"""
The device site counter (bin3c_b200/csrc/sites.cu, seq_sites.fasta_site_table(device=True)) against the host counter:
the same dict, the same keys in the same order, Python ints, for every file of tests/fasta_cases.py at slabs of 1, 7 and
4096 bytes and the default, plain and gzip'd, with and without tips; and ContactMap(gpu_sites=True) against
gpu_sites=False.
"""
import gzip
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import bam_writer                                   # noqa: E402
import fasta_cases                                  # noqa: E402
from bin3c_b200 import seq_sites                    # noqa: E402

pytestmark = pytest.mark.gpu
SLABS = (1, 7, 4096, seq_sites.DEFAULT_SLAB_BYTES)


@pytest.fixture(scope='module')
def torch():
    t = pytest.importorskip('torch')
    if not t.cuda.is_available():
        pytest.skip('needs a CUDA device')
    return t


def _ints(info):
    for v in info.values():
        s = v['sites']
        assert type(v['length']) is int and all(type(x) is int for x in (s if isinstance(s, list) else [s]))


def _same(path, enzymes=fasta_cases.ENZYMES, min_len=0, tip_size=None, slabs=SLABS):
    want = seq_sites.fasta_site_table(str(path), enzymes, min_len, tip_size=tip_size)
    for slab in slabs:
        got = seq_sites.fasta_site_table(str(path), enzymes, min_len, tip_size=tip_size, device=True, slab_bytes=slab)
        assert list(got.items()) == list(want.items()), slab
        _ints(got)
    return want


def _write(tmp_path, data, name='a.fa'):
    p = tmp_path / name
    p.write_bytes(data)
    return p


@pytest.mark.parametrize('name', sorted(fasta_cases.fixed_cases()))
def test_device_equals_host_counter(torch, tmp_path, name):
    _same(_write(tmp_path, fasta_cases.fixed_cases()[name]))


def test_every_builtin_enzyme_and_duplicates(torch, tmp_path):
    rich = b'>all\n' + b''.join(s.encode() for s in seq_sites.RECOGNITION.values()) * 3 + b'\n'
    for data in (fasta_cases.random_fasta(11, n_records=20), rich):
        p = _write(tmp_path, data)
        for enz in (sorted(seq_sites.RECOGNITION), ['DpnII', 'MboI'], ['HinfI', 'DdeI', 'ApoI']):
            _same(p, enz)


def test_non_palindromic_site(torch, tmp_path, monkeypatch):
    monkeypatch.setitem(seq_sites.RECOGNITION, 'BbsI', 'GAAGAC')
    want = _same(_write(tmp_path, b'>a\nGAAGACGTCTTCGAAG\nAC\n>b\ngtcttc\n'), ['BbsI', 'MluCI'])
    assert want['a']['sites'] == 3 and want['b']['sites'] == 1
    _same(_write(tmp_path, fasta_cases.random_fasta(12)), ['BbsI', 'HinfI'])


def test_min_len_boundary(torch, tmp_path):
    p = _write(tmp_path, fasta_cases.fixed_cases()['lf'])     # a: 12 bases, b: 8
    for min_len in (7, 8, 9, 12, 13):
        _same(p, min_len=min_len)


@pytest.mark.parametrize('tip_size', [1, 4, 8, 13])
def test_tip_windows(torch, tmp_path, tip_size):
    _same(_write(tmp_path, fasta_cases.tip_case()), tip_size=tip_size)
    _same(_write(tmp_path, fasta_cases.fixed_cases()['ws_run_across']), tip_size=tip_size)


def test_tip_windows_of_long_sequences(torch, tmp_path):
    p = _write(tmp_path, fasta_cases.fixed_cases()['long_line'])
    for tip_size in (100, 7499, 7500, 7501, 20000):
        _same(p, tip_size=tip_size, slabs=(7, 4096, seq_sites.DEFAULT_SLAB_BYTES))


@pytest.mark.parametrize('members', [1, 3])
def test_gzip(torch, tmp_path, members):
    data = fasta_cases.random_fasta(21, n_records=25) + fasta_cases.fixed_cases()['long_line']
    cut = [len(data) * k // members for k in range(members + 1)]
    p = _write(tmp_path, b''.join(gzip.compress(data[a:b]) for a, b in zip(cut, cut[1:])), 'a.fa.gz')
    want = _same(p, slabs=(7, 4096, seq_sites.DEFAULT_SLAB_BYTES))
    assert want == seq_sites.fasta_site_table(str(_write(tmp_path, data)), fasta_cases.ENZYMES)
    _same(p, tip_size=50, slabs=(4096,))


def test_byte_above_0x7f_in_a_sequence_line_raises(torch, tmp_path):
    p = _write(tmp_path, b'>caf\xc3\xa9 ok\nGATC\n>b\nGATC\xc3\xa9AATT\n')
    for slab in (1, 7, seq_sites.DEFAULT_SLAB_BYTES):
        with pytest.raises(ValueError, match='host counter'):
            seq_sites.fasta_site_table(str(p), fasta_cases.ENZYMES, device=True, slab_bytes=slab)
    _same(_write(tmp_path, b'>caf\xc3\xa9 x\nGATC\n'))


def test_seeded_assembly_200mbp(torch, tmp_path):
    p = tmp_path / 'asm.fa'
    n = fasta_cases.seeded_assembly(str(p), 200_000_000, seed=5)
    want = _same(p, slabs=(seq_sites.DEFAULT_SLAB_BYTES,))
    assert len(want) == n and sum(v['length'] for v in want.values()) >= 200_000_000


def _hic_setup(tmp_path):
    rng = np.random.default_rng(2718)
    n_refs = 90
    lengths = rng.integers(600, 4000, n_refs)
    seqs = [''.join(rng.choice(list('ACGT'), int(ln))) for ln in lengths]
    names = ['ctg%03d' % i for i in range(n_refs)]
    fasta = str(tmp_path / 'asm.fa')
    with open(fasta, 'w') as fh:
        for i, (nm, sq) in enumerate(zip(names, seqs)):
            if i == 7:
                continue
            fh.write('>{} some description\n'.format(nm))
            for k in range(0, len(sq), 70):
                fh.write(sq[k:k + 70] + '\n')
    alns = []
    for k in range(40_000):
        a = int(rng.integers(n_refs))
        b = a if rng.random() < 0.6 else int((a + rng.integers(1, 6)) % n_refs)
        good = rng.random() < 0.85
        proper = a == b and rng.random() < 0.5
        p1 = int(rng.integers(0, max(1, lengths[a] - 300)))
        p2 = p1 + int(rng.integers(50, 900)) if proper else int(rng.integers(0, max(1, lengths[b] - 100)))
        f1, f2 = 0x41 | (0x2 if proper else 0), 0x81 | (0x2 if proper else 0)
        if rng.random() < 0.5:
            (a, p1, f1), (b, p2, f2) = (b, p2, f2), (a, p1, f1)
        alns.append(dict(name='q%06d' % k, flag=f1, tid=a, pos=p1, mapq=60 if good else 11, cigar=[(0, 100)]))
        alns.append(dict(name='q%06d' % k, flag=f2, tid=b, pos=p2, mapq=60, cigar=[(0, 100)]))
    path = str(tmp_path / 'hic.bam')
    bam_writer.write_bam(path, names, lengths.tolist(), alns, block_bytes=40000, level=1)
    return path, fasta


@pytest.mark.parametrize('gpu_decode', [False, True])
def test_contact_map_with_gpu_sites(torch, tmp_path, gpu_decode):
    from bin3c_b200 import cluster
    from bin3c_b200.contact_map import ContactMap
    path, fasta = _hic_setup(tmp_path)
    maps = {}
    for flag in (False, True):
        cm = ContactMap(path, ['MluCI', 'Sau3AI'], fasta, 400, 60, min_len=1000, min_sig=2, random_seed=1,
                        gpu_decode=gpu_decode, gpu_sites=flag)
        maps[flag] = (cm.seq_map, dict(cm.pair_counts), cluster.to_edges(cm, norm=True, bisto=True, scale=True),
                      [(s.name, s.length, s.sites) for s in cm.seq_info])
    (sa, ca, ea, ia), (sb, cb, eb, ib) = maps[False], maps[True]
    assert np.array_equal(sa.row, sb.row) and np.array_equal(sa.col, sb.col) and np.array_equal(sa.data, sb.data)
    assert ca == cb and ia == ib
    for x, y in zip(ea[:3], eb[:3]):
        assert np.array_equal(x, y)
    assert ea[3] == eb[3]


def test_contact_map_with_gpu_sites_and_tips(torch, tmp_path):
    from bin3c_b200.contact_map import ContactMap
    path, fasta = _hic_setup(tmp_path)
    maps = {}
    for flag in (False, True):
        cm = ContactMap(path, ['MluCI', 'Sau3AI'], fasta, 400, 60, min_len=1000, min_sig=2, random_seed=1,
                        tip_size=500, gpu_sites=flag)
        assert cm.is_tipbased()
        maps[flag] = (cm.seq_map, dict(cm.pair_counts), [(s.name, s.length, s.sites) for s in cm.seq_info],
                      cm.get_primary_acceptance_mask())
    (sa, ca, ia, ma), (sb, cb, ib, mb) = maps[False], maps[True]
    assert np.array_equal(sa.coords, sb.coords) and np.array_equal(sa.data, sb.data)
    assert ca == cb and ia == ib and np.array_equal(ma, mb)
    assert all(isinstance(s, list) and len(s) == 2 for _, _, s in ib)
