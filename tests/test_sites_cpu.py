"""
CPU side of the device site counter: the state machine and matcher of bin3c_b200/csrc/sites.cuh, built with g++
through tests/native/sites_check.cpp and run the way sites.cu runs them, over slab cuts of 1, 7, 4096 bytes, random
cuts and one slab, against seq_sites.fasta_site_table; and the argument checks of fasta_site_table(device=True) that
come before any device work.
"""
import gzip
import os
import shutil
import struct
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import fasta_cases                                  # noqa: E402
from bin3c_b200 import seq_sites                    # noqa: E402
from bin3c_b200.exceptions import UnknownEnzymeException      # noqa: E402

SRC = os.path.join(ROOT, 'tests', 'native', 'sites_check.cpp')
CUTS = ['1', '7', '4096', str(1 << 26), 'r1', 'r2']


@pytest.fixture(scope='module')
def tool(tmp_path_factory):
    if shutil.which('g++') is None:
        pytest.skip('no g++')
    exe = str(tmp_path_factory.mktemp('sites') / 'sites_check')
    res = subprocess.run(['g++', '-std=c++17', '-O2', '-Wall', '-Werror', SRC, '-o', exe], stdout=subprocess.PIPE,
                         stderr=subprocess.STDOUT, text=True)
    assert res.returncode == 0, res.stdout
    return exe


def _pattern_file(path, enzymes):
    masks, lengths, weights = fasta_cases.device_patterns(enzymes)
    with open(path, 'wb') as f:
        f.write(struct.pack('<i', len(lengths)))
        for m, n, w in zip(masks, lengths, weights):
            f.write(struct.pack('<ii', int(n), int(w)) + m.tobytes())


def _harness(tool, tmp_path, data, enzymes, cut, min_len=0, tip_size=None):
    fa, pf, out = tmp_path / 'in.fa', tmp_path / 'pat.bin', tmp_path / 'out.bin'
    fa.write_bytes(data)
    _pattern_file(pf, enzymes)
    res = subprocess.run([tool, str(fa), str(pf), str(tip_size or 0), cut, str(out)], stdout=subprocess.PIPE,
                         stderr=subprocess.PIPE, text=True, timeout=300)
    if res.returncode == 3:
        raise ValueError(res.stdout)
    assert res.returncode == 0, res.stderr
    raw = out.read_bytes()
    n, na = struct.unpack('<qq', raw[:16])
    rows = np.frombuffer(raw[16:16 + 40 * n], dtype=np.int64)
    return seq_sites.site_table_from_rows(rows, raw[16 + 40 * n:16 + 40 * n + na], min_len, tip_size)


def _host(tmp_path, data, enzymes, min_len=0, tip_size=None):
    fa = tmp_path / 'host.fa'
    fa.write_bytes(data)
    return seq_sites.fasta_site_table(str(fa), enzymes, min_len, tip_size=tip_size)


def _same(tool, tmp_path, data, enzymes=fasta_cases.ENZYMES, min_len=0, tip_size=None, cuts=CUTS):
    want = _host(tmp_path, data, enzymes, min_len, tip_size)
    for cut in cuts:
        got = _harness(tool, tmp_path, data, enzymes, cut, min_len, tip_size)
        assert list(got.items()) == list(want.items()), cut
    return want


@pytest.mark.parametrize('name', sorted(fasta_cases.fixed_cases()))
def test_harness_equals_host_counter(tool, tmp_path, name):
    _same(tool, tmp_path, fasta_cases.fixed_cases()[name])


def test_every_builtin_enzyme_and_duplicates(tool, tmp_path):
    data = fasta_cases.random_fasta(11, n_records=20)
    rich = b'>all\n' + b''.join(s.encode() for s in seq_sites.RECOGNITION.values()) * 3 + b'\n'
    for enz in (sorted(seq_sites.RECOGNITION), ['DpnII', 'MboI'], ['HinfI', 'DdeI', 'ApoI']):
        for d in (data, rich):
            _same(tool, tmp_path, d, enz, cuts=['1', '7', 'r3', str(1 << 26)])


def test_non_palindromic_site_counts_both_strands(tool, tmp_path, monkeypatch):
    monkeypatch.setitem(seq_sites.RECOGNITION, 'BbsI', 'GAAGAC')
    data = b'>a\nGAAGACGTCTTCGAAG\nAC\n>b\ngtcttc\n'
    want = _same(tool, tmp_path, data, ['BbsI', 'MluCI'])
    assert want['a']['sites'] == 3 and want['b']['sites'] == 1


def test_min_len_boundary(tool, tmp_path):
    data = fasta_cases.fixed_cases()['lf']                  # a: 12 bases, b: 8
    for min_len in (7, 8, 9, 12, 13):
        _same(tool, tmp_path, data, min_len=min_len)


@pytest.mark.parametrize('tip_size', [1, 4, 8, 13])
def test_tip_windows(tool, tmp_path, tip_size):
    _same(tool, tmp_path, fasta_cases.tip_case(), tip_size=tip_size)
    _same(tool, tmp_path, fasta_cases.fixed_cases()['mixed_no_final_eol'], tip_size=tip_size)
    _same(tool, tmp_path, fasta_cases.fixed_cases()['ws_run_across'], tip_size=tip_size)


def test_tip_windows_of_long_sequences(tool, tmp_path):
    data = fasta_cases.fixed_cases()['long_line']
    for tip_size in (100, 7499, 7500, 7501, 20000):
        _same(tool, tmp_path, data, tip_size=tip_size, cuts=['7', '4096', 'r4'])


def test_byte_above_0x7f_in_a_sequence_line_is_refused(tool, tmp_path):
    data = b'>caf\xc3\xa9 ok\nGATC\n>b\nGATC\xc3\xa9AATT\n'
    assert _host(tmp_path, data, fasta_cases.ENZYMES)['b']['length'] == 9      # one character, two bytes
    with pytest.raises(ValueError, match='ERR 22 195'):
        _harness(tool, tmp_path, data, fasta_cases.ENZYMES, '7')
    # in a header it is only part of the name
    ok = b'>caf\xc3\xa9 x\nGATC\n'
    assert _same(tool, tmp_path, ok) == {'caf\xe9': {'sites': 1, 'length': 4}}


def test_device_without_cuda_raises(tmp_path, monkeypatch):
    torch = pytest.importorskip('torch')
    monkeypatch.setattr(torch.cuda, 'is_available', lambda: False)
    fa = tmp_path / 'a.fa'
    fa.write_bytes(b'>a\nGATC\n')
    with pytest.raises(RuntimeError, match='host counter'):
        seq_sites.fasta_site_table(str(fa), ['MluCI'], device=True)


def test_bad_enzymes_and_long_sites_raise_before_device_work(tmp_path, monkeypatch):
    torch = pytest.importorskip('torch')

    def no_device():
        raise AssertionError('device work started')
    monkeypatch.setattr(torch.cuda, 'is_available', no_device)
    fa = tmp_path / 'a.fa'
    fa.write_bytes(b'>a\nGATC\n')
    with pytest.raises(UnknownEnzymeException):
        seq_sites.fasta_site_table(str(fa), ['HindII'], device=True)
    monkeypatch.setitem(seq_sites.RECOGNITION, 'Long', 'GATC' * 4 + 'A')
    with pytest.raises(ValueError, match='17 bases'):
        seq_sites.fasta_site_table(str(fa), ['MluCI', 'Long'], device=True)
    # 16 bases is still taken (the check passes and the device step is reached)
    monkeypatch.setitem(seq_sites.RECOGNITION, 'Long', 'GATC' * 4)
    with pytest.raises(AssertionError, match='device work started'):
        seq_sites.fasta_site_table(str(fa), ['Long'], device=True)


def test_gzip_host_counter_reads_multi_member(tmp_path):
    """the device path reads .gz files with gzip.open like the host counter, members one after the other"""
    data = fasta_cases.random_fasta(5)
    fa = tmp_path / 'm.fa.gz'
    fa.write_bytes(gzip.compress(data[:len(data) // 2]) + gzip.compress(data[len(data) // 2:]))
    plain = tmp_path / 'm.fa'
    plain.write_bytes(data)
    assert seq_sites.fasta_site_table(str(fa), fasta_cases.ENZYMES) == \
        seq_sites.fasta_site_table(str(plain), fasta_cases.ENZYMES)
