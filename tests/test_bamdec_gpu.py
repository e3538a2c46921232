"""
The GPU BAM decoder (bin3c_b200/csrc/bamdec.cu, bam_io.pair_records_from_bam(device=True)) against the host reader
(libbin3c_io.so), which is itself pinned to the reference's pairing loop (tests/test_io.py): the same records in the same
order and the same stats, for every block cut, slab size, matcher mode and error the host reader handles.
"""
import os
import random
import struct
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import bam_writer                                   # noqa: E402
from bin3c_b200 import bam_io                       # noqa: E402
from test_io import random_alignments, lut_for, _golden_binmap      # noqa: E402

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def torch():
    t = pytest.importorskip('torch')
    if not t.cuda.is_available():
        pytest.skip('needs a CUDA device')
    return t


def _host(path, sites=None, min_mapq=60, strong=None, min_insert=None, min_len=None):
    rec, st = bam_io.pair_records_from_bam(path, sites=sites, min_mapq=min_mapq, strong=strong, min_insert=min_insert,
                                           min_len=min_len)
    return rec.records, st


def _same(torch, path, **kw):
    """Decode on the device and on the host; assert equal records and stats; return them."""
    dev_kw = {k: kw.pop(k) for k in ('slab_bytes', 'slab_blocks') if k in kw}
    want, st_host = _host(path, **kw)
    pr, st_dev = bam_io.pair_records_from_bam(path, device=True, **dict(kw, **dev_kw))
    got = pr.records
    assert isinstance(got, torch.Tensor) and got.is_cuda and got.dtype == torch.uint64
    assert torch.equal(got.cpu(), torch.from_numpy(want)), 'records differ from the host reader'
    assert st_dev == st_host
    return want, st_host, pr


def write_record_aligned(path, refs, lengths, alns, level=6, limit=65280):
    """A BAM file cut the way htslib cuts it: the header in its own blocks, then a block is flushed before a record
    that would not fit, so every block starts a record."""
    head = bam_writer.encode_header(refs, lengths)
    with open(path, 'wb') as out:
        for o in range(0, len(head), limit):
            out.write(bam_writer.bgzf_block(head[o:o + limit], level))
        cur = b''
        for a in alns:
            r = bam_writer.encode_alignment(a)
            if cur and len(cur) + len(r) > limit:
                out.write(bam_writer.bgzf_block(cur, level))
                cur = b''
            cur += r
        if cur:
            out.write(bam_writer.bgzf_block(cur, level))
        out.write(bam_writer.BGZF_EOF)


def _community(seed, n_templates=3000, n_refs=40):
    rng = random.Random(seed)
    refs = ['contig_{}'.format(i) for i in range(n_refs)]
    lengths = [rng.choice([300, 800, 1500, 20000]) for _ in range(n_refs)]
    return refs, lengths, random_alignments(rng, n_refs, n_templates)


MODES = {'mapq': dict(min_mapq=30), 'strong': dict(min_mapq=30, strong=40),
         'insert': dict(min_mapq=30, min_insert=1200, min_len=1000)}


@pytest.mark.parametrize('level', [1, 6])
@pytest.mark.parametrize('block_bytes', [4096, 8000, 20000, 65280])
@pytest.mark.parametrize('mode', ['mapq', 'strong', 'insert'])
def test_device_records_equal_the_host_reader(torch, tmp_path, mode, block_bytes, level):
    refs, lengths, alns = _community(block_bytes + level)
    path = str(tmp_path / 'x.bam')
    bam_writer.write_bam(path, refs, lengths, alns, block_bytes=block_bytes, level=level)
    want, st, _ = _same(torch, path, **MODES[mode])
    assert len(want) > 500 and st['unpaired'] > 0
    if mode == 'insert':
        assert st['short_insert'] > 0


@pytest.mark.parametrize('mode', ['mapq', 'strong', 'insert'])
def test_record_aligned_blocks(torch, tmp_path, mode):
    refs, lengths, alns = _community(31, 6000)
    path = str(tmp_path / 'aligned.bam')
    write_record_aligned(path, refs, lengths, alns)
    _, st, pr = _same(torch, path, **MODES[mode])
    assert pr.meta['repaired_blocks'] == 0              # every guess holds: no block walked twice
    assert st['bgzf_blocks'] > 5


@pytest.mark.parametrize('slab_blocks', [1, 2, 7])
@pytest.mark.parametrize('layout', ['cut', 'aligned'])
def test_small_slabs(torch, tmp_path, slab_blocks, layout):
    """Slabs of 1, 2 and 7 blocks: records straddle slabs, a pending first mate ends a slab, and the file ends with
    an orphan."""
    refs, lengths, alns = _community(slab_blocks, 1500)
    alns.append(dict(name='zz_last_orphan', flag=0x41, tid=1, pos=5, mapq=60, cigar=[(0, 50)]))
    path = str(tmp_path / 's.bam')
    if layout == 'cut':
        bam_writer.write_bam(path, refs, lengths, alns, block_bytes=1500, level=6)
    else:
        write_record_aligned(path, refs, lengths, alns, limit=3000)
    want, st, pr = _same(torch, path, slab_bytes=1, slab_blocks=slab_blocks, **MODES['insert'])
    assert pr.meta['slabs'] >= st['bgzf_blocks'] // slab_blocks
    # the same file in one slab gives the same records
    _same(torch, path, **MODES['insert'])
    # a record longer than a whole slab: 2000 bytes of tags in 1500-byte blocks
    big = [dict(a, tags=b'XZZ' + b'q' * 2000 + b'\0') if k % 50 == 0 else a for k, a in enumerate(alns)]
    path2 = str(tmp_path / 'big.bam')
    bam_writer.write_bam(path2, refs, lengths, big, block_bytes=1500, level=1)
    _same(torch, path2, slab_bytes=1, slab_blocks=slab_blocks, **MODES['strong'])


def test_long_cigar_in_cg_tag(torch, tmp_path):
    """The CG:B,I tag behind the <l_seq>S<span>N placeholder carries the real CIGAR (the file of
    test_io.test_bam_long_cigar_in_cg_tag_and_reverse_read_without_cigar)."""
    refs, lengths = ['a', 'b'], [50000, 40000]
    real = [(0, 30), (2, 5), (0, 20), (1, 2), (3, 1000), (0, 40)]
    l_seq = sum(n for op, n in real if op in (0, 1, 4, 7, 8))
    tag = b'CGBI' + struct.pack('<I', len(real)) + b''.join(struct.pack('<I', (n << 4) | op) for op, n in real)
    other = b'NMC\x03' + b'XZZabc\0'
    alns = [dict(name='p0', flag=0x41 | 0x10, tid=0, pos=1000, mapq=60, cigar=[(4, l_seq), (3, 1095)], seq_len=l_seq,
                 tags=other + tag),
            dict(name='p0', flag=0x81, tid=1, pos=700, mapq=60, cigar=[(0, 100)])]
    path = str(tmp_path / 'cg.bam')
    bam_writer.write_bam(path, refs, lengths, alns)
    want, _, _ = _same(torch, path, min_mapq=30, strong=35)
    assert len(want) == 1 and (int(want[0]) >> 31) & 1 == 1
    want, _, _ = _same(torch, path, min_mapq=30, strong=41)
    assert (int(want[0]) >> 31) & 1 == 0
    bad = [dict(name='q', flag=0x41 | 0x10, tid=0, pos=10, mapq=60, cigar=[]),
           dict(name='q', flag=0x81, tid=1, pos=20, mapq=60, cigar=[(0, 50)])]
    path2 = str(tmp_path / 'nocigar.bam')
    bam_writer.write_bam(path2, refs, lengths, bad)
    want, _, _ = _same(torch, path2, min_mapq=30, strong=10)
    assert len(want) == 1


def test_reference_bin_map_counts_through_the_gpu_decoder(torch, tmp_path):
    """tests/golden/binmap.npz: what the reference's own ContactMap._bin_map produced.  The records the GPU decoder
    extracts from a BAM file of the same alignments reproduce its contig map and counters."""
    from oracle import oracle
    g, alns = _golden_binmap()
    lengths = g['lengths']
    n_refs = len(lengths)
    keep = lengths >= int(g['min_len'])
    lut = np.where(keep, np.cumsum(keep) - 1, -1).astype(np.int32)
    n_seq = int(keep.sum())
    path = str(tmp_path / 'g.bam')
    bam_writer.write_bam(path, ['r%d' % i for i in range(n_refs)], lengths.tolist(), alns, block_bytes=20000, level=1)
    for k in range(int(g['n_params'])):
        kw = dict(min_mapq=int(g['p%d_min_mapq' % k]), strong=int(g['p%d_strong' % k]) or None,
                  min_insert=int(g['p%d_min_insert' % k]) or None)
        pr, st = bam_io.pair_records_from_bam(path, device=True, min_len=int(g['min_len']), **kw)
        rec = pr.records.cpu().numpy()
        m31 = np.uint64(0x7fffffff)
        ok = ((rec >> np.uint64(31)) & np.uint64(1)).astype(bool)
        dok, counts = oracle.bin_pairs_loop((rec & m31).astype(np.int64), ((rec >> np.uint64(32)) & m31).astype(np.int64),
                                            ok, {t: int(i) for t, i in enumerate(lut) if i >= 0}, n_seq)
        m = oracle.dok_to_coo(dok, n_seq)
        assert [counts['accepted'], counts['ref_excluded'], counts['poor_match'], st['short_insert']] == \
            g['p%d_counts' % k].tolist()
        assert m.shape[0] == int(g['p%d_seq_map_n' % k])
        assert np.array_equal(m.row, g['p%d_seq_map_row' % k]) and np.array_equal(m.col, g['p%d_seq_map_col' % k])
        assert np.array_equal(m.data, g['p%d_seq_map_data' % k])


def _stream_file(path, stream, block_bytes=4096, eof=True):
    with open(path, 'wb') as out:
        for o in range(0, len(stream), block_bytes):
            out.write(bam_writer.bgzf_block(stream[o:o + block_bytes], 6))
        if eof:
            out.write(bam_writer.BGZF_EOF)


def _raises_like_host(torch, path, exc=ValueError):
    with pytest.raises(exc):
        _host(path, min_mapq=20)
    with pytest.raises(exc):
        bam_io.pair_records_from_bam(path, device=True, min_mapq=20, slab_bytes=20000)


def test_malformed_files_raise_like_the_host_reader(torch, tmp_path):
    refs, lengths, alns = _community(77, 1500)
    good = str(tmp_path / 'good.bam')
    bam_writer.write_bam(good, refs, lengths, alns, block_bytes=4096)
    raw = open(good, 'rb').read()
    cases = {}
    cases['truncated'] = raw[:len(raw) * 2 // 3]
    cases['truncated_record'] = None
    offs, o = [], 0
    while o < len(raw):
        offs.append(o)
        o += struct.unpack_from('<H', raw, o + 16)[0] + 1
    b = bytearray(raw)
    mid = offs[len(offs) // 2]
    end = offs[len(offs) // 2 + 1]
    b[end - 8] ^= 0x01                                   # the CRC in the trailer
    cases['crc'] = bytes(b)
    b = bytearray(raw)
    for k in range(3):
        b[mid + 18 + 11 * k] ^= 0xff                     # the deflate payload
    cases['deflate'] = bytes(b)
    # record-level errors, in the uncompressed stream
    head = bam_writer.encode_header(refs, lengths)
    recs = [bam_writer.encode_alignment(a) for a in alns]
    k = len(recs) // 2
    over = bytearray(recs[k])
    struct.pack_into('<H', over, 4 + 12, 0xffff)         # n_cigar_op: 32 + l_name + 4 n_cig > block_size
    short = struct.pack('<i', 20) + b'\0' * 20           # block_size below the fixed fields
    stream_over = head + b''.join(recs[:k]) + bytes(over) + b''.join(recs[k + 1:])
    stream_short = head + b''.join(recs[:k]) + short + b''.join(recs[k:])
    stream_cut = head + b''.join(recs)[:-7]              # the file ends inside the last record
    unterm = dict(name='u', flag=0x41, tid=0, pos=10, mapq=60, cigar=[(4, 10), (3, 100)], seq_len=10,
                  tags=b'XZZabc')                        # CG placeholder: the tags are read; no NUL
    stream_unterm = head + b''.join(recs[:k]) + bam_writer.encode_alignment(unterm) + b''.join(recs[k:])
    for name, stream in (('overrun', stream_over), ('short', stream_short), ('cut', stream_cut),
                         ('unterminated', stream_unterm)):
        p = str(tmp_path / (name + '.bam'))
        _stream_file(p, stream)
        cases[name] = open(p, 'rb').read()
    cases.pop('truncated_record')
    for name, data in cases.items():
        p = str(tmp_path / (name + '.bam'))
        with open(p, 'wb') as f:
            f.write(data)
        _raises_like_host(torch, p)
        _same(torch, good, min_mapq=20)                  # the process decodes the next file exactly
    # not name-sorted: IOError, as the host reader
    p = str(tmp_path / 'coord.bam')
    bam_writer.write_bam(p, refs, lengths, alns, sort_order='coordinate')
    _raises_like_host(torch, p, IOError)
    # an empty alignment section without an EOF marker
    p = str(tmp_path / 'empty.bam')
    bam_writer.write_bam(p, refs, lengths, [], eof_marker=False)
    want, st, _ = _same(torch, p)
    assert len(want) == 0 and st['alignments'] == 0


def test_contact_map_with_gpu_decode(torch, tmp_path):
    """ContactMap(bam path, ..., gpu_decode=True) on the setup of test_contact_map_from_bam_and_fasta_paths: the same
    contact map, counters and edges as with the host reader."""
    from bin3c_b200 import cluster
    from bin3c_b200.contact_map import ContactMap
    rng = np.random.default_rng(2718)
    n_refs, min_len, min_insert = 90, 1000, 400
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
    maps = {}
    for flag in (False, True):
        cm = ContactMap(path, ['MluCI', 'Sau3AI'], fasta, min_insert, 60, min_len=min_len, min_sig=2, random_seed=1,
                        gpu_decode=flag)
        maps[flag] = (cm.seq_map, dict(cm.pair_counts), cluster.to_edges(cm, norm=True, bisto=True, scale=True))
    (sa, ca, ea), (sb, cb, eb) = maps[False], maps[True]
    assert np.array_equal(sa.row, sb.row) and np.array_equal(sa.col, sb.col) and np.array_equal(sa.data, sb.data)
    assert sa.data.dtype == sb.data.dtype and sa.shape == sb.shape
    assert ca == cb and ca['short_insert'] > 100
    for x, y in zip(ea[:3], eb[:3]):
        assert np.array_equal(x, y)
    assert ea[3] == eb[3]
