"""
Host IO library (include/bin3c_io.h, SURVEY.md 8f ranks 1 and 2): BAM -> packed pair records against the
oracle's restatement of the reference pairing loop (contact_map.py:612-629, :720-766), and the edge-list
writer against what nx.write_edgelist prints (cluster.py:139-151).  CPU only.
"""
import os
import random
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import bam_writer                                   # noqa: E402
from bin3c_b200 import bam_io                       # noqa: E402
from oracle import oracle, ref_exec                 # noqa: E402


def random_alignments(rng, n_refs, n_templates, weird=True):
    """A name-sorted alignment stream with everything the pairing loop looks at."""
    alns = []
    for t in range(n_templates):
        name = 'read{:07d}'.format(t) if rng.random() < 0.9 else 'r{}'.format(t)
        kind = rng.random()
        n_rec = 2 if kind < 0.75 else rng.choice([1, 1, 3, 4])
        for k in range(n_rec):
            flag = 0x1 | (0x40 if k % 2 == 0 else 0x80)
            if rng.random() < 0.5:
                flag |= 0x10
            if rng.random() < 0.6:
                flag |= 0x2
            if weird and rng.random() < 0.08:
                flag |= rng.choice([0x4, 0x100, 0x800])
            tid = rng.randrange(n_refs)
            if weird and rng.random() < 0.01:
                tid = n_refs + 3                               # out of the header's table
            if rng.random() < 0.1:
                cigar = []
            else:
                m = rng.randrange(1, 150)
                cigar = [(0, m)]
                if rng.random() < 0.3:
                    cigar = [(4, rng.randrange(1, 30))] + cigar
                if rng.random() < 0.3:
                    cigar = cigar + [(4, rng.randrange(1, 30))]
            alns.append(dict(name=name, flag=flag, tid=tid, pos=rng.randrange(0, 5000), mapq=rng.randrange(0, 61),
                             cigar=cigar))
    return alns


def lut_for(lengths, min_len):
    keep = np.asarray(lengths) >= min_len
    return np.where(keep, np.cumsum(keep) - 1, -1).astype(np.int32)


@pytest.mark.parametrize('block_bytes,threads', [(65280, 0), (997, 3), (64, 1)])
@pytest.mark.parametrize('mode', ['mapq', 'strong', 'insert'])
def test_bam_pairs_match_oracle(tmp_path, block_bytes, threads, mode):
    rng = random.Random(block_bytes * 7 + len(mode))
    n_refs = 40
    refs = ['contig_{}'.format(i) for i in range(n_refs)]
    lengths = [rng.choice([300, 800, 1500, 20000]) for _ in range(n_refs)]
    alns = random_alignments(rng, n_refs, 3000 if block_bytes > 100 else 300)
    path = str(tmp_path / 'x.bam')
    bam_writer.write_bam(path, refs, lengths, alns, block_bytes=block_bytes)
    kw = dict(min_mapq=30)
    if mode == 'strong':
        kw['strong'] = 40
    lut = None
    if mode == 'insert':
        kw['min_insert'] = 1200
        lut = lut_for(lengths, 1000)
    want, st = oracle.pair_alignments(alns, n_refs, idx_of=lut, **kw)
    with bam_io.BamPairReader(path, threads=threads) as bam:
        assert bam.references == refs
        assert bam.lengths.tolist() == lengths
        assert '@HD' in bam.header_text and 'SO:queryname' in bam.header_text
        bam.set_filter(tid2idx=lut, **kw)
        parts = []
        while True:                                            # odd chunk size: records continue across calls
            r = bam.read_pairs(701)
            if len(r) == 0:
                break
            parts.append(r.copy())
        got = np.concatenate(parts) if parts else np.empty(0, np.uint64)
        stats = bam.stats()
    assert np.array_equal(got, want)
    for k in ('alignments', 'informative', 'pairs', 'short_insert', 'unpaired'):
        assert stats[k] == st[k], k
    assert stats['uncompressed_bytes'] > 0 and stats['bgzf_blocks'] >= 2
    if mode == 'insert':
        assert st['short_insert'] > 0


def test_bam_large_multibatch(tmp_path):
    """More than one batch of BGZF blocks (256 blocks each) and many threads."""
    rng = random.Random(7)
    n_refs = 500
    refs = ['c{}'.format(i) for i in range(n_refs)]
    lengths = [1000 + i for i in range(n_refs)]
    alns = random_alignments(rng, n_refs, 60000, weird=True)
    path = str(tmp_path / 'big.bam')
    bam_writer.write_bam(path, refs, lengths, alns, block_bytes=8000, level=1)
    want, st = oracle.pair_alignments(alns, n_refs, min_mapq=20)
    with bam_io.BamPairReader(path, threads=8) as bam:
        bam.set_filter(min_mapq=20)
        got = bam.read_all(chunk=10000)
        stats = bam.stats()
    assert stats['bgzf_blocks'] > 600
    assert np.array_equal(got, want)
    assert stats['pairs'] == st['pairs'] and stats['unpaired'] == st['unpaired']


def test_pair_records_from_bam_feeds_the_oracle_path(tmp_path):
    """BAM -> PairRecords -> the same (tid_i, tid_j, pass) arrays the accumulation oracle takes."""
    rng = random.Random(11)
    n_refs = 30
    refs = ['s{}'.format(i) for i in range(n_refs)]
    lengths = [rng.choice([500, 5000]) for _ in range(n_refs)]
    alns = random_alignments(rng, n_refs, 2000, weird=False)
    path = str(tmp_path / 'p.bam')
    bam_writer.write_bam(path, refs, lengths, alns)
    pr, stats = bam_io.pair_records_from_bam(path, min_mapq=10)
    assert pr.references == refs and pr.lengths.tolist() == lengths
    rec = pr.records
    ti = (rec & np.uint64(0x7fffffff)).astype(np.int64)
    tj = ((rec >> np.uint64(32)) & np.uint64(0x7fffffff)).astype(np.int64)
    ok = ((rec >> np.uint64(31)) & np.uint64(1)).astype(bool)
    lut = lut_for(lengths, 1000)
    n_seq = int((lut >= 0).sum())
    want, _ = oracle.pair_alignments(alns, n_refs, min_mapq=10)
    assert np.array_equal(rec, want) and stats['pairs'] == len(rec)
    # the records drive the accumulation oracle exactly as records from the synthetic generator do
    dok, counts = oracle.bin_pairs_loop(ti, tj, ok, {t: int(i) for t, i in enumerate(lut) if i >= 0}, n_seq)
    assert counts['accepted'] > 100
    assert counts['accepted'] + counts['ref_excluded'] + counts['poor_match'] == len(rec)
    assert sum(dok.values()) == counts['accepted']


def test_bam_errors(tmp_path):
    refs, lengths = ['a', 'b'], [1000, 2000]
    alns = [dict(name='q', flag=0x41, tid=0, pos=1, mapq=60, cigar=[(0, 50)]),
            dict(name='q', flag=0x81, tid=1, pos=9, mapq=60, cigar=[(0, 50)])]
    p1 = str(tmp_path / 'coord.bam')
    bam_writer.write_bam(p1, refs, lengths, alns, sort_order='coordinate')
    with pytest.raises(IOError, match='sorted by read name'):
        bam_io.BamPairReader(p1)
    with bam_io.BamPairReader(p1, require_queryname=False) as bam:       # the check is the caller's choice
        assert len(bam.read_all()) == 1
    p2 = str(tmp_path / 'nohd.bam')
    bam_writer.write_bam(p2, refs, lengths, alns, hd=False)
    with pytest.raises(IOError):
        bam_io.BamPairReader(p2)
    with pytest.raises(IOError):
        bam_io.BamPairReader(str(tmp_path / 'missing.bam'))
    p3 = str(tmp_path / 'garbage.bam')
    with open(p3, 'wb') as out:
        out.write(b'this is not a BGZF file at all' * 10)
    with pytest.raises(ValueError):
        bam_io.BamPairReader(p3)
    # truncated in the middle of the alignment section
    p4 = str(tmp_path / 'full.bam')
    many = []
    for t in range(500):
        many += [dict(name='t{}'.format(t), flag=0x41, tid=0, pos=1, mapq=60, cigar=[(0, 50)]),
                 dict(name='t{}'.format(t), flag=0x81, tid=1, pos=9, mapq=60, cigar=[(0, 50)])]
    bam_writer.write_bam(p4, refs, lengths, many, block_bytes=4096)
    raw = open(p4, 'rb').read()
    p5 = str(tmp_path / 'trunc.bam')
    with open(p5, 'wb') as out:
        out.write(raw[:len(raw) * 2 // 3])
    with pytest.raises(ValueError):
        with bam_io.BamPairReader(p5) as bam:
            bam.read_all()
    # a flipped payload byte fails the CRC / inflate
    p6 = str(tmp_path / 'corrupt.bam')
    bad = bytearray(raw)
    bad[len(bad) // 2] ^= 0x55
    with open(p6, 'wb') as out:
        out.write(bytes(bad))
    with pytest.raises(ValueError):
        with bam_io.BamPairReader(p6) as bam:
            bam.read_all()
    # empty alignment section, no EOF marker
    p7 = str(tmp_path / 'empty.bam')
    bam_writer.write_bam(p7, refs, lengths, [], eof_marker=False)
    with bam_io.BamPairReader(p7) as bam:
        assert len(bam.read_all()) == 0 and bam.stats()['alignments'] == 0
    # min_insert without the index table
    with bam_io.BamPairReader(p4) as bam:
        with pytest.raises(AssertionError):
            bam.set_filter(min_insert=100)
        bam.read_pairs(10)
        with pytest.raises(AssertionError):
            bam.set_filter(min_mapq=5)                                   # too late


WEIGHTS = [1.0, 0.1, 1.0 / 3.0, 2.0 / 3.0, 1e-5, 1.5e-5, 9.999e-5, 0.0001, 0.00012345678901234567, 1e15, 1e16,
           123456789012345678.0, 5e-324, 2.2250738585072014e-308, 1.7976931348623157e308, 0.0, -2.5, 100.0,
           0.30000000000000004, 1e22, 1e-7, 0.999999999999, 0.9999999999999999, 0.5, 1e12, 1e13, 999999999999.5,
           123456789012.0, 1234567890123.0, 7.0e-10, float('inf'), float('-inf'), float('nan'), -0.0]


def test_format_weight_matches_python():
    rng = np.random.default_rng(3)
    ws = list(WEIGHTS) + rng.random(2000).tolist() + (10.0 ** rng.uniform(-12, 20, 2000)).tolist() + \
        np.frombuffer(rng.bytes(8 * 2000), dtype=np.float64).tolist()
    for w in ws:
        assert bam_io.format_weight(w) == repr(float(w)), w
        t = '%.12g' % w
        if not ('.' in t or 'e' in t or 'n' in t):
            t += '.0'
        assert bam_io.format_weight(w, bam_io.FLOAT_STR12) == t, w


@pytest.mark.parametrize('n,threads', [(0, 0), (1, 1), (1000, 2), (300000, 0), (300000, 5)])
def test_write_edges_matches_networkx_text(tmp_path, n, threads):
    rng = np.random.default_rng(n + 1)
    u = rng.integers(0, 50000, n).astype(np.int32)
    v = rng.integers(0, 50000, n).astype(np.int32)
    w = rng.random(n) * 10.0 ** rng.integers(-8, 1, n)
    if n:
        w[0] = 1.0
    for style, py2 in ((bam_io.FLOAT_REPR, False), (bam_io.FLOAT_STR12, True)):
        path = str(tmp_path / 'e{}.edges'.format(style))
        nbytes = bam_io.write_edges(u, v, w, path, float_style=style, threads=threads)
        text = open(path).read()
        assert nbytes == len(text)
        assert text == oracle.edge_lines(u, v, w, py2=py2)
    if n == 1000:
        nx = pytest.importorskip('networkx')
        g = nx.Graph()
        uu, idx = np.unique(np.stack([np.minimum(u, v), np.maximum(u, v)]), axis=1, return_index=True)
        for a, b, c in zip(uu[0], uu[1], w[idx]):
            g.add_edge(int(a), int(b), weight=float(c))
        p_nx, p_b3 = str(tmp_path / 'nx.edges'), str(tmp_path / 'b3.edges')
        nx.write_edgelist(g, p_nx, data=['weight'], delimiter=' ')
        e = list(g.edges(data='weight'))
        bam_io.write_edges([a for a, _, _ in e], [b for _, b, _ in e], [c for _, _, c in e], p_b3)
        assert open(p_nx).read() == open(p_b3).read()


def test_cluster_write_edges_uses_the_native_writer(tmp_path):
    from bin3c_b200 import cluster
    u = np.array([0, 0, 1], dtype=np.int32)
    v = np.array([0, 2, 2], dtype=np.int32)
    w = np.array([1.0, 0.25, 1.0 / 3.0])
    f = cluster.write_edges(u, v, w, str(tmp_path))
    assert os.path.basename(f) == 'cm_graph.edges'
    assert open(f).read() == '0 0 1.0\n0 2 0.25\n1 2 0.3333333333333333\n'
    f = cluster.write_edges(u, v, w, str(tmp_path), base_name='py2', py2_str=True)
    assert open(f).read() == '0 0 1.0\n0 2 0.25\n1 2 0.333333333333\n'


INFOMAP = os.path.join(ref_exec.REFERENCE_ROOT, 'external', 'Infomap')


@pytest.mark.skipif(not os.access(INFOMAP, os.X_OK), reason='no reference checkout with a built Infomap binary '
                                                             '(oracle/_ref/ or $BIN3C_REFERENCE)')
def test_infomap_partition_from_native_edge_file(tmp_path):
    """
    The hand-off itself: the reference's own Infomap binary, run with the reference's flags (cluster.py:182-185) on
    the edge file the native writer produces from the golden edge list, accepts it and returns a partition of all
    nodes; the file the oracle's restatement of nx.write_edgelist writes gives the identical tree (same graph file
    -> same clustering), and so do the Python-2 ('%.12g') and Python-3 (repr) weight layouts on this community.
    """
    import subprocess
    d = np.load(os.path.join(ROOT, 'tests', 'golden', 'c1mini.npz'))
    u, v, w = d['edge_u'], d['edge_v'], d['edge_w']
    parts = {}
    for name, style, writer in (('native_repr', bam_io.FLOAT_REPR, 'native'), ('native_py2', bam_io.FLOAT_STR12, 'native'),
                                ('oracle_py2', None, 'oracle')):
        work = tmp_path / name
        work.mkdir()
        f = str(work / 'cm_graph.edges')
        if writer == 'native':
            bam_io.write_edges(u, v, w, f, float_style=style)
        else:
            with open(f, 'w') as out:
                out.write(oracle.edge_lines(u, v, w, py2=True))
        subprocess.check_call([INFOMAP, '-u', '-v', '-z', '-i', 'link-list', '-s', '1234', '-N', '10', f, str(work)],
                              stdout=subprocess.DEVNULL, stderr=subprocess.STDOUT)
        parts[name] = oracle.read_tree(str(work / 'cm_graph.tree'))
    n_nodes = int(d['sub_n'])
    for p in parts.values():
        members = sorted(m for cl in p for m in cl)
        assert members == list(range(n_nodes))                      # zero-based, gapless ids (-z)
    assert open(str(tmp_path / 'native_py2' / 'cm_graph.edges')).read() == \
        open(str(tmp_path / 'oracle_py2' / 'cm_graph.edges')).read()
    assert parts['native_py2'] == parts['oracle_py2'] == parts['native_repr']
    assert len(parts['native_py2']) > 1


@pytest.mark.parametrize('B,n_refs', [(5, 400_000), (6, 5_000_000), (8, 2 ** 31 - 2)])
def test_narrow_records_round_trip(B, n_refs):
    """b3c_records_pack / unpack: B-byte little-endian records, tid1 | pass << tb | tid2 << (tb + 1), tb = (8B - 1) / 2;
    out-of-table ids (the native 0x7fffffff marker) map to the all-ones id of the narrow layout and back."""
    assert bam_io.records_bytes(n_refs) == B
    assert bam_io.records_bytes((1 << 19) - 2) == 5 and bam_io.records_bytes((1 << 19) - 1) == 6
    assert bam_io.records_bytes((1 << 23) - 2) == 6 and bam_io.records_bytes((1 << 23) - 1) == 8
    rng = np.random.default_rng(B)
    for n in (0, 1, 5, 100_003):
        t1 = rng.integers(0, n_refs, n, dtype=np.uint64)
        t2 = rng.integers(0, n_refs, n, dtype=np.uint64)
        ok = rng.integers(0, 2, n, dtype=np.uint64)
        t1[::97] = 0x7fffffff
        rec = t1 | (ok << np.uint64(31)) | (t2 << np.uint64(32))
        packed = bam_io.pack_records(rec, B, threads=3)
        assert packed.dtype == np.uint8 and len(packed) == (n * B + 7) // 8 * 8
        assert not packed[n * B:].any()
        assert np.array_equal(bam_io.unpack_records(packed, n, B), rec)
        if n:                                     # the documented bit layout, checked independently on record 1 (or 0)
            k = min(1, n - 1)
            tb = (8 * B - 1) // 2
            v = int.from_bytes(packed[k * B:(k + 1) * B].tobytes(), 'little')
            a = int(rec[k]) & 0x7fffffff
            assert v & ((1 << tb) - 1) == min(a, (1 << tb) - 1)
            assert (v >> tb) & 1 == (int(rec[k]) >> 31) & 1
            assert (v >> (tb + 1)) & ((1 << tb) - 1) == (int(rec[k]) >> 32) & 0x7fffffff
    with pytest.raises(AssertionError):
        bam_io.pack_records(np.zeros(4, np.uint64), 7)


@pytest.mark.parametrize('sanitizer', ['thread', 'address,undefined'])
def test_io_sources_under_sanitizers(tmp_path, sanitizer):
    """The library's own sources, instrumented (TSan for the reader / inflate-pool / parser hand-over and the formatter
    pool, ASan + UBSan for the record parsing), over good, truncated and corrupted BAM files."""
    import shutil
    import subprocess
    if shutil.which('g++') is None:
        pytest.skip('no g++')
    src = os.path.join(ROOT, 'bin3c_b200', 'csrc')
    exe = str(tmp_path / 'io_sanitize')
    cmd = ['g++', '-O1', '-g', '-std=c++17', '-pthread', '-fsanitize=' + sanitizer, '-fno-omit-frame-pointer',
           os.path.join(ROOT, 'tests', 'native', 'io_sanitize.cpp'), os.path.join(src, 'io_bam.cpp'),
           os.path.join(src, 'io_edges.cpp'), '-o', exe, '-lz']
    res = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if res.returncode != 0:
        pytest.skip('sanitizer build not available here: ' + res.stdout[-300:])
    rng = random.Random(3)
    n_refs = 300
    refs = ['c{}'.format(i) for i in range(n_refs)]
    lengths = [1000 + i for i in range(n_refs)]
    alns = random_alignments(rng, n_refs, 40000, weird=True)
    good = str(tmp_path / 'good.bam')
    bam_writer.write_bam(good, refs, lengths, alns, block_bytes=6000, level=1)      # ~900 blocks: several batches
    want, _ = oracle.pair_alignments(alns, n_refs, min_mapq=20, strong=30)
    raw = open(good, 'rb').read()
    trunc, corrupt = str(tmp_path / 'trunc.bam'), str(tmp_path / 'corrupt.bam')
    open(trunc, 'wb').write(raw[:len(raw) * 3 // 5])
    bad = bytearray(raw)
    for k in range(5):
        bad[len(bad) // 7 * (k + 1)] ^= 0xa5
    open(corrupt, 'wb').write(bytes(bad))
    env = dict(os.environ, TSAN_OPTIONS='halt_on_error=1 exitcode=66', ASAN_OPTIONS='detect_leaks=1 exitcode=66',
               UBSAN_OPTIONS='halt_on_error=1 exitcode=66')
    for path, threads in ((good, 1), (good, 8), (trunc, 4), (corrupt, 4)):
        out = subprocess.run([exe, path, str(threads), '20', '30', str(tmp_path / 'e.edges')], stdout=subprocess.PIPE,
                             stderr=subprocess.PIPE, text=True, env=env, timeout=600)
        assert out.returncode == 0, out.stderr[-2000:]
        status, n, x, nbytes = out.stdout.split()
        if path == good:
            h = 0
            for r in want.tolist():
                h ^= (r * 0x9e3779b97f4a7c15) & 0xffffffffffffffff
            assert int(status) == 0 and int(n) == len(want) and int(x) == h and int(nbytes) > 0
        else:
            assert int(status) < 0


@pytest.mark.parametrize('bin_size,block_bytes', [(1000, 65280), (2500, 1999), (400, 65280)])
def test_bam_extent_records_match_oracle(tmp_path, bin_size, block_bytes):
    """The extent map's bin-level records (contact_map.py:756-788): 5'-end positions (reverse reads: pos + reference
    span of the CIGAR), find_nearest over the bin edges of ExtentGrouping, excluded references marked; against the
    oracle's restatement, together with the ordinary pair records of the same pass."""
    from bin3c_b200.contact_map import ExtentGrouping
    rng = random.Random(bin_size)
    n_refs = 60
    refs = ['contig_{}'.format(i) for i in range(n_refs)]
    lengths = [rng.choice([300, 800, 1500, 2499, 2500, 7000, 20000]) for _ in range(n_refs)]
    alns = random_alignments(rng, n_refs, 2500)
    for a in alns:                                             # richer CIGARs and positions up to the contig end
        if not a['cigar'] and a['flag'] & 0x10 and not a['flag'] & 0x4:
            a['cigar'] = [(0, 50)]          # a mapped reverse read without a CIGAR has no 5' end (separate test)
        if a['cigar'] and rng.random() < 0.5:
            a['cigar'] = a['cigar'] + [(2, rng.randrange(1, 9)), (0, rng.randrange(1, 50)), (1, 3), (3, 100)]
        if 0 <= a['tid'] < n_refs:
            a['pos'] = rng.randrange(0, lengths[a['tid']])
    path = str(tmp_path / 'x.bam')
    bam_writer.write_bam(path, refs, lengths, alns, block_bytes=block_bytes)
    lut = lut_for(lengths, 1000)
    kept = [l for l in lengths if l >= 1000]
    og = oracle.extent_grouping(kept, bin_size)
    g = ExtentGrouping.from_lengths(kept, bin_size)
    assert g.total_bins == og['total_bins'] and all(np.array_equal(a, b) for a, b in zip(g.map, og['map']))
    want, want_ext, st = oracle.pair_alignments(alns, n_refs, min_mapq=30, idx_of=lut, grouping=og)
    with bam_io.BamPairReader(path, threads=3) as bam:
        bam.set_extent(lut, g)
        bam.set_filter(min_mapq=30)                            # keeps the extent table
        recs, exts = [], []
        while True:
            r, e = bam.read_pairs_extent(997)
            if len(r) == 0:
                break
            recs.append(r.copy())
            exts.append(e.copy())
        assert bam.stats()['pairs'] == st['pairs']
    got, got_ext = np.concatenate(recs), np.concatenate(exts)
    assert np.array_equal(got, want)
    assert np.array_equal(got_ext, want_ext)
    b1 = got_ext & np.uint64(0x7fffffff)
    assert (b1[b1 != 0x7fffffff] < g.total_bins).all() and (b1 == 0x7fffffff).any()
    # through the accumulation oracle: the extent map tallies exactly the pairs the contig map accepts
    ti, tj, ok = (got & np.uint64(0x7fffffff)).astype(np.int64), ((got >> np.uint64(32)) & np.uint64(0x7fffffff)).astype(np.int64), \
        ((got >> np.uint64(31)) & np.uint64(1)).astype(bool)
    _, c_seq = oracle.bin_pairs_loop(ti, tj, ok, {t: int(i) for t, i in enumerate(lut) if i >= 0}, len(kept))
    bi, bj = (got_ext & np.uint64(0x7fffffff)).astype(np.int64), ((got_ext >> np.uint64(32)) & np.uint64(0x7fffffff)).astype(np.int64)
    dok, c_ext = oracle.bin_pairs_loop(bi, bj, ok, {b: b for b in range(g.total_bins)}, g.total_bins)
    assert c_ext == c_seq and sum(dok.values()) == c_seq['accepted']
    # pair_records_from_bam carries both
    pr, _ = bam_io.pair_records_from_bam(path, min_mapq=30, min_len=1000, bin_size=bin_size)
    assert np.array_equal(pr.records, want) and np.array_equal(pr.extent_records, want_ext)


def test_bam_extent_argument_errors(tmp_path):
    from bin3c_b200.contact_map import ExtentGrouping
    refs, lengths = ['a', 'b', 'c'], [1000, 5000, 400]
    alns = [dict(name='q', flag=0x41, tid=0, pos=1, mapq=60, cigar=[(0, 50)]),
            dict(name='q', flag=0x91, tid=1, pos=4000, mapq=60, cigar=[(0, 50), (2, 10), (0, 40)])]
    path = str(tmp_path / 'e.bam')
    bam_writer.write_bam(path, refs, lengths, alns)
    g = ExtentGrouping.from_lengths([1000, 5000], 1000)
    with bam_io.BamPairReader(path) as bam:
        with pytest.raises(AssertionError):
            bam.read_pairs_extent(10)                          # set_extent first
        with pytest.raises(AssertionError):
            bam.set_extent(np.array([0, 1], dtype=np.int32), g)            # table must cover all references
        with pytest.raises(AssertionError):
            bam.set_extent(np.array([0, 5, -1], dtype=np.int32), g)        # index outside the sequences
        bam.set_extent(np.array([0, 1, -1], dtype=np.int32), g)
        r, e = bam.read_pairs_extent(10)
        # mate 1 forward at 1 -> bin 0 of contig a; mate 2 reverse: 4000 + 100 reference bases = 4100 -> 5th bin of b
        assert len(r) == 1 and int(e[0]) == 0 | (1 << 31) | ((1 + 4) << 32)
    with pytest.raises(Exception):
        ExtentGrouping.from_lengths([1000, 0], 1000)


def _golden_binmap():
    with np.load(os.path.join(ROOT, 'tests', 'golden', 'binmap.npz')) as z:
        g = {k: z[k] for k in z.files}            # an NpzFile re-reads an array on every access
    ptr = g['cig_ptr']
    alns = []
    for k in range(len(g['name'])):
        cig = [(int(o), int(n)) for o, n in zip(g['cig_op'][ptr[k]:ptr[k + 1]], g['cig_len'][ptr[k]:ptr[k + 1]])]
        alns.append(dict(name='t%d' % g['name'][k], flag=int(g['flag'][k]), tid=int(g['tid'][k]), pos=int(g['pos'][k]),
                         mapq=int(g['mapq'][k]), cigar=cig))
    return g, alns


def _maps_from_records(rec, ext, lut, n_seq, n_bins):
    ok = ((rec >> np.uint64(31)) & np.uint64(1)).astype(bool)
    m31 = np.uint64(0x7fffffff)
    dok, counts = oracle.bin_pairs_loop((rec & m31).astype(np.int64), ((rec >> np.uint64(32)) & m31).astype(np.int64), ok,
                                        {t: int(i) for t, i in enumerate(lut) if i >= 0}, n_seq)
    dx, cx = oracle.bin_pairs_loop((ext & m31).astype(np.int64), ((ext >> np.uint64(32)) & m31).astype(np.int64), ok,
                                   {b: b for b in range(n_bins)}, n_bins)
    assert cx == counts
    return oracle.dok_to_coo(dok, n_seq), oracle.dok_to_coo(dx, n_bins), counts


@pytest.mark.parametrize('via', ['oracle', 'native'])
def test_pair_loop_against_the_reference_bin_map(tmp_path, via):
    """
    tests/golden/binmap.npz holds what the REFERENCE'S OWN ContactMap._bin_map (exec'd verbatim on duck-typed records,
    tests/golden/make_golden_binmap.py) produced: contig map, extent map and counters for three filter settings.
    'oracle': the oracle's restatement of the loop reproduces them; 'native': so do the records the C++ BAM reader
    extracts from a real BAM file of the same alignments, accumulated by the oracle.
    """
    from bin3c_b200.contact_map import ExtentGrouping
    g, alns = _golden_binmap()
    lengths = g['lengths']
    n_refs = len(lengths)
    keep = lengths >= int(g['min_len'])
    lut = np.where(keep, np.cumsum(keep) - 1, -1).astype(np.int32)
    n_seq = int(keep.sum())
    grouping = ExtentGrouping.from_lengths(lengths[keep], int(g['bin_size']))
    og = oracle.extent_grouping(lengths[keep], int(g['bin_size']))
    if via == 'native':
        path = str(tmp_path / 'g.bam')
        bam_writer.write_bam(path, ['r%d' % i for i in range(n_refs)], lengths.tolist(), alns, block_bytes=20000, level=1)
    for k in range(int(g['n_params'])):
        kw = dict(min_mapq=int(g['p%d_min_mapq' % k]), strong=int(g['p%d_strong' % k]) or None,
                  min_insert=int(g['p%d_min_insert' % k]) or None)
        if via == 'oracle':
            rec, ext, st = oracle.pair_alignments(alns, n_refs, idx_of=lut, grouping=og, **kw)
            short = st['short_insert']
        else:
            with bam_io.BamPairReader(path, threads=4) as bam:
                bam.set_extent(lut, grouping)
                bam.set_filter(tid2idx=lut, **kw)
                parts = []
                while True:
                    r, e = bam.read_pairs_extent(4099)
                    if len(r) == 0:
                        break
                    parts.append((r.copy(), e.copy()))
                short = bam.stats()['short_insert']
            rec, ext = np.concatenate([p[0] for p in parts]), np.concatenate([p[1] for p in parts])
        seq_map, ext_map, counts = _maps_from_records(rec, ext, lut, n_seq, grouping.total_bins)
        want = g['p%d_counts' % k].tolist()
        assert [counts['accepted'], counts['ref_excluded'], counts['poor_match'], short] == want
        for nm, m in (('seq_map', seq_map), ('extent_map', ext_map)):
            assert m.shape[0] == int(g['p%d_%s_n' % (k, nm)])
            assert np.array_equal(m.row, g['p%d_%s_row' % (k, nm)]) and np.array_equal(m.col, g['p%d_%s_col' % (k, nm)])
            assert np.array_equal(m.data, g['p%d_%s_data' % (k, nm)])


def test_bam_long_cigar_in_cg_tag_and_reverse_read_without_cigar(tmp_path):
    """CIGARs of more than 65535 operations live in the CG:B,I tag behind the placeholder <l_seq>S<span>N (SAM
    specification 4.2.2; htslib hands the tag's operations to the caller): the strong matcher and the reference span of
    a reverse read must come from the tag.  A mapped reverse read WITHOUT any CIGAR has `alen` None in the reference,
    whose `r.pos + r.alen` raises: the reader reports a format error instead of a silent span of zero."""
    import struct
    from bin3c_b200.contact_map import ExtentGrouping
    refs, lengths = ['a', 'b'], [50000, 40000]
    real = [(0, 30), (2, 5), (0, 20), (1, 2), (3, 1000), (0, 40)]                  # spans 30+5+20+1000+40 = 1095
    l_seq = sum(n for op, n in real if op in (0, 1, 4, 7, 8))
    tag = b'CGBI' + struct.pack('<I', len(real)) + b''.join(struct.pack('<I', (n << 4) | op) for op, n in real)
    other = b'NMC\x03' + b'XZZabc\0'                                             # tags in front of CG are skipped
    alns = [dict(name='p0', flag=0x41 | 0x10, tid=0, pos=1000, mapq=60, cigar=[(4, l_seq), (3, 1095)], seq_len=l_seq,
                 tags=other + tag),
            dict(name='p0', flag=0x81, tid=1, pos=700, mapq=60, cigar=[(0, 100)])]
    path = str(tmp_path / 'cg.bam')
    bam_writer.write_bam(path, refs, lengths, alns)
    lut = np.array([0, 1], dtype=np.int32)
    g = ExtentGrouping.from_lengths(lengths, 500)
    with bam_io.BamPairReader(path) as bam:
        bam.set_extent(lut, g)
        bam.set_filter(min_mapq=30, strong=35)                 # the tag's last operation is 40M: a strong match
        rec, ext = bam.read_pairs_extent(10)
    assert len(rec) == 1 and (int(rec[0]) >> 31) & 1 == 1
    og = oracle.extent_grouping(lengths, 500)
    b1 = oracle.find_nearest(og['map'][0], 1000 + 1095)        # the reverse read's 5' end: pos + span of the REAL CIGAR
    b2 = oracle.find_nearest(og['map'][1], 700)
    assert int(ext[0]) & 0x7fffffff == b1 and (int(ext[0]) >> 32) & 0x7fffffff == b2
    with bam_io.BamPairReader(path) as bam:                    # with the placeholder (1 op of 'S') it would not match
        bam.set_filter(min_mapq=30, strong=41)
        assert (int(bam.read_pairs(10)[0]) >> 31) & 1 == 0
    # mapped reverse read without a CIGAR: an error when 5' ends are needed, as in the reference
    bad = [dict(name='q', flag=0x41 | 0x10, tid=0, pos=10, mapq=60, cigar=[]),
           dict(name='q', flag=0x81, tid=1, pos=20, mapq=60, cigar=[(0, 50)])]
    path2 = str(tmp_path / 'nocigar.bam')
    bam_writer.write_bam(path2, refs, lengths, bad)
    with bam_io.BamPairReader(path2) as bam:
        bam.set_extent(lut, g)
        with pytest.raises(ValueError) as ei:
            bam.read_pairs_extent(10)
        assert 'without a CIGAR' in str(ei.value)
    with bam_io.BamPairReader(path2) as bam:                   # the contig map alone does not need the 5' end
        assert len(bam.read_pairs(10)) == 1
    with pytest.raises(TypeError):
        oracle.pair_alignments(bad, 2, idx_of=lut, grouping=og)


def test_split_records_round_trip():
    """b3c_records_split: same-reference pairs as 3- / 4-byte records, the others as pair records, input order kept
    within each part; counts-only call; argument errors; single- and multi-threaded packing agree."""
    rng = np.random.default_rng(8)
    for n_refs, n in ((1000, 0), (1000, 5), (300_000, 70_001), (9_000_000, 66_000)):
        a = rng.integers(0, n_refs, n).astype(np.uint64)
        b = np.where(rng.random(n) < 0.7, a, rng.integers(0, n_refs, n).astype(np.uint64))
        ok = (rng.random(n) < 0.8).astype(np.uint64)
        rec = a | (ok << np.uint64(31)) | (b << np.uint64(32))
        if n > 4:
            rec[3] = np.uint64(0x7fffffff) | (np.uint64(0x7fffffff) << np.uint64(32))
            rec[4] = np.uint64(0x7fffffff) | (np.uint64(2) << np.uint64(32)) | np.uint64(1 << 31)
        sp1 = bam_io.split_records(rec, n_refs, threads=1)
        sp4 = bam_io.split_records(rec, n_refs, threads=4)
        assert sp1.bytes_same == bam_io.lib.b3c_records_same_bytes(n_refs) == (3 if n_refs < (1 << 23) - 1 else 4)
        assert sp1.bytes_pair == bam_io.records_bytes(n_refs)
        assert np.array_equal(sp1.same.numpy(), sp4.same.numpy()) and np.array_equal(sp1.pairs.numpy(), sp4.pairs.numpy())
        same = (a == b) if n <= 4 else ((rec & np.uint64(0x7fffffff)) == ((rec >> np.uint64(32)) & np.uint64(0x7fffffff)))
        assert sp1.n_same == int(same.sum()) and sp1.n_pairs == n - int(same.sum())
        assert np.array_equal(bam_io.unsplit_records(sp1), np.concatenate([rec[same], rec[~same]]))
    cnt = np.zeros(2, dtype=np.int64)
    r = np.zeros(4, dtype=np.uint64)
    assert bam_io.lib.b3c_records_split(r.ctypes.data, 4, 5, 3, None, None, cnt.ctypes.data, 1) == 4 and cnt.tolist() == [4, 0]
    out = np.zeros(64, dtype=np.uint8)
    with pytest.raises(AssertionError):
        bam_io.check(bam_io.lib.b3c_records_split(r.ctypes.data, 4, 7, 3, out.ctypes.data, out.ctypes.data, cnt.ctypes.data, 1))
    with pytest.raises(AssertionError):
        bam_io.check(bam_io.lib.b3c_records_split(r.ctypes.data, 4, 5, 2, out.ctypes.data, out.ctypes.data, cnt.ctypes.data, 1))
    with pytest.raises(AssertionError):
        bam_io.check(bam_io.lib.b3c_records_split(r.ctypes.data, 4, 5, 3, out.ctypes.data, None, cnt.ctypes.data, 1))
