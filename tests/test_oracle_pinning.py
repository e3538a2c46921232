"""
Live pinning: where a checkout of the reference is present (oracle/_ref/ or
$BIN3C_REFERENCE, see oracle/ref_exec.py), run its own functions verbatim beside the
oracle restatement on fresh seeded inputs (the tests marked needs_reference; skipped
without one).  The committed golden vectors carry the same checks without a checkout:
tests/test_oracle.py, and the tests at the end of this module.
"""
import numpy as np
import pytest
import scipy.sparse as sp

from bin3c_b200 import synth
from oracle import oracle, ref_exec

needs_reference = pytest.mark.skipif(not ref_exec.available(), reason='reference tree not present')


@pytest.fixture(scope='module')
def fns():
    return ref_exec.load()


@needs_reference
@pytest.mark.parametrize('seed,n,p', [(101, 120, 4000), (102, 700, 25000), (103, 64, 300)])
def test_reference_functions_vs_oracle(fns, seed, n, p):
    com = synth.make_community(n_genomes=3, n_contigs=n, n_pairs=p, seed=seed)
    ti, tj, ok = synth.unpack_pairs(com.records)
    idx_of = {int(t): k for k, t in enumerate(com.ref_index)}
    dok, counts = oracle.bin_pairs_loop(ti, tj, ok, idx_of, n)

    acc = fns['Sparse2DAccumulator'](n)
    for (i, j), c in dok.items():
        acc[i, j] = c
    ref_map = acc.get_coo()
    mine = oracle.dok_to_coo(dok, n)
    assert ref_map.dtype == mine.dtype == np.uint32
    assert np.array_equal(ref_map.row, mine.row) and np.array_equal(ref_map.col, mine.col)
    assert np.array_equal(ref_map.data, mine.data)

    assert np.array_equal(np.asarray(fns['max_offdiag'](ref_map)), oracle.max_offdiag(mine))

    s = oracle.get_sites(com.sites)
    fm = sp.coo_matrix((oracle.norm_by_sites(mine.row, mine.col, mine.data.astype(float), s),
                        (mine.row, mine.col)), shape=mine.shape)
    rb, rx, rn, _ = ref_exec.kr_with_iterations(fns, fm)
    ob, ox, on = oracle.kr_biostochastic(fm)
    assert rn == on
    assert np.max(np.abs(rx - ox) / np.abs(rx)) <= 1e-12
    assert abs(rb - ob).max() <= 1e-12 * abs(rb).max()

    mask = oracle.acceptance_mask(com.lengths, mine, 1000, 2)
    if 0 < mask.sum() < n:
        rc = fns['compress'](rb.tocoo(), mask).tocsr()
        oc = oracle.compress(rb.tocoo(), mask).tocsr()
        assert rc.shape == oc.shape and abs(rc - oc).max() == 0


@needs_reference
def test_reference_extent_grouping_vs_oracle():
    """The reference's ExtentGrouping class and find_nearest_jit, exec'd live (Python 2 division shimmed)."""
    import random
    make_grouping, find_nearest = ref_exec.load_extent()
    rng = random.Random(77)
    lengths = [rng.randrange(1, 30000) for _ in range(300)]
    for bs in (13, 1000, 4096):
        r = make_grouping(lengths, bs)
        o = oracle.extent_grouping(lengths, bs)
        assert r.total_bins == o['total_bins'] and np.array_equal(np.asarray(r.bins), o['bins'])
        for a, b in zip(r.map, o['map']):
            assert np.array_equal(np.asarray(a), b)
        for k in range(0, 300, 11):
            for x in (0, lengths[k] // 2, lengths[k], lengths[k] + 5):
                assert int(find_nearest(np.asarray(r.map[k]), x)) == oracle.find_nearest(o['map'][k], x)


@needs_reference
def test_reference_bin_map_loop_vs_oracle():
    """The reference's _bin_map, exec'd live on a fresh random alignment stream, against the oracle's loop."""
    import os
    import random
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden'))
    import make_golden_binmap as mg
    rng = random.Random(5)
    n_refs = 50
    lengths = [rng.choice([500, 1000, 2100, 12000]) for _ in range(n_refs)]
    alns = [dict(a, name='q%d' % a['name']) for a in mg.make_alignments(rng, n_refs, lengths, 3000)]
    keep = np.array(lengths) >= 1000
    lut = np.where(keep, np.cumsum(keep) - 1, -1)
    idx = {t: int(i) for t, i in enumerate(lut) if i >= 0}
    kept = [l for l in lengths if l >= 1000]
    make_grouping, _ = ref_exec.load_extent()
    for kw in (dict(min_mapq=25), dict(min_mapq=25, strong=30), dict(min_mapq=10, min_insert=900)):
        ref = ref_exec.run_bin_map(alns, lengths, idx, len(kept), grouping=make_grouping(kept, 700), **kw)
        og = oracle.extent_grouping(kept, 700)
        rec, ext, st = oracle.pair_alignments(alns, n_refs, idx_of=lut, grouping=og, **kw)
        m31 = np.uint64(0x7fffffff)
        ok = ((rec >> np.uint64(31)) & np.uint64(1)).astype(bool)
        dok, c = oracle.bin_pairs_loop((rec & m31).astype(np.int64), ((rec >> np.uint64(32)) & m31).astype(np.int64), ok,
                                       idx, len(kept))
        dx, _ = oracle.bin_pairs_loop((ext & m31).astype(np.int64), ((ext >> np.uint64(32)) & m31).astype(np.int64), ok,
                                      {b: b for b in range(og['total_bins'])}, og['total_bins'])
        rc = ref['counts']
        assert [rc[k] for k in ('accepted', 'ref_excluded', 'poor_match')] == [c[k] for k in ('accepted', 'ref_excluded', 'poor_match')]
        assert rc['short_insert'] == st['short_insert']
        for got, want in ((oracle.dok_to_coo(dok, len(kept)), ref['seq_map']),
                          (oracle.dok_to_coo(dx, og['total_bins']), ref['extent_map'])):
            assert np.array_equal(got.row, want.row) and np.array_equal(got.col, want.col)
            assert np.array_equal(got.data, want.data)


@needs_reference
def test_reference_to_graph_vs_oracle_edges(tmp_path):
    """
    The reference's to_graph (cluster.py:278-325), exec'd on the compressed balanced map of a synthetic community:
    same edge set and the same scale 1/max (Q8) as the oracle's edge list; every weight within 2 ulp (the
    reference keeps the LAST of the two mirrored entries it adds, the oracle and the product the upper one, Q9).
    The edge file networkx writes from that graph equals the native writer's on the graph's own weights.
    """
    pytest.importorskip('networkx')
    import networkx as nx
    from bin3c_b200 import bam_io
    com = synth.make_community(n_genomes=4, n_contigs=300, n_pairs=60000, seed=55)
    ti, tj, ok = synth.unpack_pairs(com.records)
    ref = oracle.run_path(ti, tj, ok, com.tid2idx(), com.lengths, com.sites, min_len=1000, min_sig=2)
    sub = ref['sub_map'] if 'sub_map' in ref else None
    if sub is None:
        bal, _x, _n = oracle.kr_biostochastic(sp.coo_matrix(
            (oracle.norm_by_sites(ref['seq_map'].row, ref['seq_map'].col, ref['seq_map'].data.astype(float),
                                  oracle.get_sites(com.sites)), (ref['seq_map'].row, ref['seq_map'].col)),
            shape=ref['seq_map'].shape))
        sub = oracle.compress(bal.tocoo(), ref['mask'])
    g = ref_exec.run_to_graph(sub.tocoo(), int(ref['mask'].sum()), scale=True)
    u, v, w, scl = oracle.graph_edges(sub, scale=True)
    assert g.number_of_edges() == len(u)
    gw = np.array([g[int(a)][int(b)]['weight'] for a, b in zip(u, v)])
    assert np.max(np.abs(gw - w) / w) <= 4.5e-16                       # <= 2 ulp
    assert gw.max() == w.max()                                           # the scale and the largest entry agree exactly
    lower = sub.tocsr()
    k = len(u) // 2
    assert gw[k] == lower[int(v[k]), int(u[k])] * scl                    # last writer = the mirrored (lower) entry
    f_nx, f_b3 = str(tmp_path / 'nx.edges'), str(tmp_path / 'b3.edges')
    nx.write_edgelist(g, f_nx, data=['weight'], delimiter=' ')
    e = list(g.edges(data='weight'))
    bam_io.write_edges([a for a, _, _ in e], [b for _, b, _ in e], [c for _, _, c in e], f_b3)
    assert open(f_nx).read() == open(f_b3).read()


@needs_reference
def test_whole_reference_path_vs_oracle():
    """The reference's ContactMap and SeqOrder classes exec'd live and driven end to end (oracle/ref_exec.py:
    run_reference_path), against oracle.run_path on a fresh community, with an extent map on the side."""
    import os
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden'))
    import make_golden_refpath as mg
    com = synth.make_community(n_genomes=3, n_contigs=150, n_pairs=20000, seed=909)
    lengths = np.full(com.n_refs, 500, dtype=np.int64)
    sites = np.ones(com.n_refs, dtype=np.int64)
    lengths[com.ref_index] = com.lengths
    sites[com.ref_index] = com.sites
    res = ref_exec.run_reference_path(mg.alignments_of(com.records), lengths, sites, 1000, 2, min_mapq=60, bin_size=3000)
    ti, tj, ok = synth.unpack_pairs(com.records)
    ref = oracle.run_path(ti, tj, ok, com.tid2idx(), com.lengths, com.sites, min_len=1000, min_sig=2)
    assert {k: res['counts'][k] for k in ('accepted', 'ref_excluded', 'poor_match')} == ref['counts']
    a, b = res['seq_map'], ref['seq_map']
    assert np.array_equal(a.row, b.row) and np.array_equal(a.col, b.col) and np.array_equal(a.data, b.data)
    assert np.array_equal(np.asarray(res['mask']), ref['mask'])
    assert np.max(np.abs(res['bisto_scale'] - ref['x']) / np.abs(ref['x'])) <= 1e-12
    g = res['graph']
    assert g.number_of_edges() == len(ref['u'])
    gw = np.array([g[int(x)][int(y)]['weight'] for x, y in zip(ref['u'], ref['v'])])
    assert np.max(np.abs(gw - ref['w']) / ref['w']) <= 4.5e-16
    assert res['extent_map'].shape[0] == res['cm'].grouping.total_bins and res['extent_map'].sum() > 0


@needs_reference
def test_reference_seqorder_and_mask_rules_vs_product_host_logic():
    """
    The product's host-side SeqOrder (pure NumPy, no GPU) beside the reference's SeqOrder class on random masks, and
    the acceptance-mask rules (contact_map.py:856-909, Q5: falsy thresholds fall back to the instance's, the mask is
    cached unless `update`) of the reference's ContactMap beside oracle.acceptance_mask.
    """
    import os
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden'))
    import make_golden_refpath as mg
    from bin3c_b200.contact_map import SeqOrder
    com = synth.make_community(n_genomes=3, n_contigs=200, n_pairs=30000, seed=4711)
    lengths = np.full(com.n_refs, 500, dtype=np.int64)
    sites = np.ones(com.n_refs, dtype=np.int64)
    lengths[com.ref_index] = com.lengths
    sites[com.ref_index] = com.sites
    res = ref_exec.run_reference_path(mg.alignments_of(com.records), lengths, sites, 1000, 3, min_mapq=60)
    cm = res['cm']
    mine = SeqOrder(cm.seq_info)
    mine.set_mask_only(np.asarray(res['mask']))     # positions depend on the history of masks: replay the reference's one
    assert np.array_equal(np.asarray(cm.order.order['pos']), mine.order['pos'])
    rng = np.random.default_rng(3)
    for frac in (1.0, 0.7, 0.2, 0.0):
        m = rng.random(cm.total_seq) < frac
        cm.order.set_mask_only(m)
        mine.set_mask_only(m)
        assert np.array_equal(np.asarray(cm.order.order['pos']), mine.order['pos'])
        assert np.array_equal(np.asarray(cm.order.order['mask']), mine.order['mask'])
        assert np.array_equal(np.asarray(cm.order.mask_vector()), mine.mask_vector())
        assert cm.order.count_accepted() == mine.count_accepted() == int(m.sum())
        assert cm.order.count_excluded() == mine.count_excluded()
        assert np.array_equal(np.asarray(cm.order.accepted()), mine.accepted())
        assert np.array_equal(np.asarray(cm.order.excluded()), mine.excluded())
        assert np.array_equal(np.asarray(cm.order.lengths()), mine.lengths())
        assert np.array_equal(np.asarray(cm.order.lengths(exclude_masked=True)), mine.lengths(exclude_masked=True))
    sm = res['seq_map']
    seq_len = np.array([s.length for s in cm.seq_info], dtype=np.int64)
    first = cm.get_primary_acceptance_mask().copy()
    assert np.array_equal(first, oracle.acceptance_mask(seq_len, sm, 1000, 3))
    cm.set_primary_acceptance_mask(min_len=5000, min_sig=20)                 # no update: the cached mask stays
    assert np.array_equal(cm.get_primary_acceptance_mask(), first)
    for ml, ms in ((5000, 20), (2000, 1), (1000, 50)):
        cm.set_primary_acceptance_mask(min_len=ml, min_sig=ms, update=True)
        assert np.array_equal(cm.get_primary_acceptance_mask(), oracle.acceptance_mask(seq_len, sm, ml, ms))
    cm.set_primary_acceptance_mask(min_len=0, min_sig=0, update=True)       # falsy -> the instance's 1000 / 3
    assert np.array_equal(cm.get_primary_acceptance_mask(), first)


@needs_reference
def test_infomap_partition_reference_graph_vs_product_edge_list(tmp_path):
    """
    North-star: "the resulting Infomap clustering is identical".  The reference's graph (its own to_graph on its own
    ContactMap) written as its pinned Python 2.7 / networkx 1.11 would write it (12 significant digits), and the
    oracle's edge list (what the CUDA path is held to within 1e-9) written by the native writer in the same layout:
    the two files are byte-identical here (1-2 ulp differences vanish in 12 digits), and the reference's Infomap
    binary returns the same partition for both, and for the full-precision (repr) layout too.
    """
    import os
    import subprocess
    import sys
    infomap = os.path.join(ref_exec.REFERENCE_ROOT, 'external', 'Infomap')
    if not os.access(infomap, os.X_OK):
        pytest.skip('no Infomap binary in the reference tree')
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden'))
    import make_golden_refpath as mg
    from bin3c_b200 import bam_io
    com = synth.make_community(n_genomes=5, n_contigs=400, n_pairs=80000, seed=31337)
    lengths = np.full(com.n_refs, 500, dtype=np.int64)
    sites = np.ones(com.n_refs, dtype=np.int64)
    lengths[com.ref_index] = com.lengths
    sites[com.ref_index] = com.sites
    res = ref_exec.run_reference_path(mg.alignments_of(com.records), lengths, sites, 1000, 3, min_mapq=60)
    ti, tj, ok = synth.unpack_pairs(com.records)
    ref = oracle.run_path(ti, tj, ok, com.tid2idx(), com.lengths, com.sites, min_len=1000, min_sig=3)
    g = res['graph']
    e = sorted((min(a, b), max(a, b), w) for a, b, w in g.edges(data='weight'))
    parts = {}
    files = {}
    for name, (u, v, w), style in (
            ('reference_py2', ([a for a, _, _ in e], [b for _, b, _ in e], [c for _, _, c in e]), bam_io.FLOAT_STR12),
            ('product_py2', (ref['u'], ref['v'], ref['w']), bam_io.FLOAT_STR12),
            ('product_repr', (ref['u'], ref['v'], ref['w']), bam_io.FLOAT_REPR)):
        work = tmp_path / name
        work.mkdir()
        f = str(work / 'cm_graph.edges')
        if name == 'reference_py2':                      # written independently of the native writer
            with open(f, 'w') as out:
                out.write(oracle.edge_lines(u, v, w, py2=True))
        else:
            bam_io.write_edges(u, v, w, f, float_style=style)
        files[name] = open(f).read()
        subprocess.check_call([infomap, '-u', '-v', '-z', '-i', 'link-list', '-s', '1234', '-N', '10', f, str(work)],
                              stdout=subprocess.DEVNULL, stderr=subprocess.STDOUT)
        parts[name] = oracle.read_tree(str(work / 'cm_graph.tree'))
    assert files['reference_py2'] == files['product_py2']
    assert parts['reference_py2'] == parts['product_py2'] == parts['product_repr']
    assert len(parts['product_py2']) >= 3


def _read_edge_file_gz(path):
    import gzip
    u, v, w = [], [], []
    with gzip.open(path, 'rt') as fh:
        for line in fh:
            a, b, c = line.split(' ')
            u.append(int(a))
            v.append(int(b))
            w.append(float(c))
    return np.array(u), np.array(v), np.array(w)


@needs_reference
def test_infomap_partition_of_gpu_edge_file(tmp_path):
    """
    North-star bar 3 on CUDA OUTPUT: tests/golden/c1_gpu.edges.gz and c1_gpu_py2.edges.gz are the edge files the CUDA
    path wrote on a B200 for BASELINE config 1 at full size (tests/test_gpu_configs.py::
    test_c1_full_size_against_the_reference_own_output checks that it still writes them; committed gzip'd).
    They hold the reference's own edges (c1full.npz: the reference's classes exec'd on the same 1M pairs) to 1e-9,
    and the reference's Infomap binary, run here with the flags of cluster.py:182-185, returns for both the partition it
    returns for the reference's own graph file (stored in c1full.npz by make_golden_c1.py).
    """
    import gzip
    import os
    import shutil
    import subprocess
    import sys
    from conftest import load_golden, GOLDEN_DIR
    g = load_golden('c1full')
    u, v, w = _read_edge_file_gz(os.path.join(GOLDEN_DIR, 'c1_gpu.edges.gz'))
    assert np.array_equal(u, g['edge_u']) and np.array_equal(v, g['edge_v'])
    assert np.max(np.abs(w - g['edge_w']) / np.abs(g['edge_w'])) <= 1e-9
    # in the reference's own 12-digit layout the GPU file is the reference's file, byte for byte
    with gzip.open(os.path.join(GOLDEN_DIR, 'c1_gpu_py2.edges.gz'), 'rt') as fh:
        gpu_py2 = fh.read()
    ref_py2 = oracle.edge_lines(g['edge_u'], g['edge_v'], g['edge_w'], py2=True)
    differing = sum(1 for a, b in zip(gpu_py2.splitlines(), ref_py2.splitlines()) if a != b)
    assert len(gpu_py2.splitlines()) == len(ref_py2.splitlines()) and differing <= 3, differing
    infomap = os.path.join(ref_exec.REFERENCE_ROOT, 'external', 'Infomap')
    if not os.access(infomap, os.X_OK):
        pytest.skip('no Infomap binary in the reference tree')
    sys.path.insert(0, GOLDEN_DIR)
    import make_golden_c1 as mc
    want = (g['part_node'], g['part_label'])
    assert want[1].max() + 1 == 10                       # the ten genomes of C1
    for name in ('c1_gpu.edges.gz', 'c1_gpu_py2.edges.gz'):
        work = tmp_path / name.replace('.', '_')
        work.mkdir()
        f = str(work / 'cm_graph.edges')
        with gzip.open(os.path.join(GOLDEN_DIR, name), 'rb') as src, open(f, 'wb') as dst:
            shutil.copyfileobj(src, dst)
        node, label = mc.partition_arrays(mc.infomap_partition(f, str(work)))
        assert np.array_equal(node, want[0]) and np.array_equal(label, want[1]), name


@needs_reference
def test_reference_tip_based_path_vs_oracle():
    """The tip-based map (SURVEY.md 8f rank 4), live: the reference's _bin_map with tip_size, its Sparse4DAccumulator and
    4-D functions over SparseShim, and its ContactMap class driven to the graph, beside the oracle on a fresh stream."""
    import random
    import sys
    import os
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden'))
    from make_golden_binmap import make_alignments
    rng = random.Random(777)
    n_refs = 40
    lengths = [rng.choice([500, 1000, 1300, 2100, 5000, 12000]) for _ in range(n_refs)]
    alns = [dict(a, name='q%d' % a['name']) for a in make_alignments(rng, n_refs, lengths, 5000)]
    sites2 = [[rng.randrange(0, 12), rng.randrange(0, 12)] for _ in range(n_refs)]
    keep = np.array(lengths) >= 1000
    lut = np.where(keep, np.cumsum(keep) - 1, -1)
    idx = {t: int(i) for t, i in enumerate(lut) if i >= 0}
    n_seq = int(keep.sum())
    for tip, kw in ((250, dict(min_mapq=20)), (3000, dict(min_mapq=10, min_insert=800))):
        res = ref_exec.run_bin_map(alns, lengths, idx, n_seq, tip_size=tip, **kw)
        cells, c = oracle.tip_pairs_loop(alns, lengths, idx, n_seq, tip, **kw)
        assert {k: res['counts'][k] for k in c} == c
        coords, data = oracle.tip_tensor(cells, n_seq)
        assert np.array_equal(res['seq_map'].coords, coords) and np.array_equal(res['seq_map'].data, data)
        path = ref_exec.run_reference_path(alns, lengths, sites2, 1000, 2, min_mapq=kw['min_mapq'],
                                           min_insert=kw.get('min_insert'), tip_size=tip)
        mine = oracle.run_tip_path(cells, np.array(lengths)[keep], np.array(sites2)[keep], 1000, 2)
        assert np.array_equal(path['mask'], mine['mask'])
        assert np.max(np.abs(path['bisto_scale'] - mine['x']) / np.abs(mine['x'])) <= 1e-12
        e = sorted((min(u, v), max(u, v), d['weight']) for u, v, d in path['graph'].edges(data=True))
        assert [x[0] for x in e] == mine['u'].tolist() and [x[1] for x in e] == mine['v'].tolist()
        assert np.max(np.abs(np.array([x[2] for x in e]) - mine['w']) / np.abs(mine['w'])) <= 1e-12


# ---- the same comparisons against outputs of the reference stored under tests/golden (no reference checkout) ----

def _refpath_and_oracle():
    """tests/golden/refpath.npz (the reference's own path, make_golden_refpath.py) and oracle.run_path on its inputs."""
    from conftest import load_golden
    g = load_golden('refpath')
    keep = (g['lengths'] >= int(g['min_len'])) & (g['sites'] >= 0)
    lut = np.where(keep, np.cumsum(keep) - 1, -1).astype(np.int32)
    ti, tj, ok = synth.unpack_pairs(g['records'])
    ref = oracle.run_path(ti, tj, ok, lut, g['lengths'][keep], g['sites'][keep], min_len=int(g['min_len']),
                          min_sig=int(g['min_sig']))
    return g, ref


def test_stored_reference_graph_weights_are_its_mirrored_entries(tmp_path):
    """
    The graph the reference's to_graph built (refpath.npz): its scale is exactly the oracle's 1/max of the compressed
    balanced map (Q8), and every weight is the reference's own balanced map at the mirrored (lower) position times that
    scale -- the last of the two entries it adds wins (Q9).  The edge file networkx writes from that graph equals the
    native writer's on the graph's own weights.
    """
    nx = pytest.importorskip('networkx')
    from bin3c_b200 import bam_io
    g, ref = _refpath_and_oracle()
    n = len(g['mask'])
    acc = np.flatnonzero(g['mask'])
    sub = sp.coo_matrix((g['bal_data'], (g['bal_row'], g['bal_col'])), shape=(n, n)).tocsr()[acc][:, acc]
    assert ref['scl'] == 1.0 / sub.max()
    assert g['edge_w'].max() == ref['w'].max()
    u, v, w = g['edge_u'], g['edge_v'], g['edge_w']
    assert np.array_equal(w, np.asarray(sub[v, u]).ravel() * ref['scl'])
    graph = nx.Graph()
    for a, b, c in zip(u, v, w):
        graph.add_edge(int(a), int(b), weight=float(c))
    f_nx, f_b3 = str(tmp_path / 'nx.edges'), str(tmp_path / 'b3.edges')
    nx.write_edgelist(graph, f_nx, data=['weight'], delimiter=' ')
    e = list(graph.edges(data='weight'))
    bam_io.write_edges([a for a, _, _ in e], [b for _, b, _ in e], [c for _, _, c in e], f_b3)
    assert open(f_nx).read() == open(f_b3).read()


def test_stored_reference_edge_file_equals_the_native_writers(tmp_path):
    """The reference's graph (refpath.npz) in the 12-significant-digit layout its pinned Python 2.7 / networkx 1.11
    write, and the oracle's edge list written by the native writer in that layout: byte-identical files, so Infomap
    reads the same graph from both."""
    from bin3c_b200 import bam_io
    g, ref = _refpath_and_oracle()
    f = str(tmp_path / 'cm_graph.edges')
    bam_io.write_edges(ref['u'], ref['v'], ref['w'], f, float_style=bam_io.FLOAT_STR12)
    assert open(f).read() == oracle.edge_lines(g['edge_u'], g['edge_v'], g['edge_w'], py2=True)


def test_gpu_edge_files_hold_the_reference_edges():
    """tests/golden/c1_gpu.edges.gz and c1_gpu_py2.edges.gz, the edge files the CUDA path wrote on a B200 for BASELINE
    config 1, hold the reference's own edges (c1full.npz) to 1e-9; in the reference's 12-digit layout the GPU file is
    the reference's file but for at most 3 lines."""
    import gzip
    import os
    from conftest import load_golden, GOLDEN_DIR
    g = load_golden('c1full')
    u, v, w = _read_edge_file_gz(os.path.join(GOLDEN_DIR, 'c1_gpu.edges.gz'))
    assert np.array_equal(u, g['edge_u']) and np.array_equal(v, g['edge_v'])
    assert np.max(np.abs(w - g['edge_w']) / np.abs(g['edge_w'])) <= 1e-9
    with gzip.open(os.path.join(GOLDEN_DIR, 'c1_gpu_py2.edges.gz'), 'rt') as fh:
        gpu_py2 = fh.read()
    ref_py2 = oracle.edge_lines(g['edge_u'], g['edge_v'], g['edge_w'], py2=True)
    differing = sum(1 for a, b in zip(gpu_py2.splitlines(), ref_py2.splitlines()) if a != b)
    assert len(gpu_py2.splitlines()) == len(ref_py2.splitlines()) and differing <= 3, differing
