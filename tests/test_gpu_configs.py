"""
GPU parity tests (-m gpu) at the sizes of the BASELINE configs, all through the C ABI:

  C1 (2,000 contigs, 1M pairs)     whole path against golden vectors produced by the REFERENCE'S OWN code on the full
                                   config (tests/golden/c1full.npz, make_golden_c1.py); the edge files the CUDA path
                                   writes hold the committed ones (tests/golden/c1_gpu*.edges.gz) that the reference's
                                   Infomap binary is run on (tests/test_oracle_pinning.py::
                                   test_infomap_partition_of_gpu_edge_file)
  C2 (50k contigs, 50M pairs)      whole path against oracle.run_path on the same records: counts, counters, mask,
                                   edge structure bit-exact, n_iter equal, x and w <= 1e-9
  C3 (250k contigs; a 100M-pair    the same against the oracle (36-bit keys, 9 column slabs, ~40 SpMV); the pair
      prefix of its 500M pairs)    stream is the counter-based one, generated on the device and mirrored on the host
  the device pair stream           bit-identical to its NumPy mirror (what the oracle is fed from)
  KR error paths on the device     exact tie (Q13) -> ValueError, n_iter > max_iter -> RuntimeError, NaN -> RuntimeError
"""
import gzip
import os

import numpy as np
import pytest
import scipy.sparse as sp

from conftest import load_golden, GOLDEN_DIR

pytestmark = pytest.mark.gpu

REL_TOL = 1e-9          # north_star tolerance for KR scale vector and edge weights


@pytest.fixture(scope='module')
def dev():
    import torch
    if not torch.cuda.is_available():
        pytest.skip('no CUDA device')
    from bin3c_b200 import device
    return device


def _relerr(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    if a.size == 0:
        return 0.0
    return float(np.max(np.abs(a - b) / np.maximum(np.abs(b), 1e-300)))


def _run_and_compare(dev, com_tables, records_dev, records_host, min_len=1000, min_sig=5, threads=16):
    """HotPath (fused and staged forms) on device records against oracle.run_path on the same records."""
    from bin3c_b200 import synth
    from bin3c_b200.pipeline import HotPath
    from oracle import oracle
    tid2idx, lengths, sites = com_tables
    hp = HotPath(tid2idx, lengths, sites, min_len=min_len, min_sig=min_sig, pair_capacity=int(records_dev.numel()))
    res = hp.run(records_dev)
    n = int(res['n_edges'])
    u, v, w = [res[k][:n].cpu().numpy().copy() for k in ('u', 'v', 'w')]
    ti, tj, ok = synth.unpack_pairs(records_host)
    ref = oracle.run_path(ti, tj, ok, tid2idx, lengths, sites, min_len=min_len, min_sig=min_sig, threads=threads)
    del ti, tj, ok
    # contact matrix, counters, map weight: bit-exact
    got = hp.seq_map.to_scipy_coo()
    want = ref['seq_map']
    assert got.dtype == np.uint32 and got.nnz == want.nnz
    assert np.array_equal(got.row, want.row) and np.array_equal(got.col, want.col)
    assert np.array_equal(got.data, want.data)
    assert {k: hp.acc_info[k] for k in ref['counts']} == ref['counts']
    assert hp.acc_info['map_weight'] == int(want.data.sum(dtype=np.int64))
    # acceptance mask: bit-exact
    assert np.array_equal(hp.mask.cpu().numpy().astype(bool), ref['mask'])
    # KR: identical iteration count, x within 1e-9
    assert hp.kr_info['n_iter'] == ref['n_iter']
    x_err = _relerr(hp.x.cpu().numpy(), ref['x'])
    assert x_err <= REL_TOL
    # edge list: structure exact, weights within 1e-9
    assert n == len(ref['u'])
    assert np.array_equal(u, ref['u']) and np.array_equal(v, ref['v'])
    w_err = _relerr(w, ref['w'])
    assert w_err <= REL_TOL
    assert _relerr(float(res['scl'].cpu()[0]), ref['scl']) <= REL_TOL
    return hp, ref, dict(x_err=x_err, w_err=w_err, u=u, v=v, w=w)


def _read_edge_file(path):
    with (gzip.open(path, 'rt') if path.endswith('.gz') else open(path)) as fh:
        rows = [line.split(' ') for line in fh]
    return (np.array([int(r[0]) for r in rows]), np.array([int(r[1]) for r in rows]),
            np.array([float(r[2]) for r in rows]))


def test_c1_full_size_against_the_reference_own_output(dev, tmp_path):
    """BASELINE config 1 at full size: every output of the CUDA path against what the reference's own classes
    produced for the same 1M pairs (c1full.npz).  The edge file it writes holds the committed tests/golden/c1_gpu.edges.gz
    (same edges, weights within 1e-9); in the reference's 12-digit layout it is the reference's own file but for at
    most 3 lines, the bound the committed c1_gpu_py2.edges.gz meets."""
    import torch
    from oracle import oracle
    from bin3c_b200 import synth, cluster
    from bin3c_b200.contact_map import ContactMap, PairRecords
    g = load_golden('c1full')
    com = synth.make_config('C1')
    cm = ContactMap(PairRecords.from_community(com), ['synthetic'], None, None, min_mapq=60,
                    min_len=int(g['min_len']), min_sig=int(g['min_sig']), random_seed=1)
    u, v, w, scl = cluster.to_edges(cm, norm=True, bisto=True, scale=True)
    torch.cuda.synchronize()
    sm = cm.seq_map
    assert np.array_equal(sm.row, g['map_row']) and np.array_equal(sm.col, g['map_col'])
    assert np.array_equal(sm.data, g['map_data'])
    pc = cm.pair_counts
    assert [pc['accepted'], pc['ref_excluded'], pc['poor_match']] == g['counts'].tolist()
    assert np.array_equal(cm.get_primary_acceptance_mask().astype(np.uint8), g['mask'])
    assert cm.kr_info['n_iter'] == int(g['kr_n_iter'])
    assert _relerr(cm.bisto_scale, g['kr_x']) <= REL_TOL
    assert np.array_equal(u, g['edge_u']) and np.array_equal(v, g['edge_v'])
    assert _relerr(w, g['edge_w']) <= REL_TOL
    fu, fv, fw = _read_edge_file(cluster.write_edges(u, v, w, str(tmp_path), base_name='c1_gpu'))
    gu, gv, gw = _read_edge_file(os.path.join(GOLDEN_DIR, 'c1_gpu.edges.gz'))
    assert np.array_equal(fu, gu) and np.array_equal(fv, gv) and _relerr(fw, gw) <= REL_TOL
    # the 12-digit file Infomap reads: the reference's own file but for at most 3 lines, as the committed one is
    with open(cluster.write_edges(u, v, w, str(tmp_path), base_name='c1_gpu_py2', py2_str=True)) as fh:
        got = fh.read().splitlines()
    want = oracle.edge_lines(g['edge_u'], g['edge_v'], g['edge_w'], py2=True).splitlines()
    differing = sum(1 for a, b in zip(got, want) if a != b)
    assert len(got) == len(want) and differing <= 3, differing


def test_c2_full_size_against_the_oracle(dev):
    """BASELINE config 2 at full size (50k contigs, 50M pairs): exact against oracle.run_path (seconds on 16
    threads), plus idempotence and fused == staged."""
    from bin3c_b200 import synth
    com = synth.make_config('C2')
    rec = dev.to_device(com.records)
    hp, ref, out = _run_and_compare(dev, (com.tid2idx(), com.lengths, com.sites), rec, com.records)
    x = hp.x.cpu().numpy().copy()
    # bistochastic on the working matrix (zero diagonals -> 1, Q2)
    m = hp.seq_map.to_scipy_csr()
    assert (m != m.T).nnz == 0
    for fused in (False, True):
        r2 = hp.run(rec, fused=fused)
        n = int(r2['n_edges'])
        assert n == len(out['u'])
        for k in ('u', 'v'):
            assert np.array_equal(r2[k][:n].cpu().numpy(), out[k])
        if fused:           # the same form again: the same bits
            assert np.array_equal(r2['w'][:n].cpu().numpy(), out['w']) and np.array_equal(hp.x.cpu().numpy(), x)
        else:               # the staged form iterates on fp64 values, the fused one on counts: equal to rounding
            assert _relerr(r2['w'][:n].cpu().numpy(), out['w']) <= 1e-12 and _relerr(hp.x.cpu().numpy(), x) <= 1e-12
            assert hp.kr_info['n_iter'] == ref['n_iter']
        if not fused:
            wk = hp.normed.to_scipy_csr()
            work = wk + sp.diags((wk.diagonal() == 0).astype(float))
            assert np.max(np.abs(x * work.dot(x) - 1)) < 1e-4


def test_c3_prefix_against_the_oracle(dev):
    """BASELINE config 3's community (250k contigs -> 36-bit keys, 9 column slabs) on the first 100M pairs of its
    counter-based stream: generated on the device, mirrored on the host for the oracle."""
    from bin3c_b200 import synth
    tab, stream, _ = synth.make_stream('C3')
    P = 100_000_000
    rec = stream.device_records(0, P)
    host = rec.cpu().numpy().view(np.uint64)          # the device stream; a slice of it re-derived by the host mirror
    assert np.array_equal(host[77_000_000:78_000_000], stream.host_records(77_000_000, 1_000_000))
    com = tab.community(host)
    hp, ref, out = _run_and_compare(dev, (com.tid2idx(), com.lengths, com.sites), rec, host)
    assert hp.kr_info['slabs'] == 9 and tab.N == 250_000


@pytest.mark.parametrize('name,first,count', [('C3', 0, 1_000_003), ('C3', 499_000_000, 1_000_000),
                                              ('C4', (1 << 31) + 12345, 2_000_001), ('C4', 0, 7)])
def test_device_pair_stream_equals_host_mirror(dev, name, first, count):
    """b3c_synth_pairs (csrc/synth.cu) == StreamV2.host_records bit for bit, at offsets beyond 2^31 too."""
    import torch
    from bin3c_b200 import synth
    tab, stream, P = synth.make_stream(name)
    got = stream.device_records(first, count)
    torch.cuda.synchronize()
    want = stream.host_records(first, count)
    assert np.array_equal(got.cpu().numpy().view(np.uint64), want)
    ti, tj, ok = synth.unpack_pairs(want)
    assert ti.max() < tab.n_refs and tj.max() < tab.n_refs
    if count > 100_000:
        lut = tab.community(want).tid2idx()
        i, j = lut[ti], lut[tj]
        keep = (i >= 0) & (j >= 0)
        assert 0.70 < np.mean(i[keep] == j[keep]) < 0.90          # ~80 % intra-contig pairs
        assert 0.015 < np.mean(~keep) < 0.025                     # ~2 % of pairs touch an excluded reference
        assert 0.84 < ok.mean() < 0.86


# ---- KR error paths driven on the device ---------------------------------------------------------------

@pytest.mark.parametrize('n', [1, 37, 4096, 5000])
def test_kr_exact_tie_raises_value_error(dev, n):
    """Q13 (sparse_utils.py:179-181): max(ynew) == Delta with no element above Delta -> the reference's np.amin of an
    empty selection raises ValueError.  A = 0.125 I makes every quantity exact: v = 1/8, rk = 7/8, Z = p = 7,
    w = 7/4, alpha = 1/2, ynew = 4.5 in every row, so Delta = 4.5 is an exact tie on the first CG step."""
    from oracle import oracle
    m = sp.identity(n, format='csr', dtype=np.float64) * 0.125
    with pytest.raises(ValueError):
        oracle.kr_scale_vector(m, Delta=4.5)
    with pytest.raises(ValueError):
        dev.kr_scale_vector(dev.DeviceCSR.from_scipy(m), Delta=4.5)
    # one ulp either side of the tie is not an error, and agrees with the oracle
    for Delta in (np.nextafter(4.5, 0.0), np.nextafter(4.5, 9.0)):
        res = oracle.kr_scale_vector(m, Delta=Delta)
        x, info = dev.kr_scale_vector(dev.DeviceCSR.from_scipy(m), Delta=Delta)
        assert info['n_iter'] == res.n_iter
        assert _relerr(x.cpu().numpy(), res.x) <= REL_TOL


@pytest.mark.parametrize('max_iter', [1, 2, 3, 5, 8, 13])
def test_kr_max_iter_behaviour_matches_the_reference(dev, max_iter):
    """sparse_utils.py:146,213-221: the outer loop stops once n_iter >= max_iter; n_iter > max_iter raises
    RuntimeError, n_iter == max_iter only warns.  Same outcome and same n_iter / x as the oracle for every cap."""
    import torch
    from oracle import oracle
    from conftest import golden_lut
    g = load_golden('c1mini')
    from bin3c_b200 import synth
    ti, tj, ok = synth.unpack_pairs(g['records'])
    up, _ = oracle.bin_pairs_fast(ti, tj, ok, golden_lut(g), len(g['lengths']))
    sm = oracle.symmetrise(up)
    s = oracle.get_sites(g['sites'])
    m = sp.coo_matrix((oracle.norm_by_sites(sm.row, sm.col, sm.data.astype(np.float64), s), (sm.row, sm.col)),
                      shape=sm.shape).tocsr()
    try:
        res, want_err = oracle.kr_scale_vector(m, max_iter=max_iter), None
    except RuntimeError as e:
        res, want_err = None, str(e)
    a = dev.DeviceCSR.from_scipy(m)
    if want_err is not None:
        with pytest.raises(RuntimeError) as ei:
            dev.kr_scale_vector(a, max_iter=max_iter)
        assert 'failed to converge' in str(ei.value) and str(ei.value) == want_err
    else:
        x, info = dev.kr_scale_vector(a, max_iter=max_iter)
        assert info['n_iter'] == res.n_iter
        assert _relerr(x.cpu().numpy(), res.x) <= REL_TOL
    torch.cuda.synchronize()


def test_kr_nan_input_raises_runtime_error(dev):
    """A NaN in the matrix: the reference's guard (sparse_utils.py:192-193) has the message below; its loop test
    `rout > rt` is False for a NaN residual, so the reference itself would fall through and hand back a NaN-bearing
    x without reaching the guard.  The CUDA path reports it (deliberately stricter; DESIGN.md section 2)."""
    rng = np.random.default_rng(3)
    n = 3000
    up = sp.triu(sp.random(n, n, density=0.01, random_state=rng, data_rvs=lambda k: rng.uniform(0.1, 5.0, k)), k=1)
    m = (up + up.T + sp.diags(rng.uniform(0.5, 2.0, n))).tocsr()
    m.data[m.nnz // 2] = np.nan
    with pytest.raises(RuntimeError) as ei:
        dev.kr_scale_vector(dev.DeviceCSR.from_scipy(m))
    assert 'invalid values' in str(ei.value)
