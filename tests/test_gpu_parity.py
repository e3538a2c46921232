"""
GPU parity tests (-m gpu): the CUDA path, called through the C ABI, against the golden vectors
produced by the reference's own functions and against the CPU oracle on seeded inputs.

Bars (BASELINE.json north_star): contact matrix, counters and acceptance mask bit-exact;
KR scale vector and edge weights within 1e-9 max relative error, identical iteration count.
"""
import numpy as np
import pytest
import scipy.sparse as sp

from conftest import golden_lut

pytestmark = pytest.mark.gpu

REL_TOL = 1e-9          # north_star tolerance for KR scale vector and edge weights


@pytest.fixture(scope='module')
def dev():
    import torch
    if not torch.cuda.is_available():
        pytest.skip('no CUDA device')
    from bin3c_b200 import device
    return device


def _accumulate(dev, records, lut, n, symmetric=True, chunks=1, capacity=None):
    import torch
    rec = dev.to_device(np.ascontiguousarray(records, dtype=np.uint64))
    acc = dev.Accumulator(n, lut, capacity if capacity is not None else max(len(records), 1))
    if len(records):
        step = -(-len(records) // chunks)
        step += step & 1                      # keep chunk starts 16-byte aligned
        for lo in range(0, len(records), step):
            acc.add(rec[lo:lo + step])
    csr, info = acc.finish(symmetric=symmetric)
    torch.cuda.synchronize()
    return csr, info


def _relerr(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    if a.size == 0:
        return 0.0
    return float(np.max(np.abs(a - b) / np.maximum(np.abs(b), 1e-300)))


# ---------------------------------------------------------------------------------------------
# accumulation
# ---------------------------------------------------------------------------------------------

def test_accumulate_golden(dev, golden):
    g = golden
    n = len(g['lengths'])
    csr, info = _accumulate(dev, g['records'], golden_lut(g), n)
    coo = csr.to_scipy_coo()
    assert coo.dtype == np.uint32
    assert np.array_equal(coo.row, g['map_row'])
    assert np.array_equal(coo.col, g['map_col'])
    assert np.array_equal(coo.data, g['map_data'])
    assert [info['accepted'], info['ref_excluded'], info['poor_match']] == g['counts'].tolist()
    assert info['map_weight'] == int(g['map_weight'])


def test_accumulate_chunked_and_upper(dev, golden):
    from oracle import oracle
    from bin3c_b200 import synth
    g = golden
    n = len(g['lengths'])
    ti, tj, ok = synth.unpack_pairs(g['records'])
    up, counts = oracle.bin_pairs_fast(ti, tj, ok, golden_lut(g), n)
    up = up.tocsr()
    up.sort_indices()
    csr, info = _accumulate(dev, g['records'], golden_lut(g), n, symmetric=False, chunks=3)
    got = csr.to_scipy_csr()
    assert np.array_equal(got.indptr, up.indptr)
    assert np.array_equal(got.indices, up.indices)
    assert np.array_equal(got.data, up.data)
    assert info['nnz_upper'] == up.nnz


def _oracle_full(records, lut, n):
    from oracle import oracle
    from bin3c_b200 import synth
    ti, tj, ok = synth.unpack_pairs(records)
    up, counts = oracle.bin_pairs_fast(ti, tj, ok, lut, n)
    return oracle.symmetrise(up), counts


@pytest.mark.parametrize('case', ['empty', 'all_excluded', 'all_poor', 'all_diag', 'single', 'one_cell'])
def test_accumulate_edge_cases(dev, case):
    from bin3c_b200 import synth
    n, n_refs = 37, 45
    lut = np.full(n_refs, -1, dtype=np.int32)
    keep = np.sort(np.random.default_rng(5).choice(n_refs, n, replace=False))
    lut[keep] = np.arange(n, dtype=np.int32)
    excl = np.setdiff1d(np.arange(n_refs), keep)
    rng = np.random.default_rng(7)
    if case == 'empty':
        rec = np.zeros(0, dtype=np.uint64)
    elif case == 'all_excluded':
        rec = synth.pack_pairs(rng.choice(excl, 999), rng.choice(keep, 999), np.ones(999, bool))
    elif case == 'all_poor':
        rec = synth.pack_pairs(rng.choice(keep, 1001), rng.choice(keep, 1001), np.zeros(1001, bool))
    elif case == 'all_diag':
        a = rng.choice(keep, 5000)
        rec = synth.pack_pairs(a, a, np.ones(5000, bool))
    elif case == 'single':
        rec = synth.pack_pairs([keep[3]], [keep[1]], [True])
    else:
        rec = synth.pack_pairs(np.full(70000, keep[2]), np.full(70000, keep[30]), np.ones(70000, bool))
    csr, info = _accumulate(dev, rec, lut, n)
    want, counts = _oracle_full(rec, lut, n)
    got = csr.to_scipy_coo()
    assert np.array_equal(got.row, want.row) and np.array_equal(got.col, want.col)
    assert np.array_equal(got.data, want.data)
    assert {k: info[k] for k in counts} == counts


@pytest.mark.parametrize('n,n_refs,p,rank_lut', [
    (1000, 1200, 200_000, True),          # shared-memory diagonal + rank table
    (1000, 1200, 200_000, False),         # arbitrary tid->index map: gather fallback
    (70_000, 80_000, 400_000, True),      # 17-bit indices: global diagonal, 64-bit staging
    (70_000, 80_000, 400_000, False),
    (300_000, 2_400_000, 300_000, True),  # rank table too large for shared memory
    (1_000_000, 1_100_000, 400_000, True),    # two-level rank table (C4's size: bitmap + 16-bit relative prefixes)
    (900_000, 1_048_576, 300_000, True),      # ... with the sentinel word opening a block of its own
    (257, 257, 50_001, True),             # odd sizes, no excluded refs
])
def test_accumulate_random(dev, n, n_refs, p, rank_lut):
    from bin3c_b200 import synth
    rng = np.random.default_rng(n + p + int(rank_lut))
    keep = np.sort(rng.choice(n_refs, n, replace=False))
    lut = np.full(n_refs, -1, dtype=np.int32)
    lut[keep] = np.arange(n, dtype=np.int32) if rank_lut else rng.permutation(n).astype(np.int32)
    # heavy duplicates + a tid beyond the table (must count as excluded)
    a = rng.integers(0, n_refs, p)
    b = np.where(rng.random(p) < 0.6, a, rng.integers(0, min(n_refs, 3000), p))
    a[:5] = n_refs + 11
    rec = synth.pack_pairs(a, b, rng.random(p) < 0.9)
    csr, info = _accumulate(dev, rec, lut, n, chunks=2)
    want, counts = _oracle_full(rec, lut, n)
    got = csr.to_scipy_coo()
    assert got.nnz == want.nnz
    assert np.array_equal(got.row, want.row) and np.array_equal(got.col, want.col)
    assert np.array_equal(got.data, want.data)
    assert {k: info[k] for k in counts} == counts
    assert info['map_weight'] == int(want.sum(dtype=np.uint64))


@pytest.mark.parametrize('B', [5, 6, 8])
@pytest.mark.parametrize('n_pairs', [0, 1, 7, 4099, 300_001])
def test_accumulate_narrow_records(dev, B, n_pairs):
    """Narrow (5- and 6-byte) records give exactly the matrix and counters of the native 8-byte records: device-
    resident in one call and in ragged chunks, and streamed from the host through HotPath's staging ring."""
    import torch
    from bin3c_b200 import bam_io, synth
    from bin3c_b200.pipeline import HotPath
    com = synth.make_community(n_genomes=6, n_contigs=900, n_pairs=max(n_pairs, 1), seed=31 + B)
    rec = com.records[:n_pairs].copy()
    if n_pairs > 20:
        rec[5] = np.uint64(0x7fffffff) | (rec[5] & np.uint64(0xffffffff80000000))     # out-of-table id in mate 1
        rec[11] = (rec[11] & np.uint64(0xffffffff)) | (np.uint64(0x7fffffff) << np.uint64(32))
    lut = com.tid2idx()
    want, winfo = _accumulate(dev, rec, lut, com.n_contigs)
    packed = bam_io.pack_records(rec, B)
    assert np.array_equal(bam_io.unpack_records(packed, n_pairs, B), rec)
    dpk = torch.from_numpy(packed).cuda()
    for chunk in (max(n_pairs, 8), 1000):                 # one call; ragged chunks of a multiple of 8 records
        acc = dev.Accumulator(com.n_contigs, lut, max(n_pairs, 1))
        for lo in range(0, n_pairs, chunk):
            hi = min(lo + chunk, n_pairs)
            nb = ((hi - lo) * B + 7) // 8 * 8
            piece = dpk[lo * B:lo * B + nb]
            if piece.data_ptr() % 16:                     # a chunk that does not start on 16 bytes is re-staged
                piece = piece.clone()
            acc.add_packed(piece, hi - lo, B)
        got, ginfo = acc.finish()
        torch.cuda.synchronize()
        assert ginfo == winfo
        assert np.array_equal(got.indptr.cpu().numpy(), want.indptr.cpu().numpy())
        assert np.array_equal(got.indices.cpu().numpy(), want.indices.cpu().numpy())
        assert np.array_equal(got.data.cpu().numpy(), want.data.cpu().numpy())
    if n_pairs >= 4099 and B != 8:
        hp = HotPath(lut, com.lengths, com.sites, pair_capacity=n_pairs, min_sig=1)
        r8 = hp.run(dev.to_device(rec))
        n = int(r8['n_edges'])
        ref = [r8[k][:n].cpu().numpy().copy() for k in ('u', 'v', 'w')]
        out = hp.run(torch.from_numpy(packed).pin_memory(), to_host=True, record_bytes=B, n_records=n_pairs)
        assert hp.h2d_bytes == len(packed) and out['n_edges'] == n
        for k, w in zip(('u', 'v', 'w'), ref):
            assert np.array_equal(out[k], w)
        hp.reset()
        hp.accumulate(packed, chunk_records=1000, record_bytes=B, n_records=n_pairs)      # pageable, many chunks
        assert hp.acc_info == winfo


@pytest.mark.parametrize('n_pairs', [0, 9, 4099, 300_001])
def test_accumulate_split_records(dev, n_pairs):
    """The narrowest hand-over (bam_io.split_records): pairs on one reference as 3-byte records, the others as pair
    records -- the same matrix, counters and edges as the native 8-byte records, device-resident and streamed from the
    host in ragged chunks; out-of-table ids included (an all-ones same-reference record counts as excluded)."""
    import torch
    from bin3c_b200 import bam_io, synth
    from bin3c_b200.pipeline import HotPath
    com = synth.make_community(n_genomes=6, n_contigs=900, n_pairs=max(n_pairs, 1), seed=47)
    rec = com.records[:n_pairs].copy()
    if n_pairs > 20:
        rec[5] = np.uint64(0x7fffffff) | (rec[5] & np.uint64(0xffffffff80000000))          # out-of-table id in mate 1
        rec[6] = np.uint64(0x7fffffff) | (np.uint64(0x7fffffff) << np.uint64(32)) | np.uint64(1 << 31)   # in both
    lut = com.tid2idx()
    want, winfo = _accumulate(dev, rec, lut, com.n_contigs)
    sp_host = bam_io.split_records(rec, com.n_refs)
    assert sp_host.bytes_same == 3 and sp_host.bytes_pair == 5 and sp_host.n_records == n_pairs
    m31 = np.uint64(0x7fffffff)
    same = (rec & m31) == ((rec >> np.uint64(32)) & m31)
    assert sp_host.n_same == int(same.sum())
    assert np.array_equal(bam_io.unsplit_records(sp_host), np.concatenate([rec[same], rec[~same]]))
    acc = dev.Accumulator(com.n_contigs, lut, max(n_pairs, 1))
    for part, n, B, sm in sp_host.cuda().parts():
        if n:
            acc.add_packed(part, n, B, same=sm)
    got, ginfo = acc.finish()
    torch.cuda.synchronize()
    assert ginfo == winfo
    assert np.array_equal(got.indptr.cpu().numpy(), want.indptr.cpu().numpy())
    assert np.array_equal(got.indices.cpu().numpy(), want.indices.cpu().numpy())
    assert np.array_equal(got.data.cpu().numpy(), want.data.cpu().numpy())
    if n_pairs >= 4099:
        hp = HotPath(lut, com.lengths, com.sites, pair_capacity=n_pairs, min_sig=1)
        r8 = hp.run(dev.to_device(rec))
        n = int(r8['n_edges'])
        ref = [r8[k][:n].cpu().numpy().copy() for k in ('u', 'v', 'w')]
        out = hp.run(bam_io.split_records(rec, com.n_refs, pin=True), to_host=True)
        assert hp.h2d_bytes == sp_host.nbytes and out['n_edges'] == n
        for k, w in zip(('u', 'v', 'w'), ref):
            assert np.array_equal(out[k], w)
        out = hp.run(sp_host.cuda())                                              # device-resident split records
        assert int(out['n_edges']) == n
        hp.reset()
        hp.accumulate(sp_host, chunk_records=1000)                                # pageable, many chunks
        assert hp.acc_info == winfo


def test_accumulate_same_records_need_a_small_table(dev):
    import torch
    acc = dev.Accumulator(64, np.arange(64, dtype=np.int32), 16)
    z = torch.zeros(64, dtype=torch.uint8, device='cuda')
    acc.add_packed(z, 8, 3, same=True)
    acc.add_packed(z, 8, 4, same=True)
    with pytest.raises(AssertionError):
        acc.add_packed(z, 8, 5, same=True)
    lut = np.arange(9_000_000, dtype=np.int32)            # more references than the 23 bits of a 3-byte record hold
    acc = dev.Accumulator(9_000_000, lut, 16)
    with pytest.raises(AssertionError):
        acc.add_packed(z, 8, 3, same=True)
    acc.add_packed(z, 8, 4, same=True)


def test_accumulate_narrow_records_need_a_small_table(dev):
    import torch
    lut = np.arange(600_000, dtype=np.int32)              # more references than 19 bits hold
    acc = dev.Accumulator(600_000, lut, 16)
    with pytest.raises(AssertionError):
        acc.add_packed(torch.zeros(64, dtype=torch.uint8, device='cuda'), 8, 5)
    acc.add_packed(torch.zeros(64, dtype=torch.uint8, device='cuda'), 8, 6)
    with pytest.raises(AssertionError):
        acc.add_packed(torch.zeros(64, dtype=torch.uint8, device='cuda'), 8, 7)


def test_accumulate_capacity_error(dev):
    from bin3c_b200 import synth
    from bin3c_b200._cabi import B3CError
    lut = np.arange(64, dtype=np.int32)
    rng = np.random.default_rng(3)
    rec = synth.pack_pairs(rng.integers(0, 64, 10000), rng.integers(0, 64, 10000), np.ones(10000, bool))
    with pytest.raises(B3CError):
        _accumulate(dev, rec, lut, 64, capacity=100)


# ---------------------------------------------------------------------------------------------
# mask, normalisation
# ---------------------------------------------------------------------------------------------

def _golden_map_dev(dev, g):
    n = len(g['lengths'])
    m = sp.coo_matrix((g['map_data'], (g['map_row'], g['map_col'])), shape=(n, n), dtype=np.uint32)
    return dev.DeviceCSR.from_scipy(m, np.uint32), m


def test_mask_golden(dev, golden):
    import torch
    g = golden
    csr, _ = _golden_map_dev(dev, g)
    sig = dev.max_offdiag(csr)
    assert np.array_equal(sig.cpu().numpy().view(np.uint32), g['signal'])
    mask = dev.acceptance_mask(dev.to_device(g['lengths'], torch.int32), sig, int(g['min_len']), int(g['min_sig']))
    assert np.array_equal(mask.cpu().numpy().astype(bool), g['mask'])


def test_site_norm_exact(dev, golden):
    import torch
    from oracle import oracle
    g = golden
    csr, m = _golden_map_dev(dev, g)
    sites = g['sites'].copy()
    sites[::7] = 0                                  # exercise the zero -> one rule (Q6)
    out = dev.site_norm(csr, dev.to_device(sites, torch.int32))
    want = oracle.norm_by_sites(m.row, m.col, m.data.astype(np.float64), oracle.get_sites(sites))
    assert np.array_equal(out.data.cpu().numpy(), want)       # same operations, same rounding


# ---------------------------------------------------------------------------------------------
# Knight-Ruiz
# ---------------------------------------------------------------------------------------------

def _normed_dev(dev, g):
    import torch
    csr, _ = _golden_map_dev(dev, g)
    return dev.site_norm(csr, dev.to_device(g['sites'], torch.int32))


def test_kr_golden(dev, golden):
    g = golden
    a = _normed_dev(dev, g)
    x, info = dev.kr_scale_vector(a)
    assert info['n_iter'] == int(g['kr_n_iter'])
    assert info['zero_diag'] == int(g['kr_zero_diag'])
    assert _relerr(x.cpu().numpy(), g['kr_x']) <= REL_TOL
    bal = dev.kr_apply(a, x).to_scipy_csr()
    assert np.array_equal(bal.indptr, g['bal_indptr']) and np.array_equal(bal.indices, g['bal_indices'])
    assert _relerr(bal.data, g['bal_data']) <= REL_TOL


def test_kr_deterministic(dev):
    from conftest import load_golden
    g = load_golden('c1mini')
    a = _normed_dev(dev, g)
    x1, _ = dev.kr_scale_vector(a)
    x2, _ = dev.kr_scale_vector(a)
    assert np.array_equal(x1.cpu().numpy(), x2.cpu().numpy())


@pytest.mark.parametrize('n,density,seed', [(3000, 0.01, 1), (20000, 0.002, 2), (1500, 0.2, 3), (5, 0.9, 4)])
def test_kr_random_vs_oracle(dev, n, density, seed):
    from oracle import oracle
    rng = np.random.default_rng(seed)
    up = sp.random(n, n, density=density, random_state=rng, data_rvs=lambda k: rng.uniform(0.1, 5.0, k))
    up = sp.triu(up, k=1)
    d = rng.uniform(0.5, 2.0, n)
    d[rng.random(n) < 0.1] = 0.0                      # zero diagonals (Q2)
    m = (up + up.T + sp.diags(d)).tocsr()
    m.eliminate_zeros()
    res = oracle.kr_scale_vector(m)
    x, info = dev.kr_scale_vector(dev.DeviceCSR.from_scipy(m))
    assert info['n_iter'] == res.n_iter
    assert info['zero_diag'] == res.n_zero_diag
    assert _relerr(x.cpu().numpy(), res.x) <= REL_TOL


def test_kr_long_rows_and_empty_rows(dev):
    """Rows far longer than an SpMV tile, rows straddling tiles, and completely empty rows (Q3)."""
    from oracle import oracle
    rng = np.random.default_rng(9)
    n = 20000
    rows = [np.full(7000, 0), np.full(5000, 1), rng.integers(2, n // 2, 60000)]
    cols = [rng.choice(n // 2, 7000, replace=False), rng.choice(n // 2, 5000, replace=False),
            rng.integers(2, n // 2, 60000)]
    r = np.concatenate(rows)
    c = np.concatenate(cols)
    up = sp.coo_matrix((rng.uniform(0.2, 3.0, len(r)), (np.minimum(r, c), np.maximum(r, c))), shape=(n, n)).tocsr()
    up = sp.triu(up, k=1)
    m = (up + up.T + sp.diags(np.r_[rng.uniform(1, 2, n // 2), np.zeros(n - n // 2)])).tocsr()
    m.eliminate_zeros()
    assert (np.diff(m.indptr) == 0).sum() > 1000 and np.diff(m.indptr).max() > 4096
    res = oracle.kr_scale_vector(m)
    x, info = dev.kr_scale_vector(dev.DeviceCSR.from_scipy(m))
    assert info['n_iter'] == res.n_iter
    assert _relerr(x.cpu().numpy(), res.x) <= REL_TOL


@pytest.mark.parametrize('n,nnz_row', [(1, 1), (100, 1), (5000, 3), (4097, 40), (3000, 900)])
def test_spmv_vs_scipy(dev, n, nnz_row):
    rng = np.random.default_rng(n)
    m = sp.random(n, n, density=min(1.0, nnz_row / n), random_state=rng, format='csr')
    m.sort_indices()
    u = rng.standard_normal(n)
    y = dev.spmv(dev.DeviceCSR.from_scipy(m), dev.to_device(u)).cpu().numpy()
    want = m.dot(u)
    assert np.max(np.abs(y - want)) <= 1e-12 * max(1.0, np.max(np.abs(want)))


class _kr_options(object):
    """Temporarily change the slab shape of KR's SpMV operand (b3c_set_option)."""

    def __init__(self, dev, width=None, max_slabs=None):
        self.dev, self.width, self.max_slabs = dev, width, max_slabs

    def __enter__(self):
        if self.width is not None:
            self.dev.check(self.dev.lib.b3c_set_option(1, self.width))
        if self.max_slabs is not None:
            self.dev.check(self.dev.lib.b3c_set_option(2, self.max_slabs))

    def __exit__(self, *a):
        self.dev.check(self.dev.lib.b3c_set_option(1, 28672))
        self.dev.check(self.dev.lib.b3c_set_option(2, 16))


def _sym_matrix(n, nnz_row, seed, zero_diag_frac=0.1):
    rng = np.random.default_rng(seed)
    k = int(n * nnz_row / 2)
    r, c = rng.integers(0, n, k), rng.integers(0, n, k)
    up = sp.coo_matrix((rng.uniform(0.1, 5.0, k), (np.minimum(r, c), np.maximum(r, c))), shape=(n, n)).tocsr()
    up = sp.triu(up, k=1)
    d = rng.uniform(0.5, 2.0, n)
    d[rng.random(n) < zero_diag_frac] = 0.0
    m = (up + up.T + sp.diags(d)).tocsr()
    m.eliminate_zeros()
    m.sort_indices()
    return m


# slab shapes: (width cap, slab cap).  None = defaults; (1000, 16) forces several narrow slabs on small matrices;
# (126, 48) many narrow slabs (up to the table cap); (None, 0) forces the form that gathers through L1/L2
SLAB_SHAPES = [(None, None), (1000, 16), (334, 16), (126, 48), (None, 0)]


@pytest.mark.parametrize('shape', SLAB_SHAPES)
@pytest.mark.parametrize('n,nnz_row', [(1, 1), (100, 1), (5000, 3), (4097, 40), (3000, 900)])
def test_spmv_slab_shapes(dev, n, nnz_row, shape):
    rng = np.random.default_rng(n)
    m = sp.random(n, n, density=min(1.0, nnz_row / n), random_state=rng, format='csr')
    m.sort_indices()
    u = rng.standard_normal(n)
    with _kr_options(dev, *shape):
        y = dev.spmv(dev.DeviceCSR.from_scipy(m), dev.to_device(u)).cpu().numpy()
    want = m.dot(u)
    assert np.max(np.abs(y - want)) <= 1e-12 * max(1.0, np.max(np.abs(want)))


@pytest.mark.parametrize('n,nnz_row', [(60000, 20), (130000, 6), (450000, 4)])
def test_spmv_wide(dev, n, nnz_row):
    """Default slab shape on matrices that need 3 and 5 slabs, and one too wide for slabs (gather form)."""
    m = _sym_matrix(n, nnz_row, seed=n)
    u = np.random.default_rng(1).standard_normal(n)
    csr = dev.DeviceCSR.from_scipy(m)
    y = dev.spmv(csr, dev.to_device(u)).cpu().numpy()
    want = m.dot(u)
    assert np.max(np.abs(y - want)) <= 1e-12 * max(1.0, np.max(np.abs(want)))


@pytest.mark.parametrize('shape', SLAB_SHAPES[1:])
def test_kr_slab_shapes(dev, shape):
    """The scale vector must not depend on how the SpMV operand is cut (beyond summation order)."""
    from oracle import oracle
    m = _sym_matrix(5000, 30, seed=17)
    res = oracle.kr_scale_vector(m)
    with _kr_options(dev, *shape):
        x, info = dev.kr_scale_vector(dev.DeviceCSR.from_scipy(m))
    assert info['slabs'] == (0 if shape[1] == 0 else -(-5000 // shape[0]))
    assert info['n_iter'] == res.n_iter
    assert info['zero_diag'] == res.n_zero_diag
    assert _relerr(x.cpu().numpy(), res.x) <= REL_TOL


@pytest.mark.parametrize('nnz_row,slabs', [(300, 40), (30, 0)])
def test_kr_wide_matrix_form_follows_cell_density(dev, nnz_row, slabs):
    """Beyond 16 slabs the slab form is kept only while the (row, slab) cells hold >= 6 entries on average."""
    from oracle import oracle
    m = _sym_matrix(5000, nnz_row, seed=29)
    res = oracle.kr_scale_vector(m)
    with _kr_options(dev, 126, None):                      # 40 slabs needed, slab cap left at its default
        x, info = dev.kr_scale_vector(dev.DeviceCSR.from_scipy(m))
    assert info['slabs'] == slabs
    assert info['n_iter'] == res.n_iter
    assert _relerr(x.cpu().numpy(), res.x) <= REL_TOL


def test_kr_three_slabs_vs_oracle(dev):
    from oracle import oracle
    m = _sym_matrix(60000, 12, seed=23)
    res = oracle.kr_scale_vector(m)
    x, info = dev.kr_scale_vector(dev.DeviceCSR.from_scipy(m))
    assert info['slabs'] == 3
    assert info['n_iter'] == res.n_iter
    assert _relerr(x.cpu().numpy(), res.x) <= REL_TOL


def test_kr_rejects_unsorted_columns(dev):
    m = _sym_matrix(3000, 10, seed=5)
    csr = dev.DeviceCSR.from_scipy(m)
    lo, hi = int(m.indptr[7]), int(m.indptr[8])
    assert hi - lo >= 2
    csr.indices[lo], csr.indices[hi - 1] = csr.indices[hi - 1].clone(), csr.indices[lo].clone()
    with _kr_options(dev, 1000, 16):
        with pytest.raises(AssertionError):
            dev.kr_scale_vector(csr)


# ---------------------------------------------------------------------------------------------
# compress + edges, whole path
# ---------------------------------------------------------------------------------------------

def test_compress_edges_golden(dev, golden):
    import torch
    from oracle import oracle
    g = golden
    n = len(g['lengths'])
    bal = sp.csr_matrix((g['bal_data'], g['bal_indices'], g['bal_indptr']), shape=(n, n))
    res = dev.compress_edges(dev.DeviceCSR.from_scipy(bal), dev.to_device(g['mask'].astype(np.uint8), torch.uint8))
    assert res['n_accepted'] == int(g['sub_n']) and res['n_kept'] == int(g['sub_nnz'])
    want = oracle.compress(bal.tocoo(), g['mask']).tocsr()
    want.sort_indices()
    got = res['sub'].to_scipy_csr()
    assert np.array_equal(got.indptr, want.indptr) and np.array_equal(got.indices, want.indices)
    assert np.array_equal(got.data, want.data)
    assert float(res['scl'].cpu()[0]) == float(g['scl'])
    assert np.array_equal(res['u'].cpu().numpy(), g['edge_u'])
    assert np.array_equal(res['v'].cpu().numpy(), g['edge_v'])
    assert _relerr(res['w'].cpu().numpy(), g['edge_w']) <= REL_TOL


def _contact_map(g):
    from bin3c_b200.contact_map import ContactMap, PairRecords
    lengths = np.full(int(g['n_refs']), 500, dtype=np.int64)
    sites = np.ones(int(g['n_refs']), dtype=np.int64)
    lengths[g['ref_index']] = g['lengths']
    sites[g['ref_index']] = g['sites']
    pr = PairRecords(lengths, sites, g['records'])
    return ContactMap(pr, ['synthetic'], None, None, min_mapq=60, min_len=int(g['min_len']),
                      min_sig=int(g['min_sig']), random_seed=1)


def test_contact_map_end_to_end(dev, golden):
    import pickle
    from bin3c_b200 import cluster
    g = golden
    # the golden cases use min_len thresholds at or above the 1000 bp floor of their contigs
    if int(g['min_len']) > 1000:
        pytest.skip('constructor-level length filter changes N for this case')
    cm = _contact_map(g)
    assert cm.total_seq == len(g['lengths'])
    assert [cm.pair_counts[k] for k in ('accepted', 'ref_excluded', 'poor_match')] == g['counts'].tolist()
    assert cm.map_weight() == int(g['map_weight'])
    assert np.array_equal(cm.get_primary_acceptance_mask(), g['mask'])
    sm = cm.seq_map
    assert sp.isspmatrix_coo(sm) and sm.dtype == np.uint32
    assert np.array_equal(sm.row, g['map_row']) and np.array_equal(sm.col, g['map_col'])
    assert np.array_equal(sm.data, g['map_data'])

    u, v, w, scl = cluster.to_edges(cm, norm=True, bisto=True, scale=True)
    assert cm.kr_info['n_iter'] == int(g['kr_n_iter'])
    assert _relerr(cm.bisto_scale, g['kr_x']) <= REL_TOL
    assert np.array_equal(u, g['edge_u']) and np.array_equal(v, g['edge_v'])
    assert _relerr(w, g['edge_w']) <= REL_TOL
    assert abs(scl - float(g['scl'])) <= REL_TOL * float(g['scl'])

    sub = cm.get_subspace(marginalise=True, flatten=False)
    assert sp.isspmatrix_coo(sub) and sub.shape == (int(g['sub_n']),) * 2 and sub.nnz == int(g['sub_nnz'])

    gph = cluster.to_graph(cm, norm=True, bisto=True, scale=True)
    assert gph.number_of_edges() == len(g['edge_u'])

    # the whole object pickles with host containers only (bin3C.py:165)
    cm2 = pickle.loads(pickle.dumps(cm))
    assert cm2._dev == {} and np.array_equal(cm2.seq_map.data, g['map_data'])
    assert _relerr(cm2.processed_map.tocsr().data, g['bal_data']) <= REL_TOL

    # the stock-layout stream (io_utils.save_object(stock=True), SURVEY 8f-5) read back: the map a `cluster` stage
    # would start from gives the same edges
    from bin3c_b200 import io_utils
    cm3 = io_utils.loads(io_utils.dumps_stock(cm))
    assert cm3._dev == {} and np.array_equal(cm3.seq_map.data, g['map_data'])
    u3, v3, w3, scl3 = cluster.to_edges(cm3, norm=True, bisto=True, scale=True)
    assert np.array_equal(u3, u) and np.array_equal(v3, v) and np.array_equal(w3, w) and scl3 == scl


def test_bam_file_to_edge_file(dev, tmp_path):
    """
    The path with the steps either side of it: a name-sorted BAM written from the golden community's records (plus
    unmapped / secondary / supplementary / unpaired records the pairing loop must skip) -> native BAM reader ->
    ContactMap -> edge list -> native edge writer; matrix, counters, mask and edges against the golden vector.
    """
    import bam_writer
    from conftest import load_golden
    from bin3c_b200 import bam_io, cluster
    from bin3c_b200.contact_map import ContactMap
    g = load_golden('c1mini')
    rec = g['records']
    ti = (rec & np.uint64(0x7fffffff)).astype(np.int64)
    tj = ((rec >> np.uint64(32)) & np.uint64(0x7fffffff)).astype(np.int64)
    ok = ((rec >> np.uint64(31)) & np.uint64(1)).astype(bool)
    n_refs = int(g['n_refs'])
    lengths = np.full(n_refs, 500, dtype=np.int64)
    sites = np.ones(n_refs, dtype=np.int64)
    lengths[g['ref_index']] = g['lengths']
    sites[g['ref_index']] = g['sites']
    rng = np.random.default_rng(5)
    alns = []
    for k, (a, b, p) in enumerate(zip(ti.tolist(), tj.tolist(), ok.tolist())):
        name = 'pair%07d' % k
        q1, q2 = (60, 60) if p else ((60, 3) if k & 1 else (7, 60))            # a failed pair has one poor mate
        alns.append(dict(name=name, flag=0x41, tid=a, pos=10, mapq=q1, cigar=[(0, 100)]))
        if k % 97 == 0:                                                         # a supplementary record between the mates
            alns.append(dict(name=name, flag=0x841, tid=int(rng.integers(n_refs)), pos=5, mapq=60, cigar=[(0, 30)]))
        alns.append(dict(name=name, flag=0x81, tid=b, pos=50, mapq=q2, cigar=[(0, 100)]))
        if k % 131 == 0:                                                        # an unpaired informative read
            alns.append(dict(name='single%d' % k, flag=0x41, tid=a, pos=1, mapq=60, cigar=[(0, 50)]))
        if k % 173 == 0:                                                        # an unmapped pair
            alns.append(dict(name='unm%d' % k, flag=0x4d, tid=-1, pos=-1, mapq=0, cigar=[]))
            alns.append(dict(name='unm%d' % k, flag=0x8d, tid=-1, pos=-1, mapq=0, cigar=[]))
    path = str(tmp_path / 'hic.bam')
    bam_writer.write_bam(path, ['ref%05d' % i for i in range(n_refs)], lengths.tolist(), alns, block_bytes=30000, level=1)
    pr, stats = bam_io.pair_records_from_bam(path, sites=sites, min_mapq=60)
    assert stats['pairs'] == len(rec) and np.array_equal(pr.records, rec)
    cm = ContactMap(pr, ['synthetic'], None, None, min_mapq=60, min_len=int(g['min_len']), min_sig=int(g['min_sig']),
                    random_seed=1)
    assert [cm.pair_counts[k] for k in ('accepted', 'ref_excluded', 'poor_match')] == g['counts'].tolist()
    sm = cm.seq_map
    assert np.array_equal(sm.row, g['map_row']) and np.array_equal(sm.col, g['map_col'])
    assert np.array_equal(sm.data, g['map_data'])
    assert np.array_equal(cm.get_primary_acceptance_mask(), g['mask'])
    u, v, w, scl = cluster.to_edges(cm, norm=True, bisto=True, scale=True)
    assert np.array_equal(u, g['edge_u']) and np.array_equal(v, g['edge_v'])
    assert _relerr(w, g['edge_w']) <= REL_TOL
    f = cluster.write_edges(u, v, w, str(tmp_path))
    lines = open(f).read().splitlines()
    assert len(lines) == len(u)
    a, b, c = lines[0].split(' ')
    assert (int(a), int(b)) == (int(u[0]), int(v[0])) and float(c) == float(w[0])       # repr round-trips


def test_none_accepted(dev):
    from conftest import load_golden
    from bin3c_b200.exceptions import NoneAcceptedException
    g = load_golden('dups')
    g['min_sig'] = np.int64(10 ** 9)
    cm = _contact_map(g)
    assert cm.get_primary_acceptance_mask().sum() == 0
    with pytest.raises(NoneAcceptedException):
        cm.prepare_seq_map(norm=True, bisto=True)


def test_sparse_utils_dropin(dev, golden):
    from bin3c_b200 import sparse_utils as su
    from oracle import oracle
    g = golden
    n = len(g['lengths'])
    m = sp.coo_matrix((g['map_data'], (g['map_row'], g['map_col'])), shape=(n, n), dtype=np.uint32)
    assert np.array_equal(su.max_offdiag(m), g['signal'])
    s = oracle.get_sites(g['sites'])
    fm = sp.coo_matrix((oracle.norm_by_sites(m.row, m.col, m.data.astype(float), s), (m.row, m.col)), shape=m.shape)
    assert su.is_hermitian(fm)
    bal, x = su.kr_biostochastic(fm)
    assert su.kr_biostochastic.last_info['n_iter'] == int(g['kr_n_iter'])
    assert _relerr(x, g['kr_x']) <= REL_TOL
    sub = su.compress(bal, g['mask'])
    assert sp.isspmatrix_coo(sub) and sub.shape[0] == int(g['sub_n']) and sub.nnz == int(g['sub_nnz'])
    # the per-pair protocol and the bulk entry agree
    acc = su.Sparse2DAccumulator(n, tid2idx=golden_lut(g))
    acc.add_pairs(records=g['records'])
    coo = acc.get_coo()
    assert np.array_equal(coo.row, g['map_row']) and np.array_equal(coo.data, g['map_data'])
    acc2 = su.Sparse2DAccumulator(4)
    acc2[0, 1] += 3
    acc2[2, 2] += 1
    assert acc2[0, 1] == 3 and acc2[1, 0] == 0
    assert np.array_equal(acc2.get_coo().toarray(), np.array([[0, 3, 0, 0], [3, 0, 0, 0], [0, 0, 1, 0], [0, 0, 0, 0]]))
    asym = sp.csr_matrix(np.array([[1.0, 2.0], [2.5, 1.0]]))
    assert not su.is_hermitian(asym)


def test_medium_config_properties(dev):
    """A mid-size community (N=20k, P=4M): exact counts vs the vectorised oracle, KR bistochastic."""
    import torch
    from bin3c_b200 import synth
    from oracle import oracle
    com = synth.make_community(n_genomes=40, n_contigs=20_000, n_pairs=4_000_000, seed=77)
    lut = com.tid2idx()
    csr, info = _accumulate(dev, com.records, lut, com.n_contigs, chunks=4)
    want, counts = _oracle_full(com.records, lut, com.n_contigs)
    got = csr.to_scipy_coo()
    assert np.array_equal(got.row, want.row) and np.array_equal(got.col, want.col)
    assert np.array_equal(got.data, want.data)
    assert {k: info[k] for k in counts} == counts
    normed = dev.site_norm(csr, dev.to_device(com.sites, torch.int32))
    x, kinfo = dev.kr_scale_vector(normed)
    a = normed.to_scipy_csr()
    work = a + sp.diags((a.diagonal() == 0).astype(float))
    xx = x.cpu().numpy()
    assert np.max(np.abs(xx * work.dot(xx) - 1)) < 1e-5
    res = oracle.kr_scale_vector(a)
    assert kinfo['n_iter'] == res.n_iter
    assert _relerr(xx, res.x) <= REL_TOL


def test_full_size_c2_properties(dev):
    """
    BASELINE config C2 at full size (50k contigs, 50M pairs), through properties that do not need the oracle's
    minutes: the three counters and every row marginal against vectorised NumPy over the records (a checksum of
    checksums), canonical + symmetric CSR, the bistochastic property of x, a sorted edge list with weights in
    (0, 1] and max 1, and a second run that is bit-identical (idempotence).
    """
    import torch
    from bin3c_b200 import synth
    from bin3c_b200.pipeline import HotPath
    com = synth.make_config('C2')
    P, N = com.n_pairs, com.n_contigs
    hp = HotPath(com.tid2idx(), com.lengths, com.sites, pair_capacity=P)
    rec = dev.to_device(com.records)
    r1 = hp.run(rec, fused=False)
    n = int(r1['n_edges'])
    first = [r1[k][:n].cpu().numpy().copy() for k in ('u', 'v', 'w')]
    x = hp.x.cpu().numpy().copy()

    # counters and marginals from the records themselves
    ti, tj, ok = synth.unpack_pairs(com.records)
    lut = com.tid2idx().astype(np.int64)
    safe = lambda t: np.where(t < len(lut), lut[np.minimum(t, len(lut) - 1)], -1)
    ii, jj = safe(ti.astype(np.int64)), safe(tj.astype(np.int64))
    excl = (ii < 0) | (jj < 0)
    poor = ~excl & ~ok.astype(bool)
    acc = ~excl & ~poor
    assert hp.acc_info['ref_excluded'] == int(excl.sum())
    assert hp.acc_info['poor_match'] == int(poor.sum())
    assert hp.acc_info['accepted'] == int(acc.sum())
    a, b = ii[acc], jj[acc]
    marg = np.bincount(a, minlength=N) + np.bincount(b, minlength=N) - np.bincount(a[a == b], minlength=N)
    m = hp.seq_map.to_scipy_csr()
    assert m.dtype == np.uint32 and m.has_sorted_indices
    assert np.array_equal(np.asarray(m.sum(axis=1, dtype=np.int64)).ravel(), marg)
    assert int(m.sum(dtype=np.int64)) == 2 * int(acc.sum()) - int((a == b).sum())      # map_weight (Q7)
    assert (m != m.T).nnz == 0
    assert np.all(np.diff(m.indptr) >= 0) and m.nnz == hp.acc_info['nnz_full']

    # bistochastic on the working matrix (zero diagonals -> 1, Q2)
    w = hp.normed.to_scipy_csr()
    work = w + sp.diags((w.diagonal() == 0).astype(float))
    assert np.max(np.abs(x * work.dot(x) - 1)) < 1e-4
    assert hp.kr_info['n_iter'] < 100

    # the edge list: upper triangle of the accepted sub-matrix, sorted, scaled by 1/max (Q8)
    u, v, wts = first
    assert np.all(u <= v) and np.all(np.diff(u.astype(np.int64) * N + v) > 0)
    assert 1.0 - 4e-16 <= wts.max() <= 1.0 and wts.min() > 0.0          # max * (1.0 / max), as the reference scales
    mask = hp.mask.cpu().numpy().astype(bool)
    assert int(r1['n_accepted']) == int(mask.sum()) and u.max() < mask.sum() and v.max() < mask.sum()
    sub = sp.triu(m[mask][:, mask].tocsr(), k=0)
    assert n == sub.nnz

    # idempotence (the staged form again: the same bits); the fused form iterates on counts: equal to rounding
    for fused in (False, True):
        r2 = hp.run(rec, fused=fused)
        assert int(r2['n_edges']) == n
        for k, want in zip(('u', 'v'), first):
            assert np.array_equal(r2[k][:n].cpu().numpy(), want)
        if fused:
            assert _relerr(r2['w'][:n].cpu().numpy(), first[2]) <= 1e-12 and _relerr(hp.x.cpu().numpy(), x) <= 1e-12
        else:
            assert np.array_equal(r2['w'][:n].cpu().numpy(), first[2]) and np.array_equal(hp.x.cpu().numpy(), x)


def test_hotpath_host_records_match_device_records(dev):
    """HotPath.run with (pinned / pageable) HOST records streamed through the staging ring and the
    edge list read back into pinned host buffers == the same run with device-resident records."""
    import torch
    from bin3c_b200 import synth
    from bin3c_b200.pipeline import HotPath
    com = synth.make_community(n_genomes=12, n_contigs=3000, n_pairs=700_001, seed=99)
    hp = HotPath(com.tid2idx(), com.lengths, com.sites, pair_capacity=com.n_pairs)
    rec = torch.from_numpy(com.records.view(np.int64))
    r0 = hp.run(rec.to('cuda'), fused=False)             # the staged form, as driven stage by stage below
    n = int(r0['n_edges'])
    want = [r0[k][:n].cpu().numpy().copy() for k in ('u', 'v', 'w')] + [float(r0['scl'].cpu()[0])]
    for host, chunk in ((rec.pin_memory(), 100_000), (rec, 1 << 24), (rec.pin_memory(), 233_334)):
        hp.reset()
        hp.accumulate(host, chunk_records=chunk)          # 8, 1 and 4 chunks (ragged tail)
        assert hp.h2d_bytes == 8 * com.n_pairs
        hp.compute_mask(); hp.normalise(); hp.balance(); hp.edges()
        got = hp.edge_res
        assert int(got['n_edges']) == n
        for k, w in zip(('u', 'v', 'w'), want):
            assert np.array_equal(got[k][:n].cpu().numpy(), w)
    r1 = hp.run(rec.to('cuda'))                          # the fused form, device records ...
    want = [r1[k][:n].cpu().numpy().copy() for k in ('u', 'v', 'w')] + [float(r1['scl'].cpu()[0])]
    out = hp.run(rec.pin_memory(), to_host=True)         # ... and host records in, host edges out
    assert out['n_edges'] == n and hp.d2h_bytes == 16 * n + 8
    for k, w in zip(('u', 'v', 'w'), want):
        assert np.array_equal(out[k], w)
    assert out['scl'] == want[3]


def test_fused_counts_form_matches_the_staged_form(dev):
    """KR on raw counts and the fused edge emission against the staged results (site_norm -> KR -> kr_apply ->
    compress): same n_iter, same edge structure; x and w agree to rounding -- the counts form factors the site
    normalisation out of the row sums ((1/s_i) sum_j c_ij (u_j / s_j), 6 B per stream entry), so the last bits of
    the iteration differ -- and with B3C_OPT_KR_COUNT_STREAM = 0 (fp64 values c_ij / (s_i s_j) in the stream) the two
    forms are bit-identical.  Zero site counts included (Q6)."""
    import torch
    from bin3c_b200 import synth
    from bin3c_b200.pipeline import HotPath
    com = synth.make_community(n_genomes=10, n_contigs=4000, n_pairs=900_000, seed=123)
    sites = com.sites.copy()
    sites[::17] = 0
    hp = HotPath(com.tid2idx(), com.lengths, sites, pair_capacity=com.n_pairs, min_sig=3)
    rec = dev.to_device(com.records)
    r_staged = hp.run(rec, fused=False)
    n = int(r_staged['n_edges'])
    staged = [r_staged[k][:n].cpu().numpy().copy() for k in ('u', 'v', 'w')] + [r_staged['scl'].cpu().numpy().copy()]
    x_staged, it_staged = hp.x.cpu().numpy().copy(), hp.kr_info['n_iter']
    r_fused = hp.run(rec, fused=True)
    assert int(r_fused['n_edges']) == n and hp.kr_info['n_iter'] == it_staged
    assert _relerr(hp.x.cpu().numpy(), x_staged) <= 1e-12
    for k, w in zip(('u', 'v'), staged):
        assert np.array_equal(r_fused[k][:n].cpu().numpy(), w)
    assert _relerr(r_fused['w'][:n].cpu().numpy(), staged[2]) <= 1e-12
    assert _relerr(r_fused['scl'].cpu().numpy(), staged[3]) <= 1e-12
    x_fused = hp.x.cpu().numpy().copy()
    hp.run(rec, fused=True)
    assert np.array_equal(hp.x.cpu().numpy(), x_fused)                  # the same form twice: the same bits
    dev.check(dev.lib.b3c_set_option(5, 0))                             # B3C_OPT_KR_COUNT_STREAM off
    try:
        r_f64 = hp.run(rec, fused=True)
        assert np.array_equal(hp.x.cpu().numpy(), x_staged)
        for k, w in zip(('u', 'v', 'w'), staged):
            assert np.array_equal(r_f64[k][:n].cpu().numpy(), w)
        assert np.array_equal(r_f64['scl'].cpu().numpy(), staged[3])
    finally:
        dev.check(dev.lib.b3c_set_option(5, 2))


@pytest.mark.parametrize('offdiag_big', ['none', 'few', 'many'])
def test_packed_count_stream_large_counts(dev, offdiag_big):
    """The packed stream (16-bit count | 16-bit column, 4 B per entry; B3C_OPT_KR_COUNT_STREAM = 2, the default in the
    slab form): diagonal counts above 65535 -- intra-contig pair counts of long contigs -- keep their low 16 bits in
    the stream and their high part as a per-row term; the high part of an OFF-diagonal count above 65535 goes to a short
    side list sorted by (row, column) that the row sums add in (rows with a zero diagonal, a large diagonal and several
    large off-diagonal counts among them); more than 4096 such counts make the build fall back to 32-bit counts.
    Either way: n_iter equal to the oracle's and to the 32-bit stream's, x <= 1e-9 (measured ~1e-15), the same bits
    when run twice, and the stream width reported."""
    import torch
    from oracle import oracle
    rng = np.random.default_rng(77)
    n = 3000
    up = sp.triu(sp.random(n, n, density=0.004, random_state=5, data_rvs=lambda k: rng.integers(1, 400, size=k)), 1).tocsr()
    diag = rng.integers(0, 3000, size=n).astype(np.int64)
    diag[[3, 70, 71, 500, 2999]] = [65535, 65536, 65537, 4_000_000_000, 1_234_567]
    if offdiag_big == 'few':
        up = up.tolil()
        up[10, 2000] = 70000
        up[10, 2500] = 3_000_000_000
        up[11, 12] = 65536
        up[70, 71] = 131072                # both rows have a large diagonal too
        up[0, 2999] = 65537
        up[40, 41] = 100000                # rows 40 and 2000 have a zero diagonal (Q2)
        up = up.tocsr()
        diag[[40, 2000]] = 0
    elif offdiag_big == 'many':
        up = (up * 1000).tocsr()           # ~9000 of the 18000 upper entries exceed 65535
    m = (up + up.T + sp.diags(diag, dtype=np.int64)).tocsr()
    m.eliminate_zeros()
    m = m.astype(np.uint32)
    m.sort_indices()
    sites = rng.integers(0, 60, size=n).astype(np.int32)
    s1 = np.where(sites == 0, 1, sites).astype(np.float64)
    norm = m.astype(np.float64).tocoo()
    norm.data = norm.data * (1.0 / (s1[norm.row] * s1[norm.col]))
    _, x_ref, it_ref = oracle.kr_biostochastic(norm.tocsr())
    csr = dev.DeviceCSR.from_scipy(m, np.uint32)
    d_sites = dev.to_device(sites, torch.int32)
    got = {}
    for mode in (2, 1, 22):
        dev.check(dev.lib.b3c_set_option(5, mode % 10))
        try:
            x, info = dev.kr_scale_vector(csr, sites=d_sites)
        finally:
            dev.check(dev.lib.b3c_set_option(5, 2))
        got[mode] = (x.cpu().numpy().copy(), info)
    assert got[2][1]['stream_bytes_per_entry'] == (6 if offdiag_big == 'many' else 4)
    assert got[1][1]['stream_bytes_per_entry'] == 6
    assert got[2][1]['n_iter'] == got[1][1]['n_iter']
    assert got[2][1]['n_iter'] == it_ref
    assert _relerr(got[2][0], x_ref) <= REL_TOL and _relerr(got[1][0], x_ref) <= REL_TOL
    assert _relerr(got[2][0], got[1][0]) <= 1e-12
    assert np.array_equal(got[2][0], got[22][0])                  # the side list is sorted: the same bits every run


def test_extent_map_from_bam(dev, tmp_path):
    """ContactMap(bin_size=...): the binned extent map (contact_map.py:687-691, 779-788, 801-803) accumulated from the
    BAM reader's bin-level records with the same sort-reduce kernels, against the oracle's restatement."""
    import random
    import bam_writer
    from bin3c_b200 import bam_io
    from bin3c_b200.contact_map import ContactMap
    from oracle import oracle
    rng = random.Random(9)
    n_refs = 80
    refs = ['c{}'.format(i) for i in range(n_refs)]
    lengths = [rng.choice([400, 1200, 2600, 9000, 30000]) for _ in range(n_refs)]
    alns = []
    for t in range(6000):
        a = rng.randrange(n_refs)
        b = a if rng.random() < 0.6 else rng.randrange(n_refs)
        for k, tid in enumerate((a, b)):
            flag = 0x1 | (0x40 if k == 0 else 0x80) | (0x10 if rng.random() < 0.5 else 0)
            alns.append(dict(name='r%06d' % t, flag=flag, tid=tid, pos=rng.randrange(0, lengths[tid]),
                             mapq=rng.choice([0, 20, 60, 60, 60]), cigar=[(0, rng.randrange(20, 150))]))
    path = str(tmp_path / 'ext.bam')
    bam_writer.write_bam(path, refs, lengths, alns, level=1)
    bin_size, min_len = 1000, 1000
    pr, _ = bam_io.pair_records_from_bam(path, min_mapq=30, min_len=min_len, bin_size=bin_size)
    cm = ContactMap(pr, ['synthetic'], None, None, min_mapq=30, min_len=min_len, min_sig=1, bin_size=bin_size)
    keep = np.array(lengths) >= min_len
    lut = np.where(keep, np.cumsum(keep) - 1, -1)
    og = oracle.extent_grouping(np.array(lengths)[keep], bin_size)
    want, want_ext, _ = oracle.pair_alignments(alns, n_refs, min_mapq=30, idx_of=lut, grouping=og)
    assert np.array_equal(pr.extent_records, want_ext)
    ok = ((want_ext >> np.uint64(31)) & np.uint64(1)).astype(bool)
    bi = (want_ext & np.uint64(0x7fffffff)).astype(np.int64)
    bj = ((want_ext >> np.uint64(32)) & np.uint64(0x7fffffff)).astype(np.int64)
    nb = og['total_bins']
    dok, counts = oracle.bin_pairs_loop(bi, bj, ok, {b: b for b in range(nb)}, nb)
    ref = oracle.dok_to_coo(dok, nb)
    assert cm.grouping.total_bins == nb and cm.extent_map.shape == (nb, nb)
    got = cm.extent_map
    assert got.dtype == np.uint32
    assert np.array_equal(got.row, ref.row) and np.array_equal(got.col, ref.col) and np.array_equal(got.data, ref.data)
    assert cm.pair_counts['accepted'] == counts['accepted'] > 1000
    # without extent records the constructor refuses a bin size
    from bin3c_b200.contact_map import PairRecords
    with pytest.raises(AssertionError):
        ContactMap(PairRecords(pr.lengths, pr.sites, pr.records), ['synthetic'], None, None, min_mapq=30,
                   min_len=min_len, min_sig=1, bin_size=bin_size)


def test_cuda_path_vs_whole_reference_path(dev):
    """
    The CUDA path against outputs of the REFERENCE ITSELF: tests/golden/refpath.npz comes from the reference's own
    ContactMap / SeqOrder / sparse_utils / to_graph code run end to end (tests/golden/make_golden_refpath.py), not
    from the oracle.  Counts, contact matrix and mask bit-exact; identical KR iteration count; x, the balanced map and
    the edge weights within 1e-9 (north-star tolerance; zero site counts included, Q6).
    """
    import os
    from bin3c_b200 import cluster
    from bin3c_b200.contact_map import ContactMap, PairRecords
    with np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'refpath.npz')) as z:
        g = {k: z[k] for k in z.files}
    cm = ContactMap(PairRecords(g['lengths'], g['sites'], g['records']), ['synthetic'], None, None, min_mapq=60,
                    min_len=int(g['min_len']), min_sig=int(g['min_sig']), random_seed=1)
    assert [cm.pair_counts[k] for k in ('accepted', 'ref_excluded', 'poor_match')] == g['counts'].tolist()
    sm = cm.seq_map
    assert np.array_equal(sm.row, g['map_row']) and np.array_equal(sm.col, g['map_col'])
    assert np.array_equal(sm.data, g['map_data'])
    assert np.array_equal(cm.get_primary_acceptance_mask(), g['mask'].astype(bool))
    u, v, w, scl = cluster.to_edges(cm, norm=True, bisto=True, scale=True)
    assert cm.kr_info['n_iter'] == int(g['kr_n_iter'])
    assert _relerr(cm.bisto_scale, g['kr_x']) <= REL_TOL
    assert np.array_equal(u, g['edge_u']) and np.array_equal(v, g['edge_v'])
    assert _relerr(w, g['edge_w']) <= REL_TOL
    pm = cm.processed_map.tocoo()
    o1, o2 = np.lexsort((pm.col, pm.row)), np.lexsort((g['bal_col'], g['bal_row']))
    assert np.array_equal(pm.row[o1], g['bal_row'][o2]) and np.array_equal(pm.col[o1], g['bal_col'][o2])
    assert _relerr(pm.data[o1], g['bal_data'][o2]) <= REL_TOL


def test_contact_map_mask_rules_against_the_reference_mask(dev):
    """
    The acceptance-mask rules of ContactMap.set_primary_acceptance_mask (contact_map.py:856-909, Q5) on the reference's
    own path (refpath.npz): the mask is cached unless `update`; updated masks follow oracle.acceptance_mask on the
    reference's contact matrix; falsy thresholds fall back to the instance's and give the reference's stored mask
    again.  SeqOrder under that mask accepts exactly the reference's accepted contigs, in order, at the front.
    """
    import os
    from oracle import oracle
    from bin3c_b200.contact_map import ContactMap, PairRecords
    with np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'refpath.npz')) as z:
        g = {k: z[k] for k in z.files}
    min_len, min_sig = int(g['min_len']), int(g['min_sig'])
    cm = ContactMap(PairRecords(g['lengths'], g['sites'], g['records']), ['synthetic'], None, None, min_mapq=60,
                    min_len=min_len, min_sig=min_sig, random_seed=1)
    want = g['mask'].astype(bool)
    n = len(want)
    seq_len = g['lengths'][(g['lengths'] >= min_len) & (g['sites'] >= 0)]
    sm = sp.coo_matrix((g['map_data'], (g['map_row'], g['map_col'])), shape=(n, n))
    assert len(seq_len) == n
    assert np.array_equal(cm.get_primary_acceptance_mask(), want)
    cm.set_primary_acceptance_mask(min_len=5000, min_sig=20)                 # no update: the cached mask stays
    assert np.array_equal(cm.get_primary_acceptance_mask(), want)
    for ml, ms in ((5000, 20), (2000, 1), (1000, 50)):
        cm.set_primary_acceptance_mask(min_len=ml, min_sig=ms, update=True)
        assert np.array_equal(cm.get_primary_acceptance_mask(), oracle.acceptance_mask(seq_len, sm, ml, ms))
    cm.set_primary_acceptance_mask(min_len=0, min_sig=0, update=True)       # falsy -> the instance's thresholds
    assert np.array_equal(cm.get_primary_acceptance_mask(), want)
    cm.order.set_mask_only(cm.get_primary_acceptance_mask())
    assert np.array_equal(cm.order.mask_vector(), want) and cm.order.count_accepted() == int(want.sum())
    assert np.array_equal(cm.order.accepted(), np.flatnonzero(want))
    assert np.array_equal(cm.order.excluded(), np.flatnonzero(~want))
    assert np.array_equal(np.sort(cm.order.order['pos'][want]), np.arange(int(want.sum())))


def test_contact_map_from_bam_and_fasta_paths(dev, tmp_path):
    """
    The call bin3C.py mkmap makes (bin3C.py:148-158): ContactMap(BAM path, enzymes, FASTA path, min_insert, ...).  The
    BAM is decoded by the native reader with the map's own matcher and insert filter, the site counts come from the
    FASTA; matrix, counters (short_insert included) and edges against the oracle's pairing loop + path on the same
    alignments, site counts against a naive count.
    """
    import bam_writer
    from bin3c_b200 import cluster, synth
    from bin3c_b200.contact_map import ContactMap
    from bin3c_b200.exceptions import UnknownEnzymeException
    from oracle import oracle
    rng = np.random.default_rng(2718)
    n_refs, min_len, min_insert = 90, 1000, 400
    lengths = rng.integers(600, 4000, n_refs)
    seqs = [''.join(rng.choice(list('ACGT'), int(ln))) for ln in lengths]
    names = ['ctg%03d' % i for i in range(n_refs)]
    fasta = str(tmp_path / 'asm.fa')
    with open(fasta, 'w') as fh:
        for i, (nm, sq) in enumerate(zip(names, seqs)):
            if i == 7:
                continue                                    # one long-enough reference is missing from the FASTA
            fh.write('>{} some description\n'.format(nm))
            for k in range(0, len(sq), 70):
                fh.write(sq[k:k + 70] + '\n')
    naive = lambda sq: sum(1 for k in range(len(sq) - 3) if sq[k:k + 4] in ('AATT', 'GATC'))      # MluCI + Sau3AI
    keep = np.array([lengths[i] >= min_len and i != 7 for i in range(n_refs)])
    idx_of = np.where(keep, np.cumsum(keep) - 1, -1)
    n_seq = int(keep.sum())
    # alignments: pairs mostly inside a handful of "genomes", some proper pairs with short inserts
    alns = []
    for k in range(40_000):
        a = int(rng.integers(n_refs))
        b = a if rng.random() < 0.6 else int((a + rng.integers(1, 6)) % n_refs)
        good = rng.random() < 0.85
        proper = a == b and rng.random() < 0.5
        p1 = int(rng.integers(0, max(1, lengths[a] - 300)))
        p2 = p1 + int(rng.integers(50, 900)) if proper else int(rng.integers(0, max(1, lengths[b] - 100)))
        f1, f2 = 0x41 | (0x2 if proper else 0), 0x81 | (0x2 if proper else 0)
        if rng.random() < 0.5:                              # read 2 first in the file
            (a, p1, f1), (b, p2, f2) = (b, p2, f2), (a, p1, f1)
        alns.append(dict(name='q%06d' % k, flag=f1, tid=a, pos=p1, mapq=60 if good else 11, cigar=[(0, 100)]))
        alns.append(dict(name='q%06d' % k, flag=f2, tid=b, pos=p2, mapq=60, cigar=[(0, 100)]))
    path = str(tmp_path / 'hic.bam')
    bam_writer.write_bam(path, names, lengths.tolist(), alns, block_bytes=40000, level=1)

    cm = ContactMap(path, ['MluCI', 'Sau3AI'], fasta, min_insert, 60, min_len=min_len, min_sig=2, random_seed=1)
    assert cm.total_seq == n_seq and cm.min_insert == min_insert
    assert [si.sites for si in cm.seq_info] == [naive(seqs[i]) for i in range(n_refs) if keep[i]]
    assert [si.refid for si in cm.seq_info] == np.flatnonzero(keep).tolist()
    rec, st = oracle.pair_alignments(alns, n_refs, min_mapq=60, min_insert=min_insert, idx_of=idx_of)
    assert st['short_insert'] > 100 and cm.pair_counts['short_insert'] == st['short_insert']
    ti, tj, ok = synth.unpack_pairs(rec)
    sites = np.array([si.sites for si in cm.seq_info], dtype=np.int64)
    ref = oracle.run_path(ti, tj, ok, idx_of.astype(np.int32), lengths[keep], sites, min_len=min_len, min_sig=2)
    assert {k: cm.pair_counts[k] for k in ref['counts']} == ref['counts']
    sm = cm.seq_map
    assert np.array_equal(sm.row, ref['seq_map'].row) and np.array_equal(sm.col, ref['seq_map'].col)
    assert np.array_equal(sm.data, ref['seq_map'].data)
    u, v, w, scl = cluster.to_edges(cm, norm=True, bisto=True, scale=True)
    assert np.array_equal(u, ref['u']) and np.array_equal(v, ref['v']) and _relerr(w, ref['w']) <= REL_TOL
    # site counts handed over directly (array / dict / callable) give the same map
    by_name = {nm: naive(sq) for i, (nm, sq) in enumerate(zip(names, seqs)) if i != 7}
    for seq_file in (np.array([by_name.get(nm, -1) for nm in names]), by_name, lambda nm, ln: by_name.get(nm, -1)):
        cm2 = ContactMap(path, ['MluCI', 'Sau3AI'], seq_file, min_insert, 60, min_len=min_len, min_sig=2)
        assert np.array_equal(cm2.seq_map.data, sm.data) and cm2.pair_counts == cm.pair_counts
    with pytest.raises(UnknownEnzymeException):
        ContactMap(path, ['MluC1'], fasta, None, 60, min_len=min_len)
    # records read with one insert filter cannot describe a map with another
    from bin3c_b200 import bam_io
    pr, _ = bam_io.pair_records_from_bam(path, sites=np.array([by_name.get(nm, -1) for nm in names]), min_mapq=60,
                                         min_insert=min_insert, min_len=min_len)
    with pytest.raises(AssertionError):
        ContactMap(pr, ['x'], None, None, 60, min_len=min_len)


def test_extent_map_post_processing_vs_reference(dev, tmp_path):
    """
    SURVEY 8f-3 complete: bin3C mkmap --bin-size from a BAM file, then ContactMap.get_extent_map / _norm_extent /
    _compress_extent on the device against what the REFERENCE'S OWN class returned for the same alignments
    (tests/golden/extentmap.npz: every mean type, raw, and balanced).
    """
    import bam_writer
    from conftest import load_golden
    from bin3c_b200.contact_map import ContactMap
    g = load_golden('extentmap')
    n_refs = len(g['lengths'])
    alns = [dict(name='q%d' % (k // 2), flag=int(f), tid=int(t), pos=int(p), mapq=int(q), cigar=[(0, 100)])
            for k, (t, p, f, q) in enumerate(zip(g['a_tid'], g['a_pos'], g['a_flag'], g['a_mapq']))]
    path = str(tmp_path / 'ext.bam')
    bam_writer.write_bam(path, ['r%03d' % i for i in range(n_refs)], g['lengths'].tolist(), alns, block_bytes=50000, level=1)
    cm = ContactMap(path, ['synthetic'], g['sites'], None, 60, min_len=int(g['min_len']), min_sig=int(g['min_sig']),
                    bin_size=int(g['bin_size']))
    assert np.array_equal(cm.grouping.bins, g['bins'])
    assert np.array_equal(cm.get_primary_acceptance_mask().astype(np.uint8), g['mask'])
    em = cm.extent_map.tocoo()
    em.sum_duplicates()
    o = np.lexsort((em.col, em.row))
    assert np.array_equal(em.row[o], g['ext_row']) and np.array_equal(em.col[o], g['ext_col'])
    assert np.array_equal(em.data[o].astype(np.int64), g['ext_data'])

    def check(m, tag, tol):
        m = sp.coo_matrix(m)
        m.sum_duplicates()
        oo = np.lexsort((m.col, m.row))
        assert np.array_equal(m.row[oo], g[tag + '_row']) and np.array_equal(m.col[oo], g[tag + '_col']), tag
        assert _relerr(m.data[oo], g[tag + '_data']) <= tol, tag

    # as in the reference, the sequence mask reaches the order (and with it the extent map) in prepare_seq_map
    assert cm.get_extent_map(norm=False).shape == em.shape
    cm.prepare_seq_map(norm=True, bisto=True)
    for tag, kw, tol in (('geo', dict(norm=True, mean_type='geometric'), 1e-14),
                         ('har', dict(norm=True, mean_type='harmonic'), 1e-14),
                         ('ari', dict(norm=True, mean_type='arithmetic'), 1e-14),
                         ('raw', dict(norm=False), 0.0),
                         ('geo_bisto', dict(norm=True, bisto=True), REL_TOL)):
        m = cm.get_extent_map(**kw)
        assert list(m.shape) == g[tag + '_shape'].tolist()
        check(m, tag, tol)
    normed = cm._norm_extent(cm.extent_map.astype(float), 'geometric')
    assert sp.isspmatrix_lil(normed)
    check(normed, 'normonly', 1e-14)
    comp = cm._compress_extent(normed)
    assert sp.isspmatrix_coo(comp)
    check(comp, 'geo', 1e-14)
    with pytest.raises(RuntimeError):
        cm.get_extent_map(mean_type='quadratic')
    with pytest.raises(NotImplementedError):
        cm.get_extent_map(permute=True)


def test_accumulate_mirror_composite_count_escape(dev):
    """The composite of the mirror half carries (column, row, count) in 64 bits: with 27-bit indices only 10 bits are
    left for the count, so cells counted 1023 times or more take the escape (exact count looked up by bisection in the
    unique keys).  70M contigs, a few hot cells and many ordinary ones, against the oracle."""
    from bin3c_b200 import synth
    n = 70_000_000
    lut = np.arange(n, dtype=np.int32)
    rng = np.random.default_rng(11)
    a = rng.integers(0, n, 40_000)
    b = rng.integers(0, n, 40_000)
    hot_a = np.repeat(np.array([5, 69_999_999, 123_456, 5]), [1022, 1023, 5000, 70_000])
    hot_b = np.repeat(np.array([7, 3, 69_000_000, 60_000_001]), [1022, 1023, 5000, 70_000])
    ti, tj = np.concatenate([a, hot_a, hot_b[:2045]]), np.concatenate([b, hot_b, hot_a[:2045]])
    rec = synth.pack_pairs(ti, tj, np.ones(len(ti), bool))
    csr, info = _accumulate(dev, rec, lut, n)
    want, counts = _oracle_full(rec, lut, n)
    got = csr.to_scipy_coo()
    assert np.array_equal(got.row, want.row) and np.array_equal(got.col, want.col)
    assert np.array_equal(got.data, want.data) and got.data.max() == 70_000
    assert {k: info[k] for k in counts} == counts


# ---------------------------------------------------------------------------------------------
# tip-based N x N x 2 x 2 map (SURVEY.md 8f rank 4)
# ---------------------------------------------------------------------------------------------

def test_tip_based_map_vs_reference(dev, tmp_path):
    """ContactMap(tip_size=...) end to end from a BAM file -- the reader's tip records, the device accumulation over the
    doubled ids, mask from the tensor's marginal, site normalisation per (sequence, tip), KR on the marginal, compress,
    marginalise / flatten, edges -- and the sparse_utils 4-D drop-ins, against tests/golden/tipmap.npz: what the
    REFERENCE'S OWN classes and functions produced (contact_map.py:631-670, 791-798, sparse_utils.py:317-509, exec'd by
    tests/golden/make_golden_tip.py).  Tensor, counters and mask exact; scale factors, processed tensor and edge
    weights <= 1e-9."""
    import pickle
    import bam_writer
    from test_tips import golden_tip, params
    from bin3c_b200 import sparse_utils as su
    from bin3c_b200.cluster import to_edges
    from bin3c_b200.contact_map import ContactMap
    g, alns = golden_tip()
    lengths = g['lengths']
    n_refs = len(lengths)
    min_len, min_sig = int(g['min_len']), int(g['min_sig'])
    keep = lengths >= min_len
    n_seq = int(keep.sum())
    path = str(tmp_path / 'tips.bam')
    bam_writer.write_bam(path, ['r%d' % i for i in range(n_refs)], lengths.tolist(), alns, block_bytes=30000, level=1)
    for k in range(int(g['n_params'])):
        p, kw, tip = params(g, k)
        cm = ContactMap(path, ['MluCI'], g['sites2'], kw['min_insert'], min_mapq=kw['min_mapq'], min_len=min_len,
                        min_sig=min_sig, strong=kw['strong'], tip_size=tip)
        assert cm.is_tipbased() and cm.total_seq == n_seq
        c = cm.pair_counts
        assert [c['accepted'], c['ref_excluded'], c['poor_match'], c['short_insert'], c['not_tip']] == g[p + 'counts'].tolist()
        sm = cm.seq_map
        assert sm.shape == (n_seq, n_seq, 2, 2) and sm.data.dtype == np.uint32
        assert np.array_equal(sm.coords, g[p + 'coords']) and np.array_equal(sm.data, g[p + 'data'])
        assert cm.map_weight() == int(g[p + 'data'].sum())
        assert np.array_equal(cm.get_primary_acceptance_mask(), g[p + 'mask'])
        # the 4-D drop-ins on the tensor
        assert np.array_equal(su.max_offdiag_4d(sm), g[p + 'signal'])
        fl = su.flatten_tensor_4d(sm)
        assert np.array_equal(fl.row, g[p + 'flat_row']) and np.array_equal(fl.col, g[p + 'flat_col'])
        assert np.array_equal(fl.data, g[p + 'flat_data'])
        cp = su.compress_4d(sm, np.arange(n_seq) % 4 != 1)
        assert cp.shape == (int(g[p + 'cmp_n']),) * 2 + (2, 2)
        assert np.array_equal(cp.coords, g[p + 'cmp_coords']) and np.array_equal(cp.data, g[p + 'cmp_data'])
        bal, scl = su.kr_biostochastic_4d(sm)
        assert _relerr(scl, g[p + 'kr_scl']) <= REL_TOL and _relerr(bal.data, g[p + 'kr_data']) <= REL_TOL
        # the path: prepare_seq_map(norm, bisto) -> get_subspace(marginalise) -> edges
        u, v, w, scale = to_edges(cm, norm=True, bisto=True, scale=True)
        assert _relerr(cm.bisto_scale, g[p + 'bisto_scale']) <= REL_TOL
        assert np.array_equal(cm.processed_map.coords, g[p + 'proc_coords'])
        assert _relerr(cm.processed_map.data, g[p + 'proc_data']) <= REL_TOL
        assert np.array_equal(u, g[p + 'edge_u']) and np.array_equal(v, g[p + 'edge_v'])
        assert _relerr(w, g[p + 'edge_w']) <= REL_TOL
        fs = cm.get_subspace(marginalise=False, flatten=True).tocsr()
        fs.sort_indices()
        assert np.array_equal(fs.indptr, g[p + 'fsub_indptr']) and np.array_equal(fs.indices, g[p + 'fsub_indices'])
        assert _relerr(fs.data, g[p + 'fsub_data']) <= REL_TOL
        assert pickle.loads(pickle.dumps(cm)).seq_map.nnz == sm.nnz
    # the per-pair protocol of the reference's accumulator (a dict of 2 x 2 cells, contact_map.py:798)
    acc = su.Sparse4DAccumulator(5)
    cell = np.zeros((2, 2), dtype=np.uint32)
    cell[1, 0] = 1
    acc[1, 3] += cell
    acc[1, 3] += cell
    acc[2, 2] += cell
    t = acc.get_coo()
    assert t.coords.T.tolist() == [[1, 3, 1, 0], [2, 2, 1, 0], [3, 1, 0, 1]] and t.data.tolist() == [2, 1, 2]
