"""
Kernel-level tests (-m gpu): the row-wise kernels (rowops.cu), the compress / edge kernels in their staged and fused
forms, and the KR tuning variants (kr.cu), each against a plain float64 (or np.longdouble) restatement of the
operation, on matrices built to put rows exactly at the kernels' switch points:

- the row-segment edge kernels cut a row into pieces of T = max(4096, ceil(nnz / n_local)) entries and walk a piece in
  four 32-entry windows per trip, so the adversarial matrix has rows of 0, 1, 31..33, 127..129, 4095..4097,
  8192, 8193 and 3 * 4096 + 1 entries, diagonals on piece boundaries, missing and zero diagonals, and upper triangles
  that start mid-window or are only the last entry; the dense block has a mean row length above 4096 with T odd;
- every row-wise entry point takes (row_lo, n_local), so each matrix is also cut into row blocks at 1024-aligned and at
  odd row_lo, with a local indptr and global columns, as the sharded driver hands them over;
- the KR flag bits (B3C_OPT_KR_FLAGS) and the SpMV operand layouts they select.

Where the kernel promises the reference's operations in the reference's order, the comparison is bit for bit.  The
generator and the references are checked on the CPU by tests/test_kernel_refs.py.
"""
import sys

import numpy as np
import pytest
import scipy.sparse as sp

pytestmark = pytest.mark.gpu

EDGE_SEG = 4096                   # rowops.cu: minimum row-segment length of the fused edge kernels

# ---------------------------------------------------------------------------------------------
# adversarial CSR builder
# ---------------------------------------------------------------------------------------------

N_ADV = 20000
ADV_ROW0 = 9990                   # the designated rows sit here, with ~10k ordinary rows on either side
U32_MAX = 2 ** 32 - 1

# (label, row length including the diagonal, columns below the row, diagonal: 'yes' | 'none' | 'zero' (stored 0))
ADV_ROWS = (
    [('len%d' % L, L, L // 2, 'yes') for L in (1, 31, 32, 33, 127, 128, 129, 4095, 4096, 4097, 8192, 8193)]
    + [('len0', 0, 0, 'none'),
       ('len12289', 3 * EDGE_SEG + 1, 6144, 'yes'),
       ('diag_first_of_piece2', 2 * EDGE_SEG + 1, EDGE_SEG, 'yes'),       # diagonal is entry 4096
       ('diag_last_of_piece1', 2 * EDGE_SEG, EDGE_SEG - 1, 'yes'),        # diagonal is entry 4095
       ('diag_last_of_piece2', 3 * EDGE_SEG + 1, 2 * EDGE_SEG - 1, 'yes'),
       ('diag_last_entry', EDGE_SEG, EDGE_SEG - 1, 'yes'),                # the diagonal is the only upper entry
       ('no_diag', EDGE_SEG + 1, 2000, 'none'),
       ('zero_diag', 129, 60, 'zero'),
       ('upper_mid_window', 200, 45, 'yes'),                              # upper triangle starts at entry 45
       ('upper_last_only', EDGE_SEG + 1, EDGE_SEG, 'none'),               # only upper entry: the last one
       ('upper_last_only_short', 33, 32, 'none'),
       ('max_is_diag', 50, 20, 'yes'),                                    # diagonal 2^32-1, larger than the rest
       ('diag_only_zero_site', 1, 0, 'yes')])


def _counts(rng, k):
    """uint32 counts spread over the whole range: log-uniform in [1, 2^32 - 1], some exactly 1 and 2^32 - 1."""
    c = np.floor(2.0 ** rng.uniform(0.0, 32.0, k)).astype(np.int64)
    c[rng.random(k) < 0.02] = 1
    c[rng.random(k) < 0.02] = U32_MAX
    return np.clip(c, 1, U32_MAX)


def _csr_from_keys(n, row, col, data):
    """CSR (indptr int64, indices int32, data) from unique (row, col) keys, columns sorted."""
    o = np.lexsort((col, row))
    indptr = np.zeros(n + 1, dtype=np.int64)
    np.cumsum(np.bincount(row, minlength=n), out=indptr[1:])
    return indptr, col[o].astype(np.int32), data[o]


def adversarial_counts(seed=11):
    """
    Symmetric uint32 count matrix of N_ADV contigs: ordinary rows with ~16 entries and the designated rows of ADV_ROWS
    at ADV_ROW0.., whose columns are drawn from the ordinary rows only, so their lengths and diagonal positions are
    exactly as listed.  Returns dict(indptr, indices, counts, rows={label: row}, sites, x, bin_len).
    """
    rng = np.random.default_rng(seed)
    n = N_ADV
    rows = {lab: ADV_ROW0 + i for i, (lab, _, _, _) in enumerate(ADV_ROWS)}
    designated = np.zeros(n, dtype=bool)
    designated[list(rows.values())] = True
    ordinary = np.flatnonzero(~designated)
    r_up, c_up, d_up = [], [], []
    # background among the ordinary rows: ~8 upper entries per row, and most diagonals
    k = 8 * len(ordinary)
    a, b = rng.choice(ordinary, k), rng.choice(ordinary, k)
    keep = a != b
    key = np.unique(np.minimum(a, b)[keep].astype(np.int64) * n + np.maximum(a, b)[keep])
    r_up.append(key // n)
    c_up.append(key % n)
    d_up.append(_counts(rng, len(key)))
    dg = ordinary[rng.random(len(ordinary)) < 0.8]
    r_up.append(dg)
    c_up.append(dg)
    d_up.append(_counts(rng, len(dg)))
    for lab, L, below, diag in ADV_ROWS:
        r = rows[lab]
        n_diag = 0 if diag == 'none' else 1
        lo_pool, hi_pool = ordinary[ordinary < r], ordinary[ordinary > r]
        cols = np.r_[rng.choice(lo_pool, below, replace=False), rng.choice(hi_pool, L - below - n_diag, replace=False)]
        r_up.append(np.minimum(cols, r))
        c_up.append(np.maximum(cols, r))
        d = _counts(rng, len(cols))
        d_up.append(np.minimum(d, 2 ** 31) if lab == 'max_is_diag' else d)
        if n_diag:
            r_up.append(np.array([r]))
            c_up.append(np.array([r]))
            d_up.append(np.array([0 if diag == 'zero' else U32_MAX if lab == 'max_is_diag' else 7]))
    ru, cu, du = (np.concatenate(t).astype(np.int64) for t in (r_up, c_up, d_up))
    assert len(np.unique(ru * n + cu)) == len(ru)
    off = ru != cu
    row, col = np.r_[ru, cu[off]], np.r_[cu, ru[off]]
    indptr, indices, counts = _csr_from_keys(n, row, col, np.r_[du, du[off]].astype(np.uint32))
    sites = rng.integers(0, 60, n).astype(np.int32)
    sites[rng.random(n) < 0.1] = 0                                   # zero sites read as one (Q6)
    sites[rows['diag_only_zero_site']] = 0
    x = 10.0 ** rng.uniform(-3.0, 3.0, n)
    bin_len = np.floor(10.0 ** rng.uniform(3.0, 6.5, n)) + rng.integers(0, 2, n)
    return dict(n=n, indptr=indptr, indices=indices, counts=counts, rows=rows, sites=sites, x=x, bin_len=bin_len)


DENSE_TOTAL, DENSE_LO, DENSE_N = 16384, 6001, 3000
DENSE_LENGTHS = (0, 1, 129, 4500, 4501, 4502, 9002, 9003, 9004, 13503)      # mean 5414.5: T = 5415 (odd)


def dense_block(seed=5):
    """
    Rows [DENSE_LO, DENSE_LO + DENSE_N) of a DENSE_TOTAL-contig count matrix (local indptr, global columns) whose mean
    row length is above 4096, so the edge kernels' piece length T = ceil(nnz / n_local) is odd and not a multiple of
    32.  Rows of 9003 entries have their diagonal at entry T (first of piece 2), rows of 9002 at entry T - 1 (last of
    piece 1); the other rows hold it at random or not at all.
    """
    rng = np.random.default_rng(seed)
    lengths = np.resize(np.array(DENSE_LENGTHS, dtype=np.int64), DENSE_N)
    T = seg_len(np.r_[0, np.cumsum(lengths)])
    cols = []
    for r, L in enumerate(lengths):
        gr = DENSE_LO + r
        if L in (9002, 9003):
            below = T - 1 if L == 9002 else T
            c = np.r_[rng.choice(gr, below, replace=False), gr,
                      gr + 1 + rng.choice(DENSE_TOTAL - gr - 1, L - below - 1, replace=False)]
        else:
            c = rng.choice(DENSE_TOTAL, L, replace=False)
        cols.append(np.sort(c))
    indptr = np.r_[0, np.cumsum(lengths)].astype(np.int64)
    indices = np.concatenate(cols).astype(np.int32)
    sites = rng.integers(0, 60, DENSE_TOTAL).astype(np.int32)
    sites[rng.random(DENSE_TOTAL) < 0.1] = 0
    return dict(n=DENSE_TOTAL, row_lo=DENSE_LO, indptr=indptr, indices=indices,
                counts=_counts(rng, len(indices)).astype(np.uint32), sites=sites,
                x=10.0 ** rng.uniform(-3.0, 3.0, DENSE_TOTAL), T=T)


# ---------------------------------------------------------------------------------------------
# float64 references, in the kernels' operation order
# ---------------------------------------------------------------------------------------------

def seg_len(indptr):
    """The piece length of the fused edge kernels for a block: max(4096, ceil(nnz / n_local))."""
    nl = len(indptr) - 1
    return max(EDGE_SEG, -(-int(indptr[-1] - indptr[0]) // nl))


def row_of_entry(indptr, row_lo=0):
    return np.repeat(np.arange(len(indptr) - 1, dtype=np.int64), np.diff(indptr)) + row_lo


def site_values(sites):
    s = np.asarray(sites, dtype=np.float64).copy()
    s[s == 0] = 1.0
    return s


def ref_max_offdiag(indptr, indices, data, row_lo=0):
    """Per row of the block: the largest value off the diagonal, 0 if there is none."""
    gr = row_of_entry(indptr, row_lo)
    out = np.zeros(len(indptr) - 1, dtype=data.dtype)
    off = indices != gr
    np.maximum.at(out, gr[off] - row_lo, data[off])
    return out


def ref_site_norm(indptr, indices, data, sites, row_lo=0):
    """c * (1.0 / (s_i * s_j)), zero sites read as one."""
    s = site_values(sites)
    return data.astype(np.float64) * (1.0 / (s[row_of_entry(indptr, row_lo)] * s[indices]))


def ref_extent_norm(indptr, indices, data, bin_len, mean_type, row_lo=0):
    """v / (1e-3 * mean(L_i, L_j)); mean_type 0 sqrt(Li Lj), 1 ((2 Li) Lj) / (Li + Lj), 2 0.5 (Li + Lj), -1 a copy."""
    v = data.astype(np.float64)
    if mean_type < 0:
        return v
    li, lj = bin_len[row_of_entry(indptr, row_lo)], bin_len[indices]
    m = {0: lambda: np.sqrt(li * lj), 1: lambda: (2.0 * li) * lj / (li + lj), 2: lambda: 0.5 * (li + lj)}[mean_type]()
    return v / (1e-3 * m)


def ref_kr_scale(indptr, indices, a, x, row_lo=0):
    """x_i * (a_ij * x_j)."""
    return x[row_of_entry(indptr, row_lo)] * (a * x[indices])


def ref_fused_values(indptr, indices, counts, sites, x, row_lo=0):
    """The fused edge value x_i * ((c * (1.0 / (s_i * s_j))) * x_j): site_norm followed by kr_scale."""
    return ref_kr_scale(indptr, indices, ref_site_norm(indptr, indices, counts, sites, row_lo), x, row_lo)


def ref_compress(indptr, indices, vals, mask, row_lo=0):
    """
    compress + edge list of a block: entries whose row and column are accepted are kept, the kept ones with column >=
    row are edges (in CSR order), ids are gapless over the accepted contigs.  Returns the per-block quantities; the
    weights need the global maximum: w = vals[edge] * (1.0 / vmax).
    """
    mask = np.asarray(mask, dtype=bool)
    gr = row_of_entry(indptr, row_lo)
    newidx = np.where(mask, np.cumsum(mask) - 1, -1)
    keep = mask[gr] & mask[indices]
    edge = keep & (indices >= gr)
    kept_rows = np.bincount(gr[keep] - row_lo, minlength=len(indptr) - 1)
    acc_rows = mask[row_lo:row_lo + len(indptr) - 1]
    return dict(n_accepted=int(mask.sum()), n_kept=int(keep.sum()), n_edges=int(edge.sum()),
                vmax=float(vals[keep].max()) if keep.any() else 0.0,
                u=newidx[gr[edge]].astype(np.int32), v=newidx[indices[edge]].astype(np.int32), w_unscaled=vals[edge],
                sub_indptr=np.r_[0, np.cumsum(kept_rows[acc_rows])].astype(np.int64),
                sub_indices=newidx[indices[keep]].astype(np.int32), sub_data=vals[keep])


def ref_scale(vmax):
    """cluster.py:316: scl = 1.0 / max, infinite when nothing is kept."""
    with np.errstate(divide='ignore'):
        return np.float64(1.0) / np.float64(vmax)


def ref_asymmetry_count(n, indptr, indices, a, tol):
    """Stored entries with |a_ij - a_ji| >= tol, a missing mirror counting as 0."""
    r = row_of_entry(indptr)
    key = r * n + indices
    mk = indices.astype(np.int64) * n + r
    pos = np.minimum(np.searchsorted(key, mk), len(key) - 1)
    mirror = np.where(key[pos] == mk, a[pos], 0.0)
    return int(np.count_nonzero(np.abs(a - mirror) >= tol))


def dense_is_hermitian(n, indptr, indices, a, tol):
    """sparse_utils.py:10-18 on the dense matrix: |m - m.H| < tol everywhere."""
    d = sp.csr_matrix((a, indices, indptr), shape=(n, n)).toarray()
    return bool(np.all(np.abs(d - d.conj().T) < tol))


# ---------------------------------------------------------------------------------------------
# fixtures
# ---------------------------------------------------------------------------------------------

# b3c_set_option keys and their defaults: slab width, max slabs, KR flags, count stream, graphs
DEFAULT_OPTIONS = ((1, 28672), (2, 16), (3, 22), (5, 2), (6, 1))


@pytest.fixture(scope='module')
def dev():
    import torch
    if not torch.cuda.is_available():
        pytest.skip('no CUDA device')
    from bin3c_b200 import device
    return device


@pytest.fixture(autouse=True)
def _restore_options():
    """Options are process-global: put every one back after each test, whether it passed or not."""
    yield
    cabi = sys.modules.get('bin3c_b200._cabi')
    if cabi is not None:
        for key, value in DEFAULT_OPTIONS:
            cabi.check(cabi.lib.b3c_set_option(key, value))


def _set_options(dev, **kw):
    keys = dict(width=1, max_slabs=2, flags=3, count_stream=5)
    for k, v in kw.items():
        if v is not None:
            dev.check(dev.lib.b3c_set_option(keys[k], int(v)))


@pytest.fixture(scope='module')
def adv():
    m = adversarial_counts()
    m['normed'] = ref_site_norm(m['indptr'], m['indices'], m['counts'], m['sites'])
    return m


@pytest.fixture(scope='module')
def dense():
    return dense_block()


def tiling(name, n=N_ADV):
    """Row blocks: the whole matrix; 1024-aligned row_lo; odd row_lo (1, 333, ...) through the designated rows."""
    cuts = {'whole': [0, n],
            'aligned': [0, 1024, 9216, 10240, n],
            'odd': [0, 1, 334, ADV_ROW0 + 11, ADV_ROW0 + 12, ADV_ROW0 + 21, n]}[name]
    return list(zip(cuts[:-1], cuts[1:]))


TILINGS = ['whole', 'aligned', 'odd']


def _block(m, lo, hi):
    """Host arrays of rows [lo, hi): local indptr from 0, global columns, and the slice of entries."""
    a, b = int(m['indptr'][lo]), int(m['indptr'][hi])
    return m['indptr'][lo:hi + 1] - a, m['indices'][a:b], slice(a, b)


def _dev_block(dev, m, lo, hi, data):
    """DeviceCSR of rows [lo, hi) with `data` (uint32 counts or float64 values of the block's entries)."""
    indptr, indices, _ = _block(m, lo, hi)
    counts = data.dtype == np.uint32
    return dev.DeviceCSR(hi - lo, dev.to_device(indptr), dev.to_device(indices), dev.to_device(data), counts=counts,
                         row_lo=lo, n_total=m['n'])


def _np(t):
    return t.cpu().numpy()


# ---------------------------------------------------------------------------------------------
# B. row-wise kernels, whole matrices and row blocks
# ---------------------------------------------------------------------------------------------

def test_adversarial_rows_reach_the_switch_points(adv):
    """The designated rows sit where they should relative to the pieces of T = 4096 entries (whole matrix)."""
    assert seg_len(adv['indptr']) == EDGE_SEG
    ip, idx, rows = adv['indptr'], adv['indices'], adv['rows']
    for lab, L, below, diag in ADV_ROWS:
        r = rows[lab]
        assert ip[r + 1] - ip[r] == L, lab
        if diag != 'none':
            assert idx[ip[r] + below] == r, lab


@pytest.mark.parametrize('tile', TILINGS)
def test_max_offdiag(dev, adv, tile):
    from oracle import oracle
    m = sp.csr_matrix((adv['counts'], adv['indices'], adv['indptr']), shape=(adv['n'],) * 2)
    want_u32 = oracle.max_offdiag(m)
    want_f64 = oracle.max_offdiag(sp.csr_matrix((adv['normed'], adv['indices'], adv['indptr']), shape=m.shape))
    rows = adv['rows']
    assert want_u32[rows['len1']] == 0 and want_u32[rows['len0']] == 0            # only a diagonal / empty
    r = rows['max_is_diag']
    assert want_u32[r] < m[r, r] == U32_MAX
    for lo, hi in tiling(tile):
        _, _, s = _block(adv, lo, hi)
        got = dev.max_offdiag(_dev_block(dev, adv, lo, hi, adv['counts'][s]))
        assert np.array_equal(_np(got).view(np.uint32), want_u32[lo:hi]), (lo, hi)
        got = dev.max_offdiag(_dev_block(dev, adv, lo, hi, adv['normed'][s]))
        assert np.array_equal(_np(got), want_f64[lo:hi]), (lo, hi)


@pytest.mark.parametrize('tile', TILINGS)
def test_site_norm(dev, adv, tile):
    import torch
    sites = dev.to_device(adv['sites'], torch.int32)
    for lo, hi in tiling(tile):
        ip, idx, s = _block(adv, lo, hi)
        want = ref_site_norm(ip, idx, adv['counts'][s], adv['sites'], lo)
        assert np.array_equal(want, adv['normed'][s])
        got = dev.site_norm(_dev_block(dev, adv, lo, hi, adv['counts'][s]), sites)          # uint32 -> float64
        assert np.array_equal(_np(got.data), want), (lo, hi)
        raw = adv['counts'][s].astype(np.float64)
        csr = _dev_block(dev, adv, lo, hi, raw)
        out = dev.site_norm(csr, sites)                                                     # float64, in place
        assert out.data.data_ptr() == csr.data.data_ptr()
        assert np.array_equal(_np(out.data), want), (lo, hi)


@pytest.mark.parametrize('mean', ['arithmetic', 'harmonic', None, 'geometric'])
@pytest.mark.parametrize('tile', TILINGS)
def test_extent_norm(dev, adv, tile, mean):
    from oracle import oracle
    mt = dev.MEAN_TYPES[mean]
    L = dev.to_device(adv['bin_len'])
    for lo, hi in tiling(tile):
        ip, idx, s = _block(adv, lo, hi)
        got = _np(dev.extent_norm(_dev_block(dev, adv, lo, hi, adv['counts'][s]), L, mean).data)
        assert np.array_equal(got, ref_extent_norm(ip, idx, adv['counts'][s], adv['bin_len'], mt, lo)), (lo, hi)
    if mean is None or tile != 'whole':
        return
    # the oracle's own formula: the same bits for the arithmetic and harmonic means, 1 ulp for (Li Lj) ** 0.5
    n = adv['n']
    m = sp.csr_matrix((adv['counts'], adv['indices'], adv['indptr']), shape=(n, n)).tocoo()
    want = oracle.norm_extent(m, adv['bin_len'], np.ones(n, dtype=np.int64), mean).data
    if mean == 'geometric':
        assert np.all(np.abs(got - want) <= np.spacing(np.abs(want)))
    else:
        assert np.array_equal(got, want)


@pytest.mark.parametrize('tile', TILINGS)
def test_kr_scale(dev, adv, tile):
    x = dev.to_device(adv['x'])
    for lo, hi in tiling(tile):
        ip, idx, s = _block(adv, lo, hi)
        got = dev.kr_apply(_dev_block(dev, adv, lo, hi, adv['normed'][s]), x)
        assert np.array_equal(_np(got.data), ref_kr_scale(ip, idx, adv['normed'][s], adv['x'], lo)), (lo, hi)


ASYM_TOL = 2.0 ** -20


def _asym_case(adv, case):
    """A principal sub-matrix of the normalised adversarial matrix (rows up to ~3000 entries), perturbed.
    Returns (n, indptr, indices, a, the expected count)."""
    lo, hi = ADV_ROW0 - 1500, ADV_ROW0 + 1500
    n = hi - lo
    full = sp.csr_matrix((adv['normed'], adv['indices'], adv['indptr']), shape=(adv['n'],) * 2)
    c = full[lo:hi, lo:hi].tocoo()
    row, col, a = c.row.astype(np.int64), c.col.astype(np.int64), c.data.copy()
    i, j = adv['rows']['len8193'] - lo, adv['rows']['len4097'] - lo             # two long rows
    off = (row < col) & (row != i) & (row != j) & (col != i) & (col != j)
    p = np.flatnonzero(off)[len(np.flatnonzero(off)) // 2]                     # an ordinary pair (p_r, p_c)
    pr, pc = row[p], col[p]
    q = np.flatnonzero((row == pc) & (col == pr))[0]
    want = 0
    if case in ('tol', 'half_tol'):
        a[p] = a[q] = 0.5
        a[p] = 0.5 + (ASYM_TOL if case == 'tol' else ASYM_TOL / 2)             # |difference| exactly tol / tol/2
        want = 2 if case == 'tol' else 0
    elif case == 'missing_mirror':
        keep = np.ones(len(a), dtype=bool)
        keep[q] = False
        row, col, a = row[keep], col[keep], a[keep]
        want = 1
    elif case == 'explicit_zero':
        ir = np.flatnonzero(row == i)
        mine = set(col[ir].tolist()) | set(row[col == i].tolist())
        k = next(k for k in range(n) if k not in mine and k != i)
        row, col, a = np.r_[row, i], np.r_[col, k], np.r_[a, 0.0]               # stored 0 at (i, k), nothing at (k, i)
    elif case == 'long_row_entry':
        e = np.flatnonzero((row == i) & (col > i))[-1]                          # the last upper entry of a long row
        a[e] = a[e] + 4 * ASYM_TOL
        want = 2
    indptr, indices, data = _csr_from_keys(n, row, col, a)
    return n, indptr, indices, data, want


@pytest.mark.parametrize('case', ['symmetric', 'tol', 'half_tol', 'missing_mirror', 'explicit_zero',
                                  'long_row_entry'])
def test_asymmetry_count(dev, adv, case):
    n, indptr, indices, a, want = _asym_case(adv, case)
    assert ref_asymmetry_count(n, indptr, indices, a, ASYM_TOL) == want
    csr = dev.DeviceCSR(n, dev.to_device(indptr), dev.to_device(indices), dev.to_device(a))
    got = dev.asymmetry_count(csr, ASYM_TOL)
    assert got == want
    assert (got == 0) == dense_is_hermitian(n, indptr, indices, a, ASYM_TOL)


def test_asymmetry_count_whole_adversarial(dev, adv):
    """Every row length of the adversarial matrix, exactly symmetric (0), then with the mirror of the last entry of its
    longest row perturbed by exactly tol (2)."""
    n, ip, idx = adv['n'], adv['indptr'], adv['indices']
    a = adv['normed'].copy()
    assert dev.asymmetry_count(dev.DeviceCSR(n, dev.to_device(ip), dev.to_device(idx), dev.to_device(a)), ASYM_TOL) == 0
    r = adv['rows']['len12289']
    e = ip[r + 1] - 1
    c = idx[e]
    q = ip[c] + np.searchsorted(idx[ip[c]:ip[c + 1]], r)
    a[e] = a[q] = 0.25
    a[q] = 0.25 + ASYM_TOL
    assert ref_asymmetry_count(n, ip, idx, a, ASYM_TOL) == 2
    assert dev.asymmetry_count(dev.DeviceCSR(n, dev.to_device(ip), dev.to_device(idx), dev.to_device(a)), ASYM_TOL) == 2


def adv_mask(adv, kind):
    n = adv['n']
    mask = np.ones(n, dtype=bool)
    if kind == 'none_in_block':
        mask[1:334] = False                              # every row of the odd tiling's second block
        mask[ADV_ROW0 + 11] = False                      # and the one-row block of the 8193-entry row
    elif kind == 'alternating':
        mask[1::2] = False
    elif kind == 'long_row_diag':
        mask[adv['rows']['len12289']] = False            # only the contig that holds the longest row's diagonal
    return mask


def _run_compress(dev, m, lo, hi, mask, fused, vals, want_global, sites=None, x=None, block_max=None):
    """compress_edges on rows [lo, hi); `reduce_max` records the block's maximum and installs the global one, as the
    sharded driver's all-reduce does."""
    import torch
    whole = (lo, hi) == (0, m['n'])
    _, _, s = _block(m, lo, hi)
    seen = []

    def reduce_max(t):
        seen.append(float(t.cpu()[0]))
        t.fill_(want_global)

    data = m['counts'][s] if fused else vals[s]
    kw = dict(sites=dev.to_device(sites, torch.int32), x=dev.to_device(x)) if fused else {}
    res = dev.compress_edges(_dev_block(dev, m, lo, hi, data), dev.to_device(mask.astype(np.uint8), torch.uint8),
                             want_sub=whole and not fused, reduce_max=None if whole else reduce_max, **kw)
    if not whole:
        assert seen == [block_max]
    return res


def _check_block(res, want, scl):
    assert (res['n_accepted'], res['n_kept'], res['n_edges']) == (want['n_accepted'], want['n_kept'], want['n_edges'])
    n = want['n_edges']
    assert res['u'].numel() == res['v'].numel() == res['w'].numel() == n
    assert np.array_equal(_np(res['u']), want['u']) and np.array_equal(_np(res['v']), want['v'])
    assert np.array_equal(_np(res['w']), want['w_unscaled'] * scl)
    assert _np(res['scl'])[0] == scl or (np.isinf(scl) and np.isinf(_np(res['scl'])[0]))


def _compress_case(dev, m, blocks, mask, fused):
    """Every block against the reference, the global scale through reduce_max, and the concatenated block lists
    against the whole-matrix list."""
    vals = (ref_fused_values(m['indptr'], m['indices'], m['counts'], m['sites'], m['x'], m.get('row_lo', 0)) if fused
            else m['normed'])
    ip, idx = m['indptr'], m['indices']
    wants = []
    for lo, hi in blocks:
        bip, bidx, s = _block(m, lo, hi)
        wants.append(ref_compress(bip, bidx, vals[s], mask, lo + m.get('row_lo', 0)))
    gmax = max(w['vmax'] for w in wants)
    scl = ref_scale(gmax)
    got_u, got_v, got_w = [], [], []
    for (lo, hi), want in zip(blocks, wants):
        res = _run_compress(dev, m, lo, hi, mask, fused, vals, gmax, m['sites'], m['x'], want['vmax'])
        _check_block(res, want, scl)
        got_u.append(_np(res['u'])); got_v.append(_np(res['v'])); got_w.append(_np(res['w']))
        if res['sub'] is not None:
            sub = res['sub']
            assert sub.n == want['n_accepted']
            assert np.array_equal(_np(sub.indptr), want['sub_indptr'])
            assert np.array_equal(_np(sub.indices), want['sub_indices'])
            assert np.array_equal(_np(sub.data), want['sub_data'])
    whole = ref_compress(ip, idx, vals, mask, m.get('row_lo', 0))
    assert np.array_equal(np.concatenate(got_u), whole['u']) and np.array_equal(np.concatenate(got_v), whole['v'])
    assert np.array_equal(np.concatenate(got_w), whole['w_unscaled'] * scl)
    return wants


@pytest.mark.parametrize('fused', [False, True], ids=['staged', 'fused'])
@pytest.mark.parametrize('mask_kind', ['all', 'none_in_block', 'alternating', 'long_row_diag'])
@pytest.mark.parametrize('tile', TILINGS)
def test_compress_edges(dev, adv, tile, mask_kind, fused):
    wants = _compress_case(dev, adv, tiling(tile), adv_mask(adv, mask_kind), fused)
    if mask_kind == 'none_in_block' and tile == 'odd':
        assert wants[1]['n_edges'] == wants[3]['n_edges'] == 0         # blocks [1, 334) and the 8193-entry row


@pytest.mark.parametrize('fused', [False, True], ids=['staged', 'fused'])
@pytest.mark.parametrize('mask_kind', ['all', 'alternating'])
def test_compress_edges_dense_block(dev, dense, mask_kind, fused):
    """A block whose pieces are T = 5415 entries (odd, not a multiple of 32), diagonals on piece boundaries; another
    rank holds the global maximum."""
    import torch
    assert dense['T'] == seg_len(dense['indptr']) == 5415
    ip, idx = dense['indptr'], dense['indices']
    mask = np.ones(DENSE_TOTAL, dtype=bool)
    if mask_kind == 'alternating':
        mask[::2] = False
    if fused:
        vals = ref_fused_values(ip, idx, dense['counts'], dense['sites'], dense['x'], DENSE_LO)
    else:
        vals = ref_site_norm(ip, idx, dense['counts'], dense['sites'], DENSE_LO)
    want = ref_compress(ip, idx, vals, mask, DENSE_LO)
    gmax = want['vmax'] * 2.0
    seen = []

    def reduce_max(t):
        seen.append(float(t.cpu()[0]))
        t.fill_(gmax)

    csr = dev.DeviceCSR(DENSE_N, dev.to_device(ip), dev.to_device(idx), dev.to_device(dense['counts'] if fused else vals),
                        counts=fused, row_lo=DENSE_LO, n_total=DENSE_TOTAL)
    kw = dict(sites=dev.to_device(dense['sites'], torch.int32), x=dev.to_device(dense['x'])) if fused else {}
    res = dev.compress_edges(csr, dev.to_device(mask.astype(np.uint8), torch.uint8), want_sub=False,
                             reduce_max=reduce_max, **kw)
    assert seen == [want['vmax']]
    _check_block(res, want, ref_scale(gmax))
    got = dev.max_offdiag(csr)
    want_max = ref_max_offdiag(ip, idx, dense['counts'] if fused else vals, DENSE_LO)
    assert np.array_equal(_np(got).view(want_max.dtype), want_max)


# ---- zero edges -------------------------------------------------------------------------------

def _no_edge_matrix():
    """Accepted contigs 0, 2, 4 without a diagonal, each paired only with a rejected contig (1, 3, 5); the rejected
    contigs 5..9 also pair among themselves."""
    n = 10
    up = [(0, 1, 40), (2, 3, 7), (4, 5, 12), (5, 6, 3), (6, 6, 9), (7, 9, 100), (8, 8, 1)]
    r = np.array([t[0] for t in up]); c = np.array([t[1] for t in up]); d = np.array([t[2] for t in up])
    off = r != c
    indptr, indices, counts = _csr_from_keys(n, np.r_[r, c[off]], np.r_[c, r[off]], np.r_[d, d[off]].astype(np.uint32))
    mask = np.zeros(n, dtype=bool)
    mask[[0, 2, 4]] = True
    sites = np.array([3, 0, 5, 2, 1, 1, 4, 0, 2, 2], dtype=np.int32)
    x = 10.0 ** np.linspace(-3, 3, n)
    m = dict(n=n, indptr=indptr, indices=indices, counts=counts, sites=sites, x=x)
    m['normed'] = ref_site_norm(indptr, indices, counts, sites)
    return m, mask


@pytest.mark.parametrize('fused', [False, True], ids=['staged', 'fused'])
def test_zero_edges_whole_matrix(dev, fused):
    """No kept entry at all: 0 edges, the accepted count, and scl = 1/0 = inf, as the reference computes it."""
    m, mask = _no_edge_matrix()
    wants = _compress_case(dev, m, [(0, m['n'])], mask, fused)
    assert wants[0]['n_edges'] == 0 and wants[0]['n_kept'] == 0 and wants[0]['n_accepted'] == 3
    assert np.isinf(ref_scale(wants[0]['vmax']))


@pytest.mark.parametrize('fused', [False, True], ids=['staged', 'fused'])
def test_zero_edges_block(dev, adv, fused):
    """A row block with no accepted row: 0 edges, and the global scale set through reduce_max."""
    mask = adv_mask(adv, 'none_in_block')
    wants = _compress_case(dev, adv, [(0, 1), (1, 334), (334, adv['n'])], mask, fused)
    assert wants[1]['n_edges'] == 0 and wants[1]['n_kept'] == 0


@pytest.mark.parametrize('fused', [False, True], ids=['staged', 'fused'])
def test_zero_edges_hotpath(dev, fused):
    """The whole path on a community whose accepted contigs pair only with contigs too short to be accepted."""
    from bin3c_b200 import synth
    from bin3c_b200.pipeline import HotPath
    n = 12
    lengths = np.where(np.arange(n) % 2 == 0, 5000, 500)            # odd contigs fall below min_len
    ti = np.repeat(np.arange(0, n, 2), 10)
    tj = ti + 1
    rec = synth.pack_pairs(ti, tj, np.ones(len(ti), dtype=bool))
    hp = HotPath(np.arange(n, dtype=np.int32), lengths, np.full(n, 3), min_len=1000, min_sig=5)
    for _ in range(2):                                              # a second run reuses the pool's buffers
        res = hp.run(dev.to_device(rec), fused=fused)
        assert res['n_accepted'] == n // 2 and res['n_edges'] == 0
        assert res['u'].numel() == res['v'].numel() == res['w'].numel() == 0
        assert np.isinf(_np(res['scl'])[0])
    out = hp.run(rec, fused=fused, to_host=True)
    assert out['n_edges'] == 0 and len(out['u']) == 0 and np.isinf(out['scl'])


# ---------------------------------------------------------------------------------------------
# C. KR tuning flags and SpMV layouts
# ---------------------------------------------------------------------------------------------

# 22 = slab-aligned CTA ranges (2) | single-word barrier (4) | peer hand-over of p.w as flagged words (16)
FLAG_SETS = [22, 0, 22 | 1, 22 | 8, 22 | 32, 22 | 96, 22 | 128, 22 & ~2, 22 & ~4, 255]
REL_TOL = 1e-9


def _relerr(a, b):
    return float(np.max(np.abs(a - b) / np.maximum(np.abs(b), 1e-300)))


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


def _side_list_counts():
    """The counts matrix of test_packed_count_stream_large_counts['few']: diagonal counts above 65535 and a handful of
    off-diagonal ones (the packed stream's side list), zero diagonals and zero sites."""
    rng = np.random.default_rng(77)
    n = 3000
    up = sp.triu(sp.random(n, n, density=0.004, random_state=5, data_rvs=lambda k: rng.integers(1, 400, size=k)),
                 1).tolil()
    diag = rng.integers(0, 3000, size=n).astype(np.int64)
    diag[[3, 70, 71, 500, 2999]] = [65535, 65536, 65537, 4_000_000_000, 1_234_567]
    up[10, 2000] = 70000
    up[10, 2500] = 3_000_000_000
    up[11, 12] = 65536
    up[70, 71] = 131072
    up[0, 2999] = 65537
    up[40, 41] = 100000
    up = up.tocsr()
    diag[[40, 2000]] = 0
    m = (up + up.T + sp.diags(diag, dtype=np.int64)).tocsr()
    m.eliminate_zeros()
    m = m.astype(np.uint32)
    m.sort_indices()
    sites = rng.integers(0, 60, size=n).astype(np.int32)
    return m, sites


# operand form: (matrix kind, slab width, max slabs, count stream, expected slabs)
KR_FORMS = {
    'f64_slabs': ('f64', 1000, 16, None, 5),
    'f64_gather': ('f64', None, 0, None, 0),
    'counts2': ('counts', 1000, 16, 2, 3),
    'counts1': ('counts', 1000, 16, 1, 3),
    'counts0': ('counts', 1000, 16, 0, 3),
    'counts_gather': ('counts', None, 0, 2, 0),       # counts in the gather form: 32-bit counts, 8 B per entry
    'counts_s9': ('counts', 334, 16, 2, 9),
    'counts_s24': ('counts', 126, 48, 2, 24),         # beyond 12 slabs: the batched rounds of rows_q
}


@pytest.fixture(scope='module')
def kr_mats():
    """The two matrices and their oracle results, computed once."""
    from oracle import oracle
    m = _sym_matrix(5000, 30, seed=17)
    res = oracle.kr_scale_vector(m)
    c, sites = _side_list_counts()
    s1 = site_values(sites)
    norm = c.astype(np.float64).tocoo()
    norm.data = norm.data * (1.0 / (s1[norm.row] * s1[norm.col]))
    _, x_ref, it_ref = oracle.kr_biostochastic(norm.tocsr())
    return {'f64': (m, None, res.x, res.n_iter), 'counts': (c, sites, x_ref, it_ref)}


_KR_DEFAULT = {}


def _kr_run(dev, mats, form, flags):
    import torch
    kind, width, max_slabs, stream, _ = KR_FORMS[form]
    m, sites, _, _ = mats[kind]
    _set_options(dev, width=width, max_slabs=max_slabs, count_stream=stream, flags=flags)
    if kind == 'f64':
        x, info = dev.kr_scale_vector(dev.DeviceCSR.from_scipy(m))
    else:
        x, info = dev.kr_scale_vector(dev.DeviceCSR.from_scipy(m, np.uint32), sites=dev.to_device(sites, torch.int32))
    return _np(x).copy(), info


def _order_bits(form):
    """Flag bits that may move the fp64 summation order of this operand form (see test_kr_flags)."""
    kind, _, max_slabs, stream, _ = KR_FORMS[form]
    if max_slabs == 0:
        return 0                                     # gather form: 1, 2 and 128 act on the slab form only
    bits = 2 | 128
    if kind == 'f64' or stream == 0:
        bits |= 1                                    # bank order reorders the fp64 stream only (kr.cu, kr_prepare_t)
    return bits


@pytest.mark.parametrize('flags', FLAG_SETS, ids=['flags%d' % f for f in FLAG_SETS])
@pytest.mark.parametrize('form', list(KR_FORMS))
def test_kr_flags(dev, kr_mats, form, flags):
    """
    Every flag set on every operand form: n_iter equal to the oracle's, x within 1e-9, the same bits on a second run,
    the operand layout (slabs, stream bytes per entry) unchanged by the flags, and against the default flags (22):

    - bits 4 (barrier), 32 / 64 (L2 prefetch) change only synchronisation or prefetching: the same bits;
    - bit 8 (flagged partial words) carries the very partial every chunk would have stored, and reduce_parts adds the
      partials in chunk order either way: the same bits;
    - bit 2 (slab-aligned CTA ranges) moves the CTA range boundaries, so the (row, slab) segments that straddle them are
      stitched at other points (a different association of the row sum), and bits 1 and 128 reorder entries inside
      a piece: within 1e-12 where they apply (slab form; bit 1 only with an fp64 stream), the same bits elsewhere.
    """
    kind, _, _, _, slabs = KR_FORMS[form]
    _, _, x_ref, it_ref = kr_mats[kind]
    if form not in _KR_DEFAULT:
        _KR_DEFAULT[form] = _kr_run(dev, kr_mats, form, 22)
    x0, info0 = _KR_DEFAULT[form]
    x1, info1 = _kr_run(dev, kr_mats, form, flags)
    x2, _ = _kr_run(dev, kr_mats, form, flags)
    assert info1['slabs'] == info0['slabs'] == slabs
    assert info1['stream_bytes_per_entry'] == info0['stream_bytes_per_entry']
    assert info1['n_iter'] == it_ref
    assert _relerr(x1, x_ref) <= REL_TOL
    assert np.array_equal(x1, x2)
    if (flags ^ 22) & _order_bits(form):
        assert _relerr(x1, x0) <= 1e-12
    else:
        assert np.array_equal(x1, x0)


SLAB_SHAPES = [(None, None), (1000, 16), (334, 16), (126, 48), (None, 0)]
SPMV_CASES = [(1, 1), (5000, 3), (4097, 40), (3000, 900)]
_SPMV_REF = {}


def _spmv_case(n, nnz_row):
    """Values log-uniform in [1e-6, 1e6], mixed-sign u; the row sums in long double and their error bound."""
    key = (n, nnz_row)
    if key not in _SPMV_REF:
        rng = np.random.default_rng(n + nnz_row)
        m = sp.random(n, n, density=min(1.0, nnz_row / n), random_state=rng, format='csr',
                      data_rvs=lambda k: 10.0 ** rng.uniform(-6.0, 6.0, k))
        m.sort_indices()
        us = [rng.standard_normal(n) * 10.0 ** rng.uniform(-6.0, 6.0, n) for _ in range(2)]
        refs = []
        rows = row_of_entry(m.indptr)
        k = np.diff(m.indptr)
        for u in us:
            prod = m.data.astype(np.longdouble) * u[m.indices].astype(np.longdouble)
            y = np.zeros(n, dtype=np.longdouble)
            np.add.at(y, rows, prod)
            mag = np.zeros(n)
            np.add.at(mag, rows, np.abs(m.data * u[m.indices]))
            refs.append((y, 2.0 * k * np.finfo(np.float64).eps * mag))
        _SPMV_REF[key] = (m, us, refs)
    return _SPMV_REF[key]


def _spmv_check(y, ref):
    want, bound = ref
    err = np.abs(y.astype(np.longdouble) - want)
    bad = np.flatnonzero(err > bound)
    assert bad.size == 0, (bad[:5], y[bad[:5]], want[bad[:5]], bound[bad[:5]])


@pytest.mark.parametrize('flags', [0, 1, 128, 255], ids=['flags0', 'flags1', 'flags128', 'flags255'])
@pytest.mark.parametrize('shape', SLAB_SHAPES, ids=['default', 'w1000', 'w334', 'w126s48', 'gather'])
@pytest.mark.parametrize('n,nnz_row', SPMV_CASES)
def test_spmv_flags(dev, n, nnz_row, shape, flags):
    """Every row within 2 k_i eps sum_j |a_ij u_j| of the long-double row sum -- one dropped, duplicated or misplaced
    entry breaks it -- for a fresh operand and for a prepared one reused with another u."""
    import torch
    m, us, refs = _spmv_case(n, nnz_row)
    _set_options(dev, width=shape[0], max_slabs=shape[1], flags=flags)
    csr = dev.DeviceCSR.from_scipy(m)
    ws = torch.empty(dev.lib.b3c_kr_workspace_bytes(n, m.nnz), dtype=torch.uint8, device='cuda')
    _spmv_check(_np(dev.spmv(csr, dev.to_device(us[0]), ws=ws)), refs[0])
    _spmv_check(_np(dev.spmv(csr, dev.to_device(us[1]), ws=ws, prepared=True)), refs[1])
