"""
CPU tests of KR's operand references (tests/kr_operand_cases.py) and of the operand layout the library plans
(b3c_kr_plan, host-only): the long-double row sum against scipy and the oracle's zero-diagonal rule, the per-row bound
rejecting each kind of defect it is there to catch, the form rule at its density threshold, and the workspace queries
bounding every layout a row block can take.
"""
import ctypes

import numpy as np
import pytest
import scipy.sparse as sp

import kr_operand_cases as K

# b3c_set_option keys and their defaults: slab width, max slabs, count stream
DEFAULTS = ((1, K.SLAB_W_MAX), (2, K.SLAB_S_MAX), (5, 2))


@pytest.fixture(scope='module')
def lib():
    from bin3c_b200.csrc import build
    build.build()
    from bin3c_b200 import _cabi
    return _cabi.lib


@pytest.fixture
def opts(lib):
    def set_(width=None, max_slabs=None, count_stream=None):
        for key, val in ((1, width), (2, max_slabs), (5, count_stream)):
            if val is not None:
                assert lib.b3c_set_option(key, int(val)) == 0
    yield set_
    for key, val in DEFAULTS:
        assert lib.b3c_set_option(key, val) == 0


def plan(lib, n, nnz, rows, counts):
    out = (ctypes.c_int64 * 5)()
    assert lib.b3c_kr_plan(n, nnz, rows, counts, out) == 0
    return tuple(int(x) for x in out)


# ---------------------------------------------------------------------------------------------
# the reference row sum and its bound
# ---------------------------------------------------------------------------------------------

def _case(seed=3, n=700):
    upper = [(5, 9, 65536), (5, 300, 2 ** 31), (17, 18, 2 ** 32 - 1), (40, 41, 65537)]
    indptr, indices, counts = K.symmetric_counts(n, 12, seed, upper=upper,
                                                 diag={7: 0, 40: 0, 17: 4_000_000_000, 9: 65536})
    return indptr, indices, counts, K.sites_for(n, seed), K.mixed_v(n, seed + 1)


def test_reference_matches_scipy_and_the_oracle_zero_diagonal_rule():
    """The site-normalised matrix times v (scipy) plus v_r on the rows the oracle's working matrix gets a 1 on the
    diagonal (oracle.kr_scale_vector, Q2); zero sites read as one; the fp64 form of the same reference agrees."""
    from oracle import oracle
    indptr, indices, counts, sites, v = _case()
    n = len(indptr) - 1
    s = K.site_values(sites)
    norm = sp.csr_matrix((counts.astype(np.float64), indices, indptr), shape=(n, n)).tocoo()
    norm.data = norm.data / (s[norm.row] * s[norm.col])
    norm = norm.tocsr()
    a = sp.csr_matrix(norm, copy=True)
    zero_d = a.diagonal() == 0                        # the oracle's rule, as it builds its working matrix
    assert zero_d[[7, 40]].all() and zero_d.sum() > 2
    work = (a + sp.diags(zero_d.astype(np.float64))).tocsr()
    want = work @ v
    q, mag, k = K.ref_rowsum(indptr, indices, counts, v, sites=sites)
    assert np.all(np.abs(q.astype(np.float64) - want) <= 1e-12 * mag)
    qf, magf, _ = K.ref_rowsum(indptr, indices, norm.data, v)
    assert np.all(np.abs(qf - q) <= 1e-13 * mag)
    # k counts the side-list terms of the large off-diagonal counts on both rows that hold them
    assert k[5] == np.diff(indptr)[5] + 2 and k[300] == np.diff(indptr)[300] + 1 and k[17] == np.diff(indptr)[17] + 1


def test_reference_of_a_row_block():
    """A row block (local indptr, global columns) gives the whole matrix's rows."""
    indptr, indices, counts, sites, v = _case(seed=4, n=3000)
    q, mag, k = K.ref_rowsum(indptr, indices, counts, v, sites=sites)
    lo, hi = 1024, 2048
    a, b = indptr[lo], indptr[hi]
    qb, magb, kb = K.ref_rowsum(indptr[lo:hi + 1] - a, indices[a:b], counts[a:b], v, row_lo=lo, sites=sites)
    assert np.array_equal(qb, q[lo:hi]) and np.array_equal(magb, mag[lo:hi]) and np.array_equal(kb, k[lo:hi])


def _fp64_rowsum(indptr, indices, counts, sites, v, drop=None, dup=None, lost=None, no_dfix=False):
    """The counts form's row sums in fp64, in the kernel's steps (us = v * inv_s, products, sums, * inv_s_r, + dfix),
    optionally with one defect: entry `drop` left out, entry `dup` added twice, entry `lost` 65536 short, or the
    packed diagonal's high part / the zero-diagonal one left out."""
    n = len(indptr) - 1
    inv = 1.0 / K.site_values(sites)
    us = v * inv
    lr = K.row_of_entry(indptr)
    c = counts.astype(np.float64).copy()
    if lost is not None:
        c[lost] -= 65536.0
    t = c * us[indices]
    if drop is not None:
        t[drop] = 0.0
    q = np.zeros(n)
    np.add.at(q, lr, t)
    if dup is not None:
        q[lr[dup]] += t[dup]
    q *= inv
    on = indices == lr
    diag = np.zeros(n)
    np.add.at(diag, lr[on], counts[on].astype(np.float64))
    dfix = np.where(diag == 0, 1.0, 0.0)
    if no_dfix:
        dfix[:] = 0.0
    return q + dfix * v


def test_bound_accepts_rounding_and_rejects_each_defect():
    """The fp64 sums pass the bound on every row; each defect is caught on the row that carries it: the entry with the
    largest |a_rj v_j| dropped or duplicated, a count of 2^32 - 1 that lost 65536, a zero diagonal's term left out, and
    the high part of a large diagonal count left out (the kernel's dfix, modelled here as the diagonal entry losing it)."""
    indptr, indices, counts, sites, v = _case()
    ref = K.ref_rowsum(indptr, indices, counts, v, sites=sites)
    assert K.bad_rows(_fp64_rowsum(indptr, indices, counts, sites, v), ref).size == 0
    lr = K.row_of_entry(indptr)
    s = K.site_values(sites)
    term = np.abs(counts / (s[lr] * s[indices]) * v[indices])
    for r in (0, 5, 17, 40, 699):
        e = indptr[r] + int(np.argmax(term[indptr[r]:indptr[r + 1]]))
        assert r in K.bad_rows(_fp64_rowsum(indptr, indices, counts, sites, v, drop=e), ref)
        assert r in K.bad_rows(_fp64_rowsum(indptr, indices, counts, sites, v, dup=e), ref)
    e = indptr[17] + int(np.flatnonzero(indices[indptr[17]:indptr[18]] == 18)[0])
    assert counts[e] == 2 ** 32 - 1
    assert 17 in K.bad_rows(_fp64_rowsum(indptr, indices, counts, sites, v, lost=e), ref)
    bad = K.bad_rows(_fp64_rowsum(indptr, indices, counts, sites, v, no_dfix=True), ref)
    assert {7, 40} <= set(bad.tolist())
    d17 = indptr[17] + int(np.flatnonzero(indices[indptr[17]:indptr[18]] == 17)[0])
    lo16 = counts.copy()
    lo16[d17] &= 0xffff
    assert 17 in K.bad_rows(_fp64_rowsum(indptr, indices, lo16, sites, v), ref)


# ---------------------------------------------------------------------------------------------
# b3c_kr_plan: the form rule and the workspace queries
# ---------------------------------------------------------------------------------------------

# (n, slab width): 35 slabs of 126 columns, and the default width at 1M rows (35 slabs)
WIDE = [(4396, 126), (5000, 126), (1_000_000, K.SLAB_W_MAX)]


@pytest.mark.parametrize('n,width', WIDE)
@pytest.mark.parametrize('packed', [True, False], ids=['packed', 'fp64'])
def test_plan_follows_the_density_rule_at_its_threshold(lib, opts, n, width, packed):
    """b3c_kr_plan against the transcription of the rule at dense * rows * S - 1 and dense * rows * S (rows rounded up
    to whole chunks), for the whole matrix and for blocks of 1, 300, 1024, 1025 and 2048 rows; the slab form flips
    exactly there.  Packed counts ask for form 2 in the slab form and 1 in the gather form; fp64 for 0."""
    opts(width=width)
    dense = K.DENSE_PACKED if packed else K.DENSE
    S = -(-n // width)
    for rows in (n, 1, 300, 1024, 1025, 2048):
        thr = dense * K.align_up(rows, K.CHUNK) * S
        for nnz in (thr - 1, thr):
            got = plan(lib, n, nnz, rows, 1 if packed else 0)
            want = K.form_rule(n, nnz, rows, packed, width=width)
            assert got[:3] == want, (rows, nnz, got, want)
            assert got[3] == ((2 if want[0] else 1) if packed else 0)
            assert (got[0] > 0) == (nnz == thr)
    opts(count_stream=1)
    assert plan(lib, n, thr, n, 1)[3] == 1
    opts(count_stream=0)
    assert plan(lib, n, thr, n, 1)[3] == 0


def test_plan_below_the_slab_cap_and_with_the_cap_lowered(lib, opts):
    """Within 16 slabs the slab form always; max slabs 0 forces the gather form whatever the density; 48 slabs is
    the widest the dense rule keeps, 49 never."""
    assert plan(lib, 100_000, 10, 100_000, 1)[:3] == (4, 4, 25000)
    opts(max_slabs=0)
    assert plan(lib, 100_000, 10 ** 9, 100_000, 1)[:3] == (0, 1, 100_000)
    opts(max_slabs=16, width=100)
    assert plan(lib, 4800, 10 ** 8, 4800, 1)[0] == 48
    assert plan(lib, 4801, 10 ** 8, 4801, 1)[0] == 0


@pytest.mark.parametrize('n,width,nnzs', [
    (4396, 126, [0, 20000, 42000, 60000, 143359, 143360, 300000]),
    (5000, 126, [50000, 143359, 600000]),
    (600_000, K.SLAB_W_MAX, [30000, 50000, 80000, 3_000_000]),
])
def test_every_block_fits_the_workspace_queries(lib, opts, n, width, nnzs):
    """For every row count 1 .. n -- tail blocks under 1024 rows included -- and both stream kinds the layout fits
    b3c_krp_workspace_bytes(n, nnz), and the whole matrix fits b3c_kr_workspace_bytes(n, nnz).  (Counting a tail
    block's own rows in the density rule let a 300-row block take the slab form where b3c_krp_workspace_bytes had
    sized the gather form: 10.9 MB against 1.8 MB at n = 4396, width 126.)"""
    opts(width=width)
    step = 1 if n < 10000 else 97
    for nnz in nnzs:
        krp = lib.b3c_krp_workspace_bytes(n, nnz)
        kr = lib.b3c_kr_workspace_bytes(n, nnz)
        for counts in (0, 1):
            assert plan(lib, n, nnz, n, counts)[4] <= kr
            for rows in list(range(1, n + 1, step)) + [n - n % K.CHUNK or n, n]:
                got = plan(lib, n, nnz, rows, counts)
                assert got[4] <= krp, (nnz, rows, counts, got, krp)


# C2, C3, C4 (the KR matrix of each bench config: n and stored entries of the last recorded bench lines) and the C5
# SpMV points; then the forms they take, as the rule stood before tail blocks were rounded up to whole chunks
BENCH = {'C2': (50_000, 9_305_590), 'C3': (250_000, 73_407_779), 'C4': (1_000_000, 210_581_950),
         'C5a': (250_000, 83_000_000), 'C5b': (1_000_000, 93_000_000), 'C5c': (1_000_000, 251_000_000),
         'C5d': (3_000_000, 300_000_000)}


def _old_rule(n, nnz, rows, packed):
    s_need = -(-n // K.SLAB_W_MAX)
    dense = K.DENSE_PACKED if packed else K.DENSE
    slab = s_need <= K.SLAB_S_MAX or (s_need <= K.SLAB_S_CAP and nnz >= dense * rows * s_need)
    return s_need if slab else 0


@pytest.mark.parametrize('name', list(BENCH))
def test_bench_forms_unchanged(lib, name):
    """The forms of the bench configs' whole matrices and of their 1024-aligned row blocks (2, 4 and 8 ranks) are
    those the rule chose before it rounded the block's rows up to whole chunks; C3 keeps 9 slabs and C4 35."""
    n, nnz = BENCH[name]
    for counts in (0, 1):
        got = plan(lib, n, nnz, n, counts)
        assert got[0] == _old_rule(n, nnz, n, counts == 1)
        for g in (2, 4, 8):
            n_chunks = -(-n // K.CHUNK)
            for r in range(g):
                lo, hi = n_chunks * r // g * K.CHUNK, min(n, n_chunks * (r + 1) // g * K.CHUNK)
                if hi - lo < K.CHUNK or hi % K.CHUNK:
                    continue
                nl = int(nnz * (hi - lo) / n)
                assert plan(lib, n, nl, hi - lo, counts)[0] == _old_rule(n, nl, hi - lo, counts == 1)
    if name == 'C3':
        assert plan(lib, n, nnz, n, 1)[:2] == (9, 9)
    if name == 'C4':
        assert plan(lib, n, nnz, n, 1)[0] == 35


def test_plan_rejects_bad_arguments(lib):
    out = (ctypes.c_int64 * 5)()
    assert lib.b3c_kr_plan(100, 10, 0, 0, out) < 0
    assert lib.b3c_kr_plan(100, 10, 101, 0, out) < 0
    assert lib.b3c_kr_plan(0, 10, 1, 0, out) < 0
    assert lib.b3c_kr_plan(100, -1, 1, 0, out) < 0
    assert lib.b3c_kr_plan(100, 10, 1, 0, None) < 0
