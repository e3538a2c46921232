"""
The row sums of KR's SpMV operand (csrc/kr.cu, rows_q) restated in np.longdouble, the per-row error bound the kernel
must meet, a transcription of the operand's form rule (kr_layout), and builders of controlled count matrices -- most
counts below 65536, large ones exactly where a case puts them.  Checked on the CPU by tests/test_kr_operand_refs.py and
used against the kernels by tests/test_gpu_kr_operand.py.
"""
import numpy as np

EPS = np.finfo(np.float64).eps
CHUNK = 1024                      # kr.cu: rows per reduction chunk (the stream lays out whole chunks of rows)
SLAB_W_MAX = 28672                # default slab width
SLAB_S_MAX = 16                   # default slab cap
SLAB_S_CAP = 48                   # the most slabs the dense-cell rule may keep
DENSE_PACKED, DENSE = 4, 6        # SLAB_DENSE_CELL_PACKED, SLAB_DENSE_CELL
BIG_CAP = 4096                    # side list of off-diagonal counts above 65535
BOUND_C = 8


def site_values(sites):
    """Site counts as the normalisation reads them: zero read as one."""
    s = np.asarray(sites, dtype=np.float64).copy()
    s[s == 0] = 1.0
    return s


def align_up(a, b):
    return -(-int(a) // b) * b


def form_rule(n, nnz, rows, packed, width=SLAB_W_MAX, max_slabs=SLAB_S_MAX):
    """(slabs, S, W) of kr_layout: slabs = 0 for the gather form.  The slab form whenever n fits max_slabs slabs of
    `width` columns; a wider matrix of at most 48 slabs keeps it (at the default cap) when its (row, slab) cells -- the
    block's rows rounded up to whole 1024-row chunks, times S -- hold `dense` entries or more on average."""
    s_need = -(-int(n) // int(width))
    dense = DENSE_PACKED if packed else DENSE
    dense_cells = max_slabs >= SLAB_S_MAX and s_need <= SLAB_S_CAP and nnz >= dense * align_up(rows, CHUNK) * s_need
    if s_need <= max_slabs or dense_cells:
        return s_need, s_need, align_up(-(-int(n) // s_need), 2)
    return 0, 1, int(n)


def row_of_entry(indptr):
    return np.repeat(np.arange(len(indptr) - 1, dtype=np.int64), np.diff(indptr))


def ref_rowsum(indptr, indices, vals, v, row_lo=0, sites=None):
    """
    q_r = sum_j a_rj v_j + [a_rr == 0] v_r for the rows of the block (local indptr, global columns), in np.longdouble:
    a = vals (fp64 values), or, with `sites`, a_rj = c_rj / (s_r s_j) with zero sites read as one.  A missing or zero
    diagonal counts as one (Q2, sparse_utils.py:110-115).  Returns (q, mag, k):
    mag_r = sum_j |a_rj v_j| (plus |v_r| for the zero-diagonal term) and k_r = the row's stream entries plus its
    side-list terms (off-diagonal counts above 65535 are summed twice, as a low and a high part).
    """
    nl = len(indptr) - 1
    lr = row_of_entry(indptr)
    gr = lr + row_lo
    v = np.asarray(v, dtype=np.float64)
    vl = v.astype(np.longdouble)
    if sites is None:
        a = np.asarray(vals, dtype=np.float64).astype(np.longdouble)
        big = np.zeros(len(indices), dtype=bool)
    else:
        s = site_values(sites).astype(np.longdouble)
        c = np.asarray(vals, dtype=np.uint32)
        a = c.astype(np.longdouble) / (s[gr] * s[indices])
        big = (c > 0xffff) & (indices != gr)
    t = a * vl[indices]
    q = np.zeros(nl, dtype=np.longdouble)
    np.add.at(q, lr, t)
    mag = np.zeros(nl, dtype=np.longdouble)
    np.add.at(mag, lr, np.abs(t))
    diag = np.zeros(nl, dtype=np.longdouble)
    on = indices == gr
    np.add.at(diag, lr[on], a[on])
    zero = diag == 0
    rows = np.arange(nl) + row_lo
    q[zero] += vl[rows[zero]]
    mag[zero] += np.abs(vl[rows[zero]])
    k = np.diff(indptr) + np.bincount(lr[big], minlength=nl)
    return q, mag.astype(np.float64), k


def row_bound(mag, k, c=BOUND_C):
    """
    |q_r - fl(q_r)| <= (2 k_r + c) eps mag_r.  Counting the roundings a term meets on its way into the counts form's
    row sum fl(fl(fl(sum_j c_rj us_j + sum_big hi_rj us_j) * fl(1 / s_r)) + fl(dfix_r v_r)):
    - fl(1 / s_j) and us_j = fl(v_j * inv_s_j): 2;
    - the product c_rj * us_j (or hi_rj * us_j): 1;
    - the sums: a row of k_r stream and side-list terms (zero padding adds exactly) goes through at most k_r - 1 adds
      whatever their association -- piece trees, segment stitching, the slab-order adds of rows_q;
    - the final * fl(1 / s_r): 2;
    - the dfix term: dfix = fl(fl(hi_rr * inv_s_r) * inv_s_r) is 4 roundings (exact 1 for a zero diagonal), its
      product with v_r 1, and the add into the row sum 1: 6.
    So a stream term meets at most k_r + 5 roundings and the dfix term 6: the error is at most gamma_{k_r + 6} mag_r,
    which (2 k_r + 8) eps mag_r covers with room to spare (the fp64 form meets fewer: k_r + 1).  One dropped, doubled or
    misplaced entry, a count that lost 65536 or a missing dfix term moves the sum by a whole term instead.
    """
    return (2.0 * np.asarray(k, dtype=np.float64) + c) * EPS * mag


def bad_rows(q, ref):
    """Local rows whose q is outside the bound around the reference (NaN counts as outside)."""
    want, mag, k = ref
    err = np.abs(np.asarray(q, dtype=np.float64).astype(np.longdouble) - want)
    return np.flatnonzero(~(err <= row_bound(mag, k)))


def csr_from_keys(n_rows, row, col, data):
    """CSR (indptr int64, indices int32, data) of unique (local row, column) keys, columns sorted."""
    o = np.lexsort((col, row))
    indptr = np.zeros(n_rows + 1, dtype=np.int64)
    np.cumsum(np.bincount(row, minlength=n_rows), out=indptr[1:])
    return indptr, np.asarray(col)[o].astype(np.int32), np.asarray(data)[o]


def small_counts(rng, k, hi=60000):
    """Counts 1 .. hi, log-uniform: they fit the packed stream's 16 bits."""
    return np.clip(np.floor(2.0 ** rng.uniform(0.0, np.log2(hi), k)), 1, hi).astype(np.uint32)


def random_block(n, rows, nnz, seed, row_lo=0, entries=(), empty_rows=(), diag_frac=0.8):
    """
    Rows [row_lo, row_lo + rows) of an n-column count matrix (not symmetric: the row sums do not need it) with exactly
    `nnz` entries: random columns with small counts, most rows holding their diagonal.  `entries` = (global row, column,
    count) placed on top (replacing a random entry, so nnz stays exact); `empty_rows` (global) hold nothing.
    """
    rng = np.random.default_rng(seed)
    fixed = {(int(r) - row_lo, int(c)): int(x) for r, c, x in entries}
    empty = np.array(sorted(int(r) - row_lo for r in empty_rows), dtype=np.int64)
    ok_rows = np.setdiff1d(np.arange(rows), empty)
    want = nnz - len(fixed)
    assert 0 <= want <= len(ok_rows) * n - len(fixed)
    keys = set(r * n + c for r, c in fixed)
    dg = ok_rows[rng.random(len(ok_rows)) < diag_frac]
    dkeys = [int(r) * n + int(r) + row_lo for r in dg if int(r) * n + int(r) + row_lo not in keys][:want]
    keys.update(dkeys)
    pool = ok_rows[rng.integers(0, len(ok_rows), 2 * (want + 16))] * n + rng.integers(0, n, 2 * (want + 16))
    for kk in pool:
        if len(keys) >= nnz:
            break
        keys.add(int(kk))
    while len(keys) < nnz:                        # dense corner cases: fill up deterministically
        r = int(ok_rows[rng.integers(0, len(ok_rows))])
        keys.add(r * n + int(rng.integers(0, n)))
    key = np.array(sorted(keys), dtype=np.int64)
    assert len(key) == nnz
    row, col = key // n, key % n
    cnt = small_counts(rng, len(key))
    for (r, c), x in fixed.items():
        cnt[np.searchsorted(key, r * n + c)] = x
    indptr, indices, counts = csr_from_keys(rows, row, col, cnt)
    return indptr, indices, counts.astype(np.uint32)


def symmetric_counts(n, nnz_row, seed, upper=(), diag=None):
    """Symmetric n x n counts: ~nnz_row entries per row with small counts, `upper` = (r, c, count) with r < c placed
    (and mirrored), diag = {row: count} (0 removes the diagonal).  Returns (indptr, indices, counts)."""
    rng = np.random.default_rng(seed)
    k = n * nnz_row // 2
    a, b = rng.integers(0, n, k), rng.integers(0, n, k)
    keep = a != b
    key = set((np.minimum(a, b)[keep].astype(np.int64) * n + np.maximum(a, b)[keep]).tolist())
    vals = {kk: int(x) for kk, x in zip(sorted(key), small_counts(rng, len(key)))}
    for r, c, x in upper:
        assert r < c
        vals[int(r) * n + int(c)] = int(x)
    d = {int(r): int(x) for r, x in zip(np.flatnonzero(rng.random(n) < 0.9), small_counts(rng, n))}
    d.update(diag or {})
    up = np.array(sorted(vals), dtype=np.int64)
    uv = np.array([vals[kk] for kk in up.tolist()], dtype=np.int64)
    dr = np.array(sorted(r for r, x in d.items() if x), dtype=np.int64)
    dv = np.array([d[r] for r in dr.tolist()], dtype=np.int64)
    ur, uc = up // n, up % n
    row = np.r_[ur, uc, dr]
    col = np.r_[uc, ur, dr]
    return csr_from_keys(n, row, col, np.r_[uv, uv, dv].astype(np.uint32))


def mixed_v(n, seed):
    """Operand of mixed sign, magnitudes log-uniform over 1e-6 .. 1e6."""
    rng = np.random.default_rng(seed)
    return rng.choice([-1.0, 1.0], n) * 10.0 ** rng.uniform(-6.0, 6.0, n)


def sites_for(n, seed):
    """Site counts with zeros (read as one), ones and 2^20 among ordinary values."""
    rng = np.random.default_rng(seed)
    s = rng.integers(2, 60, n).astype(np.int32)
    s[rng.random(n) < 0.1] = 0
    s[rng.random(n) < 0.05] = 1
    s[rng.random(n) < 0.05] = 1 << 20
    return s
