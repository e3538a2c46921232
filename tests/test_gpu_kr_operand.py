"""
KR's SpMV operand against the long-double row sums of tests/kr_operand_cases.py (-m gpu), through b3c_kr_rowsum: the
operand built exactly as b3c_kr_run* / b3c_kr_run_peer* build it, multiplied by the SpMV kernel of its form, and the row
sums rows_q hands to the iteration -- segment sums in rounds of 4 or 12 slabs, the side list of off-diagonal counts
above 65535, the row's 1 / s_i, the zero-diagonal term and the high part of a packed diagonal count.

Every case checks every local row against the bound (2 k_r + 8) eps sum_j |a_rj v_j|, with v taken as the CG operand
u and as x of a residual (different v each, so that one read in place of the other fails), the form reported against
b3c_kr_plan, and the same bits on a second call.
"""
import ctypes

import numpy as np
import pytest

import kr_operand_cases as K

pytestmark = pytest.mark.gpu

# b3c_set_option keys and their defaults: slab width, max slabs, KR flags, count stream
DEFAULT_OPTIONS = ((1, 28672), (2, 16), (3, 22), (5, 2))


@pytest.fixture(scope='module')
def dev():
    import torch
    if not torch.cuda.is_available():
        pytest.skip('no CUDA device')
    from bin3c_b200 import device
    return device


@pytest.fixture(autouse=True)
def _restore_options():
    yield
    import sys
    cabi = sys.modules.get('bin3c_b200._cabi')
    if cabi is not None:
        for key, value in DEFAULT_OPTIONS:
            cabi.check(cabi.lib.b3c_set_option(key, value))


def _opts(dev, width=None, max_slabs=None, count_stream=None):
    for key, val in ((1, width), (2, max_slabs), (5, count_stream)):
        if val is not None:
            dev.check(dev.lib.b3c_set_option(key, int(val)))


def _plan(dev, n, nnz, rows, counts):
    out = (ctypes.c_int64 * 5)()
    dev.check(dev.lib.b3c_kr_plan(n, nnz, rows, counts, out))
    return [int(x) for x in out]


def _dev(dev, a, dtype):
    import torch
    a = np.ascontiguousarray(a)
    if len(a) == 0:                                    # a real pointer for an empty block
        a = np.zeros(1, dtype=a.dtype)
    return dev.to_device(a.view(np.int32) if a.dtype == np.uint32 else a, dtype)


def rowsum(dev, n, indptr, indices, vals, v, row_lo=0, sites=None, which=0, ws_bytes=None):
    """b3c_kr_rowsum of rows [row_lo, row_lo + len(indptr) - 1): returns (rc, q, h_info)."""
    import torch
    rows = len(indptr) - 1
    nnz = len(indices)
    whole = row_lo == 0 and rows == n
    if ws_bytes is None:
        ws_bytes = dev.lib.b3c_kr_workspace_bytes(n, nnz) if whole else dev.lib.b3c_krp_workspace_bytes(n, nnz)
    ws = torch.empty(int(ws_bytes), dtype=torch.uint8, device='cuda')
    d_indptr = _dev(dev, np.asarray(indptr, dtype=np.int64), torch.int64)
    d_idx = _dev(dev, np.asarray(indices, dtype=np.int32), torch.int32)
    if sites is None:
        d_data, d_counts, d_sites = _dev(dev, np.asarray(vals, dtype=np.float64), torch.float64), None, None
    else:
        d_data = None
        d_counts = _dev(dev, np.asarray(vals, dtype=np.uint32), torch.int32)
        d_sites = dev.to_device(np.asarray(sites, dtype=np.int32), torch.int32)
    d_v = dev.to_device(np.asarray(v, dtype=np.float64))
    q = torch.full((rows,), float('nan'), dtype=torch.float64, device='cuda')
    info = (ctypes.c_int64 * 8)()
    p = dev._ptr
    rc = dev.lib.b3c_kr_rowsum(n, row_lo, row_lo + rows, nnz, p(d_indptr), p(d_idx), p(d_data), p(d_counts),
                               p(d_sites), which, p(d_v), p(q), p(ws), int(ws_bytes), info, dev._stream())
    torch.cuda.synchronize()
    return rc, q.cpu().numpy().copy(), [int(x) for x in info]


def check_case(dev, n, indptr, indices, vals, row_lo=0, sites=None, ws_bytes=None, bytes_per_entry=None, seed=1):
    """Both operands, every local row within the bound, the form of b3c_kr_plan, the same bits twice."""
    rows = len(indptr) - 1
    counts = sites is not None
    plan = _plan(dev, n, len(indices), rows, 1 if counts else 0)
    infos = []
    for which in (0, 1):
        v = K.mixed_v(n, seed + 17 * which)
        ref = K.ref_rowsum(indptr, indices, vals, v, row_lo=row_lo, sites=sites)
        rc, q, info = rowsum(dev, n, indptr, indices, vals, v, row_lo, sites, which, ws_bytes)
        dev.check(rc)
        bad = K.bad_rows(q, ref)
        assert bad.size == 0, ('which', which, 'rows', bad[:8] + row_lo, q[bad[:8]], ref[0][bad[:8]])
        rc2, q2, info2 = rowsum(dev, n, indptr, indices, vals, v, row_lo, sites, which, ws_bytes)
        dev.check(rc2)
        assert np.array_equal(q.view(np.int64), q2.view(np.int64)) and info2 == info
        infos.append(info)
    info = infos[0]
    assert infos[1] == info
    assert info[0] == plan[0] and info[1] == plan[1] and info[7] == plan[4], (info, plan)
    slab = plan[0] > 0
    natural = {0: 10 if slab else 12, 1: 6 if slab else 8, 2: 4}[plan[3]]
    assert info[2] == (bytes_per_entry or natural), (info, plan)
    assert info[5] <= info[4] and info[4] % 2048 == 0
    return info


def _normed(indptr, indices, counts, sites, row_lo=0):
    s = K.site_values(sites)
    gr = K.row_of_entry(indptr) + row_lo
    return counts.astype(np.float64) * (1.0 / (s[gr] * s[indices]))


def _block(indptr, indices, vals, lo, hi):
    a, b = int(indptr[lo]), int(indptr[hi])
    return indptr[lo:hi + 1] - a, indices[a:b], vals[a:b]


# ---------------------------------------------------------------------------------------------
# forms of a whole matrix
# ---------------------------------------------------------------------------------------------

N_FORMS = 5000
# (slab width, max slabs) for S = 1, 3, 9, 40 slabs and the gather form at n = 5000
SHAPES = {'s1': (None, None, 1), 's3': (1668, None, 3), 's9': (560, None, 9), 's40': (126, 48, 40), 'gather': (None, 0, 0)}


@pytest.fixture(scope='module')
def forms_matrix():
    upper = [(0, 4999, 65536), (1, 2, 2 ** 31), (1023, 1024, 2 ** 32 - 1), (700, 2500, 65537), (3000, 3001, 70000)]
    indptr, indices, counts = K.symmetric_counts(N_FORMS, 30, 21, upper=upper,
                                                 diag={5: 0, 1023: 0, 1: 65536, 4999: 4_000_000_000, 6: 65535})
    sites = K.sites_for(N_FORMS, 21)
    return indptr, indices, counts, sites


FORMS = [(kind, shape) for kind in ('f64', 'packed') for shape in SHAPES] + \
        [('counts32', 's9'), ('counts32', 'gather'), ('counts0', 's9'), ('counts0', 's40')]


@pytest.mark.parametrize('kind,shape', FORMS, ids=['%s-%s' % f for f in FORMS])
def test_forms_whole_matrix(dev, forms_matrix, kind, shape):
    """fp64 values and packed counts at S = 1, 3, 9, 40 and in the gather form, 32-bit counts in the slab and the
    gather form (6 and 8 B per entry), and counts with the fp64 stream (B3C_OPT_KR_COUNT_STREAM = 0).  Packed counts in
    the gather form are 32-bit counts: the packed stream needs the 16-bit slab columns."""
    indptr, indices, counts, sites = forms_matrix
    width, max_slabs, S = SHAPES[shape]
    _opts(dev, width=width, max_slabs=max_slabs, count_stream={'packed': 2, 'counts32': 1, 'counts0': 0}.get(kind))
    if kind == 'f64':
        info = check_case(dev, N_FORMS, indptr, indices, _normed(indptr, indices, counts, sites))
    else:
        info = check_case(dev, N_FORMS, indptr, indices, counts, sites=sites)
    assert info[0] == S
    gr = K.row_of_entry(indptr)
    diag = np.zeros(N_FORMS)
    np.add.at(diag, gr[indices == gr], counts[indices == gr].astype(np.float64))
    assert info[6] == np.count_nonzero(diag == 0) and diag[5] == diag[1023] == 0
    if kind == 'packed' and S:
        assert info[3] == np.count_nonzero((counts > 0xffff) & (indices != gr)) == 10


@pytest.mark.parametrize('shape', list(SHAPES))
def test_fp64_rows_equal_spmv_bitwise(dev, forms_matrix, shape):
    """fp64 form: where the diagonal is stored, q is b3c_spmv's y bit for bit (the same segment sums added in slab
    order); on a zero-diagonal row q = fl(y + v_r)."""
    import torch
    indptr, indices, counts, sites = forms_matrix
    width, max_slabs, _ = SHAPES[shape]
    _opts(dev, width=width, max_slabs=max_slabs)
    vals = _normed(indptr, indices, counts, sites)
    v = K.mixed_v(N_FORMS, 5)
    rc, q, _ = rowsum(dev, N_FORMS, indptr, indices, vals, v, which=0)
    dev.check(rc)
    import scipy.sparse as sp
    csr = dev.DeviceCSR.from_scipy(sp.csr_matrix((vals, indices, indptr), shape=(N_FORMS, N_FORMS)))
    ws = torch.empty(dev.lib.b3c_kr_workspace_bytes(N_FORMS, len(indices)), dtype=torch.uint8, device='cuda')
    y = dev.spmv(csr, dev.to_device(v), ws=ws).cpu().numpy()
    d = sp.csr_matrix((vals, indices, indptr), shape=(N_FORMS, N_FORMS)).diagonal()
    z = d == 0
    assert z[5] and z[1023] and not z.all()
    assert np.array_equal(q[~z].view(np.int64), y[~z].view(np.int64))
    assert np.array_equal(q[z].view(np.int64), (y[z] + v[z]).view(np.int64))


@pytest.mark.parametrize('shape', ['s3', 's40', 'gather'])
def test_counts_fp64_stream_equals_fp64_hook_on_site_norm(dev, forms_matrix, shape):
    """B3C_OPT_KR_COUNT_STREAM = 0 streams c_ij / (s_i s_j) as fp64: its row sums are those of the fp64 operand of
    b3c_site_norm's output, bit for bit, for both operands."""
    indptr, indices, counts, sites = forms_matrix
    width, max_slabs, _ = SHAPES[shape]
    _opts(dev, width=width, max_slabs=max_slabs, count_stream=0)
    import torch
    import scipy.sparse as sp
    csr = dev.DeviceCSR.from_scipy(sp.csr_matrix((counts, indices, indptr), shape=(N_FORMS, N_FORMS)), np.uint32)
    normed = dev.site_norm(csr, dev.to_device(sites, torch.int32)).data.cpu().numpy()
    for which in (0, 1):
        v = K.mixed_v(N_FORMS, 9 + which)
        rc, qc, ic = rowsum(dev, N_FORMS, indptr, indices, counts, v, sites=sites, which=which)
        dev.check(rc)
        rc, qf, i_f = rowsum(dev, N_FORMS, indptr, indices, normed, v, which=which)
        dev.check(rc)
        assert ic[2] == i_f[2] and np.array_equal(qc.view(np.int64), qf.view(np.int64))


# ---------------------------------------------------------------------------------------------
# the density switch of a 35-slab matrix
# ---------------------------------------------------------------------------------------------

N_WIDE = 4396                     # 35 slabs of 126 columns


@pytest.mark.parametrize('packed', [True, False], ids=['packed', 'fp64'])
@pytest.mark.parametrize('block', [(0, N_WIDE), (1024, 2048)], ids=['whole', 'block'])
@pytest.mark.parametrize('below', [0, 1], ids=['at', 'below'])
def test_density_switch(dev, packed, block, below):
    """nnz exactly at dense * rows * S and one entry below it: the slab form (35 slabs) at the threshold, the gather
    form below, for the whole matrix (rows rounded up to 5120) and a 1024-row block."""
    _opts(dev, width=126)
    lo, hi = block
    dense = K.DENSE_PACKED if packed else K.DENSE
    nnz = dense * K.align_up(hi - lo, K.CHUNK) * 35 - below
    indptr, indices, counts = K.random_block(N_WIDE, hi - lo, nnz, 31 + lo, row_lo=lo)
    sites = K.sites_for(N_WIDE, 31)
    if packed:
        info = check_case(dev, N_WIDE, indptr, indices, counts, row_lo=lo, sites=sites)
    else:
        info = check_case(dev, N_WIDE, indptr, indices, _normed(indptr, indices, counts, sites, lo), row_lo=lo)
    assert info[0] == (0 if below else 35)


# ---------------------------------------------------------------------------------------------
# the side list
# ---------------------------------------------------------------------------------------------

SPECIAL = [65536, 65537, 2 ** 31, 2 ** 32 - 1]         # off-diagonal counts that go to the side list


def _big_entries(n, rows, row_lo, k, seed, width):
    """k large off-diagonal counts in rows [row_lo, row_lo + rows): the special values first, on the first and last
    rows of the block, the last row of a chunk and rows 0 / n - 1, at columns that open or close a cell (0, W - 1, W,
    n - 1) and at random places."""
    rng = np.random.default_rng(seed)
    pick_rows = [row_lo, row_lo + rows - 1, row_lo + min(rows, K.CHUNK) - 1, 0, n - 1]
    pick_cols = [0, width - 1, width, n - 1, 7, 8]
    out, seen = [], set()
    i = 0
    while len(out) < k:
        if i < 60:
            r = pick_rows[i % len(pick_rows)]
            c = pick_cols[(i // len(pick_rows)) % len(pick_cols)]
        else:
            r, c = int(rng.integers(row_lo, row_lo + rows)), int(rng.integers(0, n))
        i += 1
        if not (row_lo <= r < row_lo + rows) or r == c or (r, c) in seen:
            continue
        seen.add((r, c))
        val = SPECIAL[len(out) % len(SPECIAL)] if len(out) < 40 else int(rng.integers(65536, 2 ** 32))
        out.append((r, c, val))
    return out


SIDE = {'none': (0, (0, 3000), 4), 'one': (1, (0, 3000), 4), 'cap': (4096, (0, 3000), 4),
        'cap_plus_block': (4097, (1024, 3000), 6)}


@pytest.mark.parametrize('case', list(SIDE))
def test_side_list_sizes(dev, case):
    """0, 1 and 4096 large off-diagonal counts keep the packed stream (n_big reported, 4 B per entry); 4097 in a block
    fall back to 32-bit counts (6 B, n_big = 0).  Rows with a zero diagonal, and with diagonal counts 65535 .. 2^32 - 1,
    among the rows that hold them."""
    k, (lo, hi), bpe = SIDE[case]
    n, width = 3000, 1000
    _opts(dev, width=width)
    ent = _big_entries(n, hi - lo, lo, k, 40 + k, width)
    diag_big = [(lo + 3, lo + 3, 65536), (lo + 4, lo + 4, 2 ** 32 - 1), (lo + 5, lo + 5, 65535), (hi - 1, hi - 1, 2 ** 31),
                (lo + 6, lo + 9, 65535)]
    indptr, indices, counts = K.random_block(n, hi - lo, 40000, 50 + k, row_lo=lo, entries=ent + diag_big)
    gr = K.row_of_entry(indptr) + lo
    n_big = int(np.count_nonzero((counts > 0xffff) & (indices != gr)))
    assert n_big == k
    dg = np.zeros(hi - lo)
    np.add.at(dg, gr[indices == gr] - lo, 1)
    if k > 1:
        assert (dg[np.array([r for r, c, x in ent]) - lo] == 0).any()   # listed rows with a zero diagonal among them
    info = check_case(dev, n, indptr, indices, counts, row_lo=lo, sites=K.sites_for(n, 3), bytes_per_entry=bpe)
    assert info[3] == (n_big if bpe == 4 else 0)
    if case == 'cap':
        assert n_big == 4096 and info[3] == 4096
    if case == 'cap_plus_block':
        assert n_big == 4097


def test_side_list_overflow_whole_symmetric(dev):
    """2049 large upper counts mirrored: 4098 side-list entries, one too many for the list -- the build falls back to
    32-bit counts (6 B per entry)."""
    n = 3000
    rng = np.random.default_rng(8)
    upper, seen = [], set()
    while len(upper) < 2049:
        r, c = sorted(int(x) for x in rng.integers(0, n, 2))
        if r < c and (r, c) not in seen:
            seen.add((r, c))
            upper.append((r, c, SPECIAL[len(upper) % 4] if len(upper) < 40 else int(rng.integers(65536, 2 ** 32))))
    indptr, indices, counts = K.symmetric_counts(n, 20, 8, upper=upper)
    gr = K.row_of_entry(indptr)
    assert np.count_nonzero((counts > 0xffff) & (indices != gr)) == 4098
    _opts(dev, width=1000)
    check_case(dev, n, indptr, indices, counts, sites=K.sites_for(n, 8), bytes_per_entry=6)


# ---------------------------------------------------------------------------------------------
# row blocks
# ---------------------------------------------------------------------------------------------

N_BLK = 5000
BLOCKS = {'first': (0, 1024), 'second': (1024, 2048), 'to_end': (3072, N_BLK), 'one_chunk': (3072, 4096),
          'tail': (4096, N_BLK)}
BLOCK_FORMS = {'f64': None, 'packed': 2, 'counts32': 1, 'counts_gather': 1}


@pytest.fixture(scope='module')
def blk_matrix():
    upper = [(0, 1, 2 ** 31), (1023, 1024, 65536), (2047, 4000, 2 ** 32 - 1), (3072, 3073, 65537), (4095, 4096, 70000),
             (4096, 4999, 100000)]
    indptr, indices, counts = K.symmetric_counts(N_BLK, 24, 12, upper=upper,
                                                 diag={0: 0, 1024: 0, 3072: 2 ** 32 - 1, 4999: 0, 4096: 65536})
    return indptr, indices, counts, K.sites_for(N_BLK, 12)


@pytest.mark.parametrize('form', list(BLOCK_FORMS))
@pytest.mark.parametrize('blk', list(BLOCKS))
def test_row_blocks(dev, blk_matrix, blk, form):
    """Row blocks as the peer-mode driver hands them over (local indptr, global columns): row_lo 0, 1024 and 3072,
    row_hi aligned or n, a one-chunk block and the 904-row tail, in every operand form, with a workspace of exactly
    b3c_krp_workspace_bytes."""
    indptr, indices, counts, sites = blk_matrix
    lo, hi = BLOCKS[blk]
    bi, bx, bc = _block(indptr, indices, counts, lo, hi)
    _opts(dev, width=1000, max_slabs=0 if form == 'counts_gather' else None, count_stream=BLOCK_FORMS[form])
    if form == 'f64':
        check_case(dev, N_BLK, bi, bx, _normed(bi, bx, bc, sites, lo), row_lo=lo)
    else:
        check_case(dev, N_BLK, bi, bx, bc, row_lo=lo, sites=sites)


@pytest.mark.parametrize('packed', [True, False], ids=['packed', 'fp64'])
def test_tail_block_fits_the_peer_workspace(dev, packed):
    """A 300-row tail block [4096, 4396) of a 35-slab matrix holding 60000 entries, run with exactly
    b3c_krp_workspace_bytes: it takes the form of a 1024-row block with the same entries (gather), for which the
    workspace was sized.  (Counting its own 300 rows, it took the slab form and the call failed with "KR workspace too
    small".)"""
    _opts(dev, width=126)
    lo, hi = 4096, N_WIDE
    indptr, indices, counts = K.random_block(N_WIDE, hi - lo, 60000, 77, row_lo=lo)
    sites = K.sites_for(N_WIDE, 77)
    ws = dev.lib.b3c_krp_workspace_bytes(N_WIDE, len(indices))
    if packed:
        info = check_case(dev, N_WIDE, indptr, indices, counts, row_lo=lo, sites=sites, ws_bytes=ws)
    else:
        info = check_case(dev, N_WIDE, indptr, indices, _normed(indptr, indices, counts, sites, lo), row_lo=lo,
                          ws_bytes=ws)
    assert info[0] == 0 and info[7] <= ws


@pytest.mark.parametrize('form', ['f64', 'packed'])
def test_empty_block_and_empty_rows(dev, form):
    """A block with no entries at all (every row's sum is its zero-diagonal term, v_r) and a block whose rows are
    partly empty, among them its first and last rows."""
    n, lo, hi = N_BLK, 1024, 3072
    _opts(dev, width=1000)
    sites = K.sites_for(n, 4)
    indptr = np.zeros(hi - lo + 1, dtype=np.int64)
    indices = np.zeros(0, dtype=np.int32)
    counts = np.zeros(0, dtype=np.uint32)
    empty = [lo, lo + 1, lo + 500, lo + 1023, lo + 1024, hi - 1] + list(range(lo + 1100, lo + 1400))
    bi, bx, bc = K.random_block(n, hi - lo, 30000, 4, row_lo=lo, empty_rows=empty)
    for ip, ix, ic in ((indptr, indices, counts), (bi, bx, bc)):
        if form == 'f64':
            info = check_case(dev, n, ip, ix, _normed(ip, ix, ic, sites, lo), row_lo=lo)
        else:
            info = check_case(dev, n, ip, ix, ic, row_lo=lo, sites=sites)
        if len(ix) == 0:
            assert info[5] == 0 and info[6] == hi - lo


# ---------------------------------------------------------------------------------------------
# segment shapes
# ---------------------------------------------------------------------------------------------

CELL_LENGTHS = (0, 1, 7, 8, 9, 511, 512, 513, 2047, 2048, 2049)


@pytest.mark.parametrize('form', ['f64', 'packed', 'counts32'])
def test_segment_shapes(dev, form):
    """Rows whose cell in slab 1 holds 0, 1, 7, 8, 9, 511, 512, 513 and 2047 .. 2049 entries (pieces of 8, chunks of
    512, tiles of 2048 entries), a big count as the first and the last entry of such cells, rows that span all three
    slabs, and cells far longer than one CTA's share of the short stream (boundary_fix stitches them)."""
    n, width = 7680, 2560
    rng = np.random.default_rng(6)
    ent = []
    for i, L in enumerate(CELL_LENGTHS):
        r = 100 + i
        cols = np.sort(rng.choice(np.arange(width, 2 * width), L, replace=False))
        for j, c in enumerate(cols):
            big = (j == 0 or j == L - 1 or j == 7 or j == 8) and i % 2 == 0
            ent.append((r, int(c), 70000 + j if big else int(rng.integers(1, 60000))))
    for r in (0, 2000, n - 1):                           # rows across every slab, from the first to the last column
        for c in np.sort(rng.choice(n, 3000, replace=False)):
            if c != r:
                ent.append((r, int(c), int(rng.integers(1, 60000))))
    rows_taken = {e[0] for e in ent}
    base_rows = np.array(sorted(set(range(n)) - rows_taken))
    rr = base_rows[rng.integers(0, len(base_rows), 40000)]
    cc = rng.integers(0, n, 40000)
    keys = {(int(a), int(b)) for a, b in zip(rr, cc)}
    keys |= {(int(r), int(r)) for r in base_rows[rng.random(len(base_rows)) < 0.9]}
    allk = {(a, b): int(x) for (a, b), x in zip(sorted(keys), K.small_counts(rng, len(keys)))}
    allk.update({(r, c): x for r, c, x in ent})
    key = np.array(sorted(allk), dtype=np.int64)
    indptr, indices, counts = K.csr_from_keys(n, key[:, 0], key[:, 1],
                                              np.array([allk[tuple(k)] for k in key.tolist()], dtype=np.uint32))
    sites = K.sites_for(n, 6)
    _opts(dev, width=width, count_stream={'packed': 2, 'counts32': 1}.get(form))
    if form == 'f64':
        info = check_case(dev, n, indptr, indices, _normed(indptr, indices, counts, sites))
    else:
        info = check_case(dev, n, indptr, indices, counts, sites=sites)
    assert info[0] == 3
    assert info[4] // 148 < 2049                          # the longest cell is longer than a CTA's share
