"""
Pair accumulation (accum.cu) at its switch points (-m gpu), every comparison exact -- indptr, indices, counts and the
info dict -- against the NumPy reference of tests/test_accum_refs.py:

- classify plans: one case per reachable (shared-memory diagonal, rank-table mode, partial diagonal) class of plan(),
  each with the dense rank map, a permuted map (the device's rank-map check fails: gather path) and a map with one
  value >= n_seq; records hit the rank-table word edges, ids beyond the table, the partial diagonal's last and first
  global contig, both matcher values, bit 63, and tiles of accepted off-diagonal pairs only (a staging flush per tile);
- key widths b = 1..28: every radix pass count, digit width and buffer parity of the key and composite sorts;
- the composite's count escape (count >= 2^cbits - 1) for b = 18..28;
- narrow records (5- / 6-byte pairs, 3- / 4-byte same-reference records) at full id width;
- capacity, workspace reuse, CUDA-graph replay against direct launches, recycled workspace addresses;
- the host-driven row-block kernels (row_hist, route, reduce_block, emit_block) on one GPU with virtual ranks.

Every case asserts the plan it was written for through b3c_accum_plan, so a change to plan() fails here instead of
quietly testing another branch.
"""
import sys

import numpy as np
import pytest

import test_accum_refs as R

pytestmark = pytest.mark.gpu

OPT_USE_GRAPHS = 6


@pytest.fixture(scope='module')
def dev():
    import torch
    if not torch.cuda.is_available():
        pytest.skip('no CUDA device')
    from bin3c_b200 import device
    return device


@pytest.fixture(autouse=True)
def _restore_options():
    """Options are process-global: graph replay back on after each test, whether it passed or not."""
    yield
    cabi = sys.modules.get('bin3c_b200._cabi')
    if cabi is not None:
        cabi.check(cabi.lib.b3c_set_option(OPT_USE_GRAPHS, 1))


def _plan(dev, n_seq, n_refs, cls=None):
    got = R.device_plan(dev.lib, n_seq, n_refs)
    want = R.py_plan(n_seq, n_refs)
    assert {k: got[k] for k in want} == want, (n_seq, n_refs, got)
    if cls is not None:
        assert R.plan_class(got) == cls, (n_seq, n_refs, got)
    return got


def _result(csr, info):
    indptr, indices, data = csr.host_arrays()
    return dict(indptr=indptr.copy(), indices=indices.copy(), data=data.copy(), info=dict(info))


def _assert_equal(got, want, what=''):
    assert got['info'] == want['info'], (what, got['info'], want['info'])
    assert np.array_equal(got['indptr'], want['indptr']), what
    assert np.array_equal(got['indices'], want['indices']), what
    assert np.array_equal(got['data'], want['data']), what


def _run(dev, acc, adds, symmetric):
    """begin, the add calls, finish -> host arrays."""
    import torch
    acc.begin()
    for add in adds:
        add(acc)
    out = _result(*acc.finish(symmetric=symmetric))
    torch.cuda.synchronize()
    return out


def _native_add(rec_dev):
    return lambda acc: acc.add(rec_dev)


def _identity(n):
    return lambda t: np.where(np.asarray(t, dtype=np.int64) < n, np.asarray(t, dtype=np.int64), -1)


# ---------------------------------------------------------------------------------------------
# classify plans
# ---------------------------------------------------------------------------------------------

def _plan_records(rng, n_seq, n_refs, keep, diag_k):
    """Native records for one plan case (numpy uint64) and the all-off-diagonal head it starts with."""
    n_warps = 148 * 32
    # head: two warp tiles per warp of accepted off-diagonal pairs (a staging flush at every tile when cap_w = 128)
    h = 2 * n_warps * R.CLS_WTILE
    i = rng.integers(0, n_seq, h)
    j = (i + 1 + rng.integers(0, max(n_seq - 1, 1), h)) % n_seq
    parts = [(keep[i], keep[j], np.ones(h, bool))]
    # rank-table word edges, the last reference, ids beyond the table
    edges = [[0, n_refs - 1, n_refs, n_refs + 1, 2 ** 31 - 1], rng.integers(n_refs, 2 ** 31, 8)]
    for step in (12, 32, 64, 2048):
        w = rng.integers(1, max(2, n_refs // step + 1), 8)
        edges += [step * w - 1, step * w]
    edges = np.concatenate(edges)
    edges = np.unique(np.clip(edges, 0, 2 ** 31 - 1))
    m = 20000
    e1 = rng.choice(edges, m)
    e2 = np.where(rng.random(m) < 0.5, rng.choice(keep, m), rng.choice(edges, m))
    parts.append((e1, e2, rng.random(m) < 0.7))
    # diagonal pairs on the partial diagonal's last and first global contig, and on both ends
    dc = [c for c in {0, n_seq - 1, diag_k - 1, diag_k} if 0 <= c < n_seq]
    d = np.repeat(np.asarray(dc), 3000)
    parts.append((keep[d], keep[d], rng.random(len(d)) < 0.9))
    # ordinary map: heavy duplicates, mostly intra-contig, some non-kept ids
    p = 300000
    a = keep[rng.integers(0, min(n_seq, 4000), p)]
    b = np.where(rng.random(p) < 0.5, a, keep[rng.integers(0, n_seq, p)])
    a = np.where(rng.random(p) < 0.05, rng.integers(0, n_refs, p), a)
    parts.append((a, b, rng.random(p) < 0.85))
    ti = np.concatenate([x[0] for x in parts]).astype(np.int64)
    tj = np.concatenate([x[1] for x in parts]).astype(np.int64)
    ok = np.concatenate([x[2] for x in parts])
    return ti, tj, ok, R.pack_native(ti, tj, ok, bit63=rng.random(len(ti)) < 0.5)


def _plan_case(dev, n_seq, n_refs, cls, luts=('rank', 'permuted', 'beyond')):
    import torch
    plan = _plan(dev, n_seq, n_refs, cls)
    rng = np.random.default_rng(n_seq * 7 + n_refs)
    keep = np.sort(rng.choice(n_refs, n_seq, replace=False)) if n_refs > n_seq else np.arange(n_seq)
    keep[-1] = n_refs - 1                                   # the last reference is kept
    keep = np.unique(keep)
    assert len(keep) == n_seq
    ti, tj, ok, rec = _plan_records(rng, n_seq, n_refs, keep, plan['diag_k'])
    rec_dev = dev.to_device(rec)
    for kind in luts:
        lut = np.full(n_refs, -1, dtype=np.int32)
        lut[keep] = rng.permutation(n_seq) if kind == 'permuted' else np.arange(n_seq)
        if kind == 'beyond':
            lut[keep[7]] = n_seq + 3
        acc = dev.Accumulator(n_seq, lut, len(rec))
        for symmetric in (True, False):
            got = _run(dev, acc, [_native_add(rec_dev)], symmetric)
            want = R.ref_accumulate(ti, tj, ok, R.lut_index(lut, n_seq), n_seq, symmetric)
            _assert_equal(got, want, (kind, symmetric))
        del acc
    torch.cuda.synchronize()


@pytest.mark.parametrize('cls', sorted(R.PLAN_CASES), ids=lambda c: 'diag%d_rank%d_%s' % (c[0], c[1], 'partial' if c[2] else 'none'))
def test_classify_plan(dev, cls):
    n_seq, n_refs = R.PLAN_CASES[cls]
    _plan_case(dev, n_seq, n_refs, cls)


@pytest.mark.parametrize('n_seq,n_refs', R.MODE3_EDGE_CASES)
def test_classify_two_level_table_sentinel_block(dev, n_seq, n_refs):
    """Two-level rank table whose bitmap word count is 1 or 31 mod 32: the zero sentinel word in a block of its own
    or at the end of the last block."""
    plan = _plan(dev, n_seq, n_refs)
    assert plan['smem_rank'] == 3
    _plan_case(dev, n_seq, n_refs, None, luts=('rank',))


# ---------------------------------------------------------------------------------------------
# key widths
# ---------------------------------------------------------------------------------------------

def test_width_cases_cover_every_sort_shape(dev):
    reached = set()
    for b, n_seq in R.WIDTH_CASES:
        reached.update(R.sort_shape(_plan(dev, n_seq, n_seq)))
    assert reached == R.all_sort_shapes(28)


@pytest.mark.parametrize('b,n_seq', R.WIDTH_CASES, ids=lambda v: str(v))
def test_key_width(dev, b, n_seq):
    import torch
    plan = _plan(dev, n_seq, n_seq)
    assert plan['b'] == b
    rng = np.random.default_rng(b * 1000 + n_seq % 997)
    pool = np.unique(np.concatenate([rng.integers(0, n_seq, 48), [0, n_seq - 1, max(n_seq - 2, 0)]]))
    p = 200000
    ti = pool[rng.integers(0, len(pool), p)]
    tj = np.where(rng.random(p) < 0.3, ti, pool[rng.integers(0, len(pool), p)])
    ti[:64] = n_seq - 1                                  # index n_seq - 1 in both positions
    tj[32:96] = n_seq - 1
    ti[-4:] = n_seq + 5                                  # beyond the table
    ok = rng.random(p) < 0.9
    rec = dev.to_device(R.pack_native(ti, tj, ok))
    lut = torch.arange(n_seq, dtype=torch.int32, device='cuda')
    acc = dev.Accumulator(n_seq, lut, p)
    for symmetric in (True, False):
        got = _run(dev, acc, [_native_add(rec)], symmetric)
        want = R.ref_accumulate(ti, tj, ok, _identity(n_seq), n_seq, symmetric)
        _assert_equal(got, want, symmetric)
    del acc, lut, rec
    torch.cuda.empty_cache()


# ---------------------------------------------------------------------------------------------
# composite count escape
# ---------------------------------------------------------------------------------------------

@pytest.mark.parametrize('b', list(range(18, 29)))
def test_composite_count_escape(dev, b):
    """The mirror composite keeps cbits = 64 - 2b bits for the count; a count >= 2^cbits - 1 is stored as the escape
    and looked up by bisection in k_emit.  Three hot cells counted 2^cbits - 2, 2^cbits - 1 and 2^cbits (half of each
    cell's records with the mates swapped) beside a seeded random map.  b = 18 takes ~0.8 G keys and ~30 GB of
    workspace.  Out of scope: b = 17 (cbits 30, ~3.2 G keys) and b <= 16, where cbits = 32 and no count below the 2^32
    pair capacity escapes."""
    import torch
    n_seq = (1 << (b - 1)) + 1
    plan = _plan(dev, n_seq, n_seq)
    cb = plan['cbits']
    assert plan['b'] == b and cb == 64 - 2 * b
    hot = [((0, n_seq - 1), (1 << cb) - 2), ((n_seq - 2, n_seq - 1), (1 << cb) - 1), ((1, 2), 1 << cb)]
    rng = np.random.default_rng(b)
    p = 100000
    ti = rng.integers(0, n_seq, p)
    tj = np.where(rng.random(p) < 0.3, ti, rng.integers(0, n_seq, p))
    lo, hi = np.minimum(ti, tj), np.maximum(ti, tj)
    clash = np.zeros(p, bool)
    for (i, j), _ in hot:
        clash |= (lo == i) & (hi == j)
    ti, tj = ti[~clash], tj[~clash]
    ok = rng.random(len(ti)) < 0.9
    parts = [dev.to_device(R.pack_native(ti, tj, ok))]
    for (i, j), c in hot:
        for x, y, k in ((i, j, c // 2), (j, i, c - c // 2)):
            parts.append(torch.full((k,), int(R.pack_native([x], [y], [True])[0]), dtype=torch.int64, device='cuda'))
    rec = torch.cat(parts)
    del parts
    n_rec = rec.numel()
    lut = torch.arange(n_seq, dtype=torch.int32, device='cuda')
    acc = dev.Accumulator(n_seq, lut, n_rec)
    got = _run(dev, acc, [_native_add(rec)], True)
    del acc, rec, lut
    torch.cuda.empty_cache()
    # reference: the random map, plus the hot cells analytically
    bb = R.key_bits(n_seq)
    acc_m = ok
    a, c = np.minimum(ti[acc_m], tj[acc_m]), np.maximum(ti[acc_m], tj[acc_m])
    keys, cnt = np.unique((a[a != c] << bb) | c[a != c], return_counts=True)
    hk = np.array([(i << bb) | j for (i, j), _ in hot], dtype=np.int64)
    hc = np.array([k for _, k in hot], dtype=np.int64)
    diag = np.bincount(a[a == c], minlength=n_seq)
    counters = dict(accepted=int(acc_m.sum() + hc.sum()), ref_excluded=0, poor_match=int((~ok).sum()))
    want = R.ref_from_cells(n_seq, np.concatenate([keys, hk]), np.concatenate([cnt, hc]), diag, counters)
    _assert_equal(got, want)


# ---------------------------------------------------------------------------------------------
# narrow records at full id width
# ---------------------------------------------------------------------------------------------

def _aligned_chunks(chunks):
    """[(packed uint8 array, n_records)] -> one uint8 array with each chunk at a 16-byte boundary, and the offsets."""
    offs, at = [], 0
    for buf, _ in chunks:
        offs.append(at)
        at += (len(buf) + 15) // 16 * 16
    out = np.zeros(max(at, 16), dtype=np.uint8)
    for (buf, _), o in zip(chunks, offs):
        out[o:o + len(buf)] = buf
    return out, offs


@pytest.mark.parametrize('fmt', ['pair5', 'pair6', 'same3', 'same4'])
def test_narrow_records_full_width(dev, fmt):
    import torch
    B, same = int(fmt[-1]), fmt.startswith('same')
    tb, marker = R.narrow_fields(B, same)
    n_refs = marker - 1                              # the widest table the format accepts
    if fmt == 'same4':
        free, _ = torch.cuda.mem_get_info()
        if free < 40 * 2 ** 30:
            n_refs = 1 << 28                         # LUT of 1 GB instead of 8 GB
    rng = np.random.default_rng(B * 10 + int(same))
    n_keep = 300000
    keep = np.unique(np.concatenate([rng.integers(0, n_refs, n_keep), [0, n_refs - 1],
                                     1 << np.arange(n_refs.bit_length() - 1)]))
    n_seq = len(keep)
    _plan(dev, n_seq, n_refs)
    # records: kept ids over the whole range, every id bit set in every field, ids in [n_refs, marker], the marker
    p = 400003
    ti = keep[rng.integers(0, n_seq, p)]
    tj = ti.copy() if same else np.where(rng.random(p) < 0.3, ti, keep[rng.integers(0, n_seq, p)])
    nb = (n_refs - 1).bit_length()                 # id bits below the table size
    bits = 1 << np.arange(nb - 1)
    ti[:nb - 1] = bits
    ti[nb - 1:2 * nb - 2] = n_refs - 1
    if not same:
        tj[:nb - 1] = n_refs - 1
        tj[nb - 1:2 * nb - 2] = bits
    special = rng.integers(n_refs, marker + 1, 2000)
    k = np.arange(2 * nb, 2 * nb + 2000)
    ti[k] = special
    if not same:
        tj[k] = np.where(rng.random(2000) < 0.5, special, keep[rng.integers(0, n_seq, 2000)])
        tj[k[:500]], ti[k[:500]] = special[:500], keep[rng.integers(0, n_seq, 500)]
    else:
        tj[k] = special
    ti[-300:] = np.arange(n_refs - 150, n_refs + 150).clip(max=marker)
    if same:
        tj = ti.copy()
    perm = rng.permutation(p)
    ti, tj = ti[perm], tj[perm]
    ok = rng.random(p) < 0.85
    field_or = np.bitwise_or.reduce(ti[ti < n_refs]) | np.bitwise_or.reduce(tj[tj < n_refs])
    assert field_or == (1 << nb) - 1                 # every bit of an id field is set at least once
    want_sym = R.ref_accumulate(ti, tj, ok, R.rank_index(keep, n_refs), n_seq, True)

    lut = torch.full((n_refs,), -1, dtype=torch.int32, device='cuda')
    lut[torch.from_numpy(keep).cuda()] = torch.arange(n_seq, dtype=torch.int32, device='cuda')
    acc = dev.Accumulator(n_seq, lut, p)
    # one call (n at an odd residue), many calls at every residue mod 16, the native records of the same pairs
    single = dev.to_device(R.pack_narrow(ti, tj, ok, B, same))
    sizes, at = [], 0
    while at < p:
        s = min(int(16 * rng.integers(0, 40) + len(sizes) % 16) or 1, p - at)
        sizes.append(s)
        at += s
    assert {s % 16 for s in sizes[:-1]} == set(range(16))
    cuts = np.concatenate([[0], np.cumsum(sizes)])
    chunks = [(R.pack_narrow(ti[a:z], tj[a:z], ok[a:z], B, same), z - a) for a, z in zip(cuts[:-1], cuts[1:])]
    buf, offs = _aligned_chunks(chunks)
    buf_dev = dev.to_device(buf)
    native = dev.to_device(R.narrow_to_native(*R.decode_narrow(R.pack_narrow(ti, tj, ok, B, same), p, B, same),
                                              B, same))

    def many(acc):
        for (c, n), o in zip(chunks, offs):
            acc.add_packed(buf_dev[o:o + len(c)], n, B, same=same)

    runs = dict(single=[lambda a: a.add_packed(single, p, B, same=same)],
                many=[many], native=[_native_add(native)])
    for name, adds in runs.items():
        _assert_equal(_run(dev, acc, adds, True), want_sym, name)
    want_up = R.ref_accumulate(ti, tj, ok, R.rank_index(keep, n_refs), n_seq, False)
    _assert_equal(_run(dev, acc, runs['single'], False), want_up, 'single upper')
    del acc, lut
    torch.cuda.empty_cache()


# ---------------------------------------------------------------------------------------------
# capacity and workspace reuse
# ---------------------------------------------------------------------------------------------

def _rank_lut(rng, n_seq, n_refs):
    keep = np.sort(rng.choice(n_refs, n_seq, replace=False))
    lut = np.full(n_refs, -1, dtype=np.int32)
    lut[keep] = np.arange(n_seq)
    return keep, lut


def _map(rng, keep, n_refs, p, off=0.5):
    n = len(keep)
    a = keep[rng.integers(0, n, p)]
    b = np.where(rng.random(p) < off, keep[rng.integers(0, n, p)], a)
    a = np.where(rng.random(p) < 0.05, rng.integers(0, n_refs + 10, p), a)
    return a, b, rng.random(p) < 0.85


def _n_offdiag_keys(ti, tj, ok, index):
    ii, jj = index(ti), index(tj)
    return int(((ii >= 0) & (jj >= 0) & ok & (ii != jj)).sum())


def test_capacity_exact_and_recovery(dev):
    from bin3c_b200._cabi import B3CError
    rng = np.random.default_rng(61)
    n, n_refs = 1000, 1200
    _plan(dev, n, n_refs, (1, 2, False))
    keep, lut = _rank_lut(rng, n, n_refs)
    index = R.lut_index(lut, n)
    ti, tj, ok = _map(rng, keep, n_refs, 300000, off=0.2)
    K = _n_offdiag_keys(ti, tj, ok, index)
    assert 0 < K < len(ti) // 3                          # many diagonal, poor and excluded records beside the keys
    rec = dev.to_device(R.pack_native(ti, tj, ok))
    want = R.ref_accumulate(ti, tj, ok, index, n)
    _assert_equal(_run(dev, dev.Accumulator(n, lut, K), [_native_add(rec)], True), want, 'capacity == keys')
    acc = dev.Accumulator(n, lut, K - 1)
    with pytest.raises(B3CError, match='capacity'):
        _run(dev, acc, [_native_add(rec)], True)
    s1, s2, sok = _map(rng, keep, n_refs, 20000)
    assert _n_offdiag_keys(s1, s2, sok, index) <= K - 1
    small = dev.to_device(R.pack_native(s1, s2, sok))
    _assert_equal(_run(dev, acc, [_native_add(small)], True), R.ref_accumulate(s1, s2, sok, index, n), 'after error')


@pytest.mark.parametrize('n,n_refs', [(1000, 1200), (70000, 80000)])
def test_workspace_reuse_graphs_and_direct(dev, n, n_refs):
    """One accumulator runs maps of N, N/3, 0 and 1 keys and N again; the arrays are the same with the sort-reduce
    replayed as a CUDA graph and launched directly."""
    rng = np.random.default_rng(n)
    _plan(dev, n, n_refs)
    keep, lut = _rank_lut(rng, n, n_refs)
    index = R.lut_index(lut, n)
    N = 400000
    maps = [_map(rng, keep, n_refs, N), _map(rng, keep, n_refs, N // 3)]
    d = keep[rng.integers(0, n, 5000)]
    maps.append((d, d, np.ones(5000, bool)))                                 # 0 keys: diagonal only
    maps.append((np.append(d, keep[1]), np.append(d, keep[2]), np.ones(5001, bool)))  # 1 key
    maps.append(_map(rng, keep, n_refs, N))
    recs = [dev.to_device(R.pack_native(*m)) for m in maps]
    wants = [R.ref_accumulate(*m, index, n) for m in maps]
    assert [_n_offdiag_keys(*m, index) for m in maps[2:4]] == [0, 1]
    outs = {}
    for graphs in (1, 0):
        dev.check(dev.lib.b3c_set_option(OPT_USE_GRAPHS, graphs))
        acc = dev.Accumulator(n, lut, N)
        outs[graphs] = []
        for k, (rec, want) in enumerate(zip(recs, wants)):
            got = _run(dev, acc, [_native_add(rec)], k % 2 == 0)
            if k % 2:
                want = R.ref_accumulate(*maps[k], index, n, symmetric=False)
            _assert_equal(got, want, (graphs, k))
            outs[graphs].append(got)
    for g1, g0 in zip(outs[1], outs[0]):
        _assert_equal(g1, g0)


def test_two_live_accumulators_alternate(dev):
    rng = np.random.default_rng(77)
    cases = [(1000, 1200, (1, 2, False)), (70000, 80000, None)]
    accs, idx, keeps = [], [], []
    for n, n_refs, cls in cases:
        _plan(dev, n, n_refs, cls)
        keep, lut = _rank_lut(rng, n, n_refs)
        accs.append(dev.Accumulator(n, lut, 200000))
        idx.append(R.lut_index(lut, n))
        keeps.append((keep, n_refs, n))
    for rnd in range(3):
        for acc, index, (keep, n_refs, n) in zip(accs, idx, keeps):
            m = _map(rng, keep, n_refs, 150000 + 1000 * rnd)
            got = _run(dev, acc, [_native_add(dev.to_device(R.pack_native(*m)))], rnd != 1)
            _assert_equal(got, R.ref_accumulate(*m, index, n, symmetric=rnd != 1), rnd)


def test_recycled_workspace_address_replans(dev):
    """A freed accumulator's workspace handed to a new one of another n_seq: the new one must not replay the old
    workspace's captured sort-reduce (b3c_accum_begin forgets the address's graphs)."""
    import torch
    rng = np.random.default_rng(5)
    n1, n2, n_refs = 6000, 5000, 7000
    keep1, lut1 = _rank_lut(rng, n1, n_refs)
    keep2, lut2 = _rank_lut(rng, n2, n_refs)
    m1, m2 = _map(rng, keep1, n_refs, 300000), _map(rng, keep2, n_refs, 300000)
    cap1, cap2 = 5_000_000, 4_990_000
    _plan(dev, n1, n_refs)
    _plan(dev, n2, n_refs)
    a = dev.Accumulator(n1, lut1, cap1)
    _assert_equal(_run(dev, a, [_native_add(dev.to_device(R.pack_native(*m1)))], True),
                  R.ref_accumulate(*m1, R.lut_index(lut1, n1), n1))
    addr = a.ws.data_ptr()
    del a
    torch.cuda.synchronize()
    b = dev.Accumulator(n2, lut2, cap2)
    if b.ws.data_ptr() != addr:
        pytest.skip('the caching allocator did not hand the freed workspace to the new accumulator')
    _assert_equal(_run(dev, b, [_native_add(dev.to_device(R.pack_native(*m2)))], True),
                  R.ref_accumulate(*m2, R.lut_index(lut2, n2), n2))


def test_many_tiny_adds_equal_one(dev):
    """1000 add calls of one to three records each (every launch flushes its shared-memory diagonal) == one call."""
    rng = np.random.default_rng(3)
    n, n_refs = 1000, 1200
    _plan(dev, n, n_refs, (1, 2, False))
    keep, lut = _rank_lut(rng, n, n_refs)
    sizes = rng.integers(1, 4, 1000)
    ti, tj, ok = _map(rng, keep, n_refs, int(sizes.sum()), off=0.3)
    rec = R.pack_native(ti, tj, ok)
    offs = np.concatenate([[0], np.cumsum((sizes + 1) // 2 * 2)])      # even offsets: 16-byte aligned starts
    spread = np.zeros(int(offs[-1]), dtype=np.uint64)
    cuts = np.concatenate([[0], np.cumsum(sizes)])
    for k in range(len(sizes)):
        spread[offs[k]:offs[k] + sizes[k]] = rec[cuts[k]:cuts[k + 1]]
    sp_dev = dev.to_device(spread)
    adds = [(lambda o, s: (lambda acc: acc.add(sp_dev[o:o + s])))(int(offs[k]), int(sizes[k])) for k in range(1000)]
    acc = dev.Accumulator(n, lut, len(rec))
    want = R.ref_accumulate(ti, tj, ok, R.lut_index(lut, n), n)
    many = _run(dev, acc, adds, True)
    one = _run(dev, acc, [_native_add(dev.to_device(rec))], True)
    _assert_equal(many, want)
    _assert_equal(one, want)


# ---------------------------------------------------------------------------------------------
# row-block kernels on one GPU
# ---------------------------------------------------------------------------------------------

RB_N, RB_REFS = 3000, 3500
RB_HEAVY = 1234                      # the heaviest row
RB_DIAG_ONLY = (2000, 2005)          # rows with diagonal entries only
RB_EMPTY = (2500, 2505)              # rows with no entry


@pytest.fixture(scope='module')
def rb_map():
    rng = np.random.default_rng(2024)
    keep = np.sort(rng.choice(RB_REFS, RB_N, replace=False))
    lut = np.full(RB_REFS, -1, dtype=np.int32)
    lut[keep] = np.arange(RB_N)
    free = np.setdiff1d(np.arange(RB_N), np.r_[RB_DIAG_ONLY[0]:RB_DIAG_ONLY[1], RB_EMPTY[0]:RB_EMPTY[1]])
    p = 120000
    i = free[rng.integers(0, len(free), p)]
    j = np.where(rng.random(p) < 0.4, i, free[rng.integers(0, len(free), p)])
    i[:20000] = RB_HEAVY
    d = np.repeat(np.arange(*RB_DIAG_ONLY), 50)
    i, j = np.concatenate([i, d]), np.concatenate([j, d])
    ok = rng.random(len(i)) < 0.9
    ok[-len(d):] = True
    ti, tj = keep[i], keep[j]
    ti[:30] = RB_REFS + 4                                              # beyond the table
    perm = rng.permutation(len(ti))
    ti, tj, ok = ti[perm], tj[perm], ok[perm]
    index = R.lut_index(lut, RB_N)
    ref = R.ref_accumulate(ti, tj, ok, index, RB_N)
    deg = np.diff(ref['indptr'])
    assert int(np.argmax(deg)) == RB_HEAVY
    assert all(deg[r] == 1 and ref['indices'][ref['indptr'][r]] == r for r in range(*RB_DIAG_ONLY))
    assert all(deg[r] == 0 for r in range(*RB_EMPTY))
    return dict(lut=lut, ti=ti, tj=tj, ok=ok, index=index, ref=ref, sites=np.ones(RB_N, np.int32),
                lengths=np.full(RB_N, 5000, np.int32))


def _shard(dev, m, splits, n_src=None, empty_src=(), capacity=None):
    """Virtual ranks: one CudaEngine per rank on this device, the collectives done here as the sharded driver does
    them.  Returns {rank: (indptr, indices, counts) host copies}; asserts row_hist, route counts and counters."""
    import torch
    from bin3c_b200 import dist
    G = len(splits) - 1
    n_src = G if n_src is None else n_src
    rng = np.random.default_rng(G)
    owner = rng.integers(0, n_src, len(m['ti']))
    for g in empty_src:
        owner[owner == g] = (g + 1) % n_src
    cap = capacity or 2 * len(m['ti'])                 # a rank may receive both directions of every key
    engines = [dist.CudaEngine(m['lut'], m['lengths'], m['sites'], cap) for _ in range(n_src)]
    srcs = [np.flatnonzero(owner == g) for g in range(n_src)]
    for e, s in zip(engines, srcs):
        e.classify(dev.to_device(R.pack_native(m['ti'][s], m['tj'][s], m['ok'][s])))
    rowcnt = sum(e.row_hist().clone() for e in engines)
    dk, _ = R.directed_keys(m['ti'], m['tj'], m['ok'], m['index'], RB_N)
    b = R.key_bits(RB_N)
    assert np.array_equal(rowcnt.cpu().numpy(), np.bincount(dk >> b, minlength=RB_N))
    send, counters = [], dict(accepted=0, ref_excluded=0, poor_match=0)
    for e, s in zip(engines, srcs):
        out, counts, c = e.route(splits)
        dks, _ = R.directed_keys(m['ti'][s], m['tj'][s], m['ok'][s], m['index'], RB_N)
        want = [int(((dks >> b) >= splits[g]).sum() - ((dks >> b) >= splits[g + 1]).sum()) for g in range(G)]
        assert counts == want
        offs = np.concatenate([[0], np.cumsum(counts)])
        send.append([out[offs[g]:offs[g + 1]].clone() for g in range(G)])
        for k in counters:
            counters[k] += c[k]
    assert counters == {k: m['ref']['info'][k] for k in counters}
    diag = sum(e.diag_counts().to(torch.int64) for e in engines).to(torch.int32)
    for e in engines:
        e.diag_counts().copy_(diag)
    blocks = {}
    for g in range(G):
        lo, hi = int(splits[g]), int(splits[g + 1])
        if hi <= lo:
            continue
        keys = torch.cat([send[s][g] for s in range(n_src)])
        blk = engines[g % n_src].build_block(keys, lo, hi)
        blocks[g] = tuple(a.copy() for a in blk.host_arrays())       # before the engine's pool reuses them
    torch.cuda.synchronize()
    return blocks


def _assert_blocks(m, splits, blocks):
    ref = m['ref']
    ip = ref['indptr']
    for g in range(len(splits) - 1):
        lo, hi = int(splits[g]), int(splits[g + 1])
        if hi <= lo:
            assert g not in blocks
            continue
        indptr, indices, counts = blocks[g]
        assert np.array_equal(indptr, ip[lo:hi + 1] - ip[lo]), g
        assert np.array_equal(indices, ref['indices'][ip[lo]:ip[hi]]), g
        assert np.array_equal(counts, ref['data'][ip[lo]:ip[hi]]), g


RB_SPLITS = {
    'one_rank': [0, RB_N],
    'two_balanced': [0, RB_N // 2, RB_N],
    'unaligned': [0, 1, 333, RB_N - 1, RB_N],
    'empty_ranks': [0, 0, 700, 700, 1700, RB_N, RB_N],
    'heaviest_row_alone': [0, RB_HEAVY, RB_HEAVY + 1, RB_N],
    'diag_only_and_empty_blocks': [0, RB_DIAG_ONLY[0], RB_DIAG_ONLY[1], RB_EMPTY[0], RB_EMPTY[1], RB_N],
}


@pytest.mark.parametrize('name', sorted(RB_SPLITS))
def test_row_blocks(dev, rb_map, name):
    _plan(dev, RB_N, RB_REFS, (1, 2, False))
    splits = RB_SPLITS[name]
    _assert_blocks(rb_map, splits, _shard(dev, rb_map, splits, empty_src=(1,) if len(splits) > 3 else ()))


def test_row_blocks_64_ranks(dev, rb_map):
    rng = np.random.default_rng(64)
    cuts = np.sort(rng.integers(0, RB_N + 1, 63))
    cuts[10] = cuts[11]                                   # an empty rank in the middle
    splits = [0] + cuts.tolist() + [RB_N]
    _assert_blocks(rb_map, splits, _shard(dev, rb_map, splits, empty_src=(5,)))


def test_route_refuses_65_ranks(dev, rb_map):
    from bin3c_b200 import dist
    e = dist.CudaEngine(rb_map['lut'], rb_map['lengths'], rb_map['sites'], 1000)
    e.classify(dev.to_device(R.pack_native(rb_map['ti'][:1000], rb_map['tj'][:1000], rb_map['ok'][:1000])))
    with pytest.raises(AssertionError, match='rank count'):
        e.route(np.linspace(0, RB_N, 66).astype(np.int32))


def test_row_block_over_capacity_raises(dev, rb_map):
    from bin3c_b200._cabi import B3CError
    G = 4
    cap = len(rb_map['ti']) // G + 100                     # each source fits; rank 0 receives every directed key
    with pytest.raises(B3CError, match='capacity'):
        _shard(dev, rb_map, [0, RB_N, RB_N, RB_N, RB_N], capacity=cap)
