"""
The device half of the sharded path (bin3c_b200/dist.py, DESIGN section 5) with W virtual ranks on one GPU (-m gpu):
one engine per rank on this device, every kernel launched for rank 0, 1, ..., W-1 in turn, and a device
synchronisation wherever the product puts a peer barrier.  No call here waits on another rank's kernel, so nothing
can spin: the flag barrier, the arena all-reduce and the persistent peer KR kernel at more than one rank stay covered
by tests/test_gpu_dist.py on multi-GPU machines only.

- Peer-arena accumulation (b3c_shard_publish / scatter / reduce_block, b3c_accum_emit_block, b3c_peer_put) at
  W = 2, 3, 5 and 8: splits against a NumPy restatement of k_shard_splits, every block, the counters and the keys each
  owner received exactly against tests/test_accum_refs.py, the mask and x regions of every arena; tail chunks, heavy
  rows, idle sources, narrow and split records, empty row blocks, receive-buffer overflow, graph replay, the chunk cap.
- The row-block KR phase API (b3c_krp_*) through the product's own dist.kr_block_loop at W = 2, 3, 4 and 8: the phase
  contract checked at every collective (u zero outside the rank's rows, partials at their identity in chunks it does
  not own), the loop-control trace against tests/np_engine.py on the same blocks, n_iter, zero diagonals and x against
  the oracle and the one-GPU kernel; both SpMV forms in one solve; the tie, max_iter and NaN outcomes, also through
  ShardedHotPath.balance(), whose exceptions must be those of dev.kr_scale_vector.
- The whole path end to end (accumulation -> masks -> site_norm -> balance -> kr_apply -> compress_edges) against
  oracle.run_path with the bars of tests/test_gpu_dist.py.
"""
import contextlib
import ctypes as C
import sys

import numpy as np
import pytest
import scipy.sparse as sp

import kr_operand_cases as K
import test_accum_refs as R
from conftest import load_golden, golden_lut

pytestmark = pytest.mark.gpu

OPT_KR_SLAB_WIDTH, OPT_KR_MAX_SLABS, OPT_USE_GRAPHS = 1, 2, 6
DEFAULT_OPTIONS = {OPT_KR_SLAB_WIDTH: 28672, OPT_KR_MAX_SLABS: 16, OPT_USE_GRAPHS: 1}
CHUNK = 1024                     # accum.cu XA_CHUNK = kr.cu CHUNK
XA_MAX_CHUNKS = 4096             # accum.cu: row chunks the split kernel handles
REL_TOL = 1e-9
PA, PB, PC, PMIN, PNEGMAX, PG1, PG2 = range(7)


@pytest.fixture(scope='module')
def dev():
    import torch
    if not torch.cuda.is_available():
        pytest.skip('no CUDA device')
    from bin3c_b200 import device
    return device


@pytest.fixture(autouse=True)
def _restore_options():
    """Options are process-global: back to the defaults after each test, whether it passed or not."""
    yield
    cabi = sys.modules.get('bin3c_b200._cabi')
    if cabi is not None:
        for key, value in DEFAULT_OPTIONS.items():
            cabi.check(cabi.lib.b3c_set_option(key, value))


def _relerr(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b) / np.maximum(np.abs(b), 1e-300))) if a.size else 0.0


# =================================================================================================
# A. peer-arena accumulation
# =================================================================================================

def ref_splits(dk, b, n, G):
    """k_shard_splits restated: chunk weight = directed keys whose row lies in the 1024-row chunk + the chunk's rows;
    cut k goes to the chunk boundary nearer to total * k // G along the running weight (a tie goes after the chunk
    that reaches the target), at most n // 1024 whole chunks, never below the previous cut; the last split is n."""
    nc = -(-n // CHUNK)
    keys = np.add.reduceat(np.bincount(np.asarray(dk, dtype=np.int64) >> b, minlength=n), CHUNK * np.arange(nc))
    cum = np.cumsum(keys + np.minimum(CHUNK, n - CHUNK * np.arange(nc)))
    total = int(cum[-1])
    out, prev = [0], 0
    for k in range(1, G):
        t = total * k // G
        c = int(np.searchsorted(cum, t, side='left'))          # first chunk whose running weight reaches t
        bnd = c
        if c < nc and int(cum[c]) - t <= t - (int(cum[c - 1]) if c else 0):
            bnd = c + 1
        bnd = max(min(bnd, n // CHUNK), prev)
        prev = bnd
        out.append(bnd * CHUNK)
    return out + [n]


def make_map(n, p, seed, heavy=(), heavy_pairs=15000, n_refs=None):
    """Seeded pair records over n contigs (rank LUT over n_refs ids, excluded and out-of-table ids, poor matches,
    ~40 % intra-contig) with `heavy` rows given heavy_pairs extra off-diagonal partners each."""
    rng = np.random.default_rng(seed)
    n_refs = n_refs or n + n // 8 + 3
    keep = np.sort(rng.choice(n_refs, n, replace=False))
    lut = np.full(n_refs, -1, dtype=np.int32)
    lut[keep] = np.arange(n)
    i = rng.integers(0, n, p)
    j = np.where(rng.random(p) < 0.4, i, rng.integers(0, n, p))
    hi = [np.full(heavy_pairs, r) for r in heavy]
    hj = [rng.integers(0, n, heavy_pairs) for _ in heavy]
    i, j = np.concatenate([i] + hi), np.concatenate([j] + hj)
    ti, tj = keep[i], keep[j]
    m = len(ti)
    ti[rng.random(m) < 0.01] = n_refs + 5                      # beyond the table
    excl = np.setdiff1d(np.arange(n_refs), keep)
    if len(excl):
        pick = rng.random(m) < 0.02
        tj[pick] = excl[rng.integers(0, len(excl), int(pick.sum()))]
    ok = rng.random(m) < 0.88
    perm = rng.permutation(m)
    ti, tj, ok = ti[perm], tj[perm], ok[perm]
    index = R.lut_index(lut, n)
    lengths = rng.integers(200, 5000, n).astype(np.int32)
    return dict(n=n, lut=lut, ti=ti, tj=tj, ok=ok, index=index, ref=R.ref_accumulate(ti, tj, ok, index, n),
                lengths=lengths, sites=np.ones(n, np.int32), n_refs=n_refs)


@contextlib.contextmanager
def arenas(dev, n, cap, W):
    """W peer arenas (b3c_peer_alloc) on this device, as the HOST array of device pointers every rank passes."""
    import torch
    lib = dev.lib
    nbytes = lib.b3c_xa_bytes(n, cap)
    assert nbytes > 0
    got = []
    try:
        for _ in range(W):
            p = C.c_void_p()
            dev.check(lib.b3c_peer_alloc(nbytes, C.byref(p), C.create_string_buffer(64)))
            got.append(p.value)
        yield (C.c_void_p * W)(*got)
    finally:
        torch.cuda.synchronize()
        for p in got:
            lib.b3c_peer_free(C.c_void_p(p))


def engines_for(m, W, cap):
    from bin3c_b200 import dist
    return [dist.CudaEngine(m['lut'], m['lengths'], m['sites'], cap) for _ in range(W)]


def peer_accumulate(dev, engines, ptrs, adds):
    """CudaEngine.accumulate_peer in lockstep: classify on every rank | publish on every rank | sync | scatter on every
    rank (own d_splits) | sync | reduce_block + emit_block on every rank.  Returns one dict per rank: rc (and the
    error text), sizes, the rank's d_splits, the block (DeviceCSR) and host copies of its arrays."""
    import torch
    from bin3c_b200 import _cabi
    lib, W = dev.lib, len(engines)
    d_splits = [torch.full((16,), -1, dtype=torch.int32, device='cuda') for _ in range(W)]
    for e, add in zip(engines, adds):
        e.acc.begin()
        add(e)
    for g, e in enumerate(engines):
        dev.check(lib.b3c_shard_publish(dev._ptr(e.acc.ws), ptrs, g, W, dev._stream()))
    torch.cuda.synchronize()
    for g, e in enumerate(engines):
        dev.check(lib.b3c_shard_scatter(dev._ptr(e.acc.ws), ptrs, g, W, dev._ptr(d_splits[g]), dev._stream()))
    torch.cuda.synchronize()
    out = []
    for g, e in enumerate(engines):
        sizes = (C.c_int64 * 24)()
        rc = lib.b3c_shard_reduce_block(dev._ptr(e.acc.ws), ptrs, g, W, dev._ptr(d_splits[g]), sizes, dev._stream())
        r = dict(rc=rc, msg=_cabi.last_error() if rc else '', sizes=[int(v) for v in sizes],
                 d_splits=d_splits[g][:W + 1].cpu().tolist(), block=None)
        if rc == 0 and sizes[2] > sizes[1]:
            lo, hi, nnz = int(sizes[1]), int(sizes[2]), int(sizes[0])
            indptr = torch.empty(hi - lo + 1, dtype=torch.int64, device='cuda')
            indices = torch.empty(max(nnz, 1), dtype=torch.int32, device='cuda')[:nnz]
            counts = torch.empty(max(nnz, 1), dtype=torch.int32, device='cuda')[:nnz]
            dev.check(lib.b3c_accum_emit_block(dev._ptr(e.acc.ws), lo, hi, dev._ptr(indptr), dev._ptr(indices),
                                               dev._ptr(counts), dev._stream()))
            r['block'] = dev.DeviceCSR(hi - lo, indptr, indices, counts, counts=True, row_lo=lo, n_total=e.n)
            r['host'] = tuple(a.copy() for a in r['block'].host_arrays())
        out.append(r)
    torch.cuda.synchronize()
    return out


def native_adds(dev, m, owner, W):
    recs = [dev.to_device(R.pack_native(m['ti'][owner == g], m['tj'][owner == g], m['ok'][owner == g]))
            for g in range(W)]
    return [(lambda r: (lambda e: e.add_records(r)))(r) for r in recs]


def mixed_adds(dev, m, owner, W):
    """Rank g classifies its records as 5-byte, 6-byte, split (same-reference 3 / 4 bytes + pair records) or native
    records, by g % 4."""
    from bin3c_b200 import bam_io
    adds = []
    for g in range(W):
        s = owner == g
        ti, tj, ok = m['ti'][s], m['tj'][s], m['ok'][s]
        kind = g % 4
        if kind in (0, 1):
            B = 5 + kind
            buf = dev.to_device(R.pack_narrow(ti, tj, ok, B))
            adds.append((lambda b, k, B: (lambda e: e.add_records(b, B, k)))(buf, len(ti), B))
        elif kind == 2:
            split = bam_io.split_records(R.pack_native(ti, tj, ok), m['n_refs'] + 6).cuda()
            assert split.n_same > 0 and split.n_pairs > 0
            adds.append((lambda sr: (lambda e: e.add_records(sr)))(split))
        else:
            rec = dev.to_device(R.pack_native(ti, tj, ok))
            adds.append((lambda r: (lambda e: e.add_records(r)))(rec))
    return adds


def check_accumulation(m, res, W, owner=None):
    """Splits, blocks, counters and received keys of every rank, exactly."""
    ref = m['ref']
    n = m['n']
    b = R.key_bits(n)
    dk, _ = R.directed_keys(m['ti'], m['tj'], m['ok'], m['index'], n)
    want_splits = ref_splits(dk, b, n, W)
    rows = dk >> b
    ip = ref['indptr']
    for g, r in enumerate(res):
        assert r['rc'] == 0, (g, r['rc'], r['msg'])
        sz = r['sizes']
        assert r['d_splits'] == want_splits, (g, r['d_splits'], want_splits)
        assert sz[8:8 + W + 1] == want_splits, g
        lo, hi = want_splits[g], want_splits[g + 1]
        assert (sz[1], sz[2]) == (lo, hi), g
        assert sz[3:6] == [ref['info'][k] for k in ('accepted', 'ref_excluded', 'poor_match')], g
        assert sz[6] == int(((rows >= lo) & (rows < hi)).sum()), g
        if hi <= lo:
            assert r['block'] is None and sz[0] == 0, g
            continue
        indptr, indices, counts = r['host']
        assert sz[0] == ip[hi] - ip[lo], g
        assert np.array_equal(indptr, ip[lo:hi + 1] - ip[lo]), g
        assert np.array_equal(indices, ref['indices'][ip[lo]:ip[hi]]), g
        assert np.array_equal(counts, ref['data'][ip[lo]:ip[hi]]), g
    return want_splits


def arena_region(ptrs, g, off, n, dtype):
    from bin3c_b200 import dist
    return dist._device_view(ptrs[g] + off, n, dtype).cpu().numpy()


def check_arena_regions(dev, m, engines, res, ptrs, cap, min_len=1000, min_sig=3):
    """Every rank puts its block mask and a float64 slice into all arenas: afterwards every arena holds the whole
    mask (the oracle's) and the whole vector."""
    import torch
    from oracle import oracle
    n, W = m['n'], len(engines)
    offs = (C.c_int64 * 4)()
    dev.check(dev.lib.b3c_xa_offsets(n, cap, offs))
    vec = torch.from_numpy(np.random.default_rng(n).uniform(-3.0, 3.0, n)).cuda()
    for g, (e, r) in enumerate(zip(engines, res)):
        if r['block'] is None:
            continue
        lo = r['block'].row_lo
        mask = e.block_mask(r['block'], min_len, min_sig)
        dev.check(dev.lib.b3c_peer_put(ptrs, W, int(offs[0]) + lo, dev._ptr(mask), mask.numel(), dev._stream()))
        xs = vec[lo:lo + r['block'].n].contiguous()
        dev.check(dev.lib.b3c_peer_put(ptrs, W, int(offs[1]) + 8 * lo, dev._ptr(xs), 8 * xs.numel(), dev._stream()))
        torch.cuda.synchronize()                       # the pool's mask buffer is the next rank's too
    ref = m['ref']
    seq = sp.csr_matrix((ref['data'], ref['indices'], ref['indptr']), shape=(n, n))
    want_mask = oracle.acceptance_mask(m['lengths'], seq, min_len, min_sig)
    assert 0 < want_mask.sum() < n
    for g in range(W):
        assert np.array_equal(arena_region(ptrs, g, int(offs[0]), n, torch.uint8).astype(bool), want_mask), g
        assert np.array_equal(arena_region(ptrs, g, int(offs[1]), n, torch.float64), vec.cpu().numpy()), g


def uneven_owner(rng, m_len, W, empty=()):
    """Source rank of every record: weights 1, 2, ..., W shuffled, sources in `empty` get nothing."""
    w = rng.permutation(np.arange(1, W + 1)).astype(np.float64)
    w[list(empty)] = 0.0
    return rng.choice(W, m_len, p=w / w.sum())


# name: (W, n, pairs, heavy rows, idle sources, records)
PEER_CASES = {
    'w2_tail_chunk': (2, 5000, 150000, (1023, 1024), (), 'native'),
    'w3_heavy_at_split': (3, 9000, 200000, (1023, 1024, 'split'), (), 'native'),
    'w5_idle_source': (5, 12000, 200000, (7000,), (2,), 'native'),
    'w3_narrow_and_split_records': (3, 7000, 150000, (1024,), (), 'mixed'),
    'w8_few_keys_one_heavy_row': (8, 8 * 1024 + 500, 4000, (100,), (), 'native'),
    'w8_fewer_chunks_than_ranks': (8, 3000, 80000, (1023,), (6,), 'native'),
    'w5_fewer_chunks_than_ranks': (5, 4 * 1024 + 7, 60000, (), (), 'mixed'),
}


def peer_case(name):
    W, n, p, heavy, empty, kind = PEER_CASES[name]
    seed = sum(map(ord, name))
    rows = [r for r in heavy if r != 'split']
    if 'split' in heavy:
        # a heavy row right at a cut: place it at the first split of the map without it, then make sure it still is
        base = make_map(n, p, seed, rows)
        dk, _ = R.directed_keys(base['ti'], base['tj'], base['ok'], base['index'], n)
        s = ref_splits(dk, R.key_bits(n), n, W)[1]
        rows.append(s)
    m = make_map(n, p, seed, rows)
    dk, _ = R.directed_keys(m['ti'], m['tj'], m['ok'], m['index'], n)
    splits = ref_splits(dk, R.key_bits(n), n, W)
    if 'split' in heavy:
        assert any(r in splits or r + 1 in splits for r in rows[-1:]), (rows, splits)
    return m, W, empty, kind, splits


@pytest.mark.parametrize('name', sorted(PEER_CASES))
def test_peer_accumulation(dev, name):
    m, W, empty, kind, splits = peer_case(name)
    rng = np.random.default_rng(W)
    owner = uneven_owner(rng, len(m['ti']), W, empty)
    if 'fewer_chunks' in name:
        assert any(lo == hi for lo, hi in zip(splits[:-1], splits[1:]))       # some ranks own no rows
    cap = 2 * len(m['ti']) + 1024
    engines = engines_for(m, W, cap)
    adds = (mixed_adds if kind == 'mixed' else native_adds)(dev, m, owner, W)
    with arenas(dev, m['n'], cap, W) as ptrs:
        res = peer_accumulate(dev, engines, ptrs, adds)
        check_accumulation(m, res, W)
        check_arena_regions(dev, m, engines, res, ptrs, cap)


def test_peer_accumulation_receive_overflow_then_recovery(dev):
    """Every source fits its own keys, but each owner receives about both directions of everybody's: more than the
    capacity.  The owner's reduce_block reports B3C_ERR_CAPACITY with the count; a second run in the same workspaces
    and arenas with room is exact (b3c_shard_publish clears the overflow word)."""
    from bin3c_b200._cabi import B3C_ERR_CAPACITY
    W = 2
    m = make_map(5000, 120000, 91)
    rng = np.random.default_rng(91)
    owner = rng.integers(0, W, len(m['ti']))
    n, b = m['n'], R.key_bits(m['n'])
    local = [len(R.directed_keys(m['ti'][owner == g], m['tj'][owner == g], m['ok'][owner == g], m['index'], n)[0]) // 2
             for g in range(W)]
    dk, _ = R.directed_keys(m['ti'], m['tj'], m['ok'], m['index'], n)
    splits = ref_splits(dk, b, n, W)
    received = [int(((dk >> b >= lo) & (dk >> b < hi)).sum()) for lo, hi in zip(splits[:-1], splits[1:])]
    cap = max(local) + 16
    assert all(r > cap for r in received)
    engines = engines_for(m, W, cap)
    with arenas(dev, n, cap, W) as ptrs:
        res = peer_accumulate(dev, engines, ptrs, native_adds(dev, m, owner, W))
        for g, r in enumerate(res):
            assert r['rc'] == B3C_ERR_CAPACITY, (g, r)
            assert r['msg'] == 'received {} directed keys, accumulator capacity is {}'.format(received[g], cap)
        # a third of the records: every owner's share fits
        keep = rng.random(len(m['ti'])) < 0.3
        small = make_subset(m, keep)
        res = peer_accumulate(dev, engines, ptrs, native_adds(dev, small, owner[keep], W))
        check_accumulation(small, res, W)


def make_subset(m, keep):
    s = dict(m)
    s['ti'], s['tj'], s['ok'] = m['ti'][keep], m['tj'][keep], m['ok'][keep]
    s['ref'] = R.ref_accumulate(s['ti'], s['tj'], s['ok'], m['index'], m['n'])
    return s


def test_peer_accumulation_replay(dev):
    """Runs in the same workspaces and arenas with two record splits, with the sort-reduce replayed as a CUDA graph
    (one per workspace and arena) and launched directly: every block exact, hence identical."""
    W = 3
    m = make_map(9000, 150000, 17, (4000,))
    rng = np.random.default_rng(17)
    owners = [uneven_owner(rng, len(m['ti']), W), rng.integers(0, W, len(m['ti']))]
    cap = 2 * len(m['ti']) + 1024
    engines = engines_for(m, W, cap)
    blocks = []
    with arenas(dev, m['n'], cap, W) as ptrs:
        for graphs in (1, 0, 1):
            dev.check(dev.lib.b3c_set_option(OPT_USE_GRAPHS, graphs))
            for owner in owners:
                res = peer_accumulate(dev, engines, ptrs, native_adds(dev, m, owner, W))
                check_accumulation(m, res, W)
                blocks.append([r['host'] for r in res])
    for other in blocks[1:]:
        for a, b in zip(blocks[0], other):
            assert all(np.array_equal(x, y) for x, y in zip(a, b))


def test_shard_scatter_refuses_too_many_chunks(dev):
    n = XA_MAX_CHUNKS * CHUNK + 1
    acc = dev.Accumulator(n, np.arange(n, dtype=np.int32), 64)
    d_splits = dev.to_device(np.zeros(16, np.int32))
    with arenas(dev, n, acc.capacity, 2) as ptrs:
        with pytest.raises(AssertionError) as ei:
            dev.check(dev.lib.b3c_shard_scatter(dev._ptr(acc.ws), ptrs, 0, 2, dev._ptr(d_splits), dev._stream()))
    assert str(ei.value) == 'sharded accumulation supports at most {} row chunks ({} contigs)'.format(
        XA_MAX_CHUNKS, XA_MAX_CHUNKS * CHUNK)


# =================================================================================================
# B. the row-block KR phase loop
# =================================================================================================

class Views(list):
    """Per-rank views of one vector (`u`) or of rows of the partials (`part`, a slice of PA..PG2)."""

    def __init__(self, items, what):
        list.__init__(self, items)
        self.what = what


class _Parts(object):
    def __init__(self, engines):
        self.engines = engines

    def __getitem__(self, idx):
        return Views([e.part[idx] for e in self.engines], idx)


class LockstepEngine(object):
    """One engine per virtual rank; every call goes to all of them in rank order.  Blocks, normalised blocks and
    balanced blocks are lists with one entry per rank.  kr_scalar records the state after every scalar step (all
    ranks must agree)."""

    def __init__(self, engines, splits):
        self.engines = engines
        self.splits = [int(s) for s in splits]
        self.trace = []

    @property
    def n(self):
        return self.engines[0].n

    def site_norm(self, blocks):
        return [e.site_norm(b) for e, b in zip(self.engines, blocks)]

    def kr_setup(self, blocks, tol, delta, Delta, max_iter):
        for e, b in zip(self.engines, blocks):
            e.kr_setup(b, tol, delta, Delta, max_iter)

    def kr_phase(self, phase):
        for e in self.engines:
            e.kr_phase(phase)

    def kr_scalar(self, which):
        for e in self.engines:
            e.kr_scalar(which)
        st = self.kr_state()
        self.trace.append((which, st['state'], st['k'], st['outer'], st['n_spmv']))

    def kr_state(self):
        sts = [e.kr_state() for e in self.engines]
        keys = ('state', 'status', 'n_iter', 'k', 'outer', 'n_spmv')
        for g, st in enumerate(sts[1:], 1):
            assert {k: int(st[k]) for k in keys} == {k: int(sts[0][k]) for k in keys}, (g, st, sts[0])
        out = {k: int(sts[0][k]) for k in keys}
        out['zero_diag'] = sum(int(st['zero_diag']) for st in sts)
        return out

    @property
    def u(self):
        return Views([e.u for e in self.engines], 'u')

    @property
    def part(self):
        return _Parts(self.engines)

    @property
    def x(self):
        """The scale vector assembled from every rank's own rows."""
        import torch
        x0 = self.engines[0].x
        x = torch.zeros(self.n, dtype=torch.float64, device=x0.device)
        for e, lo, hi in zip(self.engines, self.splits[:-1], self.splits[1:]):
            x[lo:hi] = e.x[lo:hi]
        return x

    def kr_apply(self, blocks, x):
        return [e.kr_apply(b, x) for e, b in zip(self.engines, blocks)]

    def compress_edges(self, blocks, mask, reduce_max, scale=True):
        """Two passes: the first records each rank's block maximum, the second runs with the global one filled in."""
        vmax = []
        for e, b in zip(self.engines, blocks):
            e.compress_edges(b, mask, lambda t: vmax.append(float(t.cpu()[0])), scale=scale)
        g = max(vmax)
        out = []
        for e, b in zip(self.engines, blocks):
            r = e.compress_edges(b, mask, lambda t: t.fill_(g), scale=scale)
            out.append({k: r[k].cpu().numpy().copy() for k in ('u', 'v', 'w')})
        return out

    def synchronize(self):
        import torch
        torch.cuda.synchronize()


class LockstepComm(object):
    """world == 1 to the driver.  An all-reduce of per-rank views first checks the phase contract exactly -- u is 0.0
    outside the rank's rows, the sum partials 0.0 and the minimum partials +inf in chunks it does not own -- then
    reduces in rank order and writes the result into every rank's view."""
    rank, world = 0, 1

    def __init__(self, splits):
        self.splits = [int(s) for s in splits]
        self.checked = 0

    def all_reduce(self, t, op='sum'):
        if not isinstance(t, Views):
            return t                                     # already global (the lockstep engine sums zero_diag)
        import torch
        for g, v in enumerate(t):
            lo, hi = self.splits[g], self.splits[g + 1]
            if t.what == 'u':
                outside = torch.cat([v[:lo], v[hi:]])
                assert bool((outside == 0.0).all()), ('u outside the rows of rank', g)
            else:
                rows = range(7)[t.what]
                rows = [rows] if isinstance(rows, int) else list(rows)
                vv = v.view(len(rows), -1)
                nc = vv.shape[1]
                own = torch.zeros(nc, dtype=torch.bool, device=v.device)
                own[lo // CHUNK:-(-hi // CHUNK)] = True
                for i, p in enumerate(rows):
                    ident = 0.0 if p <= PC else float('inf')
                    assert bool((vv[i][~own] == ident).all()), ('partial', p, 'of rank', g, vv[i][~own])
        self.checked += 1
        acc = t[0].clone()
        for v in t[1:]:
            acc = acc + v if op == 'sum' else torch.minimum(acc, v)
        for v in t:
            v.copy_(acc)
        return t

    def barrier(self):
        pass


def count_blocks(indptr, indices, counts, splits):
    """Row blocks [(local indptr, indices, counts)] of a whole count CSR."""
    return [(indptr[lo:hi + 1] - indptr[lo], indices[indptr[lo]:indptr[hi]], counts[indptr[lo]:indptr[hi]])
            for lo, hi in zip(splits[:-1], splits[1:])]


def device_blocks(dev, blocks, splits, n, counts=True):
    import torch
    out = []
    for (ip, ix, d), lo in zip(blocks, splits[:-1]):
        data = dev.to_device(np.asarray(d, np.uint32).view(np.int32)) if counts else \
            dev.to_device(np.asarray(d, np.float64))
        out.append(dev.DeviceCSR(len(ip) - 1, dev.to_device(np.asarray(ip, np.int64)),
                                 dev.to_device(np.asarray(ix, np.int32)) if len(ix) else
                                 torch.empty(0, dtype=torch.int32, device='cuda'),
                                 data, counts=counts, row_lo=lo, n_total=n))
    return out


def numpy_blocks(blocks, splits, n):
    from np_engine import Block
    return [Block(sp.csr_matrix((np.asarray(d), np.asarray(ix), np.asarray(ip)), shape=(len(ip) - 1, n)), lo, n)
            for (ip, ix, d), lo in zip(blocks, splits[:-1])]


def sym_counts(n, seed, nnz_row=12, regions=(), empty=(), zero_diag=(), heavy=()):
    """Symmetric n x n uint32 counts: ~nnz_row random off-diagonal entries per row, plus, for every (lo, hi, k) in
    `regions`, about k more per row with both ends in [lo, hi); rows in `empty` hold nothing, rows in `zero_diag` no
    diagonal, each row in `heavy` is linked to a tenth of all rows.  Returns the CSR (indptr, indices, counts)."""
    rng = np.random.default_rng(seed)
    parts = [(rng.integers(0, n, n * nnz_row // 2), rng.integers(0, n, n * nnz_row // 2))]
    for lo, hi, k in regions:
        m = (hi - lo) * k // 2
        parts.append((rng.integers(lo, hi, m), rng.integers(lo, hi, m)))
    for r in heavy:
        c = rng.choice(n, n // 10, replace=False)
        parts.append((np.full(len(c), r), c))
    a = np.concatenate([p[0] for p in parts]).astype(np.int64)
    b = np.concatenate([p[1] for p in parts]).astype(np.int64)
    drop = np.zeros(n, bool)
    drop[list(empty)] = True
    keep = (a != b) & ~drop[a] & ~drop[b]
    key = np.unique(np.minimum(a, b)[keep] * n + np.maximum(a, b)[keep])
    cnt = K.small_counts(rng, len(key), hi=500).astype(np.int64)
    d = np.flatnonzero(~drop)
    nd = np.zeros(n, bool)
    nd[list(zero_diag)] = True
    d = d[~nd[d]]
    dc = K.small_counts(rng, len(d), hi=500).astype(np.int64)
    row = np.concatenate([key // n, key % n, d])
    col = np.concatenate([key % n, key // n, d])
    return K.csr_from_keys(n, row, col, np.concatenate([cnt, cnt, dc]).astype(np.uint32))


def sites_of(n, seed):
    rng = np.random.default_rng(seed)
    s = rng.integers(2, 40, n).astype(np.int32)
    s[rng.random(n) < 0.1] = 0
    return s


def normed_whole(indptr, indices, counts, sites, n):
    from oracle import oracle
    row = K.row_of_entry(indptr)
    data = oracle.norm_by_sites(row, indices, np.asarray(counts).astype(np.float64), oracle.get_sites(sites))
    return sp.csr_matrix((data, indices, indptr), shape=(n, n))


def run_lockstep(engines, blocks, splits, params, normalise=True):
    """site_norm (optional) + kr_setup + dist.kr_block_loop over the virtual ranks; returns (engine, comm, state)."""
    from bin3c_b200 import dist
    eng, comm = LockstepEngine(engines, splits), LockstepComm(splits)
    normed = eng.site_norm(blocks) if normalise else blocks
    eng.kr_setup(normed, *params)
    st = dist.kr_block_loop(eng, comm)
    assert comm.checked > 0
    return eng, comm, st


def cuda_engines(n, sites, W):
    from bin3c_b200 import dist
    return [dist.CudaEngine(np.arange(n, dtype=np.int32), np.full(n, 5000, np.int32), sites, 1024) for _ in range(W)]


def numpy_engines(n, sites, W):
    from np_engine import NumpyEngine
    return [NumpyEngine(np.arange(n), np.full(n, 5000), sites, 1024) for _ in range(W)]


# name: (n, splits, matrix builder kwargs)
KR_CASES = {
    'w2_tail_alone': (1500, [0, 1024, 1500], dict(zero_diag=(3, 1200))),
    'w3_tail_next_to_full': (4 * 1024 + 300, [0, 2048, 4096, 4396], dict(zero_diag=(10, 2100, 4390), heavy=(4100,))),
    'w4_one_chunk_block_and_empty_rows': (12000, [0, 1024, 3072, 9216, 12000],
                                          dict(empty=range(4000, 7000), zero_diag=(0, 1500, 10000))),
    'w8_heavy_row': (8 * 1024 + 77, [0, 1024, 2048, 3072, 4096, 5120, 6144, 7168, 8269],
                     dict(heavy=(2047,), zero_diag=(5, 3000, 8200))),
}


@pytest.mark.parametrize('name', sorted(KR_CASES))
def test_kr_block_loop(dev, name):
    from oracle import oracle
    n, splits, kw = KR_CASES[name]
    W = len(splits) - 1
    indptr, indices, counts = sym_counts(n, sum(map(ord, name)), **kw)
    sites = sites_of(n, len(name))
    whole = normed_whole(indptr, indices, counts, sites, n)
    want = oracle.kr_scale_vector(whole)
    blocks = count_blocks(indptr, indices, counts, splits)
    params = (1e-6, 0.1, 3.0, 1000)
    eng, comm, st = run_lockstep(cuda_engines(n, sites, W), device_blocks(dev, blocks, splits, n), splits, params)
    ref_eng, _, ref_st = run_lockstep(numpy_engines(n, sites, W), numpy_blocks(blocks, splits, n), splits, params)
    assert eng.trace == ref_eng.trace
    assert st['status'] == 0 and st['state'] == 0
    x1, info = dev.kr_scale_vector(dev.DeviceCSR.from_scipy(whole))
    assert st['n_iter'] == want.n_iter == info['n_iter'] == ref_st['n_iter']
    assert st['zero_diag'] == want.n_zero_diag
    x = eng.x.cpu().numpy()
    for lo, hi in zip(splits[:-1], splits[1:]):
        assert _relerr(x[lo:hi], want.x[lo:hi]) <= REL_TOL, (lo, hi)
    if kw.get('empty'):
        e = list(kw['empty'])
        assert np.all(np.diff(indptr)[e] == 0) and np.allclose(want.x[e], 1.0)


def test_kr_block_loop_slab_and_gather_blocks(dev):
    """512-column slabs (18 slabs for 9000 columns, more than the 16 of B3C_OPT_KR_MAX_SLABS): the dense rows [0, 4096)
    keep the slab form by the dense-cell rule, the sparse block [4096, 9000) takes the gather form -- in one solve."""
    from oracle import oracle
    from bin3c_b200 import _cabi
    n, splits = 9000, [0, 4096, 9000]
    dev.check(dev.lib.b3c_set_option(OPT_KR_SLAB_WIDTH, 512))
    indptr, indices, counts = sym_counts(n, 29, nnz_row=16, regions=[(0, 4096, 250)], zero_diag=(7, 5000))
    sites = sites_of(n, 29)
    blocks = count_blocks(indptr, indices, counts, splits)
    forms = []
    for (ip, _, _), lo, hi in zip(blocks, splits[:-1], splits[1:]):
        nnz = int(ip[-1])
        plan = []
        for rows in (hi - lo, n):                        # the block's rows, and the whole matrix's
            h = (C.c_int64 * 5)()
            _cabi.check(_cabi.lib.b3c_kr_plan(n, nnz, rows, 0, h))
            assert (int(h[0]), int(h[1]), int(h[2])) == K.form_rule(n, nnz, rows, False, width=512), (lo, rows)
            plan.append(int(h[0]))
        assert plan[0] == plan[1], (lo, plan)
        forms.append(plan[0])
    assert forms == [18, 0], forms
    whole = normed_whole(indptr, indices, counts, sites, n)
    want = oracle.kr_scale_vector(whole)
    params = (1e-6, 0.1, 3.0, 1000)
    eng, _, st = run_lockstep(cuda_engines(n, sites, 2), device_blocks(dev, blocks, splits, n), splits, params)
    ref_eng, _, _ = run_lockstep(numpy_engines(n, sites, 2), numpy_blocks(blocks, splits, n), splits, params)
    assert eng.trace == ref_eng.trace
    assert st['status'] == 0 and st['n_iter'] == want.n_iter and st['zero_diag'] == want.n_zero_diag
    assert _relerr(eng.x.cpu().numpy(), want.x) <= REL_TOL


# ---- outcomes other than convergence, through kr_block_loop and ShardedHotPath.balance() ------------------------

def lockstep_path(engines, blocks, splits, n, sites, max_iter=1000, Delta=3.0):
    """ShardedHotPath on the lockstep engine and comm, host-driven KR, torch.distributed-style exchanges, with the row
    blocks set as the accumulation would leave them."""
    from bin3c_b200.dist import ShardedHotPath
    eng, comm = LockstepEngine(engines, splits), LockstepComm(splits)
    hp = ShardedHotPath(np.arange(n, dtype=np.int32), np.full(n, 5000, np.int32), sites, 1024, Delta=Delta,
                        max_iter=max_iter, comm=comm, engine=eng, host_driven_kr=True, peer_exchange=False)
    hp.block, hp.splits = blocks, np.asarray(splits, dtype=np.int32)
    return hp


def float_blocks(dev, m, splits):
    m = sp.csr_matrix(m)
    m.sort_indices()
    ip, ix, d = m.indptr.astype(np.int64), m.indices.astype(np.int32), m.data
    return device_blocks(dev, count_blocks(ip, ix, d, splits), splits, m.shape[0], counts=False)


def kr_error(fn):
    try:
        fn()
    except Exception as e:                              # noqa: BLE001 -- the type is what is compared
        return type(e), str(e)
    return None


@pytest.mark.parametrize('splits', [[0, 2048, 5000], [0, 1024, 3072, 5000]], ids=['w2', 'w3'])
def test_kr_block_loop_exact_tie(dev, splits):
    """Q13 over row blocks: A = 0.125 I makes ynew = 4.5 in every row on the first CG step, so Delta = 4.5 is an exact
    tie -- every rank ends with B3C_ERR_TIE, and balance() raises what b3c_kr_run raises.  One ulp either side is
    not an error and agrees with the oracle."""
    from oracle import oracle
    from bin3c_b200._cabi import B3C_ERR_TIE
    n, W = 5000, len(splits) - 1
    m = sp.identity(n, format='csr', dtype=np.float64) * 0.125
    ones = np.ones(n, np.int32)
    for Delta in (4.5, np.nextafter(4.5, 0.0), np.nextafter(4.5, 9.0)):
        eng, _, st = run_lockstep(cuda_engines(n, ones, W), float_blocks(dev, m, splits), splits,
                                  (1e-6, 0.1, Delta, 1000), normalise=False)
        sts = [e.kr_state() for e in eng.engines]
        if Delta == 4.5:
            assert all(s['status'] == B3C_ERR_TIE for s in sts)
            want = kr_error(lambda: dev.kr_scale_vector(dev.DeviceCSR.from_scipy(m), Delta=Delta))
            assert want is not None and want[0] is ValueError
            with pytest.raises(ValueError):
                oracle.kr_scale_vector(m, Delta=Delta)
            hp = lockstep_path(cuda_engines(n, ones, W), float_blocks(dev, m, splits), splits, n, ones, Delta=Delta)
            assert kr_error(hp.balance) == want
        else:
            res = oracle.kr_scale_vector(m, Delta=Delta)
            assert all(s['status'] == 0 for s in sts) and st['n_iter'] == res.n_iter
            assert _relerr(eng.x.cpu().numpy(), res.x) <= REL_TOL


@pytest.fixture(scope='module')
def c1mini_normed():
    from oracle import oracle
    from bin3c_b200 import synth
    g = load_golden('c1mini')
    ti, tj, ok = synth.unpack_pairs(g['records'])
    up, _ = oracle.bin_pairs_fast(ti, tj, ok, golden_lut(g), len(g['lengths']))
    sm = oracle.symmetrise(up)
    s = oracle.get_sites(g['sites'])
    return sp.coo_matrix((oracle.norm_by_sites(sm.row, sm.col, sm.data.astype(np.float64), s), (sm.row, sm.col)),
                         shape=sm.shape).tocsr()


@pytest.mark.parametrize('max_iter', [1, 2, 3, 5, 8, 13])
def test_kr_block_loop_max_iter(dev, c1mini_normed, max_iter):
    """The outer loop stops once n_iter >= max_iter; n_iter > max_iter raises.  Over two row blocks: the same outcome
    and n_iter as the oracle, and balance() raises exactly what dev.kr_scale_vector raises."""
    from oracle import oracle
    m = c1mini_normed
    n = m.shape[0]
    splits = [0, CHUNK, n] if n > CHUNK else None
    assert splits is not None, n
    ones = np.ones(n, np.int32)
    try:
        res, want_err = oracle.kr_scale_vector(m, max_iter=max_iter), None
    except RuntimeError as e:
        res, want_err = None, str(e)
    eng, _, st = run_lockstep(cuda_engines(n, ones, 2), float_blocks(dev, m, splits), splits,
                              (1e-6, 0.1, 3.0, max_iter), normalise=False)
    dev_err = kr_error(lambda: dev.kr_scale_vector(dev.DeviceCSR.from_scipy(m), max_iter=max_iter))
    hp = lockstep_path(cuda_engines(n, ones, 2), float_blocks(dev, m, splits), splits, n, ones, max_iter=max_iter)
    path_err = kr_error(hp.balance)
    if want_err is not None:
        assert st['n_iter'] > max_iter
        assert dev_err == (RuntimeError, want_err) and path_err == dev_err
    else:
        assert dev_err is None and path_err is None
        assert st['status'] == 0 and st['n_iter'] == res.n_iter
        assert _relerr(eng.x.cpu().numpy(), res.x) <= REL_TOL
        assert _relerr(hp.x.cpu().numpy(), res.x) <= REL_TOL


def test_kr_block_loop_nan_in_one_block(dev):
    """A NaN in the last rank's block: every rank stops with B3C_ERR_NAN, and balance() raises what
    dev.kr_scale_vector raises for the whole matrix."""
    from bin3c_b200._cabi import B3C_ERR_NAN
    n, splits = 5000, [0, 1024, 3072, 5000]
    rng = np.random.default_rng(3)
    up = sp.triu(sp.random(n, n, density=0.004, random_state=rng, data_rvs=lambda k: rng.uniform(0.1, 5.0, k)), k=1)
    m = (up + up.T + sp.diags(rng.uniform(0.5, 2.0, n))).tocsr()
    m.sort_indices()
    at = m.indptr[4000]
    m.data[at] = np.nan
    ones = np.ones(n, np.int32)
    eng, _, st = run_lockstep(cuda_engines(n, ones, 3), float_blocks(dev, m, splits), splits,
                              (1e-6, 0.1, 3.0, 1000), normalise=False)
    assert all(e.kr_state()['status'] == B3C_ERR_NAN for e in eng.engines)
    want = kr_error(lambda: dev.kr_scale_vector(dev.DeviceCSR.from_scipy(m)))
    assert want == (RuntimeError, 'scale vector has developed invalid values (NANs)!')
    hp = lockstep_path(cuda_engines(n, ones, 3), float_blocks(dev, m, splits), splits, n, ones)
    assert kr_error(hp.balance) == want


# =================================================================================================
# C. the whole sharded path on virtual ranks
# =================================================================================================

@pytest.mark.parametrize('cfg,W', [('CFG', 2), ('BIG', 8)])
def test_sharded_path_virtual_ranks(dev, cfg, W):
    """Peer accumulation -> block masks through b3c_peer_put -> site_norm -> balance() -> kr_apply -> compress_edges
    over W virtual ranks: the one-GPU stand-in for test_gpu_dist.test_sharded_path_ranks, with its bars."""
    import torch
    import test_gpu_dist as D
    from bin3c_b200 import dist, synth
    com = synth.make_community(**getattr(D, cfg))
    n, min_sig = com.n_contigs, 3
    per = -(-com.n_pairs // W)
    per += per & 1
    cap = int(2.5 * per) + 1024
    engines = [dist.CudaEngine(com.tid2idx(), com.lengths, com.sites, cap) for _ in range(W)]
    recs = [dev.to_device(com.records[g * per:(g + 1) * per]) for g in range(W)]
    adds = [(lambda r: (lambda e: e.add_records(r)))(r) for r in recs]
    offs = (C.c_int64 * 4)()
    dev.check(dev.lib.b3c_xa_offsets(n, cap, offs))
    with arenas(dev, n, cap, W) as ptrs:
        res = peer_accumulate(dev, engines, ptrs, adds)
        assert all(r['rc'] == 0 and r['block'] is not None for r in res)
        splits = res[0]['d_splits']
        for g, (e, r) in enumerate(zip(engines, res)):
            mask = e.block_mask(r['block'], 1000, min_sig)
            dev.check(dev.lib.b3c_peer_put(ptrs, W, int(offs[0]) + r['block'].row_lo, dev._ptr(mask), mask.numel(),
                                           dev._stream()))
            torch.cuda.synchronize()
        masks = [arena_region(ptrs, g, int(offs[0]), n, torch.uint8) for g in range(W)]
        assert all(np.array_equal(mk, masks[0]) for mk in masks)
        hp = lockstep_path(engines, [r['block'] for r in res], splits, n, com.sites)
        hp.min_sig = min_sig
        hp.mask = torch.from_numpy(masks[0]).cuda()
        hp.balance()
        edges = hp.edges()
        x = hp.x.cpu().numpy()
        parts = []
        for g, r in enumerate(res):
            indptr, indices, data = r['host']
            row = np.repeat(np.arange(r['block'].n), np.diff(indptr)) + r['block'].row_lo
            sz = r['sizes']
            parts.append(dict(row=row, col=indices, data=data, mask=masks[g], x=x, n_iter=hp.kr_info['n_iter'],
                              counts=np.array(sz[3:6]), **edges[g]))
    D._check(parts, com, min_sig)
