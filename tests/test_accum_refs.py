"""
CPU checks of the pair-accumulation reference that tests/test_gpu_accum.py holds the device to, and of the plan hook
(b3c_accum_plan) that names the code path each device case takes.

The reference is plain NumPy: it decodes native and narrow records with its own bit arithmetic, maps reference ids to
contig indices (an id beyond the table, a LUT value < 0 or >= n_seq: excluded), applies the matcher bit, counts the
diagonal, reduces the off-diagonal keys min * 2^b + max with np.unique and builds the upper and the symmetric CSR
(int64 indptr, sorted int32 columns, uint32 counts) with the counters and map_weight of ContactMap._bin_map.  Here it
is checked against the oracle (oracle.bin_pairs_fast + oracle.symmetrise) on the golden cases and on seeded maps, and
its narrow decoder against the host packer (bam_io.pack_records / unpack_records / split_records).
"""
import ctypes

import numpy as np
import pytest

from conftest import golden_lut

TID = np.uint64(0x7fffffff)
CLS_WTILE = 128                   # accum.cu: records per warp tile of k_classify
RS_BITS = 9                       # accum.cu: widest radix digit


# ---------------------------------------------------------------------------------------------
# records
# ---------------------------------------------------------------------------------------------

def pack_native(ti, tj, ok, bit63=None):
    """(tid1, tid2, matcher) -> native 8-byte records: tid1 in bits 0..30, matcher bit 31, tid2 in bits 32..62.
    bit63: bit 63 set where true (not part of any field; the accumulation must ignore it)."""
    r = np.asarray(ti, dtype=np.uint64) | (np.asarray(tj, dtype=np.uint64) << np.uint64(32))
    r |= np.asarray(ok, dtype=bool).astype(np.uint64) << np.uint64(31)
    if bit63 is not None:
        r |= np.asarray(bit63, dtype=bool).astype(np.uint64) << np.uint64(63)
    return r


def decode_native(rec):
    rec = np.asarray(rec, dtype=np.uint64)
    return ((rec & TID).astype(np.int64), ((rec >> np.uint64(32)) & TID).astype(np.int64),
            ((rec >> np.uint64(31)) & np.uint64(1)).astype(bool))


def narrow_fields(B, same):
    """(id bits per field, all-ones marker) of a B-byte pair record or same-reference record."""
    tb = 8 * B - 1 if same else (8 * B - 1) // 2
    return tb, (1 << tb) - 1


def pack_narrow(ti, tj, ok, B, same=False):
    """Narrow records written bit by bit: pair records hold tid1 in bits [0, tb), the matcher in bit tb and tid2 in
    bits [tb + 1, 2 tb + 1), tb = (8 B - 1) // 2; same-reference records hold one id in bits [0, 8 B - 1) and the
    matcher in the top bit.  Ids must fit the field (the marker, all ones, included).  Padded to 8 bytes."""
    tb, marker = narrow_fields(B, same)
    ti = np.asarray(ti, dtype=np.uint64)
    tj = np.asarray(tj, dtype=np.uint64)
    assert ti.size == 0 or (int(ti.max()) <= marker and int(tj.max()) <= marker)
    if same:
        assert np.array_equal(ti, tj)
        v = ti | (np.asarray(ok, dtype=bool).astype(np.uint64) << np.uint64(tb))
    else:
        v = ti | (np.asarray(ok, dtype=bool).astype(np.uint64) << np.uint64(tb)) | (tj << np.uint64(tb + 1))
    n = len(v)
    out = np.zeros((n * B + 7) // 8 * 8, dtype=np.uint8)
    for k in range(B):
        out[k:n * B:B] = ((v >> np.uint64(8 * k)) & np.uint64(0xff)).astype(np.uint8)
    return out


def decode_narrow(buf, n, B, same=False):
    """Narrow records -> (tid1, tid2, matcher) as the device widens them: the marker stays all ones of the field."""
    tb, marker = narrow_fields(B, same)
    b = np.asarray(buf, dtype=np.uint8)
    v = np.zeros(n, dtype=np.uint64)
    for k in range(B):
        v |= b[k:n * B:B].astype(np.uint64) << np.uint64(8 * k)
    m = np.uint64(marker)
    t1 = (v & m).astype(np.int64)
    t2 = t1.copy() if same else ((v >> np.uint64(tb + 1)) & m).astype(np.int64)
    return t1, t2, ((v >> np.uint64(tb)) & np.uint64(1)).astype(bool)


def narrow_to_native(ti, tj, ok, B, same=False):
    """Decoded narrow fields -> native records, the marker mapped to 0x7fffffff as the host unpacker does."""
    _, marker = narrow_fields(B, same)
    ti = np.where(ti == marker, 0x7fffffff, ti)
    tj = np.where(tj == marker, 0x7fffffff, tj)
    return pack_native(ti, tj, ok)


# ---------------------------------------------------------------------------------------------
# reference accumulation
# ---------------------------------------------------------------------------------------------

def key_bits(n_seq):
    b = 1
    while (1 << b) < n_seq:
        b += 1
    return b


def lut_index(lut, n_seq):
    """tid -> contig index through a LUT (int array; -1 excluded); -1 for ids beyond it and values >= n_seq."""
    lut = np.asarray(lut, dtype=np.int64)

    def f(t):
        t = np.asarray(t, dtype=np.int64)
        inr = t < len(lut)
        v = np.where(inr, lut[np.minimum(t, len(lut) - 1)], -1)
        return np.where((v >= 0) & (v < n_seq), v, -1)
    return f


def rank_index(keep, n_refs):
    """tid -> rank among the sorted kept ids (the dense rank map) without a table of n_refs entries."""
    keep = np.asarray(keep, dtype=np.int64)

    def f(t):
        t = np.asarray(t, dtype=np.int64)
        p = np.searchsorted(keep, t)
        hit = (p < len(keep)) & (keep[np.minimum(p, len(keep) - 1)] == t) & (t < n_refs)
        return np.where(hit, p, -1)
    return f


def csr_from_cells(n, row, col, cnt):
    o = np.lexsort((col, row))
    indptr = np.zeros(n + 1, dtype=np.int64)
    np.cumsum(np.bincount(row, minlength=n), out=indptr[1:])
    return indptr, col[o].astype(np.int32), cnt[o].astype(np.uint32)


def ref_from_cells(n_seq, off_keys, off_cnt, diag, counters, symmetric=True):
    """Unique off-diagonal keys min * 2^b + max with counts, the diagonal counts -> dict(indptr, indices, data, info)."""
    b = key_bits(n_seq)
    off_keys = np.asarray(off_keys, dtype=np.int64)
    off_cnt = np.asarray(off_cnt, dtype=np.int64)
    assert off_cnt.size == 0 or int(off_cnt.max()) < 2 ** 32
    i, j = off_keys >> b, off_keys & ((1 << b) - 1)
    d = np.flatnonzero(diag)
    rows = [i, d] + ([j] if symmetric else [])
    cols = [j, d] + ([i] if symmetric else [])
    cnts = [off_cnt, np.asarray(diag, dtype=np.int64)[d]] + ([off_cnt] if symmetric else [])
    indptr, indices, data = csr_from_cells(n_seq, np.concatenate(rows), np.concatenate(cols), np.concatenate(cnts))
    info = dict(nnz_upper=len(off_keys) + len(d), nnz_full=2 * len(off_keys) + len(d),
                map_weight=2 * int(off_cnt.sum()) + int(np.asarray(diag, dtype=np.int64).sum()), **counters)
    return dict(indptr=indptr, indices=indices, data=data, info=info)


def ref_accumulate(ti, tj, ok, index, n_seq, symmetric=True):
    """The accumulation of (tid1, tid2, matcher) with `index` (lut_index / rank_index)."""
    ii, jj = index(ti), index(tj)
    ok = np.asarray(ok, dtype=bool)
    valid = (ii >= 0) & (jj >= 0)
    acc = valid & ok
    counters = dict(accepted=int(acc.sum()), ref_excluded=int((~valid).sum()), poor_match=int((valid & ~ok).sum()))
    a, c = np.minimum(ii[acc], jj[acc]), np.maximum(ii[acc], jj[acc])
    diag = np.bincount(a[a == c], minlength=n_seq).astype(np.int64)
    b = key_bits(n_seq)
    keys, cnt = np.unique((a[a != c] << b) | c[a != c], return_counts=True)
    return ref_from_cells(n_seq, keys, cnt, diag, counters, symmetric)


def directed_keys(ti, tj, ok, index, n_seq):
    """Directed keys (row << b | col) of the accepted off-diagonal pairs, both directions, and the diagonal."""
    ii, jj = index(ti), index(tj)
    acc = (ii >= 0) & (jj >= 0) & np.asarray(ok, dtype=bool)
    a, c = ii[acc], jj[acc]
    off = a != c
    b = key_bits(n_seq)
    lo, hi = np.minimum(a[off], c[off]), np.maximum(a[off], c[off])
    return np.concatenate([(lo << b) | hi, (hi << b) | lo]), np.bincount(a[~off], minlength=n_seq)


# ---------------------------------------------------------------------------------------------
# plan: Python transcription of accum.cu plan() / radix_sort, to be held against b3c_accum_plan
# ---------------------------------------------------------------------------------------------

def _align(x, a=16):
    return (x + a - 1) // a * a


def py_plan(n_seq, n_refs):
    SMEM_MAX, WARPS, CAPW_MAX = 232448, 32, 512
    b = key_bits(n_seq)
    rw = -(-n_refs // 64)
    rank64 = _align((rw * 2 + 1) * 8)
    rank32 = _align((-(-n_refs // 12) + 1) * 4)
    rank3 = _align((rw + 1) * 8) + _align((rw + 1) * 2) + _align((rw // 32 + 2) * 4)
    diag = _align(n_seq * 4)

    def cap_w(fixed, kb):
        c = min((SMEM_MAX - fixed) // (WARPS * kb), CAPW_MAX) & ~31
        return c if c >= CLS_WTILE else 0

    def mode(other, kb):
        if b <= 20 and cap_w(other + rank32, kb) >= 256:
            return 2, rank32
        if cap_w(other + rank64, kb):
            return 1, rank64
        if b <= 20 and cap_w(other + rank32, kb):
            return 2, rank32
        if cap_w(other + rank3, kb):
            return 3, rank3
        return 0, 0
    if b <= 16 and mode(diag, 4)[0]:
        sd, (rm, rb) = True, mode(diag, 4)
        fixed, kb = rb + diag, 4
    elif b <= 16 and cap_w(diag, 4):
        sd, rm, fixed, kb = True, 0, diag, 4
    else:
        sd, (rm, rb) = False, mode(0, 8)
        fixed, kb = rb, 8
    cw, dk = cap_w(fixed, kb), 0
    if not sd:
        room = (SMEM_MAX - fixed - WARPS * CLS_WTILE * kb) // 4
        if room >= n_seq // 20 and room > 0:
            cw, dk = CLS_WTILE, min(room, n_seq)
    return dict(b=b, smem_diag=int(sd), smem_rank=rm, cap_w=cw, diag_k=dk)


def radix_shape(bits):
    """(passes, digit bits) of radix_sort over `bits` bits."""
    p = -(-bits // RS_BITS) if bits > 0 else 0
    return p, (-(-bits // p) if p else 0)


def comp_cbits(b):
    return min(64 - 2 * b, 32)


PLAN_FIELDS = ('b', 'smem_diag', 'smem_rank', 'cap_w', 'diag_k', 'key_passes', 'key_digit', 'comp_passes',
               'comp_digit', 'cbits')


def device_plan(lib, n_seq, n_refs, cap=1000):
    """b3c_accum_plan as a dict (host-only: needs the library, not a GPU)."""
    out = (ctypes.c_int64 * len(PLAN_FIELDS))()
    rc = lib.b3c_accum_plan(int(cap), int(n_seq), int(n_refs), out)
    assert rc == 0, rc
    return dict(zip(PLAN_FIELDS, (int(v) for v in out)))


def sort_shape(plan):
    """(passes, wide, parity) of the key sort and of the composite sort.  The parity of the key sort says which key
    buffer holds the sorted keys (and the composite written over them); the composite sort's, where it ends up."""
    return ((plan['key_passes'], plan['key_digit'] > 8, plan['key_passes'] & 1),
            (plan['comp_passes'], plan['comp_digit'] > 8, plan['comp_passes'] & 1))


def plan_class(plan):
    return (plan['smem_diag'], plan['smem_rank'], plan['diag_k'] > 0)


# (smem diag, rank mode, partial diag) -> (n_seq, n_refs): every reachable class of plan()
PLAN_CASES = {
    (1, 2, False): (1000, 1200),
    (1, 1, False): (2048, 819200),
    (1, 3, False): (8192, 819200),
    (1, 0, False): (4096, 1638400),
    (0, 2, True): (65536, 65536),
    (0, 2, False): (300000, 450000),
    (0, 1, True): (65536, 524288),
    (0, 1, False): (524288, 524288),
    (0, 3, True): (65536, 1048576),
    (0, 3, False): (262144, 1048576),
    (0, 0, True): (65536, 2621440),
    (0, 0, False): (1048576, 1572864),
}
# two-level table (mode 3) sizes whose bitmap word count is 1 or 31 mod 32 (the sentinel word's block)
MODE3_EDGE_CASES = [(8192, 819201), (8192, 819131), (65536, 1048577), (65536, 1048449)]

# key widths 1..28: n_seq = 2^(b-1) + 1 and 2^b (b = 1: 1 and 2; b = 28 only at 2^27 + 1)
WIDTH_CASES = sorted({(1, 1), (1, 2)} | {(b, (1 << (b - 1)) + 1) for b in range(2, 29)} |
                     {(b, 1 << b) for b in range(2, 28)})


def all_sort_shapes(max_b=28):
    """Every (passes, wide, parity) the key sort (2b bits) and the composite sort (b bits) take for b <= max_b."""
    out = set()
    for b in range(1, max_b + 1):
        for bits in (2 * b, b):
            p, d = radix_shape(bits)
            out.add((p, d > 8, p & 1))
    return out


# ---------------------------------------------------------------------------------------------
# tests
# ---------------------------------------------------------------------------------------------

def _oracle(ti, tj, ok, lut, n):
    from oracle import oracle
    up, counts = oracle.bin_pairs_fast(ti, tj, ok, lut, n)
    return up, oracle.symmetrise(up), counts


def _assert_ref_equals_oracle(ti, tj, ok, lut, n):
    up, full, counts = _oracle(ti, tj, ok, lut, n)
    for symmetric, want in ((True, full), (False, up)):
        r = ref_accumulate(ti, tj, ok, lut_index(lut, n), n, symmetric=symmetric)
        w = want.tocsr()
        w.sort_indices()
        assert np.array_equal(r['indptr'], w.indptr)
        assert np.array_equal(r['indices'], w.indices)
        assert np.array_equal(r['data'], w.data.astype(np.uint32))
        assert {k: r['info'][k] for k in counts} == counts
    assert r['info']['map_weight'] == int(full.sum(dtype=np.uint64))
    assert r['info']['nnz_full'] == full.nnz and r['info']['nnz_upper'] == up.nnz


def test_reference_matches_oracle_golden(golden):
    g = golden
    ti, tj, ok = decode_native(g['records'])
    n = len(g['lengths'])
    _assert_ref_equals_oracle(ti, tj, ok, golden_lut(g), n)
    r = ref_accumulate(ti, tj, ok, lut_index(golden_lut(g), n), n)
    assert [r['info'][k] for k in ('accepted', 'ref_excluded', 'poor_match')] == g['counts'].tolist()
    assert r['info']['map_weight'] == int(g['map_weight'])


@pytest.mark.parametrize('n,n_refs,seed', [(1, 1, 1), (2, 5, 2), (37, 45, 3), (1000, 1200, 4), (5000, 70000, 5)])
def test_reference_matches_oracle_seeded(n, n_refs, seed):
    rng = np.random.default_rng(seed)
    keep = np.sort(rng.choice(n_refs, n, replace=False))
    lut = np.full(n_refs, -1, dtype=np.int32)
    lut[keep] = rng.permutation(n)
    p = 30000
    a = rng.integers(0, n_refs + 3, p)
    b = np.where(rng.random(p) < 0.5, a, rng.integers(0, n_refs + 3, p))
    _assert_ref_equals_oracle(a, b, rng.random(p) < 0.8, lut, n)


def test_reference_rank_index_equals_lut():
    rng = np.random.default_rng(9)
    n_refs = 100000
    keep = np.sort(rng.choice(n_refs, 3000, replace=False))
    lut = np.full(n_refs, -1, dtype=np.int32)
    lut[keep] = np.arange(len(keep))
    t = np.concatenate([rng.integers(0, n_refs, 50000), keep, [n_refs, n_refs + 1, 2 ** 31 - 1]])
    assert np.array_equal(rank_index(keep, n_refs)(t), lut_index(lut, len(keep))(t))


def test_reference_excludes_lut_values_beyond_n_seq():
    lut = np.array([0, 1, 5, 2], dtype=np.int32)           # 5 >= n_seq: excluded like -1
    r = ref_accumulate([0, 2, 3, 1], [1, 1, 3, 9], [True] * 4, lut_index(lut, 3), 3)
    assert r['info'] == dict(nnz_upper=2, nnz_full=3, map_weight=3, accepted=2, ref_excluded=2, poor_match=0)


@pytest.mark.parametrize('B', [5, 6])
def test_narrow_decoder_matches_host_packer(B):
    from bin3c_b200 import bam_io
    rng = np.random.default_rng(B)
    tb, marker = narrow_fields(B, False)
    n = 4099
    ti = rng.integers(0, marker, n)
    tj = rng.integers(0, marker, n)
    ti[:tb] = 1 << np.arange(tb)                            # every id bit alone, on every byte offset
    tj[tb:2 * tb] = 1 << np.arange(tb)
    ti[-5:] = 2 ** 31 - 1                                  # beyond the field: the packer writes the marker
    ok = rng.random(n) < 0.5
    rec = pack_native(ti, tj, ok)
    packed = bam_io.pack_records(rec, B)
    assert {(i * B) % 8 for i in range(n)} == {(i * B) % 8 for i in range(8)}
    d1, d2, dok = decode_narrow(packed, n, B)
    assert np.array_equal(narrow_to_native(d1, d2, dok, B), bam_io.unpack_records(packed, n, B))
    ti[-5:] = marker
    assert np.array_equal(d1, ti) and np.array_equal(d2, tj) and np.array_equal(dok, ok)
    assert np.array_equal(pack_narrow(ti, tj, ok, B), packed)


@pytest.mark.parametrize('n_refs', [1000, (1 << 23) - 1])
def test_same_reference_decoder_matches_host_splitter(n_refs):
    from bin3c_b200 import bam_io
    rng = np.random.default_rng(n_refs)
    n = 2051
    t = rng.integers(0, n_refs, n)
    t[:30] = 1 << np.arange(30) % 23
    t[-3:] = 2 ** 31 - 1
    ok = rng.random(n) < 0.5
    rec = pack_native(t, t, ok)
    sp_ = bam_io.split_records(rec, n_refs)
    Bs = sp_.bytes_same
    assert sp_.n_same == n and Bs == bam_io.lib.b3c_records_same_bytes(n_refs)
    buf = sp_.same.numpy()
    d1, d2, dok = decode_narrow(buf, n, Bs, same=True)
    assert np.array_equal(narrow_to_native(d1, d2, dok, Bs, same=True), bam_io.unsplit_records(sp_))
    _, marker = narrow_fields(Bs, True)
    t[-3:] = marker
    assert np.array_equal(pack_narrow(t, t, ok, Bs, same=True), buf)


@pytest.fixture(scope='module')
def cabi():
    from bin3c_b200.csrc import build
    build.build()
    from bin3c_b200 import _cabi
    return _cabi


def test_plan_hook_matches_transcription(cabi):
    sizes = list(PLAN_CASES.values()) + MODE3_EDGE_CASES + [(n, n) for _, n in WIDTH_CASES] + \
        [(1, 1), (3, 1 << 20), (70000, 80000), (300000, 2400000), (1000000, 1100000), (900000, 1048576)]
    for n_seq, n_refs in sizes:
        got = device_plan(cabi.lib, n_seq, n_refs)
        want = py_plan(n_seq, n_refs)
        assert {k: got[k] for k in want} == want, (n_seq, n_refs)
        b = want['b']
        assert (got['key_passes'], got['key_digit']) == radix_shape(2 * b)
        assert (got['comp_passes'], got['comp_digit']) == radix_shape(b)
        assert got['cbits'] == comp_cbits(b)


def test_plan_cases_reach_every_class(cabi):
    for cls, (n_seq, n_refs) in PLAN_CASES.items():
        assert plan_class(device_plan(cabi.lib, n_seq, n_refs)) == cls, (cls, n_seq, n_refs)
    for n_seq, n_refs in MODE3_EDGE_CASES:
        assert device_plan(cabi.lib, n_seq, n_refs)['smem_rank'] == 3
    assert sorted(-(-r // 64) % 32 for _, r in MODE3_EDGE_CASES) == [1, 1, 31, 31]
    # plan() can reach no other class: sweep the sizes the accumulation accepts (coarsely)
    seen = set()
    for n_seq in sorted({int(x) for x in np.geomspace(1, 2 ** 28, 60)}):
        for f in (1.0, 1.2, 2.0, 8.0, 100.0, 400.0):
            n_refs = min(int(n_seq * f), 2 ** 31 - 2)
            seen.add(plan_class(py_plan(n_seq, n_refs)))
    assert seen <= set(PLAN_CASES)


def test_width_cases_reach_every_sort_shape(cabi):
    reached = set()
    for b, n_seq in WIDTH_CASES:
        plan = device_plan(cabi.lib, n_seq, n_seq)
        assert plan['b'] == b
        reached.update(sort_shape(plan))
    assert reached == all_sort_shapes(28)
    assert {radix_shape(2 * b)[0] for b in range(1, 29)} == set(range(1, 8))
