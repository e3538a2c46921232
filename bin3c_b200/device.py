"""
Device-resident stages of the contact-map hot path.

Thin host-side wrappers over the C ABI (include/bin3c_b200.h).  PyTorch tensors are used
only as device buffers and for the current CUDA stream; every operation here is a call
into hand-written sm_100a kernels -- there is no torch arithmetic on the data path and no
CPU fallback.
"""
import ctypes as C

import numpy as np
import torch

from . import _cabi
from ._cabi import lib, check


class nvtx_range(object):
    """NVTX range around a stage of the path (SURVEY.md section 5: tracing), so nsys / ncu timelines show
    `b3c:accumulate`, `b3c:mask`, `b3c:kr`, `b3c:edges` ...  A push/pop pair costs nothing measurable without a
    profiler attached."""

    def __init__(self, name):
        self.name = 'b3c:' + name

    def __enter__(self):
        torch.cuda.nvtx.range_push(self.name)
        return self

    def __exit__(self, *exc):
        torch.cuda.nvtx.range_pop()
        return False


class pipeline_stream(object):
    """
    Run a pass of the path on a capturable stream.  The sort-reduce sequences replay as CUDA graphs
    (include/bin3c_b200.h: B3C_OPT_USE_GRAPHS), and a graph cannot be captured on the legacy default stream -- which is
    what torch hands out unless the caller chose a stream.  So: if the current stream is the default one, the pass
    runs on the pipeline's own stream, ordered after everything already enqueued, and the default stream is ordered
    after the pass on exit; a caller's own stream is used as it is.
    """
    _own = {}

    def __enter__(self):
        cur = torch.cuda.current_stream()
        self._ctx = None
        if cur.cuda_stream == 0:
            d = torch.cuda.current_device()
            side = pipeline_stream._own.get(d)
            if side is None:
                side = pipeline_stream._own[d] = torch.cuda.Stream()
            side.wait_stream(cur)
            self._outer, self._side = cur, side
            self._ctx = torch.cuda.stream(side)
            self._ctx.__enter__()
        return self

    def __exit__(self, *exc):
        if self._ctx is not None:
            self._ctx.__exit__(*exc)
            self._outer.wait_stream(self._side)
        return False


def require_cuda():
    if not torch.cuda.is_available():
        raise RuntimeError('bin3c_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback')


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t):
    return C.c_void_p(0 if t is None else t.data_ptr())


def _empty(n, dtype, device=None):
    return torch.empty(max(int(n), 0), dtype=dtype, device=device or 'cuda')


class BufferPool(object):
    """
    Grow-only named device buffers, so a pipeline that runs the path repeatedly does not go through
    the allocator (or cudaMalloc) on every step.  get() returns a view of the first n elements.
    """

    def __init__(self):
        self._bufs = {}

    def get(self, name, n, dtype):
        n = max(int(n), 0)
        t = self._bufs.get(name)
        if t is None or t.dtype != dtype or t.numel() < n:
            t = torch.empty(n + n // 4 + 16, dtype=dtype, device='cuda')
            self._bufs[name] = t
        return t[:n]


def grown(t, rows, keep):
    """A larger buffer for a full one: a tensor like t with `rows` rows (dim 0), holding t's first `keep` rows."""
    g = torch.empty((int(rows),) + tuple(t.shape[1:]), dtype=t.dtype, device=t.device)
    g[:keep].copy_(t[:keep])
    return g


def _alloc(pool, name, n, dtype):
    return _empty(n, dtype) if pool is None else pool.get(name, n, dtype)


def to_device(a, dtype=None, non_blocking=False):
    """numpy array / torch tensor -> contiguous CUDA tensor (H2D copy when needed)."""
    if isinstance(a, torch.Tensor):
        t = a
    else:
        a = np.ascontiguousarray(a)
        if a.dtype == np.uint64:
            a = a.view(np.int64)
        elif a.dtype == np.uint32:
            a = a.view(np.int32)
        t = torch.from_numpy(a)
    if dtype is not None and t.dtype != dtype:
        t = t.to(dtype)
    return t.to('cuda', non_blocking=non_blocking).contiguous()


class DeviceCSR(object):
    """CSR on the device: int64 indptr[n+1], int32 indices[nnz], data[nnz] (int32 bits of uint32 counts, or float64)."""

    def __init__(self, n, indptr, indices, data, counts=False, row_lo=0, n_total=None):
        self.n = int(n)                # rows held here (a whole matrix, or a row block of one)
        self.indptr = indptr
        self.indices = indices
        self.data = data
        self.counts = counts           # True: data holds uint32 counts (stored in an int32 tensor)
        self.row_lo = int(row_lo)      # global index of the first row
        self.n_total = int(n_total) if n_total is not None else self.n     # columns / global rows

    def like(self, data, counts=False):
        """Same structure, other values."""
        return DeviceCSR(self.n, self.indptr, self.indices, data, counts=counts, row_lo=self.row_lo,
                         n_total=self.n_total)

    @property
    def nnz(self):
        return int(self.indices.numel())

    @classmethod
    def from_scipy(cls, m, dtype=np.float64):
        """Canonical CSR (duplicates summed, sorted columns) of a scipy matrix, copied to the device."""
        import scipy.sparse as sp
        c = sp.csr_matrix(m, copy=True)
        c.sum_duplicates()
        c.sort_indices()
        counts = np.dtype(dtype) == np.uint32
        return cls(c.shape[0], to_device(c.indptr.astype(np.int64)), to_device(c.indices.astype(np.int32)),
                   to_device(c.data.astype(dtype)), counts=counts)

    def host_arrays(self):
        indptr = self.indptr.cpu().numpy()
        indices = self.indices.cpu().numpy()
        data = self.data.cpu().numpy()
        if self.counts:
            data = data.view(np.uint32)
        return indptr, indices, data

    def to_scipy_csr(self):
        import scipy.sparse as sp
        indptr, indices, data = self.host_arrays()
        return sp.csr_matrix((data, indices, indptr), shape=(self.n, self.n))

    def to_scipy_coo(self):
        import scipy.sparse as sp
        indptr, indices, data = self.host_arrays()
        row = np.repeat(np.arange(self.n, dtype=np.int32), np.diff(indptr))
        return sp.coo_matrix((data, (row, indices)), shape=(self.n, self.n))


# --------------------------------------------------------------------------------------
# pair accumulation
# --------------------------------------------------------------------------------------

class Accumulator(object):
    """
    Device accumulator for packed pair records (include/bin3c_b200.h, "Pair accumulation").
    Usage: add(records) any number of times, then finish().
    """

    def __init__(self, n_seq, tid2idx, pair_capacity):
        require_cuda()
        self.n_seq = int(n_seq)
        self.tid2idx = to_device(tid2idx, torch.int32)
        self.n_refs = int(self.tid2idx.numel())
        self.capacity = int(pair_capacity)
        nbytes = lib.b3c_accum_workspace_bytes(self.capacity, self.n_seq, self.n_refs)
        if nbytes < 0:
            raise AssertionError('invalid accumulator sizes')
        self.ws = _empty(nbytes, torch.uint8)
        check(lib.b3c_accum_begin(_ptr(self.ws), self.ws.numel(), self.capacity, self.n_seq,
                                  _ptr(self.tid2idx), self.n_refs, _stream()))
        self.info = None

    def begin(self):
        """Start another map over the same reference table."""
        check(lib.b3c_accum_reset(_ptr(self.ws), _stream()))
        self.info = None

    def add(self, records):
        """records: CUDA int64/uint64-bit tensor of packed pair records (16-byte aligned)."""
        assert records.is_cuda and records.element_size() == 8 and records.is_contiguous()
        check(lib.b3c_accum_add_pairs(_ptr(self.ws), _ptr(records), records.numel(), _stream()))

    def add_packed(self, packed, n_records, bytes_per_record, same=False):
        """packed: CUDA uint8 tensor of narrow records (bam_io.pack_records), 16-byte aligned, padded to 8 bytes.
        same=True: 3- or 4-byte records of pairs on one reference (bam_io.split_records)."""
        assert packed.is_cuda and packed.element_size() == 1 and packed.is_contiguous()
        assert packed.numel() >= (int(n_records) * int(bytes_per_record) + 7) // 8 * 8
        fn = lib.b3c_accum_add_pairs_same if same else lib.b3c_accum_add_pairs_packed
        check(fn(_ptr(self.ws), _ptr(packed), int(n_records), int(bytes_per_record), _stream()))

    def finish(self, symmetric=True, pool=None):
        """Sort-reduce and emit the canonical CSR.  Returns (DeviceCSR[uint32 counts], info dict)."""
        sizes = (C.c_int64 * 8)()
        check(lib.b3c_accum_reduce(_ptr(self.ws), sizes, _stream()))
        nnz = int(sizes[1] if symmetric else sizes[0])
        indptr = _alloc(pool, 'map_indptr', self.n_seq + 1, torch.int64)
        indices = _alloc(pool, 'map_indices', nnz, torch.int32)
        counts = _alloc(pool, 'map_counts', nnz, torch.int32)
        check(lib.b3c_accum_emit_csr(_ptr(self.ws), 1 if symmetric else 0, _ptr(indptr), _ptr(indices),
                                     _ptr(counts), _stream()))
        self.info = dict(nnz_upper=int(sizes[0]), nnz_full=int(sizes[1]), accepted=int(sizes[2]),
                         ref_excluded=int(sizes[3]), poor_match=int(sizes[4]), map_weight=int(sizes[5]))
        return DeviceCSR(self.n_seq, indptr, indices, counts, counts=True), self.info


class SplitRecords(object):
    """
    Host (or device) pair records in the narrowest layout (bam_io.split_records): the pairs whose mates lie on one
    reference as 3- or 4-byte records (`same`, uint8 tensor), the rest as 5- / 6- / 8-byte pair records (`pairs`).
    The contact map does not depend on the order of its records, so the two parts are simply accumulated one after
    the other.
    """

    def __init__(self, same, n_same, bytes_same, pairs, n_pairs, bytes_pair):
        self.same, self.n_same, self.bytes_same = same, int(n_same), int(bytes_same)
        self.pairs, self.n_pairs, self.bytes_pair = pairs, int(n_pairs), int(bytes_pair)

    def parts(self):
        return ((self.same, self.n_same, self.bytes_same, True), (self.pairs, self.n_pairs, self.bytes_pair, False))

    @property
    def n_records(self):
        return self.n_same + self.n_pairs

    @property
    def nbytes(self):
        return int(self.same.numel()) + int(self.pairs.numel()) * self.pairs.element_size()

    @property
    def is_cuda(self):
        return bool(self.same.is_cuda)

    def pin_memory(self):
        return SplitRecords(self.same.pin_memory(), self.n_same, self.bytes_same, self.pairs.pin_memory(), self.n_pairs,
                            self.bytes_pair)

    def cuda(self):
        return SplitRecords(self.same.cuda(), self.n_same, self.bytes_same, self.pairs.cuda(), self.n_pairs,
                            self.bytes_pair)


class RecordStreamer(object):
    """
    Host pair records -> accumulator through a ring of two device staging buffers: the H2D copy of chunk k+1 runs
    on a side stream while chunk k is classified (use pinned memory for a truly asynchronous copy).  The chunk is
    large on purpose: every classify launch flushes its per-CTA diagonal histograms.  Used by HotPath (one GPU) and
    by the sharded driver (every rank streams its own shard).  Returns the bytes copied.
    """

    def __init__(self, pool):
        self.pool = pool
        self._copy_stream = None
        self._ring_ev = None

    def feed(self, acc, records, n_rec=None, record_bytes=8, chunk_records=1 << 24, same=False):
        if isinstance(records, SplitRecords):
            # same-reference records first, then the pair records: one stream through the same ring
            total = 0
            for part, n, B, sm in records.parts():
                if n:
                    total += self.feed(acc, part, n, B, chunk_records, same=sm)
            return total
        B = int(record_bytes)
        main = torch.cuda.current_stream()
        if self._copy_stream is None:
            self._copy_stream = torch.cuda.Stream()
            self._ring_ev = [[torch.cuda.Event(), torch.cuda.Event()] for _ in range(2)]
        copy_stream = self._copy_stream
        if B == 8:
            n_rec = int(records.numel())
            chunk = int(min(chunk_records, max(n_rec, 1)))
            chunk += chunk & 1                           # chunk starts stay 16-byte aligned
            ring = [self.pool.get('stage%d' % k, chunk, torch.int64) for k in range(2)]
        else:
            n_rec = int(n_rec)
            assert records.dtype == torch.uint8 and records.numel() >= (n_rec * B + 7) // 8 * 8
            chunk = max(8, int(min(chunk_records, max(n_rec, 1))) // 8 * 8)
            ring = [self.pool.get('stage_b%d' % k, chunk * B + 8, torch.uint8) for k in range(2)]
        copied_bytes = 0
        copy_stream.wait_stream(main)
        for k, lo in enumerate(range(0, n_rec, chunk)):
            hi = min(lo + chunk, n_rec)
            if B == 8:
                src, nel = records[lo:hi], hi - lo
            else:
                nel = ((hi - lo) * B + 7) // 8 * 8
                src = records[lo * B:lo * B + nel]
            buf, (copied, consumed) = ring[k & 1][:nel], self._ring_ev[k & 1]
            if k >= 2:
                copy_stream.wait_event(consumed)
            with torch.cuda.stream(copy_stream):
                buf.copy_(src, non_blocking=True)
                copied.record(copy_stream)
            main.wait_event(copied)
            if B == 8:
                acc.add(buf)
            else:
                acc.add_packed(buf, hi - lo, B, same=same)
            consumed.record(main)
            copied_bytes += nel * (8 if B == 8 else 1)
        return copied_bytes


# --------------------------------------------------------------------------------------
# mask + normalisation
# --------------------------------------------------------------------------------------

def max_offdiag(csr, pool=None):
    out = _alloc(pool, 'signal', csr.n, csr.data.dtype)
    fn = lib.b3c_max_offdiag_u32 if csr.counts else lib.b3c_max_offdiag_f64
    if not csr.counts:
        assert csr.data.dtype == torch.float64
    check(fn(csr.n, csr.row_lo, _ptr(csr.indptr), _ptr(csr.indices), _ptr(csr.data), _ptr(out), _stream()))
    return out


def acceptance_mask(lengths, signal, min_len, min_sig, pool=None):
    n = int(lengths.numel())
    mask = _alloc(pool, 'mask', n, torch.uint8)
    check(lib.b3c_acceptance_mask(n, _ptr(lengths), _ptr(signal), int(min_len), int(min_sig), _ptr(mask), _stream()))
    return mask


def site_norm(csr, sites, pool=None):
    """counts (uint32) or float64 matrix -> float64 matrix scaled by 1/(s_i*s_j); float input is scaled in place."""
    if csr.counts:
        out = _alloc(pool, 'normed', csr.nnz, torch.float64)
        check(lib.b3c_site_norm(csr.n, csr.row_lo, _ptr(csr.indptr), _ptr(csr.indices), _ptr(csr.data), _ptr(sites),
                                _ptr(out), _stream()))
        return csr.like(out)
    check(lib.b3c_site_norm_f64(csr.n, csr.row_lo, _ptr(csr.indptr), _ptr(csr.indices), _ptr(csr.data), _ptr(sites),
                                _stream()))
    return csr


MEAN_TYPES = {'geometric': 0, 'harmonic': 1, 'arithmetic': 2, None: -1}


def extent_norm(csr, bin_len, mean_type='geometric', pool=None):
    """Extent-map counts (uint32) -> float64 divided by 1e-3 * mean(L_r, L_c) (contact_map.py:1147-1165); mean_type
    None only converts.  bin_len: CUDA float64, the sequence length of every bin."""
    assert csr.counts, 'the extent map holds raw uint32 counts'
    if mean_type not in MEAN_TYPES:
        raise RuntimeError('unsupported mean type [{}]'.format(mean_type))        # contact_map.py:46
    out = _alloc(pool, 'extent_normed', csr.nnz, torch.float64)
    check(lib.b3c_extent_norm(csr.n, csr.row_lo, _ptr(csr.indptr), _ptr(csr.indices), _ptr(csr.data), _ptr(bin_len),
                              MEAN_TYPES[mean_type], _ptr(out), _stream()))
    return csr.like(out)


# --------------------------------------------------------------------------------------
# Knight-Ruiz
# --------------------------------------------------------------------------------------

_KR_WS = {}


def _kr_workspace(n, nnz):
    nbytes = lib.b3c_kr_workspace_bytes(n, nnz)
    dev = torch.cuda.current_device()
    ws = _KR_WS.get(dev)
    if ws is None or ws.numel() < nbytes:
        ws = _empty(nbytes, torch.uint8)
        _KR_WS[dev] = ws
    return ws


def kr_scale_vector(csr, tol=1e-6, delta=0.1, Delta=3, max_iter=1000, pool=None, sites=None):
    """
    Returns (x CUDA float64[n], info dict) for a symmetric float64 DeviceCSR -- or, with `sites`, for a
    uint32 count matrix that is site-normalised on the fly (the normalised matrix is never written).
    """
    ws = _kr_workspace(csr.n, csr.nnz)
    x = _alloc(pool, 'kr_x', csr.n, torch.float64)
    info = (C.c_int64 * 32)()
    if sites is not None:
        assert csr.counts, 'the counts form takes the raw uint32 contact matrix'
        rc = lib.b3c_kr_run_counts(csr.n, csr.nnz, _ptr(csr.indptr), _ptr(csr.indices), _ptr(csr.data), _ptr(sites),
                                   float(tol), float(delta), float(Delta), int(max_iter), _ptr(x), _ptr(ws),
                                   ws.numel(), info, _stream())
    else:
        assert csr.data.dtype == torch.float64
        rc = lib.b3c_kr_run(csr.n, csr.nnz, _ptr(csr.indptr), _ptr(csr.indices), _ptr(csr.data), float(tol),
                            float(delta), float(Delta), int(max_iter), 0, _ptr(x), _ptr(ws), ws.numel(), info,
                            _stream())
    names = ('init', 'spmv', 'reduce', 'resid', 'dir', 'w', 'step', 'update', 'scalar')
    out = dict(n_iter=int(info[0]), zero_diag=int(info[1]), outer=int(info[2]), n_spmv=int(info[3]),
               grid=int(info[4]), cycles=int(info[5]),
               work_cycles={k: int(info[6 + i]) for i, k in enumerate(names)},
               sync_cycles={k: int(info[15 + i]) for i, k in enumerate(names)},
               slabs=int(info[24]), nnz_stream=int(info[25]), segments=int(info[26]), kernel_us=int(info[27]),
               cta_spmv_cycles=dict(min=int(info[28]), max=int(info[29]), mean=int(info[30])),
               stream_bytes_per_entry=int(info[31]))
    check(rc)
    return x, out


def kr_apply(csr, x, pool=None):
    """diag(x) . A . diag(x) entry-wise (sparse_utils.py:223-224)."""
    out = _alloc(pool, 'balanced', csr.nnz, torch.float64)
    check(lib.b3c_kr_scale(csr.n, csr.row_lo, _ptr(csr.indptr), _ptr(csr.indices), _ptr(csr.data), _ptr(x), _ptr(out),
                           _stream()))
    return csr.like(out)


def asymmetry_count(csr, tol):
    scratch = _empty(1, torch.int64)
    cnt = (C.c_int64 * 1)()
    check(lib.b3c_asymmetry_count(csr.n, _ptr(csr.indptr), _ptr(csr.indices), _ptr(csr.data), float(tol),
                                  _ptr(scratch), cnt, _stream()))
    return int(cnt[0])


def spmv(csr, u, y=None, ws=None, prepared=False):
    """y = A.u with KR's SpMV kernels.  Pass the same ws with prepared=True to reuse the tile plan."""
    if ws is None:
        ws = _kr_workspace(csr.n, csr.nnz)
    if y is None:
        y = _empty(csr.n, torch.float64)
    check(lib.b3c_spmv(csr.n, csr.nnz, _ptr(csr.indptr), _ptr(csr.indices), _ptr(csr.data), _ptr(u), _ptr(y),
                       _ptr(ws), ws.numel(), 1 if prepared else 0, _stream()))
    return y


# --------------------------------------------------------------------------------------
# compress + edge weighting
# --------------------------------------------------------------------------------------

def compress_edges(csr, mask, want_sub=True, want_edges=True, scale=True, pool=None, reduce_max=None, sites=None,
                   x=None):
    """
    Drop rejected contigs and produce the compressed matrix and/or the weighted edge list of a
    matrix or row block.  `mask` covers all csr.n_total contigs.  `reduce_max(tensor)` lets a
    multi-GPU driver all-reduce the block maximum before the weights are scaled.
    Fused form: csr holds the raw uint32 counts and `sites`, `x` (site counts, KR scale vector) are
    given -- the edge weights are normalised and balanced on the fly (edge list only).
    Returns dict(n_accepted, sub=DeviceCSR|None, u, v, w, scl) with CUDA tensors.
    """
    fused = sites is not None
    if fused:
        assert csr.counts and x is not None and not want_sub and want_edges
    else:
        assert csr.data.dtype == torch.float64
    n, nl = csr.n_total, csr.n
    whole = (csr.row_lo == 0 and nl == n)
    assert whole or not want_sub, 'the compressed matrix is only produced for a whole matrix'
    nbytes = lib.b3c_compress_workspace_bytes(n)
    ws = _alloc(pool, 'compress_ws', nbytes, torch.uint8)
    newidx = _alloc(pool, 'newidx', n, torch.int32)
    vmax = _alloc(pool, 'vmax', 1, torch.float64)
    h = (C.c_int64 * 4)()
    if fused:
        check(lib.b3c_edges_count(n, csr.row_lo, nl, _ptr(csr.indptr), _ptr(csr.indices), _ptr(csr.data), _ptr(sites),
                                  _ptr(x), _ptr(mask), _ptr(newidx), _ptr(ws), ws.numel(), _ptr(vmax), h, _stream()))
    else:
        check(lib.b3c_compress_count(n, csr.row_lo, nl, _ptr(csr.indptr), _ptr(csr.indices), _ptr(csr.data),
                                     _ptr(mask), _ptr(newidx), _ptr(ws), ws.numel(), _ptr(vmax), h, _stream()))
    if reduce_max is not None:
        reduce_max(vmax)
    n_acc, n_kept, n_edges = int(h[0]), int(h[1]), int(h[2])
    sub_indptr = sub_indices = sub_data = eu = ev = ew = None
    if want_sub:
        sub_indptr = _alloc(pool, 'sub_indptr', n_acc + 1, torch.int64)
        sub_indices = _alloc(pool, 'sub_indices', n_kept, torch.int32)
        sub_data = _alloc(pool, 'sub_data', n_kept, torch.float64)
    if want_edges:
        # at least one element: a zero-length tensor (or view) reports a null address, which the fused fill refuses as
        # missing edge arrays; a block or a matrix without edges gets zero-length views of real buffers
        eu = _alloc(pool, 'edge_u', max(n_edges, 1), torch.int32)
        ev = _alloc(pool, 'edge_v', max(n_edges, 1), torch.int32)
        ew = _alloc(pool, 'edge_w', max(n_edges, 1), torch.float64)
    scl = _alloc(pool, 'scl', 1, torch.float64)
    if fused:
        check(lib.b3c_edges_fill(n, csr.row_lo, nl, _ptr(csr.indptr), _ptr(csr.indices), _ptr(csr.data), _ptr(ws),
                                 _ptr(vmax), 1 if scale else 0, _ptr(eu), _ptr(ev), _ptr(ew), _ptr(scl), _stream()))
    else:
        check(lib.b3c_compress_fill(n, csr.row_lo, nl, _ptr(csr.indptr), _ptr(csr.indices), _ptr(csr.data),
                                    _ptr(mask), _ptr(newidx), _ptr(ws), _ptr(vmax), 1 if scale else 0,
                                    _ptr(sub_indptr), _ptr(sub_indices), _ptr(sub_data), _ptr(eu), _ptr(ev), _ptr(ew),
                                    _ptr(scl), _stream()))
    sub = DeviceCSR(n_acc, sub_indptr, sub_indices, sub_data) if want_sub else None
    if want_edges:
        eu, ev, ew = eu[:n_edges], ev[:n_edges], ew[:n_edges]
    return dict(n_accepted=n_acc, n_kept=n_kept, n_edges=n_edges, sub=sub, u=eu, v=ev, w=ew, scl=scl, newidx=newidx)


def launch_count():
    return _cabi.launch_count()
