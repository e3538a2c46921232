"""
Multi-GPU driver of the hot path (SURVEY.md section 8e): one process per GPU, torch.distributed
(NCCL over NVLink / NVSwitch) for the exchanges, the C-ABI kernels for all arithmetic.

  accumulation   pair records are sharded by chunk (each rank classifies its own records).  Row
                 ranges are cut so that every rank owns about the same number of matrix entries
                 (all-reduced row histogram, 1024-row aligned).  Every canonical key (i<j) becomes
                 the directed keys (i,j) and (j,i), each routed to the owner of its row with ONE
                 all-to-all; the diagonal counts are all-reduced.  Each rank then sorts and
                 run-length reduces what it received: the result is its row block of the full
                 symmetric matrix, with exact integer counts whatever the number of ranks.
  mask / norm    per row block; the mask slices are combined with an all-reduce.
  KR             row block per rank.  Product path (CudaEngine.kr_run_peer): every rank runs the
                 persistent KR kernel on its block; u and the fixed-shape chunk partials live in
                 exchange buffers that all ranks of the node map over NVLink (CUDA IPC) and write
                 into directly, with flag barriers in the same buffers -- no host round trip and no
                 collective call inside the iteration.  Host-driven form (kr_block_loop, used by the
                 gloo tests and as the reference for the peer form): per SpMV the vector u is
                 assembled with an all-reduce (the slices a rank does not own are zero, so SUM is
                 exact), the partials are all-reduced, and the loop control runs on the device
                 from those partials (b3c_krp_*).  Every rank takes the same branches either way.
  compress/edges per row block; the scale 1/max needs one all-reduce(MAX).

The collective layer (`Comm`) and the per-rank compute layer (`engine`) are separate so the host
logic can be exercised on CPU with the gloo backend (tests/test_dist_gloo.py injects a NumPy
engine); the product engine is CudaEngine and has no CPU fallback.
"""
import ctypes as C
import time

import numpy as np
import torch
import torch.distributed as dist

CHUNK = 1024          # row alignment of KR row blocks (kr.cu: CHUNK)

KRP_INIT, KRP_SPMV, KRP_RESID, KRP_DIR, KRP_W, KRP_STEP, KRP_UPDATE = range(7)
KRS_OUTER_FIRST, KRS_OUTER, KRS_ALPHA, KRS_DECIDE = range(4)
STATE_DONE, STATE_INNER, STATE_UPDATE = 0, 1, 2
PA, PB, PC, PMIN, PNEGMAX, PG1, PG2 = range(7)


# ------------------------------------------------------------------------------------------------
# pure host logic
# ------------------------------------------------------------------------------------------------

def balanced_row_splits(row_weight, n_ranks, align=CHUNK):
    """
    Cut [0, n) into n_ranks contiguous row ranges of about equal total weight, boundaries rounded
    to multiples of `align` (the last boundary is n).  Ranges may be empty when n is small.
    Returns int32[n_ranks + 1].
    """
    w = np.asarray(row_weight, dtype=np.float64)
    n = len(w)
    cum = np.concatenate([[0.0], np.cumsum(w + 1e-9)])          # strictly increasing
    targets = cum[-1] * np.arange(1, n_ranks) / n_ranks
    cuts = np.searchsorted(cum, targets, side='left')
    cuts = (np.round(cuts / float(align)) * align).astype(np.int64)
    cuts = np.clip(cuts, 0, (n // align) * align)
    splits = np.concatenate([[0], np.maximum.accumulate(cuts), [n]]).astype(np.int32)
    return splits


class Comm(object):
    """The collectives the driver needs; world size 1 short-circuits everything."""

    def __init__(self, group=None):
        self.group = group
        self.on = dist.is_available() and dist.is_initialized()
        self.rank = dist.get_rank(group) if self.on else 0
        self.world = dist.get_world_size(group) if self.on else 1

    def all_reduce(self, t, op='sum'):
        if self.world > 1:
            ops = {'sum': dist.ReduceOp.SUM, 'min': dist.ReduceOp.MIN, 'max': dist.ReduceOp.MAX}
            dist.all_reduce(t, op=ops[op], group=self.group)
        return t

    def exchange_counts(self, send_counts):
        """send_counts[g] = elements this rank sends to g  ->  elements it receives from each g."""
        if self.world == 1:
            return list(send_counts)
        dev = 'cuda' if dist.get_backend(self.group) == 'nccl' else 'cpu'
        s = torch.tensor(send_counts, dtype=torch.int64, device=dev)
        r = torch.empty_like(s)
        dist.all_to_all_single(r, s, group=self.group)
        return [int(v) for v in r.cpu()]

    def all_to_all_v(self, send, send_counts, recv_counts):
        if self.world == 1:
            return send[:send_counts[0]]
        recv = torch.empty(int(sum(recv_counts)), dtype=send.dtype, device=send.device)
        dist.all_to_all_single(recv, send[:int(sum(send_counts))], output_split_sizes=list(recv_counts),
                               input_split_sizes=list(send_counts), group=self.group)
        return recv

    def barrier(self):
        if self.world > 1:
            dist.barrier(group=self.group)

    def all_gather_object(self, obj):
        if self.world == 1:
            return [obj]
        out = [None] * self.world
        dist.all_gather_object(out, obj, group=self.group)
        return out

    def gather_object(self, obj, dst=0):
        """Python objects of all ranks, in rank order, on rank `dst` (None elsewhere)."""
        if self.world == 1:
            return [obj]
        out = [None] * self.world if self.rank == dst else None
        dist.gather_object(obj, out, dst=dst, group=self.group)
        return out


# ------------------------------------------------------------------------------------------------
# the product engine: everything a rank computes, through the C ABI
# ------------------------------------------------------------------------------------------------

class _CAI(object):
    """Raw device memory as a __cuda_array_interface__ object (for torch.as_tensor)."""

    def __init__(self, ptr, n, typestr):
        self.__cuda_array_interface__ = dict(shape=(int(n),), typestr=typestr, data=(int(ptr), False), version=2)


def _device_view(ptr, n, dtype):
    """A torch tensor over n elements of device memory this process did not allocate through torch."""
    typestr = {torch.uint8: '|u1', torch.float64: '<f8', torch.int64: '<i8', torch.int32: '<i4'}[dtype]
    return torch.as_tensor(_CAI(ptr, n, typestr), device='cuda')


class CudaEngine(object):

    def __init__(self, tid2idx, lengths, sites, pair_capacity):
        from . import device as dev
        self.dev = dev
        dev.require_cuda()
        self.lib, self.check = dev.lib, dev.check
        self.n = int(len(lengths))
        self.tid2idx = dev.to_device(np.asarray(tid2idx, dtype=np.int32), torch.int32)
        self.lengths = dev.to_device(np.asarray(lengths, dtype=np.int32), torch.int32)
        self.sites = dev.to_device(np.asarray(sites, dtype=np.int32), torch.int32)
        self.acc = dev.Accumulator(self.n, self.tid2idx, pair_capacity)
        offs = (C.c_int64 * 4)()
        self.check(self.lib.b3c_accum_offsets(dev._ptr(self.acc.ws), offs))
        self._o_diag = int(offs[1])
        self.pool = dev.BufferPool()
        self.scratch = torch.zeros(256, dtype=torch.int64, device='cuda')
        self.kr_ws = None

    # ---- peer exchange arena (NVLink-mapped; see include/bin3c_b200.h, "Peer exchange arena") --------
    def open_arena(self, comm):
        """Allocate this rank's arena, map everybody else's (once); views of the mask and x regions."""
        if getattr(self, '_arena', None) is not None:
            return self._arena
        lib, dev = self.lib, self.dev
        assert comm.world <= 8, 'the peer arena spans the GPUs of one node (at most 8 ranks)'
        self._xa_cap = int(self.acc.capacity)
        nbytes = lib.b3c_xa_bytes(self.n, self._xa_cap)
        own = C.c_void_p()
        handle = C.create_string_buffer(64)
        self.check(lib.b3c_peer_alloc(nbytes, C.byref(own), handle))
        handles = comm.all_gather_object(handle.raw)
        ptrs = (C.c_void_p * comm.world)()
        self._a_opened = []
        for g, h in enumerate(handles):
            if g == comm.rank:
                ptrs[g] = own.value
            else:
                q = C.c_void_p()
                self.check(lib.b3c_peer_open(h, C.byref(q)))
                ptrs[g] = q.value
                self._a_opened.append(q.value)
        offs = (C.c_int64 * 4)()
        self.check(lib.b3c_xa_offsets(self.n, self._xa_cap, offs))
        self._a_off = dict(mask=int(offs[0]), x=int(offs[1]))
        self._a_own = own.value
        self._arena = ptrs
        self._epoch = 0
        self.mask_view = _device_view(own.value + self._a_off['mask'], self.n, torch.uint8)
        self.x_view = _device_view(own.value + self._a_off['x'], self.n, torch.float64)
        self._scal = torch.zeros(8, dtype=torch.float64, device='cuda')
        self._splits_dev = torch.zeros(16, dtype=torch.int32, device='cuda')
        comm.barrier()
        return ptrs

    def close_arena(self):
        if getattr(self, '_arena', None) is None:
            return
        torch.cuda.synchronize()
        self.mask_view = self.x_view = None
        for q in self._a_opened:
            self.lib.b3c_peer_close(C.c_void_p(q))
        self.lib.b3c_peer_free(C.c_void_p(self._a_own))
        self._arena = None

    def peer_barrier(self, comm):
        self._epoch += 1
        self.check(self.lib.b3c_peer_barrier(self._arena, comm.rank, comm.world, self.n, self._xa_cap, self._epoch,
                                             self.dev._stream()))

    def peer_put(self, comm, region, elem_offset, src):
        """src (CUDA tensor) -> every rank's arena, `elem_offset` elements into the named region."""
        off = self._a_off[region] + int(elem_offset) * src.element_size()
        self.check(self.lib.b3c_peer_put(self._arena, comm.world, off, self.dev._ptr(src),
                                         src.numel() * src.element_size(), self.dev._stream()))

    def peer_allreduce(self, comm, t, op='sum'):
        """In-place all-reduce of a small float64 CUDA tensor (<= 8 values) through the arenas."""
        assert t.dtype == torch.float64 and t.numel() <= 8 and t.is_contiguous()
        self._epoch += 1
        self.check(self.lib.b3c_peer_allreduce_f64(self._arena, comm.rank, comm.world, self.n, self._xa_cap, self._epoch,
                                                   0 if op == 'sum' else 1, self.dev._ptr(t), t.numel(),
                                                   self.dev._stream()))
        return t

    def add_records(self, records, record_bytes=8, n_records=None):
        """Classify this rank's pair records: a CUDA tensor in place, or HOST records (pinned for an asynchronous
        copy; native 8-byte or narrow 5/6-byte, bam_io.pack_records) streamed through the staging ring."""
        B = int(record_bytes)
        self.h2d_bytes = 0
        if isinstance(records, self.dev.SplitRecords):
            if records.is_cuda:
                for part, n, pb, same in records.parts():
                    if n:
                        self.acc.add_packed(part, n, pb, same=same)
                return
            if getattr(self, '_streamer', None) is None:
                self._streamer = self.dev.RecordStreamer(self.pool)
            self.h2d_bytes = self._streamer.feed(self.acc, records)
            return
        if records.is_cuda:
            if B == 8:
                self.acc.add(records)
            else:
                self.acc.add_packed(records, int(n_records), B)
            return
        if getattr(self, '_streamer', None) is None:
            self._streamer = self.dev.RecordStreamer(self.pool)
        self.h2d_bytes = self._streamer.feed(self.acc, records, n_records, B)

    def accumulate_peer(self, records, comm, record_bytes=8, n_records=None):
        """
        The sharded accumulation with every exchange done by kernels over the peer arenas: classify ->
        publish chunk weights | barrier | splits + route/scatter into the owners' buffers | barrier |
        sort + reduce the received keys -> this rank's row block.  One host synchronisation (the sizes).
        Returns (block DeviceCSR or None, info dict).
        """
        dev, lib = self.dev, self.lib
        ptrs = self.open_arena(comm)
        mark = self._mark
        mark('start')
        self.acc.begin()
        self.add_records(records, record_bytes, n_records)
        mark('classify')
        ws = dev._ptr(self.acc.ws)
        self.check(lib.b3c_shard_publish(ws, ptrs, comm.rank, comm.world, dev._stream()))
        mark('publish')
        self.peer_barrier(comm)
        mark('barrier1')
        self.check(lib.b3c_shard_scatter(ws, ptrs, comm.rank, comm.world, dev._ptr(self._splits_dev), dev._stream()))
        mark('route')
        self.peer_barrier(comm)
        mark('barrier2')
        sizes = (C.c_int64 * 24)()
        self.check(lib.b3c_shard_reduce_block(ws, ptrs, comm.rank, comm.world, dev._ptr(self._splits_dev), sizes,
                                              dev._stream()))
        mark('sort_reduce')
        nnz, row_lo, row_hi = int(sizes[0]), int(sizes[1]), int(sizes[2])
        info = dict(accepted=int(sizes[3]), ref_excluded=int(sizes[4]), poor_match=int(sizes[5]),
                    keys_received=int(sizes[6]), splits=[int(sizes[8 + g]) for g in range(comm.world + 1)])
        block = None
        if row_hi > row_lo:
            nl = row_hi - row_lo
            indptr = self.pool.get('blk_indptr', nl + 1, torch.int64)
            indices = self.pool.get('blk_indices', nnz, torch.int32)
            counts = self.pool.get('blk_counts', nnz, torch.int32)
            self.check(lib.b3c_accum_emit_block(ws, row_lo, row_hi, dev._ptr(indptr), dev._ptr(indices),
                                                dev._ptr(counts), dev._stream()))
            block = dev.DeviceCSR(nl, indptr, indices, counts, counts=True, row_lo=row_lo, n_total=self.n)
        mark('emit')
        return block, info

    # sub-step CUDA events of the sharded accumulation (bench.py's stage table; off unless `events` is a list)
    events = None

    def _mark(self, name):
        if self.events is not None:
            ev = torch.cuda.Event(enable_timing=True)
            ev.record()
            self.events.append((name, ev))

    def substep_ms(self):
        """{sub-step: ms} from the recorded events (call after a synchronize); clears them."""
        out = {}
        evs, self.events = self.events or [], []
        for (na, a), (nb, b) in zip(evs[:-1], evs[1:]):
            if nb != 'start':
                out[nb] = out.get(nb, 0.0) + a.elapsed_time(b)
        return out

    # ---- accumulation ------------------------------------------------------------------------
    def classify(self, records, record_bytes=8, n_records=None):
        self.acc.begin()
        self.add_records(records, record_bytes, n_records)

    def row_hist(self):
        dev = self.dev
        h = self.pool.get('rowcnt', self.n, torch.int64)
        h.zero_()
        self.check(self.lib.b3c_accum_row_hist(dev._ptr(self.acc.ws), dev._ptr(h), dev._stream()))
        return h

    def diag_counts(self):
        """int32 view of the accumulator's diagonal counts (to be all-reduced in place)."""
        return self.acc.ws[self._o_diag:self._o_diag + 4 * self.n].view(torch.int32)

    def route(self, splits):
        dev = self.dev
        G = len(splits) - 1
        d_splits = dev.to_device(np.asarray(splits, dtype=np.int32), torch.int32)
        out = self.pool.get('route_out', 2 * self.acc.capacity, torch.int64)
        h = (C.c_int64 * (G + 8))()
        self.check(self.lib.b3c_accum_route(dev._ptr(self.acc.ws), dev._ptr(d_splits), G, dev._ptr(out), out.numel(),
                                            dev._ptr(self.scratch), h, dev._stream()))
        offs = [int(h[g]) for g in range(G + 1)]
        counters = dict(accepted=int(h[G + 1]), ref_excluded=int(h[G + 2]), poor_match=int(h[G + 3]))
        return out, [offs[g + 1] - offs[g] for g in range(G)], counters

    def build_block(self, keys, row_lo, row_hi):
        dev = self.dev
        sizes = (C.c_int64 * 8)()
        n_keys = int(keys.numel())
        self.check(self.lib.b3c_accum_reduce_block(dev._ptr(self.acc.ws), dev._ptr(keys) if n_keys else None, n_keys,
                                                   row_lo, row_hi, sizes, dev._stream()))
        nnz = int(sizes[0])
        nl = row_hi - row_lo
        indptr = self.pool.get('blk_indptr', nl + 1, torch.int64)
        indices = self.pool.get('blk_indices', nnz, torch.int32)
        counts = self.pool.get('blk_counts', nnz, torch.int32)
        self.check(self.lib.b3c_accum_emit_block(dev._ptr(self.acc.ws), row_lo, row_hi, dev._ptr(indptr),
                                                 dev._ptr(indices), dev._ptr(counts), dev._stream()))
        return dev.DeviceCSR(nl, indptr, indices, counts, counts=True, row_lo=row_lo, n_total=self.n)

    # ---- mask / norm ---------------------------------------------------------------------------
    def block_mask(self, csr, min_len, min_sig):
        dev = self.dev
        sig = dev.max_offdiag(csr, pool=self.pool)
        return dev.acceptance_mask(self.lengths[csr.row_lo:csr.row_lo + csr.n], sig, min_len, min_sig, pool=self.pool)

    def new_mask(self):
        m = self.pool.get('mask_full', self.n, torch.uint8)
        m.zero_()
        return m

    def site_norm(self, csr):
        return self.dev.site_norm(csr, self.sites, pool=self.pool)

    # ---- KR phases -------------------------------------------------------------------------------
    def kr_setup(self, csr, tol, delta, Delta, max_iter):
        dev, lib = self.dev, self.lib
        nbytes = lib.b3c_krp_workspace_bytes(self.n, csr.nnz)
        if self.kr_ws is None or self.kr_ws.numel() < nbytes:
            self.kr_ws = torch.empty(nbytes, dtype=torch.uint8, device='cuda')
        offs = (C.c_int64 * 8)()
        self.check(lib.b3c_krp_setup(self.n, csr.row_lo, csr.row_lo + csr.n, csr.nnz, dev._ptr(csr.indptr),
                                     dev._ptr(csr.indices), dev._ptr(csr.data), float(tol), float(delta), float(Delta),
                                     int(max_iter), dev._ptr(self.kr_ws), self.kr_ws.numel(), offs, dev._stream()))
        n, nc = self.n, int(offs[3])
        ws = self.kr_ws
        self.u = ws[int(offs[0]):int(offs[0]) + 8 * n].view(torch.float64)
        self.x = ws[int(offs[1]):int(offs[1]) + 8 * n].view(torch.float64)
        self.part = ws[int(offs[2]):int(offs[2]) + 8 * 7 * nc].view(torch.float64).view(7, nc)

    def kr_phase(self, phase):
        self.check(self.lib.b3c_krp_phase(self.dev._ptr(self.kr_ws), phase, self.dev._stream()))

    def kr_scalar(self, which):
        self.check(self.lib.b3c_krp_scalar(self.dev._ptr(self.kr_ws), which, self.dev._stream()))

    def kr_state(self):
        h = (C.c_int64 * 8)()
        self.check(self.lib.b3c_krp_state(self.dev._ptr(self.kr_ws), h, self.dev._stream()))
        return dict(state=int(h[0]), status=int(h[1]), n_iter=int(h[2]), k=int(h[3]), outer=int(h[4]),
                    n_spmv=int(h[5]), zero_diag=int(h[6]))

    # ---- KR, peer form ---------------------------------------------------------------------------------
    def _peer_buffers(self, comm):
        """This rank's exchange buffer plus the mapped buffers of all other ranks (made once)."""
        if getattr(self, '_xbuf', None) is not None:
            return self._xbuf
        lib = self.lib
        assert comm.world <= 8, 'peer-mode KR handles the GPUs of one node (at most 8 ranks)'
        nbytes = lib.b3c_kr_exchange_bytes(self.n)
        own = C.c_void_p()
        handle = C.create_string_buffer(64)
        self.check(lib.b3c_peer_alloc(nbytes, C.byref(own), handle))
        handles = comm.all_gather_object(handle.raw)
        ptrs = (C.c_void_p * comm.world)()
        self._x_opened = []
        for g, h in enumerate(handles):
            if g == comm.rank:
                ptrs[g] = own.value
            else:
                p = C.c_void_p()
                self.check(lib.b3c_peer_open(h, C.byref(p)))
                ptrs[g] = p.value
                self._x_opened.append(p.value)
        self._x_own = own.value
        self._xbuf = ptrs
        comm.barrier()
        return ptrs

    def close_peers(self):
        self.close_arena()
        if getattr(self, '_xbuf', None) is None:
            return
        torch.cuda.synchronize()
        for p in self._x_opened:
            self.lib.b3c_peer_close(C.c_void_p(p))
        self.lib.b3c_peer_free(C.c_void_p(self._x_own))
        self._xbuf = None

    fused = True      # KR and the edge emission take the raw counts (normalised / balanced on the fly)

    def kr_run_peer(self, csr, tol, delta, Delta, max_iter, comm):
        """The whole KR iteration of this rank's row block in one persistent kernel (see module docstring).
        csr: float64 normalised block, or the raw uint32 count block (site-normalised on the fly)."""
        dev, lib = self.dev, self.lib
        ptrs = self._peer_buffers(comm)
        nbytes = lib.b3c_krp_workspace_bytes(self.n, csr.nnz)
        if self.kr_ws is None or self.kr_ws.numel() < nbytes:
            self.kr_ws = torch.empty(nbytes, dtype=torch.uint8, device='cuda')
        x = self.pool.get('kr_x', self.n, torch.float64)
        info = (C.c_int64 * 32)()
        if csr.counts:
            rc = lib.b3c_kr_run_peer_counts(self.n, csr.row_lo, csr.row_lo + csr.n, csr.nnz, dev._ptr(csr.indptr),
                                            dev._ptr(csr.indices), dev._ptr(csr.data), dev._ptr(self.sites), float(tol),
                                            float(delta), float(Delta), int(max_iter), comm.rank, comm.world, ptrs,
                                            dev._ptr(x), dev._ptr(self.kr_ws), self.kr_ws.numel(), info, dev._stream())
        else:
            rc = lib.b3c_kr_run_peer(self.n, csr.row_lo, csr.row_lo + csr.n, csr.nnz, dev._ptr(csr.indptr),
                                     dev._ptr(csr.indices), dev._ptr(csr.data), float(tol), float(delta), float(Delta),
                                     int(max_iter), comm.rank, comm.world, ptrs, dev._ptr(x), dev._ptr(self.kr_ws),
                                     self.kr_ws.numel(), info, dev._stream())
        self.x = x
        st = dict(state=0, status=0, n_iter=int(info[0]), zero_diag=int(info[1]), outer=int(info[2]),
                  n_spmv=int(info[3]), kernel_us=int(info[27]), slabs=int(info[24]), nnz_stream=int(info[25]),
                  cycles=int(info[5]))
        names = ('init', 'spmv', 'reduce', 'resid', 'dir', 'w', 'step', 'update', 'scalar')
        st['work_cycles'] = {k: int(info[6 + i]) for i, k in enumerate(names)}
        st['sync_cycles'] = {k: int(info[15 + i]) for i, k in enumerate(names)}
        if rc == -6:
            st['status'] = -6
        else:
            self.check(rc)
        return st

    # ---- scaling + edges ----------------------------------------------------------------------------
    def kr_apply(self, csr, x):
        return self.dev.kr_apply(csr, x, pool=self.pool)

    def compress_edges(self, csr, mask, reduce_max, scale=True, x=None):
        """csr: the balanced float64 block, or (with x) the raw count block -- fused form."""
        return self.dev.compress_edges(csr, mask, want_sub=False, want_edges=True, scale=scale, pool=self.pool,
                                       reduce_max=reduce_max, sites=self.sites if x is not None else None, x=x)

    def synchronize(self):
        torch.cuda.synchronize()


# ------------------------------------------------------------------------------------------------
# the driver
# ------------------------------------------------------------------------------------------------

def kr_block_loop(eng, comm, max_phases=1_000_000):
    """
    The Knight-Ruiz iteration over row blocks (sparse_utils.py:123-221): phases on the engine,
    collectives in between, loop control on the device (see include/bin3c_b200.h, "Row-block
    phase API").  Returns the final state dict.
    """
    def spmv():
        comm.all_reduce(eng.u, 'sum')
        eng.kr_phase(KRP_SPMV)

    eng.kr_phase(KRP_INIT)
    spmv()
    eng.kr_phase(KRP_RESID)
    comm.all_reduce(eng.part[PA], 'sum')
    eng.kr_scalar(KRS_OUTER_FIRST)
    st = eng.kr_state()
    n = 0
    while st['state'] != STATE_DONE and n < max_phases:
        n += 1
        if st['state'] == STATE_INNER:
            eng.kr_phase(KRP_DIR)
            spmv()
            eng.kr_phase(KRP_W)
            comm.all_reduce(eng.part[PA:PB + 1], 'sum')
            eng.kr_scalar(KRS_ALPHA)
            eng.kr_phase(KRP_STEP)
            comm.all_reduce(eng.part[PC], 'sum')
            comm.all_reduce(eng.part[PMIN:PG2 + 1], 'min')
            eng.kr_scalar(KRS_DECIDE)
        else:
            eng.kr_phase(KRP_UPDATE)
            spmv()
            eng.kr_phase(KRP_RESID)
            comm.all_reduce(eng.part[PA], 'sum')
            eng.kr_scalar(KRS_OUTER)
        st = eng.kr_state()
    return st


class _no_range(object):
    """Stand-in for device.nvtx_range when the engine is not the CUDA engine (gloo tests)."""

    def __init__(self, name):
        pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        return False


class _Trace(object):
    """Optional wall-clock trace of the driver's sub-steps (device-synchronised; for tuning, never in timed runs)."""

    def __init__(self):
        self.on, self.t, self.out = False, 0.0, {}

    def start(self):
        self.on, self.out = True, {}
        torch.cuda.synchronize()
        self.t = time.perf_counter()

    def mark(self, name):
        if self.on:
            torch.cuda.synchronize()
            now = time.perf_counter()
            self.out[name] = self.out.get(name, 0.0) + (now - self.t) * 1e3
            self.t = now


def _raise_kr_status(status, n_iter, max_iter):
    """Raise what b3c_kr_run* raises for the same outcome of the iteration: the exception type _cabi.check gives the
    status, with the message kr.cu's set_error writes for it (b3c_krp_state reports the status without a message)."""
    if status == 0 and n_iter <= max_iter:
        return
    from . import _cabi
    if status == _cabi.B3C_ERR_TIE:
        msg = 'KR: max(ynew) == Delta with no element above Delta (reference raises ValueError here)'
    elif status == _cabi.B3C_ERR_NAN:
        msg = 'scale vector has developed invalid values (NANs)!'
    elif status in (0, _cabi.B3C_ERR_NOCONV):
        status = _cabi.B3C_ERR_NOCONV
        msg = 'matrix balancing failed to converge in {} iterations'.format(n_iter)
    else:
        msg = 'KR phase loop ended with status {}'.format(status)
    raise _cabi.error(status, msg)


class ShardedHotPath(object):
    """The whole path over `comm.world` ranks.  Each rank passes its own chunk of pair records."""

    def __init__(self, tid2idx, lengths, sites, pair_capacity, min_len=1000, min_sig=5, tol=1e-6, delta=0.1,
                 Delta=3, max_iter=1000, comm=None, engine=None, host_driven_kr=False, peer_exchange=None):
        self.comm = comm or Comm()
        self.host_driven_kr = host_driven_kr          # True: kr_block_loop (collectives between phases)
        self.trace = _Trace()
        self.n = int(len(lengths))
        self.min_len, self.min_sig = int(min_len), int(min_sig)
        self.kr_params = (tol, delta, Delta, max_iter)
        # every rank may receive up to both directions of every key: size the buffers for the
        # directed keys of a balanced split with head-room
        self.engine = engine or CudaEngine(tid2idx, lengths, sites, pair_capacity)
        # peer exchange: keys, mask / x slices and the small reductions move through NVLink-mapped arenas
        # written by our own kernels; otherwise (CPU engines, host-driven form) through torch.distributed
        self.peer = (hasattr(self.engine, 'accumulate_peer') and not host_driven_kr) if peer_exchange is None \
            else bool(peer_exchange)
        self.info = {}

    def _check_splits(self):
        """Every rank needs rows: the KR driver and the peer barriers have no form for an idle rank.  The splits are
        the same on every rank, so all of them raise together (nobody is left spinning at a barrier)."""
        if np.any(np.diff(self.splits) <= 0):
            raise ValueError('{} contigs cannot be cut into {} row blocks of whole {}-row chunks (splits {}): run '
                             'this community on fewer GPUs'.format(self.n, self.comm.world, CHUNK, self.splits.tolist()))

    def stage_barrier(self):
        """All ranks' streams meet here (a device-side barrier when the peer arenas are open): bench.py puts one in
        front of every stage it times, so that a stage does not absorb the skew left by its predecessors."""
        eng, comm = self.engine, self.comm
        if self.peer and getattr(eng, '_arena', None) is not None:
            eng.peer_barrier(comm)
        elif comm.world > 1:
            eng.synchronize()
            comm.barrier()

    @property
    def h2d_bytes(self):
        return int(getattr(self.engine, 'h2d_bytes', 0))

    def accumulate(self, records, record_bytes=8, n_records=None):
        eng, comm = self.engine, self.comm
        tr = self.trace
        if self.peer:
            self.block, info = eng.accumulate_peer(records, comm, record_bytes, n_records)
            self.splits = np.asarray(info['splits'], dtype=np.int32)
            self.row_lo, self.row_hi = int(self.splits[comm.rank]), int(self.splits[comm.rank + 1])
            self.info.update(info)
            tr.mark('accumulate(peer)')
            self._check_splits()
            return self.block
        if record_bytes != 8:
            eng.classify(records, record_bytes, n_records)
        else:
            eng.classify(records)
        tr.mark('classify')
        rowcnt = comm.all_reduce(eng.row_hist(), 'sum')
        tr.mark('row_hist+allreduce')
        weight = rowcnt.cpu().numpy().astype(np.float64) + 1.0        # +1: the diagonal entry
        self.splits = balanced_row_splits(weight, comm.world)
        tr.mark('splits(host)')
        send, send_counts, counters = eng.route(self.splits)
        tr.mark('route')
        recv_counts = comm.exchange_counts(send_counts)
        keys = comm.all_to_all_v(send, send_counts, recv_counts)
        tr.mark('all_to_all')
        comm.all_reduce(eng.diag_counts(), 'sum')
        tr.mark('diag allreduce')
        self.row_lo, self.row_hi = int(self.splits[comm.rank]), int(self.splits[comm.rank + 1])
        dev = keys.device
        c = torch.tensor([counters['accepted'], counters['ref_excluded'], counters['poor_match']],
                         dtype=torch.int64, device=dev)
        comm.all_reduce(c, 'sum')
        c = c.cpu().tolist()
        self.info.update(accepted=c[0], ref_excluded=c[1], poor_match=c[2], splits=self.splits.tolist(),
                         keys_received=int(keys.numel()))
        tr.mark('counters')
        if self.row_hi > self.row_lo:
            self.block = eng.build_block(keys, self.row_lo, self.row_hi)
        else:
            self.block = None
        tr.mark('build_block')
        self._check_splits()
        return self.block

    def compute_mask(self):
        eng, comm = self.engine, self.comm
        if self.peer:
            if self.block is not None:
                eng.peer_put(comm, 'mask', self.row_lo, eng.block_mask(self.block, self.min_len, self.min_sig))
            eng.peer_barrier(comm)
            self.mask = eng.mask_view
            self.trace.mark('mask')
            return self.mask
        mask = eng.new_mask()
        if self.block is not None:
            mask[self.row_lo:self.row_hi].copy_(eng.block_mask(self.block, self.min_len, self.min_sig))
        self.mask = comm.all_reduce(mask, 'sum')
        self.trace.mark('mask')
        return self.mask

    def balance(self):
        eng, comm = self.engine, self.comm
        self._check_splits()
        peer = hasattr(eng, 'kr_run_peer') and not self.host_driven_kr
        self.fused = peer and getattr(eng, 'fused', False)
        if self.fused:
            self.normed = None
            st = eng.kr_run_peer(self.block, *self.kr_params, comm=comm)
        elif peer:
            self.normed = eng.site_norm(self.block)
            self.trace.mark('site_norm')
            st = eng.kr_run_peer(self.normed, *self.kr_params, comm=comm)
        else:
            self.normed = eng.site_norm(self.block)
            self.trace.mark('site_norm')
            eng.kr_setup(self.normed, *self.kr_params)
            st = kr_block_loop(eng, comm)
        self.trace.mark('kr')
        if self.peer:
            # the persistent kernel leaves the WHOLE scale vector on every rank (x lives in the exchange buffers);
            # only the zero-diagonal count, kept per row block, is summed through the arenas
            eng._scal[0] = float(st['zero_diag'])
            self._zero_diag_dev = eng.peer_allreduce(comm, eng._scal[:1], 'sum').clone()
            st['zero_diag'] = None                 # read back with the edge sizes (edges()): no host sync of its own
        else:
            z = torch.tensor([st['zero_diag']], dtype=torch.int64, device=eng.x.device)
            st['zero_diag'] = int(comm.all_reduce(z, 'sum').cpu()[0])
        self.kr_info = st
        _raise_kr_status(st['status'], st['n_iter'], self.kr_params[3])
        # x: every rank wrote its own slice; assemble the whole vector
        xs = eng.x
        if peer:
            pass                                   # complete on every rank already
        elif comm.world > 1:
            full = torch.zeros_like(xs)
            full[self.row_lo:self.row_hi].copy_(xs[self.row_lo:self.row_hi])
            xs = comm.all_reduce(full, 'sum')
        self.x = xs
        self.trace.mark('x allreduce')
        if self.fused:
            self.balanced = None
        else:
            self.balanced = eng.kr_apply(self.normed, self.x)
            self.trace.mark('kr_apply')
        return self.balanced

    def edges(self, scale=True):
        eng, comm = self.engine, self.comm
        if self.peer:
            reduce_max = lambda t: eng.peer_allreduce(comm, t, 'max')         # noqa: E731
        else:
            reduce_max = lambda t: comm.all_reduce(t, 'max')                  # noqa: E731
        if self.fused:
            self.edge_res = eng.compress_edges(self.block, self.mask, reduce_max, scale=scale, x=self.x)
        else:
            self.edge_res = eng.compress_edges(self.balanced, self.mask, reduce_max, scale=scale)
        if getattr(self, '_zero_diag_dev', None) is not None and self.kr_info.get('zero_diag') is None:
            self.kr_info['zero_diag'] = int(self._zero_diag_dev.cpu()[0])     # the stream has just been synchronised
            self._zero_diag_dev = None
        self.trace.mark('edges')
        return self.edge_res

    def traced_run(self, records):
        """One run with a device sync after every sub-step; returns {sub-step: ms}."""
        self.trace.start()
        self.run(records)
        self.trace.on = False
        return dict(self.trace.out)

    def run(self, records, record_bytes=8, n_records=None):
        dev = getattr(self.engine, 'dev', None)
        rng = getattr(dev, 'nvtx_range', None) or _no_range
        with (dev.pipeline_stream() if dev is not None else _no_range('')):
            with rng('accumulate(sharded)'):
                self.accumulate(records, record_bytes, n_records)
            with rng('mask'):
                self.compute_mask()
            with rng('kr(row block)'):
                self.balance()
            with rng('edges'):
                return self.edges()
