"""
ctypes binding of libbin3c_io.so (include/bin3c_io.h): the two host-side steps either side of the
contact-map hot path (SURVEY.md 8f, ranks 1 and 2).

* `BamPairReader` / `pair_records_from_bam` -- name-sorted BAM -> header reference table + packed pair
  records, i.e. what the reference does with pysam in contact_map.py:534-545 (header, sort-order check)
  and :624-629, :720-766 (informative records, mate pairing, matchers, min_insert).  The result feeds
  `ContactMap(PairRecords(...))` / `Sparse2DAccumulator.add_pairs`.
* `write_edges` -- edge arrays -> the `cm_graph.edges` text file nx.write_edgelist produces
  (cluster.py:139-151).

Like the device library there is no Python fallback: a missing .so raises ImportError.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'libbin3c_io.so')

B3C_IO_OK = 0
B3C_IO_ERR_ARG = -1
B3C_IO_ERR_OPEN = -2
B3C_IO_ERR_FORMAT = -3
B3C_IO_ERR_SORT = -4

DEFAULT_SLAB_BYTES = 256 << 20    # compressed bytes per slab of the device decoder

FLOAT_REPR = 0       # Python 3 str(float) == repr(float)
FLOAT_STR12 = 1      # Python 2.7 str(float): '%.12g' (+ '.0'), what the reference's pinned interpreter prints

if not os.path.exists(LIB_PATH):
    raise ImportError('{} is missing: build it with `python -m bin3c_b200.csrc.build`'.format(LIB_PATH))

lib = C.CDLL(LIB_PATH)

_p = C.c_void_p
_i32 = C.c_int32
_i64 = C.c_int64

# name: (restype, argtypes) -- must list every function declared in include/bin3c_io.h
SIGNATURES = {
    'b3c_io_version': (C.c_int, []),
    'b3c_io_last_error': (C.c_char_p, []),
    'b3c_bam_open': (C.c_int, [C.c_char_p, _i32, _i32, C.POINTER(C.c_void_p)]),
    'b3c_bam_close': (None, [_p]),
    'b3c_bam_n_refs': (_i32, [_p]),
    'b3c_bam_ref_name': (C.c_char_p, [_p, _i32]),
    'b3c_bam_ref_lengths': (_i64, [_p, _p, _i32]),
    'b3c_bam_header_text': (_i64, [_p, _p, _i64]),
    'b3c_bam_data_offset': (_i64, [_p]),
    'b3c_bgzf_scan': (_i64, [_p, _i64, _i32, _p, _p, _p, _i64, _p]),
    'b3c_bam_set_filter': (C.c_int, [_p, _i32, _i32, _i32, _p, _i32]),
    'b3c_bam_read_pairs': (_i64, [_p, _p, _i64]),
    'b3c_bam_set_extent': (C.c_int, [_p, _p, _i32, _p, _p, _p, _i32]),
    'b3c_bam_read_pairs_extent': (_i64, [_p, _p, _p, _i64]),
    'b3c_bam_set_tips': (C.c_int, [_p, _i64, _p, _i32]),
    'b3c_bam_read_pairs_tips': (_i64, [_p, _p, _p, _i64]),
    'b3c_bam_stats': (C.c_int, [_p, _p, _i32]),
    'b3c_edges_write': (_i64, [C.c_char_p, _p, _p, _p, _i64, C.c_char, _i32]),
    'b3c_edges_write_fmt': (_i64, [C.c_char_p, _p, _p, _p, _i64, C.c_char, _i32, _i32]),
    'b3c_records_bytes': (_i32, [_i64]),
    'b3c_records_pack': (_i64, [_p, _i64, _i32, _p, _i32]),
    'b3c_records_unpack': (_i64, [_p, _i64, _i32, _p]),
    'b3c_records_same_bytes': (_i32, [_i64]),
    'b3c_records_split': (_i64, [_p, _i64, _i32, _i32, _p, _p, _p, _i32]),
    'b3c_format_weight': (_i32, [C.c_double, _p, _i32]),
    'b3c_format_weight_fmt': (_i32, [C.c_double, _i32, _p, _i32]),
}

for _name, (_res, _args) in SIGNATURES.items():
    _fn = getattr(lib, _name)
    _fn.restype = _res
    _fn.argtypes = _args


def last_error():
    return lib.b3c_io_last_error().decode('utf-8', 'replace')


def check(rc):
    """Map a b3c_io_status to the exception the reference raises for the same condition."""
    if rc >= 0:
        return rc
    msg = last_error()
    if rc == B3C_IO_ERR_ARG:
        raise AssertionError(msg)
    if rc == B3C_IO_ERR_SORT:
        raise IOError(msg)                        # contact_map.py:537-538
    if rc == B3C_IO_ERR_OPEN:
        raise IOError(msg)
    raise ValueError(msg)                         # malformed file (pysam raises ValueError / OSError here)


STAT_NAMES = ('alignments', 'informative', 'pairs', 'short_insert', 'unpaired', 'bgzf_blocks', 'compressed_bytes',
              'uncompressed_bytes', 'not_tip')


class BamPairReader(object):
    """
    A name-sorted BAM file as a stream of packed pair records.

    :param path: BAM file
    :param threads: inflate threads (<= 0: one per online core)
    :param require_queryname: raise IOError unless @HD SO:queryname (contact_map.py:537-538)
    """

    def __init__(self, path, threads=0, require_queryname=True):
        self._h = C.c_void_p()
        check(lib.b3c_bam_open(os.fsencode(path), int(threads), 1 if require_queryname else 0, C.byref(self._h)))
        n = lib.b3c_bam_n_refs(self._h)
        self.references = [lib.b3c_bam_ref_name(self._h, i).decode('ascii', 'replace') for i in range(n)]
        self.lengths = np.empty(n, dtype=np.int64)
        check(lib.b3c_bam_ref_lengths(self._h, self.lengths.ctypes.data, n))
        m = lib.b3c_bam_header_text(self._h, None, 0)
        buf = C.create_string_buffer(int(m) + 1)
        lib.b3c_bam_header_text(self._h, C.cast(buf, C.c_void_p), int(m) + 1)
        self.header_text = buf.value.decode('utf-8', 'replace')

    @property
    def n_refs(self):
        return len(self.references)

    def set_filter(self, min_mapq=0, strong=None, min_insert=None, tid2idx=None):
        """The matcher (contact_map.py:612-622) and the insert filter (:761-766); before the first read."""
        t = None
        if tid2idx is not None:
            t = np.ascontiguousarray(tid2idx, dtype=np.int32)
        check(lib.b3c_bam_set_filter(self._h, int(min_mapq), int(strong or 0), int(min_insert or 0),
                                     t.ctypes.data if t is not None else None, len(t) if t is not None else 0))

    def set_extent(self, tid2idx, grouping):
        """Also emit extent records (contact_map.py:779-788); `grouping` is a contact_map.ExtentGrouping."""
        t = np.ascontiguousarray(tid2idx, dtype=np.int32)
        first = np.ascontiguousarray(grouping.first_bin, dtype=np.int64)
        ptr = np.ascontiguousarray(grouping.edge_ptr, dtype=np.int64)
        upper = np.ascontiguousarray(grouping.upper_edges, dtype=np.int64)
        check(lib.b3c_bam_set_extent(self._h, t.ctypes.data, len(t), first.ctypes.data, ptr.ctypes.data,
                                     upper.ctypes.data, len(first)))

    def read_pairs_extent(self, capacity):
        """Up to `capacity` further (pair records, extent records); empty arrays at end of file."""
        rec = np.empty(int(capacity), dtype=np.uint64)
        ext = np.empty(int(capacity), dtype=np.uint64)
        n = check(lib.b3c_bam_read_pairs_extent(self._h, rec.ctypes.data, ext.ctypes.data, int(capacity)))
        return rec[:n], ext[:n]

    def set_tips(self, tip_size, tid2idx):
        """Emit tip records (contact_map.py:631-670, 791-798): doubled ids 2 * tid + tip; before the first read."""
        t = np.ascontiguousarray(tid2idx, dtype=np.int32)
        check(lib.b3c_bam_set_tips(self._h, int(tip_size), t.ctypes.data, len(t)))

    def read_pairs_tips(self, capacity):
        """Up to `capacity` further (tip records, flags of the accepted same-sequence (tail, head) pairs)."""
        rec = np.empty(int(capacity), dtype=np.uint64)
        t10 = np.empty(int(capacity), dtype=np.uint8)
        n = check(lib.b3c_bam_read_pairs_tips(self._h, rec.ctypes.data, t10.ctypes.data, int(capacity)))
        return rec[:n], t10[:n]

    def read_pairs(self, capacity, out=None):
        """Up to `capacity` further records (an empty array at end of file)."""
        if out is None:
            out = np.empty(int(capacity), dtype=np.uint64)
        assert out.dtype == np.uint64 and out.flags.c_contiguous and len(out) >= capacity
        n = check(lib.b3c_bam_read_pairs(self._h, out.ctypes.data, int(capacity)))
        return out[:n]

    def read_all(self, chunk=1 << 22):
        parts = []
        while True:
            r = self.read_pairs(chunk)
            if len(r) == 0:
                break
            parts.append(r.copy() if len(r) < chunk else r)
        return np.concatenate(parts) if parts else np.empty(0, dtype=np.uint64)

    def stats(self):
        s = np.zeros(len(STAT_NAMES), dtype=np.int64)
        check(lib.b3c_bam_stats(self._h, s.ctypes.data, len(s)))
        return dict(zip(STAT_NAMES, s.tolist()))

    def close(self):
        if self._h:
            lib.b3c_bam_close(self._h)
            self._h = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def pair_records_from_bam(path, sites=None, min_mapq=60, strong=None, min_insert=None, min_len=None, threads=0,
                          bin_size=None, tip_size=None, device=False, slab_bytes=DEFAULT_SLAB_BYTES, slab_blocks=None):
    """
    BAM file -> (PairRecords, stats): the object `ContactMap(bam_file=...)` takes in this package.

    :param sites: restriction-site count per BAM reference (the FASTA pass, contact_map.py:520-531, is not
                  part of this path); None -> ones.  A negative value marks "not in the FASTA".
    :param min_insert: needs `min_len` (and `sites`) to know which references are excluded, because the
                  reference applies the insert filter only to pairs that passed the exclusion test.
    :param tip_size: tip-based map (contact_map.py:631-670): records carry doubled ids 2 * tid + tip and
                  PairRecords.tip10 the same-sequence (tail, head) pairs; needs `min_len` like min_insert; `sites`
                  may then be an (n_refs, 2) array of (head, tail) site counts (seq_utils.py:146-158).
    :param device: decode on the GPU (bin3c_b200/csrc/bamdec.cu): the records come back as a CUDA uint64 tensor
                  with the values, order and stats of the host reader.  Only compressed bytes cross PCIe.  Contig-map
                  records only: with bin_size or tip_size it raises NotImplementedError.
    :param slab_bytes, slab_blocks: the device decoder reads the file in slabs of whole BGZF blocks, about slab_bytes
                  compressed bytes and at most slab_blocks blocks (default 65536) each
    """
    from .contact_map import PairRecords
    if device:
        if bin_size or tip_size:
            raise NotImplementedError('extent and tip records are not decoded on the GPU: read this BAM file with the '
                                      'host reader (device=False)')
        return _pair_records_on_device(path, sites, min_mapq, strong, min_insert, min_len, slab_bytes, slab_blocks)
    with BamPairReader(path, threads=threads) as bam:
        s = np.ones(bam.n_refs, dtype=np.int64) if sites is None else np.asarray(sites, dtype=np.int64)
        assert len(s) == bam.n_refs, 'one site count per BAM reference'
        in_fasta = (s >= 0) if s.ndim == 1 else (s >= 0).all(axis=1)
        tid2idx = None
        tip10 = None
        assert not (bin_size and tip_size), 'extent records and tip records do not combine in this build'
        if min_insert:
            assert min_len is not None, 'min_insert needs min_len'
            keep = (bam.lengths >= min_len) & in_fasta                 # contact_map.py:545-564
            tid2idx = np.where(keep, np.cumsum(keep) - 1, -1).astype(np.int32)
        if tip_size:
            assert min_len is not None, 'tip_size needs min_len'
            keep = (bam.lengths >= min_len) & in_fasta
            tid2idx = np.where(keep, np.cumsum(keep) - 1, -1).astype(np.int32)
            bam.set_tips(tip_size, tid2idx)
        extent = None
        if bin_size:
            # the extent map (bin3C mkmap --bin-size): bins over the sequences that pass the length filter
            from .contact_map import ExtentGrouping
            assert min_len is not None, 'bin_size needs min_len'
            keep = (bam.lengths >= min_len) & in_fasta
            tid2idx = np.where(keep, np.cumsum(keep) - 1, -1).astype(np.int32)
            bam.set_extent(tid2idx, ExtentGrouping.from_lengths(bam.lengths[keep], bin_size))
        bam.set_filter(min_mapq=min_mapq, strong=strong, min_insert=min_insert, tid2idx=tid2idx)
        if bin_size:
            parts = []
            while True:
                r, e = bam.read_pairs_extent(1 << 22)
                if len(r) == 0:
                    break
                parts.append((r, e))
            records = np.concatenate([p[0] for p in parts]) if parts else np.empty(0, dtype=np.uint64)
            extent = np.concatenate([p[1] for p in parts]) if parts else np.empty(0, dtype=np.uint64)
        elif tip_size:
            parts = []
            while True:
                r, t = bam.read_pairs_tips(1 << 22)
                if len(r) == 0:
                    break
                parts.append((r, t))
            records = np.concatenate([p[0] for p in parts]) if parts else np.empty(0, dtype=np.uint64)
            flags = np.concatenate([p[1] for p in parts]) if parts else np.empty(0, dtype=np.uint8)
            # BAM reference ids of the accepted same-sequence (tail, head) pairs
            tip10 = ((records[flags != 0] & np.uint64(0x7fffffff)) >> np.uint64(1)).astype(np.int64)
        else:
            records = bam.read_all()
        stats = bam.stats()
        meta = dict(min_mapq=min_mapq, strong=strong, min_insert=min_insert or None, min_len=min_len,
                    bin_size=bin_size or None, short_insert=stats['short_insert'], tip_size=tip_size or None,
                    not_tip=stats['not_tip'])
        return PairRecords(bam.lengths, s, records, references=bam.references, extent_records=extent, meta=meta,
                           tip10=tip10), stats


def _pair_records_on_device(path, sites, min_mapq, strong, min_insert, min_len, slab_bytes, slab_blocks):
    """
    pair_records_from_bam(device=True).  A read-ahead slab ring reads the file into two pinned slabs and lists each
    slab's BGZF blocks (b3c_bgzf_scan) while the device decodes the previous slab (include/bin3c_b200.h:
    b3c_bamdec_*); each slab goes to the device with one asynchronous copy, and the record tensor grows as slabs finish.
    """
    import torch
    from . import _cabi, slab_ring
    from .contact_map import PairRecords
    from .device import grown
    if not torch.cuda.is_available():
        raise RuntimeError('pair_records_from_bam(device=True) needs a CUDA device; the host reader is device=False')
    with BamPairReader(path, threads=1) as bam:                 # header, sort order, reference table
        references, lengths = bam.references, bam.lengths.copy()
        data_offset = int(check(lib.b3c_bam_data_offset(bam._h)))
    n_refs = len(references)
    s = np.ones(n_refs, dtype=np.int64) if sites is None else np.asarray(sites, dtype=np.int64)
    assert len(s) == n_refs, 'one site count per BAM reference'
    tid2idx = None
    if min_insert:
        assert min_len is not None, 'min_insert needs min_len'
        keep = (lengths >= min_len) & ((s >= 0) if s.ndim == 1 else (s >= 0).all(axis=1))
        tid2idx = np.where(keep, np.cumsum(keep) - 1, -1).astype(np.int32)
    slab_bytes = max(int(slab_bytes), 1)
    max_blocks = int(slab_blocks) if slab_blocks else 1 << 16
    assert max_blocks >= 1, 'slab_blocks must be positive'
    cap = slab_bytes + 65536                                    # always holds one whole block (BSIZE < 2^16)

    dev = torch.device('cuda', torch.cuda.current_device())
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    ws = torch.empty(int(_cabi.lib.b3c_bamdec_workspace_bytes(max_blocks, n_refs)), dtype=torch.uint8, device=dev)
    d_tid = torch.from_numpy(tid2idx).to(dev) if tid2idx is not None else None
    _cabi.check(_cabi.lib.b3c_bamdec_begin(ws.data_ptr(), ws.numel(), int(min_mapq), int(strong or 0),
                                           int(min_insert or 0), d_tid.data_ptr() if d_tid is not None else None,
                                           n_refs, data_offset, stream))

    pinned = [torch.empty(cap, dtype=torch.uint8, pin_memory=True) for _ in range(2)]
    left, eof = np.empty(0, dtype=np.uint8), False

    def fill(a):                                                # the ring's thread: the carried bytes, then the file
        nonlocal left, eof
        n = len(left)
        a[:n] = left
        while n < cap and not eof:
            m = f.readinto(memoryview(a)[n:cap])
            eof = not m
            n += m or 0
        offs = np.empty(max_blocks, dtype=np.int64)
        bsz = np.empty(max_blocks, dtype=np.int32)
        isz = np.empty(max_blocks, dtype=np.int32)
        used = np.zeros(1, dtype=np.int64)
        nb = lib.b3c_bgzf_scan(a.ctypes.data, n, 1 if eof else 0, offs.ctypes.data, bsz.ctypes.data,
                               isz.ctypes.data, max_blocks, used.ctypes.data)
        if nb < 0:
            raise ValueError('{}: {}'.format(path, last_error()))  # the reader's status for a bad BGZF block
        c = int(used[0])
        left = a[c:n].copy()
        return int(nb), c, offs[:nb], bsz[:nb], isz[:nb], eof and c == n

    with open(path, 'rb') as f, slab_ring.SlabRing([p.numpy() for p in pinned], fill=fill) as ring:
        d_comp = torch.empty(cap, dtype=torch.uint8, device=dev)
        u_bufs = [None, None]
        out = torch.empty(1 << 20, dtype=torch.uint64, device=dev)
        n_out, stream_off, next_rec = 0, 0, data_offset
        prev_u, prev_u0, repaired, n_slabs = None, 0, 0, 0
        res = (C.c_int64 * 4)()
        for k, (nb, c, offs, bsz, isz, last) in ring:
            tbl = np.empty((nb, 3), dtype=np.int64)
            tbl[:, 0] = offs
            tbl[:, 1] = bsz.astype(np.int64) | (isz.astype(np.int64) << 32)
            u_off = np.cumsum(isz, dtype=np.int64)
            tbl[:, 2] = u_off - isz
            u_bytes = int(u_off[-1]) if nb else 0
            carry = max(0, stream_off - next_rec)
            slot = n_slabs & 1
            need = carry + u_bytes
            if u_bufs[slot] is None or u_bufs[slot].numel() < max(need, 1):
                u_bufs[slot] = None
                u_bufs[slot] = torch.empty(max(need + need // 4, 1 << 16), dtype=torch.uint8, device=dev)
            u = u_bufs[slot]
            d_carry = prev_u.data_ptr() + (next_rec - prev_u0) if carry else None
            bound = need // 72 + 2
            if out.numel() - n_out < bound:
                out = grown(out, max(2 * out.numel(), n_out + bound), n_out)
            if c:
                d_comp[:c].copy_(pinned[k][:c], non_blocking=True)
            d_tbl = torch.from_numpy(tbl.reshape(-1)).pin_memory().to(dev, non_blocking=True) if nb else None
            rc = _cabi.lib.b3c_bamdec_slab(ws.data_ptr(), d_comp.data_ptr(), d_tbl.data_ptr() if nb else None, nb,
                                           stream_off, u_bytes, d_carry, carry, u.data_ptr(), u.numel(),
                                           1 if last else 0, out.data_ptr() + 8 * n_out, out.numel() - n_out, res,
                                           stream)
            ring.release(k)                                     # the slab call synchronised: the pinned slab is free
            if rc == _cabi.B3C_ERR_FORMAT:
                raise ValueError('{}: {}'.format(path, _cabi.last_error()))
            _cabi.check(rc)
            n_out += int(res[0])
            prev_u, prev_u0 = u, stream_off - carry
            next_rec = int(res[1])
            repaired += int(res[2])
            stream_off += u_bytes
            n_slabs += 1
    st = np.zeros(8, dtype=np.int64)
    _cabi.check(_cabi.lib.b3c_bamdec_stats(ws.data_ptr(), st.ctypes.data_as(C.POINTER(C.c_int64)), 8, stream))
    stats = dict(zip(STAT_NAMES, st.tolist() + [0]))
    meta = dict(min_mapq=min_mapq, strong=strong, min_insert=min_insert or None, min_len=min_len, bin_size=None,
                short_insert=stats['short_insert'], tip_size=None, not_tip=0, gpu_decode=True, slabs=n_slabs,
                repaired_blocks=repaired)
    return PairRecords(lengths, s, out[:n_out], references=references, meta=meta), stats


def records_bytes(n_refs):
    """The narrowest record (5, 6 or 8 bytes) that holds the reference ids of a table of n_refs entries."""
    return int(lib.b3c_records_bytes(int(n_refs)))


def pack_records(records, bytes_per_record, out=None, threads=0):
    """uint64 native records -> narrow records (uint8 array, length a multiple of 8) for HotPath / add_pairs_packed."""
    r = np.ascontiguousarray(records, dtype=np.uint64)
    nbytes = (len(r) * bytes_per_record + 7) // 8 * 8
    if out is None:
        out = np.empty(nbytes, dtype=np.uint8)
    assert out.dtype == np.uint8 and out.flags.c_contiguous and len(out) >= nbytes
    check(lib.b3c_records_pack(r.ctypes.data, len(r), int(bytes_per_record), out.ctypes.data, int(threads)))
    return out[:nbytes]


def split_records(records, n_refs, pin=False, threads=0):
    """
    uint64 native records -> device.SplitRecords, the narrowest form for the host->device copy: the pairs whose mates
    lie on one reference as 3- / 4-byte records, the rest as 5- / 6- / 8-byte pair records (b3c_records_split).
    `pin`: allocate the two buffers in pinned host memory (asynchronous copies).
    """
    import torch
    from .device import SplitRecords
    r = np.ascontiguousarray(records, dtype=np.uint64)
    B, Bs = records_bytes(n_refs), int(lib.b3c_records_same_bytes(int(n_refs)))
    assert Bs in (3, 4), 'reference table too large for same-reference records'
    cnt = np.zeros(2, dtype=np.int64)
    check(lib.b3c_records_split(r.ctypes.data, len(r), B, Bs, None, None, cnt.ctypes.data, int(threads)))
    n_same, n_pair = int(cnt[0]), int(cnt[1])
    same = torch.empty((n_same * Bs + 7) // 8 * 8, dtype=torch.uint8, pin_memory=bool(pin))
    pair = torch.empty((n_pair * B + 7) // 8 * 8, dtype=torch.uint8, pin_memory=bool(pin))
    check(lib.b3c_records_split(r.ctypes.data, len(r), B, Bs, same.numpy().ctypes.data, pair.numpy().ctypes.data,
                                cnt.ctypes.data, int(threads)))
    return SplitRecords(same, n_same, Bs, pair, n_pair, B)


def unsplit_records(split):
    """device.SplitRecords (host) -> uint64 native records: the same-reference ones first, then the others."""
    s = np.ascontiguousarray(split.same.numpy())
    Bs, ts = split.bytes_same, 8 * split.bytes_same - 1
    v = np.zeros(split.n_same, dtype=np.uint64)
    for k in range(Bs):
        v |= s[k:split.n_same * Bs:Bs].astype(np.uint64) << np.uint64(8 * k)
    t = v & np.uint64((1 << ts) - 1)
    t[t == np.uint64((1 << ts) - 1)] = np.uint64(0x7fffffff)
    same = t | (((v >> np.uint64(ts)) & np.uint64(1)) << np.uint64(31)) | (t << np.uint64(32))
    pairs = unpack_records(split.pairs.numpy(), split.n_pairs, split.bytes_pair)
    return np.concatenate([same, pairs])


def unpack_records(packed, n, bytes_per_record):
    b = np.ascontiguousarray(packed, dtype=np.uint8)
    out = np.empty(int(n), dtype=np.uint64)
    check(lib.b3c_records_unpack(b.ctypes.data, int(n), int(bytes_per_record), out.ctypes.data))
    return out


def format_weight(w, float_style=FLOAT_REPR):
    buf = C.create_string_buffer(40)
    n = lib.b3c_format_weight_fmt(float(w), int(float_style), C.cast(buf, C.c_void_p), 40)
    check(n)
    return buf.value.decode('ascii')


def _is_cuda(x):
    return bool(getattr(x, 'is_cuda', False))


def write_edges(u, v, w, path, sep=' ', float_style=FLOAT_REPR, threads=0):
    """
    One 'u v weight' line per edge, as nx.write_edgelist(g, path, data=['weight'], delimiter=sep).  Returns the bytes
    written.  Host arrays are formatted by the host writer (b3c_edges_write_fmt, `threads` threads); when u, v and w
    are all CUDA tensors (cluster.to_edges(..., device=True)) the lines are formatted on their device and only the
    text crosses PCIe (_write_edges_on_device).  The file is the same byte for byte either way.
    """
    cuda = [_is_cuda(x) for x in (u, v, w)]
    if any(cuda):
        assert all(cuda), 'u, v and w must be all CUDA tensors or all host arrays'
        return _write_edges_on_device(u, v, w, path, sep, float_style)
    u = np.ascontiguousarray(u, dtype=np.int32)
    v = np.ascontiguousarray(v, dtype=np.int32)
    w = np.ascontiguousarray(w, dtype=np.float64)
    assert len(u) == len(v) == len(w)
    assert isinstance(sep, str) and len(sep) == 1, 'single-character separator'
    return check(lib.b3c_edges_write_fmt(os.fsencode(path), u.ctypes.data, v.ctypes.data, w.ctypes.data, len(u),
                                         sep.encode('ascii'), int(float_style), int(threads)))


DEFAULT_EDGE_CHUNK = 1 << 21      # edges per device formatting call (text buffers of 49 bytes per edge)


def _write_edges_on_device(u, v, w, path, sep=' ', float_style=FLOAT_REPR, chunk_edges=DEFAULT_EDGE_CHUNK):
    """
    write_edges for CUDA tensors.  The device formats chunk_edges edges at a time into a text buffer
    (include/bin3c_b200.h: b3c_edges_text); each chunk's text is copied into one of two pinned host slabs, and a
    write-behind slab ring writes slab k to the file while the device formats chunk k + 1.  Returns the bytes written.
    """
    import torch
    from . import _cabi, slab_ring
    assert len(u) == len(v) == len(w)
    assert isinstance(sep, str) and len(sep) == 1, 'single-character separator'
    sep_byte = sep.encode('ascii')[0]
    assert float_style in (FLOAT_REPR, FLOAT_STR12), 'float_style is FLOAT_REPR or FLOAT_STR12'
    dev = u.device
    assert v.device == dev and w.device == dev, 'u, v and w must be on one device'
    chunk = max(1, int(chunk_edges))
    n = len(u)
    with open(path, 'wb') as f, torch.cuda.device(dev):
        if n == 0:
            return 0
        u = u.reshape(-1).to(torch.int32).contiguous()
        v = v.reshape(-1).to(torch.int32).contiguous()
        w = w.reshape(-1).to(torch.float64).contiguous()
        chunk = min(chunk, n)
        cap = _cabi.B3C_EDGES_MAX_LINE_BYTES * chunk
        stream = torch.cuda.current_stream()
        ws = torch.empty(int(_cabi.lib.b3c_edges_text_workspace_bytes(chunk)), dtype=torch.uint8, device=dev)
        text = torch.empty(cap, dtype=torch.uint8, device=dev)
        slabs = [torch.empty(cap, dtype=torch.uint8, pin_memory=True) for _ in range(2 if n > chunk else 1)]
        nbytes = C.c_int64()
        total = 0
        with slab_ring.SlabRing([s.numpy() for s in slabs], drain=lambda a, nb: f.write(memoryview(a)[:nb])) as ring:
            for lo in range(0, n, chunk):
                m = min(chunk, n - lo)
                _cabi.check(_cabi.lib.b3c_edges_text(ws.data_ptr(), ws.numel(), u.data_ptr() + 4 * lo,
                                                     v.data_ptr() + 4 * lo, w.data_ptr() + 8 * lo, m, sep_byte,
                                                     int(float_style), text.data_ptr(), cap, C.byref(nbytes),
                                                     C.c_void_p(stream.cuda_stream)))
                k = ring.acquire()
                nb = int(nbytes.value)
                slabs[k][:nb].copy_(text[:nb], non_blocking=True)
                stream.synchronize()
                ring.release(k, nb)
                total += nb
    return total
