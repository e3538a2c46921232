"""
Serialisation of whole objects, as the reference's stage hand-off does it (mzd/io_utils.py:12-32: gzip +
cPickle of the whole ContactMap after `mkmap`, bin3C.py:165; read back by `cluster`, bin3C.py:176).

    save_object(file_name, obj)                 io_utils.py:12-21   (.gz appended if missing)
    load_object(file_name)                      io_utils.py:24-32   (gzip / bz2 / plain by suffix)
    save_object(file_name, obj, stock=True)     the same file written so that a STOCK bin3C run can read it
    save_object(file_name, obj, device=True)    the same pickle, deflated on the GPU as BGZF-framed gzip
    load_object(file_name, device=True)         a file of save_object(device=True), inflated on the GPU

The device path (include/bin3c_b200.h: b3c_bgzf_*) writes a multi-member gzip file: the pickle cut into 65280-byte
pieces, each one gzip member with the BGZF header, then the 28-byte BGZF end-of-file member.  Python's gzip (2.7 and
3) reads it, so load_object(device=False) and a stock `cluster` open it unchanged; the file carries no name or time
and is the same on every run.  load_object(device=True) reads only such BGZF files.

Interchange with a stock run (SURVEY section 8f-5).  A stock run is Python 2.7 + NumPy 1.14 + SciPy 1.1, and its
classes live in `mzd.contact_map`.  A Python 3 pickle of this package's ContactMap is useless to it three times
over: protocol > 2, module paths that do not exist there (`numpy._core`, `scipy.sparse._coo`, `bin3c_b200.*`) and
object layouts that changed (SciPy's `coo_matrix.coords`, NumPy's `RandomState` state dict).  `stock=True` therefore
does not use the pickle module to write: `_StockWriter` emits the protocol-2 opcodes itself --

  * `ContactMap`, `SeqOrder` and `ExtentGrouping` as instances of the reference's CLASSIC classes (MARK, GLOBAL,
    OBJ, state dict, BUILD: what cPickle emits for `class ContactMap:`), with the reference's attribute set
    (contact_map.py:492-518: `seq_map` / `processed_map` as plain attributes, no device or cache fields);
  * `SeqInfo` as `mzd.contact_map.SeqInfo(*fields)`;
  * arrays and dtypes through their own `__reduce__` under the NumPy 1.14 paths (`numpy.core.multiarray._reconstruct`,
    raw data as a Python 2 `str`);
  * sparse matrices as `scipy.sparse.coo.coo_matrix` / `csr.csr_matrix` with SciPy 1.1's attribute layout
    (`row`, `col`, `data`, `_shape`, `maxprint`);
  * `RandomState` through `numpy.random.__RandomState_ctor` with the legacy state tuple;
  * ASCII text as Python 2 `str` (attribute names, sequence names, enzyme names), anything else as `unicode`.

`load_object` reads both directions: files written here, and files written by a stock run (protocol 0 INST / OBJ
records of `mzd.contact_map.*`, `scipy.sparse.coo.coo_matrix` state with `row` / `col`, latin-1 byte strings).
There is no Python 2 interpreter in this image, so the stock side of the interchange is checked structurally (every
global the stream names exists in the pinned stack, no opcode beyond protocol 2: tests/test_io_utils.py) and by
reading the stream back through the stock-layout loader; it has not been loaded by a Python 2 process.
"""
import bz2
import gzip
import io
import pickle
import struct

import numpy as np
import scipy.sparse as scisp

# default buffer for incremental read/write (io_utils.py:9)
DEF_BUFFER = 16384

STOCK_MODULE = 'mzd.contact_map'

# attributes of the reference's ContactMap (contact_map.py:492-518, 568-574) in a stock pickle
STOCK_CONTACT_MAP_ATTRS = (
    'strong', 'bam_file', 'bin_size', 'min_mapq', 'min_insert', 'min_len', 'min_sig', 'min_extent', 'min_size',
    'max_fold', 'random_state', 'seq_info', 'seq_map', 'seq_file', 'grouping', 'extent_map', 'order', 'tip_size',
    'precount', 'total_reads', 'cov_info', 'processed_map', 'primary_acceptance_mask', 'bisto_scale', 'seq_analyzer',
    'enzymes', 'total_len', 'total_seq', 'current_mask')
STOCK_SEQ_ORDER_ATTRS = ('_positions', 'order')
STOCK_GROUPING_ATTRS = ('bins', 'bin_size', 'map', 'borders', 'centers', 'total_bins')


def open_input(file_name):
    """Open a file for reading; the suffix says whether it is compressed (io_utils.py:35-50)."""
    suffix = file_name.split('.')[-1].lower()
    if suffix == 'bz2':
        return bz2.BZ2File(file_name, 'r')
    elif suffix == 'gz':
        return gzip.GzipFile(file_name, 'r')
    return open(file_name, 'rb')


def open_output(file_name, append=False, compress=None, gzlevel=6):
    """Open a file for writing, optionally compressed; the suffix is appended if missing (io_utils.py:53-88)."""
    mode = 'ab' if append else 'wb'
    if compress == 'bzip2':
        if not file_name.endswith('.bz2'):
            file_name += '.bz2'
        return bz2.BZ2File(file_name, mode[0])
    elif compress == 'gzip':
        if not file_name.endswith('.gz'):
            file_name += '.gz'
        return gzip.GzipFile(file_name, mode, compresslevel=gzlevel)
    elif compress is None:
        return open(file_name, mode)
    raise RuntimeError('Unknown compression type {}'.format(compress))


def save_object(file_name, obj, stock=False, device=False, slab_members=None):
    """
    Serialise an object to a gzip-compressed file (io_utils.py:12-21).  stock=True: readable by a stock bin3C.
    device=True: deflated on the GPU (BGZF framing, see the module docstring); slab_members = 65280-byte members per
    host slab (default DEFAULT_SLAB_MEMBERS), which changes nothing in the file.
    """
    if device:
        return _save_on_device(file_name, obj, stock, slab_members or DEFAULT_SLAB_MEMBERS)
    with open_output(file_name, compress='gzip') as out_h:
        if stock:
            out_h.write(dumps_stock(obj))
        else:
            pickle.dump(obj, out_h, protocol=pickle.HIGHEST_PROTOCOL)


def load_object(file_name, device=False, slab_bytes=None):
    """
    Deserialise an object written by save_object here or by a stock bin3C run (io_utils.py:24-32).  device=True:
    a file of save_object(device=True), inflated on the GPU and read slab_bytes compressed bytes at a time.
    """
    if device:
        return loads(_inflate_on_device(file_name, slab_bytes or DEFAULT_LOAD_SLAB_BYTES))
    with open_input(file_name) as in_h:
        return loads(in_h.read())


# ---- the device path: BGZF-framed gzip deflated and inflated on the GPU -------------------------------------------

MEMBER_INPUT = 65280                  # pickle bytes per gzip member (include/bin3c_b200.h: B3C_BGZF_MEMBER_INPUT)
MEMBER_MAX = 65536
DEFAULT_SLAB_MEMBERS = 512            # 33 MB of pickle per host slab
DEFAULT_LOAD_SLAB_BYTES = 64 << 20
BGZF_EOF = bytes.fromhex('1f8b08040000000000ff0600424302001b0003000000000000000000')


class _SlabWriter(object):
    """The file object pickle writes to: fills the write-behind ring's slabs and hands each full one over."""

    def __init__(self, ring, views):
        self.ring, self.views = ring, views
        self.k, self.n = ring.acquire(), 0

    def write(self, b):
        mv = memoryview(b).cast('B')
        done, total = 0, len(mv)
        while done < total:
            a = self.views[self.k]
            m = min(len(a) - self.n, total - done)
            a[self.n:self.n + m] = mv[done:done + m]
            self.n += m
            done += m
            if self.n == len(a):
                self.ring.release(self.k, self.n)
                self.k, self.n = self.ring.acquire(), 0
        return total

    def close(self):
        if self.n:
            self.ring.release(self.k, self.n)
        self.n = 0


def _cuda(what):
    import torch
    if not torch.cuda.is_available():
        raise RuntimeError('{}(device=True) needs a CUDA device; the host path is device=False'.format(what))
    return torch


def _save_on_device(file_name, obj, stock, slab_members):
    """
    save_object(device=True).  pickle writes into pinned slabs of slab_members members; a write-behind slab ring
    deflates each full slab on the device (b3c_bgzf_deflate) and writes its members to the file while the next
    slab fills.
    """
    import ctypes as C
    torch = _cuda('save_object')
    from . import _cabi, slab_ring
    if not file_name.endswith('.gz'):
        file_name += '.gz'
    k = int(slab_members)
    assert k >= 1, 'slab_members must be positive'
    with open(file_name, 'wb') as f:
        dev = torch.device('cuda', torch.cuda.current_device())
        ws = torch.empty(int(_cabi.lib.b3c_bgzf_deflate_workspace_bytes(k)), dtype=torch.uint8, device=dev)
        d_in = torch.empty(k * MEMBER_INPUT, dtype=torch.uint8, device=dev)
        d_out = torch.empty(k * MEMBER_MAX, dtype=torch.uint8, device=dev)
        h_out = torch.empty(k * MEMBER_MAX, dtype=torch.uint8, pin_memory=True)
        slabs = [torch.empty(k * MEMBER_INPUT, dtype=torch.uint8, pin_memory=True) for _ in range(2)]
        out_bytes = C.c_int64()

        def drain(slab, nbytes):                        # the ring's thread
            with torch.cuda.device(dev):
                stream = torch.cuda.current_stream()
                d_in[:nbytes].copy_(slab[:nbytes], non_blocking=True)
                _cabi.check(_cabi.lib.b3c_bgzf_deflate(ws.data_ptr(), ws.numel(), d_in.data_ptr(), nbytes,
                                                       d_out.data_ptr(), d_out.numel(), C.byref(out_bytes),
                                                       C.c_void_p(stream.cuda_stream)))
                m = int(out_bytes.value)
                h_out[:m].copy_(d_out[:m])
            f.write(memoryview(h_out.numpy())[:m])

        with slab_ring.SlabRing(slabs, drain=drain) as ring:
            w = _SlabWriter(ring, [t.numpy() for t in slabs])
            if stock:
                w.write(dumps_stock(obj))
            else:
                pickle.dump(obj, w, protocol=pickle.HIGHEST_PROTOCOL)
            w.close()
        f.write(BGZF_EOF)


def _inflate_on_device(file_name, slab_bytes):
    """
    The bytes of a file of save_object(device=True).  A read-ahead slab ring reads the file into two pinned slabs
    and lists each slab's members (b3c_bgzf_scan of libbin3c_io.so) while the device inflates the previous slab
    and checks every member's CRC-32 and ISIZE (b3c_bgzf_inflate).
    """
    import ctypes as C
    torch = _cuda('load_object')
    from . import _cabi, bam_io, slab_ring
    cap = max(int(slab_bytes), 1) + MEMBER_MAX           # always holds one whole member
    max_blocks = cap // 28 + 1                           # the shortest member is the end-of-file one
    dev = torch.device('cuda', torch.cuda.current_device())
    with open(file_name, 'rb') as f:
        pinned = [torch.empty(cap, dtype=torch.uint8, pin_memory=True) for _ in range(2)]
        left, eof, first = np.empty(0, dtype=np.uint8), False, [True]

        def fill(a):                                     # the ring's thread: the carried bytes, then the file
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
            nb = bam_io.lib.b3c_bgzf_scan(a.ctypes.data, n, 1 if eof else 0, offs.ctypes.data, bsz.ctypes.data,
                                          isz.ctypes.data, max_blocks, used.ctypes.data)
            if nb < 0:
                msg = bam_io.last_error()
                if first[0] and 'not a BGZF file' in msg:
                    msg += ': load_object(device=True) reads the BGZF files of save_object(device=True); ' \
                           'read this file with device=False'
                raise ValueError('{}: {}'.format(file_name, msg))
            first[0] = False
            c = int(used[0])
            left = a[c:n].copy()
            last_eof = bool(nb) and isz[nb - 1] == 0 and bytes(a[offs[nb - 1]:c]) == BGZF_EOF
            return int(nb), c, offs[:nb], bsz[:nb], isz[:nb], last_eof, eof and c == n

        parts, ends_with_eof = [], False
        stream = torch.cuda.current_stream()
        ws = torch.empty(8, dtype=torch.uint8, device=dev)
        d_comp = torch.empty(cap, dtype=torch.uint8, device=dev)
        d_u = h_u = None
        with slab_ring.SlabRing([p.numpy() for p in pinned], fill=fill) as ring:
            for k, (nb, c, offs, bsz, isz, last_eof, last) in ring:
                ends_with_eof = last_eof if nb else ends_with_eof
                tbl = np.empty((nb, 3), dtype=np.int64)
                tbl[:, 0] = offs
                tbl[:, 1] = bsz.astype(np.int64) | (isz.astype(np.int64) << 32)
                u_off = np.cumsum(isz, dtype=np.int64)
                tbl[:, 2] = u_off - isz
                u_bytes = int(u_off[-1]) if nb else 0
                if u_bytes and (d_u is None or d_u.numel() < u_bytes):
                    d_u = torch.empty(u_bytes, dtype=torch.uint8, device=dev)
                    h_u = torch.empty(u_bytes, dtype=torch.uint8, pin_memory=True)
                if c:
                    d_comp[:c].copy_(pinned[k][:c], non_blocking=True)
                d_tbl = torch.from_numpy(tbl.reshape(-1)).to(dev) if nb else None
                rc = _cabi.lib.b3c_bgzf_inflate(ws.data_ptr(), ws.numel(), d_comp.data_ptr(),
                                                d_tbl.data_ptr() if nb else None, nb,
                                                d_u.data_ptr() if u_bytes else None, u_bytes,
                                                C.c_void_p(stream.cuda_stream))
                ring.release(k)                          # the call synchronised: the pinned slab is free
                if rc == _cabi.B3C_ERR_FORMAT:
                    raise ValueError('{}: {}'.format(file_name, _cabi.last_error()))
                _cabi.check(rc)
                if u_bytes:
                    h_u[:u_bytes].copy_(d_u[:u_bytes])
                    parts.append(h_u[:u_bytes].numpy().tobytes())
    if not ends_with_eof:
        raise ValueError('{}: the file does not end with the BGZF end-of-file member (truncated?)'.format(file_name))
    return b''.join(parts)


# ---- writer: protocol-2 opcodes for the stock stack -----------------------------------------------------------

class _StockWriter(object):

    def __init__(self):
        self.out = io.BytesIO()
        self.w = self.out.write

    # -- primitives
    def glob(self, module, name):
        self.w(b'c' + module.encode('ascii') + b'\n' + name.encode('ascii') + b'\n')

    def py2_str(self, raw):
        n = len(raw)
        if n < 256:
            self.w(b'U' + bytes([n]) + raw)
        else:
            self.w(b'T' + struct.pack('<i', n) + raw)

    def text(self, s):
        try:
            self.py2_str(s.encode('ascii'))
        except UnicodeEncodeError:
            raw = s.encode('utf-8')
            self.w(b'X' + struct.pack('<I', len(raw)) + raw)

    def integer(self, v):
        if 0 <= v < 256:
            self.w(b'K' + bytes([v]))
        elif 0 <= v < 65536:
            self.w(b'M' + struct.pack('<H', v))
        elif -0x80000000 <= v <= 0x7fffffff:
            self.w(b'J' + struct.pack('<i', v))
        else:
            raw = v.to_bytes((v.bit_length() + 8) // 8, 'little', signed=True)
            self.w(b'\x8a' + bytes([len(raw)]) + raw)

    def sequence(self, items, empty, add_many):
        self.w(empty)
        items = list(items)
        for i in range(0, len(items), 1000):
            self.w(b'(')
            for it in items[i:i + 1000]:
                self.save(it)
            self.w(add_many)

    def mapping(self, d):
        self.w(b'}')
        items = list(d.items())
        for i in range(0, len(items), 1000):
            self.w(b'(')
            for k, v in items[i:i + 1000]:
                self.save(k)
                self.save(v)
            self.w(b'u')

    def tup(self, t):
        n = len(t)
        if n == 0:
            self.w(b')')
            return
        if n > 3:
            self.w(b'(')
        for it in t:
            self.save(it)
        self.w({1: b'\x85', 2: b'\x86', 3: b'\x87'}.get(n, b't'))

    def classic_instance(self, name, state):
        # what cPickle writes for an instance of a classic class without __getinitargs__
        self.w(b'(')
        self.glob(STOCK_MODULE, name)
        self.w(b'o')
        self.mapping(state)
        self.w(b'b')

    # -- NumPy / SciPy
    _np_globals = None

    def np_reduce(self, obj):
        fn, args, state = obj.__reduce__()[:3]
        if fn is np.dtype or isinstance(obj, np.dtype):
            self.glob('numpy', 'dtype')
        else:
            self.glob('numpy.core.multiarray', '_reconstruct')
        self.tup(args)
        self.w(b'R')
        self.save(state)
        self.w(b'b')

    def sparse(self, m):
        if scisp.isspmatrix_coo(m) or isinstance(m, scisp.coo_array):
            self.glob('scipy.sparse.coo', 'coo_matrix')
            state = {'row': m.row, 'col': m.col, 'data': m.data}
        elif scisp.isspmatrix_csr(m) or isinstance(m, scisp.csr_array):
            self.glob('scipy.sparse.csr', 'csr_matrix')
            state = {'indices': m.indices, 'indptr': m.indptr, 'data': m.data}
        else:
            raise TypeError('stock pickle: sparse format {} is not stored on a ContactMap'.format(m.format))
        state['_shape'] = tuple(int(x) for x in m.shape)
        state['maxprint'] = 50
        self.w(b')\x81')                     # NEWOBJ: cls.__new__(cls)
        self.mapping(state)
        self.w(b'b')

    def random_state(self, rs):
        self.glob('numpy.random', '__RandomState_ctor')
        self.w(b')R')
        kind, key, pos, has_gauss, cached = rs.get_state(legacy=True)
        self.tup((kind, np.asarray(key, dtype=np.uint32), int(pos), int(has_gauss), float(cached)))
        self.w(b'b')

    # -- dispatch
    def save(self, obj):
        from . import contact_map as cm
        if obj is None:
            self.w(b'N')
        elif obj is True or (isinstance(obj, np.bool_) and bool(obj)):
            self.w(b'\x88')
        elif obj is False or isinstance(obj, np.bool_):
            self.w(b'\x89')
        elif isinstance(obj, (int, np.integer)):
            self.integer(int(obj))
        elif isinstance(obj, (float, np.floating)):
            self.w(b'G' + struct.pack('>d', float(obj)))
        elif isinstance(obj, str):
            self.text(obj)
        elif isinstance(obj, (bytes, bytearray)):
            self.py2_str(bytes(obj))
        elif isinstance(obj, cm.SeqInfo):
            self.glob(STOCK_MODULE, 'SeqInfo')
            self.tup(tuple(obj))
            self.w(b'R')
        elif isinstance(obj, tuple):
            self.tup(obj)
        elif isinstance(obj, list):
            self.sequence(obj, b']', b'e')
        elif isinstance(obj, dict):
            self.mapping(obj)
        elif isinstance(obj, type) and issubclass(obj, np.generic):
            self.glob('numpy', obj.__name__)                    # e.g. the ndarray subtype slot of _reconstruct
        elif obj is np.ndarray:
            self.glob('numpy', 'ndarray')
        elif isinstance(obj, (np.ndarray, np.dtype)):
            self.np_reduce(obj)
        elif scisp.issparse(obj):
            self.sparse(obj)
        elif isinstance(obj, np.random.RandomState):
            self.random_state(obj)
        elif isinstance(obj, cm.ContactMap):
            self.classic_instance('ContactMap', stock_state(obj))
        elif isinstance(obj, cm.SeqOrder):
            self.classic_instance('SeqOrder', {k: getattr(obj, k) for k in STOCK_SEQ_ORDER_ATTRS})
        elif isinstance(obj, cm.ExtentGrouping):
            self.classic_instance('ExtentGrouping', {k: getattr(obj, k) for k in STOCK_GROUPING_ATTRS})
        else:
            raise TypeError('stock pickle: no Python 2 form for {!r}'.format(type(obj)))


def stock_state(cmap):
    """The attribute dict a stock ContactMap carries (contact_map.py:492-518) taken from one of ours."""
    state = {}
    for k in STOCK_CONTACT_MAP_ATTRS:
        v = getattr(cmap, k, None)
        if k == 'seq_file' and not isinstance(v, (str, type(None))):
            v = None                         # site counts were given as an array / dict / callable
        state[k] = v
    return state


def dumps_stock(obj):
    """Protocol-2 pickle of `obj` in the layout of the reference's pinned stack (see the module docstring)."""
    wr = _StockWriter()
    wr.w(b'\x80\x02')
    wr.save(obj)
    wr.w(b'.')
    return wr.out.getvalue()


# ---- reader: this package's pickles and a stock run's -----------------------------------------------------------

class _StockSparse(object):
    """Stand-in for a SciPy 1.1 sparse matrix while a stock pickle loads (its state names `row` / `col`, which are
    read-only properties of today's classes); `real()` builds today's object."""
    kind = None

    def __setstate__(self, state):
        self.__dict__.update(state)

    def real(self):
        if self.kind == 'coo':
            return scisp.coo_matrix((np.asarray(self.data), (np.asarray(self.row), np.asarray(self.col))),
                                    shape=tuple(self._shape))
        return scisp.csr_matrix((np.asarray(self.data), np.asarray(self.indices), np.asarray(self.indptr)),
                                shape=tuple(self._shape))


class _StockCoo(_StockSparse):
    kind = 'coo'


class _StockCsr(_StockSparse):
    kind = 'csr'


def unstock(v):
    """Stand-ins of a stock pickle -> today's objects (containers are walked)."""
    if isinstance(v, _StockSparse):
        return v.real()
    if isinstance(v, list):
        return [unstock(x) for x in v]
    if isinstance(v, dict):
        return {k: unstock(x) for k, x in v.items()}
    return v


class _Unpickler(pickle.Unpickler):

    def find_class(self, module, name):
        from . import contact_map as cm
        if module == STOCK_MODULE and name in ('ContactMap', 'SeqOrder', 'ExtentGrouping', 'SeqInfo'):
            return getattr(cm, name)
        if module in ('scipy.sparse.coo', 'scipy.sparse._coo') and name == 'coo_matrix' and module.endswith('.coo'):
            return _StockCoo
        if module == 'scipy.sparse.csr' and name == 'csr_matrix':
            return _StockCsr
        if module == 'numpy.core.multiarray' and name == '_reconstruct':
            return np.ndarray.__reduce__(np.empty(0))[0]
        if module == 'numpy.random' and name == '__RandomState_ctor':
            return _random_state_ctor
        if module == 'mzd.exceptions':
            from . import exceptions
            return getattr(exceptions, name)
        return super(_Unpickler, self).find_class(module, name)


def _random_state_ctor():
    return np.random.RandomState(seed=0)


def loads(raw):
    """Object from a pickle written here (any protocol) or by a stock bin3C run (Python 2 byte strings as latin-1)."""
    obj = _Unpickler(io.BytesIO(raw), encoding='latin1').load()
    return unstock(obj)
