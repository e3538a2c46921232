"""
TEST INFRASTRUCTURE -- NOT PRODUCT CODE.

Runs the reference's own hot-path functions (cerebis/bin3C, Python 2.7) verbatim under
Python 3 by exec'ing line ranges of its source, from a checkout of the reference at
$BIN3C_REFERENCE (default oracle/_ref/, which git ignores): cerebis/bin3C at commit
76ad2a9, with its Infomap binary built at external/Infomap.  No reference source is
committed to this repository.  It is used by tests/golden/make_golden*.py to produce
the committed golden vectors that pin oracle/oracle.py, and by the "pinning" tests,
which skip when no reference checkout is present.

Shims (SURVEY.md section 8c): np.int/np.float/np.bool aliases, xrange = range, and a
`.H` property on SciPy sparse classes (removed from SciPy >= 1.14) used by
sparse_utils.py:18.
"""
import logging
import os
import textwrap

import numpy as np
import scipy.sparse as scisp

REFERENCE_ROOT = os.environ.get('BIN3C_REFERENCE', os.path.join(os.path.dirname(os.path.abspath(__file__)), '_ref'))

# (file, first line, last line) of each function executed verbatim
SLICES = {
    'is_hermitian': ('mzd/sparse_utils.py', 10, 18),
    'kr_biostochastic': ('mzd/sparse_utils.py', 90, 224),
    'Sparse2DAccumulator': ('mzd/sparse_utils.py', 227, 266),
    'max_offdiag': ('mzd/sparse_utils.py', 269, 281),
    'compress': ('mzd/sparse_utils.py', 284, 314),
}


def available():
    return os.path.isfile(os.path.join(REFERENCE_ROOT, 'mzd', 'sparse_utils.py'))


class _NpShim(object):
    """numpy with the aliases removed in NumPy >= 1.24 put back."""
    int = int
    float = float
    bool = bool

    def __getattr__(self, name):
        return getattr(np, name)


def _install_H():
    # sparse_utils.py:18 uses m.H; SciPy dropped the attribute
    for cls in (scisp.csr_matrix, scisp.csc_matrix, scisp.coo_matrix, scisp.lil_matrix):
        if not hasattr(cls, 'H'):
            cls.H = property(lambda self: self.conj().transpose())


class IterCapture(logging.Handler):
    """Collects the 'It took N iterations' debug line of sparse_utils.py:218."""

    def __init__(self):
        logging.Handler.__init__(self, level=logging.DEBUG)
        self.n_iter = None
        self.warnings = []

    def emit(self, record):
        msg = record.getMessage()
        if msg.startswith('It took '):
            self.n_iter = int(msg.split()[2])
        elif record.levelno >= logging.WARNING:
            self.warnings.append(msg)


def load(skip_hermitian_check=False):
    """
    Exec the sliced reference functions and return them in a dict, plus the logger they
    write to (name 'mzd.sparse_utils', as in the reference).
    """
    if not available():
        raise RuntimeError('reference tree not found at {}'.format(REFERENCE_ROOT))
    _install_H()
    logger = logging.getLogger('mzd.sparse_utils')
    logger.setLevel(logging.DEBUG)
    ns = {'np': _NpShim(), 'scisp': scisp, 'logger': logger, 'xrange': range}
    for name, (rel, lo, hi) in SLICES.items():
        with open(os.path.join(REFERENCE_ROOT, rel), 'r') as fh:
            lines = fh.readlines()[lo - 1:hi]
        exec(compile(textwrap.dedent(''.join(lines)), '{}:{}-{}'.format(rel, lo, hi), 'exec'), ns)
    if skip_hermitian_check:
        # Q11: the dense NxN check cannot run beyond N ~ 50k; it only logs a warning
        ns['is_hermitian'] = lambda m, tol=1e-6: True
    out = {k: ns[k] for k in SLICES}
    out['logger'] = logger
    return out


def kr_with_iterations(fns, m, **kw):
    """Run the reference kr_biostochastic and also return its iteration count."""
    cap = IterCapture()
    fns['logger'].addHandler(cap)
    try:
        bal, x = fns['kr_biostochastic'](m, **kw)
    finally:
        fns['logger'].removeHandler(cap)
    return bal, x, cap.n_iter, cap.warnings


# ---- the tip-based tensor functions (sparse_utils.py:317-509) over a stand-in for pydata `sparse` -------------------
class SparseShim(object):
    """
    Stand-in for the `sparse` module (sparse==0.3.1, Pipfile.lock:381; not installed here): the part of sparse.COO the
    reference's 4-D functions touch.  COO(coords, data, shape, has_duplicates): coordinates sorted row-major,
    duplicates summed when flagged (COO.__init__ of 0.3.1 sorts unless sorted=True and sums when has_duplicates);
    .coords .data .shape .nnz .astype() .sum(axis=(2, 3)) -> 2-D COO with .tocsr() / .to_scipy_sparse().
    TEST INFRASTRUCTURE: lets the reference's own code run here; it is not the reference's dependency itself.
    """

    class COO(object):
        def __init__(self, coords, data=None, shape=None, has_duplicates=True, sorted=False):
            coords = np.asarray(coords, dtype=np.int64)
            data = np.asarray(data)
            if coords.ndim == 1:
                coords = coords.reshape(len(shape), -1)
            self.shape = tuple(int(v) for v in shape)
            if not sorted and coords.shape[1]:
                lin = np.ravel_multi_index(tuple(coords), self.shape)
                o = np.argsort(lin, kind='stable')
                coords, data, lin = coords[:, o], data[o], lin[o]
                if has_duplicates and len(lin) > 1:
                    first = np.concatenate([[True], lin[1:] != lin[:-1]])
                    if not first.all():
                        data = np.add.reduceat(data, np.flatnonzero(first)).astype(data.dtype)
                        coords = coords[:, first]
            self.coords, self.data = coords, data

        @property
        def nnz(self):
            return self.coords.shape[1]

        @property
        def ndim(self):
            return len(self.shape)

        def astype(self, dtype):
            return SparseShim.COO(self.coords.copy(), self.data.astype(dtype), self.shape, has_duplicates=False,
                                  sorted=True)

        def sum(self, axis=None):
            if axis is None:
                return self.data.sum()
            keep = [a for a in range(self.ndim) if a not in tuple(axis)]
            data = self.data
            if np.issubdtype(data.dtype, np.unsignedinteger):
                data = data.astype(np.uint64)              # numpy's sum of uint32 accumulates in uint64
            return SparseShim.COO(self.coords[keep], data, tuple(self.shape[a] for a in keep), has_duplicates=True)

        def to_scipy_sparse(self):
            assert self.ndim == 2
            return scisp.coo_matrix((self.data, (self.coords[0], self.coords[1])), shape=self.shape)

        def tocsr(self):
            return self.to_scipy_sparse().tocsr()

        def to_coo(self):
            return self

    class DOK(object):
        pass


SLICES_4D = {
    'Sparse4DAccumulator': ('mzd/sparse_utils.py', 317, 409),
    'max_offdiag_4d': ('mzd/sparse_utils.py', 412, 421),
    'flatten_tensor_4d': ('mzd/sparse_utils.py', 424, 443),
    'compress_4d': ('mzd/sparse_utils.py', 446, 477),
    'dotdot': ('mzd/sparse_utils.py', 480, 492),
    'kr_biostochastic_4d': ('mzd/sparse_utils.py', 495, 509),
}


def load_4d():
    """Exec the reference's tip-based tensor functions (sparse_utils.py:317-509) with SparseShim as `sparse`; returns
    them in a dict together with the 2-D functions they call."""
    fns = load()
    ns = {'np': _NpShim(), 'scisp': scisp, 'sparse': SparseShim, 'logger': fns['logger'], 'xrange': range,
          'max_offdiag': fns['max_offdiag'], 'kr_biostochastic': fns['kr_biostochastic']}
    for name, (rel, lo, hi) in SLICES_4D.items():
        with open(os.path.join(REFERENCE_ROOT, rel), 'r') as fh:
            lines = fh.readlines()[lo - 1:hi]
        exec(compile(textwrap.dedent(''.join(lines)), '{}:{}-{}'.format(rel, lo, hi), 'exec'), ns)
    out = dict(fns)
    out.update({k: ns[k] for k in SLICES_4D})
    return out


# ---- the extent map's bins (contact_map.py:116-156) and find_nearest_jit (:49-62) -----------------------------
class Py2Int(int):
    """An int whose `/` is Python 2's: integer division when the other operand is an int (contact_map.py:132), true
    division when it is a float (:137).  Lets ExtentGrouping run verbatim under Python 3."""

    def __truediv__(self, other):
        if isinstance(other, int):
            return Py2Int(int(self) // int(other))
        return int(self) / other

    def __mod__(self, other):
        return int(self) % other


def load_extent():
    """
    Exec the reference's ExtentGrouping class and find_nearest_jit body.  Shims: np.int, tqdm.tqdm = identity,
    the numba decorator dropped (the @jit line is not part of the slice), and sequence lengths wrapped in Py2Int.
    Returns (make_grouping(lengths, bin_size) -> reference ExtentGrouping instance, find_nearest(group_sites, x)).
    """
    if not available():
        raise RuntimeError('reference tree not found at {}'.format(REFERENCE_ROOT))
    import collections

    class _Tqdm(object):
        @staticmethod
        def tqdm(it, **kw):
            return it

    ns = {'np': _NpShim(), 'tqdm': _Tqdm, 'ZeroLengthException': ValueError}
    path = os.path.join(REFERENCE_ROOT, 'mzd', 'contact_map.py')
    with open(path, 'r') as fh:
        lines = fh.readlines()
    for lo, hi in ((50, 62), (116, 156)):              # def find_nearest_jit (without @jit at :49), class ExtentGrouping
        exec(compile(textwrap.dedent(''.join(lines[lo - 1:hi])), 'mzd/contact_map.py:{}-{}'.format(lo, hi), 'exec'), ns)
    Seq = collections.namedtuple('Seq', ['length', 'id'])

    def make_grouping(lengths, bin_size):
        return ns['ExtentGrouping']([Seq(Py2Int(int(l)), n) for n, l in enumerate(lengths)], bin_size)

    return make_grouping, ns['find_nearest_jit']


# ---- the reference's own _bin_map (contact_map.py:602-809) over duck-typed alignment records ----------------
class FakeAlignment(object):
    """The pysam.AlignedSegment attributes _bin_map touches, from an alignment dict (name, flag, tid, pos, mapq, cigar)."""
    _OPS = 'MIDNSHP=X'

    def __init__(self, a):
        f = a['flag']
        self.query_name = a['name']
        self.reference_id = a['tid']
        self.mapping_quality = a['mapq']
        self.pos = self.reference_start = a['pos']
        cig = a.get('cigar') or None
        self.cigartuples = list(cig) if cig else None
        self.cigarstring = ''.join('{}{}'.format(n, self._OPS[op]) for op, n in cig) if cig else None
        self.alen = sum(n for op, n in cig if op in (0, 2, 3, 7, 8)) if cig else None      # pysam reference_length
        self.reference_end = self.pos + self.alen if cig else None
        self.is_unmapped = bool(f & 0x4)
        self.is_secondary = bool(f & 0x100)
        self.is_supplementary = bool(f & 0x800)
        self.is_reverse = bool(f & 0x10)
        self.is_read2 = bool(f & 0x80)
        self.is_proper_pair = bool(f & 0x2)


class _FakeBam(object):
    def __init__(self, alignments, lengths):
        self._alns = alignments
        self.lengths = list(lengths)

    def reset(self):
        pass

    def fetch(self, until_eof=True):
        bam = self

        class It(object):                      # the reference calls _bam_iter.next() (Python 2 protocol)
            def __init__(self):
                self._it = iter(bam._alns)

            def next(self):
                return FakeAlignment(next(self._it))
        return It()


def run_bin_map(alignments, ref_lengths, idx_of, n_seq, min_mapq=0, strong=None, min_insert=None, grouping=None,
                tip_size=None):
    """
    Exec the reference's ContactMap._bin_map verbatim (contact_map.py:602-809) on a stub instance and a fake BAM of
    duck-typed records; Sparse2DAccumulator and find_nearest_jit are the reference's own too.  `grouping` is an
    exec'd reference ExtentGrouping (load_extent) or None.  A mapped record without CIGAR has alen None, which the
    reference cannot add to a position: feed such records only as forward reads.
    With `tip_size` the map is the tip-based tensor: the reference's own Sparse4DAccumulator (over SparseShim) and
    _on_tip_withlocs; seq_map is then a SparseShim.COO of shape (N, N, 2, 2).
    Returns dict(seq_map coo, extent_map coo or None, counts dict).
    """
    import collections
    fns = load_4d() if tip_size else load()
    _, find_nearest = load_extent()
    logger = logging.getLogger('mzd.contact_map.exec')
    captured = {}

    class Cap(logging.Handler):
        def emit(self, record):
            msg = record.getMessage()
            if msg.startswith('Pair accounting: '):
                captured['counts'] = msg[len('Pair accounting: '):]
    cap = Cap(level=logging.INFO)
    logger.addHandler(cap)
    logger.setLevel(logging.INFO)

    class SU(object):
        Sparse2DAccumulator = fns['Sparse2DAccumulator']
        Sparse4DAccumulator = fns.get('Sparse4DAccumulator')

    ns = {'np': _NpShim(), 'sparse_utils': SU, 'logger': logger, 'OrderedDict': collections.OrderedDict,
          'find_nearest_jit': find_nearest, 'xrange': range}
    with open(os.path.join(REFERENCE_ROOT, 'mzd', 'contact_map.py'), 'r') as fh:
        lines = fh.readlines()[602 - 1:809]
    exec(compile(textwrap.dedent(''.join(lines)), 'mzd/contact_map.py:602-809', 'exec'), ns)

    class Stub(object):
        pass
    me = Stub()
    me.strong, me.min_insert, me.min_mapq = strong, min_insert, min_mapq
    me.total_seq, me.total_len, me.total_reads = n_seq, 0, None
    me.bin_size = grouping.bin_size if grouping is not None else None
    me.grouping, me.tip_size = grouping, tip_size
    me.extent_map = me.seq_map = None
    me.is_tipbased = lambda: tip_size is not None
    me.make_reverse_index = lambda field: dict(idx_of)
    me.map_weight = lambda: int(me.seq_map.data.sum()) if tip_size else int(me.seq_map.sum())
    try:
        ns['_bin_map'](me, _FakeBam(alignments, ref_lengths))
    finally:
        logger.removeHandler(cap)
    counts = eval(captured['counts'], {'OrderedDict': collections.OrderedDict})
    return dict(seq_map=me.seq_map, extent_map=me.extent_map, counts=dict(counts))


# ---- the reference's own to_graph (cluster.py:278-325) on a stub contact map -------------------------------------
def run_to_graph(sub_map, n_accepted, scale=True, contact_map=None):
    """
    Exec cluster.to_graph verbatim; `sub_map` is what contact_map.get_subspace(marginalise=True, flatten=False) returns
    (the compressed, balanced map).  Shims: itertools.izip = zip, nx.info (removed in networkx 3) = '', tqdm = identity.
    Returns the nx.Graph the reference builds.
    """
    import networkx
    import scipy.sparse as sp

    class NX(object):
        Graph = networkx.Graph

        @staticmethod
        def info(g):
            return ''

    class IT(object):
        izip = zip

    class TQ(object):
        @staticmethod
        def tqdm(it, **kw):
            return it

    class Order(object):
        @staticmethod
        def count_accepted():
            return n_accepted

    class CM(object):
        processed_map = object()
        order = Order()
        seq_info = None

        @staticmethod
        def set_primary_acceptance_mask(*a, **kw):
            pass

        @staticmethod
        def get_subspace(marginalise=False, flatten=True):
            return sub_map

    ns = {'nx': NX, 'itertools': IT, 'tqdm': TQ, 'sp': sp, 'logger': logging.getLogger('mzd.cluster.exec')}
    with open(os.path.join(REFERENCE_ROOT, 'mzd', 'cluster.py'), 'r') as fh:
        lines = fh.readlines()[278 - 1:325]
    exec(compile(textwrap.dedent(''.join(lines)), 'mzd/cluster.py:278-325', 'exec'), ns)
    return ns['to_graph'](contact_map if contact_map is not None else CM, norm=True, bisto=True, scale=scale)


# ---- the whole reference path: SeqOrder + ContactMap classes exec'd, driven as bin3C.py mkmap / cluster do ------------
def run_reference_path(alignments, ref_lengths, ref_sites, min_len, min_sig, min_mapq=60, strong=None, min_insert=None,
                       bin_size=None, seed=1, tip_size=None):
    """
    Exec the reference's SeqOrder and ContactMap classes (contact_map.py:159-485, 486-end), find_nearest_jit,
    fast_norm_fullseq_bysite (without their numba decorators) and ExtentGrouping, build a ContactMap without its
    __init__ (which needs pysam and Biopython: the attribute set-up of :492-600 is replayed here from the reference
    table), then call the reference's own methods in the order bin3C.py mkmap / cluster call them:
        _bin_map(fake bam) -> set_primary_acceptance_mask() -> to_graph(...) [prepare_seq_map(norm, bisto),
        get_subspace(marginalise=True, flatten=False)]
    With `tip_size` the map is the tip-based tensor (`ref_sites` then holds (head, tail) pairs, seq_utils.py:146-158):
    the 4-D functions of sparse_utils.py:317-509 over SparseShim and fast_norm_tipbased_bysite (contact_map.py:84-97,
    without its numba decorator, whose signature -- float64 arrays of 4, 2 and 2 dimensions, :83 -- is not what
    _norm_seq passes).
    Returns dict(cm, seq_map, mask, bisto_scale, processed_map, sub_map, graph, counts).
    """
    import collections
    fns = load_4d() if tip_size else load(skip_hermitian_check=False)
    _, find_nearest = load_extent()
    logger = logging.getLogger('mzd.contact_map.exec')
    captured = {}

    class Cap(logging.Handler):
        def emit(self, record):
            msg = record.getMessage()
            if msg.startswith('Pair accounting: '):
                captured['counts'] = msg[len('Pair accounting: '):]
    cap = Cap(level=logging.INFO)
    logger.addHandler(cap)
    logger.setLevel(logging.INFO)

    class SU(object):
        Sparse2DAccumulator = fns['Sparse2DAccumulator']
        max_offdiag = staticmethod(fns['max_offdiag'])
        compress = staticmethod(fns['compress'])
        kr_biostochastic = staticmethod(fns['kr_biostochastic'])
        if tip_size:
            Sparse4DAccumulator = fns['Sparse4DAccumulator']
            max_offdiag_4d = staticmethod(fns['max_offdiag_4d'])
            flatten_tensor_4d = staticmethod(fns['flatten_tensor_4d'])
            compress_4d = staticmethod(fns['compress_4d'])
            kr_biostochastic_4d = staticmethod(fns['kr_biostochastic_4d'])

    class NoneAcceptedException(Exception):
        pass

    class TQ(object):
        @staticmethod
        def tqdm(it=None, **kw):
            class Bar(object):
                def __enter__(self_):
                    return self_

                def __exit__(self_, *a):
                    return False

                def update(self_, n=1):
                    pass
            return it if it is not None else Bar()

    SeqInfo = collections.namedtuple('SeqInfo', ['offset', 'refid', 'name', 'length', 'sites'])
    ns = {'np': _NpShim(), 'sp': scisp, 'sparse_utils': SU, 'logger': logger, 'OrderedDict': collections.OrderedDict,
          'namedtuple': collections.namedtuple, 'xrange': range, 'tqdm': TQ, 'SeqInfo': SeqInfo,
          'NoneAcceptedException': NoneAcceptedException, 'find_nearest_jit': find_nearest}
    with open(os.path.join(REFERENCE_ROOT, 'mzd', 'contact_map.py'), 'r') as fh:
        lines = fh.readlines()
    for lo, hi in ((25, 46), (84, 97), (101, 113), (116, 156), (159, 485), (486, len(lines))):      # mean_selector: :25-46
        exec(compile(textwrap.dedent(''.join(lines[lo - 1:hi])), 'mzd/contact_map.py:{}-{}'.format(lo, hi), 'exec'), ns)
    # tqdm is imported inside _bin_map ("import tqdm"): give it the stub through sys.modules for the call
    import sys
    import types
    stub = types.ModuleType('tqdm')
    stub.tqdm = TQ.tqdm
    saved = sys.modules.get('tqdm')
    sys.modules['tqdm'] = stub

    CM = ns['ContactMap']
    # _norm_extent (contact_map.py:1147-1165) leaves NumPy arrays in the rows of its LIL matrix (`list /= ndarray`);
    # SciPy 1.1 converted such a matrix, SciPy 1.18's LIL -> CSR wants lists again: same values, list rows
    _norm_extent_ref = CM._norm_extent

    def _norm_extent_lists(self, _map, mean_type='geometric'):
        out = _norm_extent_ref(self, _map, mean_type)
        for i in range(out.shape[0]):
            out.data[i] = [float(v) for v in np.asarray(out.data[i], dtype=np.float64).ravel()]
        return out
    CM._norm_extent = _norm_extent_lists
    cm = CM.__new__(CM)
    cm.strong, cm.bam_file, cm.bin_size, cm.min_mapq, cm.min_insert = strong, None, bin_size, min_mapq, min_insert
    cm.min_len, cm.min_sig, cm.min_extent, cm.min_size, cm.max_fold = min_len, min_sig, 0, 0, None
    cm.random_state = np.random.RandomState(seed)
    cm.seq_info, cm.seq_map, cm.seq_file, cm.grouping, cm.extent_map, cm.order = [], None, None, None, None, None
    cm.tip_size, cm.precount, cm.total_reads, cm.cov_info, cm.processed_map = tip_size, False, None, None, None
    cm.primary_acceptance_mask, cm.bisto_scale, cm.seq_analyzer, cm.enzymes = None, None, None, ['synthetic']
    offset = 0
    for n, (rlen, sites) in enumerate(zip(ref_lengths, ref_sites)):                 # contact_map.py:545-564
        if rlen < min_len or np.min(sites) < 0:
            continue
        cm.seq_info.append(SeqInfo(offset, n, 'ref{:07d}'.format(n), Py2Int(int(rlen)),
                                   [int(v) for v in sites] if tip_size else int(sites)))
        offset += int(rlen)
    cm.total_len, cm.total_seq = offset, len(cm.seq_info)
    cm.current_mask = np.ones(cm.total_seq, dtype=bool)
    if bin_size:
        cm.grouping = ns['ExtentGrouping'](cm.seq_info, bin_size)
    cm.order = ns['SeqOrder'](cm.seq_info)
    try:
        cm._bin_map(_FakeBam(alignments, ref_lengths))
        cm.set_primary_acceptance_mask()
        graph = run_to_graph(None, None, scale=True, contact_map=cm)
    finally:
        logger.removeHandler(cap)
        if saved is not None:
            sys.modules['tqdm'] = saved
        else:
            del sys.modules['tqdm']
    counts = dict(eval(captured['counts'], {'OrderedDict': collections.OrderedDict}))
    return dict(cm=cm, seq_map=cm.seq_map, extent_map=cm.extent_map, mask=cm.get_primary_acceptance_mask(),
                bisto_scale=cm.bisto_scale, processed_map=cm.processed_map, graph=graph, counts=counts)
