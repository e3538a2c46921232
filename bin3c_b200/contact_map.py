"""
Host-side mirror of the hot-path surface of the reference's mzd/contact_map.py
(cerebis/bin3C @ 76ad2a9): the ContactMap methods that build, filter, normalise and balance
the contig x contig contact matrix, with the same names, arguments and error behaviour.

    ContactMap.__init__ (reference table part)   contact_map.py:545-600
    ContactMap._bin_map                          contact_map.py:602-809
    ContactMap.make_reverse_index                contact_map.py:818-832
    ContactMap.map_weight / is_empty             contact_map.py:834-844
    ContactMap.set_primary_acceptance_mask       contact_map.py:856-909
    ContactMap.prepare_seq_map                   contact_map.py:911-945
    ContactMap.get_subspace                      contact_map.py:947-999
    ContactMap._bisto_seq / _get_sites / _norm_seq   contact_map.py:1087-1145
    SeqOrder (the five bookkeeping methods the path uses)   contact_map.py:159-447
    ExtentGrouping + the extent (binned) map accumulation   contact_map.py:116-156, 779-788, 801-803

The difference from the reference is the input: BAM decoding (pysam) is outside the path
(SURVEY.md section 8f), so `bam_file` is a PairRecords object -- the BAM header's reference
table plus the packed pair-record stream -- instead of a file name.  Device buffers live in
`self._dev` and never reach a pickle: seq_map / processed_map materialise on the host as the
same SciPy containers the reference stores (Q10) the first time they are read.
"""
import logging
from collections import OrderedDict

import numpy as np
import scipy.sparse as scisp

from . import device as dev
from .exceptions import NoneAcceptedException, ParsingError
from .synth import SeqInfo

logger = logging.getLogger('mzd.contact_map')


class PairRecords(object):
    """
    What the path needs from a name-sorted BAM: the header's reference table and, per usable
    read pair, one packed record (see include/bin3c_b200.h).

    :param references: reference names (or None -> 'ref{n}')
    :param lengths: reference lengths, int array [n_refs]   (bam.lengths)
    :param sites: restriction-site count per reference; stands in for the FASTA pass of
                  contact_map.py:520-531.  A negative value marks "not present in the FASTA".
    :param records: uint64 packed pair records, NumPy array (host) or CUDA tensor (device)
    :param extent_records: optional, same length: the pair's records at BIN level (global bin numbers of the two
                  5'-end positions in place of reference ids; bam_io.pair_records_from_bam(bin_size=...)),
                  needed by ContactMap(bin_size=...)
    """

    def __init__(self, lengths, sites, records, references=None, extent_records=None, meta=None, tip10=None):
        self.extent_records = extent_records      # bin-level records for the extent map (bam_io, bin_size=...)
        # tip-based map (bam_io, tip_size=...): the records carry doubled ids 2 * tid + tip; tip10 = BAM reference ids
        # of the accepted same-sequence pairs whose tips are (tail, head) in read order; sites is then [n_refs, 2]
        self.tip10 = tip10
        # how the records were made (bam_io.pair_records_from_bam): min_mapq, strong, min_insert, min_len, bin_size and
        # the reader's short_insert count.  ContactMap checks its own arguments against these, so that e.g. an extent
        # map is never built over bins other than the ones the reader used.
        self.meta = dict(meta) if meta else None
        self.lengths = np.asarray(lengths, dtype=np.int64)
        self.sites = np.asarray(sites, dtype=np.int64)
        assert self.lengths.shape == self.sites.shape[:1] and (self.sites.ndim == 1 or self.sites.shape[1] == 2)
        self.references = references
        self.records = records

    @property
    def n_refs(self):
        return len(self.lengths)

    def name(self, n):
        return self.references[n] if self.references is not None else 'ref{:07d}'.format(n)

    @classmethod
    def from_community(cls, com, short_len=500):
        """PairRecords of a synthetic Community: excluded references are short (length < min_len)."""
        lengths = np.full(com.n_refs, short_len, dtype=np.int64)
        sites = np.ones(com.n_refs, dtype=np.int64)
        lengths[com.ref_index] = com.lengths
        sites[com.ref_index] = com.sites
        return cls(lengths, sites, com.records)


class ExtentGrouping(object):
    """
    The bins of the extent map (contact_map.py:116-156).  A sequence gets length // bin_size bins (the reference is
    Python 2: `/` on ints), at least one, and one more when the remainder is half a bin or more; the bin edges are
    np.linspace(0, length, num_bins + 1) truncated to integers.  `map[i]` is the reference's per-sequence array of
    (upper edge, global bin) pairs; `first_bin`, `edge_ptr` and `upper_edges` are the same thing as flat arrays for
    the BAM reader (include/bin3c_io.h: b3c_bam_set_extent).
    """

    def __init__(self, seq_info, bin_size):
        self._build([s.length for s in seq_info], bin_size)

    @classmethod
    def from_lengths(cls, lengths, bin_size):
        g = cls.__new__(cls)
        g._build(np.asarray(lengths).tolist(), bin_size)
        return g

    def _build(self, lengths, bin_size):
        from .exceptions import ZeroLengthException
        self.bin_size = bin_size
        self.bins, self.map, self.borders, self.centers = [], [], [], []
        self.total_bins = 0
        first, upper = [], []
        for n, length in enumerate(lengths):
            length = int(length)
            if length == 0:
                raise ZeroLengthException(n)
            num_bins = length // bin_size
            if num_bins == 0:
                num_bins += 1
            # non-integer discrepancy: contract / expand all bins equally, the threshold being half a bin
            if length % bin_size != 0 and length / float(bin_size) - num_bins >= 0.5:
                num_bins += 1
            edges = np.linspace(0, length, num_bins + 1, endpoint=True).astype(np.int64)
            self.bins.append(num_bins)
            first_bin, last_bin = self.total_bins, self.total_bins + num_bins
            self.map.append(np.vstack((edges[1:], np.arange(first_bin, last_bin))).T)
            self.borders.append(np.array([first_bin, last_bin], dtype=np.int64))
            self.total_bins += num_bins
            c_nk = edges[:-1] + 0.5 * (edges[1] - edges[0]) - 0.5 * length
            self.centers.append(c_nk.reshape((1, len(c_nk))))
            first.append(first_bin)
            upper.append(edges[1:])
        self.bins = np.array(self.bins)
        self.first_bin = np.array(first, dtype=np.int64)
        self.edge_ptr = np.concatenate([[0], np.cumsum(self.bins)]).astype(np.int64)
        self.upper_edges = np.concatenate(upper).astype(np.int64) if upper else np.empty(0, dtype=np.int64)


class SeqOrder(object):
    """Ordering / masking state of the sequences (contact_map.py:159-483); only what the path uses."""

    FORWARD = 1
    REVERSE = -1
    ACCEPTED = True
    EXCLUDED = False

    STRUCT_TYPE = np.dtype([('pos', np.int32), ('ori', np.int8), ('mask', np.bool_), ('length', np.int32)])

    def __init__(self, seq_info):
        n = len(seq_info)
        self._positions = None
        self.order = np.empty(n, dtype=SeqOrder.STRUCT_TYPE)
        self.order['pos'] = np.arange(n, dtype=np.int32)
        self.order['ori'] = SeqOrder.FORWARD
        self.order['mask'] = SeqOrder.ACCEPTED
        self.order['length'] = np.fromiter((s.length for s in seq_info), dtype=np.int32, count=n)
        self._update_positions()

    def _update_positions(self):
        # masked sequences last, then by current position (contact_map.py:203-213), without the Python loop
        sorted_indices = np.lexsort([self.order['pos'], ~self.order['mask']])
        self.order['pos'][sorted_indices] = np.arange(len(sorted_indices), dtype=np.int32)
        self._positions = np.argsort(self.order['pos'])

    def set_mask_only(self, _mask):
        _mask = np.asarray(_mask, dtype=np.bool_)
        assert len(_mask) == len(self.order), 'supplied mask must be the same length as existing order'
        self.order['mask'] = _mask
        self._update_positions()

    def mask_vector(self):
        return self.order['mask']

    def count_accepted(self):
        return self.order['mask'].sum()

    def count_excluded(self):
        return len(self.order) - self.count_accepted()

    def accepted(self):
        return np.where(self.order['mask'])[0]

    def excluded(self):
        return np.where(~self.order['mask'])[0]

    def lengths(self, exclude_masked=False):
        if exclude_masked:
            return self.order['length'][self.order['mask']]
        return self.order['length']


class ContactMap(object):

    def __init__(self, bam_file, enzymes, seq_file, min_insert, min_mapq=0, min_len=0, min_sig=1, min_extent=0,
                 min_size=0, max_fold=None, random_seed=None, strong=None, bin_size=None, tip_size=None,
                 precount=False, gpu_decode=False, gpu_sites=False):

        assert not (tip_size and bin_size), 'tip records and extent records do not combine in this build'
        if not isinstance(bam_file, PairRecords):
            # the call bin3C.py mkmap makes (bin3C.py:148-158): a BAM path and a FASTA path.  The BAM is decoded by
            # the native reader (libbin3c_io.so) with this map's matcher, insert filter and bins; the site counts come
            # from the FASTA (seq_sites.fasta_site_table), or from `seq_file` given as an array / dict / callable.
            # gpu_decode=True decodes the BAM on the GPU instead (bam_io.pair_records_from_bam(device=True)): the
            # same records, left on the device for the accumulation.  gpu_sites=True counts the FASTA's sites on the
            # GPU (seq_sites.fasta_site_table(device=True)): the same counts.
            bam_file = self._open_bam(bam_file, enzymes, seq_file, min_insert, min_mapq, min_len, strong, bin_size,
                                      tip_size, gpu_decode=gpu_decode, gpu_sites=gpu_sites)
        meta = bam_file.meta
        if tip_size:
            assert meta is not None and meta.get('tip_size') == tip_size and meta.get('min_len') == min_len, \
                'tip_size needs tip records: bam_io.pair_records_from_bam(path, tip_size=..., min_len=...) with the ' \
                "map's own tip_size and min_len"
            assert bam_file.sites.ndim == 2, 'a tip-based map takes (head, tail) site counts per reference'
        else:
            assert meta is None or not meta.get('tip_size'), 'these are tip records: the map needs tip_size'
        assert not bin_size or bam_file.extent_records is not None, \
            'bin_size needs extent records: bam_io.pair_records_from_bam(path, bin_size=..., min_len=...)'
        if meta is None:
            assert not min_insert, 'min_insert needs alignment positions: read the BAM with ' \
                                   'bam_io.pair_records_from_bam(path, min_insert=...) or pass its path'
        else:
            # the records were cut with these settings: the map must be described by the same ones
            assert (meta.get('min_insert') or None) == (min_insert or None), \
                'records were read with min_insert={}, the map asks for {}'.format(meta.get('min_insert'), min_insert)
            if bin_size:
                assert meta.get('bin_size') == bin_size and meta.get('min_len') == min_len, \
                    'extent records were binned with bin_size={}, min_len={}; the map asks for {}, {}'.format(
                        meta.get('bin_size'), meta.get('min_len'), bin_size, min_len)
            if min_insert:
                assert meta.get('min_len') == min_len, \
                    'the insert filter was applied with min_len={}; the map asks for {}'.format(meta.get('min_len'), min_len)

        self.strong = strong
        self.bam_file = None            # records are not retained on the (pickled) instance
        self.bin_size = bin_size
        self.min_mapq = min_mapq
        self.min_insert = min_insert
        self.min_len = min_len
        self.min_sig = min_sig
        self.min_extent = min_extent
        self.min_size = min_size
        self.max_fold = max_fold
        self.random_state = np.random.RandomState(random_seed)
        self.seq_info = []
        self.seq_file = seq_file
        self.grouping = None
        self.extent_map = None
        self.order = None
        self.tip_size = tip_size
        self.precount = precount
        self.total_reads = None
        self.cov_info = None
        self.primary_acceptance_mask = None
        self.bisto_scale = None
        self.seq_analyzer = None
        self.enzymes = enzymes
        self.pair_counts = None
        self.kr_info = None
        self._host = {}                 # lazily materialised SciPy containers
        self._dev = {}                  # device-resident state, never pickled

        # the set of active sequences, first filtration step is by length (contact_map.py:545-564)
        ref_count = {'seq_missing': 0, 'too_short': 0}
        logger.info('Reading sequences...')
        too_short = bam_file.lengths < min_len
        missing = ~too_short & ((bam_file.sites < 0) if bam_file.sites.ndim == 1 else (bam_file.sites < 0).any(axis=1))
        ref_count['too_short'] = int(too_short.sum())
        ref_count['seq_missing'] = int(missing.sum())
        keep = np.flatnonzero(~too_short & ~missing)
        offset = 0
        for n in keep:
            rlen = int(bam_file.lengths[n])
            # tip-based: [head sites, tail sites] (seq_utils.py:146-158)
            st = [int(v) for v in bam_file.sites[n]] if bam_file.sites.ndim == 2 else int(bam_file.sites[n])
            self.seq_info.append(SeqInfo(offset, int(n), bam_file.name(n), rlen, st))
            offset += rlen

        self.total_len = offset
        self.total_seq = len(self.seq_info)
        self.n_refs = bam_file.n_refs
        self.current_mask = np.ones(self.total_seq, dtype=np.bool_)

        if self.total_seq == 0:
            logger.info('No sequences in BAM found in FASTA')
            raise ParsingError('No sequences in BAM found in FASTA')

        logger.info('Accepted {} sequences covering {} bp'.format(self.total_seq, self.total_len))
        logger.info('References excluded: {}'.format(ref_count))

        self.order = SeqOrder(self.seq_info)

        if self.bin_size:
            self.grouping = ExtentGrouping(self.seq_info, self.bin_size)      # contact_map.py:581-583

        # accumulate
        self._bin_map(bam_file)

        # create an initial acceptance mask
        self.set_primary_acceptance_mask()

    @staticmethod
    def _open_bam(path, enzymes, seq_file, min_insert, min_mapq, min_len, strong, bin_size, tip_size=None,
                  gpu_decode=False, gpu_sites=False):
        """BAM path -> PairRecords with this map's filters (contact_map.py:520-564: FASTA pass, header, reference table).
        `seq_file`: a FASTA path; or per-reference site counts as an array (one per BAM reference), a dict
        {reference name: sites} (absent = not in the FASTA), or a callable (name, length) -> sites."""
        import os
        from . import bam_io
        with bam_io.BamPairReader(path) as hdr:
            names, lengths = list(hdr.references), np.asarray(hdr.lengths, dtype=np.int64)
        if callable(seq_file):
            sites = np.array([seq_file(nm, int(ln)) for nm, ln in zip(names, lengths)], dtype=np.int64)
        elif isinstance(seq_file, dict):
            sites = np.array([seq_file.get(nm, [-1, -1] if tip_size else -1) for nm in names], dtype=np.int64)
        elif isinstance(seq_file, (str, bytes, os.PathLike)):
            from .seq_sites import fasta_site_table
            logger.info('Analyzing sites...')
            info = fasta_site_table(seq_file, enzymes, min_len or 0, tip_size=tip_size, device=gpu_sites)
            sites = np.full((len(names), 2) if tip_size else len(names), -1, dtype=np.int64)
            for n, (nm, ln) in enumerate(zip(names, lengths)):
                fa = info.get(nm)
                if fa is None:
                    if ln >= (min_len or 0):
                        logger.info('Sequence: "{}" was not present in reference fasta'.format(nm))
                    continue
                assert fa['length'] == ln, \
                    'Sequence lengths in {} do not agree: bam {} fasta {}'.format(nm, fa['length'], ln)
                sites[n] = fa['sites']
        else:
            sites = np.asarray(seq_file, dtype=np.int64)
            assert sites.shape[:1] == lengths.shape, 'one site count per BAM reference'
        if tip_size and sites.ndim == 1:
            sites = np.array([[v, v] if np.ndim(v) == 0 else list(v) for v in sites.tolist()], dtype=np.int64)
        rec, _ = bam_io.pair_records_from_bam(path, sites=sites, min_mapq=min_mapq, strong=strong, min_insert=min_insert,
                                              min_len=min_len, bin_size=bin_size, tip_size=tip_size, device=gpu_decode)
        return rec

    # ---- pickling: host containers only ------------------------------------------------------
    def __getstate__(self):
        state = dict(self.__dict__)
        state['_host'] = {'seq_map': self.seq_map, 'processed_map': self.processed_map}
        state['_dev'] = {}
        return state

    def __setstate__(self, state):
        """Accepts this package's own state and a STOCK bin3C ContactMap's attribute dict (contact_map.py:492-518:
        `seq_map` / `processed_map` as plain attributes; io_utils.load_object maps the classes)."""
        from .io_utils import unstock
        state = dict(state)
        host = dict(state.pop('_host', None) or {})
        for k in ('seq_map', 'processed_map'):
            if k in state:
                host[k] = state.pop(k)
        state['_host'] = {k: unstock(v) for k, v in host.items()}
        state['_dev'] = {}
        if 'extent_map' in state:
            state['extent_map'] = unstock(state['extent_map'])
        self.__dict__.update(state)
        self.__dict__.setdefault('pair_counts', None)
        self.__dict__.setdefault('kr_info', None)
        if 'n_refs' not in self.__dict__ and self.__dict__.get('seq_info'):
            self.n_refs = max(si.refid for si in self.seq_info) + 1      # a stock map does not keep the table size

    @property
    def seq_map(self):
        """coo_matrix[uint32], symmetric, canonical row-major -- what get_coo() returns (Q10)."""
        if self._host.get('seq_map') is None and 'seq_map' in self._dev:
            self._host['seq_map'] = self._dev['seq_map'].to_scipy_coo()
        return self._host.get('seq_map')

    @seq_map.setter
    def seq_map(self, m):
        self._host['seq_map'] = m
        self._dev.pop('seq_map', None)

    @property
    def processed_map(self):
        if self._host.get('processed_map') is None and 'processed_map' in self._dev:
            self._host['processed_map'] = self._dev['processed_map'].to_scipy_csr()
        return self._host.get('processed_map')

    @processed_map.setter
    def processed_map(self, m):
        self._host['processed_map'] = m
        self._dev.pop('processed_map', None)

    def _seq_map_dev(self):
        if 'seq_map' not in self._dev:
            self._dev['seq_map'] = dev.DeviceCSR.from_scipy(self._host['seq_map'], np.uint32)
        return self._dev['seq_map']

    def _processed_dev(self):
        if 'processed_map' not in self._dev:
            self._dev['processed_map'] = dev.DeviceCSR.from_scipy(self._host['processed_map'], np.float64)
        return self._dev['processed_map']

    # ---- accumulation ------------------------------------------------------------------------
    def _bin_map(self, bam, chunk_records=1 << 24):
        """
        Accumulate read-pair observations from the supplied pair records (contact_map.py:602-809).
        Filter order, canonicalisation and counters follow the reference loop (:733-739, :774-777,
        :796); the matcher outcome (:612-622) arrives as the record's pass bit.

        Host records are streamed to the device in chunks on a side stream so the copy of chunk k+1
        overlaps the classification of chunk k.
        """
        import torch
        dev.require_cuda()
        counts = OrderedDict({
            'accepted': 0,
            'not_tip': 0,
            'short_insert': 0,
            'ref_excluded': 0,
            'median_excluded': 0,
            'end_buffered': 0,
            'poor_match': 0})

        lut = np.full(self.n_refs, -1, dtype=np.int32)
        idx = self.make_reverse_index('refid')
        lut[np.fromiter(idx.keys(), dtype=np.int64, count=len(idx))] = \
            np.fromiter(idx.values(), dtype=np.int32, count=len(idx))

        if self.is_tipbased():
            # each tip is tracked separately: the single count becomes a 2x2 interaction matrix and the map a tensor
            # of dimension NxNx2x2 (contact_map.py:681-684); accumulated on the device over the doubled ids
            from . import sparse_utils
            n_rec = int(bam.records.numel()) if isinstance(bam.records, torch.Tensor) else len(bam.records)
            acc = sparse_utils.Sparse4DAccumulator(self.total_seq, tid2idx=lut, pair_capacity=max(n_rec, 1))
            acc.add_tip_pairs(bam.records, bam.tip10)
            self._dev.pop('seq_map', None)
            self._host['seq_map'] = acc.get_coo()
            counts.update(acc.counts)
            counts['short_insert'] = int(bam.meta.get('short_insert') or 0)
            counts['not_tip'] = int(bam.meta.get('not_tip') or 0)
            self.pair_counts = counts
            self._map_weight = int(self._host['seq_map'].data.sum(dtype=np.uint64))
            logger.info('Pair accounting: {}'.format(counts))
            logger.info('Total extent map weight {}'.format(self.map_weight()))
            return

        from .pipeline import HotPath
        hp = HotPath(lut, self.order.lengths(), np.array([si.sites for si in self.seq_info], dtype=np.int32),
                     min_len=self.min_len or 1, min_sig=self.min_sig or 1)
        csr = hp.accumulate(bam.records, chunk_records=chunk_records)
        info = hp.acc_info
        self._host['seq_map'] = None
        self._dev['seq_map'] = csr
        counts['accepted'] = info['accepted']
        counts['ref_excluded'] = info['ref_excluded']
        counts['poor_match'] = info['poor_match']
        if bam.meta is not None:
            # pairs the reader dropped for a short insert (contact_map.py:761-766) never became records
            counts['short_insert'] = int(bam.meta.get('short_insert') or 0)
        self.pair_counts = counts
        self._map_weight = info['map_weight']

        if self.bin_size:
            # the extent map (contact_map.py:687-691, 779-788, 801-803): the same sort-reduce over the bin-level
            # records, bins being their own index table; every pair the contig map accepts is tallied
            logger.info('Initialising contact map of {0}x{0} fragment bins, representing {1} bp over {2} sequences'
                        .format(self.grouping.total_bins, self.total_len, self.total_seq))
            nb = self.grouping.total_bins
            ident = np.arange(nb, dtype=np.int32)
            ext = bam.extent_records
            n_ext = int(ext.numel()) if isinstance(ext, torch.Tensor) else len(ext)
            hx = HotPath(ident, np.ones(nb, dtype=np.int32), np.ones(nb, dtype=np.int32), min_len=1, min_sig=1,
                         pair_capacity=n_ext)
            ecsr = hx.accumulate(ext, chunk_records=chunk_records)
            assert hx.acc_info['accepted'] == info['accepted'], 'extent records disagree with the pair records'
            self.extent_map = ecsr.to_scipy_coo()
            hx = None

        logger.info('Pair accounting: {}'.format(counts))
        logger.info('Total extent map weight {}'.format(self.map_weight()))

    @staticmethod
    def get_fields():
        return SeqInfo._fields

    def make_reverse_index(self, field_name):
        """Reverse look-up from a seq_info field to the internal index (contact_map.py:818-832)."""
        rev_idx = {}
        for n, seq in enumerate(self.seq_info):
            fv = getattr(seq, field_name)
            if fv in rev_idx:
                raise RuntimeError('field contains non-unique entries, a 1-1 mapping cannot be made')
            rev_idx[fv] = n
        return rev_idx

    def map_weight(self):
        """:return: the total map weight (sum ij) -- off-diagonals count twice (Q7)"""
        if getattr(self, '_map_weight', None) is not None:
            return self._map_weight
        return self.seq_map.sum()

    def is_empty(self):
        return self.map_weight() == 0

    def is_tipbased(self):
        return self.tip_size is not None

    # ---- filtering ---------------------------------------------------------------------------
    def get_primary_acceptance_mask(self):
        assert self.primary_acceptance_mask is not None, 'Primary acceptance mask has not be initialized'
        return self.primary_acceptance_mask.copy()

    def set_primary_acceptance_mask(self, min_len=None, min_sig=None, max_fold=None, update=False):
        """
        Determine and set the filter mask (contact_map.py:856-909):
        (length >= min_len) & (max off-diagonal raw count >= min_sig)   (Q4, Q5).
        """
        import torch
        assert max_fold is None, 'Filtering on max_fold is currently disabled'

        if not min_len:
            min_len = self.min_len
        if not min_sig:
            min_sig = self.min_sig

        assert min_len, 'Filtering criteria min_len is None'
        assert min_sig, 'Filtering criteria min_sig is None'

        logger.debug('Setting primary acceptance mask with '
                     'filtering criterion min_len: {} min_sig: {}'.format(min_len, min_sig))

        if not update and self.primary_acceptance_mask is not None:
            logger.debug('Using existing mask')
            return self.get_primary_acceptance_mask()

        if self.is_tipbased():
            # signal of a tensor: maximum off-diagonal of its 2-D marginal (sparse_utils.max_offdiag_4d, :896-897)
            from . import sparse_utils
            acceptance_mask = np.ones(self.total_seq, dtype=np.bool_)
            _mask = self.order.lengths() >= min_len
            logger.debug('Minimum length threshold removing: {}'.format(self.total_seq - _mask.sum()))
            acceptance_mask &= _mask
            _mask = sparse_utils.max_offdiag_4d(self.seq_map) >= min_sig
            logger.debug('Minimum signal threshold removing: {}'.format(self.total_seq - _mask.sum()))
            acceptance_mask &= _mask
            self.primary_acceptance_mask = acceptance_mask
            logger.debug('Accepted sequences: {}'.format(self.primary_acceptance_mask.sum()))
            return self.get_primary_acceptance_mask()

        csr = self._seq_map_dev()
        lengths = dev.to_device(np.ascontiguousarray(self.order.lengths()), torch.int32)
        signal = dev.max_offdiag(csr)
        self._dev['signal'] = signal
        mask_len = dev.acceptance_mask(lengths, signal, min_len, 0)
        mask_sig = dev.acceptance_mask(lengths, signal, np.iinfo(np.int32).min, min_sig)
        mask = dev.acceptance_mask(lengths, signal, min_len, min_sig)
        self._dev['mask'] = mask
        host = torch.stack([mask_len, mask_sig, mask]).cpu().numpy().astype(np.bool_)
        logger.debug('Minimum length threshold removing: {}'.format(self.total_seq - host[0].sum()))
        logger.debug('Minimum signal threshold removing: {}'.format(self.total_seq - host[1].sum()))

        self.primary_acceptance_mask = host[2]
        logger.debug('Accepted sequences: {}'.format(self.primary_acceptance_mask.sum()))
        return self.get_primary_acceptance_mask()

    # ---- normalisation + balancing -----------------------------------------------------------------
    def prepare_seq_map(self, norm=True, bisto=False, mean_type='geometric'):
        """
        Prepare the sequence map by normalisation and balancing (contact_map.py:911-945).  KR runs
        on the full N x N map, before masked contigs are removed, as the reference does (Q3).
        """
        logger.info('Preparing sequence map with full dimensions: {}'.format((self.total_seq, self.total_seq)))

        _mask = self.get_primary_acceptance_mask()
        self.order.set_mask_only(_mask)

        if self.order.count_accepted() < 1:
            raise NoneAcceptedException()

        if self.is_tipbased():
            from . import sparse_utils
            _map = self.seq_map.astype(np.float64)
            if norm:
                _map = self._norm_seq(_map, True, mean_type=mean_type, use_sites=True)
                logger.debug('Map normalized')
            if bisto:
                _map, scl = sparse_utils.kr_biostochastic_4d(_map)
                self.kr_info = sparse_utils.kr_biostochastic.last_info
                self.bisto_scale = scl
                logger.debug('Map balanced')
            self._dev.pop('processed_map', None)
            self._host['processed_map'] = _map
            return

        _map = self._seq_map_dev()

        if norm:
            _map = self._norm_seq(_map, self.is_tipbased(), mean_type=mean_type, use_sites=True)
            logger.debug('Map normalized')
        else:
            import torch
            _map = dev.DeviceCSR(_map.n, _map.indptr, _map.indices,
                                 dev.site_norm(_map, dev.to_device(np.ones(_map.n, np.int32), torch.int32)).data)

        if bisto:
            _map, scl = self._bisto_seq(_map)
            self.bisto_scale = scl
            logger.debug('Map balanced')

        self._host['processed_map'] = None
        self._dev['processed_map'] = _map

    def _bisto_seq(self, _map):
        """Make a contact map bistochastic (contact_map.py:1087-1101)."""
        logger.debug('Balancing contact map')
        if isinstance(_map, dev.DeviceCSR):
            x, info = dev.kr_scale_vector(_map)
            self.kr_info = info
            sp_logger = logging.getLogger('mzd.sparse_utils')
            if info['zero_diag']:
                sp_logger.warning('treating {} zeros on diagonal as ones'.format(info['zero_diag']))
            sp_logger.debug('It took {} iterations to achieve bistochasticity'.format(info['n_iter']))
            return dev.kr_apply(_map, x), x.cpu().numpy()
        from . import sparse_utils
        return sparse_utils.kr_biostochastic(_map)

    def _get_sites(self):
        _sites = np.array([si.sites for si in self.seq_info], dtype=np.float64)
        # all sequences are assumed to have a minimum of 1 site -- even if not observed (Q6)
        _sites[np.where(_sites == 0)] = 1
        return _sites

    def _norm_seq(self, _map, tip_based, use_sites=True, mean_type='geometric'):
        """
        Normalise a sequence map by the restriction-site counts of the interacting contigs
        (contact_map.py:1110-1145 with fast_norm_fullseq_bysite, :100-113).
        """
        import torch
        if tip_based:
            # fast_norm_tipbased_bysite (contact_map.py:84-97): data[n] *= 1.0 / (sites[i, k] * sites[j, l]) over the
            # (head, tail) site counts, zeros taken as one (:1103-1108)
            assert use_sites, 'length-based normalisation is dead code from the bin3C CLI'
            logger.debug('Doing site based normalisation')
            _sites = self._get_sites()
            _map = _map.astype(np.float64)
            i, j, k, l = _map.coords
            _map.data *= 1.0 / (_sites[i, k] * _sites[j, l])
            return _map
        if not use_sites:
            raise NotImplementedError('length-based normalisation is dead code from the bin3C CLI '
                                      '(prepare_seq_map hard-codes use_sites=True, contact_map.py:933)')
        logger.debug('Doing site based normalisation')
        sites = dev.to_device(np.array([si.sites for si in self.seq_info], dtype=np.int32), torch.int32)
        if isinstance(_map, dev.DeviceCSR):
            return dev.site_norm(_map, sites)
        # host matrix in, host matrix out (same container type as given)
        csr = dev.DeviceCSR.from_scipy(_map, np.float64)
        out = dev.site_norm(csr, sites).to_scipy_csr()
        return out.asformat(_map.getformat())

    # ---- subspace ------------------------------------------------------------------------------
    def get_subspace(self, permute=False, external_mask=None, marginalise=False, flatten=True, dtype=np.float64):
        """
        Using an already normalized full seq_map, return the map without filtered elements
        (contact_map.py:947-999).  Returns a coo_matrix, as sparse_utils.compress does.
        """
        assert (not marginalise and not flatten) or np.logical_xor(marginalise, flatten), \
            'marginalise and flatten are mutually exclusive'
        if permute:
            raise NotImplementedError('reordering is plot-only (contact_map.py:1066-1085) and out of scope')

        if self.is_tipbased():
            from . import sparse_utils
            _map = self.processed_map.astype(dtype)
            if external_mask is not None:
                _mask = self.get_primary_acceptance_mask()
                logger.info('Beginning with sequences after primary filtering: {}'.format(_mask.sum()))
                _mask &= external_mask
                logger.info('Active sequences after applying external mask: {}'.format(_mask.sum()))
                self.order.set_mask_only(_mask)
            if self.order.count_accepted() < self.total_seq:
                _map = sparse_utils.compress_4d(_map, self.order.mask_vector())
                logger.info('After removing filtered sequences map dimensions: {}'.format(_map.shape))
            if marginalise:
                logger.debug('Marginalising NxNx2x2 tensor to NxN matrix')
                _map = _map.sum(axis=(2, 3)).to_scipy_sparse()
            elif flatten:
                logger.debug('Flattening NxNx2x2 tensor to 2Nx2N matrix')
                _map = sparse_utils.flatten_tensor_4d(_map)
            return _map

        res = self._subspace_dev(external_mask, want_sub=True, want_edges=False, scale=False)
        if res is None:
            return self.processed_map.tocoo().astype(dtype)
        logger.info('After removing filtered sequences map dimensions: {}'.format((res['n_accepted'],) * 2))
        return res['sub'].to_scipy_coo().astype(dtype)

    # ---- extent (binned) map post-processing (contact_map.py:1001-1036, 1147-1165, 1197-1249) -----------------------
    def _extent_dev(self, _map=None):
        """The extent map (or a caller's matrix of the same shape) as a device CSR of raw counts."""
        m = self.extent_map if _map is None else _map
        assert scisp.isspmatrix(m), 'Extent matrix is not a scipy matrix type'
        return dev.DeviceCSR.from_scipy(m, np.uint32)

    def _bin_vectors(self):
        """Per bin: the length of its sequence (float64, device) and whether that sequence is accepted (uint8)."""
        import torch
        bins = np.asarray(self.grouping.bins, dtype=np.int64)
        bin_len = np.repeat(self.order.lengths().astype(np.float64), bins)
        bin_ok = np.repeat(self.order.mask_vector().astype(np.uint8), bins)
        return dev.to_device(bin_len), dev.to_device(bin_ok, torch.uint8)

    def _norm_extent(self, _map, mean_type='geometric'):
        """
        Normalise an extent map by the mean of the interacting sequences' lengths (contact_map.py:1147-1165):
        every entry is divided by 1e-3 * mean(L_i, L_j) on the device (b3c_extent_norm).

        :return: a normalized extent map in lil_matrix format
        """
        assert scisp.isspmatrix(_map), 'Extent matrix is not a scipy matrix type'
        bin_len, _ = self._bin_vectors()
        return dev.extent_norm(self._extent_dev(_map), bin_len, mean_type).to_scipy_csr().tolil()

    def _compress_extent(self, _map):
        """
        Compress the extent map for each sequence that is presently masked: all bins of a masked sequence are
        removed and the remaining bins renumbered (contact_map.py:1197-1249), with the device compaction kernels.

        :return: a scipy.sparse.coo_matrix pertaining to only the unmasked sequences.
        """
        assert scisp.isspmatrix(_map), 'Extent matrix is not a scipy sparse matrix type'
        _, bin_ok = self._bin_vectors()
        csr = dev.DeviceCSR.from_scipy(_map, np.float64)
        res = dev.compress_edges(csr, bin_ok, want_sub=True, want_edges=False, scale=False)
        return res['sub'].to_scipy_coo()

    def get_extent_map(self, norm=True, bisto=False, permute=False, mean_type='geometric'):
        """
        Return the extent map after applying specified processing steps. Masked sequences are always removed
        (contact_map.py:1001-1036).  Normalisation, compaction and balancing all run on the device; nothing but the
        result comes back to the host.

        :param norm: sequence length normalisation
        :param bisto: make map bistochastic
        :param permute: permute the map using current order (plot-only, contact_map.py:1167-1195: not built)
        :param mean_type: length normalisation mean (geometric, harmonic, arithmetic)
        :return: processed extent map
        """
        assert self.extent_map is not None, 'this map was built without bin_size'
        if permute:
            raise NotImplementedError('reordering is plot-only (contact_map.py:1167-1195) and out of scope')
        logger.info('Preparing extent map with fill dimensions: {}'.format(self.extent_map.shape))
        bin_len, bin_ok = self._bin_vectors()
        m = dev.extent_norm(self._extent_dev(), bin_len, mean_type if norm else None)
        if norm:
            logger.debug('Map normalized')
        compressed = self.order.count_accepted() < self.total_seq
        if compressed:
            m = dev.compress_edges(m, bin_ok, want_sub=True, want_edges=False, scale=False)['sub']
            logger.info('After removing filtered sequences map dimensions: {}'.format((m.n, m.n)))
        if bisto:
            x, _ = dev.kr_scale_vector(m)
            m = dev.kr_apply(m, x)
            logger.debug('Map balanced')
            return m.to_scipy_csr()
        if compressed:
            return m.to_scipy_coo()
        return m.to_scipy_csr().tolil() if norm else m.to_scipy_coo()

    def _subspace_dev(self, external_mask, want_sub, want_edges, scale, force=False):
        import torch
        if external_mask is not None:
            _mask = self.get_primary_acceptance_mask()
            logger.info('Beginning with sequences after primary filtering: {}'.format(_mask.sum()))
            _mask &= external_mask
            logger.info('Active sequences after applying external mask: {}'.format(_mask.sum()))
            self.order.set_mask_only(_mask)
        if not force and not self.order.count_accepted() < self.total_seq:
            return None
        mask = dev.to_device(self.order.mask_vector().astype(np.uint8), torch.uint8)
        return dev.compress_edges(self._processed_dev(), mask, want_sub=want_sub, want_edges=want_edges, scale=scale)
