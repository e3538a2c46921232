"""
Restriction-site counts per sequence of a multi-FASTA: the part of ContactMap.__init__ (contact_map.py:520-531,
seq_utils.py:95-161 SiteCounter) that precedes the hot path, so that `ContactMap(bam_path, enzymes, fasta_path, ...)`
-- the call bin3C.py mkmap makes (bin3C.py:148-158) -- works end to end without Biopython.  The reference counts with
Bio.Restriction (`len(enzyme.search(seq, linear=True))` summed over the enzymes, seq_utils.py:134-150): the number of
occurrences of each enzyme's recognition site, overlapping ones included.  Not pinned against Biopython (absent here);
a caller that has its own counts passes them instead (ContactMap's `seq_file` also takes an array, dict or callable).

Two counters give the same table: the host counter below (the specification), and with `device=True` the GPU counter
(bin3c_b200/csrc/sites.cu): one host thread reads -- and for .gz files inflates -- the file into pinned slabs while
the device classifies lines, strips whitespace, and counts every pattern on the previous slab.
"""
import gzip
import locale
import re
import time
from difflib import SequenceMatcher

import numpy as np

from .exceptions import UnknownEnzymeException

# recognition sites (NEB spelling) of the enzymes Hi-C / Meta3C protocols use; IUPAC codes allowed
RECOGNITION = {
    'MluCI': 'AATT', 'Sau3AI': 'GATC', 'DpnII': 'GATC', 'MboI': 'GATC', 'BfuCI': 'GATC', 'HindIII': 'AAGCTT',
    'NcoI': 'CCATGG', 'NlaIII': 'CATG', 'HinfI': 'GANTC', 'DdeI': 'CTNAG', 'MseI': 'TTAA', 'Csp6I': 'GTAC',
    'CviQI': 'GTAC', 'CviAII': 'CATG', 'EcoRI': 'GAATTC', 'BglII': 'AGATCT', 'XhoI': 'CTCGAG', 'SphI': 'GCATGC',
    'ApoI': 'RAATTY', 'HpyCH4IV': 'ACGT', 'AluI': 'AGCT', 'BamHI': 'GGATCC', 'SacI': 'GAGCTC', 'PstI': 'CTGCAG',
    'HpaII': 'CCGG', 'MspI': 'CCGG', 'TaqI': 'TCGA', 'XbaI': 'TCTAGA', 'NheI': 'GCTAGC', 'SalI': 'GTCGAC',
}
_IUPAC = {'A': 'A', 'C': 'C', 'G': 'G', 'T': 'T', 'R': '[AG]', 'Y': '[CT]', 'S': '[CG]', 'W': '[AT]', 'K': '[GT]',
          'M': '[AC]', 'B': '[CGT]', 'D': '[AGT]', 'H': '[ACT]', 'V': '[ACG]', 'N': '[ACGT]'}
_COMP = str.maketrans('ACGTRYSWKMBDHVN', 'TGCAYRSWMKVHDBN')


# IUPAC code -> the set of bases as a 4-bit mask (A 1, C 2, G 4, T 8): the device counter's form of a pattern
_MASK = {'A': 1, 'C': 2, 'G': 4, 'T': 8, 'R': 5, 'Y': 10, 'S': 6, 'W': 9, 'K': 12, 'M': 3, 'B': 14, 'D': 13, 'H': 11,
         'V': 7, 'N': 15}
MAX_SITE_LEN = 16               # include/bin3c_b200.h: B3C_SITES_MAX_LEN
MAX_DEVICE_PATTERNS = 64        # B3C_SITES_MAX_PATTERNS (distinct patterns)
MAX_SLAB_BYTES = 1 << 30        # B3C_SITES_MAX_SLAB
DEFAULT_SLAB_BYTES = 64 << 20   # file bytes per slab of the device counter


def _sites(enzyme_names):
    """The searched sites in search order: per enzyme, in list order, the sorted set {site, reverse complement}."""
    if isinstance(enzyme_names, str):
        enzyme_names = [enzyme_names]
    sites = []
    for name in enzyme_names:
        site = RECOGNITION.get(name)
        if site is None:        # strict about names, helpful about near misses (seq_utils.py:119-131)
            similar = [k for k in RECOGNITION if SequenceMatcher(None, name.lower(), k.lower()).ratio() >= 0.8]
            raise UnknownEnzymeException(name, similar)
        both = {site, site.translate(_COMP)[::-1]}           # a non-palindromic site is searched on both strands
        sites.extend(sorted(both))
    return sites


def _patterns(enzyme_names):
    return [re.compile('(?=' + ''.join(_IUPAC[c] for c in s) + ')') for s in _sites(enzyme_names)]


def count_sites(seq, patterns):
    """Occurrences of every pattern (overlapping ones included) in an upper-case sequence string."""
    return sum(sum(1 for _ in p.finditer(seq)) for p in patterns)


def tip_sites(seq, patterns, tip_size):
    """[head sites, tail sites] of a tip-based map (SiteCounter.count_sites, seq_utils.py:146-158): the first and last
    tip_size bases, or the two halves of a sequence shorter than 2 tip_size -- with Python 2's integer division,
    seq[:n/2] and seq[-n/2:]: -n/2 rounds towards minus infinity, so the tail half of an odd-length sequence is the
    longer one."""
    n = len(seq)
    if n < 2 * tip_size:
        l_tip, r_tip = seq[:n // 2], seq[(-n) // 2:]
    else:
        l_tip, r_tip = seq[:tip_size], seq[-tip_size:]
    return [count_sites(l_tip, patterns), count_sites(r_tip, patterns)]


def fasta_site_table(path, enzyme_names, min_len=0, tip_size=None, device=False, slab_bytes=DEFAULT_SLAB_BYTES):
    """{sequence id: {'sites': n, 'length': L}} for the sequences of at least min_len bases -- the reference's
    `fasta_info` (contact_map.py:520-531).  Plain or gzip'd FASTA.  With tip_size, 'sites' is [head, tail].

    device=True counts on the GPU and returns the same dict (same keys in the same order, Python ints).  It raises
    RuntimeError without a CUDA device, and ValueError for a byte >= 0x80 in a sequence line (text mode counts such
    characters, not bytes), for a site longer than MAX_SITE_LEN bases and for more than MAX_DEVICE_PATTERNS distinct
    sites; the host counter (device=False) takes all of these.  slab_bytes: file bytes the device counts per step.
    """
    pats = _patterns(enzyme_names)
    if device:
        return _site_table_on_device(path, _device_patterns(_sites(enzyme_names)), min_len, tip_size, slab_bytes)
    opener = gzip.open if str(path).endswith('.gz') else open
    info = {}

    def flush(name, parts):
        if name is None:
            return
        seq = ''.join(parts).upper()
        if len(seq) >= min_len:
            info[name] = {'sites': tip_sites(seq, pats, tip_size) if tip_size else count_sites(seq, pats),
                          'length': len(seq)}

    name, parts = None, []
    with opener(path, 'rt') as fh:
        for line in fh:
            if line.startswith('>'):
                flush(name, parts)
                name, parts = line[1:].split()[0] if len(line) > 1 and line[1:].split() else '', []
            else:
                parts.append(line.strip())
    flush(name, parts)
    return info


def _device_patterns(sites):
    """Sites -> (masks uint8[n, MAX_SITE_LEN], lengths int32[n], weights int32[n]): one entry per distinct site,
    weighted by how often it is searched."""
    distinct = {}
    for site in sites:
        if not 1 <= len(site) <= MAX_SITE_LEN:
            raise ValueError('site {!r} has {} bases: the device counter takes 1 to {}; count with the host counter '
                             '(device=False)'.format(site, len(site), MAX_SITE_LEN))
        distinct[site] = distinct.get(site, 0) + 1
    if len(distinct) > MAX_DEVICE_PATTERNS:
        raise ValueError('{} distinct sites: the device counter takes at most {}; count with the host counter '
                         '(device=False)'.format(len(distinct), MAX_DEVICE_PATTERNS))
    masks = np.zeros((len(distinct), MAX_SITE_LEN), dtype=np.uint8)
    for p, site in enumerate(distinct):
        masks[p, :len(site)] = [_MASK[c] for c in site]
    lengths = np.array([len(s) for s in distinct], dtype=np.int32)
    weights = np.array(list(distinct.values()), dtype=np.int32)
    return masks, lengths, weights


def site_table_from_rows(rows, names, min_len, tip_size):
    """The dict fasta_site_table returns, from the per-sequence table of the device counter (include/bin3c_b200.h:
    b3c_sites_finish: length, name range, sites or head sites, tail sites) and its name arena.  Names are split as
    the host counter splits them: decoded with the encoding text mode uses."""
    enc = locale.getpreferredencoding(False)
    info = {}
    for length, lo, hi, s, t in np.asarray(rows, dtype=np.int64).reshape(-1, 5).tolist():
        if length >= min_len:
            toks = names[lo:hi].decode(enc).split()
            info[toks[0] if toks else ''] = {'sites': [s, t] if tip_size else s, 'length': length}
    return info


def _site_table_on_device(path, patterns, min_len, tip_size, slab_bytes, timing=None):
    """
    fasta_site_table(device=True).  One host thread reads (and inflates) the file into two pinned slabs while the
    device counts the previous one (include/bin3c_b200.h: b3c_sites_*); each slab crosses with one asynchronous copy
    and one synchronisation.  The per-sequence table and the name arena stay on the device until the end.
    `timing`: a dict that receives the seconds spent reading / inflating, in slab calls, and waiting for the reader.
    """
    import ctypes as C
    import queue
    import threading
    import torch
    if not torch.cuda.is_available():
        raise RuntimeError('fasta_site_table(device=True) needs a CUDA device; the host counter is device=False')
    from . import _cabi
    masks, lengths, weights = patterns
    slab = max(1, min(int(slab_bytes), MAX_SLAB_BYTES))
    tip = int(tip_size) if tip_size else 0
    dev = torch.device('cuda', torch.cuda.current_device())
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    nws = int(_cabi.lib.b3c_sites_workspace_bytes(slab, tip))
    _cabi.check(0 if nws > 0 else int(nws))
    ws = torch.empty(nws, dtype=torch.uint8, device=dev)
    _cabi.check(_cabi.lib.b3c_sites_begin(ws.data_ptr(), nws, slab, masks.ctypes.data, lengths.ctypes.data,
                                          weights.ctypes.data, len(lengths), tip, stream))
    pinned = [torch.empty(slab, dtype=torch.uint8, pin_memory=True) for _ in range(2)]
    free, ready = queue.Queue(), queue.Queue()
    for k in range(2):
        free.put(k)
    t = {'read_s': 0.0, 'slab_s': 0.0, 'wait_s': 0.0, 'slabs': 0, 'bytes': 0}

    def read_slabs():
        try:
            gz = str(path).endswith('.gz')
            with (gzip.open(path, 'rb') if gz else open(path, 'rb', buffering=0)) as f:
                while True:
                    k = free.get()
                    if k is None:
                        return
                    view = memoryview(pinned[k].numpy())
                    n, t0 = 0, time.perf_counter()
                    while n < slab:
                        m = f.readinto(view[n:])
                        if not m:
                            break
                        n += m
                    t['read_s'] += time.perf_counter() - t0
                    ready.put((k, n))
                    if n < slab:
                        return
        except BaseException as e:                              # handed to the counting thread
            ready.put((None, e))

    reader = threading.Thread(target=read_slabs, name='fasta-slab-reader', daemon=True)
    reader.start()
    d_buf = torch.empty(slab, dtype=torch.uint8, device=dev)
    seq_cap, name_cap = 1 << 12, 1 << 16
    seqs = torch.empty((seq_cap, 5), dtype=torch.int64, device=dev)
    names = torch.empty(name_cap, dtype=torch.uint8, device=dev)
    res = (C.c_int64 * 3)()
    try:
        while True:
            t0 = time.perf_counter()
            k, n = ready.get()
            t['wait_s'] += time.perf_counter() - t0
            if k is None:
                raise n
            if n == 0:
                break
            t0 = time.perf_counter()
            d_buf[:n].copy_(pinned[k][:n], non_blocking=True)
            while True:
                rc = _cabi.lib.b3c_sites_slab(ws.data_ptr(), d_buf.data_ptr(), n, seqs.data_ptr(), seq_cap,
                                              names.data_ptr(), name_cap, res, stream)
                if rc != _cabi.B3C_ERR_CAPACITY:
                    break
                if res[0] > seq_cap:                            # grow, keep what is written, count the slab again
                    seq_cap = max(2 * seq_cap, int(res[0]))
                    grown = torch.empty((seq_cap, 5), dtype=torch.int64, device=dev)
                    grown[:len(seqs)].copy_(seqs)
                    seqs = grown
                if res[1] > name_cap:
                    name_cap = max(2 * name_cap, int(res[1]))
                    grown = torch.empty(name_cap, dtype=torch.uint8, device=dev)
                    grown[:len(names)].copy_(names)
                    names = grown
            free.put(k)                                         # the slab call synchronised: the pinned slab is free
            t['slab_s'] += time.perf_counter() - t0
            t['slabs'] += 1
            t['bytes'] += n
            if rc == _cabi.B3C_ERR_FORMAT:
                raise ValueError('{}: {}; count this file with the host counter (device=False)'.format(
                    path, _cabi.last_error()))
            _cabi.check(rc)
            if n < slab:
                break
    finally:
        free.put(None)
        reader.join()
    n_seq = int(res[0])
    out = torch.empty((max(n_seq, 1), 5), dtype=torch.int64, device=dev)
    _cabi.check(_cabi.lib.b3c_sites_finish(ws.data_ptr(), seqs.data_ptr(), out.data_ptr(), n_seq, res, stream))
    rows = out[:n_seq].cpu().numpy()
    arena = bytes(names[:int(res[1])].cpu().numpy())
    if timing is not None:
        timing.update(t)
    return site_table_from_rows(rows, arena, min_len, tip_size)
