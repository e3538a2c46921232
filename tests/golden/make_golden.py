"""
Generate the golden vectors under tests/golden/ by running the REFERENCE's own functions
(exec'd verbatim from a reference checkout by oracle/ref_exec.py) on seeded synthetic inputs.

With a reference checkout (see oracle/ref_exec.py):   python tests/golden/make_golden.py

What is reference-verbatim: Sparse2DAccumulator (+get_coo), max_offdiag, kr_biostochastic
(+is_hermitian), compress  (sparse_utils.py:227-266, 269-281, 90-224, 284-314).
What had to be re-driven because it cannot execute here (no pysam / numba typing / Py2
itertools): the pair loop of contact_map.py:720-798 (driven over packed records through
the reference accumulator's __getitem__/__setitem__ protocol), the site normalisation of
contact_map.py:110-113, the mask of :888-905, and the nx.Graph edge loop of
cluster.py:314-321 (run here with the installed networkx, last-writer-wins included).

Later in the round those pieces were made to execute too -- the pair loop on duck-typed alignment records
(make_golden_binmap.py), ExtentGrouping with a Python-2 division shim (make_golden_extent.py) and the whole path
through the reference's own SeqOrder / ContactMap classes and to_graph (make_golden_refpath.py): those vectors
contain no re-driven glue.  The five cases made by this script are kept as they are.
"""
import os
import sys

import numpy as np
import networkx as nx

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, '..', '..'))

from bin3c_b200 import synth            # noqa: E402
from oracle import ref_exec             # noqa: E402

CASES = {
    # name: (community kwargs, min_len, min_sig)
    'small': (dict(n_genomes=4, n_contigs=300, n_pairs=30_000, seed=11), 1000, 3),
    'dups': (dict(n_genomes=2, n_contigs=40, n_pairs=20_000, seed=12), 1000, 5),
    'sparse': (dict(n_genomes=5, n_contigs=500, n_pairs=3_000, seed=13), 2000, 2),
    'c1mini': (dict(n_genomes=10, n_contigs=2000, n_pairs=150_000, seed=1001), 1000, 5),
    'heavy': (dict(n_genomes=6, n_contigs=800, n_pairs=60_000, seed=14, profile='heavy'), 1500, 4),
}


def run_case(fns, kw, min_len, min_sig):
    com = synth.make_community(**kw)
    n = com.n_contigs
    tid_i, tid_j, passed = synth.unpack_pairs(com.records)
    idx_of = {int(t): k for k, t in enumerate(com.ref_index)}     # make_reverse_index('refid')

    # --- contact_map.py:720-798 driven through the reference accumulator
    acc = fns['Sparse2DAccumulator'](n)
    counts = {'accepted': 0, 'ref_excluded': 0, 'poor_match': 0}
    for a, b, ok in zip(tid_i.tolist(), tid_j.tolist(), passed.tolist()):
        if a not in idx_of or b not in idx_of:
            counts['ref_excluded'] += 1
            continue
        if not ok:
            counts['poor_match'] += 1
            continue
        ix1, ix2 = idx_of[a], idx_of[b]
        if ix2 < ix1:
            ix1, ix2 = ix2, ix1
        counts['accepted'] += 1
        acc[ix1, ix2] += 1
    seq_map = acc.get_coo()
    assert seq_map.dtype == np.uint32

    # --- contact_map.py:888-905
    signal = fns['max_offdiag'](seq_map)
    mask = (com.lengths >= min_len) & (signal >= min_sig)

    # --- contact_map.py:929, 1103-1108, 110-113
    fmap = seq_map.astype(float)
    sites = np.array(com.sites, dtype=float)
    sites[np.where(sites == 0)] = 1
    for k in range(fmap.data.shape[0]):
        fmap.data[k] *= 1.0 / (sites[fmap.row[k]] * sites[fmap.col[k]])

    # --- sparse_utils.py:90-224
    bal, x, n_iter, warns = ref_exec.kr_with_iterations(fns, fmap)

    # --- contact_map.py:966-982, sparse_utils.py:284-314
    sub = bal.astype(float)
    if mask.sum() < n:
        sub = fns['compress'](sub.tocoo(), mask)
    sub = sub.tocoo()

    # --- cluster.py:314-321
    scl = 1.0 / sub.max()
    g = nx.Graph(name='contact_graph')
    for u, v, w in zip(sub.row, sub.col, sub.data):
        g.add_edge(int(u), int(v), weight=w * scl)
    edges = sorted((min(u, v), max(u, v), d['weight']) for u, v, d in g.edges(data=True))
    eu = np.array([e[0] for e in edges], dtype=np.int64)
    ev = np.array([e[1] for e in edges], dtype=np.int64)
    ew = np.array([e[2] for e in edges], dtype=np.float64)

    balc = bal.tocsr()
    balc.sort_indices()
    return dict(
        n_refs=np.int64(com.n_refs), ref_index=com.ref_index, lengths=com.lengths, sites=com.sites,
        records=com.records, min_len=np.int64(min_len), min_sig=np.int64(min_sig),
        counts=np.array([counts['accepted'], counts['ref_excluded'], counts['poor_match']], dtype=np.int64),
        map_row=seq_map.row.astype(np.int32), map_col=seq_map.col.astype(np.int32), map_data=seq_map.data,
        map_weight=np.uint64(seq_map.sum()),
        signal=np.asarray(signal), mask=mask,
        kr_x=x, kr_n_iter=np.int64(n_iter), kr_zero_diag=np.int64((fmap.tocsr().diagonal() == 0).sum()),
        bal_indptr=balc.indptr.astype(np.int64), bal_indices=balc.indices.astype(np.int32), bal_data=balc.data,
        sub_n=np.int64(sub.shape[0]), sub_nnz=np.int64(sub.nnz), scl=np.float64(scl),
        edge_u=eu, edge_v=ev, edge_w=ew)


def main():
    fns = ref_exec.load()
    for name, (kw, min_len, min_sig) in CASES.items():
        out = run_case(fns, kw, min_len, min_sig)
        path = os.path.join(HERE, '{}.npz'.format(name))
        np.savez_compressed(path, **out)
        print('{:8s} N={} P={} nnz={} accepted={} kr_iter={} zero_diag={} edges={} -> {} ({} KB)'.format(
            name, len(out['lengths']), len(out['records']), len(out['map_data']), int(out['mask'].sum()),
            int(out['kr_n_iter']), int(out['kr_zero_diag']), len(out['edge_u']), os.path.basename(path),
            os.path.getsize(path) // 1024))


if __name__ == '__main__':
    main()
