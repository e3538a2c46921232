"""
Golden vectors of the WHOLE reference path, produced by the reference's own classes: SeqOrder and ContactMap
(contact_map.py:159-485, 486-end) exec'd verbatim under Python 3 (oracle/ref_exec.run_reference_path; __init__'s
pysam/Biopython part replayed from the reference table), driven as bin3C.py does -- _bin_map ->
set_primary_acceptance_mask -> to_graph [prepare_seq_map(norm, bisto) -> _norm_seq, _bisto_seq (kr_biostochastic);
get_subspace(marginalise=True, flatten=False) -> compress] -- on a synthetic community whose pair records are
presented as duck-typed alignment records.  Nothing here comes from oracle/oracle.py.
With a reference checkout (see oracle/ref_exec.py):  python tests/golden/make_golden_refpath.py
"""
import logging
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from bin3c_b200 import synth          # noqa: E402
from oracle import ref_exec           # noqa: E402

MIN_LEN, MIN_SIG = 1000, 3


def alignments_of(records):
    ti, tj, ok = synth.unpack_pairs(records)
    alns = []
    for k, (a, b, p) in enumerate(zip(ti.tolist(), tj.tolist(), ok.tolist())):
        q1, q2 = (60, 60) if p else ((60, 3) if k & 1 else (7, 60))
        alns.append(dict(name='p%d' % k, flag=0x41, tid=a, pos=5, mapq=q1, cigar=[(0, 100)]))
        alns.append(dict(name='p%d' % k, flag=0x81, tid=b, pos=9, mapq=q2, cigar=[(0, 100)]))
    return alns


def main():
    com = synth.make_community(n_genomes=6, n_contigs=500, n_pairs=120000, seed=8086)
    n_refs = com.n_refs
    lengths = np.full(n_refs, 500, dtype=np.int64)
    sites = np.ones(n_refs, dtype=np.int64)
    lengths[com.ref_index] = com.lengths
    sites[com.ref_index] = com.sites
    sites[com.ref_index[::41]] = 0                       # zero site counts are taken as one (Q6)
    cap = ref_exec.IterCapture()
    logging.getLogger('mzd.sparse_utils').addHandler(cap)
    res = ref_exec.run_reference_path(alignments_of(com.records), lengths, sites, MIN_LEN, MIN_SIG, min_mapq=60)
    logging.getLogger('mzd.sparse_utils').removeHandler(cap)
    g = res['graph']
    e = sorted((min(a, b), max(a, b), w) for a, b, w in g.edges(data='weight'))
    sm, pm = res['seq_map'], res['processed_map'].tocoo()
    c = res['counts']
    out = dict(lengths=lengths, sites=sites, records=com.records, min_len=np.int64(MIN_LEN), min_sig=np.int64(MIN_SIG),
               counts=np.array([c['accepted'], c['ref_excluded'], c['poor_match']], dtype=np.int64),
               map_row=sm.row.astype(np.int64), map_col=sm.col.astype(np.int64), map_data=sm.data.astype(np.int64),
               mask=np.asarray(res['mask']).astype(np.uint8), kr_x=np.asarray(res['bisto_scale'], dtype=np.float64),
               kr_n_iter=np.int64(cap.n_iter),
               bal_row=pm.row.astype(np.int64), bal_col=pm.col.astype(np.int64), bal_data=pm.data.astype(np.float64),
               edge_u=np.array([a for a, _, _ in e], dtype=np.int64), edge_v=np.array([b for _, b, _ in e], dtype=np.int64),
               edge_w=np.array([w for _, _, w in e], dtype=np.float64))
    np.savez_compressed(os.path.join(HERE, 'refpath.npz'), **out)
    print('wrote refpath.npz', os.path.getsize(os.path.join(HERE, 'refpath.npz')), 'counts', c, 'accepted contigs',
          int(out['mask'].sum()), 'kr iterations', cap.n_iter, 'edges', len(e))


if __name__ == '__main__':
    main()
