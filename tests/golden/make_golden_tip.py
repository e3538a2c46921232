"""
Golden vectors for the tip-based map (SURVEY.md 8f rank 4): the reference's own code exec'd verbatim under Python 3
(oracle/ref_exec.py) with SparseShim standing in for pydata `sparse` --
  * ContactMap._bin_map with tip_size (contact_map.py:602-809: _on_tip_withlocs, Sparse4DAccumulator) on the alignment
    stream of make_golden_binmap.py: the N x N x 2 x 2 tensor and the pair counters (incl. not_tip), for tips that do
    not overlap, tips that overlap on the shorter sequences, and the insert filter;
  * max_offdiag_4d, flatten_tensor_4d, compress_4d, kr_biostochastic_4d on that tensor (sparse_utils.py:412-509);
  * the whole path by the reference's own classes: _bin_map -> set_primary_acceptance_mask -> to_graph
    [prepare_seq_map(norm, bisto) with fast_norm_tipbased_bysite, get_subspace(marginalise=True)]: mask, scale factors,
    processed tensor, graph edges; plus get_subspace(flatten=True).
With a reference checkout (see oracle/ref_exec.py):  python tests/golden/make_golden_tip.py
"""
import os
import random
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
sys.path.insert(0, HERE)

from oracle import ref_exec                       # noqa: E402
from make_golden_binmap import make_alignments    # noqa: E402

PARAMS = [dict(min_mapq=30, tip_size=300), dict(min_mapq=30, tip_size=700, strong=40),
          dict(min_mapq=20, tip_size=5000, min_insert=1500)]
MIN_LEN, MIN_SIG = 1000, 2


def main():
    rng = random.Random(90417)
    n_refs = 90
    lengths = [rng.choice([400, 900, 1000, 1001, 1400, 1800, 2600, 9000, 30000]) for _ in range(n_refs)]
    alns = make_alignments(rng, n_refs, lengths, 14000)
    # positions exactly on the tip boundaries and in the middle of short sequences (the `<` / `>` of :638-665)
    for a in alns[::37]:
        ln = lengths[a['tid']]
        a['pos'] = rng.choice([ln // 2, 300, ln - 300, 299, ln - 299, 700, ln - 700, 0, ln - 1])
        a['pos'] = min(max(a['pos'], 0), ln - 1)
    sites2 = [[rng.choice([0, 1, 2, 5, 9, 30]), rng.choice([0, 1, 3, 7, 11])] for _ in range(n_refs)]
    keep = np.array(lengths) >= MIN_LEN
    lut = np.where(keep, np.cumsum(keep) - 1, -1)
    idx = {t: int(i) for t, i in enumerate(lut) if i >= 0}
    n_seq = int(keep.sum())
    out = {'lengths': np.array(lengths, dtype=np.int64), 'sites2': np.array(sites2, dtype=np.int64),
           'min_len': np.int64(MIN_LEN), 'min_sig': np.int64(MIN_SIG),
           'name': np.array([a['name'] for a in alns], dtype=np.int64),
           'flag': np.array([a['flag'] for a in alns], dtype=np.int64),
           'tid': np.array([a['tid'] for a in alns], dtype=np.int64),
           'pos': np.array([a['pos'] for a in alns], dtype=np.int64),
           'mapq': np.array([a['mapq'] for a in alns], dtype=np.int64),
           'cig_ptr': np.cumsum([0] + [len(a['cigar']) for a in alns]).astype(np.int64),
           'cig_op': np.array([op for a in alns for op, _ in a['cigar']], dtype=np.int64),
           'cig_len': np.array([n for a in alns for _, n in a['cigar']], dtype=np.int64),
           'n_params': np.int64(len(PARAMS))}
    named = [dict(a, name='t%d' % a['name']) for a in alns]
    fns = ref_exec.load_4d()
    for k, kw in enumerate(PARAMS):
        p = 'p%d_' % k
        res = ref_exec.run_bin_map(named, lengths, idx, n_seq, **kw)
        for key in ('min_mapq', 'strong', 'min_insert', 'tip_size'):
            out[p + key] = np.int64(kw.get(key) or 0)
        c = res['counts']
        out[p + 'counts'] = np.array([c['accepted'], c['ref_excluded'], c['poor_match'], c['short_insert'], c['not_tip']],
                                     dtype=np.int64)
        sm = res['seq_map']
        out[p + 'coords'], out[p + 'data'] = sm.coords.astype(np.int64), sm.data.astype(np.int64)
        out[p + 'signal'] = fns['max_offdiag_4d'](sm).astype(np.int64)
        fl = fns['flatten_tensor_4d'](sm)
        out[p + 'flat_row'], out[p + 'flat_col'] = fl.row.astype(np.int64), fl.col.astype(np.int64)
        out[p + 'flat_data'] = np.asarray(fl.data).astype(np.int64)
        mask = np.arange(n_seq) % 4 != 1
        cm = fns['compress_4d'](sm, mask)
        out[p + 'cmp_coords'], out[p + 'cmp_data'] = cm.coords.astype(np.int64), cm.data.astype(np.int64)
        out[p + 'cmp_n'] = np.int64(cm.shape[0])
        bal, scl = fns['kr_biostochastic_4d'](sm)
        out[p + 'kr_scl'], out[p + 'kr_data'] = scl, bal.data
        # the whole path by the reference's classes
        path = ref_exec.run_reference_path(named, lengths, sites2, MIN_LEN, MIN_SIG, min_mapq=kw['min_mapq'],
                                           strong=kw.get('strong'), min_insert=kw.get('min_insert'),
                                           tip_size=kw['tip_size'])
        assert np.array_equal(path['seq_map'].coords, sm.coords) and np.array_equal(path['seq_map'].data, sm.data)
        out[p + 'mask'] = path['mask']
        out[p + 'bisto_scale'] = path['bisto_scale']
        out[p + 'proc_coords'] = path['processed_map'].coords.astype(np.int64)
        out[p + 'proc_data'] = path['processed_map'].data
        g = path['graph']
        e = sorted((min(u, v), max(u, v), d['weight']) for u, v, d in g.edges(data=True))
        out[p + 'edge_u'] = np.array([x[0] for x in e], dtype=np.int64)
        out[p + 'edge_v'] = np.array([x[1] for x in e], dtype=np.int64)
        out[p + 'edge_w'] = np.array([x[2] for x in e], dtype=np.float64)
        out[p + 'n_nodes'] = np.int64(g.number_of_nodes())
        fsub = path['cm'].get_subspace(marginalise=False, flatten=True).tocsr()
        fsub.sort_indices()
        out[p + 'fsub_indptr'], out[p + 'fsub_indices'], out[p + 'fsub_data'] = fsub.indptr, fsub.indices, fsub.data
        print(kw, c, 'nnz', sm.nnz, 'accepted seqs', int(path['mask'].sum()), 'edges', len(e))
    np.savez_compressed(os.path.join(HERE, 'tipmap.npz'), **out)
    print('wrote tipmap.npz', os.path.getsize(os.path.join(HERE, 'tipmap.npz')))


if __name__ == '__main__':
    main()
