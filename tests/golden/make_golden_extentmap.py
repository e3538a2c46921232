"""
Golden vectors of the extent (binned) map's post-processing -- ContactMap.get_extent_map, _norm_extent and
_compress_extent (contact_map.py:1001-1036, 1147-1165, 1197-1249) -- produced by the reference's own ContactMap class
exec'd verbatim under Python 3 (oracle/ref_exec.run_reference_path with bin_size): _bin_map over duck-typed alignment
records builds seq_map and extent_map, set_primary_acceptance_mask masks some sequences, then get_extent_map is called
for every mean type, with and without balancing.  Nothing here comes from oracle/oracle.py.
With a reference checkout (see oracle/ref_exec.py):  python tests/golden/make_golden_extentmap.py
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from oracle import ref_exec           # noqa: E402

MIN_LEN, MIN_SIG, BIN_SIZE = 1000, 26, 1500


def main():
    rng = np.random.default_rng(60606)
    n_refs = 70
    lengths = rng.integers(500, 9000, n_refs)
    sites = np.maximum(1, lengths // 256)
    genome = rng.integers(0, 4, n_refs)
    alns, tid, pos, flag, mapq = [], [], [], [], []
    for k in range(30_000):
        a = int(rng.integers(n_refs))
        if rng.random() < 0.55:
            b = a
        else:
            same = np.flatnonzero(genome == genome[a])
            b = int(rng.choice(same)) if rng.random() < 0.9 else int(rng.integers(n_refs))
        rec = []
        for which, t in ((0x41, a), (0x81, b)):
            f = which | (0x10 if rng.random() < 0.5 else 0)
            p = int(rng.integers(0, max(1, lengths[t] - 100)))
            q = 60 if rng.random() < 0.9 else 5
            rec.append(dict(name='q%d' % k, flag=f, tid=t, pos=p, mapq=q, cigar=[(0, 100)]))
            tid.append(t), pos.append(p), flag.append(f), mapq.append(q)
        alns.extend(rec)
    res = ref_exec.run_reference_path(alns, lengths, sites, MIN_LEN, MIN_SIG, min_mapq=60, bin_size=BIN_SIZE)
    cm = res['cm']
    em = cm.extent_map.tocoo()
    out = dict(lengths=lengths.astype(np.int64), sites=sites.astype(np.int64), a_tid=np.array(tid, dtype=np.int32),
               a_pos=np.array(pos, dtype=np.int64), a_flag=np.array(flag, dtype=np.int32),
               a_mapq=np.array(mapq, dtype=np.int32), min_len=np.int64(MIN_LEN), min_sig=np.int64(MIN_SIG),
               bin_size=np.int64(BIN_SIZE), mask=np.asarray(res['mask']).astype(np.uint8),
               bins=np.asarray(cm.grouping.bins, dtype=np.int64),
               ext_row=em.row.astype(np.int64), ext_col=em.col.astype(np.int64), ext_data=em.data.astype(np.int64))
    print('mask', int(out['mask'].sum()), 'of', len(out['mask']))
    assert 0 < out['mask'].sum() < len(out['mask']), 'the mask must remove some, not all, sequences'
    for tag, kw in (('geo', dict(norm=True, bisto=False, mean_type='geometric')),
                    ('har', dict(norm=True, bisto=False, mean_type='harmonic')),
                    ('ari', dict(norm=True, bisto=False, mean_type='arithmetic')),
                    ('raw', dict(norm=False, bisto=False)),
                    ('geo_bisto', dict(norm=True, bisto=True, mean_type='geometric'))):
        m = cm.get_extent_map(**kw).tocoo()
        m.sum_duplicates()
        o = np.lexsort((m.col, m.row))
        out[tag + '_shape'] = np.array(m.shape, dtype=np.int64)
        out[tag + '_row'], out[tag + '_col'] = m.row[o].astype(np.int64), m.col[o].astype(np.int64)
        out[tag + '_data'] = m.data[o].astype(np.float64)
    # _norm_extent alone, on the uncompressed map (what get_extent_map does before compressing)
    m = cm._norm_extent(cm.extent_map.astype(float), 'geometric').tocoo()
    o = np.lexsort((m.col, m.row))
    out['normonly_row'], out['normonly_col'], out['normonly_data'] = m.row[o].astype(np.int64), m.col[o].astype(np.int64), \
        m.data[o].astype(np.float64)
    path = os.path.join(HERE, 'extentmap.npz')
    np.savez_compressed(path, **out)
    print('wrote', path, os.path.getsize(path), 'bytes; bins', int(out['bins'].sum()), 'extent nnz', em.nnz,
          'accepted', int(out['mask'].sum()), 'of', len(out['mask']), 'compressed shape', out['geo_shape'].tolist())


if __name__ == '__main__':
    main()
