"""
Golden vectors for the pair loop: the reference's own ContactMap._bin_map (contact_map.py:602-809), exec'd verbatim
under Python 3 (oracle/ref_exec.run_bin_map) on a fake BAM of duck-typed alignment records, with the reference's own
Sparse2DAccumulator, ExtentGrouping and find_nearest_jit.  Three filter settings (MAPQ only, strong matcher,
min_insert), each with the contig map, the binned extent map and the pair counters.  The alignment stream is stored
as flat arrays so that tests can rebuild it (and write it as a real BAM file for the native reader).
With a reference checkout (see oracle/ref_exec.py):  python tests/golden/make_golden_binmap.py
"""
import os
import random
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from oracle import ref_exec          # noqa: E402

PARAMS = [dict(min_mapq=30), dict(min_mapq=30, strong=40), dict(min_mapq=20, min_insert=1500)]
BIN_SIZE = 1000
MIN_LEN = 1000


def make_alignments(rng, n_refs, lengths, n_templates):
    alns = []
    for t in range(n_templates):
        n_rec = 2 if rng.random() < 0.8 else rng.choice([1, 1, 3, 4])
        a = rng.randrange(n_refs)
        for k in range(n_rec):
            tid = a if rng.random() < 0.55 else rng.randrange(n_refs)
            flag = 0x1 | (0x40 if k % 2 == 0 else 0x80)
            if rng.random() < 0.5:
                flag |= 0x10
            if rng.random() < 0.6:
                flag |= 0x2
            if rng.random() < 0.06:
                flag |= rng.choice([0x4, 0x100, 0x800])
            if rng.random() < 0.05:
                cigar = []
                flag &= ~0x10                     # the reference cannot add alen = None to a position
            else:
                cigar = [(0, rng.randrange(1, 150))]
                if rng.random() < 0.3:
                    cigar = [(4, rng.randrange(1, 30))] + cigar
                if rng.random() < 0.3:
                    cigar = cigar + [(2, rng.randrange(1, 9)), (0, rng.randrange(1, 60))]
                if rng.random() < 0.3:
                    cigar = cigar + [(4, rng.randrange(1, 30))]
            alns.append(dict(name=t, flag=flag, tid=tid, pos=rng.randrange(0, lengths[tid]),
                             mapq=rng.choice([0, 10, 25, 40, 60, 60, 60]), cigar=cigar))
    return alns


def main():
    rng = random.Random(60211)
    n_refs = 120
    lengths = [rng.choice([400, 900, 1000, 1800, 2600, 9000, 30000]) for _ in range(n_refs)]
    alns = make_alignments(rng, n_refs, lengths, 12000)
    keep = np.array(lengths) >= MIN_LEN
    lut = np.where(keep, np.cumsum(keep) - 1, -1)
    idx = {t: int(i) for t, i in enumerate(lut) if i >= 0}
    kept = [l for l in lengths if l >= MIN_LEN]
    make_grouping, _ = ref_exec.load_extent()
    out = {'lengths': np.array(lengths, dtype=np.int64), 'min_len': np.int64(MIN_LEN), 'bin_size': np.int64(BIN_SIZE),
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
    for k, kw in enumerate(PARAMS):
        res = ref_exec.run_bin_map(named, lengths, idx, len(kept), grouping=make_grouping(kept, BIN_SIZE), **kw)
        out['p%d_min_mapq' % k] = np.int64(kw.get('min_mapq', 0))
        out['p%d_strong' % k] = np.int64(kw.get('strong') or 0)
        out['p%d_min_insert' % k] = np.int64(kw.get('min_insert') or 0)
        c = res['counts']
        out['p%d_counts' % k] = np.array([c['accepted'], c['ref_excluded'], c['poor_match'], c['short_insert']], dtype=np.int64)
        for nm in ('seq_map', 'extent_map'):
            m = res[nm]
            out['p%d_%s_row' % (k, nm)] = m.row.astype(np.int64)
            out['p%d_%s_col' % (k, nm)] = m.col.astype(np.int64)
            out['p%d_%s_data' % (k, nm)] = m.data.astype(np.int64)
            out['p%d_%s_n' % (k, nm)] = np.int64(m.shape[0])
        print(kw, c)
    np.savez_compressed(os.path.join(HERE, 'binmap.npz'), **out)
    print('wrote binmap.npz', os.path.getsize(os.path.join(HERE, 'binmap.npz')))


if __name__ == '__main__':
    main()
