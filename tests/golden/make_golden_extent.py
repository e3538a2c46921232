"""
Golden vectors for the extent map's bins: the reference's own ExtentGrouping class and find_nearest_jit, exec'd
verbatim from the reference's mzd/contact_map.py:50-62, 116-156 under Python 3 (oracle/ref_exec.load_extent: np.int
alias, tqdm stub, numba decorator dropped, and sequence lengths wrapped in an int whose `/` is Python 2's integer
division), on seeded random sequence lengths.  With a reference checkout (see oracle/ref_exec.py):  python tests/golden/make_golden_extent.py
"""
import os
import random
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from oracle import ref_exec          # noqa: E402


def main():
    make_grouping, find_nearest = ref_exec.load_extent()
    rng = random.Random(20240)
    lengths = [rng.choice([1, 96, 97, 145, 146, 299, 300, 999, 1000, 1499, 1500, 2499, 2500, 7777, 20000, 123457])
               for _ in range(150)] + [rng.randrange(1, 30000) for _ in range(150)]
    out = {'lengths': np.array(lengths, dtype=np.int64)}
    bin_sizes = [97, 333, 1000, 2500, 50000]
    out['bin_sizes'] = np.array(bin_sizes, dtype=np.int64)
    for bs in bin_sizes:
        g = make_grouping(lengths, bs)
        out['bins_%d' % bs] = np.asarray(g.bins, dtype=np.int64)
        out['upper_%d' % bs] = np.concatenate([np.asarray(m)[:, 0] for m in g.map]).astype(np.int64)
        out['binid_%d' % bs] = np.concatenate([np.asarray(m)[:, 1] for m in g.map]).astype(np.int64)
        q_seq, q_pos, q_bin = [], [], []
        for k in range(0, len(lengths), 5):
            for x in (0, 1, lengths[k] // 3, lengths[k] // 2, lengths[k] - 1, lengths[k], lengths[k] + 17):
                q_seq.append(k)
                q_pos.append(x)
                q_bin.append(int(find_nearest(np.asarray(g.map[k]), x)))
        out['q_seq_%d' % bs] = np.array(q_seq, dtype=np.int64)
        out['q_pos_%d' % bs] = np.array(q_pos, dtype=np.int64)
        out['q_bin_%d' % bs] = np.array(q_bin, dtype=np.int64)
    np.savez_compressed(os.path.join(HERE, 'extent.npz'), **out)
    print('wrote extent.npz:', {k: v.shape for k, v in out.items() if k.startswith('bins_')})


if __name__ == '__main__':
    main()
