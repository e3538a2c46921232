"""
Golden vectors of BASELINE config 1 at FULL size (10 genomes, 2,000 contigs, 1M Hi-C pairs, seed 1001), produced by
the reference's own code: SeqOrder / ContactMap / sparse_utils / cluster.to_graph exec'd verbatim under Python 3
(oracle/ref_exec.run_reference_path, as in make_golden_refpath.py), then nx.write_edgelist in the layout the pinned
Python 2.7 / networkx 1.11 produce (12 significant digits) and the reference's own Infomap binary with the flags of
cluster.py:182-185.  Nothing here comes from oracle/oracle.py.  The pair records are not stored: they are
synth.make_config('C1') (deterministic).  Run with a reference checkout (see oracle/ref_exec.py; ~15 s):
    python tests/golden/make_golden_c1.py
"""
import logging
import os
import subprocess
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
sys.path.insert(0, HERE)

from bin3c_b200 import synth          # noqa: E402
from oracle import oracle, ref_exec   # noqa: E402
import make_golden_refpath as mg      # noqa: E402

MIN_LEN, MIN_SIG = 1000, 5             # bin3C.py:27-34 runtime defaults
INFOMAP_FLAGS = ['-u', '-v', '-z', '-i', 'link-list', '-s', '1234', '-N', '10']


def infomap_partition(edge_file, work_dir):
    infomap = os.path.join(ref_exec.REFERENCE_ROOT, 'external', 'Infomap')
    subprocess.check_call([infomap] + INFOMAP_FLAGS + [edge_file, work_dir], stdout=subprocess.DEVNULL,
                          stderr=subprocess.STDOUT)
    base = os.path.splitext(os.path.basename(edge_file))[0]
    return oracle.read_tree(os.path.join(work_dir, base + '.tree'))


def partition_arrays(part):
    """list of node sets -> (node int64[], label int64[]) sorted by node, labels renumbered by smallest member."""
    groups = sorted((sorted(int(n) for n in nodes) for nodes in part), key=lambda g: g[0])
    node = np.array([n for g in groups for n in g], dtype=np.int64)
    label = np.array([k for k, g in enumerate(groups) for _ in g], dtype=np.int64)
    o = np.argsort(node)
    return node[o], label[o]


def main():
    com = synth.make_config('C1')
    lengths = np.full(com.n_refs, 500, dtype=np.int64)
    sites = np.ones(com.n_refs, dtype=np.int64)
    lengths[com.ref_index] = com.lengths
    sites[com.ref_index] = com.sites
    cap = ref_exec.IterCapture()
    logging.getLogger('mzd.sparse_utils').addHandler(cap)
    res = ref_exec.run_reference_path(mg.alignments_of(com.records), lengths, sites, MIN_LEN, MIN_SIG, min_mapq=60)
    logging.getLogger('mzd.sparse_utils').removeHandler(cap)
    g = res['graph']
    e = sorted((min(a, b), max(a, b), w) for a, b, w in g.edges(data='weight'))
    u = np.array([a for a, _, _ in e], dtype=np.int64)
    v = np.array([b for _, b, _ in e], dtype=np.int64)
    w = np.array([c for _, _, c in e], dtype=np.float64)
    with tempfile.TemporaryDirectory() as d:
        f = os.path.join(d, 'cm_graph.edges')
        with open(f, 'w') as fh:                                  # the reference's own layout (Python 2 str(float))
            fh.write(oracle.edge_lines(u, v, w, py2=True))
        node, label = partition_arrays(infomap_partition(f, d))
    sm = res['seq_map']
    c = res['counts']
    out = dict(counts=np.array([c['accepted'], c['ref_excluded'], c['poor_match']], dtype=np.int64),
               map_row=sm.row.astype(np.int32), map_col=sm.col.astype(np.int32), map_data=sm.data.astype(np.uint32),
               mask=np.asarray(res['mask']).astype(np.uint8), kr_x=np.asarray(res['bisto_scale'], dtype=np.float64),
               kr_n_iter=np.int64(cap.n_iter), edge_u=u.astype(np.int32), edge_v=v.astype(np.int32), edge_w=w,
               part_node=node, part_label=label, min_len=np.int64(MIN_LEN), min_sig=np.int64(MIN_SIG))
    path = os.path.join(HERE, 'c1full.npz')
    np.savez_compressed(path, **out)
    print('wrote', path, os.path.getsize(path), 'bytes; counts', c, 'nnz', sm.nnz, 'accepted contigs',
          int(out['mask'].sum()), 'kr iterations', cap.n_iter, 'edges', len(e), 'clusters', int(label.max()) + 1)


if __name__ == '__main__':
    main()
