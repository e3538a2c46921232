"""
BASELINE config 1 made real: the reference's OWN code (oracle/ref_exec.run_reference_path: SeqOrder, ContactMap,
sparse_utils and cluster.to_graph exec'd verbatim under Python 3) on the synthetic C1 community (10 genomes, 2,000
contigs, 1M Hi-C pairs), then nx.write_edgelist and the reference's Infomap binary with the reference's flags --
timed stage by stage on this machine's CPU, beside the vectorised port (oracle.run_path) and with the two partitions
compared.  Needs a reference checkout (see oracle/ref_exec.py); no GPU.
    python tools/reference_c1.py [--scale 1.0]
"""
import argparse
import json
import logging
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests', 'golden'))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--scale', type=float, default=1.0)
    args = ap.parse_args()
    import networkx as nx
    from bin3c_b200 import synth, bam_io
    from oracle import oracle, ref_exec
    import make_golden_refpath as mg
    com = synth.make_config('C1', scale=args.scale)
    lengths = np.full(com.n_refs, 500, dtype=np.int64)
    sites = np.ones(com.n_refs, dtype=np.int64)
    lengths[com.ref_index] = com.lengths
    sites[com.ref_index] = com.sites
    alns = mg.alignments_of(com.records)
    marks = []

    class Clock(logging.Handler):
        def emit(self, record):
            marks.append((time.perf_counter(), record.getMessage()[:60]))
    for name in ('mzd.contact_map.exec', 'mzd.cluster.exec', 'mzd.sparse_utils'):
        lg = logging.getLogger(name)
        lg.addHandler(Clock(level=logging.DEBUG))
        lg.setLevel(logging.DEBUG)
    t0 = time.perf_counter()
    res = ref_exec.run_reference_path(alns, lengths, sites, 1000, 5, min_mapq=60)
    t_path = time.perf_counter() - t0
    stages = {}
    prev = t0
    for t, msg in marks:
        stages[msg] = round(t - prev, 3)
        prev = t
    out = {'workload': 'C1: {} contigs, {} pairs (seed {})'.format(com.n_contigs, com.n_pairs, com.seed),
           'reference_path_s': round(t_path, 2), 'reference_pairs_per_s': round(com.n_pairs / t_path),
           'reference_log_marks_s': stages}
    with tempfile.TemporaryDirectory() as d:
        g = res['graph']
        f = os.path.join(d, 'cm_graph.edges')
        t0 = time.perf_counter()
        nx.write_edgelist(g, f, data=['weight'], delimiter=' ')
        out['nx_write_edgelist_s'] = round(time.perf_counter() - t0, 3)
        infomap = os.path.join(ref_exec.REFERENCE_ROOT, 'external', 'Infomap')
        t0 = time.perf_counter()
        subprocess.check_call([infomap, '-u', '-v', '-z', '-i', 'link-list', '-s', '1234', '-N', '10', f, d],
                              stdout=subprocess.DEVNULL, stderr=subprocess.STDOUT)
        out['infomap_s'] = round(time.perf_counter() - t0, 3)
        part_ref = oracle.read_tree(os.path.join(d, 'cm_graph.tree'))
        # the vectorised port and the native writer
        ti, tj, ok = synth.unpack_pairs(com.records)
        t0 = time.perf_counter()
        port = oracle.run_path(ti, tj, ok, com.tid2idx(), com.lengths, com.sites, min_len=1000, min_sig=5)
        out['port_path_s'] = round(time.perf_counter() - t0, 3)
        d2 = os.path.join(d, 'port')
        os.mkdir(d2)
        f2 = os.path.join(d2, 'cm_graph.edges')
        t0 = time.perf_counter()
        bam_io.write_edges(port['u'], port['v'], port['w'], f2)
        out['native_write_edges_s'] = round(time.perf_counter() - t0, 4)
        subprocess.check_call([infomap, '-u', '-v', '-z', '-i', 'link-list', '-s', '1234', '-N', '10', f2, d2],
                              stdout=subprocess.DEVNULL, stderr=subprocess.STDOUT)
        part_port = oracle.read_tree(os.path.join(d2, 'cm_graph.tree'))
    out['accepted_contigs'] = int(np.asarray(res['mask']).sum())
    out['edges'] = g.number_of_edges()
    out['clusters'] = len(part_ref)
    out['partition_identical'] = part_ref == part_port
    out['x_max_rel_diff'] = float(np.max(np.abs(res['bisto_scale'] - port['x']) / np.abs(port['x'])))
    print(json.dumps(out, indent=1))


if __name__ == '__main__':
    main()
