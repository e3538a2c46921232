#!/usr/bin/env python
"""
bench.py -- the contact-map hot path on N B200s (one process per GPU).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config C1|C2|C3|C4]
                    [--dump-outputs DIR]

One "step" is one pass of the whole hot path over one batch of synthetic packed pair records:
accumulate -> acceptance mask -> site normalisation -> Knight-Ruiz balancing -> compressed, scaled edge list.

Workload.  The default at every N is BASELINE.json configs[2] (C3: 500 genomes, 250k contigs, 500M pairs -- the
config BASELINE quotes "at 1/2/4/8 B200"; it fits one GPU and its contact matrix, 0.9 GB, does not fit the L2, so the
roofline fraction is an HBM number).  N > 1 is STRONG scaling of that same community: every rank takes a contiguous
1/N of the pair stream, generated on the device (csrc/synth.cu; its NumPy mirror feeds the oracle).  At N = 1 the
line also carries `c2`, the same measurement on configs[1] (C2: 50k contigs, 50M pairs, L2-resident matrix), and
`kr_spmv_microbench` (configs[4] points).  Prints ONE JSON line (rank 0).

  value      pairs/s of the whole step with the records already resident in HBM (all ranks' pairs / max-rank time)
  e2e        the same step through the public API with the records in pinned HOST memory (narrow 5/6-byte records
             streamed through the staging ring) and the edge list read back to the host inside the timed region
  roofline   the dominant kernel's algorithmic bytes / its CUDA-event time against MEASURED_PEAKS.json
  cpu_baseline  the CPU oracle (NumPy/SciPy port of the reference path) on a bounded sample, rank 0
  parity     the CUDA path against that same oracle result, on the same sample (the whole config when it is <= 50M
             pairs), outside the timed region: contact matrix, counters, mask, edge structure bit-exact, n_iter equal,
             x and w max relative error; `digest` = order-independent checksums of the full-size result, equal
             for every N

--impl reference times the oracle port on the host cores (the reference itself is Python 2.7 and cannot run here;
see DESIGN.md), rank 0 only, on a bounded sample of the same config.
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = 'Hi-C pairs/sec into CSR; KR SpMV GB/s vs HBM peak at 1/2/4/8 B200'      # BASELINE.json:metric
METRIC_NOTE = 'value = pairs/s through the WHOLE hot path (accumulate -> mask -> KR -> edge list); accumulation alone ' \
              'is accumulate_pairs_per_s, KR SpMV GB/s is roofline.achieved / kr.spmv_gbs_by_formula'
UNIT = 'pairs/s'
DTYPE = 'u32 counts / f64 balancing'
MIN_LEN, MIN_SIG = 1000, 5           # bin3C.py:27-34 runtime defaults
CPU_SAMPLE_PAIRS = 50_000_000       # the whole of C2; a bounded prefix of the pair stream for larger configs
REL_TOL = 1e-9                      # north_star: KR scale vector and edge weights
DUMP_EDGES = 1_500_000              # --dump-outputs: u, v, w and their indices as float64 stay under 48 MB
DUMP_SEED = 1234


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--config', default=None, help='C1|C2|C3|C4 (default C3 at every N; C4 is meant for 8 GPUs)')
    ap.add_argument('--scale', type=float, default=1.0, help='shrink the pair count (debugging only)')
    ap.add_argument('--e2e-steps', type=int, default=None)
    ap.add_argument('--no-cpu-baseline', action='store_true', help='skip the CPU oracle leg (and with it the parity check)')
    ap.add_argument('--e2e-record-bytes', default='auto',
                    help="auto: the narrowest hand-over (same-reference pairs as 3/4-byte records, the rest as 5/6/8-byte "
                         "pair records); narrow: 5/6/8-byte pair records only; 8: native records")
    ap.add_argument('--no-microbench', action='store_true', help='skip the C5 KR SpMV microbench points')
    ap.add_argument('--microbench', default='default', choices=['default', 'full'], help='full: also the 3M-row C5 point')
    ap.add_argument('--no-c2', action='store_true', help='N=1: skip the secondary C2 measurement')
    ap.add_argument('--no-e2e', action='store_true')
    ap.add_argument('--parity', default='sample', choices=['sample', 'full', 'none'],
                    help='sample: oracle on the first 50M pairs; full: on the whole config (minutes and tens of GB at C3)')
    ap.add_argument('--weak', action='store_true', help='N>1: weak scaling (a full --config shard per rank) instead of strong')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='N=1: after the timed steps, write what the last timed step returned as DIR/<name>.npy '
                         '(float64; the edge list as a fixed, seeded sample when it is longer than {} edges)'.format(
                             DUMP_EDGES))
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    return args


def ncu_traffic(cfg, kernel):
    """DRAM bytes per launch of `kernel` from the committed ncu capture (profiles/traffic.json), or None."""
    try:
        with open(os.path.join(ROOT, 'profiles', 'traffic.json')) as fh:
            return int(json.load(fh)[cfg][kernel]['bytes'])
    except Exception:
        return None


def measured_peak():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    try:
        with open(path) as fh:
            return float(json.load(fh)['hbm_gbs']), 'measured (MEASURED_PEAKS.json)'
    except Exception:
        return 6650.0, 'fallback (B200_PROFILING.md)'


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons of one GPU while the timed region runs."""

    def __init__(self, index, period=0.02):
        threading.Thread.__init__(self, daemon=True)
        self.index, self.period = index, period
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop_ev = threading.Event()
        self._nv = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nv = pynvml
            self._h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self._nv = None

    def run(self):
        nv = self._nv
        if nv is None:
            return
        names = {
            'nvmlClocksEventReasonHwSlowdown': 'hw_slowdown',
            'nvmlClocksThrottleReasonHwSlowdown': 'hw_slowdown',
            'nvmlClocksEventReasonHwThermalSlowdown': 'hw_thermal_slowdown',
            'nvmlClocksThrottleReasonHwThermalSlowdown': 'hw_thermal_slowdown',
            'nvmlClocksEventReasonSwThermalSlowdown': 'sw_thermal_slowdown',
            'nvmlClocksThrottleReasonSwThermalSlowdown': 'sw_thermal_slowdown',
            'nvmlClocksEventReasonSwPowerCap': 'sw_power_cap',
            'nvmlClocksThrottleReasonSwPowerCap': 'sw_power_cap',
        }
        bits = {getattr(nv, k): v for k, v in names.items() if hasattr(nv, k)}
        get_reasons = getattr(nv, 'nvmlDeviceGetCurrentClocksEventReasons', None) or \
            getattr(nv, 'nvmlDeviceGetCurrentClocksThrottleReasons', None)
        while not self._stop_ev.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM))
                if get_reasons is not None:
                    r = get_reasons(self._h)
                    for b, nm in bits.items():
                        if r & b:
                            self.reasons.add(nm)
            except Exception:
                pass
            time.sleep(self.period)

    def stop(self):
        self._stop_ev.set()
        self.join(timeout=2)
        return {'sm_mhz': float(np.median(self.samples)) if self.samples else None,
                'sm_max_mhz': self.max_mhz, 'reasons': sorted(self.reasons), 'samples': len(self.samples)}


def cpu_threads():
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


# ---------------------------------------------------------------------------------------------------------------
# workloads
# ---------------------------------------------------------------------------------------------------------------

class Workload(object):
    """A BASELINE config made concrete: the community tables plus its pair stream (sequential host stream for C1 / C2,
    counter-based device stream for C3 / C4)."""

    def __init__(self, name, scale=1.0):
        from bin3c_b200 import synth
        self.name = name
        kw = dict(synth.CONFIGS[name])
        t0 = time.time()
        self.v2 = kw.get('stream') == 'v2'
        if self.v2:
            self.tab, self.stream, self.P = synth.make_stream(name, max(1, int(kw['n_pairs'] * scale)))
            self.com = self.tab.community(None)
        else:
            self.com = synth.make_config(name, scale=scale)
            self.tab, self.stream, self.P = None, None, self.com.n_pairs
        self.gen_s = time.time() - t0
        self.N, self.n_refs, self.seed = self.com.n_contigs, self.com.n_refs, kw['seed']
        self.n_genomes = kw['n_genomes']
        self.tid2idx, self.lengths, self.sites = self.com.tid2idx(), self.com.lengths, self.com.sites

    def describe(self):
        return '{}: {} genomes, {} contigs, {} pairs (seed {}{})'.format(
            self.name, self.n_genomes, self.N, self.P, self.seed, ', counter-based stream' if self.v2 else '')

    def device_records(self, first, count):
        from bin3c_b200 import device as dev
        if self.v2:
            return self.stream.device_records(first, count)
        return dev.to_device(self.com.records[first:first + count])

    def host_records(self, first, count):
        if self.v2:
            return self.stream.host_records(first, count)
        return self.com.records[first:first + count]


def cpu_oracle_run(work, n_pairs, records=None, threads=None):
    """One pass of the oracle port over the first n_pairs records (accumulation spread over the host threads; the
    SciPy/NumPy stages after it are single-threaded, as in the reference).  Returns (seconds, result dict)."""
    from bin3c_b200 import synth
    from oracle import oracle
    if records is None:
        records = work.host_records(0, n_pairs)
    t0 = time.perf_counter()
    ti, tj, ok = synth.unpack_pairs(records[:n_pairs])
    ref = oracle.run_path(ti, tj, ok, work.tid2idx, work.lengths, work.sites, min_len=MIN_LEN, min_sig=MIN_SIG,
                          threads=threads or cpu_threads())
    return time.perf_counter() - t0, ref


def run_reference(args, rank):
    """The reference arm: the CPU port of the reference path on the host cores, rank 0 only, on a bounded sample of
    the same config our arm runs at this N (strong scaling: the config does not depend on N)."""
    if rank != 0:
        return
    cfg = args.config or 'C3'
    work = Workload(cfg, min(1.0, args.scale))
    sample = int(min(work.P, CPU_SAMPLE_PAIRS))
    records = work.host_records(0, sample)
    for _ in range(args.warmup):
        cpu_oracle_run(work, sample, records)
    times = [cpu_oracle_run(work, sample, records)[0] for _ in range(max(args.steps, 1))]
    t = float(np.mean(times))
    val = sample / t
    line = {
        'impl': 'reference', 'metric': METRIC, 'metric_note': METRIC_NOTE, 'value': val, 'unit': UNIT,
        'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': t * 1e3,
        'higher_is_better': True, 'scaling': 'strong', 'vs_baseline': None, 'dtype': DTYPE, 'data': 'synthetic',
        'config': {'workload': work.describe()},
        'cpu_baseline': {'value': val, 'unit': UNIT, 'cores': cpu_threads(), 'kind': 'port',
                         'sample': 'each step = the first {} pairs of the workload ({} contigs), NumPy/SciPy port of the '
                                   'reference path; accumulation on {} threads, SciPy KR single-threaded; box has {} '
                                   'cores'.format(sample, work.N, cpu_threads(), os.cpu_count())},
        'e2e': {'value': val, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
    }
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------------------------
# checker side: parity against the oracle, digests of a full-size result (outside every timed region)
# ---------------------------------------------------------------------------------------------------------------

def _relerr(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    if a.shape != b.shape:
        return float('inf')
    if a.size == 0:
        return 0.0
    return float(np.max(np.abs(a - b) / np.maximum(np.abs(b), 1e-300)))


def parity_report(got, ref, sample, whole):
    """got: dict(row, col, data, counts[3], mask, n_iter, x, u, v, w) assembled from the CUDA path; ref: oracle.run_path."""
    sm = ref['seq_map']
    o = np.lexsort((got['col'], got['row']))
    rep = {
        'checked': True, 'against': 'oracle.run_path (NumPy/SciPy restatement pinned to the reference, DESIGN.md section 2)',
        'sample_pairs': int(sample), 'whole_config': bool(whole),
        'contact_matrix_exact': bool(len(o) == sm.nnz and np.array_equal(got['row'][o], sm.row) and
                                     np.array_equal(got['col'][o], sm.col) and
                                     np.array_equal(got['data'][o].astype(np.uint32), sm.data)),
        'counters_exact': [int(v) for v in got['counts']] == [ref['counts'][k] for k in
                                                              ('accepted', 'ref_excluded', 'poor_match')],
        'mask_exact': bool(np.array_equal(np.asarray(got['mask']).astype(bool), ref['mask'])),
        'n_iter': [int(got['n_iter']), int(ref['n_iter'])],
        'x_max_rel_err': _relerr(got['x'], ref['x']),
    }
    eo = np.lexsort((got['v'], got['u']))
    rep['edges_structure_exact'] = bool(len(eo) == len(ref['u']) and np.array_equal(got['u'][eo], ref['u']) and
                                        np.array_equal(got['v'][eo], ref['v']))
    rep['w_max_rel_err'] = _relerr(got['w'][eo], ref['w']) if rep['edges_structure_exact'] else float('inf')
    rep['tolerance'] = REL_TOL
    rep['ok'] = bool(rep['contact_matrix_exact'] and rep['counters_exact'] and rep['mask_exact'] and
                     rep['n_iter'][0] == rep['n_iter'][1] and rep['x_max_rel_err'] <= REL_TOL and
                     rep['edges_structure_exact'] and rep['w_max_rel_err'] <= REL_TOL)
    return rep


def _mix(torch, h):
    h = h * -7046029254386353131            # 0x9E3779B97F4A7C15 as int64 (wrapping arithmetic)
    h = h ^ (h >> 29)
    h = h * -4658895280553007687            # 0xBF58476D1CE4E5B9
    return h ^ (h >> 32)


def digest_block(torch, csr, mask, x, edges):
    """Order- and partition-independent 64-bit checksums of this rank's share of a result (wrapping sums of hashed
    entries: summing them over ranks gives the same number for every N)."""
    n_tot = int(csr.n_total)
    indptr = csr.indptr
    rows = torch.repeat_interleave(torch.arange(csr.n, device='cuda', dtype=torch.int64) + csr.row_lo,
                                   indptr[1:] - indptr[:-1])
    key = rows * n_tot + csr.indices.to(torch.int64)
    cnt = csr.data.to(torch.int64) & 0xffffffff
    d_map = int((_mix(torch, key) * (2 * cnt + 1)).sum())
    lo, hi = csr.row_lo, csr.row_lo + csr.n
    m = mask[lo:hi].to(torch.int64)
    d_mask = int((_mix(torch, torch.arange(lo, hi, device='cuda', dtype=torch.int64)) * m).sum())
    n_e = int(edges['n_edges'])
    ek = edges['u'][:n_e].to(torch.int64) * n_tot + edges['v'][:n_e].to(torch.int64)
    d_edges = int(_mix(torch, ek).sum())
    return dict(map=d_map, mask=d_mask, edges=d_edges, weight=int(cnt.sum()), x_sum=float(x[lo:hi].sum()),
                w_sum=float(edges['w'][:n_e].sum()), n_edges=n_e, nnz=int(csr.nnz))


def _wrap64(v):
    return int(v) & 0xffffffffffffffff


def dump_outputs(out_dir, res):
    """Write the edge result HotPath.run returned (the views are overwritten by the next run, so call this before it)
    as out_dir/<name>.npy, all float64 (the int32 ids are exact in it).  An edge list longer than DUMP_EDGES is written
    as the same seeded sample of positions on every run, with those positions in edge_index.npy."""
    n = int(res['n_edges'])
    out = {k: np.array([res[k]], dtype=np.float64) for k in ('n_accepted', 'n_kept', 'n_edges')}
    out['scl'] = res['scl'][:1].cpu().numpy().astype(np.float64)
    out['newidx'] = res['newidx'].cpu().numpy().astype(np.float64)
    idx = np.arange(n) if n <= DUMP_EDGES else np.sort(np.random.default_rng(DUMP_SEED).choice(n, DUMP_EDGES,
                                                                                               replace=False))
    for k in ('u', 'v', 'w'):
        out[k] = res[k][:n].cpu().numpy()[idx].astype(np.float64)
    out['edge_index'] = idx.astype(np.float64)
    total = sum(a.nbytes for a in out.values())
    assert total <= 64 << 20, 'outputs to dump take {} B'.format(total)
    os.makedirs(out_dir, exist_ok=True)
    for k, a in out.items():
        np.save(os.path.join(out_dir, k + '.npy'), a)


# ---------------------------------------------------------------------------------------------------------------
# N = 1
# ---------------------------------------------------------------------------------------------------------------

def spmv_point(dev, torch, peak, rows, nnz, reps=20, seed=1005, compare=True):
    """One BASELINE config 5 point: the KR SpMV kernel alone on a random block-structured symmetric CSR that does not
    fit in L2, GB/s by SURVEY 8d's 12*nnz + 24*N formula against the measured HBM peak; the same product with SciPy's
    single-threaded csr_matvec (what kr_biostochastic calls, sparse_utils.py:136) beside it."""
    from bin3c_b200 import synth
    indptr, indices, data = synth.make_block_csr(rows, nnz, seed=seed)
    csr = dev.DeviceCSR(rows, dev.to_device(indptr), dev.to_device(indices), dev.to_device(data))
    u = dev.to_device(np.random.default_rng(0).uniform(0.5, 1.5, csr.n))
    ws = torch.empty(dev.lib.b3c_kr_workspace_bytes(csr.n, csr.nnz), dtype=torch.uint8, device='cuda')
    y = dev.spmv(csr, u, ws=ws, prepared=False)
    for _ in range(3):
        dev.spmv(csr, u, y=y, ws=ws, prepared=True)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        dev.spmv(csr, u, y=y, ws=ws, prepared=True)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    nbytes = 12 * csr.nnz + 24 * csr.n
    out = {'workload': 'C5 point: block-structured symmetric CSR, {} rows, {} nnz (seed {}), {} MB by formula'.format(
               csr.n, csr.nnz, seed, nbytes // 1000000),
           'kernels': 'k_spmv + k_spmv_collect (the SpMV phase of k_kr_persistent as a stand-alone launch)',
           'ms_per_spmv': ms, 'gbs': nbytes / ms / 1e6, 'peak': peak, 'frac': nbytes / ms / 1e6 / peak, 'reps': reps}
    if compare:
        import scipy.sparse as sp
        m_host = sp.csr_matrix((data, indices, indptr), shape=(rows, rows))
        u_host = np.random.default_rng(0).uniform(0.5, 1.5, rows)
        m_host.dot(u_host)
        t0 = time.perf_counter()
        for _ in range(3):
            y_host = m_host.dot(u_host)
        scipy_ms = (time.perf_counter() - t0) / 3 * 1e3
        err = float(np.max(np.abs(y.cpu().numpy() - y_host)) / np.max(np.abs(y_host)))
        assert err < 1e-12, 'SpMV differs from SciPy: {}'.format(err)
        out.update({'scipy_csr_matvec_ms': scipy_ms, 'speedup_vs_scipy_1_core': scipy_ms / ms, 'max_rel_diff_vs_scipy': err})
    return out


def run_single_gpu(work, args, torch, dev, local_rank, steps, warmup, want_cpu, parity_mode, dump_dir=None):
    """Everything measured on one config on one GPU; returns the fields of a bench line.  With dump_dir, what the last
    timed step returned is written there (dump_outputs)."""
    from bin3c_b200 import bam_io
    from bin3c_b200.pipeline import HotPath
    P, N = work.P, work.N
    rec_dev = work.device_records(0, P)
    torch.cuda.synchronize()
    # key capacity: only off-diagonal accepted pairs become keys (~17 % of the synthetic streams); beyond 600M pairs
    # the buffers are sized for 30 % of them (an overflow is reported as B3C_ERR_CAPACITY, never silently)
    hp = HotPath(work.tid2idx, work.lengths, work.sites, min_len=MIN_LEN, min_sig=MIN_SIG,
                 pair_capacity=P if P <= 600_000_000 else int(0.3 * P))

    # ---- device-resident arm -----------------------------------------------------------------------
    for _ in range(warmup):
        hp.run(rec_dev)
    torch.cuda.synchronize()
    sampler = ClockSampler(local_rank)
    sampler.start()
    hp.enable_events(True)
    stage_acc, host_acc = {}, {}
    launches0 = dev.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    ev0.record()
    per_step_events = []
    kr_kernel_us = 0.0
    for _ in range(steps):
        res = hp.run(rec_dev)
        per_step_events.append(hp.events)
        kr_kernel_us += hp.kr_info['kernel_us']            # CUDA events around the persistent kernel's launch
    ev1.record()
    torch.cuda.synchronize()
    launches = dev.launch_count() - launches0
    total_ms = ev0.elapsed_time(ev1)
    for evs in per_step_events:
        hp.events = evs
        for k, v in hp.stage_ms().items():
            stage_acc[k] = stage_acc.get(k, 0.0) + v
        for k, v in hp.stage_host_ms().items():
            host_acc[k] = host_acc.get(k, 0.0) + v
    stage_ms = {k: v / steps for k, v in stage_acc.items()}
    hp.enable_events(False)
    ms_per_step = total_ms / steps
    value = P / (ms_per_step * 1e-3)
    info, kr = hp.acc_info, hp.kr_info
    nnz_full = info['nnz_full']
    n_edges = int(res['n_edges'])
    dg = digest_block(torch, hp.seq_map, hp.mask, hp.x, res)
    digest = {'map': _wrap64(dg['map']), 'mask': _wrap64(dg['mask']), 'edges': _wrap64(dg['edges']),
              'map_weight': dg['weight'], 'nnz_full': dg['nnz'], 'n_edges': dg['n_edges'], 'n_iter': kr['n_iter'],
              'x_sum': dg['x_sum'], 'w_sum': dg['w_sum']}
    if dump_dir:
        dump_outputs(dump_dir, res)

    # ---- end-to-end arm: pinned host records in, host edge list out ------------------------------------
    # The records cross PCIe in the narrowest layout the reference table allows: the pairs whose mates lie on one
    # reference (four in five) as 3-byte records, the rest as 5-byte pair records (6 / 8 for larger tables) -- what
    # the BAM reader hands over for the bulk path (bam_io.split_records / b3c_records_split).  Packing is the
    # producer's job and is not timed, like the BAM decode; the map does not depend on the order of its records.
    e2e = None
    clocks = None
    if not args.no_e2e:
        e2e_steps = args.e2e_steps or max(3, min(steps, 10))
        rec_bytes = 8 if args.e2e_record_bytes == '8' else bam_io.records_bytes(work.n_refs)
        host64 = rec_dev.cpu().numpy().view(np.uint64) if work.v2 else work.com.records
        rec_desc = rec_bytes
        if args.e2e_record_bytes == 'auto':
            e2e_in, e2e_kw = bam_io.split_records(host64, work.n_refs, pin=True), {}
            rec_desc = {'same_reference': e2e_in.bytes_same, 'pair': e2e_in.bytes_pair, 'n_same': e2e_in.n_same,
                        'n_pair': e2e_in.n_pairs, 'mean': round(e2e_in.nbytes / float(P), 3)}
        elif rec_bytes == 8:
            e2e_in, e2e_kw = torch.from_numpy(host64.view(np.int64)).pin_memory(), {}
        else:
            nb = (P * rec_bytes + 7) // 8 * 8
            e2e_in = torch.empty(nb, dtype=torch.uint8, pin_memory=True)
            bam_io.pack_records(host64, rec_bytes, out=e2e_in.numpy())
            e2e_kw = {'record_bytes': rec_bytes, 'n_records': P}
        if work.v2:
            del host64
        out = hp.run(e2e_in, to_host=True, **e2e_kw)
        assert out['n_edges'] == n_edges, 'end-to-end arm disagrees with the device-resident arm'
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            out = hp.run(e2e_in, to_host=True, **e2e_kw)
        torch.cuda.synchronize()
        e2e_s = (time.perf_counter() - t0) / e2e_steps
        e2e = {'value': P / e2e_s, 'unit': UNIT, 'h2d_bytes_per_step': int(hp.h2d_bytes),
               'd2h_bytes_per_step': int(hp.d2h_bytes), 'ms_per_step': e2e_s * 1e3, 'steps': e2e_steps,
               'record_bytes': rec_desc}
        del e2e_in
    clocks = sampler.stop()

    # ---- roofline of the dominant kernel -----------------------------------------------------------------
    peak, peak_src = measured_peak()
    t_cls = stage_ms.get('classify', 0.0)
    t_acc = t_cls + stage_ms.get('sort_reduce_emit', 0.0)
    t_kr = kr_kernel_us / steps * 1e-3                  # ms per launch of k_kr_persistent (the 'kr' stage adds its set-up)
    spmv_bytes = 12 * nnz_full + 24 * N                 # fp64 value + int32 column, int64 indptr, x read, y written
    kr_bytes = kr['n_spmv'] * spmv_bytes
    cls_bytes = 8 * P
    l2_note = 'matrix {} MB vs 126 MB L2: {}'.format(spmv_bytes // 1000000,
                                                     'HBM-bound' if spmv_bytes > 2 * 126e6 else 'L2-resident, NOT an HBM measurement')
    roof_kr = {'kernel': 'k_kr_persistent', 'bound': 'hbm', 'achieved': kr_bytes / (t_kr * 1e-3) / 1e9, 'peak': peak,
               'unit': 'GB/s', 'frac': kr_bytes / (t_kr * 1e-3) / 1e9 / peak, 'traffic': None, 'peak_source': peak_src,
               'bytes_per_launch': kr_bytes, 'ms_per_launch': t_kr,
               'note': '{} SpMV x (12*nnz + 24*N) B per launch (SURVEY 8d formula: what a CSR SpMV has to move; the kernel '
                       'streams {} B per entry, see streamed_gbs), vector phases and grid barriers are inside the launch '
                       'but add no counted bytes; {}'.format(kr['n_spmv'], kr.get('stream_bytes_per_entry', 0), l2_note)}
    # what the kernel's own operand stream amounts to (entries incl. padding x bytes per entry + the vectors), per launch
    streamed = kr['n_spmv'] * (kr['nnz_stream'] * kr.get('stream_bytes_per_entry', 0) + 24 * N)
    roof_kr['streamed_bytes_per_launch'] = streamed
    roof_kr['streamed_gbs'] = streamed / (t_kr * 1e-3) / 1e9
    roof_cls = {'kernel': 'k_classify', 'bound': 'hbm', 'achieved': cls_bytes / (t_cls * 1e-3) / 1e9, 'peak': peak,
                'unit': 'GB/s', 'frac': cls_bytes / (t_cls * 1e-3) / 1e9 / peak, 'traffic': None,
                'peak_source': peak_src, 'bytes_per_launch': cls_bytes, 'ms_per_launch': t_cls,
                'note': '8 B per packed pair record read once'}
    if args.scale == 1.0:
        roof_kr['traffic'] = ncu_traffic(work.name, 'k_kr_persistent')
        roof_cls['traffic'] = ncu_traffic(work.name, 'k_classify')
    for r in (roof_kr, roof_cls):
        # SURVEY 8d: "report fraction of both" -- the measured copy peak above and the north-star's nominal 8 TB/s;
        # and what the DRAM counters of the committed ncu capture amount to over the live launch time
        r['frac_of_nominal_8000'] = r['achieved'] / 8000.0
        if r['traffic']:
            r['traffic_gbs'] = r['traffic'] / (r['ms_per_launch'] * 1e-3) / 1e9
            r['traffic_frac'] = r['traffic_gbs'] / peak
    roofline, other = (roof_kr, roof_cls) if t_kr >= t_cls else (roof_cls, roof_kr)
    # accumulation against SURVEY 8d's strict bound: read every record once, write the upper-triangle CSR once
    key_bits = 2 * max(1, int(np.ceil(np.log2(max(N, 2)))))
    acc_bytes = 8 * P + 8 * info['nnz_upper'] + 8 * (N + 1)
    accumulation = {'pairs_per_s': P / (t_acc * 1e-3), 'ms': t_acc, 'strict_bytes': acc_bytes,
                    'strict_gbs': acc_bytes / (t_acc * 1e-3) / 1e9, 'strict_frac': acc_bytes / (t_acc * 1e-3) / 1e9 / peak,
                    'key_bits': key_bits, 'radix_passes': '{} (keys) + {} (mirror, column bits), digits of up to 9 bits'.format(
                        -(-key_bits // 9), -(-(key_bits // 2) // 9)),
                    'note': 'B_acc = 8 P + 8 nnz_upper + 8 (N + 1) (SURVEY 8d); only the off-diagonal ~20 % of the pairs '
                            'reach the sort'}

    # ---- CPU baseline on a bounded sample, and parity of the CUDA path against its result ------------------------
    cpu = parity = None
    if want_cpu:
        sample = P if parity_mode == 'full' else min(P, CPU_SAMPLE_PAIRS)
        records = rec_dev[:sample].cpu().numpy().view(np.uint64) if work.v2 else work.com.records[:sample]
        t, ref = cpu_oracle_run(work, sample, records)
        del records
        cpu = {'value': sample / t, 'unit': UNIT, 'cores': cpu_threads(), 'kind': 'port',
               'sample': 'first {} pairs of the workload, one pass, {:.1f} s, NumPy/SciPy port; accumulation on {} '
                         'threads, SciPy KR single-threaded; box has {} cores'.format(sample, t, cpu_threads(),
                                                                                     os.cpu_count())}
        if parity_mode != 'none':
            r = hp.run(rec_dev[:sample])
            ne = int(r['n_edges'])
            coo = hp.seq_map.to_scipy_coo()
            got = dict(row=coo.row, col=coo.col, data=coo.data,
                       counts=[hp.acc_info[k] for k in ('accepted', 'ref_excluded', 'poor_match')],
                       mask=hp.mask.cpu().numpy(), n_iter=hp.kr_info['n_iter'], x=hp.x.cpu().numpy(),
                       u=r['u'][:ne].cpu().numpy(), v=r['v'][:ne].cpu().numpy(), w=r['w'][:ne].cpu().numpy())
            parity = parity_report(got, ref, sample, sample == P)
        del ref

    sm_mhz = (clocks or {}).get('sm_mhz') or 1965.0
    return {
        'value': value, 'ms_per_step': ms_per_step,
        'config': {'workload': work.describe(),
                   'l2': 'input records {} MB > 126 MB L2, no explicit flush'.format(8 * P // 1000000),
                   'nnz_full': nnz_full, 'nnz_upper': info['nnz_upper'], 'accepted_contigs': int(res['n_accepted']),
                   'edges': n_edges, 'min_len': MIN_LEN, 'min_sig': MIN_SIG, 'generator_s': round(work.gen_s, 1)},
        'clocks': clocks, 'e2e': e2e, 'gpu_launches': int(launches),
        'roofline': roofline, 'roofline_other': other, 'accumulation': accumulation, 'cpu_baseline': cpu,
        'parity': parity, 'digest': digest,
        'stages_ms': {k: round(v, 4) for k, v in stage_ms.items()},
        'stages_host_ms': {k: round(v / steps, 4) for k, v in host_acc.items()},
        'kr_phase_us': {'clock_mhz': sm_mhz,
                        'work': {k: round(v / sm_mhz, 1) for k, v in kr['work_cycles'].items()},
                        'sync': {k: round(v / sm_mhz, 1) for k, v in kr['sync_cycles'].items()},
                        'total': round(kr['cycles'] / sm_mhz, 1), 'grid': kr['grid']},
        'accumulate_pairs_per_s': P / (t_acc * 1e-3),
        'kr': {'n_iter': kr['n_iter'], 'n_spmv': kr['n_spmv'], 'outer': kr['outer'], 'zero_diag': kr['zero_diag'],
               'spmv_gbs_by_formula': roof_kr['achieved'], 'kernel_ms': t_kr, 'stage_ms': stage_ms.get('kr'),
               'slabs': kr['slabs'], 'stream_entries': kr['nnz_stream'], 'segments': kr['segments'],
               'stream_bytes_per_entry': kr.get('stream_bytes_per_entry'),
               'spmv_phase_gbs': (spmv_bytes * kr['n_spmv'] / 1e9) /
                                 max((kr['work_cycles']['spmv'] + kr['sync_cycles']['spmv']) / (sm_mhz * 1e6), 1e-12)},
        'pair_counts': {k: info[k] for k in ('accepted', 'ref_excluded', 'poor_match')},
    }


def main_single(args, local_rank):
    import torch
    from bin3c_b200 import device as dev
    cfg = args.config or 'C3'
    work = Workload(cfg, args.scale)
    want_cpu = not args.no_cpu_baseline
    head = run_single_gpu(work, args, torch, dev, local_rank, args.steps, args.warmup, want_cpu, args.parity,
                          dump_dir=args.dump_outputs)
    del work
    torch.cuda.empty_cache()
    line = {'metric': METRIC, 'metric_note': METRIC_NOTE, 'value': head.pop('value'), 'unit': UNIT, 'n_gpus': 1,
            'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': head.pop('ms_per_step'),
            'higher_is_better': True, 'scaling': 'strong', 'vs_baseline': None, 'dtype': DTYPE, 'data': 'synthetic'}
    line.update(head)
    if args.config is None and not args.no_c2 and args.scale == 1.0:
        # BASELINE configs[1] beside the headline: 50k contigs / 50M pairs, the whole config checked against the oracle
        c2 = run_single_gpu(Workload('C2'), args, torch, dev, local_rank, args.steps, args.warmup, want_cpu,
                            'sample' if args.parity != 'none' else 'none')
        c2.pop('clocks', None)
        line['c2'] = c2
        torch.cuda.empty_cache()
    if not args.no_microbench and args.scale == 1.0:
        # BASELINE config 5 points (fp64 CSR in, b3c_spmv): 250k rows keep the slab form (shared-memory gathers);
        # 1M and 3M rows are wider than 16 column slabs with sparse (row, slab) cells and take the gather form
        peak, _ = measured_peak()
        pts = [(250_000, 100_000_000, True), (1_000_000, 100_000_000, False), (1_000_000, 300_000_000, False)]
        if args.microbench == 'full':
            pts.append((3_000_000, 300_000_000, False))
        line['kr_spmv_microbench'] = []
        for rows, nnz, compare in pts:
            line['kr_spmv_microbench'].append(spmv_point(dev, torch, peak, rows, nnz, compare=compare))
            torch.cuda.empty_cache()
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------------------------
# N > 1: strong scaling of the same config (one process per GPU, launched by torchrun)
# ---------------------------------------------------------------------------------------------------------------

def main_multi(args, rank, local_rank, world):
    import torch
    from bin3c_b200 import device as dev, bam_io
    from bin3c_b200.dist import ShardedHotPath, Comm
    cfg = args.config or 'C3'
    work = Workload(cfg, args.scale)
    comm = Comm()
    P, N = work.P, work.N
    if args.weak:
        first, pairs_local, total_pairs = rank * P, P, P * world
    else:
        cuts = [(P * g // world) // 2 * 2 for g in range(world)] + [P]       # even starts: 16-byte aligned slices
        first, pairs_local, total_pairs = cuts[rank], cuts[rank + 1] - cuts[rank], P
    rec_dev = work.device_records(first, pairs_local) if work.v2 or not args.weak else \
        dev.to_device(work.com.records)
    torch.cuda.synchronize()
    # key capacity per rank: its own off-diagonal keys, and the directed keys routed to it (both directions of every
    # key of its row block; the blocks are balanced by entries, so about 2 x total keys / world, with head-room)
    per_rank_max = max(pairs_local, 2 * total_pairs // world)
    cap = int(0.6 * per_rank_max) + (1 << 20)
    hp = ShardedHotPath(work.tid2idx, work.lengths, work.sites, pair_capacity=cap, min_len=MIN_LEN, min_sig=MIN_SIG,
                        comm=comm)

    def sync():
        torch.cuda.synchronize()
        comm.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        hp.run(rec_dev)
    sync()
    sampler = ClockSampler(local_rank)
    sampler.start()
    launches0 = dev.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sync()
    e0.record()
    for _ in range(args.steps):
        res = hp.run(rec_dev)
    e1.record()
    sync()
    ms = torch.tensor([e0.elapsed_time(e1) / args.steps], dtype=torch.float64, device='cuda')
    comm.all_reduce(ms, 'max')
    launches = dev.launch_count() - launches0
    kr = dict(hp.kr_info)
    splits = [int(v) for v in hp.info['splits']]
    counters = {k: hp.info[k] for k in ('accepted', 'ref_excluded', 'poor_match')}

    # ---- per-stage times from a common start: a device-side barrier over all ranks precedes every stage, so a
    # stage's time no longer contains the skew its predecessors left (max and mean over ranks) ---------------------
    names = ('accumulate', 'mask', 'kr', 'edges')
    acc_t = torch.zeros(len(names), dtype=torch.float64, device='cuda')
    n_st = max(2, min(args.steps, 5))
    sub_acc = {}
    if hasattr(hp.engine, 'substep_ms'):
        hp.engine.events = []
    for _ in range(n_st):
        marks = []
        for fn in (lambda: hp.accumulate(rec_dev), hp.compute_mask, hp.balance, hp.edges):
            hp.stage_barrier()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            marks.append((a, b))
        torch.cuda.synchronize()
        acc_t += torch.tensor([a.elapsed_time(b) for a, b in marks], dtype=torch.float64, device='cuda')
        if hasattr(hp.engine, 'substep_ms'):
            for k, v in hp.engine.substep_ms().items():
                sub_acc[k] = sub_acc.get(k, 0.0) + v / n_st
    if hasattr(hp.engine, 'substep_ms'):
        hp.engine.events = None
    sub_names = ('classify', 'publish', 'barrier1', 'route', 'barrier2', 'sort_reduce', 'emit')
    sub_t = torch.tensor([sub_acc.get(k, 0.0) for k in sub_names], dtype=torch.float64, device='cuda')
    sub_max = sub_t.clone()
    comm.all_reduce(sub_max, 'max')
    acc_t /= n_st
    st_max, st_sum = acc_t.clone(), acc_t.clone()
    comm.all_reduce(st_max, 'max')
    comm.all_reduce(st_sum, 'sum')
    krk = torch.tensor([float(hp.kr_info.get('kernel_us') or 0)], dtype=torch.float64, device='cuda')
    krk_max = krk.clone()
    comm.all_reduce(krk_max, 'max')
    res = hp.edge_res
    dg = digest_block(torch, hp.block, hp.mask, hp.x, res) if hp.block is not None else \
        dict(map=0, mask=0, edges=0, weight=0, x_sum=0.0, w_sum=0.0, n_edges=0, nnz=0)
    di = torch.tensor([dg['map'], dg['mask'], dg['edges'], dg['weight'], dg['nnz'], dg['n_edges'], pairs_local],
                      dtype=torch.int64, device='cuda')
    comm.all_reduce(di, 'sum')
    df = torch.tensor([dg['x_sum'], dg['w_sum']], dtype=torch.float64, device='cuda')
    comm.all_reduce(df, 'sum')

    # ---- end to end: this rank's records start in pinned HOST memory (narrow records through the staging ring),
    # its edge list ends on the host ---------------------------------------------------------------------------------
    e2e = None
    if not args.no_e2e:
        rec_bytes = 8 if args.e2e_record_bytes == '8' else bam_io.records_bytes(work.n_refs)
        host64 = rec_dev.cpu().numpy().view(np.uint64)
        rec_desc, run_kw = rec_bytes, {'record_bytes': rec_bytes, 'n_records': pairs_local}
        if args.e2e_record_bytes == 'auto':
            e2e_in, run_kw = bam_io.split_records(host64, work.n_refs, pin=True), {}
            rec_desc = {'same_reference': e2e_in.bytes_same, 'pair': e2e_in.bytes_pair}
        elif rec_bytes == 8:
            e2e_in = torch.from_numpy(host64.view(np.int64)).pin_memory()
        else:
            nb = (pairs_local * rec_bytes + 7) // 8 * 8
            e2e_in = torch.empty(nb, dtype=torch.uint8, pin_memory=True)
            bam_io.pack_records(host64, rec_bytes, out=e2e_in.numpy())
        del host64
        e2e_steps = args.e2e_steps or max(3, min(args.steps, 10))
        pinned = {}

        def e2e_step():
            r = hp.run(e2e_in, **run_kw)
            n = int(r['n_edges'])
            nbytes = 0
            for k, m in (('u', n), ('v', n), ('w', n), ('scl', 1)):
                h = pinned.get(k)
                if h is None or h.numel() < m:
                    h = pinned[k] = torch.empty(m + m // 4 + 16, dtype=r[k].dtype, pin_memory=True)
                h[:m].copy_(r[k][:m], non_blocking=True)
                nbytes += m * h.element_size()
            torch.cuda.current_stream().synchronize()
            return nbytes

        d2h = e2e_step()
        sync()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            d2h = e2e_step()
        sync()
        e2e_t = torch.tensor([(time.perf_counter() - t0) / e2e_steps], dtype=torch.float64, device='cuda')
        comm.all_reduce(e2e_t, 'max')
        io_t = torch.tensor([d2h, hp.h2d_bytes], dtype=torch.int64, device='cuda')
        comm.all_reduce(io_t, 'sum')
        e2e = {'value': total_pairs / float(e2e_t.cpu()[0]), 'unit': UNIT, 'h2d_bytes_per_step': int(io_t.cpu()[1]),
               'd2h_bytes_per_step': int(io_t.cpu()[0]), 'ms_per_step': float(e2e_t.cpu()[0]) * 1e3, 'steps': e2e_steps,
               'record_bytes': rec_desc}
        del e2e_in
    clocks = sampler.stop()

    # ---- parity: the sharded CUDA path on a bounded prefix of the stream (every rank takes 1/N of it) against the
    # oracle on rank 0; the CPU baseline is the oracle's time on that same sample ------------------------------------
    cpu = parity = None
    if not args.no_cpu_baseline and args.parity != 'none':
        sample = total_pairs if args.parity == 'full' else min(total_pairs, CPU_SAMPLE_PAIRS)
        cuts_s = [(sample * g // world) // 2 * 2 for g in range(world)] + [sample]
        lo, hi = cuts_s[rank], cuts_s[rank + 1]
        if args.weak:
            srec = work.device_records(lo, hi - lo)     # weak scaling draws rank-local streams; the check uses the head
        elif lo >= first and hi <= first + pairs_local:
            srec = rec_dev[lo - first:hi - first]
        else:
            srec = work.device_records(lo, hi - lo)
        r = hp.run(srec)
        torch.cuda.synchronize()
        part = None
        if hp.block is not None:
            indptr, indices, data = hp.block.host_arrays()
            ne = int(r['n_edges'])
            part = dict(row=(np.repeat(np.arange(hp.block.n), np.diff(indptr)) + hp.row_lo).astype(np.int32), col=indices,
                        data=data, u=r['u'][:ne].cpu().numpy(), v=r['v'][:ne].cpu().numpy(), w=r['w'][:ne].cpu().numpy())
        common = dict(counts=[hp.info[k] for k in ('accepted', 'ref_excluded', 'poor_match')],
                      mask=hp.mask.cpu().numpy().copy(), n_iter=hp.kr_info['n_iter'], x=hp.x.cpu().numpy().copy())
        parts = comm.gather_object((part, common))
        if rank == 0:
            t, ref = cpu_oracle_run(work, sample, work.host_records(0, sample) if not work.v2 else None)
            cpu = {'value': sample / t, 'unit': UNIT, 'cores': cpu_threads(), 'kind': 'port',
                   'sample': 'first {} pairs of the workload, one pass, {:.1f} s, NumPy/SciPy port; accumulation on {} '
                             'threads, SciPy KR single-threaded; box has {} cores'.format(sample, t, cpu_threads(),
                                                                                         os.cpu_count())}
            blocks = [p for p, _ in parts if p is not None]
            got = {k: np.concatenate([b[k] for b in blocks]) for k in ('row', 'col', 'data', 'u', 'v', 'w')}
            got.update(parts[0][1])
            parity = parity_report(got, ref, sample, sample == total_pairs)
            # every rank must hold the same mask, x and iteration count
            parity['ranks_agree'] = bool(all(np.array_equal(c['mask'], parts[0][1]['mask']) and
                                             np.array_equal(c['x'], parts[0][1]['x']) and
                                             c['n_iter'] == parts[0][1]['n_iter'] and c['counts'] == parts[0][1]['counts']
                                             for _, c in parts))
            parity['ok'] = bool(parity['ok'] and parity['ranks_agree'])
            parity['n_ranks'] = world
        comm.barrier()
    if rank != 0:
        return
    ms_per_step = float(ms.cpu()[0])
    di = [int(v) for v in di.cpu()]
    peak, peak_src = measured_peak()
    # rank 0's launch of the persistent KR kernel over its row block: every SpMV streams the block's entries and reads
    # the whole exchanged vector u
    blk = hp.block
    kr_bytes = kr['n_spmv'] * (12 * int(blk.nnz) + 16 * int(blk.n) + 8 * hp.n) if blk is not None else 0
    kr_s = (kr.get('kernel_us') or 0) * 1e-6
    ach = kr_bytes / kr_s / 1e9 if kr_s > 0 else None
    roofline = {'kernel': 'k_kr_persistent (peer mode, rank 0 row block)', 'bound': 'hbm', 'achieved': ach, 'peak': peak,
                'unit': 'GB/s', 'frac': ach / peak if ach else None, 'traffic': None, 'peak_source': peak_src,
                'bytes_per_launch': kr_bytes, 'ms_per_launch': kr_s * 1e3,
                'note': '{} SpMV x (12*nnz_block + 16*rows_block + 8*N) B; the launch also contains the vector phases and '
                        'the NVLink hand-overs; kernel time from CUDA events around the launch'.format(kr['n_spmv'])}
    line = {
        'metric': METRIC, 'metric_note': METRIC_NOTE, 'value': total_pairs / (ms_per_step * 1e-3), 'unit': UNIT,
        'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': ms_per_step,
        'higher_is_better': True, 'scaling': 'weak' if args.weak else 'strong', 'vs_baseline': None, 'dtype': DTYPE,
        'data': 'synthetic',
        'config': {'workload': work.describe() if not args.weak else 'weak scaling: a {} shard per GPU'.format(work.describe()),
                   'sharding': '{} pairs per rank (contiguous 1/{} of the stream, generated on the device)'.format(
                       pairs_local, world),
                   'l2': 'input records {} MB per GPU > 126 MB L2, no explicit flush'.format(8 * pairs_local // 1000000),
                   'nnz_full': di[4], 'edges': di[5], 'row_splits': splits, 'generator_s': round(work.gen_s, 1)},
        'clocks': clocks, 'e2e': e2e, 'gpu_launches': int(launches),
        'stages_ms_synced': {'max_over_ranks': {k: round(float(v), 4) for k, v in zip(names, st_max.cpu())},
                             'mean_over_ranks': {k: round(float(v) / world, 4) for k, v in zip(names, st_sum.cpu())},
                             'accumulate_substeps_rank0': {k: round(float(v), 4) for k, v in zip(sub_names, sub_t.cpu())},
                             'accumulate_substeps_max': {k: round(float(v), 4) for k, v in zip(sub_names, sub_max.cpu())},
                             'note': 'a device-side barrier over all ranks precedes every stage (not part of the timed '
                                     'steps above)'},
        'kr': {'n_iter': kr['n_iter'], 'n_spmv': kr['n_spmv'], 'outer': kr['outer'], 'zero_diag': kr['zero_diag'],
               'kernel_us_rank0': kr.get('kernel_us'), 'kernel_us_max': float(krk_max.cpu()[0]), 'slabs': kr.get('slabs'),
               'phase_us_work': {k: round(v / 1965.0, 1) for k, v in kr.get('work_cycles', {}).items()},
               'phase_us_sync': {k: round(v / 1965.0, 1) for k, v in kr.get('sync_cycles', {}).items()}},
        'pair_counts': counters,
        'digest': {'map': _wrap64(di[0]), 'mask': _wrap64(di[1]), 'edges': _wrap64(di[2]), 'map_weight': di[3],
                   'nnz_full': di[4], 'n_edges': di[5], 'n_iter': kr['n_iter'], 'x_sum': float(df.cpu()[0]),
                   'w_sum': float(df.cpu()[1])},
        'parity': parity, 'roofline': roofline, 'cpu_baseline': cpu,
    }
    print(json.dumps(line))


def main():
    args = parse_args()
    rank = int(os.environ.get('RANK', 0))
    local_rank = int(os.environ.get('LOCAL_RANK', 0))
    world = int(os.environ.get('WORLD_SIZE', 1))
    if args.dump_outputs and (args.impl == 'reference' or world > 1):
        raise SystemExit('--dump-outputs is for --impl ours on one GPU')

    if args.impl == 'reference':
        run_reference(args, rank)
        return

    import torch
    import __graft_entry__
    __graft_entry__.build()
    assert torch.cuda.is_available(), 'bench.py needs a CUDA device (no CPU fallback)'
    torch.cuda.set_device(local_rank)
    from bin3c_b200 import device as dev
    # everything runs on one capturable (non-default) stream: the sort-reduce sequences replay as CUDA graphs, and
    # the timing events sit on the stream the kernels are launched on
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank))
        with dev.pipeline_stream():
            main_multi(args, rank, local_rank, world)
        torch.cuda.synchronize()
        dist.destroy_process_group()
        return
    with dev.pipeline_stream():
        main_single(args, local_rank)


if __name__ == '__main__':
    main()
