"""
Per-launch device time of the radix-sort kernels (k_rs_*) over a bench.py run, from torch.profiler's CUDA
activities (the kernels launched inside the reduce graph are recorded one by one).  Profile in a run of its own:
tracing slows the host, so ms_per_step from this run is not a timing.

    python tools/sort_launch_profile.py --out prof.json -- --no-cpu-baseline --no-microbench --no-e2e --no-c2 --steps 3

Everything after `--` goes to bench.py.  Prints one JSON line per kernel name (launches, total and mean us) and
writes the same list to --out.
"""
import argparse
import json
import os
import runpy
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def main():
    argv = sys.argv[1:]
    bench_args = []
    if '--' in argv:
        i = argv.index('--')
        argv, bench_args = argv[:i], argv[i + 1:]
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', required=True)
    ap.add_argument('--match', default='k_rs_', help='keep kernels whose name contains this')
    args = ap.parse_args(argv)

    import torch
    from torch.profiler import ProfilerActivity, profile
    if not torch.cuda.is_available():
        raise SystemExit('sort_launch_profile needs a CUDA device')
    sys.path.insert(0, ROOT)
    sys.argv = [os.path.join(ROOT, 'bench.py')] + bench_args
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        runpy.run_path(os.path.join(ROOT, 'bench.py'), run_name='__main__')
        torch.cuda.synchronize()
    rows = []
    for avg in prof.key_averages():
        if args.match not in avg.key:
            continue
        t = float(getattr(avg, 'device_time_total', 0.0) or getattr(avg, 'self_device_time_total', 0.0))
        rows.append((avg.key, int(avg.count), t))
    out = [{'kernel': k, 'launches': n, 'total_us': round(t, 1), 'mean_us': round(t / max(n, 1), 2)}
           for k, n, t in sorted(rows, key=lambda r: -r[2])]
    for r in out:
        print(json.dumps(r))
    with open(args.out, 'w') as f:
        json.dump({'gpu': torch.cuda.get_device_name(0), 'bench_args': bench_args, 'kernels': out}, f, indent=1)


if __name__ == '__main__':
    main()
