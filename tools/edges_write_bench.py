"""
cm_graph.edges from an edge list: the host writer (bam_io.write_edges on NumPy arrays, all cores) against the device
writer (the same call on CUDA tensors, bin3c_b200/csrc/edgefmt.cu), in both float styles, on synthetic edge lists of
the C3 (27 M edges) and C4 (100 M edges) sizes: u < v ids below 250 k / 1 M, weights log-uniform in (1e-6, 1] with 1 %
exactly 1.0.

    python tools/edges_write_bench.py [--sizes C3,C4] [--repeats 3] [--out FILE]

Per size and style: each writer once to warm up, then --repeats timed runs (wall clock around the whole call, which
ends when the file is closed); the best run is reported.  The two files must be equal.  To show what bounds the device
writer, two of its parts are also timed alone: the formatting calls (b3c_edges_text over all chunks, with the text
left on the device; host clock around calls that synchronise) and writing the same text from one pinned host buffer
to a file (no formatting).  Files go to a temporary directory, whose filesystem type is recorded; they are written
into the page cache (no fsync).  The GPU's name and power limit are read in the same run.  Prints one JSON line (and
writes it to --out).
"""
import argparse
import ctypes as C
import filecmp
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SIZES = {'C3': (27_000_000, 250_000), 'C4': (100_000_000, 1_000_000)}


def gpu_info():
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'],
                             stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=30).stdout
        name, power = [x.strip() for x in out.strip().splitlines()[0].split(',')]
        return name, power
    except Exception as e:                              # noqa: BLE001 -- recorded, not fatal
        return 'unknown ({})'.format(e), 'unknown'


def filesystem_of(path):
    """(mount point, type) of the mount holding `path`, from /proc/mounts"""
    path = os.path.realpath(path)
    best = ('?', '?')
    try:
        with open('/proc/mounts') as f:
            for line in f:
                dev, mnt, fstype = line.split()[:3]
                if (path == mnt or path.startswith(mnt.rstrip('/') + '/')) and len(mnt) >= len(best[0]):
                    best = (mnt, fstype)
    except OSError:
        pass
    return best


def make_edges(n, n_ids, seed=1):
    rng = np.random.default_rng(seed)
    a = rng.integers(0, n_ids, n, dtype=np.int64)
    b = rng.integers(0, n_ids - 1, n, dtype=np.int64)
    b = b + (b >= a)                                    # b != a
    u, v = np.minimum(a, b).astype(np.int32), np.maximum(a, b).astype(np.int32)
    w = np.exp(rng.uniform(np.log(1e-6), 0.0, n))
    w[rng.random(n) < 0.01] = 1.0
    return u, v, w


def best_of(fn, repeats):
    fn()
    ts = []
    for _ in range(repeats):
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
    return min(ts), ts


def format_alone(torch, du, dv, dw, style, chunk, repeats):
    """seconds for the b3c_edges_text calls over all chunks (text stays on the device), and the text bytes"""
    from bin3c_b200 import _cabi
    n = du.numel()
    cap = _cabi.B3C_EDGES_MAX_LINE_BYTES * chunk
    ws = torch.empty(int(_cabi.lib.b3c_edges_text_workspace_bytes(chunk)), dtype=torch.uint8, device='cuda')
    text = torch.empty(cap, dtype=torch.uint8, device='cuda')
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    nb = C.c_int64()
    total = [0]

    def run():
        total[0] = 0
        for lo in range(0, n, chunk):
            m = min(chunk, n - lo)
            _cabi.check(_cabi.lib.b3c_edges_text(ws.data_ptr(), ws.numel(), du.data_ptr() + 4 * lo,
                                                 dv.data_ptr() + 4 * lo, dw.data_ptr() + 8 * lo, m, 32, style,
                                                 text.data_ptr(), cap, C.byref(nb), stream))
            total[0] += nb.value
    t, _ = best_of(run, repeats)
    return t, total[0]


def write_alone(torch, path, nbytes, slab, repeats):
    """seconds to write nbytes from one pinned slab to a file, slab by slab"""
    buf = torch.full((slab,), 0x31, dtype=torch.uint8, pin_memory=True)
    view = memoryview(buf.numpy())

    def run():
        with open(path, 'wb') as f:
            left = nbytes
            while left > 0:
                k = min(left, slab)
                f.write(view[:k])
                left -= k
    t, _ = best_of(run, repeats)
    os.unlink(path)
    return t


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--sizes', default='C3,C4')
    ap.add_argument('--repeats', type=int, default=3)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    import torch
    from bin3c_b200 import _cabi, bam_io
    assert torch.cuda.is_available(), 'this benchmark needs a CUDA device'
    name, power = gpu_info()
    tmp = tempfile.mkdtemp(prefix='edges_write_')
    mnt, fstype = filesystem_of(tmp)
    res = dict(bench='edges_write', gpu=name, power_limit=power, tmp_dir_fs=fstype, tmp_dir_mount=mnt,
               host_threads=os.cpu_count(), repeats=args.repeats, chunk_edges=bam_io.DEFAULT_EDGE_CHUNK, runs=[])
    try:
        for size in args.sizes.split(','):
            n, n_ids = SIZES[size]
            u, v, w = make_edges(n, n_ids)
            du, dv, dw = (torch.from_numpy(x).cuda() for x in (u, v, w))
            for style, sname in ((bam_io.FLOAT_REPR, 'repr'), (bam_io.FLOAT_STR12, 'str12')):
                ph, pd = os.path.join(tmp, 'host.edges'), os.path.join(tmp, 'dev.edges')
                t_host, ts_host = best_of(lambda: bam_io.write_edges(u, v, w, ph, float_style=style), args.repeats)
                t_dev, ts_dev = best_of(lambda: bam_io.write_edges(du, dv, dw, pd, float_style=style), args.repeats)
                size_bytes = os.path.getsize(pd)
                equal = os.path.getsize(ph) == size_bytes and filecmp.cmp(ph, pd, shallow=False)
                os.unlink(ph)
                os.unlink(pd)
                t_fmt, fmt_bytes = format_alone(torch, du, dv, dw, style, bam_io.DEFAULT_EDGE_CHUNK, args.repeats)
                t_wr = write_alone(torch, os.path.join(tmp, 'raw.bin'), size_bytes,
                                   _cabi.B3C_EDGES_MAX_LINE_BYTES * bam_io.DEFAULT_EDGE_CHUNK, args.repeats)
                run = dict(size=size, n_edges=n, style=sname, file_bytes=size_bytes, files_equal=bool(equal),
                           host_s=round(t_host, 4), device_s=round(t_dev, 4), speedup=round(t_host / t_dev, 2),
                           host_runs_s=[round(t, 4) for t in ts_host], device_runs_s=[round(t, 4) for t in ts_dev],
                           device_format_only_s=round(t_fmt, 4), file_write_only_s=round(t_wr, 4),
                           host_medges_per_s=round(n / t_host / 1e6, 1), device_medges_per_s=round(n / t_dev / 1e6, 1),
                           format_text_bytes_equal=fmt_bytes == size_bytes)
                res['runs'].append(run)
                print(json.dumps(run), file=sys.stderr, flush=True)
            del du, dv, dw
            torch.cuda.empty_cache()
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
