"""
FASTA -> restriction-site table: the host counter (seq_sites.fasta_site_table) against the device counter
(device=True, bin3c_b200/csrc/sites.cu) on a seeded assembly, three ways: wrapped at 60 columns, unwrapped (one line
per contig), and wrapped + gzip'd.  Every device result must equal the host result (same dict, same order).

    python tools/fasta_sites_bench.py [--gbp 1.0] [--repeats 3] [--slab-mb 64] [--out FILE]

Per file: the host counter once; the device counter once to warm up, then --repeats timed runs (wall clock around the
whole call, which ends in a synchronise), with the split of the last run: the reader thread's time in readinto
(for .gz files that includes gzip's inflate), the time in slab calls (host-to-device copy and the kernels) and the time
the counting thread waited for the reader.  Also: the file read alone into pinned memory (and, for the .gz file,
inflate alone), and the device kernels alone on one slab already in device memory (CUDA events).  The GPU's name and
power limit are read in the same run.  Files are written to a temporary directory; plain files are read from the page
cache after being written.  Prints one JSON line (and writes it to --out).
"""
import argparse
import ctypes as C
import gzip
import json
import os
import shutil
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))

ENZYMES = ['MluCI', 'Sau3AI']


def gpu_info():
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'],
                             stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=30).stdout
        name, power = [x.strip() for x in out.strip().splitlines()[0].split(',')]
        return name, power
    except Exception as e:                              # noqa: BLE001 -- recorded, not fatal
        return 'unknown ({})'.format(e), 'unknown'


def read_alone(path, slab):
    """seconds to read (and for .gz inflate) the file into a pinned buffer, slab by slab"""
    import torch
    buf = torch.empty(slab, dtype=torch.uint8, pin_memory=True)
    view = memoryview(buf.numpy())
    t0 = time.perf_counter()
    with (gzip.open(path, 'rb') if path.endswith('.gz') else open(path, 'rb', buffering=0)) as f:
        while f.readinto(view):
            pass
    return time.perf_counter() - t0


def kernels_alone(path, slab, reps=10):
    """device seconds per slab of the first slab of the file, counted `reps` times from device memory"""
    import torch
    from bin3c_b200 import _cabi, seq_sites
    masks, lengths, weights = seq_sites._device_patterns(seq_sites._sites(ENZYMES))
    with open(path, 'rb') as f:
        data = f.read(slab)
    dev = torch.device('cuda')
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    nws = int(_cabi.lib.b3c_sites_workspace_bytes(len(data), 0))
    ws = torch.empty(nws, dtype=torch.uint8, device=dev)
    _cabi.check(_cabi.lib.b3c_sites_begin(ws.data_ptr(), nws, len(data), masks.ctypes.data, lengths.ctypes.data,
                                          weights.ctypes.data, len(lengths), 0, stream))
    d = torch.frombuffer(bytearray(data), dtype=torch.uint8).to(dev)
    cap = 1 << 22                                       # headers of `reps` slabs of an assembly, with room to spare
    seqs = torch.empty((cap, 5), dtype=torch.int64, device=dev)
    names = torch.empty(1 << 28, dtype=torch.uint8, device=dev)
    res = (C.c_int64 * 3)()

    def one():
        _cabi.check(_cabi.lib.b3c_sites_slab(ws.data_ptr(), d.data_ptr(), len(data), seqs.data_ptr(), cap,
                                             names.data_ptr(), names.numel(), res, stream))
    one()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps - 1):
        one()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / 1e3 / (reps - 1), len(data)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gbp', type=float, default=1.0)
    ap.add_argument('--repeats', type=int, default=3)
    ap.add_argument('--slab-mb', type=int, default=64)
    ap.add_argument('--out', default=None)
    ap.add_argument('--keep-dir', default=None, help='write the assemblies here instead of a temporary directory')
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit('fasta_sites_bench.py needs a CUDA device')
    from bin3c_b200 import seq_sites
    from fasta_cases import seeded_assembly
    name, power = gpu_info()
    slab = a.slab_mb << 20
    tmp = a.keep_dir or tempfile.mkdtemp(prefix='fasta_sites_bench_')
    total = int(a.gbp * 1e9)
    result = dict(tool='fasta_sites_bench', gpu=name, power_limit=power, gbp=a.gbp, enzymes=ENZYMES, slab_bytes=slab,
                  repeats=a.repeats, files={})
    try:
        for label, wrap, gz in (('wrap60', 60, False), ('unwrapped', None, False), ('wrap60_gz', 60, True)):
            path = os.path.join(tmp, 'asm_{}.fa{}'.format(label, '.gz' if gz else ''))
            t0 = time.perf_counter()
            n_contigs = seeded_assembly(path, total, seed=7, wrap=wrap, gz=gz)
            write_s = time.perf_counter() - t0
            t0 = time.perf_counter()
            want = seq_sites.fasta_site_table(path, ENZYMES)
            host_s = time.perf_counter() - t0
            bp = sum(v['length'] for v in want.values())
            seq_sites.fasta_site_table(path, ENZYMES, device=True, slab_bytes=slab)          # warm-up
            times, split = [], {}
            for _ in range(a.repeats):
                split = {}
                t0 = time.perf_counter()
                got = seq_sites._site_table_on_device(path, seq_sites._device_patterns(seq_sites._sites(ENZYMES)), 0,
                                                      None, slab, timing=split)
                times.append(time.perf_counter() - t0)
                assert list(got.items()) == list(want.items()), 'device result differs from the host counter'
            read_s = read_alone(path, slab)
            inflate_s = None
            if gz:                                    # inflate alone = read+inflate minus reading the compressed bytes
                t0 = time.perf_counter()
                with open(path, 'rb', buffering=0) as f:
                    while f.read(slab):
                        pass
                inflate_s = read_s - (time.perf_counter() - t0)
            k_s, k_bytes = kernels_alone(path, slab) if not gz else (None, None)     # same bytes once inflated
            dev_s = statistics.median(times)
            result['files'][label] = dict(
                file_bytes=os.path.getsize(path), bp=bp, contigs=n_contigs, equal=True, write_s=round(write_s, 3),
                host_s=round(host_s, 3), host_mbp_s=round(bp / host_s / 1e6, 1),
                device_s=[round(t, 3) for t in times], device_median_s=round(dev_s, 3),
                device_mbp_s=round(bp / dev_s / 1e6, 1), speedup=round(host_s / dev_s, 2),
                split_last_run={k: (round(v, 3) if isinstance(v, float) else v) for k, v in split.items()},
                read_alone_s=round(read_s, 3), inflate_alone_s=None if inflate_s is None else round(inflate_s, 3),
                kernels_per_slab_s=None if gz else round(k_s, 5),
                kernels_gb_s=None if gz else round(k_bytes / k_s / 1e9, 1))
            print(label, json.dumps(result['files'][label]), file=sys.stderr, flush=True)
    finally:
        if not a.keep_dir:
            shutil.rmtree(tmp, ignore_errors=True)
    line = json.dumps(result)
    print(line)
    if a.out:
        with open(a.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
