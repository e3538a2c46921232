"""
The contact_map.p.gz stage hand-off (io_utils.save_object / load_object) at C2 and C3 size: pickle bytes, file bytes
and wall times of
  host_save       save_object: pickle + Python gzip level 6, one thread (what bin3C.py mkmap does)
  threaded_save   comparison arm, not product: pickle, then zlib level 6 over 65280-byte members on os.cpu_count()
                  threads with the BGZF framing of the device path
  device_save     save_object(device=True)
  pickle_only     pickle.dumps alone (the host share of every save)
  host_load / device_load
then, in a separate pass, the device kernels' times from torch.profiler.  Writes <out>/map_handoff.json.
    python tools/map_handoff_bench.py --out DIR [--configs C2,C3] [--c3-scale 0.2] [--reps 3]
"""
import argparse
import json
import os
import pickle
import struct
import subprocess
import sys
import tempfile
import time
import zlib
from concurrent.futures import ThreadPoolExecutor

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np                                   # noqa: E402
import torch                                         # noqa: E402

from bin3c_b200 import io_utils, synth               # noqa: E402
from bin3c_b200.contact_map import ContactMap, PairRecords   # noqa: E402


def threaded_gzip(raw, path, threads):
    def member(k):
        piece = raw[k:k + io_utils.MEMBER_INPUT]
        c = zlib.compressobj(6, zlib.DEFLATED, -15)
        body = c.compress(piece) + c.flush()
        size = 18 + len(body) + 8
        return (bytes.fromhex('1f8b08040000000000ff060042430200') + struct.pack('<H', size - 1) + body +
                struct.pack('<II', zlib.crc32(piece), len(piece)))
    with ThreadPoolExecutor(threads) as ex, open(path, 'wb') as f:
        for m in ex.map(member, range(0, len(raw), io_utils.MEMBER_INPUT)):
            f.write(m)
        f.write(io_utils.BGZF_EOF)


def timed(fn, reps):
    ts = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t)
    return ts


def build_map(cfg, scale):
    com = synth.make_config(cfg, scale)
    return ContactMap(PairRecords.from_community(com), ['synthetic'], None, None, min_mapq=60, min_len=1000,
                      min_sig=5, random_seed=1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', required=True)
    ap.add_argument('--configs', default='C2,C3')
    ap.add_argument('--c3-scale', type=float, default=0.2, help='fraction of the C3 pair stream the map is built from')
    ap.add_argument('--reps', type=int, default=3)
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    assert torch.cuda.is_available(), 'the device arms need a CUDA device'
    gpu = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'],
                         stdout=subprocess.PIPE, text=True).stdout.strip().splitlines()
    result = dict(gpu=gpu[0] if gpu else torch.cuda.get_device_name(), host_threads=os.cpu_count(), configs={})
    tmp = tempfile.mkdtemp(prefix='handoff_')
    io_utils.save_object(os.path.join(tmp, 'warm'), {'a': np.arange(10 ** 6)}, device=True)   # module load, pinning
    for cfg in args.configs.split(','):
        scale = args.c3_scale if cfg == 'C3' else 1.0
        t = time.perf_counter()
        cm = build_map(cfg, scale)
        built = time.perf_counter() - t
        raw = pickle.dumps(cm, pickle.HIGHEST_PROTOCOL)
        r = dict(scale=scale, map_build_s=built, nnz=int(cm.seq_map.nnz), pickle_bytes=len(raw))
        host_p, dev_p, thr_p = (os.path.join(tmp, cfg + s) for s in ('_host.p', '_dev.p', '_thr.p.gz'))
        r['pickle_only_s'] = timed(lambda: pickle.dumps(cm, pickle.HIGHEST_PROTOCOL), args.reps)
        r['host_save_s'] = timed(lambda: io_utils.save_object(host_p, cm), 1)
        r['threaded_save_s'] = timed(lambda: threaded_gzip(pickle.dumps(cm, pickle.HIGHEST_PROTOCOL), thr_p,
                                                           os.cpu_count()), args.reps)
        r['device_save_s'] = timed(lambda: io_utils.save_object(dev_p, cm, device=True), args.reps)
        r['host_load_s'] = timed(lambda: io_utils.load_object(host_p + '.gz'), 1)
        r['device_load_s'] = timed(lambda: io_utils.load_object(dev_p + '.gz', device=True), args.reps)
        for k, p in (('host_file_bytes', host_p + '.gz'), ('device_file_bytes', dev_p + '.gz'),
                     ('threaded_file_bytes', thr_p)):
            r[k] = os.path.getsize(p)
        with open(dev_p + '.gz', 'rb') as f:
            import gzip
            r['device_file_decompresses_to_pickle'] = gzip.decompress(f.read()) == raw
        r['zlib6_whole_bytes'] = len(zlib.compress(raw, 6))
        r['device_vs_zlib6'] = r['device_file_bytes'] / r['zlib6_whole_bytes']
        r['speedup_device_save_vs_host'] = min(r['host_save_s']) / min(r['device_save_s'])
        r['speedup_device_save_vs_threaded'] = min(r['threaded_save_s']) / min(r['device_save_s'])
        # per-kernel device times of one device save, in a pass of their own
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
            io_utils.save_object(dev_p, cm, device=True)
            torch.cuda.synchronize()
        kern = {}
        for e in prof.key_averages():
            dt = getattr(e, 'device_time_total', None) or getattr(e, 'cuda_time_total', 0)
            if dt and ('k_' in e.key or 'Memcpy' in e.key or 'scan' in e.key):
                kern[e.key] = dict(calls=e.count, total_ms=dt / 1e3)
        r['profile_device_save'] = kern
        result['configs'][cfg] = r
        print(json.dumps({cfg: {k: v for k, v in r.items() if k != 'profile_device_save'}}), flush=True)
        for p in (host_p + '.gz', dev_p + '.gz', thr_p):
            os.remove(p)
        del cm, raw
    with open(os.path.join(args.out, 'map_handoff.json'), 'w') as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result))


if __name__ == '__main__':
    main()
