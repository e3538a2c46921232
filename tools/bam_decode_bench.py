"""
BAM file -> packed pair records: the host reader (libbin3c_io.so, one inflate thread per core) against the GPU decoder
(bam_io.pair_records_from_bam(device=True)), in one call, on the io_bench community: name-sorted pairs over 50 000
references, 150-base reads with 120 incompressible tag bytes per alignment (about 3:1 at zlib level 1).  Two layouts of
the same stream: blocks cut before a record that would not fit (as htslib writes them) and blocks cut every 65280 bytes
(records straddle blocks; the decoder's boundary guesses then rest on field checks).

Times are file (in the page cache, read once before timing) to records in device memory, best of --repeat after one
warm-up; per-kernel device times come from a separate torch.profiler pass over one decode.
    python tools/bam_decode_bench.py [--pairs 4000000] [--repeat 5] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))

STAGES = {'inflate': ('k_inflate', 'k_crc'), 'boundaries': ('k_guess', 'k_verify'), 'parse': ('k_scan', 'k_link'),
          'pair': ('k_chain', 'k_emit')}


def make_stream(n_pairs, seed=1):
    """The alignment section as bytes (vectorised; the records of tests/bam_writer.encode_alignment) and the record
    sizes of the two mates."""
    rng = np.random.default_rng(seed)
    n_refs = 50_000
    name_len = 42                                         # 41 characters + NUL
    l_seq = 150
    sizes = []
    mates = []
    for mate, (flag, cig) in enumerate(((0x63, [(0, 150)]), (0x93, [(4, 10), (0, 140)]))):
        body = 32 + name_len + 4 * len(cig) + (l_seq + 1) // 2 + l_seq + 120
        rec = np.zeros((n_pairs, 4 + body), dtype=np.uint8)
        head = np.zeros(n_pairs, dtype=np.dtype([('bs', '<i4'), ('tid', '<i4'), ('pos', '<i4'), ('l_name', 'u1'),
                                                   ('mapq', 'u1'), ('bin', '<u2'), ('n_cig', '<u2'), ('flag', '<u2'),
                                                   ('l_seq', '<i4'), ('ntid', '<i4'), ('npos', '<i4'), ('tlen', '<i4')]))
        head['bs'] = body
        head['tid'] = rng.integers(0, n_refs, n_pairs)
        head['pos'] = 100 if mate == 0 else 400
        head['l_name'] = name_len
        head['mapq'] = 60
        head['bin'] = 4680
        head['n_cig'] = len(cig)
        head['flag'] = flag
        head['l_seq'] = l_seq
        head['ntid'] = -1
        head['npos'] = -1
        rec[:, :36] = head.view(np.uint8).reshape(n_pairs, 36)
        k = np.arange(n_pairs)
        names = np.char.add(np.char.add(np.char.add('A00123:45:HXXXXXXXX:1:', np.char.zfill((1101 + k % 500).astype(str), 4)),
                                        np.char.add(':', np.char.zfill((k % 30000).astype(str), 5))),
                            np.char.add(':', np.char.zfill(k.astype(str), 8)))
        rec[:, 36:36 + name_len - 1] = np.frombuffer(names.astype('S41').tobytes(), dtype=np.uint8).reshape(n_pairs, 41)
        o = 36 + name_len
        for op, n in cig:
            rec[:, o:o + 4] = np.frombuffer(np.uint32((n << 4) | op).tobytes(), dtype=np.uint8)
            o += 4
        rec[:, o:o + (l_seq + 1) // 2] = 0x11
        o += (l_seq + 1) // 2
        rec[:, o:o + l_seq] = 0x1e
        o += l_seq
        rec[:, o:o + 120] = rng.integers(0, 256, (n_pairs, 120), dtype=np.uint8)
        sizes.append(4 + body)
        mates.append(rec)
    stream = np.stack(mates, axis=1).reshape(-1) if sizes[0] == sizes[1] else \
        np.concatenate([mates[0], mates[1]], axis=1).reshape(-1)
    return stream, sizes


def write_bam(path, refs_header, stream, cuts, threads):
    """BGZF blocks of stream[cuts[i]:cuts[i+1]] at zlib level 1, compressed on a thread pool."""
    import bam_writer

    def block(i):
        return bam_writer.bgzf_block(stream[cuts[i]:cuts[i + 1]].tobytes(), 1)
    with open(path, 'wb') as out:
        for o in range(0, len(refs_header), 65280):
            out.write(bam_writer.bgzf_block(refs_header[o:o + 65280], 1))
        with ThreadPoolExecutor(threads) as ex:
            for b in ex.map(block, range(len(cuts) - 1), chunksize=64):
                out.write(b)
        out.write(bam_writer.BGZF_EOF)


def gpu_info():
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                             stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=60).stdout.strip()
        return out.splitlines()[0] if out else None
    except (OSError, subprocess.SubprocessError):
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--pairs', type=int, default=4_000_000)
    ap.add_argument('--repeat', type=int, default=5)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    import torch
    import bam_writer
    from bin3c_b200 import bam_io
    if not torch.cuda.is_available():
        raise SystemExit('bam_decode_bench needs a CUDA device')
    threads = os.cpu_count()
    t0 = time.perf_counter()
    stream, (s1, s2) = make_stream(args.pairs)
    n_refs = 50_000
    header = bam_writer.encode_header(['c%d' % i for i in range(n_refs)], [5000] * n_refs)
    pair = s1 + s2
    per_block = 65280 // pair
    aligned = np.arange(0, len(stream) + 1, per_block * pair, dtype=np.int64)
    if aligned[-1] != len(stream):
        aligned = np.append(aligned, len(stream))
    arbitrary = np.append(np.arange(0, len(stream), 65280, dtype=np.int64), len(stream))
    out = {'gpu': gpu_info(), 'torch_device': torch.cuda.get_device_name(0), 'host_cores': threads,
           'pairs': args.pairs, 'record_bytes': [s1, s2], 'uncompressed_bytes': int(len(stream) + len(header)),
           'page_cache': 'file read once before timing', 'layouts': {}}
    with tempfile.TemporaryDirectory() as d:
        for name, cuts in (('record_aligned', aligned), ('arbitrary_cut_65280', arbitrary)):
            path = os.path.join(d, name + '.bam')
            write_bam(path, header, stream, cuts, threads)
            fsize = os.path.getsize(path)
            with open(path, 'rb') as f:                      # into the page cache
                while f.read(1 << 24):
                    pass
            res = {'file_bytes': fsize, 'blocks': int(len(cuts) - 1)}

            def host():
                with bam_io.BamPairReader(path, threads=threads) as bam:
                    bam.set_filter(min_mapq=30, strong=50)
                    return bam.read_all(), bam.stats()

            def device():
                pr, st = bam_io.pair_records_from_bam(path, min_mapq=30, strong=50, device=True)
                torch.cuda.synchronize()
                return pr, st

            for label, fn in (('host', host), ('gpu', device)):
                fn()
                best = 1e30
                for _ in range(args.repeat):
                    t = time.perf_counter()
                    r = fn()
                    best = min(best, time.perf_counter() - t)
                res[label] = {'s': round(best, 4), 'pairs_per_s': round(args.pairs / best),
                              'compressed_gb_per_s': round(fsize / best / 1e9, 3),
                              'uncompressed_gb_per_s': round(out['uncompressed_bytes'] / best / 1e9, 3)}
                if label == 'host':
                    host_rec, host_st = r
                else:
                    pr, st = r
                    res['gpu']['slabs'] = pr.meta['slabs']
                    res['gpu']['repaired_blocks'] = pr.meta['repaired_blocks']
                    res['records_equal'] = bool(torch.equal(pr.records.cpu(), torch.from_numpy(host_rec)))
                    res['stats_equal'] = st == host_st
                    res['n_records'] = int(pr.records.numel())
            res['gpu_over_host'] = round(res['host']['s'] / res['gpu']['s'], 2)
            # per-kernel device time of one decode (a separate, profiled pass)
            from torch.profiler import profile, ProfilerActivity
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                device()
            kt = {}
            for e in prof.key_averages():
                for stage, kernels in STAGES.items():
                    if any(k in e.key for k in kernels):
                        kt.setdefault(stage, 0.0)
                        kt[stage] += e.device_time_total / 1e3
                if 'Memcpy HtoD' in e.key:
                    kt['h2d_copy'] = kt.get('h2d_copy', 0.0) + e.device_time_total / 1e3
            res['kernel_ms'] = {k: round(v, 3) for k, v in kt.items()}
            out['layouts'][name] = res
            os.remove(path)
    out['wall_s'] = round(time.perf_counter() - t0, 1)
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
