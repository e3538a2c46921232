"""
CPU side of the device BGZF encoder: the deflate core bin3c_b200/csrc/deflate.cuh, built with g++ through
tests/native/deflate_check.cpp (also under AddressSanitizer + UBSan), checked member by member against zlib's raw
inflate and inflate.cuh's host build, with the BGZF framing (header, BSIZE, CRC-32 = zlib.crc32, ISIZE) and the code
lengths of every dynamic block (at most 15 bits, 7 for the code-length code, every code complete); and the argument
checks of io_utils.save_object / load_object(device=True) that come before any device work.
"""
import gzip
import os
import pickle
import shutil
import struct
import subprocess
import sys
import zlib

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from bin3c_b200 import io_utils                     # noqa: E402
from bam_writer import BGZF_EOF                      # noqa: E402

SRC = os.path.join(ROOT, 'tests', 'native', 'deflate_check.cpp')
MEMBER = io_utils.MEMBER_INPUT


def build_tool(tmp_dir, sanitize=None):
    if shutil.which('g++') is None:
        pytest.skip('no g++')
    exe = os.path.join(str(tmp_dir), 'deflate_check' + ('_san' if sanitize else ''))
    cmd = ['g++', '-std=c++17', '-Wall', '-Werror'] + (
        ['-O1', '-g', '-fsanitize=' + sanitize, '-fno-omit-frame-pointer', '-fno-sanitize-recover=all']
        if sanitize else ['-O2']) + [SRC, '-o', exe]
    res = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if res.returncode != 0 and sanitize:
        pytest.skip('no {} runtime: {}'.format(sanitize, res.stdout[-300:]))
    assert res.returncode == 0, res.stdout
    return exe


def encode(tool, tmp_path, data, tag='in'):
    """The harness's members for `data` and its per-member report rows."""
    src, out = tmp_path / (tag + '.bin'), tmp_path / (tag + '.bgzf')
    src.write_bytes(data)
    res = subprocess.run([tool, str(src), str(out)], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True,
                         timeout=600)
    assert res.returncode == 0, res.stderr
    rows = [tuple(int(x) for x in line.split()) for line in res.stdout.splitlines()]
    return out.read_bytes(), rows


def split_members(blob):
    members, o = [], 0
    while o < len(blob):
        assert blob[o:o + 4] == b'\x1f\x8b\x08\x04'
        bsize = struct.unpack_from('<H', blob, o + 16)[0]
        members.append(blob[o:o + bsize + 1])
        o += bsize + 1
    assert o == len(blob)
    return members


def check_members(blob, rows, data):
    """Every member against zlib and its own piece of the input; returns the members."""
    members = split_members(blob)
    pieces = [data[k:k + MEMBER] for k in range(0, len(data), MEMBER)] or [b'']
    assert len(members) == len(pieces) == len(rows)
    head = bytes.fromhex('1f8b08040000000000ff06004243020000')[:16]
    for m, piece, row in zip(members, pieces, rows):
        assert row[-1] == 0, row                                  # the harness's own checks (inflate.cuh, lengths)
        assert len(m) <= 65536 and row[2] == len(m)
        assert m[:16] == head and struct.unpack_from('<H', m, 16)[0] == len(m) - 1
        d = zlib.decompressobj(-15)
        assert d.decompress(m[18:-8]) == piece and d.eof and not d.unused_data
        assert struct.unpack('<II', m[-8:]) == (zlib.crc32(piece), len(piece))
        if row[1] == 2:
            assert row[3] <= 15 and row[4] <= 15 and row[5] <= 7
    assert gzip.decompress(blob + BGZF_EOF) == data
    return members


def de_bruijn(k, n):
    """A de Bruijn sequence B(k, n) over range(k): every n-gram once (cyclically)."""
    a, seq = [0] * k * n, []

    def db(t, p):
        if t > n:
            if n % p == 0:
                seq.extend(a[1:p + 1])
        else:
            a[t] = a[t - p]
            db(t + 1, p)
            for j in range(a[t - p] + 1, k):
                a[t] = j
                db(t + 1, t)
    db(1, 1)
    return bytes(seq)


def fibonacci_bytes(rng, n_symbols=22):
    f = [1, 1]
    while len(f) < n_symbols:
        f.append(f[-1] + f[-2])
    raw = np.repeat(np.arange(n_symbols, dtype=np.uint8) * 11, f)
    return rng.permutation(raw).tobytes()


def match_lengths(rng):
    out = []
    for L in range(3, 259):
        x = rng.integers(0, 256, L, dtype=np.uint8).tobytes()
        out += [rng.integers(0, 256, 40, dtype=np.uint8).tobytes(), x, b'\x00\xff', x]
    return b''.join(out)


def distances(rng):
    out = []
    for d in (1, 2, 4, 5, 8, 9, 24576, 32767, 32768):
        x = rng.integers(0, 256, d, dtype=np.uint8).tobytes()
        out.append(x + (x * (1 + 24 // d))[:24] + rng.integers(0, 256, 64, dtype=np.uint8).tobytes())
    return b''.join(out)


def contact_map_arrays(rng, n=200_000, n_rows=30_000):
    row = np.sort(rng.integers(0, n_rows, n)).astype(np.int32)
    col = rng.integers(0, n_rows, n).astype(np.int32)
    data = rng.geometric(0.3, n).astype(np.uint32)
    return pickle.dumps({'row': row, 'col': col, 'data': data, 'shape': (n_rows, n_rows)}, pickle.HIGHEST_PROTOCOL)


def host_map_pickle():
    import test_io_utils
    return pickle.dumps(test_io_utils._host_map(n=300, seed=5), pickle.HIGHEST_PROTOCOL)


def cases():
    rng = np.random.default_rng(20261022)
    return {
        'empty': b'', 'one': b'a', 'two': b'ab', 'three': b'abc',
        'match_lengths': match_lengths(rng),
        'distances': distances(rng),
        'all_bytes': bytes(range(256)) * 300,
        'run': b'\x07' * MEMBER,
        'run_plus_one': b'\x07' * (MEMBER + 1),
        'random': rng.integers(0, 256, 3 * MEMBER + 1000, dtype=np.uint8).tobytes(),
        'fibonacci': fibonacci_bytes(rng),
        'literal_only': de_bruijn(16, 3),
        'contact_arrays': contact_map_arrays(rng),
        'host_map': host_map_pickle(),
    }


CASES = cases()


@pytest.fixture(scope='module')
def tool(tmp_path_factory):
    return build_tool(tmp_path_factory.mktemp('deflate'))


@pytest.mark.parametrize('name', sorted(CASES))
def test_members_round_trip_through_zlib(tool, tmp_path, name):
    data = CASES[name]
    blob, rows = encode(tool, tmp_path, data)
    members = check_members(blob, rows, data)
    if name == 'random':
        assert all(r[1] == 0 for r in rows), 'incompressible input is stored'
    if name in ('run', 'literal_only', 'fibonacci', 'contact_arrays', 'host_map', 'all_bytes'):
        assert all(r[1] == 2 for r in rows), rows
    if name == 'run':
        assert len(members[0]) < 300
    if name == 'literal_only':
        assert len(blob) < len(data) * 0.6


def test_every_length_and_distance_code_is_used(tool, tmp_path):
    """The match-length and distance inputs reach every length code (257-285) and the distance codes they aim at."""
    seen_l, seen_d = set(), set()
    for name in ('match_lengths', 'distances', 'run'):
        blob, _ = encode(tool, tmp_path, CASES[name], name)
        for m in split_members(blob):
            syms = _symbols(m[18:-8])
            seen_l |= {s for s in syms[0] if s >= 257}
            seen_d |= set(syms[1])
    assert seen_l == set(range(257, 286))
    assert {0, 1, 3, 4, 6, 7, 28, 29} <= seen_d


def _symbols(payload):
    """(literal/length symbols, distance codes) of a single-block raw-deflate payload, decoded in Python."""
    pos = [0]

    def bits(n):
        v = 0
        for k in range(n):
            v |= ((payload[pos[0] >> 3] >> (pos[0] & 7)) & 1) << k
            pos[0] += 1
        return v

    def table(lengths):
        codes, code, cnt = {}, 0, [0] * 16
        for ln in lengths:
            cnt[ln] += 1
        cnt[0] = 0
        nxt = [0] * 16
        for b in range(1, 16):
            code = (code + cnt[b - 1]) << 1
            nxt[b] = code
        for s, ln in enumerate(lengths):
            if ln:
                codes[(ln, nxt[ln])] = s
                nxt[ln] += 1
        return codes

    def decode(t):
        code, ln = 0, 0
        while True:
            code = (code << 1) | bits(1)
            ln += 1
            if (ln, code) in t:
                return t[(ln, code)]

    bits(1)
    if bits(2) != 2:
        return set(), set()
    hlit, hdist, hclen = bits(5) + 257, bits(5) + 1, bits(4) + 4
    order = [16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15]
    cl = [0] * 19
    for k in range(hclen):
        cl[order[k]] = bits(3)
    clt, lengths = table(cl), []
    while len(lengths) < hlit + hdist:
        s = decode(clt)
        if s < 16:
            lengths.append(s)
        elif s == 16:
            lengths += [lengths[-1]] * (3 + bits(2))
        elif s == 17:
            lengths += [0] * (3 + bits(3))
        else:
            lengths += [0] * (11 + bits(7))
    lt, dt = table(lengths[:hlit]), table(lengths[hlit:])
    lext = [0] * 8 + [k // 4 - 1 for k in range(8, 28)] + [0]
    dext = [0] * 4 + [k // 2 - 1 for k in range(4, 30)]
    lsyms, dsyms = set(), set()
    while True:
        s = decode(lt)
        lsyms.add(s)
        if s == 256:
            return lsyms, dsyms
        if s > 256:
            bits(lext[s - 257])
            d = decode(dt)
            dsyms.add(d)
            bits(dext[d])


@pytest.mark.parametrize('n,limit', [(286, 15), (30, 15), (19, 7)])
def test_fibonacci_frequencies_meet_the_length_limit(tool, n, limit):
    """Fibonacci weights make the unlimited Huffman code as deep as there are symbols; the limited code stays within
    `limit` bits, complete, and gives no heavier symbol a longer code."""
    fib = [1, 1]
    while len(fib) < 40:
        fib.append(fib[-1] + fib[-2])
    rng = np.random.default_rng(n)
    freq = [0] * n
    for k, s in enumerate(rng.permutation(n)[:min(n, 24)]):
        freq[s] = fib[k]
    res = subprocess.run([tool, 'lengths', str(limit)] + [str(f) for f in freq], stdout=subprocess.PIPE, text=True,
                         check=True)
    lengths = [int(x) for x in res.stdout.split()]
    used = [s for s in range(n) if freq[s]]
    assert max(lengths) == limit
    assert all(lengths[s] > 0 for s in used) and all(lengths[s] == 0 for s in range(n) if not freq[s])
    assert sum(2.0 ** -lengths[s] for s in used) == 1.0
    by_weight = sorted(used, key=lambda s: freq[s])
    assert all(lengths[a] >= lengths[b] for a, b in zip(by_weight, by_weight[1:]))


def test_size_against_zlib_level6(tool, tmp_path):
    """The members of a contact-map-like pickle stay within 1.10x of zlib level 6 over the whole stream."""
    for name in ('contact_arrays', 'host_map'):
        blob, _ = encode(tool, tmp_path, CASES[name], name)
        ratio = (len(blob) + len(BGZF_EOF)) / len(zlib.compress(CASES[name], 6))
        assert ratio <= 1.10, (name, ratio)


def test_members_do_not_depend_on_neighbours(tool, tmp_path):
    """A member is a function of its own input bytes: encoding a piece alone gives the same member."""
    data = CASES['contact_arrays']
    whole = split_members(encode(tool, tmp_path, data, 'whole')[0])
    for k in (0, 2):
        alone = encode(tool, tmp_path, data[k * MEMBER:(k + 1) * MEMBER], 'piece{}'.format(k))[0]
        assert alone == whole[k]


@pytest.mark.parametrize('sanitize', ['address,undefined'])
def test_members_under_sanitizers(tmp_path, sanitize):
    exe = build_tool(tmp_path, sanitize)
    for name in ('empty', 'three', 'match_lengths', 'distances', 'run_plus_one', 'random', 'fibonacci',
                 'literal_only', 'contact_arrays'):
        blob, rows = encode(exe, tmp_path, CASES[name], name)
        check_members(blob, rows, CASES[name])


def test_device_paths_need_a_cuda_device(tmp_path):
    torch = pytest.importorskip('torch')
    if torch.cuda.is_available():
        pytest.skip('a CUDA device is present')
    p = str(tmp_path / 'map.p')
    with pytest.raises(RuntimeError, match='device=False'):
        io_utils.save_object(p, {'a': 1}, device=True)
    assert not os.path.exists(p + '.gz')
    io_utils.save_object(p, {'a': 1})
    with pytest.raises(RuntimeError, match='device=False'):
        io_utils.load_object(p + '.gz', device=True)
