"""
CPU side of the device BAM decoder: the deflate core and CRC-32 of bin3c_b200/csrc/inflate.cuh, built with g++ through
tests/native/inflate_check.cpp, against zlib (also under AddressSanitizer + UBSan), and the host framing the decoder
relies on (include/bin3c_io.h: b3c_bgzf_scan, b3c_bam_data_offset).
"""
import os
import random
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

import bam_writer                                   # noqa: E402
from bin3c_b200 import bam_io                       # noqa: E402

SRC = os.path.join(ROOT, 'tests', 'native', 'inflate_check.cpp')


def _build(tmp_dir, sanitize=None):
    if shutil.which('g++') is None:
        pytest.skip('no g++')
    exe = os.path.join(str(tmp_dir), 'inflate_check' + ('_san' if sanitize else ''))
    cmd = ['g++', '-std=c++17', '-Wall', '-Werror', SRC, '-o', exe]
    cmd[1:1] = ['-O1', '-g', '-fsanitize=' + sanitize, '-fno-omit-frame-pointer', '-fno-sanitize-recover=all'] \
        if sanitize else ['-O2']
    res = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if res.returncode != 0:
        if sanitize:
            pytest.skip('sanitizer build not available here: ' + res.stdout[-300:])
        raise AssertionError(res.stdout)
    return exe


@pytest.fixture(scope='module')
def tool(tmp_path_factory):
    return _build(tmp_path_factory.mktemp('inflate'))


def _inflate(exe, tmp_path, raw, cap, env=None):
    src, dst = str(tmp_path / 'in.bin'), str(tmp_path / 'out.bin')
    with open(src, 'wb') as f:
        f.write(raw)
    res = subprocess.run([exe, 'inflate', src, dst, str(cap)], stdout=subprocess.PIPE, stderr=subprocess.PIPE,
                         text=True, env=env, timeout=120)
    assert res.returncode == 0, res.stderr[-3000:]
    status, n = (int(v) for v in res.stdout.split())
    with open(dst, 'rb') as f:
        out = f.read()
    assert len(out) == n
    return status, out


def _zlib(raw):
    """What zlib's raw inflate makes of `raw`: the output, or None when the stream is invalid or ends early."""
    d = zlib.decompressobj(-15)
    try:
        out = d.decompress(raw) + d.flush()
    except zlib.error:
        return None
    return out if d.eof else None


def _deflate(data, level=6, strategy=zlib.Z_DEFAULT_STRATEGY):
    c = zlib.compressobj(level, zlib.DEFLATED, -15, 9, strategy)
    return c.compress(data) + c.flush()


class _Bits(object):
    """LSB-first bit writer of a deflate stream."""

    def __init__(self):
        self.acc, self.n, self.out = 0, 0, bytearray()

    def put(self, v, nbits):
        self.acc |= v << self.n
        self.n += nbits
        while self.n >= 8:
            self.out.append(self.acc & 0xff)
            self.acc >>= 8
            self.n -= 8

    def huff(self, code, nbits):                     # Huffman codes go most significant bit first
        self.put(int('{:0{}b}'.format(code, nbits)[::-1], 2), nbits)

    def bytes(self):
        return bytes(self.out) + (bytes([self.acc]) if self.n else b'')


def _fixed_lit(w, sym):
    if sym < 144:
        w.huff(0x30 + sym, 8)
    elif sym < 256:
        w.huff(0x190 + sym - 144, 9)
    elif sym < 280:
        w.huff(sym - 256, 7)
    else:
        w.huff(0xc0 + sym - 280, 8)


def far_matches_stream(rng):
    """A fixed-Huffman block: 32768 literals, then matches of length 258 at distance 32768 (zlib's own compressor never
    reaches that far: it stops 262 bytes short of the window)."""
    lit = bytes(rng.getrandbits(8) for _ in range(32768))
    w = _Bits()
    w.put(1, 1)
    w.put(1, 2)
    for b in lit:
        _fixed_lit(w, b)
    for _ in range(100):
        _fixed_lit(w, 285)                           # length 258, no extra bits
        w.huff(29, 5)                                # distance code 29: 24577 + 13 extra bits
        w.put(32768 - 24577, 13)
    _fixed_lit(w, 256)
    want = lit + (lit * 2)[:258 * 100]
    return w.bytes(), want


def _inputs():
    rng = random.Random(5)
    text = b''.join('read{:07d}\t{}\t{}\tACGTTGCA\n'.format(i, i % 97, i * 7).encode() * 3 for i in range(4000))
    return {
        'empty': b'',
        'one': b'x',
        'incompressible': bytes(rng.getrandbits(8) for _ in range(65280)),
        'repetitive': b'A' * 65280,
        'period3': b'ACG' * 21760,
        'text_65280': text[:65280],
        'short_text': text[:1000],
        'bam_like': bytes(rng.choice(b'\x00\x01\x11\x1e\xffACGT') for _ in range(65280)),
    }


def test_inflate_matches_zlib_on_every_level_and_strategy(tool, tmp_path):
    cases = 0
    for name, data in _inputs().items():
        variants = [(lv, zlib.Z_DEFAULT_STRATEGY) for lv in range(10)]
        variants += [(6, zlib.Z_FIXED), (6, zlib.Z_HUFFMAN_ONLY), (6, zlib.Z_RLE), (6, zlib.Z_FILTERED), (9, zlib.Z_RLE)]
        for level, strategy in variants:
            raw = _deflate(data, level, strategy)
            assert _zlib(raw) == data
            status, out = _inflate(tool, tmp_path, raw, len(data))
            assert status == 0 and out == data, (name, level, strategy, status)
            cases += 1
    assert cases == 8 * 15


def test_inflate_far_matches_and_output_capacity(tool, tmp_path):
    raw, want = far_matches_stream(random.Random(9))
    assert _zlib(raw) == want and len(want) == 32768 + 25800
    status, out = _inflate(tool, tmp_path, raw, len(want))
    assert status == 0 and out == want
    status, _ = _inflate(tool, tmp_path, raw, len(want) - 1)        # one byte more than ISIZE allows
    assert status == -2
    # the same distance one byte too far: before the start of the output
    w = _Bits()
    w.put(1, 1)
    w.put(1, 2)
    for b in want[:32767]:
        _fixed_lit(w, b)
    _fixed_lit(w, 285)
    w.huff(29, 5)
    w.put(32768 - 24577, 13)
    _fixed_lit(w, 256)
    bad = w.bytes()
    assert _zlib(bad) is None
    status, _ = _inflate(tool, tmp_path, bad, 65536)
    assert status == -11


def _bad_streams():
    """(name, stream): truncated, bit-flipped and invalid-code-length deflate streams."""
    rng = random.Random(17)
    inputs = _inputs()
    out = []
    for name in ('text_65280', 'incompressible', 'bam_like', 'repetitive'):
        for level in (0, 1, 6, 9):
            raw = _deflate(inputs[name], level)
            for cut in (1, 2, len(raw) // 3, len(raw) // 2, len(raw) - 1):
                out.append(('{}-{}-cut{}'.format(name, level, cut), raw[:cut]))
            for k in range(6):
                b = bytearray(raw)
                pos = rng.randrange(len(b))
                b[pos] ^= 1 << rng.randrange(8)
                out.append(('{}-{}-flip{}'.format(name, level, pos), bytes(b)))
    # dynamic block headers with invalid code lengths
    w = _Bits()                                      # code-length code over-subscribed: 19 lengths of 1
    w.put(1, 1)
    w.put(2, 2)
    w.put(0, 5)
    w.put(0, 5)
    w.put(15, 4)
    for _ in range(19):
        w.put(1, 3)
    out.append(('codelen-oversubscribed', w.bytes() + b'\0' * 8))
    w = _Bits()                                      # code-length code incomplete: a single length of 2
    w.put(1, 1)
    w.put(2, 2)
    w.put(0, 5)
    w.put(0, 5)
    w.put(0, 4)
    w.put(2, 3)
    for _ in range(3):
        w.put(0, 3)
    out.append(('codelen-incomplete', w.bytes() + b'\0' * 8))
    w = _Bits()                                      # 287 literal/length codes (at most 286)
    w.put(1, 1)
    w.put(2, 2)
    w.put(30, 5)
    w.put(0, 5)
    w.put(15, 4)
    out.append(('too-many-lengths', w.bytes() + b'\0' * 16))
    w = _Bits()                                      # literal/length lengths without an end-of-block code
    w.put(1, 1)
    w.put(2, 2)
    w.put(0, 5)                                      # 257 literal/length lengths
    w.put(0, 5)                                      # 1 distance length
    w.put(14, 4)                                     # 18 code-length lengths, in the order below
    order = [16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1]
    lens = {18: 1, 0: 2, 1: 2}                       # canonical codes: 18 -> 0, 0 -> 10, 1 -> 11
    for sym in order:
        w.put(lens.get(sym, 0), 3)
    codes = {18: (0, 1), 0: (2, 2), 1: (3, 2)}
    w.huff(*codes[1])                                # literals 0 and 1 get length 1
    w.huff(*codes[1])
    w.huff(*codes[18])
    w.put(138 - 11, 7)                               # 138 zeros
    w.huff(*codes[18])
    w.put(117 - 11, 7)                               # 117 zeros: symbol 256 (end of block) has no code
    w.huff(*codes[1])                                # the distance length
    out.append(('no-end-of-block', w.bytes() + b'\0' * 16))
    out.append(('block-type-3', bytes([0x07]) + b'\0' * 8))
    out.append(('stored-nlen', bytes([0x01, 0x05, 0x00, 0x00, 0x00]) + b'abcde'))
    return out


def _check_bad_streams(exe, tmp_path, env=None):
    n_err = 0
    for name, raw in _bad_streams():
        want = _zlib(raw)
        cap = 65536 if want is None else len(want)
        status, out = _inflate(exe, tmp_path, raw, cap, env=env)
        if want is None:
            assert status < 0, name                  # zlib rejects it: so does the decoder
            n_err += 1
        else:
            assert status == 0 and out == want, name     # a flip zlib decodes without complaint: the same bytes
    return n_err


def test_inflate_rejects_what_zlib_rejects(tool, tmp_path):
    n_err = _check_bad_streams(tool, tmp_path)
    assert n_err > 80                                # the truncations and the invalid code lengths at least


def test_inflate_under_asan_and_ubsan(tmp_path):
    exe = _build(tmp_path, 'address,undefined')
    env = dict(os.environ, ASAN_OPTIONS='detect_leaks=1 exitcode=66', UBSAN_OPTIONS='halt_on_error=1 exitcode=66')
    _check_bad_streams(exe, tmp_path, env=env)
    data = _inputs()['text_65280']
    status, out = _inflate(exe, tmp_path, _deflate(data, 9), len(data), env=env)
    assert status == 0 and out == data


def test_crc32_and_combine_match_zlib(tool, tmp_path):
    rng = np.random.default_rng(2)
    for n in (0, 1, 31, 32, 33, 1000, 65279, 65280, 65536):
        data = rng.integers(0, 256, n, dtype=np.uint8).tobytes()
        p = str(tmp_path / 'c.bin')
        with open(p, 'wb') as f:
            f.write(data)
        for pieces in (1, 7, 32):
            out = subprocess.run([tool, 'crc', p, str(pieces)], stdout=subprocess.PIPE, text=True, check=True).stdout
            whole, joined = (int(v) for v in out.split())
            assert whole == zlib.crc32(data) & 0xffffffff, n
            assert joined == whole, (n, pieces)


def _walk_blocks(raw):
    """Python walk of a BGZF file: (offset, BSIZE, ISIZE) of every block."""
    out, o = [], 0
    while o < len(raw):
        xlen = struct.unpack_from('<H', raw, o + 10)[0]
        e, bsize = 0, None
        while e + 4 <= xlen:
            si1, si2, slen = raw[o + 12 + e], raw[o + 13 + e], struct.unpack_from('<H', raw, o + 14 + e)[0]
            if si1 == ord('B') and si2 == ord('C') and slen == 2:
                bsize = struct.unpack_from('<H', raw, o + 16 + e)[0]
            e += 4 + slen
        isize = struct.unpack_from('<I', raw, o + bsize + 1 - 4)[0]
        out.append((o, bsize, isize))
        o += bsize + 1
    return out


def _scan(buf, at_eof, capacity=1 << 20):
    b = np.frombuffer(buf, dtype=np.uint8) if len(buf) else np.zeros(1, np.uint8)
    offs = np.zeros(capacity, np.int64)
    bsz = np.zeros(capacity, np.int32)
    isz = np.zeros(capacity, np.int32)
    consumed = np.zeros(1, np.int64)
    n = bam_io.lib.b3c_bgzf_scan(b.ctypes.data, len(buf), int(at_eof), offs.ctypes.data, bsz.ctypes.data,
                                 isz.ctypes.data, capacity, consumed.ctypes.data)
    if n < 0:
        return n, None, int(consumed[0])
    return n, list(zip(offs[:n].tolist(), bsz[:n].tolist(), isz[:n].tolist())), int(consumed[0])


def _community(rng, n_templates=3000):
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    from test_io import random_alignments
    refs = ['contig_{}'.format(i) for i in range(40)]
    lengths = [rng.choice([300, 800, 1500, 20000]) for _ in refs]
    return refs, lengths, random_alignments(rng, len(refs), n_templates)


@pytest.mark.parametrize('block_bytes,level', [(65280, 6), (4096, 1), (997, 6), (64, 0)])
def test_bgzf_scan_matches_a_python_walk(tmp_path, block_bytes, level):
    rng = random.Random(block_bytes)
    refs, lengths, alns = _community(rng, 1500)
    path = str(tmp_path / 'x.bam')
    bam_writer.write_bam(path, refs, lengths, alns, block_bytes=block_bytes, level=level)
    raw = open(path, 'rb').read()
    want = _walk_blocks(raw)
    n, got, consumed = _scan(raw, True)
    assert n == len(want) and got == want and consumed == len(raw)
    # the table the decoder is handed: the reader's block and byte counts
    with bam_io.BamPairReader(path, threads=2) as bam:
        bam.read_all()
        st = bam.stats()
    assert st['bgzf_blocks'] == n and st['compressed_bytes'] == len(raw)
    assert st['uncompressed_bytes'] == sum(i for _, _, i in got)
    # a buffer that ends inside a block: the scan stops before it, unless the file ends there
    for cut in (len(raw) // 2, len(raw) - 3, 5, 20):
        part = raw[:cut]
        k = sum(1 for o, b, _ in want if o + b + 1 <= cut)
        n2, got2, consumed2 = _scan(part, False)
        assert n2 == k and got2 == want[:k] and consumed2 == (want[k][0] if k < len(want) else len(raw))
        assert _scan(part, True)[0] == bam_io.B3C_IO_ERR_FORMAT
    # the block capacity ends a scan early
    n3, got3, consumed3 = _scan(raw, True, capacity=2)
    assert n3 == 2 and got3 == want[:2] and consumed3 == want[2][0]


def test_bgzf_scan_errors_match_the_reader(tmp_path):
    rng = random.Random(1)
    refs, lengths, alns = _community(rng, 300)
    good = str(tmp_path / 'good.bam')
    bam_writer.write_bam(good, refs, lengths, alns, block_bytes=4096)
    raw = open(good, 'rb').read()
    blocks = _walk_blocks(raw)
    bad_magic = bytearray(raw)
    bad_magic[blocks[3][0] + 1] ^= 0xff
    no_bc = bytearray(raw)
    no_bc[blocks[2][0] + 12] = ord('X')
    big_isize = bytearray(raw)
    o, b, _ = blocks[1]
    struct.pack_into('<I', big_isize, o + b + 1 - 4, 70000)
    for name, buf in (('magic', bytes(bad_magic)), ('bc', bytes(no_bc)), ('isize', bytes(big_isize)),
                      ('truncated', raw[:blocks[4][0] + 30])):
        n, _, _ = _scan(buf, True)
        p = str(tmp_path / (name + '.bam'))
        with open(p, 'wb') as f:
            f.write(buf)
        with pytest.raises(ValueError):                  # the host reader: B3C_IO_ERR_FORMAT -> ValueError
            with bam_io.BamPairReader(p) as bam:
                bam.read_all()
        assert n == bam_io.B3C_IO_ERR_FORMAT, name
        with pytest.raises(ValueError):
            bam_io.check(n)
    assert _scan(b'', True)[:2] == (0, [])


def test_data_offset_is_the_end_of_the_header(tmp_path):
    for n_refs in (0, 1, 40, 3000):
        refs = ['r{}'.format(i) for i in range(n_refs)]
        lengths = [1000 + i for i in range(n_refs)]
        path = str(tmp_path / 'h{}.bam'.format(n_refs))
        alns = [dict(name='q', flag=0x41, tid=0, pos=1, mapq=60, cigar=[(0, 50)])] if n_refs else []
        bam_writer.write_bam(path, refs, lengths, alns, block_bytes=1000)
        with bam_io.BamPairReader(path, threads=1) as bam:
            assert bam_io.lib.b3c_bam_data_offset(bam._h) == len(bam_writer.encode_header(refs, lengths))


def test_device_decoding_is_for_contig_records_only(tmp_path):
    """Extent and tip records are not decoded on the GPU: the call says so (and names the host reader) before it
    touches a device."""
    path = str(tmp_path / 'x.bam')
    bam_writer.write_bam(path, ['a', 'b'], [5000, 5000], [dict(name='q', flag=0x41, tid=0, pos=1, mapq=60, cigar=[(0, 50)])])
    for kw in (dict(bin_size=1000), dict(tip_size=500)):
        with pytest.raises(NotImplementedError, match='host reader'):
            bam_io.pair_records_from_bam(path, device=True, min_len=1000, **kw)
