"""
CPU side of the device edge-list writer: the formatting core bin3c_b200/csrc/edgefmt.cuh, built with g++ through
tests/native/edgefmt_check.cpp, against Python's repr(float), '%.12g' plus '.0' (tests/test_io.py::
test_format_weight_matches_python), bam_io.format_weight and the host writer's file in both float styles; the
power-of-5 table it uses against one regenerated from Python integers; and the argument checks of
bam_io.write_edges for CUDA tensors that come before any device work.
"""
import os
import shutil
import struct
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import edge_cases                                   # noqa: E402
from bin3c_b200 import bam_io                       # noqa: E402
from bin3c_b200.csrc import gen_edgefmt_pow5        # noqa: E402

SRC = os.path.join(ROOT, 'tests', 'native', 'edgefmt_check.cpp')
N_RANDOM = 2_100_000                                # per class: random bit patterns, uniform / log-uniform values


@pytest.fixture(scope='module')
def tool(tmp_path_factory):
    if shutil.which('g++') is None:
        pytest.skip('no g++')
    exe = str(tmp_path_factory.mktemp('edgefmt') / 'edgefmt_check')
    res = subprocess.run(['g++', '-std=c++17', '-O2', '-Wall', '-Werror', SRC, '-o', exe], stdout=subprocess.PIPE,
                         stderr=subprocess.STDOUT, text=True)
    assert res.returncode == 0, res.stdout
    return exe


@pytest.fixture(scope='module')
def cases():
    return edge_cases.edges(np.random.default_rng(20261021), N_RANDOM)


def _harness(tool, tmp_path, u, v, w, sep, style):
    src, out = tmp_path / 'in.bin', tmp_path / 'out.txt'
    with open(src, 'wb') as f:
        f.write(struct.pack('<qii', len(u), ord(sep), style))
        f.write(np.ascontiguousarray(u, dtype=np.int32).tobytes())
        f.write(np.ascontiguousarray(v, dtype=np.int32).tobytes())
        f.write(np.ascontiguousarray(w, dtype=np.float64).tobytes())
    res = subprocess.run([tool, str(src), str(out)], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True,
                         timeout=600)
    assert res.returncode == 0, res.stdout
    return out.read_bytes()


def _host(tmp_path, u, v, w, sep, style):
    p = str(tmp_path / 'host.edges')
    n = bam_io.write_edges(u, v, w, p, sep=sep, float_style=style)
    data = open(p, 'rb').read()
    assert n == len(data)
    return data


def _py2(x):
    t = '%.12g' % x
    if not ('.' in t or 'e' in t or 'n' in t):
        t += '.0'
    return t


@pytest.mark.parametrize('style', [bam_io.FLOAT_REPR, bam_io.FLOAT_STR12])
def test_lines_equal_host_writer_and_python(tool, tmp_path, cases, style):
    u, v, w = cases
    assert len(w) >= 4_000_000
    got = _harness(tool, tmp_path, u, v, w, ' ', style)
    assert got == _host(tmp_path, u, v, w, ' ', style)
    weights = [line.rsplit(' ', 1)[1] for line in got.decode('ascii').split('\n')[:-1]]
    assert len(weights) == len(w)
    py = repr if style == bam_io.FLOAT_REPR else _py2
    wl = w.tolist()
    bad = [(x, s) for x, s in zip(wl, weights) if s != py(x)]
    assert not bad, bad[:10]
    for x, s in zip(wl[:200000], weights):
        assert s == bam_io.format_weight(x, style), x


@pytest.mark.parametrize('sep', [' ', '\t', ';', '\x00', '\x7f'])
def test_ids_and_separators(tool, tmp_path, sep):
    rng = np.random.default_rng(ord(sep) + 7)
    ids = np.array(edge_cases.INT32_EDGES + [5, 99, 100, 999999999, 1000000000, -999999999, -1000000000],
                   dtype=np.int64)
    u = np.concatenate([np.repeat(ids, len(ids)), rng.integers(-2 ** 31, 2 ** 31, 5000)]).astype(np.int32)
    v = np.concatenate([np.tile(ids, len(ids)), rng.integers(0, 1 << 20, 5000)]).astype(np.int32)
    w = rng.random(len(u))
    w[::5] = 1.0
    for style in (bam_io.FLOAT_REPR, bam_io.FLOAT_STR12):
        assert _harness(tool, tmp_path, u, v, w, sep, style) == _host(tmp_path, u, v, w, sep, style)
    line = _harness(tool, tmp_path, [-2 ** 31], [-2 ** 31], [-2.2250738585072014e-308], sep, bam_io.FLOAT_REPR)
    assert len(line) == 49                          # the line bound B3C_EDGES_MAX_LINE_BYTES
    assert line == ('-2147483648{0}-2147483648{0}-2.2250738585072014e-308\n'.format(sep)).encode('ascii')


def test_special_edges(tool, tmp_path):
    u, v, w = edge_cases.special_edges()
    for style in (bam_io.FLOAT_REPR, bam_io.FLOAT_STR12):
        assert _harness(tool, tmp_path, u, v, w, ' ', style) == _host(tmp_path, u, v, w, ' ', style)


def test_empty_input(tool, tmp_path):
    assert _harness(tool, tmp_path, [], [], [], ' ', bam_io.FLOAT_REPR) == b''


def test_pow5_table_regenerated_from_python_integers():
    with open(gen_edgefmt_pow5.HEADER) as f:
        assert f.read() == gen_edgefmt_pow5.render()
    # spot checks of the definitions themselves
    assert gen_edgefmt_pow5.pow5_split(0) == 1 << 124
    assert gen_edgefmt_pow5.pow5_split(341) == 5 ** 341 >> ((5 ** 341).bit_length() - 125)
    for i in (0, 1, 27, 28, 100, 297, 341):
        p, x = 5 ** i, gen_edgefmt_pow5.pow5_inv_split(i)
        t = p.bit_length() - 1 + 125
        assert (x - 1) * p <= 1 << t < x * p


class _FakeCuda(object):
    """stands for a CUDA tensor: the checks below must fail before anything touches it"""
    is_cuda = True

    def __init__(self, n):
        self.n = n

    def __len__(self):
        return self.n

    def __getattr__(self, name):
        raise AssertionError('device work started ({})'.format(name))


def test_device_argument_errors_come_first(tmp_path):
    pytest.importorskip('torch')
    p = tmp_path / 'never.edges'
    host = np.zeros(3)
    with pytest.raises(AssertionError, match='all CUDA tensors or all host arrays'):
        bam_io.write_edges(_FakeCuda(3), host.astype(np.int32), host, str(p))
    with pytest.raises(AssertionError, match='all CUDA tensors or all host arrays'):
        bam_io.write_edges(host.astype(np.int32), host.astype(np.int32), _FakeCuda(3), str(p))
    with pytest.raises(AssertionError):
        bam_io.write_edges(_FakeCuda(3), _FakeCuda(3), _FakeCuda(4), str(p))
    with pytest.raises(AssertionError, match='single-character separator'):
        bam_io.write_edges(_FakeCuda(3), _FakeCuda(3), _FakeCuda(3), str(p), sep='ab')
    with pytest.raises(AssertionError, match='float_style'):
        bam_io.write_edges(_FakeCuda(3), _FakeCuda(3), _FakeCuda(3), str(p), float_style=2)
    assert not p.exists()
