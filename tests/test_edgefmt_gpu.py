"""
The device edge-list writer (bin3c_b200/csrc/edgefmt.cu; bam_io.write_edges and cluster.write_edges with CUDA
tensors) against the host writer: the committed C1 edge files byte for byte in both float styles, millions of edges
of every weight class of tests/edge_cases.py at several chunk sizes, empty and one-edge lists, the end-to-end C1
contact map with and without device=True, and the errors.
"""
import ctypes as C
import gzip
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import edge_cases                                   # noqa: E402
from bin3c_b200 import bam_io, cluster              # noqa: E402

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(ROOT, 'tests', 'golden')
STYLES = (bam_io.FLOAT_REPR, bam_io.FLOAT_STR12)


@pytest.fixture(scope='module')
def torch():
    t = pytest.importorskip('torch')
    if not t.cuda.is_available():
        pytest.skip('needs a CUDA device')
    return t


def _cuda(torch, u, v, w):
    return (torch.from_numpy(np.ascontiguousarray(u, dtype=np.int32)).cuda(),
            torch.from_numpy(np.ascontiguousarray(v, dtype=np.int32)).cuda(),
            torch.from_numpy(np.ascontiguousarray(w, dtype=np.float64)).cuda())


def _host_text(tmp_path, u, v, w, sep, style):
    p = str(tmp_path / 'host.edges')
    n = bam_io.write_edges(u, v, w, p, sep=sep, float_style=style)
    data = open(p, 'rb').read()
    assert n == len(data)
    return data


def _device_text(tmp_path, du, dv, dw, sep, style, chunk=None):
    p = str(tmp_path / 'dev.edges')
    if chunk is None:
        n = bam_io.write_edges(du, dv, dw, p, sep=sep, float_style=style)
    else:
        n = bam_io._write_edges_on_device(du, dv, dw, p, sep=sep, float_style=style, chunk_edges=chunk)
    data = open(p, 'rb').read()
    assert n == len(data) == os.path.getsize(p)
    return data


def test_golden_c1_files_byte_for_byte(torch, tmp_path):
    raw = gzip.open(os.path.join(GOLDEN, 'c1_gpu.edges.gz'), 'rb').read()
    py2 = gzip.open(os.path.join(GOLDEN, 'c1_gpu_py2.edges.gz'), 'rb').read()
    rows = [line.split(b' ') for line in raw.split(b'\n')[:-1]]
    assert len(rows) == 34043
    u = np.array([int(r[0]) for r in rows], dtype=np.int32)
    v = np.array([int(r[1]) for r in rows], dtype=np.int32)
    w = np.array([float(r[2]) for r in rows])                 # repr weights read back exactly
    du, dv, dw = _cuda(torch, u, v, w)
    with open(cluster.write_edges(du, dv, dw, str(tmp_path), base_name='c1'), 'rb') as f:
        assert f.read() == raw
    with open(cluster.write_edges(du, dv, dw, str(tmp_path), base_name='c1_py2', py2_str=True), 'rb') as f:
        assert f.read() == py2


@pytest.fixture(scope='module')
def cases():
    u, v, w = edge_cases.edges(np.random.default_rng(7), 1_500_000)
    assert len(w) >= 3_000_000
    return u, v, w


@pytest.mark.parametrize('style', STYLES)
@pytest.mark.parametrize('sep', [' ', '\t'])
def test_random_edges_equal_host_writer(torch, tmp_path, cases, style, sep):
    u, v, w = cases
    du, dv, dw = _cuda(torch, u, v, w)
    want = _host_text(tmp_path, u, v, w, sep, style)
    assert _device_text(tmp_path, du, dv, dw, sep, style) == want
    assert _device_text(tmp_path, du, dv, dw, sep, style, chunk=4096) == want
    # one call per edge or per 7 edges: on the few hundred special edges of edge_cases, and a random 3000-edge prefix
    su, sv, sw = edge_cases.special_edges()
    m = 3000
    for hu, hv, hw in ((su, sv, sw), (u[:m], v[:m], w[:m])):
        small = _host_text(tmp_path, hu, hv, hw, sep, style)
        for chunk in (1, 7):
            assert _device_text(tmp_path, *_cuda(torch, hu, hv, hw), sep, style, chunk=chunk) == small


def test_other_dtypes_convert_as_the_host_writer(torch, tmp_path):
    rng = np.random.default_rng(3)
    u = rng.integers(0, 1 << 20, 10000)
    v = rng.integers(0, 1 << 20, 10000)
    w = rng.random(10000).astype(np.float32)
    want = _host_text(tmp_path, u, v, w, ' ', bam_io.FLOAT_REPR)
    got = _device_text(tmp_path, torch.from_numpy(u).cuda(), torch.from_numpy(v).cuda(), torch.from_numpy(w).cuda(),
                       ' ', bam_io.FLOAT_REPR)
    assert got == want


def test_empty_and_one_edge(torch, tmp_path):
    e = torch.empty(0, dtype=torch.int32, device='cuda')
    for style in STYLES:
        p = tmp_path / 'empty.edges'
        p.write_bytes(b'stale')
        assert bam_io.write_edges(e, e, e.double(), str(p), float_style=style) == 0
        assert p.read_bytes() == b''
        one = _cuda(torch, [3], [-7], [0.1])
        assert _device_text(tmp_path, *one, ' ', style) == _host_text(tmp_path, [3], [-7], [0.1], ' ', style)
    # the C ABI takes null pointers for no edges (a zero-length tensor reports a null address)
    from bin3c_b200 import _cabi
    nbytes = C.c_int64(-1)
    _cabi.check(_cabi.lib.b3c_edges_text(None, 0, None, None, None, 0, 32, 0, None, 0, C.byref(nbytes), None))
    assert nbytes.value == 0
    # too small a text buffer is an argument error
    du, dv, dw = _cuda(torch, [1, 2], [3, 4], [0.5, 0.25])
    ws = torch.empty(int(_cabi.lib.b3c_edges_text_workspace_bytes(2)), dtype=torch.uint8, device='cuda')
    text = torch.empty(97, dtype=torch.uint8, device='cuda')
    rc = _cabi.lib.b3c_edges_text(ws.data_ptr(), ws.numel(), du.data_ptr(), dv.data_ptr(), dw.data_ptr(), 2, 32, 0,
                                  text.data_ptr(), 97, C.byref(nbytes), None)
    assert rc == _cabi.B3C_ERR_ARG


@pytest.mark.parametrize('phase', [1, 3, 8, 15, 16])
def test_text_at_any_alignment(torch, tmp_path, phase):
    """b3c_edges_text writes d_text[0 .. bytes) at any address (a caller may append chunks into one buffer): the text
    equals the host writer's, and the guard bytes either side of it are untouched"""
    from bin3c_b200 import _cabi
    u, v, w = edge_cases.edges(np.random.default_rng(phase), 2000)
    u, v, w = u[:5000], v[:5000], w[:5000]                    # 20 blocks of 256 edges
    want = _host_text(tmp_path, u, v, w, ' ', bam_io.FLOAT_REPR)
    du, dv, dw = _cuda(torch, u, v, w)
    n = len(u)
    cap = _cabi.B3C_EDGES_MAX_LINE_BYTES * n
    ws = torch.empty(int(_cabi.lib.b3c_edges_text_workspace_bytes(n)), dtype=torch.uint8, device='cuda')
    buf = torch.full((cap + 64,), 0xA5, dtype=torch.uint8, device='cuda')
    nbytes = C.c_int64()
    _cabi.check(_cabi.lib.b3c_edges_text(ws.data_ptr(), ws.numel(), du.data_ptr(), dv.data_ptr(), dw.data_ptr(), n,
                                         32, bam_io.FLOAT_REPR, buf.data_ptr() + phase, cap, C.byref(nbytes),
                                         C.c_void_p(torch.cuda.current_stream().cuda_stream)))
    got = buf.cpu().numpy()
    assert nbytes.value == len(want)
    assert got[phase:phase + len(want)].tobytes() == want
    assert (got[:phase] == 0xA5).all() and (got[phase + len(want):] == 0xA5).all()


def test_end_to_end_c1_contact_map(torch, tmp_path):
    from conftest import load_golden
    from bin3c_b200 import synth
    from bin3c_b200.contact_map import ContactMap, PairRecords
    g = load_golden('c1full')
    cm = ContactMap(PairRecords.from_community(synth.make_config('C1')), ['synthetic'], None, None, min_mapq=60,
                    min_len=int(g['min_len']), min_sig=int(g['min_sig']), random_seed=1)
    du, dv, dw, _ = cluster.to_edges(cm, norm=True, bisto=True, scale=True, device=True)
    assert du.is_cuda and dw.is_cuda
    u, v, w, _ = cluster.to_edges(cm, norm=True, bisto=True, scale=True)
    for py2 in (False, True):
        fd = cluster.write_edges(du, dv, dw, str(tmp_path), base_name='dev', py2_str=py2)
        fh = cluster.write_edges(u, v, w, str(tmp_path), base_name='host', py2_str=py2)
        with open(fd, 'rb') as a, open(fh, 'rb') as b:
            assert a.read() == b.read()


def test_errors_then_exact(torch, tmp_path):
    u, v, w = edge_cases.edges(np.random.default_rng(11), 20000)
    du, dv, dw = _cuda(torch, u, v, w)
    p = str(tmp_path / 'e.edges')
    with pytest.raises(AssertionError):
        bam_io.write_edges(du, v, dw, p)
    with pytest.raises(AssertionError):
        bam_io.write_edges(u, v, dw, p)
    with pytest.raises(AssertionError):
        bam_io.write_edges(du, dv[:-1], dw, p)
    with pytest.raises(IOError):
        bam_io.write_edges(du, dv, dw, str(tmp_path / 'no' / 'such' / 'dir' / 'e.edges'))
    with pytest.raises(IOError):
        cluster.write_edges(du, dv, dw, str(tmp_path / 'missing'))
    for style in STYLES:
        assert _device_text(tmp_path, du, dv, dw, ' ', style, chunk=1000) == _host_text(tmp_path, u, v, w, ' ', style)
