"""
The stage hand-off on the device (io_utils.save_object / load_object(device=True); include/bin3c_b200.h: b3c_bgzf_*):
the device members byte for byte against the g++ build of deflate.cuh (tests/native/deflate_check.cpp), files that
gzip reads back to pickle.dumps(obj) / dumps_stock(obj) and that do not change between runs or slab sizes, maps read
back by both loaders, the errors of the device loader, and the size against zlib level 6.
"""
import gzip
import os
import pickle
import sys
import zlib

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import bam_writer                                    # noqa: E402
import test_bgzf_deflate_cpu as cpu                  # noqa: E402
from bin3c_b200 import io_utils                      # noqa: E402
from test_io_utils import _host_map, _same_map       # noqa: E402

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def torch():
    t = pytest.importorskip('torch')
    if not t.cuda.is_available():
        pytest.skip('needs a CUDA device')
    return t


@pytest.fixture(scope='module')
def tool(tmp_path_factory):
    return cpu.build_tool(tmp_path_factory.mktemp('deflate'))


def _device_members(torch, data):
    import ctypes as C
    from bin3c_b200 import _cabi
    n = len(data)
    members = max(1, -(-n // io_utils.MEMBER_INPUT))
    ws = torch.empty(int(_cabi.lib.b3c_bgzf_deflate_workspace_bytes(members)), dtype=torch.uint8, device='cuda')
    d_in = torch.frombuffer(bytearray(data) or bytearray(1), dtype=torch.uint8).cuda()
    out = torch.empty(members * io_utils.MEMBER_MAX, dtype=torch.uint8, device='cuda')
    nbytes = C.c_int64()
    _cabi.check(_cabi.lib.b3c_bgzf_deflate(ws.data_ptr(), ws.numel(), d_in.data_ptr(), n, out.data_ptr(), out.numel(),
                                           C.byref(nbytes), C.c_void_p(torch.cuda.current_stream().cuda_stream)))
    return out[:nbytes.value].cpu().numpy().tobytes()


@pytest.mark.parametrize('name', sorted(cpu.CASES))
def test_device_members_equal_the_host_build(torch, tool, tmp_path, name):
    data = cpu.CASES[name]
    want, _ = cpu.encode(tool, tmp_path, data)
    got = _device_members(torch, data)
    if not data:
        assert got == b''                               # no member for an empty stream
        return
    assert got == want
    assert gzip.decompress(got + bam_writer.BGZF_EOF) == data


def _c1_map():
    from conftest import load_golden
    from bin3c_b200 import synth
    from bin3c_b200.contact_map import ContactMap, PairRecords
    g = load_golden('c1full')
    return ContactMap(PairRecords.from_community(synth.make_config('C1')), ['synthetic'], None, None, min_mapq=60,
                      min_len=int(g['min_len']), min_sig=int(g['min_sig']), random_seed=1)


def _bam_map(tmp_path):
    from bin3c_b200.contact_map import ContactMap
    rng = np.random.default_rng(77)
    n_refs = 60
    lengths = rng.integers(800, 5000, n_refs)
    names = ['ctg%03d' % i for i in range(n_refs)]
    alns = []
    for k in range(20_000):
        a = int(rng.integers(n_refs))
        b = a if rng.random() < 0.6 else int(rng.integers(n_refs))
        alns.append(dict(name='q%06d' % k, flag=0x41, tid=a, pos=int(rng.integers(0, 700)), mapq=60, cigar=[(0, 100)]))
        alns.append(dict(name='q%06d' % k, flag=0x81, tid=b, pos=int(rng.integers(0, 700)), mapq=60, cigar=[(0, 100)]))
    path = str(tmp_path / 'hic.bam')
    bam_writer.write_bam(path, names, lengths.tolist(), alns, block_bytes=40000, level=1)
    return ContactMap(path, ['MluCI'], np.ones(n_refs, dtype=np.int64), None, 60, min_len=1000, min_sig=2,
                      random_seed=1, gpu_decode=True)


MAPS = ['host', 'host_bins', 'c1', 'bam']


@pytest.fixture(scope='module')
def maps(tmp_path_factory):
    return {'host': _host_map(), 'host_bins': _host_map(bin_size=5000), 'c1': _c1_map(),
            'bam': _bam_map(tmp_path_factory.mktemp('bam'))}


@pytest.mark.parametrize('stock', [False, True])
@pytest.mark.parametrize('which', MAPS)
def test_save_writes_the_pickle(torch, tmp_path, maps, which, stock):
    cm = maps[which]
    raw = io_utils.dumps_stock(cm) if stock else pickle.dumps(cm, pickle.HIGHEST_PROTOCOL)
    p = str(tmp_path / 'contact_map.p')
    io_utils.save_object(p, cm, stock=stock, device=True)
    with open(p + '.gz', 'rb') as f:
        blob = f.read()
    assert blob.endswith(bam_writer.BGZF_EOF)
    assert gzip.decompress(blob) == raw
    ratio = len(blob) / len(zlib.compress(raw, 6))
    print('{} stock={}: {} pickle bytes, {} file bytes, {:.4f} x zlib level 6'.format(which, stock, len(raw),
                                                                                     len(blob), ratio))
    assert ratio <= 1.10
    for device in (False, True):
        back = io_utils.load_object(p + '.gz', device=device)
        if which.startswith('host'):
            _same_map(cm, back)
        else:
            assert np.array_equal(back.seq_map.toarray(), cm.seq_map.toarray())
            assert back.seq_info == cm.seq_info


def test_file_is_the_same_across_runs_and_slab_sizes(torch, tmp_path, maps):
    cm = maps['c1']
    raw = pickle.dumps(cm, pickle.HIGHEST_PROTOCOL)
    assert len(raw) > 7 * io_utils.MEMBER_INPUT
    files = []
    for k, slab in enumerate([None, None, 1, 7]):
        p = str(tmp_path / 'map{}.p'.format(k))
        io_utils.save_object(p, cm, device=True, slab_members=slab)
        with open(p + '.gz', 'rb') as f:
            files.append(f.read())
    assert all(f == files[0] for f in files)
    assert gzip.decompress(files[0]) == raw


def test_load_in_small_slabs(torch, tmp_path, maps):
    cm = maps['c1']
    p = str(tmp_path / 'contact_map.p')
    io_utils.save_object(p, cm, device=True)
    for slab in (1, 100_000, 1 << 20):
        back = io_utils.load_object(p + '.gz', device=True, slab_bytes=slab)
        assert np.array_equal(back.seq_map.toarray(), cm.seq_map.toarray())


def test_small_object_round_trips(torch, tmp_path):
    p = str(tmp_path / 'small')
    io_utils.save_object(p, {'a': 1}, device=True)
    assert io_utils.load_object(p + '.gz', device=True) == {'a': 1}
    assert io_utils.load_object(p + '.gz') == {'a': 1}


def test_loader_refuses_other_files(torch, tmp_path):
    p = str(tmp_path / 'host.p')
    io_utils.save_object(p, {'a': 1})                   # Python's gzip: no BC subfield
    with pytest.raises(ValueError, match='device=False'):
        io_utils.load_object(p + '.gz', device=True)
    plain = tmp_path / 'plain.p'
    plain.write_bytes(pickle.dumps({'a': 1}))
    with pytest.raises(ValueError, match='device=False'):
        io_utils.load_object(str(plain), device=True)


def test_loader_checks_crc_and_length(torch, tmp_path, maps):
    p = str(tmp_path / 'map.p')
    io_utils.save_object(p, maps['c1'], device=True)
    with open(p + '.gz', 'rb') as f:
        blob = bytearray(f.read())
    first = cpu.split_members(bytes(blob[:-len(bam_writer.BGZF_EOF)]))[0]
    bad = bytearray(blob)
    bad[len(first) - 8] ^= 0x01                         # the first member's CRC-32
    (tmp_path / 'crc.gz').write_bytes(bytes(bad))
    with pytest.raises(ValueError, match='CRC'):
        io_utils.load_object(str(tmp_path / 'crc.gz'), device=True)
    for cut in (len(blob) // 2, len(blob) - len(bam_writer.BGZF_EOF)):
        (tmp_path / 'cut.gz').write_bytes(bytes(blob[:cut]))
        with pytest.raises(ValueError):
            io_utils.load_object(str(tmp_path / 'cut.gz'), device=True)


def test_unwritable_path_raises_ioerror(torch, tmp_path):
    with pytest.raises(IOError):
        io_utils.save_object(str(tmp_path / 'no' / 'such' / 'dir' / 'map.p'), {'a': 1}, device=True)
