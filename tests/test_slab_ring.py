"""
bin3c_b200.slab_ring on the CPU: NumPy slabs, an in-memory source and sink.  Bytes round-trip exactly in both
directions, a slab is filled again only after the caller has handed it back, exceptions on either side reach the
caller with their type, and every case ends with the ring's thread joined.
"""
import io
import threading
import time

import numpy as np
import pytest

from bin3c_b200.slab_ring import SlabRing

SLAB_SIZES = [1, 7, 4096]
LENGTHS = ['0', '1', 'one slab', '3 slabs', '3 slabs + 1']


class FillError(Exception):
    pass


class DrainError(Exception):
    pass


class ConsumerError(Exception):
    pass


@pytest.fixture(autouse=True)
def no_thread_left():
    before = set(threading.enumerate())
    yield
    assert set(threading.enumerate()) == before


def _data(length, slab):
    n = {'0': 0, '1': 1, 'one slab': slab, '3 slabs': 3 * slab, '3 slabs + 1': 3 * slab + 1}[length]
    return np.random.default_rng(n + slab).integers(0, 256, n, dtype=np.uint8).tobytes()


def _reader(src, slabs, events):
    """fill(): readinto until the slab is full or at the end, as the FASTA reader does"""
    def fill(a):
        k = next(i for i, s in enumerate(slabs) if s is a)
        events.append(('fill', k))
        n = 0
        while n < len(a):
            m = src.readinto(memoryview(a)[n:])
            if not m:
                break
            n += m
        return n, n < len(a)
    return fill


def _wait_for_worker_to_end():
    for _ in range(2000):
        if not any(t.name == 'slab-ring' for t in threading.enumerate()):
            return
        time.sleep(0.005)
    raise AssertionError('the ring thread did not end')


@pytest.mark.parametrize('slab', SLAB_SIZES)
@pytest.mark.parametrize('length', LENGTHS)
def test_read_ahead_round_trip_and_hand_back(slab, length):
    data = _data(length, slab)
    slabs = [np.zeros(slab, dtype=np.uint8) for _ in range(2)]
    events, got, order = [], bytearray(), []
    with SlabRing(slabs, fill=_reader(io.BytesIO(data), slabs, events)) as ring:
        for k, (n, last) in ring:
            order.append(k)
            got += slabs[k][:n].tobytes()
            events.append(('release', k))
            ring.release(k)
    assert bytes(got) == data
    # one slab per full slab of data, then the short (possibly empty) last one, alternating between the two slabs
    n_slabs = len(data) // slab + 1
    assert order == [j % 2 for j in range(n_slabs)]
    fills = [k for e, k in events if e == 'fill']
    assert fills == order
    # slab k is filled for the j-th time only after the consumer has released it from its (j - 1)-th use
    for i, (e, k) in enumerate(events):
        if e == 'fill':
            fills_before = sum(1 for e2, k2 in events[:i] if e2 == 'fill' and k2 == k)
            releases_before = sum(1 for e2, k2 in events[:i] if e2 == 'release' and k2 == k)
            assert releases_before == fills_before, events


@pytest.mark.parametrize('slab', SLAB_SIZES)
@pytest.mark.parametrize('length', LENGTHS)
def test_write_behind_round_trip_and_hand_back(slab, length):
    data = _data(length, slab)
    slabs = [np.zeros(slab, dtype=np.uint8) for _ in range(2)]
    sink, events = io.BytesIO(), []

    def drain(a, nb):
        k = next(i for i, s in enumerate(slabs) if s is a)
        sink.write(memoryview(a)[:nb])
        events.append(('drained', k))

    with SlabRing(slabs, drain=drain) as ring:
        for lo in range(0, len(data), slab):
            k = ring.acquire()
            events.append(('acquired', k))
            piece = np.frombuffer(data[lo:lo + slab], dtype=np.uint8)
            slabs[k][:len(piece)] = piece
            ring.release(k, len(piece))
    assert sink.getvalue() == data
    acquired = [k for e, k in events if e == 'acquired']
    assert acquired == [j % 2 for j in range(len(acquired))]
    assert [k for e, k in events if e == 'drained'] == acquired
    # a slab is handed to the caller again only after its previous contents were drained
    for i, (e, k) in enumerate(events):
        if e == 'acquired':
            uses = sum(1 for e2, k2 in events[:i] if e2 == 'acquired' and k2 == k)
            assert sum(1 for e2, k2 in events[:i] if e2 == 'drained' and k2 == k) == uses, events


def test_one_slab_write_behind():
    sink = io.BytesIO()
    slabs = [np.zeros(3, dtype=np.uint8)]
    with SlabRing(slabs, drain=lambda a, nb: sink.write(memoryview(a)[:nb])) as ring:
        for piece in (b'abc', b'de', b'f'):
            k = ring.acquire()
            slabs[k][:len(piece)] = np.frombuffer(piece, dtype=np.uint8)
            ring.release(k, len(piece))
    assert sink.getvalue() == b'abcdef'


def test_fill_error_reaches_the_caller():
    slabs = [np.zeros(7, dtype=np.uint8) for _ in range(2)]
    calls = []

    def fill(a):
        calls.append(1)
        if len(calls) == 3:
            raise FillError('bad block in slab 3')
        return len(a), False

    with pytest.raises(FillError, match='slab 3'):
        with SlabRing(slabs, fill=fill) as ring:
            for k, _ in ring:
                ring.release(k)
    assert len(calls) == 3


def test_consumer_error_stops_the_reader():
    slabs = [np.zeros(7, dtype=np.uint8) for _ in range(2)]
    calls = []

    def fill(a):                                       # an endless stream: only the consumer can end it
        calls.append(1)
        return len(a), False

    with pytest.raises(ConsumerError):
        with SlabRing(slabs, fill=fill) as ring:
            for j, (k, _) in enumerate(ring):
                ring.release(k)
                if j == 1:
                    raise ConsumerError()
    assert len(calls) <= 4                             # two slabs filled, each refilled once at most


def test_caller_error_stops_the_writer_after_what_it_submitted():
    sink = io.BytesIO()
    slabs = [np.zeros(4, dtype=np.uint8) for _ in range(2)]
    with pytest.raises(ConsumerError):
        with SlabRing(slabs, drain=lambda a, nb: sink.write(memoryview(a)[:nb])) as ring:
            k = ring.acquire()
            slabs[k][:] = np.frombuffer(b'wxyz', dtype=np.uint8)
            ring.release(k, 4)
            raise ConsumerError()
    assert sink.getvalue() == b'wxyz'


@pytest.mark.parametrize('seen_at', ['acquire', 'release', 'close'])
def test_drain_error_reaches_the_caller(seen_at):
    slabs = [np.zeros(5, dtype=np.uint8) for _ in range(2)]
    go = threading.Event()

    def drain(a, nb):
        go.wait(10)
        raise DrainError('disk full')

    with pytest.raises(DrainError, match='disk full'):
        with SlabRing(slabs, drain=drain) as ring:
            ring.release(ring.acquire(), 5)
            k = ring.acquire()                         # the second slab was free all along
            go.set()
            if seen_at != 'close':
                _wait_for_worker_to_end()
                if seen_at == 'acquire':
                    ring.acquire()
                else:
                    ring.release(k, 5)
                raise AssertionError('the drain error was not raised at the next hand-over')
