"""
Two host slabs and one host thread that stream a file, so that the file I/O on one slab overlaps the device work on
the other.  The ring takes the slabs it is given (NumPy views of pinned tensors, or any arrays) and passes their
indices between the two threads, so a slab is in one thread's hands at a time.

Read-ahead (BAM decode, FASTA site counting), SlabRing(slabs, fill=...): the thread fills slab k while the caller
consumes slab k - 1.  fill(slab) returns a tuple whose last element is true for the stream's last slab.  Iterating
over the ring yields (k, that tuple) in stream order up to that slab; release(k) hands slab k back to be filled again.

Write-behind (the edge-file writer), SlabRing(slabs, drain=...): the caller fills slab k while the thread drains slab
k - 1.  acquire() gives the caller a free slab k, and release(k, nbytes) hands it to drain(slab, nbytes).

The ring is a context manager.  Leaving the block, normally or by an exception, lets the thread finish the slabs
already handed to it, then stops and joins it.  An exception raised in the thread is raised again in the caller, with
its type unchanged, at the caller's next call on the ring or at the end of the block.
"""
import queue
import threading


class SlabRing(object):
    def __init__(self, slabs, fill=None, drain=None):
        assert (fill is None) != (drain is None), 'a ring reads ahead (fill) or writes behind (drain)'
        self.slabs, self._fill, self._drain, self._error = slabs, fill, drain, None
        self._to_worker, self._to_caller = queue.Queue(), queue.Queue()
        for k in range(len(slabs)):                     # a free slab starts with the side that fills it
            if fill:
                self._to_worker.put((k, None))
            else:
                self._to_caller.put(k)
        self._worker = threading.Thread(target=self._run, name='slab-ring', daemon=True)

    def __enter__(self):
        self._worker.start()
        return self

    def __exit__(self, exc_type, exc, tb):
        self._to_worker.put(None)
        self._worker.join()
        if exc_type is None:
            self._raise_failure()

    def _run(self):
        try:
            for k, nbytes in iter(self._to_worker.get, None):
                if self._drain:
                    self._drain(self.slabs[k], nbytes)
                    self._to_caller.put(k)
                else:
                    item = self._fill(self.slabs[k])
                    self._to_caller.put((k, item))
                    if item[-1]:
                        return
        except BaseException as e:                      # raised again in the caller
            self._error = e
            self._to_caller.put(None)                   # wakes a caller waiting for a slab

    def _raise_failure(self):
        if self._error is not None:
            raise self._error

    def acquire(self):
        """The next slab from the thread: k with drain, (k, fill's tuple) with fill."""
        got = self._to_caller.get()
        self._raise_failure()
        return got

    def release(self, k, nbytes=None):
        """Hands slab k to the thread: to be filled again, or to drain its first nbytes."""
        self._raise_failure()
        self._to_worker.put((k, nbytes))

    def __iter__(self):
        last = False
        while not last:
            k, item = self.acquire()
            last = item[-1]
            yield k, item
