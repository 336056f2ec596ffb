"""Text written on the device and copied out in blocks: two host blocks in flight, one filled by the device while the
other is consumed.  Shared by the genotype CLI (long table and matrices, written to files) and the counter
(Engine.pileup_count_text, whose per-contig text goes back to the streaming driver)."""
import ctypes as C
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np


def write_blocks(f, text, n, bufs, cap):
    """Units (rows or sites) 0 .. n-1 to file f in blocks: text(lo, addr, cap) formats as many whole units from lo as
    fit in cap bytes at addr and returns (units, bytes).  Block i is formatted into bufs[i] while the file thread still
    writes block i ^ 1.  Returns the seconds the file writes took."""
    def put(view):
        t = time.perf_counter()
        f.write(view)
        return time.perf_counter() - t
    spent, lo, i, pending = 0.0, 0, 0, None
    with ThreadPoolExecutor(1) as pool:
        while lo < n:
            units, nb = text(lo, bufs[i].addr, cap)
            if pending is not None:
                spent += pending.result()
            pending = pool.submit(put, bufs[i].view[:nb])
            lo += units
            i ^= 1
        if pending is not None:
            spent += pending.result()
    return spent


class PinnedBlock:
    """A block buffer in pinned host memory (pageable where the host refuses to pin it)."""

    def __init__(self, eng, nbytes):
        self._lib, self._ptr = eng._lib, C.c_void_p()
        self.nbytes = nbytes
        if self._lib.ls_host_alloc(C.c_size_t(nbytes), C.byref(self._ptr)) != 0:
            self._ptr, self._keep = None, C.create_string_buffer(nbytes)
            self.addr = C.addressof(self._keep)
        else:
            self.addr = self._ptr.value
        self.view = memoryview((C.c_char * nbytes).from_address(self.addr)).cast('B')

    def free(self):
        self.view.release()
        if self._ptr is not None:
            self._lib.ls_host_free(self._ptr)
            self._ptr = None


# the longest counter row besides its contig name: "\t" + 10 digits + "\t" + REF + the 24-byte INFO key, DP and NC
# (10 digits and a separator each) and five vectors of six 10-digit numbers with their separators
COUNTER_ROW_MAX = 1 + 11 + 1 + 24 + 22 + 5 * 66
COUNTER_BLOCK_BYTES = 16 << 20  # a chunk's text (~50 MB for 256 MB of BAM) in a few calls; pinning is paid once per engine


def counter_block_bytes(names):
    """Block size of the counter text: COUNTER_BLOCK_BYTES, or the longest possible row if that is longer."""
    return max(COUNTER_BLOCK_BYTES, max((len(x) for x in names), default=0) + COUNTER_ROW_MAX)


class _Into:
    """A file-like sink that copies the blocks into one array, back to back (numpy copies without the GIL)."""

    def __init__(self, nbytes):
        self.buf, self.n = np.empty(nbytes, np.uint8), 0  # pages past the text are never touched

    def write(self, view):
        k = len(view)
        self.buf[self.n:self.n + k] = np.frombuffer(view, np.uint8)
        self.n += k


def counter_text(eng, names, bufs):
    """The counter rows of the engine's last run as {tid: memoryview of the text}, each contig's rows in site order,
    formatted on the device (eng.pileup_text_load / eng.pileup_text) in blocks of whole rows through bufs (two blocks
    of equal size, each holding at least the longest possible row).  names: the contig names as bytes, indexed by tid."""
    lo, hi = eng.pileup_text_load(names)
    cap = bufs[0].nbytes
    out = {}
    for t in np.nonzero(hi > lo)[0].tolist():
        s0, s1 = int(lo[t]), int(hi[t])
        sink = _Into((s1 - s0) * (len(names[t]) + COUNTER_ROW_MAX))
        write_blocks(sink, lambda s, addr, n: eng.pileup_text(s0 + s, s1, addr, n), s1 - s0, bufs, cap)
        out[t] = memoryview(sink.buf[:sink.n])
    return out
