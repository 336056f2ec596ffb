"""Host-side orchestration shared by the drop-in CLIs: BAM -> ReadBatch, barcode -> cell ids,
window pruning, per-GPU sharding (no collective), the BaseCellCounter TSV writer and the streamed BAM (stream_chunks)
under the counter (stream_count) and the genotype scripts (stream_genotype).

Reference counterparts: BaseCellCounter.main / run_interval / concatenate_sort_temp_files_and_write
(BaseCellCounter.py:22-79,182-320,344-409).  GPU selection cannot be a CLI flag (the Snakemake
rules stay unchanged), so it comes from the environment: LONGSOM_GPUS="0,1,2,3" or LONGSOM_GPUS=4.
"""
import ctypes as C
import os
import sys
import threading
import time

import numpy as np

from . import bamio
from .batch import ReadBatch, SiteCounts, Windows
from .engine import CountParams, Engine
from .sharding import balanced_window_shards

INFO_FIELD = "DP|NC|CC|BC|BQ|BCf|BCr"
COUNTER_CONCEPTS = (
    '##INFO=DP,Description="Depth of coverage">\n'
    '##INFO=NC,Description="Number of different cells">\n'
    '##INFO=CC,Description="Cell counts [A:C:T:G:I:D:N:O], where D means deletion, I insertion and O other type of character">\n'
    '##INFO=BC,Description="Base counts [A:C:T:G:I:D:N:O], where D means deletion, I insertion and O other type of character">\n'
    '##INFO=BQ,Description="Base quality sums [A:C:T:G:I:D:N:O], where D means deletion, I insertion and O other type of character">\n'
    '##INFO=BCf,Description="Base counts in forward reads [A:C:T:G:I:D:N:O], where D means deletion, I insertion and O other type of character">\n'
    '##INFO=BCr,Description="Base counts in reverse reads [A:C:T:G:I:D:N:O], where D means deletion, I insertion and O other type of character">'
)


def devices_from_env():
    v = os.environ.get("LONGSOM_GPUS", "").strip()
    if not v:
        return [0]
    if "," in v:
        return [int(x) for x in v.split(",") if x.strip() != ""]
    n = int(v)
    return list(range(n)) if n > 0 else [0]


def _parse_cpulist(text):
    cpus = set()
    for part in text.strip().split(","):
        if not part:
            continue
        a, _, b = part.partition("-")
        cpus.update(range(int(a), int(b or a) + 1))
    return cpus


def bind_near_gpu(device):
    """Pin this process to the CPUs of the NUMA node the GPU hangs off, so that the pinned staging buffers it
    allocates afterwards (first touch) and the threads that fill them sit next to the GPU's PCIe root.  One process
    per GPU (the bench's ranks, a CLI run on one device); a no-op when the platform does not say where the GPU is
    (numa_node = -1, no sysfs) or LONGSOM_NUMA=0.  Returns the node, or None."""
    if os.environ.get("LONGSOM_NUMA", "1") == "0" or not hasattr(os, "sched_setaffinity"):
        return None
    try:
        import ctypes
        from . import _lib
        buf = ctypes.create_string_buffer(64)   # CUDA ordinal -> PCI address (honours CUDA_VISIBLE_DEVICES)
        if _lib.load().ls_device_pci_bus_id(int(device), buf, 64) != 0:
            return None
        bus = buf.value.decode().strip().lower()
        if len(bus.split(":")[0]) == 8:   # an 8-digit PCI domain; sysfs uses 4 digits
            bus = bus[4:]
        with open("/sys/bus/pci/devices/%s/numa_node" % bus) as f:
            node = int(f.read().strip())
        if node < 0:
            return None
        with open("/sys/devices/system/node/node%d/cpulist" % node) as f:
            cpus = _parse_cpulist(f.read()) & os.sched_getaffinity(0)
        if not cpus:
            return None
        os.sched_setaffinity(0, cpus)
        return node
    except Exception:
        return None


# ---- CUDA context pre-warm ---------------------------------------------------------------------------------
# Creating a CUDA context on a 180 GB device takes about a second or more; the CLIs start it in a background
# thread before they decode the BAM (the native decoder releases the GIL), so the two overlap.
_WARM = {}
_WARM_LOCK = threading.Lock()


def prewarm(devices):
    """Start creating one Engine (CUDA context + stream) per device in the background."""
    def make(dev, box):
        try:
            box["engine"] = Engine(dev)
        except Exception as e:  # surfaced by take_engine
            box["error"] = e
    for dev in devices:
        box = {}
        t = threading.Thread(target=make, args=(dev, box), daemon=True)
        with _WARM_LOCK:
            _WARM.setdefault(dev, []).append((t, box))
        t.start()


def take_engine(dev):
    """An Engine for dev: the pre-warmed one if prewarm() was called, else a new one.  The caller closes it."""
    with _WARM_LOCK:
        entry = _WARM[dev].pop() if _WARM.get(dev) else None
    if entry is None:
        return Engine(dev)
    t, box = entry
    t.join()
    if "error" in box:
        raise box["error"]
    return box["engine"]


def read_ends(batch: ReadBatch):
    """Exclusive reference end of every read (pos + M/D/N/=/X lengths)."""
    if batch.n_reads == 0:
        return np.zeros(0, np.int64)
    op = batch.cigar & 15
    ln = np.where(np.isin(op, (0, 2, 3, 7, 8)), batch.cigar >> 4, 0).astype(np.int64)
    csum = np.concatenate([[0], np.cumsum(ln)])
    span = csum[batch.cigar_off[1:].astype(np.int64)] - csum[batch.cigar_off[:-1].astype(np.int64)]
    return batch.pos.astype(np.int64) + span


def read_keys(batch: ReadBatch, ends):
    """(start, end) keys tid << 32 | position of every read; the end is at least pos + 1, as the fetch of a pileup() call
    sees it (bam_endpos)."""
    tid = batch.tid.astype(np.int64) << 32
    pos = batch.pos.astype(np.int64)
    return tid | pos, tid | np.maximum(ends, pos + 1)


def clean_barcodes_split(raw):
    """BaseCellCounter / SingleCellGenotype: barcode = CB.split('-')[0] (BaseCellCounter.py:246)."""
    return [b.split("-")[0] for b in raw]


def dense_ids(strings):
    """Map a list of strings to dense ids in first-appearance order; returns (ids array, unique list)."""
    table, ids, uniq = {}, np.zeros(len(strings), np.int32), []
    for i, s in enumerate(strings):
        j = table.get(s)
        if j is None:
            j = len(uniq)
            table[s] = j
            uniq.append(s)
        ids[i] = j
    return ids, uniq


def prune_and_sort_windows(named_windows, bam_names, batch, ends):
    """named_windows: [(chrom, start, end)].  Keeps windows whose contig is in the BAM and that at least one
    read overlaps (others cannot emit a site); returns them as (tid, start, end) sorted by (tid, start)."""
    tid_of = {n: i for i, n in enumerate(bam_names)}
    iv = sorted((tid_of[c], s, e) for c, s, e in named_windows if c in tid_of and e > s)
    if not iv or batch.n_reads == 0:
        return []
    rk_lo, rk_hi = read_keys(batch, ends)
    run_max = np.maximum.accumulate(rk_hi)
    wk_lo = np.array([(t << 32) | s for t, s, e in iv], np.int64)
    wk_hi = np.array([(t << 32) | e for t, s, e in iv], np.int64)
    nb = np.searchsorted(rk_lo, wk_hi, side="left")
    covered = (nb > 0) & (run_max[np.maximum(nb - 1, 0)] > wk_lo)
    return [iv[j] for j in np.nonzero(covered)[0]]


def count_sites(batch, windows_iv, contig_seq, params: CountParams, devices=None, stats_out=None):
    """Pileup counts for windows_iv = [(tid, start, end)] (sorted, disjoint).  The windows are cut into
    coverage-balanced shards (array slices of the batch, no copies): one per device, or
    LONGSOM_SHARDS_PER_GPU per device, in which case each device runs two engine handles (own stream and buffers in the device's one CUDA context) so that uploads, kernels
    and result copies of its shards overlap.  Results are concatenated in window order."""
    devices = devices or [0]
    if not windows_iv:
        return SiteCounts.empty(0)
    per_gpu = max(1, int(os.environ.get("LONGSOM_SHARDS_PER_GPU", "1") or 1))
    win = Windows.from_intervals(windows_iv, contig_seq)
    if len(devices) == 1 and per_gpu == 1:
        with take_engine(devices[0]) as eng:
            res = eng.pileup_count(batch, win, params)
            if stats_out is not None:
                stats_out.append(dict(device=devices[0], **eng.last_stats))
        return res
    lanes = 2 if per_gpu > 1 else 1
    engines = [take_engine(dev) for dev in devices for _ in range(lanes)]
    try:
        res = count_shards_pipelined(window_shards(batch, win, len(devices) * per_gpu), params, None, engines=engines)
        if stats_out is not None:
            stats_out.extend(dict(device=e.device, **(e.last_stats or {})) for e in engines)
    finally:
        for e in engines:
            e.close()
    return SiteCounts(np.concatenate([r.tid for r in res]), np.concatenate([r.pos for r in res]),
                      np.concatenate([r.ref for r in res]), np.concatenate([r.counts for r in res], axis=0))


def window_shards(batch: ReadBatch, windows: Windows, n_shards):
    """Cut (batch, windows) into n_shards consecutive window groups of similar aligned-base weight.  Each shard
    gets the consecutive read range that can overlap its windows (reads are position-sorted; a read that spans a
    cut is in both shards and each shard only emits the sites of its own windows).  Array slices, no copies."""
    nw = windows.n_windows
    if nw == 0 or batch.n_reads == 0 or n_shards <= 1:
        return [(batch, windows)]
    rk_lo, rk_hi = read_keys(batch, read_ends(batch))
    rk_hi = np.maximum.accumulate(rk_hi)
    wk_lo = (windows.tid.astype(np.int64) << 32) | windows.start.astype(np.int64)
    wk_hi = (windows.tid.astype(np.int64) << 32) | windows.end.astype(np.int64)
    idx = np.minimum(np.searchsorted(wk_hi, rk_lo, side="right"), nw - 1)
    weight = np.zeros(nw)
    np.add.at(weight, idx, batch.l_qseq.astype(np.float64))
    out = []
    for lo, hi in balanced_window_shards(weight, n_shards):
        if hi <= lo:
            continue
        r_lo = int(np.searchsorted(rk_hi, wk_lo[lo], side="right"))   # first read whose running end passes the shard
        r_hi = int(np.searchsorted(rk_lo, wk_hi[hi - 1], side="left"))
        out.append((batch.slice(r_lo, max(r_lo, r_hi)), windows.slice(lo, hi)))
    return out


def count_shards_pipelined(shards, params: CountParams, outs, device=0, lanes=2, engines=None):
    """Runs ls_pileup_count() on every (batch, windows) shard, shard i on engine i mod len(engines), each engine
    (CUDA context; by default `lanes` of them on ONE device) in its own host thread: while one computes or copies
    results back, another uploads its next shard, so the PCIe transfers of a job overlap with each other (H2D /
    D2H are separate engines) and with the kernels.  With engines on several devices the same loop is the
    multi-GPU path.
    outs[i] (preallocated, e.g. pinned) receives shard i's sites and the per-shard site counts are returned; with
    outs=None each shard's SiteCounts is allocated after its run and the list of SiteCounts is returned."""
    own = engines is None
    engines = engines or [take_engine(device) for _ in range(max(1, lanes))]
    n_sites = [0] * len(shards)
    errors = []

    def work(e):
        try:
            for i in range(e, len(shards), len(engines)):
                if outs is None:
                    n_sites[i] = engines[e].pileup_count(shards[i][0], shards[i][1], params)
                else:
                    n_sites[i] = engines[e].pileup_count_e2e(shards[i][0], shards[i][1], params, outs[i])
        except Exception as ex:
            errors.append(ex)
    threads = [threading.Thread(target=work, args=(e,)) for e in range(len(engines))]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    if own:
        for eng in engines:
            eng.close()
    if errors:
        raise errors[0]
    return n_sites


# ---- streamed BAM: chunks -> pinned staging -> one worker per device -> results in chunk order ------------------------
class PinnedSlot:
    """One staging buffer set in pinned host memory (ls_host_alloc): the BAM decoder writes where the H2D copy reads.
    Arrays grow on demand and are reused for every chunk that goes through the slot.  Where the host refuses pinned
    memory (no CUDA device, or the locked-memory limit) an array is pageable, and the upload stages it through the
    driver's own pinned buffers."""
    FIELDS = (("tid", np.int32, "n"), ("pos", np.int32, "n"), ("flag", np.uint16, "n"), ("mapq", np.uint8, "n"),
              ("cell", np.int32, "n"), ("l_qseq", np.int32, "n"), ("cigar_off", np.uint32, "n1"),
              ("base_off", np.uint64, "n1"), ("cigar", np.uint32, "c"), ("seq4", np.uint8, "b2"), ("qual", np.uint8, "b"))

    def __init__(self):
        from . import _lib as L
        self.lib = L.load()
        self.arrays, self.ptrs, self.caps = {}, {}, {}

    def _alloc(self, name, dtype, count):
        if self.caps.get(name, 0) >= count:
            return
        if name in self.ptrs:
            self.lib.ls_host_free(self.ptrs.pop(name))
        want = int(count * 1.25) + 1024
        nbytes = want * np.dtype(dtype).itemsize
        p = C.c_void_p()
        self.caps[name] = want
        if self.lib.ls_host_alloc(C.c_size_t(nbytes), C.byref(p)) != 0:
            self.arrays[name] = np.empty(want, dtype)
            return
        self.ptrs[name] = p
        self.arrays[name] = np.frombuffer((C.c_uint8 * nbytes).from_address(p.value), dtype=dtype, count=want)

    def __call__(self, n, nc, nb):
        size = {"n": n, "n1": n + 1, "c": nc, "b": nb, "b2": nb // 2 + 1}
        for name, dtype, kind in self.FIELDS:
            self._alloc(name, dtype, size[kind])
        return self.arrays

    def free(self):
        for p in self.ptrs.values():
            self.lib.ls_host_free(p)
        self.arrays, self.ptrs, self.caps = {}, {}, {}


def _peak_rss_gb():
    """High-water mark of THIS process image (VmHWM).  ru_maxrss is no use here: it survives exec, so a child started
    by a large parent reports the parent's resident set."""
    try:
        with open("/proc/self/status") as f:
            for line in f:
                if line.startswith("VmHWM:"):
                    return int(line.split()[1]) / 1e6
    except OSError:
        pass
    import resource
    return resource.getrusage(resource.RUSAGE_SELF).ru_maxrss / 1e6


def plan_chunk(read_start, read_end, region_start, region_end, first_region, last):
    """One chunk of a streamed run.  read_start / read_end: read_keys() of the chunk's reads in coordinate order (the
    carried reads first); region_start / region_end: keys of the regions, sorted by start and disjoint, so that their
    ends are sorted too; first_region: the first region no earlier chunk completed; last: start key of the chunk's
    last read, or None when no mapped read follows.
    A region is complete once last >= its end: every later read starts at or after `last`, so none can overlap it.
    Returns (done, send, carry): regions [first_region, done) are complete; `send` indexes the reads that overlap one
    of them, which are all the records a fetch of those regions returns; `carry` indexes the reads whose end passes the
    start of region `done`, the first incomplete one, and which go in front of the next chunk."""
    nb = region_end.shape[0]
    done = nb if last is None else max(first_region, int(np.searchsorted(region_end, last, side="right")))
    # the first region from first_region on that ends after the read starts; regions are sorted, so it is the only
    # one to test
    j = np.maximum(np.searchsorted(region_end, read_start, side="right"), first_region)
    send = np.nonzero((j < done) & (region_start[np.minimum(j, max(nb - 1, 0))] < read_end))[0] if done > first_region \
        else np.zeros(0, np.int64)
    carry = np.nonzero(read_end > region_start[done])[0] if done < nb else np.zeros(0, np.int64)
    return done, send, carry


plan_genotype_chunk = plan_chunk  # the genotype scripts' name: their regions are the genotype_bins()


def stream_chunks(bam_path, region_start, region_end, devices, cell_map, run, chunk_bytes=None, make_engine=None):
    """Streams a coordinate-sorted BAM of any size through regions with bounded host memory.
      region_start, region_end : keys tid << 32 | position of the regions, as plan_chunk() takes them;
      cell_map    : barcode text of a CB tag -> cell id, or -1; read once per barcode, on the decoder thread;
      run         : run(engine, batch, ends, lo, done) -> result, for a chunk that completes regions [lo, done): batch
                    holds the reads that overlap them, with cell ids, and ends their exclusive reference ends;
      chunk_bytes : inflated BAM per chunk (default LONGSOM_CHUNK_MB, 256 MB);
      make_engine : device -> engine of a worker (default take_engine).
    A decoder thread fills len(devices) + 1 pinned slots in turn with the next chunk behind the reads carried from the
    previous one and plans it (plan_chunk).  One worker per entry of `devices`, each with its own engine, calls `run`.
    The reader is given the regions: where the BAM has a usable .bai it reads and inflates only the BGZF members the
    index lists for them (bamio.BamStream.set_regions), which hold every record that overlaps a region, in file order;
    plan_chunk drops the others.  Without one it reads the whole file.
    Yields (result, lo, done, stats) in chunk order; stats holds the device, n_reads (reads sent), n_carried (reads
    the chunk carried in), indexed (the .bai is used), compressed_bytes / inflated_bytes / decode_s (what the reader
    read and inflated, and the decoder thread's seconds, since the previous yielded chunk) and the engine's last_stats.  After the first error the workers only drain the queue, and
    the error is raised once every thread has stopped.  Closing the generator stops the stream the same way."""
    import queue
    devices = devices or [0]
    chunk_bytes = int(chunk_bytes or float(os.environ.get("LONGSOM_CHUNK_MB", "256")) * (1 << 20))
    bs = bamio.BamStream(bam_path)
    key_tid = (np.asarray(region_start, np.int64) >> 32).astype(np.int32)
    index_note = bs.set_regions(key_tid, np.asarray(region_start, np.int64) & 0xffffffff,
                                np.asarray(region_end, np.int64) & 0xffffffff)
    if index_note is not None and not index_note.startswith("no .bai"):
        print("[longsom] %s: index not used, reading the whole BAM: %s" % (bam_path, index_note), file=sys.stderr)
    slots = [PinnedSlot() for _ in range(len(devices) + 1)]
    free_slots, todo, done_q = queue.Queue(), queue.Queue(maxsize=len(slots)), queue.Queue()
    for sl in slots:
        free_slots.put(sl)
    errors, stop = [], threading.Event()

    def decoder():
        seq, lo, carry, carry_ends, cell_of_raw = 0, 0, None, None, np.zeros(0, np.int32)
        io_sent = (0, 0)  # reader bytes already reported with an earlier chunk
        decode_s = 0.0    # decoder seconds not yet reported with a chunk
        try:
            while lo < region_end.shape[0] and not errors and not stop.is_set():
                slot = free_slots.get()
                t0 = time.perf_counter()
                got = bs.next_chunk(chunk_bytes, slot, carry, carry_ends)
                if got is None:
                    free_slots.put(slot)
                    if carry is None:
                        break
                    slot, batch, ends, n_carried, last = None, carry, carry_ends, carry.n_reads, None
                else:
                    batch, n_new, ends = got
                    n_carried = batch.n_reads - n_new
                    # unplaced reads (tid -1) close a coordinate-sorted BAM: no mapped read follows them
                    last = None if batch.tid[-1] < 0 else (int(batch.tid[-1]) << 32) | int(batch.pos[-1])
                done, send, keep = plan_chunk(*read_keys(batch, ends), region_start, region_end, lo, last)
                carry, carry_ends = (batch.select(keep), ends[keep]) if keep.shape[0] else (None, None)
                if send.shape[0]:
                    sub = batch.slice(send[0], send[-1] + 1) if send[-1] - send[0] + 1 == send.shape[0] else batch.select(send)
                    if len(bs.barcodes) > cell_of_raw.shape[0]:  # the table grows as new CB texts appear
                        new = [cell_map(b) for b in bs.barcodes[cell_of_raw.shape[0]:]]
                        cell_of_raw = np.concatenate([cell_of_raw, np.array(new, np.int32)])
                    cell = np.full(sub.n_reads, -1, np.int32)
                    tagged = sub.cell >= 0
                    cell[tagged] = cell_of_raw[sub.cell[tagged]]
                    sub.cell = cell
                    io = (bs.compressed_bytes, bs.inflated_bytes)
                    decode_s += time.perf_counter() - t0
                    todo.put((seq, sub, ends[send], n_carried, lo, done, slot,
                              dict(indexed=index_note is None, compressed_bytes=io[0] - io_sent[0],
                                   inflated_bytes=io[1] - io_sent[1], decode_s=decode_s)))
                    io_sent, decode_s = io, 0.0
                    seq += 1
                else:
                    decode_s += time.perf_counter() - t0
                    if slot is not None:
                        free_slots.put(slot)
                lo = done
                if last is None:
                    break
        except Exception as ex:  # raised by the generator
            errors.append(ex)
        finally:
            for _ in devices:
                todo.put(None)

    def worker(dev):
        eng = None
        try:
            eng = (make_engine or take_engine)(dev)
        except Exception as ex:
            errors.append(ex)
        try:
            while True:
                item = todo.get()
                if item is None:
                    break
                seq, batch, ends, n_carried, lo, done, slot, io = item
                try:
                    if not errors and not stop.is_set():  # otherwise the queue is only drained: the decoder never blocks
                        res = run(eng, batch, ends, lo, done)
                        done_q.put((seq, (res, lo, done, dict(device=dev, n_reads=batch.n_reads, n_carried=n_carried,
                                                               **io, **eng.last_stats))))
                except Exception as ex:
                    errors.append(ex)
                finally:
                    if slot is not None:
                        free_slots.put(slot)
        finally:
            if eng is not None:
                eng.close()
            done_q.put(None)

    threads = [threading.Thread(target=decoder, daemon=True)] + [
        threading.Thread(target=worker, args=(d,), daemon=True) for d in devices]
    for t in threads:
        t.start()
    try:
        pending, want, live = {}, 0, len(devices)
        while live:
            item = done_q.get()
            if item is None:
                live -= 1
                continue
            pending[item[0]] = item[1]
            while want in pending and not errors:
                yield pending.pop(want)
                want += 1
        if errors:
            raise errors[0]
    finally:
        stop.set()
        for t in threads:
            t.join()
        for sl in slots:
            sl.free()
        bs.close()


def stream_count(bam_path, named_windows, fasta, params: CountParams, out_file, ID, devices=None, chunk_bytes=None,
                 stats_out=None):
    """BaseCellCounter over a BAM of any size with bounded host memory (reference: the per-window pool of
    BaseCellCounter.py:344-409).  The windows are the regions of stream_chunks: a chunk runs ls_pileup_count on those
    of its complete windows that a read reaches, and this thread appends the rows to one file per contig.  The rows are
    formatted on the device (Engine.pileup_count_text), or from the fetched counts by ls_write_counter_rows with
    LONGSOM_COUNTER_TEXT=host and for an engine without a text writer.  The table
    lists the contigs in NAME order (collect_result sorts the window files by name), the BAM delivers them in header
    order: a contig's file is appended to the table as soon as every contig before it in name order is complete, so at
    the end only the last few are left to copy.  Returns the number of sites written; stats_out, if given, receives
    the stats of every chunk."""
    import contextlib
    import shutil
    t_start = time.time()
    bs = bamio.BamStream(bam_path)  # the header only: stream_chunks decodes the reads
    names = bs.contig_names
    bs.close()
    tid_of = {n: i for i, n in enumerate(names)}
    win = sorted((tid_of[c], s, e) for c, s, e in named_windows if c in tid_of and e > s)
    order = sorted({t for t, _s, _e in win}, key=lambda t: names[t])
    fasta_lock = threading.Lock()
    busy = {"decode": 0.0, "device": 0.0, "text": 0.0, "writer": 0.0, "concat": 0.0}
    cells = {}  # cleaned barcode (CB.split('-')[0], BaseCellCounter.py:246) -> dense id in first-appearance order
    host_text = os.environ.get("LONGSOM_COUNTER_TEXT", "device") == "host"
    names_b = [n.encode() for n in names]

    def run(eng, batch, ends, lo, done):
        """The chunk's sites as SiteCounts (rows formatted by the writer) or, where the engine writes the rows itself,
        as (n_sites, {tid: text})."""
        t0 = time.time()
        iv = prune_and_sort_windows([(names[t], s, e) for t, s, e in win[lo:done]], names, batch, ends)
        with fasta_lock:
            contig_seq = {t: fasta.contig(names[t]) for t in sorted({w[0] for w in iv})}
        w = Windows.from_intervals(iv, contig_seq)
        if host_text or not hasattr(eng, "pileup_count_text"):  # (a stand-in engine has no text writer)
            res = eng.pileup_count(batch, w, params)
        else:
            text = eng.pileup_count_text(batch, w, params, names_b)
            res = (eng.last_stats["n_sites"], text)
            busy["text"] += eng.last_stats["text_s"]
            t0 += eng.last_stats["text_s"]
        busy["device"] += time.time() - t0
        return res

    parts, out, next_part, n_sites = {}, None, 0, 0

    def append_ready(complete_tid):
        """Appends the files of the contigs that come next in name order and lie before complete_tid in the BAM."""
        nonlocal out, next_part
        t0 = time.time()
        while next_part < len(order) and order[next_part] < complete_tid:
            path = parts.pop(order[next_part], None)
            next_part += 1
            if path is None:
                continue
            if out is None:
                out = open(out_file, "wb")
                out.write(("##fileDate=%s\n" % time.strftime("%d/%m/%Y")).encode())
                out.write((COUNTER_CONCEPTS + "\n").encode())
                out.write(("\t".join(["#CHROM", "POS", "REF", "INFO", str(ID)]) + "\n").encode())
                out.flush()
            with open(path, "rb") as f:
                left = os.fstat(f.fileno()).st_size
                try:  # in-kernel copy
                    while left > 0:
                        k = os.sendfile(out.fileno(), f.fileno(), None, min(left, 1 << 30))
                        if k <= 0:
                            break
                        left -= k
                except OSError:
                    pass
                if left > 0:
                    out.seek(0, os.SEEK_END)
                    shutil.copyfileobj(f, out, 1 << 24)
                    out.flush()
            os.remove(path)
        busy["concat"] += time.time() - t0

    wk_start = np.array([(t << 32) | s for t, s, e in win], np.int64)
    wk_end = np.array([(t << 32) | e for t, s, e in win], np.int64)
    cell_map = lambda b: cells.setdefault(b.split("-")[0], len(cells))
    try:
        with contextlib.closing(stream_chunks(bam_path, wk_start, wk_end, devices, cell_map, run, chunk_bytes)) as chunks:
            for res, _lo, done, stats in chunks:
                t0 = time.time()
                busy["decode"] += stats["decode_s"]
                if stats_out is not None:
                    stats_out.append(stats)
                if isinstance(res, SiteCounts):
                    n_sites += res.n_sites
                    for t in np.unique(res.tid).tolist():
                        path = parts.setdefault(t, "%s.part.%d.%d" % (out_file, os.getpid(), t))
                        write_counter_rows(path, names[t], res, t)
                else:
                    n_sites += res[0]
                    for t, text in res[1].items():
                        path = parts.setdefault(t, "%s.part.%d.%d" % (out_file, os.getpid(), t))
                        with open(path, "ab") as f:
                            f.write(text)
                busy["writer"] += time.time() - t0
                append_ready(win[done][0] if done < len(win) else len(names))
        if n_sites == 0:
            print("No temporary files found")
            return 0
        append_ready(len(names))
        out.close()
        out = None
        if os.environ.get("LS_STREAM_TIMING"):
            print("[stream_count] busy seconds: " + ", ".join("%s %.3f" % kv for kv in sorted(busy.items())) +
                  "; wall %.3f s; peak RSS of this process %.2f GB" % (time.time() - t_start, _peak_rss_gb()),
                  file=sys.stderr)
        return n_sites
    finally:
        for path in parts.values():
            if os.path.exists(path):
                os.remove(path)
        if out is not None:   # an error after the first contigs were appended: no partial table is left behind
            out.close()
            if os.path.exists(out_file):
                os.remove(out_file)


# ---- streaming genotype scripts: BAM chunks -> K1' + K2 per chunk -> touched pairs -----------------------------------
def genotype_bins(site_tid, site_pos, bin_size):
    """The pileup() calls of a genotype run as ls_genotype derives them from the sorted site table: one per run of sites
    with the same contig and floor(POS / bin_size) of the 1-based POS, over [first pos - 1, last pos + 1) (0-based).
    Returns (first, start, end): first[b] is the first site row of bin b and first[-1] the number of sites; start / end
    are the keys tid << 32 | position of the bin's region."""
    tid = np.asarray(site_tid, np.int64)
    pos = np.asarray(site_pos, np.int64)
    code = (pos + 1) // (bin_size if bin_size > 0 else 50000)
    new = np.ones(pos.shape[0], bool)
    new[1:] = (tid[1:] != tid[:-1]) | (code[1:] != code[:-1])
    first = np.append(np.nonzero(new)[0], pos.shape[0])
    lo, hi = first[:-1], first[1:] - 1
    return first, (tid[lo] << 32) | np.maximum(pos[lo] - 1, 0), (tid[hi] << 32) | (pos[hi] + 1)


def stream_genotype(bam_path, sites, bins, n_cells, cell_map, geno_params, alpha, beta, skip_p, devices, chunk_bytes=None,
                    stats_out=None, make_engine=None):
    """Touched (site, cell) pairs of SingleCellGenotype / HCCVSingleCellGenotype over a BAM of any size with bounded host
    memory: the same (site, cell, dp, alt, p) arrays, ordered by site, that one Engine.genotype_sparse call over the
    whole file returns.
      sites       : (site_tid, site_pos, alt_class), sorted and unique, tids of the BAM header;
      bins        : the bin size of the scripts' --bin; the pileup() calls are genotype_bins();
      cell_map    : barcode text of a CB tag -> column in [0, n_cells), or -1;
      geno_params : the other keyword arguments of genotype_sparse (min_bq, min_mq, max_depth, alt_only);
      skip_p      : per site, 1 where no tail is evaluated (None: none);
      chunk_bytes, make_engine : as stream_chunks takes them.
    The bins are the regions of stream_chunks: a chunk uploads the reads that overlap its complete bins and runs
    genotype_sparse on the contiguous slice of the site table those bins hold.  A chunk then holds every record the
    whole-file call fetches for those bins, in the same order, so the depth cap drops the same records.  Sites no read
    reaches get no pairs.  stats_out, if given, receives the stats of every chunk with its site rows [site_lo, site_hi)."""
    import contextlib
    site_tid, site_pos, alt_cls = (np.ascontiguousarray(a, t) for a, t in zip(sites, (np.int32, np.int32, np.uint8)))
    skip = None if skip_p is None else np.ascontiguousarray(skip_p, np.uint8)
    first, bstart, bend = genotype_bins(site_tid, site_pos, bins)
    empty = (np.zeros(0, np.int32),) * 4 + (np.zeros(0, np.float64),)
    if bend.shape[0] == 0:
        return empty

    def run(eng, batch, _ends, lo, done):
        lo, hi = int(first[lo]), int(first[done])
        eng.upload(batch, None)
        site, cell, dp, alt, p = eng.genotype_sparse(site_tid[lo:hi], site_pos[lo:hi], alt_cls[lo:hi], n_cells, alpha,
                                                     beta, skip_p=None if skip is None else skip[lo:hi], bin_size=bins,
                                                     **geno_params)
        site += lo  # chunk-local site rows -> rows of the whole table
        return site, cell, dp, alt, p

    parts = []
    with contextlib.closing(stream_chunks(bam_path, bstart, bend, devices, cell_map, run, chunk_bytes,
                                          make_engine)) as chunks:
        for tup, lo, done, stats in chunks:
            parts.append(tup)
            if stats_out is not None:
                stats_out.append(dict(stats, site_lo=int(first[lo]), site_hi=int(first[done])))
    if not parts:
        return empty
    # chunks cover disjoint, increasing site slices: in chunk order the pairs are ordered by (site, cell)
    return tuple(np.concatenate([p[k] for p in parts]) for k in range(5))


def format_counter_lines(chrom, pos, ref, counts):
    """TSV lines of BaseCellCounter.run_interval (:297-309) for one contig."""
    lines = []
    posl = (pos + 1).tolist()
    refl = ref.tobytes().decode("latin-1")
    c = counts.tolist()
    for i in range(len(posl)):
        r = c[i]
        cc, f, rv, bq = r[2:8], r[8:14], r[14:20], r[20:26]
        lines.append("%s\t%d\t%s\t%s\t%d|%d|%s|%s|%s|%s|%s\n" % (
            chrom, posl[i], refl[i], INFO_FIELD, r[0], r[1], ":".join(map(str, cc)),
            ":".join(str(a + b) for a, b in zip(f, rv)), ":".join(map(str, bq)), ":".join(map(str, f)),
            ":".join(map(str, rv))))
    return lines


def write_counter_tsv(out_file, ID, sites: SiteCounts, bam_names):
    """Final file of concatenate_sort_temp_files_and_write (:22-79): header, then window blocks ordered by
    (chrom lexicographic, start).  Returns False (and writes nothing) when no site passed, like the
    reference ('No temporary files found')."""
    if sites.n_sites == 0:
        print("No temporary files found")
        return False
    with open(out_file, "w") as out:
        out.write("##fileDate=%s\n" % time.strftime("%d/%m/%Y"))
        out.write(COUNTER_CONCEPTS + "\n")
        out.write("\t".join(["#CHROM", "POS", "REF", "INFO", str(ID)]) + "\n")
    for t in sorted(np.unique(sites.tid).tolist(), key=lambda t: bam_names[t]):
        write_counter_rows(out_file, bam_names[t], sites, t)
    return True


def write_counter_rows(path, chrom, sites: SiteCounts, tid):
    """Appends the TSV rows of contig `tid` to path with the native formatter (ls_write_counter_rows).  The rows of one
    contig are contiguous: sites are ordered by window = (tid, start)."""
    host = bamio._load_host()
    host.ls_write_counter_rows.argtypes = [C.c_char_p, C.c_char_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64,
                                           C.c_int, C.c_int]
    host.ls_write_counter_rows.restype = C.c_int
    lo, hi = int(np.searchsorted(sites.tid, tid, "left")), int(np.searchsorted(sites.tid, tid, "right"))
    pos = np.ascontiguousarray(sites.pos[lo:hi])
    ref = np.ascontiguousarray(sites.ref[lo:hi])
    cnt = np.ascontiguousarray(sites.counts[lo:hi])
    threads = min(16, len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1))
    rc = host.ls_write_counter_rows(os.fsencode(path), chrom.encode(), pos.ctypes.data, ref.ctypes.data, cnt.ctypes.data,
                                    hi - lo, threads, 1)
    if rc != 0:
        raise IOError("ls_write_counter_rows(%s) failed: %d" % (path, rc))


def load_bam_for_counting(bam_path, mode="split"):
    """Decode a BAM and map CB tags to dense cell ids.
    mode 'split': cell = CB.split('-')[0] (BaseCellCounter.py:246).  Returns (BamData, ReadBatch, cell names)."""
    bd = bamio.read_bam(bam_path)
    cleaned = clean_barcodes_split(bd.barcodes)
    ids, uniq = dense_ids(cleaned)
    return bd, bd.with_cells(ids), uniq
