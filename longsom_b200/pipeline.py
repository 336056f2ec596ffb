"""Host-side orchestration shared by the drop-in CLIs: BAM -> ReadBatch, barcode -> cell ids,
window pruning, per-GPU sharding (no collective), the BaseCellCounter TSV writer and the streamed BAM sources of
the counter (stream_count) and of the genotype scripts (stream_genotype).

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
    rk_lo = (batch.tid.astype(np.int64) << 32) | batch.pos.astype(np.int64)
    rk_hi = (batch.tid.astype(np.int64) << 32) | np.maximum(ends, batch.pos.astype(np.int64) + 1)
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
    ends = read_ends(batch)
    rk_lo = (batch.tid.astype(np.int64) << 32) | batch.pos.astype(np.int64)
    rk_hi = np.maximum.accumulate((batch.tid.astype(np.int64) << 32) | np.maximum(ends, batch.pos.astype(np.int64) + 1))
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


# ---- streaming BaseCellCounter: BAM chunks -> pinned staging -> GPU -> per-contig row files ---------------------------
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


def stream_count(bam_path, named_windows, fasta, params: CountParams, out_file, ID, devices=None, chunk_bytes=None,
                 stats_out=None):
    """BaseCellCounter over a BAM of any size with bounded host memory (reference: the per-window pool of
    BaseCellCounter.py:344-409).  Three stages run concurrently:
      decoder : next ~chunk_bytes of the BAM -> pinned slot (behind the reads carried over from the previous chunk);
                decides which windows are COMPLETE (no later read can reach them: reads are coordinate sorted) and which
                reads must be carried on because they overlap a window that is not;
      device  : ls_pileup_count on (carried + chunk reads, complete windows), one chunk per engine at a time;
      writer  : native TSV rows appended to one file per contig; the files are concatenated in the reference's order
                (contig name, start) at the end.
    Returns the number of sites written."""
    import queue
    import shutil
    devices = devices or [0]
    chunk_bytes = int(chunk_bytes or float(os.environ.get("LONGSOM_CHUNK_MB", "256")) * (1 << 20))
    bs = bamio.BamStream(bam_path)
    tid_of = {n: i for i, n in enumerate(bs.contig_names)}
    win = sorted((tid_of[c], s, e) for c, s, e in named_windows if c in tid_of and e > s)
    wk_end = np.array([(t << 32) | e for t, s, e in win], np.int64)
    wk_start = np.array([(t << 32) | s for t, s, e in win], np.int64)
    n_slots = len(devices) + 1
    free_slots = queue.Queue()
    slots = [PinnedSlot() for _ in range(n_slots)]
    for sl in slots:
        free_slots.put(sl)
    todo, done = queue.Queue(maxsize=n_slots), queue.Queue()
    errors = []
    fasta_lock = threading.Lock()
    busy = {"decode": 0.0, "host_glue": 0.0, "device": 0.0, "writer": 0.0}
    clean_map = {"ids": np.zeros(0, np.int32), "table": {}, "names": []}

    def cell_ids(raw, barcodes):
        """raw barcode ids of the stream -> dense ids of cleaned barcodes (CB.split('-')[0], BaseCellCounter.py:246)."""
        ids = clean_map["ids"]
        if len(barcodes) > ids.shape[0]:
            new = np.zeros(len(barcodes), np.int32)
            new[:ids.shape[0]] = ids
            for i in range(ids.shape[0], len(barcodes)):
                c = barcodes[i].split("-")[0]
                j = clean_map["table"].get(c)
                if j is None:
                    j = len(clean_map["names"])
                    clean_map["table"][c] = j
                    clean_map["names"].append(c)
                new[i] = j
            clean_map["ids"] = ids = new
        out = np.full(raw.shape[0], -1, np.int32)
        m = raw >= 0
        out[m] = ids[raw[m]]
        return out

    def decoder():
        try:
            wi, seq, carry, carry_ends = 0, 0, None, None
            while True:
                slot = free_slots.get()
                t_a = time.time()
                got = bs.next_chunk(chunk_bytes, slot, carry, carry_ends)
                busy["decode"] += time.time() - t_a
                t_a = time.time()
                if got is None:
                    free_slots.put(slot)
                    batch, last, ends = carry, None, carry_ends
                    if batch is None or batch.n_reads == 0 or wi >= len(win):
                        break
                    slot = None
                else:
                    batch, _n_new, ends = got
                    last = (int(batch.tid[-1]) << 32) | int(batch.pos[-1])
                # windows no future read can overlap: every later read starts at or after `last`
                wj = len(win) if last is None else int(np.searchsorted(wk_end, last, side="right"))
                wj = max(wj, wi)
                rk_end = (batch.tid.astype(np.int64) << 32) | np.maximum(ends, batch.pos.astype(np.int64) + 1)
                if wj > wi:
                    iv = prune_and_sort_windows([(bs.contig_names[t], s, e) for t, s, e in win[wi:wj]], bs.contig_names, batch, ends)
                    if iv:
                        b2 = ReadBatch(batch.tid, batch.pos, batch.flag, batch.mapq, cell_ids(batch.cell, bs.barcodes),
                                       batch.cigar_off, batch.cigar, batch.base_off, batch.l_qseq, batch.seq4, batch.qual)
                        todo.put((seq, b2, iv, slot, win[wj][0] if wj < len(win) else (1 << 30)))
                        seq += 1
                        slot_in_use = True
                    else:
                        slot_in_use = False
                else:
                    slot_in_use = False
                wi = wj
                if last is None:
                    if slot is not None and not slot_in_use:
                        free_slots.put(slot)
                    break
                # reads that overlap a window which is not complete yet travel with the next chunk
                if wi < len(win):
                    keep = np.nonzero(rk_end > wk_start[wi])[0]
                    carry = batch.select(keep) if keep.shape[0] else None
                    carry_ends = ends[keep] if keep.shape[0] else None
                else:
                    carry, carry_ends = None, None
                if not slot_in_use:
                    free_slots.put(slot)
                busy["host_glue"] += time.time() - t_a
                if wi >= len(win):
                    break
        except Exception as ex:  # surfaced by the caller
            errors.append(ex)
        finally:
            for _ in devices:
                todo.put(None)

    def device_worker(dev):
        try:
            eng = take_engine(dev)
            try:
                while True:
                    item = todo.get()
                    if item is None:
                        break
                    seq, batch, iv, slot, complete_tid = item
                    t_a = time.time()
                    with fasta_lock:
                        contig_seq = {t: fasta.contig(bs.contig_names[t]) for t in sorted({w[0] for w in iv})}
                    w = Windows.from_intervals(iv, contig_seq)
                    sites = eng.pileup_count(batch, w, params)
                    if stats_out is not None:
                        stats_out.append(dict(device=dev, **eng.last_stats))
                    if slot is not None:
                        free_slots.put(slot)
                    busy["device"] += time.time() - t_a
                    done.put((seq, sites, complete_tid))
            finally:
                eng.close()
        except Exception as ex:
            errors.append(ex)
        finally:
            done.put(None)

    threads = [threading.Thread(target=decoder, daemon=True)] + [threading.Thread(target=device_worker, args=(d,), daemon=True)
                                                                 for d in devices]
    for t in threads:
        t.start()
    # writer (this thread): chunks in sequence order, rows appended to one temporary file per contig
    host = bamio._load_host()
    host.ls_write_counter_rows.argtypes = [C.c_char_p, C.c_char_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64,
                                           C.c_int, C.c_int]
    host.ls_write_counter_rows.restype = C.c_int
    parts, pending, want, live, n_sites = {}, {}, 0, len(devices), 0
    nthreads = min(16, len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1))
    # The table lists the contigs in NAME order (collect_result sorts the window files by name), the BAM delivers them
    # in header order: rows go to one part file per contig, and a part is appended to the output as soon as every
    # contig before it in name order is complete -- at the end only the last few contigs are left to copy.
    order = sorted({t for t, _s, _e in win}, key=lambda t: bs.contig_names[t])
    state = {"out": None, "next": 0, "complete_tid": -1}
    busy["concat"] = 0.0

    def append_ready(everything=False):
        t_cat = time.time()
        while state["next"] < len(order) and (everything or order[state["next"]] < state["complete_tid"]):
            t = order[state["next"]]
            state["next"] += 1
            path = parts.pop(t, None)
            if path is None:
                continue
            if state["out"] is None:
                state["out"] = open(out_file, "wb")
                state["out"].write(("##fileDate=%s\n" % time.strftime("%d/%m/%Y")).encode())
                state["out"].write((COUNTER_CONCEPTS + "\n").encode())
                state["out"].write(("\t".join(["#CHROM", "POS", "REF", "INFO", str(ID)]) + "\n").encode())
                state["out"].flush()
            out = state["out"]
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
        busy["concat"] += time.time() - t_cat

    while live:
        item = done.get()
        if item is None:
            live -= 1
            continue
        pending[item[0]] = (item[1], item[2])
        t_w = time.time()
        while want in pending:
            sites, complete_tid = pending.pop(want)
            want += 1
            n_sites += sites.n_sites
            for t in np.unique(sites.tid).tolist():
                lo, hi = int(np.searchsorted(sites.tid, t, "left")), int(np.searchsorted(sites.tid, t, "right"))
                path = parts.setdefault(t, "%s.part.%d.%d" % (out_file, os.getpid(), t))
                pos = np.ascontiguousarray(sites.pos[lo:hi])
                ref = np.ascontiguousarray(sites.ref[lo:hi])
                cnt = np.ascontiguousarray(sites.counts[lo:hi])
                rc = host.ls_write_counter_rows(os.fsencode(path), bs.contig_names[t].encode(), pos.ctypes.data, ref.ctypes.data,
                                                cnt.ctypes.data, hi - lo, nthreads, 1)
                if rc != 0:
                    errors.append(IOError("ls_write_counter_rows(%s) failed: %d" % (path, rc)))
            state["complete_tid"] = max(state["complete_tid"], complete_tid)
            if not errors:
                append_ready()
        busy["writer"] += time.time() - t_w
    for t in threads:
        t.join()
    for sl in slots:
        sl.free()
    bs.close()
    try:
        if errors:
            raise errors[0]
        if n_sites == 0:
            print("No temporary files found")
            return 0
        append_ready(everything=True)
        if state["out"] is not None:
            state["out"].close()
            state["out"] = None
        if os.environ.get("LS_STREAM_TIMING"):
            import resource
            print("[stream_count] busy seconds: " + ", ".join("%s %.2f" % kv for kv in sorted(busy.items())) +
                  "; peak RSS of this process %.2f GB" % _peak_rss_gb(), file=sys.stderr)
            if os.environ.get("LS_STREAM_TIMING") == "2":   # what the resident set is made of (largest mappings)
                try:
                    maps, cur = [], None
                    with open("/proc/self/smaps") as f:
                        for line in f:
                            if "-" in line.split(" ", 1)[0] and ":" not in line.split(" ", 1)[0]:
                                cur = line.split()
                            elif line.startswith("Rss:") and cur is not None:
                                maps.append((int(line.split()[1]), cur[5] if len(cur) > 5 else "[anon]", cur[0]))
                    maps.sort(reverse=True)
                    print("[stream_count] largest resident mappings (MB): " +
                          "; ".join("%d %s" % (kb // 1024, name) for kb, name, _ in maps[:10]), file=sys.stderr)
                except OSError:
                    pass
        return n_sites
    finally:
        for path in parts.values():
            if os.path.exists(path):
                os.remove(path)
        if state["out"] is not None:   # an error after the first contigs were appended: no partial table is left behind
            state["out"].close()
            if os.path.exists(out_file):
                os.remove(out_file)


# ---- streaming genotype scripts: BAM chunks -> pinned staging -> K1' + K2 per chunk -> touched pairs ------------------
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


def read_keys(batch: ReadBatch, ends):
    """(start, end) keys tid << 32 | position of every read; the end is at least pos + 1, as the fetch of a pileup() call
    sees it (bam_endpos)."""
    tid = batch.tid.astype(np.int64) << 32
    pos = batch.pos.astype(np.int64)
    return tid | pos, tid | np.maximum(ends, pos + 1)


def plan_genotype_chunk(read_start, read_end, bin_start, bin_end, first_bin, last):
    """One chunk of a streamed genotype run.  read_start / read_end: read_keys() of the chunk's reads in coordinate
    order (the carried reads first); bin_start / bin_end: region keys of genotype_bins(); first_bin: the first bin no
    earlier chunk completed; last: start key of the chunk's last read, or None when no mapped read follows.
    A bin is complete once last >= its end: every later read starts at or after `last`, so none can overlap it.
    Returns (done, send, carry): bins [first_bin, done) are complete; `send` indexes the reads that overlap one of
    them, which are all the records their pileup() calls fetch; `carry` indexes the reads whose end passes the start of
    bin `done`, the first incomplete one, and which go in front of the next chunk."""
    nb = bin_end.shape[0]
    done = nb if last is None else max(first_bin, int(np.searchsorted(bin_end, last, side="right")))
    # the first bin from first_bin on that ends after the read starts; bins are sorted, so it is the only one to test
    j = np.maximum(np.searchsorted(bin_end, read_start, side="right"), first_bin)
    send = np.nonzero((j < done) & (bin_start[np.minimum(j, max(nb - 1, 0))] < read_end))[0] if done > first_bin \
        else np.zeros(0, np.int64)
    carry = np.nonzero(read_end > bin_start[done])[0] if done < nb else np.zeros(0, np.int64)
    return done, send, carry


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
      chunk_bytes : inflated BAM per chunk (default LONGSOM_CHUNK_MB, 256 MB);
      make_engine : device -> engine of a worker (default take_engine).
    A decoder thread fills pinned slots with the next chunk behind the reads carried from the previous one and plans it
    (plan_genotype_chunk).  One worker per entry of `devices`, each with its own engine, uploads the reads that overlap
    the chunk's complete bins and runs genotype_sparse on the contiguous slice of the site table those bins hold.  A
    chunk then holds every record the whole-file call fetches for those bins, in the same order, so the depth cap drops
    the same records.  Sites no read reaches get no pairs.  stats_out, if given, receives one dict per device call."""
    import queue
    site_tid, site_pos, alt_cls = (np.ascontiguousarray(a, t) for a, t in zip(sites, (np.int32, np.int32, np.uint8)))
    skip = None if skip_p is None else np.ascontiguousarray(skip_p, np.uint8)
    first, bstart, bend = genotype_bins(site_tid, site_pos, bins)
    empty = (np.zeros(0, np.int32),) * 4 + (np.zeros(0, np.float64),)
    if bend.shape[0] == 0:
        return empty
    devices = devices or [0]
    chunk_bytes = int(chunk_bytes or float(os.environ.get("LONGSOM_CHUNK_MB", "256")) * (1 << 20))
    bs = bamio.BamStream(bam_path)
    slots = [PinnedSlot() for _ in range(len(devices) + 1)]
    free_slots = queue.Queue()
    for sl in slots:
        free_slots.put(sl)
    todo, done_q = queue.Queue(maxsize=len(slots)), queue.Queue()
    errors = []
    columns = {"of_raw": np.zeros(0, np.int32)}

    def to_columns(raw):
        """raw barcode ids of the stream -> columns; the table grows as new CB texts appear."""
        old = columns["of_raw"]
        if len(bs.barcodes) > old.shape[0]:
            columns["of_raw"] = np.concatenate([old, np.array([cell_map(b) for b in bs.barcodes[old.shape[0]:]], np.int32)])
        out = np.full(raw.shape[0], -1, np.int32)
        m = raw >= 0
        out[m] = columns["of_raw"][raw[m]]
        return out

    def decoder():
        seq = 0
        try:
            bi, carry, carry_ends = 0, None, None
            while bi < bend.shape[0] and not errors:
                slot = free_slots.get()
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
                rs, re_ = read_keys(batch, ends)
                bj, send, keep = plan_genotype_chunk(rs, re_, bstart, bend, bi, last)
                carry, carry_ends = (batch.select(keep), ends[keep]) if keep.shape[0] else (None, None)
                if send.shape[0]:
                    sub = batch.slice(send[0], send[-1] + 1) if send[-1] - send[0] + 1 == send.shape[0] else batch.select(send)
                    sub.cell = to_columns(sub.cell)
                    todo.put((seq, sub, int(first[bi]), int(first[bj]), slot, n_carried))
                    seq += 1
                elif slot is not None:
                    free_slots.put(slot)
                bi = bj
                if last is None:
                    break
        except Exception as ex:  # surfaced by the caller
            errors.append(ex)
        finally:
            for _ in devices:
                todo.put(None)

    def device_worker(dev):
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
                seq, batch, lo, hi, slot, n_carried = item
                try:
                    if not errors:  # after an error the queue is only drained, so that the decoder never blocks
                        eng.upload(batch, None)
                        site, cell, dp, alt, p = eng.genotype_sparse(
                            site_tid[lo:hi], site_pos[lo:hi], alt_cls[lo:hi], n_cells, alpha, beta,
                            skip_p=None if skip is None else skip[lo:hi], bin_size=bins, **geno_params)
                        site += lo  # chunk-local site rows -> rows of the whole table
                        if stats_out is not None:
                            stats_out.append(dict(device=dev, n_reads=batch.n_reads, n_carried=n_carried, site_lo=lo,
                                                  site_hi=hi, **eng.last_stats))
                        done_q.put((seq, (site, cell, dp, alt, p)))
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
        threading.Thread(target=device_worker, args=(d,), daemon=True) for d in devices]
    for t in threads:
        t.start()
    parts, live = {}, len(devices)
    while live:
        item = done_q.get()
        if item is None:
            live -= 1
        else:
            parts[item[0]] = item[1]
    for t in threads:
        t.join()
    for sl in slots:
        sl.free()
    bs.close()
    if errors:
        raise errors[0]
    if not parts:
        return empty
    # chunks cover disjoint, increasing site slices: in chunk order the pairs are ordered by (site, cell)
    return tuple(np.concatenate([parts[s][k] for s in sorted(parts)]) for k in range(5))


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
    host = bamio._load_host()
    host.ls_write_counter_rows.argtypes = [C.c_char_p, C.c_char_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64,
                                           C.c_int, C.c_int]
    host.ls_write_counter_rows.restype = C.c_int
    tids = np.unique(sites.tid)
    for t in sorted(tids.tolist(), key=lambda t: bam_names[t]):
        # rows of one contig are contiguous (sites are ordered by window = (tid, start)) -> native formatter
        lo, hi = int(np.searchsorted(sites.tid, t, "left")), int(np.searchsorted(sites.tid, t, "right"))
        pos = np.ascontiguousarray(sites.pos[lo:hi])
        ref = np.ascontiguousarray(sites.ref[lo:hi])
        cnt = np.ascontiguousarray(sites.counts[lo:hi])
        rc = host.ls_write_counter_rows(os.fsencode(out_file), bam_names[t].encode(), pos.ctypes.data, ref.ctypes.data,
                                        cnt.ctypes.data, hi - lo, min(16, len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)), 1)
        if rc != 0:
            raise IOError("ls_write_counter_rows(%s) failed: %d" % (out_file, rc))
    return True


def load_bam_for_counting(bam_path, mode="split"):
    """Decode a BAM and map CB tags to dense cell ids.
    mode 'split': cell = CB.split('-')[0] (BaseCellCounter.py:246).  Returns (BamData, ReadBatch, cell names)."""
    bd = bamio.read_bam(bam_path)
    cleaned = clean_barcodes_split(bd.barcodes)
    ids, uniq = dense_ids(cleaned)
    return bd, bd.with_cells(ids), uniq
