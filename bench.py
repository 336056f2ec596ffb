#!/usr/bin/env python
"""bench.py -- LongSom SNV hot path on B200: aligned bases counted / s (pileup).

  python bench.py --gpus N --steps K --warmup W            our arm (CUDA, one rank per GPU)
  python bench.py --impl reference --gpus N --steps K ...  CPU arm (oracle port, all host threads)

Workload (BASELINE.json configs[1]/[2]): whole-transcriptome synthetic PacBio-Kinnex-style
batch, 5M reads x ~1.5 kb, 5k cells; at N > 1 the SAME batch is sharded by coverage-balanced
genomic bins across the GPUs (strong scaling, no collective on the data path).
A "step" is one pass of the hot path over the resident batch: segment build -> (tile, cell)
sort -> unit expansion -> pileup-count kernel -> compaction of the passing sites into the reference's
output order (the compacted site list in HBM is what BaseCellCounter emits).  `value` is device-resident
throughput, `e2e` is the same metric from pinned HOST buffers (H2D of the batch and D2H of the compacted
site table inside the timing): the batch cut into --e2e-shards window shards, the C-ABI call ls_pileup_count()
per shard on --e2e-lanes engine handles of the GPU (own stream and buffers, one CUDA context; pipeline.count_shards_pipelined), so that transfers and
kernels of different shards overlap; the one-call figure is reported next to it (e2e.single_call_*).
One JSON line on stdout (rank 0).

  python bench.py ... --dump-outputs DIR   also writes the site table of the last timed step as DIR/<name>.npy
                                           (see dump_outputs), so that two builds can be compared output for output
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "aligned bases counted/sec (pileup)"
UNIT = "aligned_bases/s"
PARAMS = dict(min_bq=20, min_mq=60, min_dp=5, min_cc=5, min_ac=0, max_depth=200000)  # workflow values


def log(*a):
    print(*a, file=sys.stderr, flush=True)


_REAL_STDOUT = None


def quiet_stdout():
    """Libraries (NCCL prints its version banner) write to fd 1; the contract is ONE JSON line on stdout.
    Route fd 1 to stderr for the whole run and keep a private duplicate for the result line."""
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)


def emit_json(obj):
    line = (json.dumps(obj) + "\n").encode()
    sys.stdout.flush()
    if _REAL_STDOUT is not None:
        os.write(_REAL_STDOUT, line)
    else:
        sys.stdout.write(line.decode())
        sys.stdout.flush()


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


# ---------------------------------------------------------------------------------------------
def build_workload(scale, rank, world, sample_bases=None):
    """Returns dict(batch, windows, owned_aligned, total_reads, ...) for this rank's shard, or, when
    sample_bases is given, a bounded sample (a run of consecutive windows) for the CPU arm."""
    from longsom_b200 import synth
    from longsom_b200.batch import Windows, make_windows
    from longsom_b200.sharding import balanced_window_shards, reads_for_windows, window_weights
    cfg = synth.config("C2", scale=scale)
    t0 = time.time()
    plan = synth.Plan(**cfg)
    tid, pos, gend, tlen = plan.headers()
    iv = make_windows(plan.contig_lens, 50000)
    wt = np.array([i[0] for i in iv], np.int32)
    ws = np.array([i[1] for i in iv], np.int32)
    we = np.array([i[2] for i in iv], np.int32)
    weights = window_weights(wt, ws, we, tid, pos, tlen)
    if sample_bases is not None:
        # the first run of consecutive covered windows holding ~sample_bases aligned bases (genes are laid out
        # left to right with i.i.d. expression weights, so a prefix of the genome is a fair sample of the batch)
        cum = np.concatenate([[0.0], np.cumsum(weights)])
        start = int(np.argmax(weights > 0))
        end = int(np.searchsorted(cum, cum[start] + sample_bases, side="left"))
        w_lo, w_hi = start, max(start + 1, min(end, len(iv)))
    else:
        w_lo, w_hi = balanced_window_shards(weights, world)[rank]
    sel = reads_for_windows(wt, ws, we, w_lo, w_hi, tid, pos, gend)
    batch = plan.materialize(sel)
    # windows of the shard that can see a read at all (empty windows produce no output)
    keep = [j for j in range(w_lo, w_hi) if weights[j] > 0 or True]
    contig = {t: plan.ref[int(plan.contig_off[t]):int(plan.contig_off[t + 1])] for t in range(len(plan.contig_lens))}
    # drop windows no read overlaps: they cannot emit a site and only cost reference upload
    if len(sel):
        rkey_lo = (batch.tid.astype(np.int64) << 32) | batch.pos.astype(np.int64)
        rkey_hi = (batch.tid.astype(np.int64) << 32) | gend[sel].astype(np.int64)
        wkey_lo = (wt[w_lo:w_hi].astype(np.int64) << 32) | ws[w_lo:w_hi].astype(np.int64)
        wkey_hi = (wt[w_lo:w_hi].astype(np.int64) << 32) | we[w_lo:w_hi].astype(np.int64)
        # a window is covered if some read starts before its end and the running max end passes its start
        order_max_end = np.maximum.accumulate(rkey_hi)
        n_before_end = np.searchsorted(rkey_lo, wkey_hi, side="left")
        covered = (n_before_end > 0) & (order_max_end[np.maximum(n_before_end - 1, 0)] > wkey_lo)
        keep = [w_lo + j for j in np.nonzero(covered)[0]]
    windows = Windows.from_intervals([iv[j] for j in keep], contig)
    # reads "owned" by this shard: start inside [first window start, last window end)
    if w_hi > w_lo:
        lo_key = (int(wt[w_lo]) << 32) | (int(ws[w_lo]) if w_lo > 0 and wt[w_lo - 1] == wt[w_lo] else 0)
        hi_key = (int(wt[w_hi - 1]) << 32) | (int(we[w_hi - 1]) if w_hi < len(iv) and wt[w_hi] == wt[w_hi - 1] else (1 << 31))
        rk = (batch.tid.astype(np.int64) << 32) | batch.pos.astype(np.int64)
        owned = (rk >= lo_key) & (rk < hi_key)
    else:
        owned = np.zeros(batch.n_reads, bool)
    op = batch.cigar & 15
    ln = np.where((op == 0) | (op == 7) | (op == 8), batch.cigar >> 4, 0).astype(np.int64)
    per_read = np.add.reduceat(ln, batch.cigar_off[:-1].astype(np.int64)) if batch.n_reads else np.zeros(0, np.int64)
    if batch.n_reads:
        per_read[batch.cigar_off[1:] == batch.cigar_off[:-1]] = 0
    owned_aligned = int(per_read[owned].sum())
    info = dict(cfg=cfg, n_reads_total=plan.n_reads, n_cells=plan.n_cells, windows_total=len(iv),
                shard=(w_lo, w_hi), gen_s=time.time() - t0, batch_aligned=int(per_read.sum()))
    plan.close()
    return dict(batch=batch, windows=windows, owned_aligned=owned_aligned, info=info)


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu):
        super().__init__(daemon=True)
        self.gpu, self.rows, self.proc = gpu, [], None
        self.t_rows = []          # arrival time of every row
        self.t_begin = None       # rows that arrive before mark_begin() are not "under load"

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "25"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                self.rows.append([x.strip() for x in line.split(",")])
                self.t_rows.append(time.perf_counter())
        except Exception:
            pass

    def wait_ready(self, timeout=8.0):
        """nvidia-smi takes a variable time to print its first row: the timed region starts after it."""
        t0 = time.perf_counter()
        while not self.rows and time.perf_counter() - t0 < timeout:
            time.sleep(0.01)

    def mark_begin(self):
        self.t_begin = time.perf_counter()

    def n_under_load(self):
        return sum(1 for t in self.t_rows if self.t_begin is not None and t >= self.t_begin)

    def stop(self):
        if self.proc:
            self.proc.terminate()
        self.join(timeout=2)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        rows = [r for r, t in zip(self.rows, self.t_rows) if self.t_begin is None or t >= self.t_begin]
        for r in rows:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except (ValueError, IndexError):
                continue
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=max(mx) if mx else None,
                    reasons=sorted(reasons), samples=len(sm))


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def algorithmic_bytes(batch, n_tiles, tile, n_sites):
    """B_K1 of DESIGN.md: 1.5 B per query base (4-bit base + quality), 4 B per CIGAR op, 19 B per
    read (pos 4, flag 2, mapq 1, cell 4, two offsets 8), 1 B of reference per tile position,
    104 B (26 words) per emitted site."""
    qbases = int(batch.l_qseq.astype(np.int64).sum())
    return 1.5 * qbases + 4.0 * batch.cigar.shape[0] + 19.0 * batch.n_reads + 1.0 * n_tiles * tile + 104.0 * n_sites


DUMP_SITES = 200_000  # sampled rows of the site table: 30 float64 values each, ~48 MB in all


def dump_outputs(out_dir, sites, rank, world):
    """Writes what a caller of the timed step receives, the compacted site table (tid, pos, ref, counts[26]), as
    float64 .npy files.  The full table has ~1.7e7 rows at scale 1, so only a fixed, seeded sample of rows is written
    (site_index.npy holds their row numbers), together with the column sums of counts over every row.  With
    several GPUs each rank writes its own shard's table under a rank<r>_ prefix and samples a 1/world share."""
    os.makedirs(out_dir, exist_ok=True)
    n, k = sites.n_sites, DUMP_SITES // world
    idx = np.sort(np.random.default_rng(0).choice(n, size=k, replace=False)) if n > k else np.arange(n)
    prefix = "rank%d_" % rank if world > 1 else ""
    arrays = {"site_index": idx, "tid": sites.tid[idx], "pos": sites.pos[idx], "ref": sites.ref[idx],
              "counts": sites.counts[idx], "counts_column_sums": sites.counts.sum(axis=0, dtype=np.uint64)}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, prefix + name + ".npy"), a.astype(np.float64))


def cpu_oracle_rate(sample, threads, steps=1):
    """Oracle port (plain C, OpenMP over windows) on a bounded sample; aligned bases / s."""
    import oracle
    from longsom_b200.engine import CountParams
    prm = CountParams(**PARAMS)
    best = None
    n_sites = 0
    for _ in range(steps):
        t0 = time.perf_counter()
        sc, nal = oracle.pileup_count(sample["batch"], sample["windows"], prm, threads=threads)
        dt = time.perf_counter() - t0
        n_sites = sc.n_sites
        best = dt if best is None or dt < best else best
    return sample["owned_aligned"] / best, best, n_sites


# ---------------------------------------------------------------------------------------------
def run_reference(args, rank, world):
    if rank != 0:
        return
    import __graft_entry__ as g
    g.build_checker()  # generator + oracle only: this arm never loads liblongsom_b200.so
    cores = os.cpu_count() or 1
    scale = args.scale
    # size the per-step sample so that (steps + warmup) steps take ~2 minutes: probe first
    probe = build_workload(scale, 0, 1, sample_bases=2e7)
    rate, dt, _ = cpu_oracle_rate(probe, cores)
    budget = 100.0 / max(1, args.steps + args.warmup)
    target = float(min(max(rate * min(budget, 25.0), 2e7), 2e9))
    sample = build_workload(scale, 0, 1, sample_bases=target)
    for _ in range(args.warmup):
        cpu_oracle_rate(sample, cores)
    times = []
    for _ in range(args.steps):
        r, dt, ns = cpu_oracle_rate(sample, cores)
        times.append(dt)
    ms = 1e3 * float(np.mean(times))
    value = sample["owned_aligned"] / (ms / 1e3)
    desc = "%d reads / %d aligned bases (windows %d..%d of the C2 batch)" % (
        sample["batch"].n_reads, sample["owned_aligned"], sample["info"]["shard"][0], sample["info"]["shard"][1])
    out = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "u32", "data": "synthetic",
        "config": workload_config(sample["info"], scale, l2="n/a (CPU)"),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": desc},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "note": "oracle port (oracle/pileup_oracle.c, OpenMP over 50 kb windows) of BaseCellCounter.run_interval; "
                "the reference's own Python/pysam path cannot run here (pysam absent, SURVEY.md 8c)",
    }
    emit_json(out)


def workload_config(info, scale, l2):
    cfg = info["cfg"]
    return {"workload": "C2 whole-transcriptome synthetic PacBio Kinnex-style batch (BASELINE.json configs[1]); "
                        "%d reads x ~1.5 kb, %d cells, %d contigs" % (cfg["n_reads"], cfg["n_cells"],
                                                                      len(cfg["contig_lens"])),
            "scale": scale, "reads": cfg["n_reads"], "cells": cfg["n_cells"], "genes": cfg["n_genes"],
            "params": PARAMS, "partition": "coverage-balanced 50 kb-window bins, one shard per GPU, no collective",
            "l2": l2}


def run_ours(args, rank, world, local_rank):
    import torch
    import __graft_entry__ as g
    if rank == 0:
        g.build()
    dist = None
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        dist.barrier()
    else:
        torch.cuda.set_device(local_rank)
    from longsom_b200.batch import ReadBatch, SiteCounts
    from longsom_b200.engine import CountParams, Engine
    from longsom_b200 import _lib
    from longsom_b200.pipeline import bind_near_gpu
    numa_node = bind_near_gpu(local_rank)   # before the batch and the pinned buffers are allocated (first touch)
    scale = args.scale
    wl = build_workload(scale, rank, world)
    batch, windows, info = wl["batch"], wl["windows"], wl["info"]
    log("[rank %d] shard windows %s: %d reads, %.3f GB batch, generated in %.1f s" % (
        rank, info["shard"], batch.n_reads, batch.nbytes() / 1e9, info["gen_s"]))
    prm = CountParams(**PARAMS)
    eng = Engine(local_rank)
    tile = _lib.load().ls_pileup_tile_size()

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def reduce_max(x):
        if dist is None:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def reduce_sum(x):
        if dist is None:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    total_units = reduce_sum(float(wl["owned_aligned"]))

    # ---- device-resident steps ---------------------------------------------------------------
    eng.upload(batch, windows)
    n_sites = 0
    for _ in range(args.warmup):
        n_sites = eng.run(prm)
        eng.compact()
    sampler = ClockSampler(local_rank)
    sampler.start()
    sampler.wait_ready()
    barrier()
    sampler.mark_begin()
    t0 = time.perf_counter()
    ms_count, ms_total, ms_compact, launches = [], [], [], 0
    for _ in range(args.steps):
        n_sites = eng.run(prm)
        st = eng.last_stats
        ms_count.append(st["ms_count"])
        ms_total.append(st["ms_total"])
        launches += st["count_launches"]
        eng.compact()
        ms_compact.append(eng.last_stats["ms_compact"])
        launches += 1
    barrier()
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, eng.fetch(n_sites), rank, world)
    # a short timed region can end between two nvidia-smi rows: keep the same load running (untimed) until the sampler
    # has at least three rows taken under it
    extra = 0
    while sampler.n_under_load() < 3 and extra < 400 and sampler.proc is not None:
        eng.run(prm)
        eng.compact()
        extra += 1
    clocks = sampler.stop()
    clocks["untimed_steps_added_for_sampling"] = extra
    dt = reduce_max(dt)
    ms_per_step = 1e3 * dt / args.steps
    value = total_units / (dt / args.steps)

    # ---- roofline of the dominant kernel (pileup_count_kernel), live CUDA-event timing ---------
    peak, peak_src = measured_peak()
    alg = algorithmic_bytes(batch, st["n_tiles"], tile, n_sites)
    c_ms = float(np.mean(ms_compact))
    k_ms = float(np.mean(ms_count))
    achieved = alg / (k_ms * 1e-3) / 1e9 if k_ms > 0 else 0.0
    traffic = None
    tp = os.path.join(ROOT, "profiles", "k1_traffic.json")
    if os.path.exists(tp):
        try:
            traffic = json.load(open(tp)).get("dram_bytes_per_launch")
        except Exception:
            traffic = None
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "kernel": "pileup_count_kernel", "kernel_ms": k_ms,
                "algorithmic_bytes_per_launch": alg, "bytes_per_aligned_base": alg / max(1, info["batch_aligned"]),
                "peak_source": peak_src, "kernel_share_of_step": k_ms / ms_per_step if ms_per_step else None,
                "issue_slot_ceiling": "see profiles/README.md: the kernel is bound by instruction issue and shared-memory "
                                      "wavefronts, not by HBM"}

    # ---- end to end through the C-ABI with pinned host buffers ---------------------------------
    def pin(a):
        t = torch.from_numpy(np.ascontiguousarray(a))
        return t.pin_memory().numpy() if t.numel() else a
    pb = ReadBatch(*[pin(getattr(batch, f)) for f in ("tid", "pos", "flag", "mapq", "cell", "cigar_off", "cigar",
                                                      "base_off", "l_qseq", "seq4", "qual")])
    from longsom_b200.batch import Windows
    pw = Windows(*[pin(getattr(windows, f)) for f in ("tid", "start", "end", "ref_off", "ref")])
    cap = max(int(n_sites), 1)
    out = SiteCounts(pin(np.zeros(cap, np.int32)), pin(np.zeros(cap, np.int32)), pin(np.zeros(cap, np.uint8)),
                     pin(np.zeros((cap, 26), np.uint32)))
    e2e_steps = max(1, min(args.steps, 3))
    eng.pileup_count_e2e(pb, pw, prm, out)  # warm
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        ns = eng.pileup_count_e2e(pb, pw, prm, out)
        launches_e2e = eng.last_stats["count_launches"] + 1
    barrier()
    dte = reduce_max(time.perf_counter() - t0)
    h2d = batch.nbytes() + sum(getattr(windows, f).nbytes for f in ("tid", "start", "end", "ref_off", "ref"))
    d2h = int(ns) * (4 + 4 + 1 + 104)
    single_ms = 1e3 * dte / e2e_steps
    e2e = {"value": total_units / (dte / e2e_steps), "unit": UNIT, "h2d_bytes_per_step": int(reduce_sum(float(h2d))),
           "d2h_bytes_per_step": int(reduce_sum(float(d2h))), "steps": e2e_steps, "ms_per_step": single_ms,
           "api": "ls_pileup_count (C-ABI, pinned host buffers)"}
    # Pipelined variant (what the CLI-level pipeline offers for large inputs): the same batch cut into window shards,
    # ls_pileup_count() per shard on `lanes` engine handles (ls_ctx: own stream and buffers, same CUDA context), so uploads, kernels and result copies of
    # different shards overlap.  Every step still moves every input byte H2D and every result byte D2H.
    if args.e2e_shards > 1:
        from longsom_b200.pipeline import count_shards_pipelined, window_shards
        del pb, pw, out
        shards = [(ReadBatch(*[pin(getattr(b_, f)) for f in ("tid", "pos", "flag", "mapq", "cell", "cigar_off", "cigar",
                                                             "base_off", "l_qseq", "seq4", "qual")]),
                   Windows(*[pin(getattr(w_, f)) for f in ("tid", "start", "end", "ref_off", "ref")]))
                  for b_, w_ in window_shards(batch, windows, args.e2e_shards)]
        lanes = [Engine(local_rank) for _ in range(max(1, args.e2e_lanes))]  # own contexts: `eng` keeps the full batch
        sizes = []
        for b_, w_ in shards:  # sizing pass (not timed): sites per shard
            lanes[0].upload(b_, w_)
            sizes.append(int(lanes[0].run(prm)))
        assert sum(sizes) == int(n_sites), "window shards must reproduce the site count (%d vs %d)" % (sum(sizes), n_sites)
        outs = [SiteCounts(pin(np.zeros(max(c, 1), np.int32)), pin(np.zeros(max(c, 1), np.int32)),
                           pin(np.zeros(max(c, 1), np.uint8)), pin(np.zeros((max(c, 1), 26), np.uint32))) for c in sizes]
        count_shards_pipelined(shards, prm, outs, engines=lanes)  # warm
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            got = count_shards_pipelined(shards, prm, outs, engines=lanes)
        barrier()
        dtp = reduce_max(time.perf_counter() - t0)
        assert sum(got) == int(n_sites)
        h2d_p = sum(b_.nbytes() + sum(getattr(w_, f).nbytes for f in ("tid", "start", "end", "ref_off", "ref"))
                    for b_, w_ in shards)
        e2e = {"value": total_units / (dtp / e2e_steps), "unit": UNIT, "h2d_bytes_per_step": int(reduce_sum(float(h2d_p))),
               "d2h_bytes_per_step": int(reduce_sum(float(d2h))), "steps": e2e_steps, "ms_per_step": 1e3 * dtp / e2e_steps,
               "api": "longsom_b200.pipeline.count_shards_pipelined: ls_pileup_count (C-ABI, pinned host buffers) per "
                      "window shard, %d shards on %d engine handles (streams of the device's CUDA context)" % (len(shards), len(lanes)),
               "single_call_ms_per_step": single_ms, "single_call_value": total_units / (single_ms * 1e-3)}
        for l in lanes:
            l.close()
        del shards, outs

    # ---- what the box's PCIe / host memory can do at this N: every rank copies 1 GiB of pinned memory to its GPU at
    # the same time, three times (the ceiling the end-to-end number above is to be read against)
    h2d_ceiling = None
    try:
        hbuf = torch.empty(1 << 30, dtype=torch.uint8).pin_memory()
        dbuf = torch.empty(1 << 30, dtype=torch.uint8, device="cuda")
        dbuf.copy_(hbuf, non_blocking=True)
        torch.cuda.synchronize()
        barrier()
        t0 = time.perf_counter()
        for _ in range(3):
            dbuf.copy_(hbuf, non_blocking=True)
        torch.cuda.synchronize()
        barrier()
        dt_c = reduce_max(time.perf_counter() - t0)
        h2d_ceiling = {"aggregate_GBps": world * 3 * (1 << 30) / dt_c / 1e9, "per_gpu_GBps": 3 * (1 << 30) / dt_c / 1e9,
                       "how": "1 GiB pinned -> device, all ranks at once, 3 copies, max over ranks"}
        del hbuf, dbuf
    except Exception as ex:   # the number is an annotation, never a reason to fail the bench
        h2d_ceiling = {"error": repr(ex)}
    if isinstance(e2e, dict):
        e2e["h2d_ceiling"] = h2d_ceiling
        if h2d_ceiling and "aggregate_GBps" in h2d_ceiling and e2e.get("ms_per_step"):
            e2e["h2d_GBps_achieved"] = e2e["h2d_bytes_per_step"] / (e2e["ms_per_step"] * 1e-3) / 1e9

    # ---- second half of BASELINE.json's metric: candidate sites genotyped / s (K1' + K2), every N -------------------
    # 200 000 candidate sites over the whole batch (each rank takes the ones inside its window shard), all cells of
    # the workload; sparse path: touched (site, cell) tuples + on-device beta-binomial tails.
    secondary = None
    if not args.no_secondary:
        got = eng.fetch(n_sites) if n_sites else None
        share = wl["owned_aligned"] / max(1.0, total_units)
        n_cand = int(min(got.n_sites if got is not None else 0, round(200000 * args.scale * share)))
        n_cells = info["cfg"]["n_cells"]
        g_dev_ms, g_e2e_ms, n_tup, gk_ms, bb_ms, hits = 0.0, 0.0, 0, 0.0, 0.0, 0
        if n_cand >= 100:
            rng = np.random.default_rng(rank)
            idx = np.sort(rng.choice(got.n_sites, size=n_cand, replace=False))
            alt = rng.integers(0, 4, size=n_cand).astype(np.uint8)
            gt, gp = got.tid[idx].copy(), got.pos[idx].copy()
            a2, b2 = 0.2474528917555431, 162.03696139428595
            eng.genotype_sparse(gt, gp, alt, n_cells, a2, b2, min_bq=30, min_mq=60, fetch=False)  # warm
            barrier()
            t0 = time.perf_counter()
            n_tup = eng.genotype_sparse(gt, gp, alt, n_cells, a2, b2, min_bq=30, min_mq=60, fetch=False)
            barrier()
            g_dev_ms = 1e3 * (time.perf_counter() - t0)
            gs = eng.last_stats
            gk_ms, bb_ms, hits = gs["ms_count"], gs["ms_sort"], gs["n_events"]
            t0 = time.perf_counter()
            tup = eng.genotype_sparse(gt, gp, alt, n_cells, a2, b2, min_bq=30, min_mq=60)
            barrier()
            g_e2e_ms = 1e3 * (time.perf_counter() - t0)
            del tup
        else:
            for _ in range(3):
                barrier()
        tot_cand = reduce_sum(float(n_cand))
        g_dev_ms, g_e2e_ms = reduce_max(g_dev_ms), reduce_max(g_e2e_ms)
        # K1' algorithmic bytes (SURVEY 8d): 19 B per read + 4 B per CIGAR op + 13 B per site + 8 B per touched pair
        g_alg = 19.0 * batch.n_reads + 4.0 * batch.cigar.shape[0] + 13.0 * n_cand + 8.0 * n_tup
        secondary = {"metric": "candidate sites genotyped/sec (K1' sparse pileup + K2 beta-binomial tails, on device)",
                     "value": tot_cand / (g_dev_ms * 1e-3) if g_dev_ms else None, "unit": "sites/s",
                     "sites": int(tot_cand), "cells": int(n_cells), "ms": g_dev_ms,
                     "e2e": {"value": tot_cand / (g_e2e_ms * 1e-3) if g_e2e_ms else None, "ms": g_e2e_ms,
                             "note": "host site table in, touched (site, cell, Dp, Alt, p) tuples out"},
                     "rank0": {"sites": int(n_cand), "touched_pairs": int(n_tup), "pileup_hits": int(hits),
                               "k1p_ms": gk_ms, "k2_ms": bb_ms,
                               "roofline": {"bound": "hbm", "kernel": "slot count (CIGAR walk) + genotype_kernel + hit sort + reduce",
                                            "achieved": g_alg / (gk_ms * 1e-3) / 1e9 if gk_ms else None, "peak": peak,
                                            "unit": "GB/s", "frac": g_alg / (gk_ms * 1e-3) / 1e9 / peak if gk_ms else None,
                                            "algorithmic_bytes": g_alg}}}
        if world == 1:
            # K2 and K3 on their own (the step1 / step2 kernels of the path), host arrays in and out like their callers
            rng = np.random.default_rng(11)
            m2 = int(2_000_000 * min(1.0, args.scale))
            n2 = np.minimum(2 + rng.geometric(0.01, m2), 200000).astype(np.int32)
            k2 = np.minimum(1 + rng.geometric(0.25, m2), n2).astype(np.int32)
            big = rng.random(m2) < 0.002   # a few deep sites with long tails (k > 128: the staged path)
            k2[big] = np.minimum(n2[big], 129 + rng.integers(0, 2000, int(big.sum()))).astype(np.int32)
            eng.betabinom_sf(k2[:1000], n2[:1000], 0.26, 173.9)
            t0 = time.perf_counter()
            eng.betabinom_sf(k2, n2, 0.26, 173.9)
            k2_wall = time.perf_counter() - t0
            st2 = eng.last_stats
            m3, nk3 = int(2_000_000 * min(1.0, args.scale)), int(4_000_000 * min(1.0, args.scale))
            tab = (rng.integers(0, 25, nk3).astype(np.uint64) << np.uint64(32)) | rng.integers(0, 250_000_000, nk3).astype(np.uint64)
            q3 = np.concatenate([tab[rng.integers(0, nk3, m3 // 2)],
                                 (rng.integers(0, 25, m3 - m3 // 2).astype(np.uint64) << np.uint64(32)) |
                                 rng.integers(0, 250_000_000, m3 - m3 // 2).astype(np.uint64)])
            eng.site_table_load(0, tab)
            st3a = eng.last_stats
            eng.site_table_lookup(0, q3[:1000])
            t0 = time.perf_counter()
            eng.site_table_lookup(0, q3)
            k3_wall = time.perf_counter() - t0
            st3b = eng.last_stats
            secondary["k2"] = {"kernel": "bb_small_kernel (k <= 128, terms in registers) + staged terms for longer tails",
                               "queries": m2, "pmf_terms": int(st2["n_events"]), "kernel_ms": st2["ms_count"],
                               "fp64_pmf_terms_per_s": st2["n_events"] / (st2["ms_count"] * 1e-3) if st2["ms_count"] else None,
                               "queries_per_s_host_to_host": m2 / k2_wall}
            secondary["k3"] = {"kernel": "mask_lookup_kernel against a resident sorted table", "table_keys": nk3, "queries": m3,
                               "table_sort_ms": st3a["ms_sort"], "lookup_ms": st3b["ms_count"],
                               "lookups_per_s": m3 / (st3b["ms_count"] * 1e-3) if st3b["ms_count"] else None,
                               "GB_per_s": (9.0 * m3 + 8.0 * nk3) / (st3b["ms_count"] * 1e-3) / 1e9 if st3b["ms_count"] else None,
                               "bytes_note": "8 B query + 1 B hit per lookup + one pass over the table",
                               "queries_per_s_host_to_host": m3 / k3_wall}
            del tab, q3, k2, n2
        del got
    # ---- BASELINE.json configs[3] (hotspot stress: 20 genes at > 1e5 reads / locus, 10k cells), N = 1 only --------
    c4 = None
    if world == 1 and not args.no_secondary and args.scale >= 1.0:
        from longsom_b200 import synth
        from longsom_b200.batch import Windows as _W, make_windows as _mw
        d4 = synth.generate(**synth.config("C4", scale=1.0))
        w4 = _W.from_intervals(_mw(d4.contig_lens, 50000), d4.contig_seqs())
        eng.upload(d4.batch, w4)
        for _ in range(2):
            eng.run(prm)
            eng.compact()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        n4 = eng.run(prm)
        s4 = eng.last_stats
        eng.compact()
        torch.cuda.synchronize()
        dt4 = time.perf_counter() - t0
        al4 = d4.batch.aligned_bases()
        alg4 = algorithmic_bytes(d4.batch, s4["n_tiles"], tile, n4)
        c4 = {"workload": "C4 hotspot stress: %d reads, %d cells, 20 hot genes" % (d4.batch.n_reads, d4.n_cells),
              "value": al4 / dt4, "unit": UNIT, "ms_per_step": 1e3 * dt4, "kernel_ms": s4["ms_count"],
              "segments_per_tile": s4["n_segments"] / max(1, s4["n_tiles"]),
              "roofline_frac": alg4 / (s4["ms_count"] * 1e-3) / 1e9 / peak}
        del d4, w4

    # ---- the drop-in CLI, BAM on disk -> TSV on disk (streaming path), rank 0, N = 1 only ---------------------------
    e2e_cli = None
    if world == 1 and args.cli_scale > 0:
        import tempfile
        from longsom_b200 import bamio, synth
        dcli = synth.generate(**synth.config("C2", scale=args.cli_scale * scale))
        tmp = tempfile.mkdtemp(prefix="ls_bench_cli_")
        bamio.write_fasta(tmp + "/ref.fa", dcli.contig_names, [dcli.contig_seq(i) for i in range(len(dcli.contig_lens))])
        names = [synth.barcode_of(c) + "-1" for c in range(dcli.n_cells + dcli.n_extra_cells)]
        bc = dcli.batch
        bamio.write_bam(tmp + "/x.bam", dcli.contig_names, dcli.contig_lens, bc, lambda i: None if bc.cell[i] < 0 else names[bc.cell[i]])
        al_cli, n_cli, bam_mb = bc.aligned_bases(), bc.n_reads, os.path.getsize(tmp + "/x.bam") / 1e6
        del dcli, bc
        script = os.path.join(ROOT, "workflow", "scripts", "SNVCalling", "BaseCellCounter.py")
        best = None
        for _ in range(2):
            t0 = time.perf_counter()
            r = subprocess.run([sys.executable, script, "--bam", tmp + "/x.bam", "--ref", tmp + "/ref.fa", "--chrom", "all",
                                "--out_folder", tmp, "--id", "x", "--min_bq", "20", "--min_mq", "60", "--tmp_dir", tmp + "/t"],
                               stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
            dtc = time.perf_counter() - t0
            if r.returncode != 0:
                raise RuntimeError("drop-in CLI failed: " + r.stderr[-1500:])
            best = dtc if best is None or dtc < best else best
        e2e_cli = {"value": al_cli / best, "unit": UNIT, "seconds": best, "reads": int(n_cli), "bam_mb": bam_mb,
                   "tsv_mb": os.path.getsize(tmp + "/x.tsv") / 1e6, "host_cores": os.cpu_count(),
                   "api": "workflow/scripts/SNVCalling/BaseCellCounter.py as a subprocess (process start, CUDA context, "
                          "streaming BGZF decode (own DEFLATE decoder, prefetch thread) -> pinned slots -> ls_pileup_count -> native TSV rows, completed contigs appended as they finish)"}
        import shutil
        shutil.rmtree(tmp, ignore_errors=True)

    # ---- CPU baseline beside it (rank 0, N=1 only) -----------------------------------------------
    cpu = None
    if world == 1 and not args.no_cpu:
        cores = os.cpu_count() or 1
        probe = build_workload(scale, 0, 1, sample_bases=2e7)
        rate, _, _ = cpu_oracle_rate(probe, cores)
        sample = build_workload(scale, 0, 1, sample_bases=float(min(max(rate * 15.0, 2e7), 2e9)))
        rate, dtc, _ = cpu_oracle_rate(sample, cores)
        cpu = {"value": rate, "unit": UNIT, "cores": cores, "kind": "port",
               "sample": "%d reads / %d aligned bases (windows %d..%d of the C2 batch), %.1f s" % (
                   sample["batch"].n_reads, sample["owned_aligned"], sample["info"]["shard"][0],
                   sample["info"]["shard"][1], dtc)}
    if rank == 0:
        res = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "u32", "data": "synthetic",
            "config": workload_config(info, scale, l2="inputs (%.2f GB per GPU) exceed the 126 MB L2; no flush needed"
                                      % (batch.nbytes() / 1e9)),
            "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "clocks": clocks, "secondary": secondary, "c4": c4, "e2e_cli": e2e_cli,
            "gpu_launches": int(launches), "numa_node": numa_node,
            "stats": {"n_segments": st["n_segments"], "n_tiles": st["n_tiles"], "n_sites": int(n_sites),
                      "n_events": st["n_events"], "ms_segments": st["ms_segments"], "ms_sort": st["ms_sort"],
                      "ms_count": k_ms, "ms_compact": c_ms, "ms_device_total": float(np.mean(ms_total)) + c_ms, "tile": tile,
                      "aligned_bases_total": total_units},
        }
        emit_json(res)
    eng.close()
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--scale", type=float, default=float(os.environ.get("LS_BENCH_SCALE", "1.0")),
                    help="fraction of the C2 workload (1.0 = 5M reads); only for local debugging")
    ap.add_argument("--e2e-shards", type=int, default=8, help="window shards of the pipelined end-to-end leg (1 = off)")
    ap.add_argument("--e2e-lanes", type=int, default=2, help="engine handles (streams) the pipelined end-to-end leg alternates on")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-secondary", action="store_true", help="skip the genotyping metric and the C4 line")
    ap.add_argument("--cli-scale", type=float, default=0.2,
                    help="size of the BAM of the disk-to-disk CLI leg as a fraction of the workload (0 = skip; 1.0 = the "
                         "whole 5 M-read BAM, which takes ~100 s to write)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the site table of the last timed step (a seeded sample) to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    quiet_stdout()
    rank, world, local_rank = env_int("RANK", 0), env_int("WORLD_SIZE", 1), env_int("LOCAL_RANK", 0)
    # torchrun pins OMP_NUM_THREADS=1; the (untimed) synthetic generator and the CPU oracle are OpenMP code
    os.environ["OMP_NUM_THREADS"] = str(max(1, (os.cpu_count() or 1) // max(1, world)))
    if world != args.gpus and world > 1:
        log("warning: WORLD_SIZE=%d but --gpus %d" % (world, args.gpus))
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
