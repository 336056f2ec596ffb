"""Wall clock of the drop-in BaseCellCalling.step1 on a merged table built from the synthetic C2 data (BaseCellCounter on
two cell-type BAMs -- the same reads under two names -- then MergeBaseCellCounts), in two arms run in the same call:
the device arm (the row loop on the GPU, ls_step1.cu) and the host arm (the same child with Engine's step1_* methods
hidden: the host passes of ls_step1.cpp, tails on the GPU).  Each run starts after a sync; the arms alternate.  Per arm:
rows, the best / median wall time of the child, the median step1 stage time (main()) and its rows/s, the peak resident
set, and for the device arm the median busy seconds of the file reads, the device calls, the text blocks (their file
writes overlapped) and the file writes.  Also: a write floor (the same output bytes written from memory), the card and its power limit, and a
byte comparison of the two arms' tables.
usage: cli_step1_timing.py [scales, comma-separated] [repeats]"""
import json
import os
import shutil
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from longsom_b200 import bamio, synth  # noqa: E402

CHILD = r"""
import contextlib, io, json, resource, sys, time
sys.path.insert(0, %r)
from longsom_b200.cli import step1
from longsom_b200.engine import Engine
if sys.argv[1] == "host":
    for k in [k for k in vars(Engine) if k.startswith("step1_")]:
        delattr(Engine, k)
t, log = time.perf_counter(), io.StringIO()
with contextlib.redirect_stdout(log):
    step1.main(sys.argv[2:])
stage = time.perf_counter() - t
rows = int(log.getvalue().split("Step 1 variant calling: ")[1].split()[0])
print("TIMES " + json.dumps(dict(step1.last_times, rows=rows, stage=stage,
                                 peak_rss_gb=resource.getrusage(resource.RUSAGE_SELF).ru_maxrss / 1e6)))
""" % ROOT

scales = [float(x) for x in (sys.argv[1] if len(sys.argv) > 1 else "0.2").split(",")]
repeats = int(sys.argv[2]) if len(sys.argv) > 2 else 3
card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], stdout=subprocess.PIPE,
                      text=True).stdout.strip().splitlines()
print("cards:", card, "host cores:", len(os.sched_getaffinity(0)), flush=True)
scripts = os.path.join(ROOT, "workflow", "scripts", "SNVCalling")
results = []
for scale in scales:
    tmp = tempfile.mkdtemp()
    d = synth.generate(**synth.config("C2", scale=scale))
    b = d.batch
    names = [synth.barcode_of(c) + "-1" for c in range(d.n_cells + d.n_extra_cells)]
    os.makedirs(tmp + "/counts")
    for ct in ("Cancer", "Non-Cancer"):
        bamio.write_bam("%s/s.%s.bam" % (tmp, ct), d.contig_names, d.contig_lens, b,
                        lambda i: None if b.cell[i] < 0 else names[b.cell[i]])
    bamio.write_fasta(tmp + "/ref.fa", d.contig_names, [d.contig_seq(i) for i in range(len(d.contig_lens))])
    del d, b
    for ct in ("Cancer", "Non-Cancer"):
        subprocess.run([sys.executable, scripts + "/BaseCellCounter.py", "--bam", "%s/s.%s.bam" % (tmp, ct), "--ref",
                        tmp + "/ref.fa", "--chrom", "all", "--out_folder", tmp + "/counts", "--min_bq", "20", "--min_mq",
                        "60", "--tmp_dir", tmp + "/tmp_" + ct], check=True, stdout=subprocess.DEVNULL)
    subprocess.run([sys.executable, scripts + "/MergeBaseCellCounts.py", "--tsv_folder", tmp + "/counts", "--outfile",
                    tmp + "/merged.tsv"], check=True, stdout=subprocess.DEVNULL)
    merged_mb = os.path.getsize(tmp + "/merged.tsv") / 1e6
    print("scale %g: merged table %.1f MB" % (scale, merged_mb), flush=True)
    runs = {"device": [], "host": []}
    for rep in range(repeats):
        for arm in ("device", "host") if rep % 2 == 0 else ("host", "device"):
            out = "%s/out_%s" % (tmp, arm)
            os.sync()
            t0 = time.time()
            r = subprocess.run([sys.executable, "-c", CHILD, arm, "--infile", tmp + "/merged.tsv", "--outfile", out,
                                "--ref", tmp + "/ref.fa"], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
            dt = time.time() - t0
            assert r.returncode == 0, r.stderr[-3000:]
            row = json.loads([l for l in r.stdout.splitlines() if l.startswith("TIMES ")][0][6:])
            row["seconds"] = dt
            runs[arm].append(row)
            print("   %-6s %.2f s  %s" % (arm, dt, json.dumps(row)), flush=True)
    a, h = (open("%s/out_%s.calling.step1.tsv" % (tmp, x), "rb").read() for x in ("device", "host"))
    same = a == h
    os.sync()
    t0 = time.time()
    with open(tmp + "/floor.tsv", "wb") as f:
        f.write(a)
    floor = time.time() - t0
    res = dict(scale=scale, merged_mb=round(merged_mb, 1), out_mb=round(len(a) / 1e6, 1), identical=same,
               write_floor_s=round(floor, 3), card=card)
    for arm, rs in runs.items():
        med = lambda k: statistics.median(x.get(k, 0.0) for x in rs)   # the host arm reports its stage time only
        res[arm] = dict(rows=rs[0]["rows"], best_s=round(min(x["seconds"] for x in rs), 3), median_s=round(med("seconds"), 3),
                        stage_s=round(med("stage"), 3), rows_per_s=round(rs[0]["rows"] / med("stage")),
                        read_s=round(med("read_s"), 3), call_s=round(med("call_s"), 3), text_s=round(med("text_s"), 3),
                        write_s=round(med("write_s"), 3), peak_rss_gb=round(med("peak_rss_gb"), 2))
    print(json.dumps(res), flush=True)
    results.append(res)
    shutil.rmtree(tmp, ignore_errors=True)
