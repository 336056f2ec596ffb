"""Disk-to-disk wall clock of the drop-in BaseCellCounter on a synthetic C2 BAM with its rows formatted on the device
(default) and by the host writer (LONGSOM_COUNTER_TEXT=host), byte-compared.  Per arm: the best and the median wall
time of the script; the medians of the wall time of its streaming stage (pipeline.stream_count), of the busy seconds
it reports for the decoder thread, the device steps (count, text), the writer (main thread: part-file appends, or
fetch + ls_write_counter_rows) and the concatenation, and of the peak resident set; the table size.  Each run starts
after a sync; the two arms alternate.
usage: cli_counter_text_timing.py [scales, comma-separated] [repeats]"""
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

scales = [float(x) for x in (sys.argv[1] if len(sys.argv) > 1 else "0.2").split(",")]
repeats = int(sys.argv[2]) if len(sys.argv) > 2 else 5
card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], stdout=subprocess.PIPE,
                      text=True).stdout.strip().splitlines()
print("cards:", card, "host cores:", len(os.sched_getaffinity(0)), flush=True)
script = os.path.join(ROOT, "workflow", "scripts", "SNVCalling", "BaseCellCounter.py")
results = []
for scale in scales:
    tmp = tempfile.mkdtemp()
    d = synth.generate(**synth.config("C2", scale=scale))
    b = d.batch
    names = [synth.barcode_of(c) + "-1" for c in range(d.n_cells + d.n_extra_cells)]
    bamio.write_bam(tmp + "/x.bam", d.contig_names, d.contig_lens, b, lambda i: None if b.cell[i] < 0 else names[b.cell[i]])
    bamio.write_fasta(tmp + "/ref.fa", d.contig_names, [d.contig_seq(i) for i in range(len(d.contig_lens))])
    n_reads, bam_mb = int(b.n_reads), os.path.getsize(tmp + "/x.bam") / 1e6
    del d, b
    print("scale %g: %d reads, BAM %.1f MB" % (scale, n_reads, bam_mb), flush=True)
    runs = {"device": [], "host": []}
    for rep in range(repeats):
        for arm in ("device", "host") if rep % 2 == 0 else ("host", "device"):
            out = "%s/out_%s" % (tmp, arm)
            shutil.rmtree(out, ignore_errors=True)
            os.makedirs(out)
            env = dict(os.environ, LS_STREAM_TIMING="1", LONGSOM_COUNTER_TEXT=arm)
            os.sync()
            t0 = time.time()
            r = subprocess.run([sys.executable, script, "--bam", tmp + "/x.bam", "--ref", tmp + "/ref.fa", "--chrom", "all",
                                "--out_folder", out, "--id", "x", "--min_bq", "20", "--min_mq", "60", "--tmp_dir",
                                out + "/tmp"], env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
            dt = time.time() - t0
            assert r.returncode == 0, r.stderr[-3000:]
            busy = [l for l in r.stderr.splitlines() if l.startswith("[stream_count] busy seconds:")][0]
            row = dict(seconds=dt, peak_rss_gb=float([l for l in r.stderr.splitlines()
                                                       if l.startswith("[counter] peak RSS")][0].split()[3]))
            for kv in busy.split(":", 1)[1].split(";")[0].split(","):
                k, v = kv.split()
                row[k] = float(v)
            row["stream"] = float(busy.split("; wall ")[1].split()[0])
            runs[arm].append(row)
            print("   %-6s %.2f s  %s" % (arm, dt, busy.split(": ", 1)[1]), flush=True)
        if rep == 0:
            tables = [open("%s/out_%s/x.tsv" % (tmp, a), "rb").read().split(b"\n", 1)[1] for a in ("device", "host")]
            identical, table_mb = tables[0] == tables[1], len(tables[0]) / 1e6
            del tables
            assert identical, "device and host tables differ"
    summary = dict(scale=scale, reads=n_reads, bam_mb=round(bam_mb, 1), table_mb=round(table_mb, 1),
                   identical=identical, repeats=repeats)
    for arm, rs in runs.items():
        best = min(rs, key=lambda x: x["seconds"])
        summary[arm] = dict(best_s=round(best["seconds"], 2), median_s=round(statistics.median(x["seconds"] for x in rs), 2),
                            **{k: round(statistics.median(x[k] for x in rs), 3)
                               for k in ("stream", "decode", "device", "text", "writer", "concat", "peak_rss_gb")})
    print(json.dumps(summary), flush=True)
    results.append(summary)
    shutil.rmtree(tmp, ignore_errors=True)
print(json.dumps({"cards": card, "results": results}))
