"""Disk-to-disk wall clock and peak resident set of the drop-in HCCVSingleCellGenotype on a synthetic C2 BAM: streaming
path (default) against the whole-file path (LONGSOM_STREAM=0), at each GPU count asked for that the host has,
byte-compared.  HCCVSingleCellGenotype writes the same long table as SingleCellGenotype without the pandas pivot, whose
memory is the same on both paths.  The dense table has sites x cells rows, so the metadata lists only `cells` barcodes.
usage: cli_genotype_stream_timing.py [scale] [n_sites] [cells] [gpu counts, e.g. 1,8] [chunk_mb]"""
import filecmp, json, os, subprocess, sys, tempfile, time
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from longsom_b200 import synth, bamio

scale = float(sys.argv[1]) if len(sys.argv) > 1 else 0.2
n_sites = int(sys.argv[2]) if len(sys.argv) > 2 else 200_000
n_meta = int(sys.argv[3]) if len(sys.argv) > 3 else 20
gpu_counts = [int(x) for x in (sys.argv[4] if len(sys.argv) > 4 else "1,8").split(",")]
chunk_mb = sys.argv[5] if len(sys.argv) > 5 else None
card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], stdout=subprocess.PIPE,
                      text=True).stdout.strip().splitlines()
print("cards:", card, flush=True)
import torch
n_dev = torch.cuda.device_count()
d = synth.generate(**synth.config("C2", scale=scale))
tmp = tempfile.mkdtemp()
b = d.batch
names = [synth.barcode_of(c) + "-1" for c in range(d.n_cells + d.n_extra_cells)]
t = time.time()
bamio.write_bam(tmp + "/x.bam", d.contig_names, d.contig_lens, b, lambda i: None if b.cell[i] < 0 else names[b.cell[i]])
bamio.write_fasta(tmp + "/ref.fa", d.contig_names, [d.contig_seq(i) for i in range(len(d.contig_lens))])
# candidate sites: positions inside reads, as a caller's candidates would be
rng = np.random.default_rng(7)
pick = rng.choice(b.n_reads, min(b.n_reads, 3 * n_sites), replace=False)
keys = sorted({(int(b.tid[i]), int(b.pos[i]) + int(rng.integers(0, 1000))) for i in pick})
keys = [keys[i] for i in np.sort(rng.choice(len(keys), min(n_sites, len(keys)), replace=False))]
with open(tmp + "/cand.tsv", "w") as f:
    f.write("#CHROM\tStart\tEnd\tREF\tALT\n")
    for tid, p in keys:
        f.write("\t".join([d.contig_names[tid], str(p + 1), str(p + 1), "A", "ACGT"[p % 4], ".", "Cancer", ".", ".", ".",
                           ".", ".", ".", "3"]) + "\n")
with open(tmp + "/meta.tsv", "w") as f:
    f.write("Index\tCell_type\n")
    for c in range(n_meta):
        f.write("%s-1\t%s\n" % (synth.barcode_of(c), d.cell_type(c)))
print("reads %d, BAM %.1f MB, %d sites, %d cells in the table (inputs written in %.1f s), %d devices" % (
    b.n_reads, os.path.getsize(tmp + "/x.bam") / 1e6, len(keys), n_meta, time.time() - t, n_dev), flush=True)
del d, b
run = ("import sys; from longsom_b200.cli.genotype import main; from longsom_b200.pipeline import _peak_rss_gb; "
       "main(sys.argv[1:], hccv=True); print('[genotype] peak RSS %.3f GB' % _peak_rss_gb(), file=sys.stderr)")
res = []
for n in gpu_counts:
    if n > n_dev:
        print("%d GPUs: not available on this host (%d devices)" % (n, n_dev), flush=True)
        continue
    for mode, env in (("stream", {}), ("whole", {"LONGSOM_STREAM": "0"})):  # streaming first: the smaller footprint
        e = dict(os.environ, LONGSOM_GPUS=str(n), PYTHONPATH=ROOT, **env)
        if chunk_mb and mode == "stream":
            e["LONGSOM_CHUNK_MB"] = chunk_mb
        out = "%s/%s_%d.tsv" % (tmp, mode, n)
        best, rss = None, None
        for rep in range(2):
            t0 = time.time()
            r = subprocess.run([sys.executable, "-c", run, "--bam", tmp + "/x.bam", "--infile", tmp + "/cand.tsv", "--ref",
                                tmp + "/ref.fa", "--meta", tmp + "/meta.tsv", "--outfile", out, "--min_mq", "60",
                                "--tmp_dir", tmp + "/t"], env=e, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
            dt = time.time() - t0
            assert r.returncode == 0, r.stderr[-3000:]
            rss = max(rss or 0.0, float([l for l in r.stderr.splitlines() if l.startswith("[genotype] peak RSS")][0].split()[3]))
            best = dt if best is None else min(best, dt)
        res.append(dict(gpus=n, mode=mode, seconds=round(best, 2), peak_rss_gb=rss, out_mb=round(os.path.getsize(out) / 1e6, 1)))
        print("%d GPU(s) %-6s %.2f s, peak RSS %.2f GB, table %.0f MB" % (n, mode, best, rss, os.path.getsize(out) / 1e6),
              flush=True)
    assert filecmp.cmp("%s/stream_%d.tsv" % (tmp, n), "%s/whole_%d.tsv" % (tmp, n), shallow=False), "tables differ"
    print("tables identical", flush=True)
print(json.dumps({"cards": card, "scale": scale, "sites": len(keys), "cells": n_meta, "runs": res}))
