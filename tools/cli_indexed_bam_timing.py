"""Disk-to-disk wall clock, bytes read and inflated, and peak resident set of the three streamed scripts on a synthetic
C2 BAM, with its .bai (indexed arm) and on a copy without it (whole-file arm), byte-compared.  The BAM is indexed by
routing every barcode to one cell type through ls_bam_split with its filters off, as SplitBamCellTypes would.  Each run
starts after a sync; the two arms alternate.
  HCCVSingleCellGenotype at 1e2, 1e3, 1e4 sites; SingleCellGenotype at 1e3, 1e4 sites;
  BaseCellCounter --chrom <one contig> and --chrom all (the row that must not regress).
usage: cli_indexed_bam_timing.py [scale] [repeats]"""
import ctypes as C
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from longsom_b200 import bamio, synth  # noqa: E402

scale = float(sys.argv[1]) if len(sys.argv) > 1 else 0.2
repeats = int(sys.argv[2]) if len(sys.argv) > 2 else 2
card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], stdout=subprocess.PIPE,
                      text=True).stdout.strip().splitlines()
print("cards:", card, flush=True)
d = synth.generate(**synth.config("C2", scale=scale))
tmp = tempfile.mkdtemp()
b = d.batch
names = [synth.barcode_of(c) + "-1" for c in range(d.n_cells + d.n_extra_cells)]
t = time.time()
bamio.write_bam(tmp + "/raw.bam", d.contig_names, d.contig_lens, b, lambda i: None if b.cell[i] < 0 else names[b.cell[i]])
bamio.write_fasta(tmp + "/ref.fa", d.contig_names, [d.contig_seq(i) for i in range(len(d.contig_lens))])
os.makedirs(tmp + "/idx")
os.makedirs(tmp + "/plain")
host = bamio._load_host()
host.ls_bam_split.restype = C.c_int
keys = [synth.barcode_of(c).encode() for c in range(d.n_cells + d.n_extra_cells)]
off = (C.c_uint32 * (len(keys) + 1))(*np.concatenate([[0], np.cumsum([len(k) for k in keys])]).tolist())
err = C.create_string_buffer(512)
rc = host.ls_bam_split(os.fsencode(tmp + "/raw.bam"), 1, (C.c_char_p * 1)(os.fsencode(tmp + "/idx/x.bam")), b"".join(keys),
                       off, (C.c_int32 * len(keys))(*([0] * len(keys))), C.c_int64(len(keys)), 0, -1, -1, 0,
                       min(32, os.cpu_count() or 1), 6, (C.c_int64 * 36)(), (C.c_int64 * 32)(), err, 512)
assert rc == 0, err.value
os.remove(tmp + "/raw.bam")
shutil.copy(tmp + "/idx/x.bam", tmp + "/plain/x.bam")
bam_mb = os.path.getsize(tmp + "/idx/x.bam") / 1e6
whole = bamio.read_bam(tmp + "/idx/x.bam").batch
rng = np.random.default_rng(7)


def sites_file(n, name):
    """n candidate sites inside reads, as a caller's candidates would be."""
    pick = rng.choice(whole.n_reads, min(whole.n_reads, 3 * n), replace=False)
    ks = sorted({(int(whole.tid[i]), int(whole.pos[i]) + int(rng.integers(0, 1000))) for i in pick})
    ks = [ks[i] for i in np.sort(rng.choice(len(ks), min(n, len(ks)), replace=False))]
    path = "%s/%s.tsv" % (tmp, name)
    with open(path, "w") as f:
        f.write("#CHROM\tStart\tEnd\tREF\tALT\n")
        for tid, p in ks:
            f.write("\t".join([contig_names[tid], str(p + 1), str(p + 1), "A", "ACGT"[p % 4], ".", "Cancer", ".", ".",
                               ".", ".", ".", ".", "3"]) + "\n")
    return path


with open(tmp + "/meta.tsv", "w") as f:
    f.write("Index\tCell_type\n")
    for c in range(20):
        f.write("%s-1\t%s\n" % (synth.barcode_of(c), d.cell_type(c)))
print("reads %d, BAM %.1f MB (inputs written in %.1f s)" % (b.n_reads, bam_mb, time.time() - t), flush=True)
contig_names = list(d.contig_names)
del b

GENO = ("import sys; from longsom_b200.cli.genotype import main; from longsom_b200.pipeline import _peak_rss_gb; "
        "main(sys.argv[2:], hccv=sys.argv[1] == 'hccv'); print('[run] peak RSS %.3f GB' % _peak_rss_gb(), file=sys.stderr)")
COUNT = ("import sys; from longsom_b200.cli.counter import main; from longsom_b200.pipeline import _peak_rss_gb; "
         "main(sys.argv[1:]); print('[run] peak RSS %.3f GB' % _peak_rss_gb(), file=sys.stderr)")
runs = []
for n in (100, 1000, 10000):
    runs.append(("HCCVSingleCellGenotype %d sites" % n, GENO, ["hccv", "--infile", sites_file(n, "h%d" % n), "--ref",
                 tmp + "/ref.fa", "--meta", tmp + "/meta.tsv", "--min_mq", "60"], "--outfile", ""))
for n in (1000, 10000):
    runs.append(("SingleCellGenotype %d sites" % n, GENO, ["geno", "--infile", sites_file(n, "g%d" % n), "--ref",
                 tmp + "/ref.fa", "--meta", tmp + "/meta.tsv", "--fusions", "--min_mq", "60"], "--outfile", ""))
for chrom in (contig_names[0], "all"):
    runs.append(("BaseCellCounter --chrom %s" % chrom, COUNT, ["--ref", tmp + "/ref.fa", "--chrom", chrom, "--min_bq", "20",
                 "--min_mq", "60"], "--out_folder", ""))


def outputs(kind, out):
    if kind == "--out_folder":
        return [os.path.join(out, f) for f in sorted(os.listdir(out)) if f.endswith(".tsv")]
    return sorted(os.path.join(os.path.dirname(out), f) for f in os.listdir(os.path.dirname(out))
                  if f.startswith(os.path.basename(out)))


res = []
for label, code, args, out_flag, _ in runs:
    row = dict(run=label)
    produced = {}
    for rep in range(repeats):
        for arm in ("indexed", "whole") if rep % 2 == 0 else ("whole", "indexed"):
            bam = tmp + ("/idx/x.bam" if arm == "indexed" else "/plain/x.bam")
            out = "%s/out_%s_%s" % (tmp, arm, abs(hash(label)))
            shutil.rmtree(out, ignore_errors=True)
            os.makedirs(out)
            dest = out if out_flag == "--out_folder" else out + "/o"
            extra = ["--id", "x.t"] if out_flag == "--out_folder" else []
            os.sync()
            t0 = time.time()
            r = subprocess.run([sys.executable, "-c", code] + args + ["--bam", bam, out_flag, dest, "--tmp_dir", out + "/t"]
                               + extra, env=dict(os.environ, PYTHONPATH=ROOT, LS_BAM_TIMING="1"),
                               stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
            dt = time.time() - t0
            assert r.returncode == 0, r.stderr[-3000:]
            comp = infl = 0
            used = False
            for line in r.stderr.splitlines():
                if line.startswith("[ls_bamstream]") and "compressed bytes read" in line:
                    tail = line.split("compressed bytes read ")[1]
                    comp += int(tail.split(",")[0])
                    infl += int(tail.split("inflated bytes ")[1].split(",")[0])
                    used |= "index used" in line
            rss = float([l for l in r.stderr.splitlines() if l.startswith("[run] peak RSS")][0].split()[3])
            prev = row.get(arm)
            if prev is None or dt < prev["seconds"]:
                row[arm] = dict(seconds=round(dt, 2), compressed_mb=round(comp / 1e6, 1), inflated_mb=round(infl / 1e6, 1),
                                peak_rss_gb=rss, index_used=used)
            produced[arm] = outputs(out_flag, dest)
    a, w = produced["indexed"], produced["whole"]
    assert [os.path.basename(p) for p in a] == [os.path.basename(p) for p in w] and a, (a, w)
    for x, y in zip(a, w):  # the counter's ##fileDate line aside, byte for byte
        strip = lambda path: [l for l in open(path, "rb") if not l.startswith(b"##fileDate")]
        assert strip(x) == strip(y), "outputs differ: " + x
    res.append(row)
    i, w = row["indexed"], row["whole"]
    print("%-34s indexed %7.2f s %8.1f MB read %8.1f MB inflated %.2f GB RSS | whole %7.2f s %8.1f MB read %8.1f MB "
          "inflated %.2f GB RSS | outputs identical" % (label, i["seconds"], i["compressed_mb"], i["inflated_mb"],
                                                         i["peak_rss_gb"], w["seconds"], w["compressed_mb"], w["inflated_mb"],
                                                         w["peak_rss_gb"]), flush=True)
print(json.dumps({"cards": card, "scale": scale, "bam_mb": round(bam_mb, 1), "reads": int(whole.n_reads), "runs": res}))
shutil.rmtree(tmp, ignore_errors=True)
