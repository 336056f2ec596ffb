"""Wall clock and peak resident set of the drop-in SingleCellGenotype on a synthetic C2 BAM, with its two output stages
timed on their own.
- Long table: the device writer (write_long_table with the run's engine) and the host writer (the same child with
  write_long_table forced to engine=None), both at each size, their tables compared byte for byte.  The device arm also
  reports the write kernels' and device-to-host copies' time from events and the time of its file writes; each size
  reports a write floor, the same number of bytes written from memory to the same directory in blocks of the same size.
  HCCVSingleCellGenotype gets both arms at the largest size.
- Matrices: the device writer (write_matrices) at each size, and the reference's pandas pivots (pivot_long_dataframe) at
  the sizes listed for them, with the files of the two compared byte for byte.  At every size a seeded sample of matrix
  rows is checked against the long table's own values.
Sizes are long-table entries (sites x cells); the metadata lists `cells` barcodes.
usage: cli_genotype_matrix_timing.py [scale] [cells] [sizes, e.g. 1e6,1e7,1e8] [pandas sizes, e.g. 1e6,1e7]"""
import filecmp, json, os, subprocess, sys, tempfile, time
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from longsom_b200 import synth, bamio

scale = float(sys.argv[1]) if len(sys.argv) > 1 else 0.2
n_meta = int(sys.argv[2]) if len(sys.argv) > 2 else 5000
sizes = [int(float(x)) for x in (sys.argv[3] if len(sys.argv) > 3 else "1e6,1e7,1e8").split(",")]
pandas_sizes = [int(float(x)) for x in (sys.argv[4] if len(sys.argv) > 4 else "1e6,1e7").split(",") if x]
card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], stdout=subprocess.PIPE,
                      text=True).stdout.strip().splitlines()
print("cards:", card, flush=True)
d = synth.generate(**synth.config("C2", scale=scale))
tmp = tempfile.mkdtemp()
b = d.batch
names = [synth.barcode_of(c) + "-1" for c in range(max(d.n_cells + d.n_extra_cells, n_meta))]
bamio.write_bam(tmp + "/x.bam", d.contig_names, d.contig_lens, b, lambda i: None if b.cell[i] < 0 else names[b.cell[i]])
bamio.write_fasta(tmp + "/ref.fa", d.contig_names, [d.contig_seq(i) for i in range(len(d.contig_lens))])
with open(tmp + "/meta.tsv", "w") as f:
    f.write("Index\tCell_type\n")
    for c in range(n_meta):
        f.write("%s\t%s\n" % (names[c], d.cell_type(c) if c < d.n_cells else "Cancer"))
rng = np.random.default_rng(7)
pick = rng.choice(b.n_reads, min(b.n_reads, 3 * max(sizes) // n_meta), replace=False)
all_keys = sorted({(int(b.tid[i]), int(b.pos[i]) + int(rng.integers(0, 100))) for i in pick})
print("reads %d, BAM %.1f MB, %d candidate sites available, %d cells" % (b.n_reads, os.path.getsize(tmp + "/x.bam") / 1e6,
                                                                        len(all_keys), n_meta), flush=True)

# the stages run in the child: the stage functions are wrapped with timers; the pandas arm skips the matrix writer and
# the host arm takes the long table from the host writer
RUN = r"""
import json, sys, time
from longsom_b200.cli import genotype as G
from longsom_b200.pipeline import _peak_rss_gb
T = {}
def timed(name, f):
    def w(*a, **k):
        t = time.time(); r = f(*a, **k); T[name] = T.get(name, 0.0) + time.time() - t; return r
    return w
arm, hccv = sys.argv.pop(1), sys.argv.pop(1) == "hccv"
long_table = G.write_long_table
def write_long_table(*a, engine=None):
    if len(a) > 8:
        a, engine = a[:8], a[8]
    src = long_table(*a, engine=None if arm == "host" else engine)
    T["long_stats"] = src.long_stats
    return src
G.write_long_table = timed("long_table", write_long_table)
G.pivot_long_dataframe = timed("pandas", G.pivot_long_dataframe)
if arm == "pandas":
    G.write_matrices = lambda *a, **k: False
else:
    G.write_matrices = timed("matrices", G.write_matrices)
G.main(sys.argv[1:], hccv=hccv)
print("[timing] " + json.dumps(dict(T, peak_rss_gb=_peak_rss_gb())), file=sys.stderr)
"""
KINDS = ("DpMatrix", "AltMatrix", "VAFMatrix", "BinaryMatrix")


def check_sample(prefix, n_sample=20):
    """Rows of the matrices against the long table's own values, on a seeded sample of rows: Dp, Alt, VAF and
    BinMutationStatus of every (site, cell), read from the long table with plain Python."""
    with open(prefix + ".DpMatrix.tsv") as f:
        cols = f.readline().rstrip("\n").split("\t")[1:]
        labels = [line.split("\t", 1)[0] for line in f]
    want = set(np.random.default_rng(3).choice(len(labels), min(n_sample, len(labels)), replace=False).tolist())
    want_labels = {labels[i] for i in want}
    vals = {}
    with open(prefix + ".SingleCellGenotype.tsv") as f:
        f.readline()
        for line in f:
            e = line.rstrip("\n").split("\t")
            if e[15] in want_labels:
                vals[(e[15], e[7])] = (e[9], e[10], e[11], e[14])
    for k, name in enumerate(KINDS):
        with open(prefix + "." + name + ".tsv") as f:
            f.readline()
            for i, line in enumerate(f):
                if i in want:
                    e = line.rstrip("\n").split("\t")
                    assert [vals[(e[0], c)][k] for c in cols] == e[1:], (name, e[0])
    return len(want)


def same_bytes(a, b, block=64 << 20):
    if os.path.getsize(a) != os.path.getsize(b):
        return False
    with open(a, "rb") as fa, open(b, "rb") as fb:
        while True:
            x, y = fa.read(block), fb.read(block)
            if x != y:
                return False
            if not x:
                return True


def write_floor(nbytes, path, block=64 << 20):
    """Seconds to write nbytes from memory to path in blocks of `block` bytes, as the long table's writer does."""
    buf = memoryview(bytes(b"0123456789abcdef" * (block // 16)))
    t = time.time()
    with open(path, "wb") as f:
        left = nbytes
        while left > 0:
            f.write(buf[:min(block, left)])
            left -= block
    dt = time.time() - t
    os.remove(path)
    return dt


def run(arm, hccv, prefix):
    """One child run of one script: its row of the table and the path of its long table."""
    os.sync()  # every arm starts without the previous arm's dirty pages
    script = ["--fusions", "--outfile", prefix] if not hccv else ["--outfile", prefix + ".hccv.tsv"]
    t0 = time.time()
    r = subprocess.run([sys.executable, "-c", RUN, arm, "hccv" if hccv else "scg", "--bam", tmp + "/x.bam", "--infile",
                        tmp + "/cand.tsv", "--ref", tmp + "/ref.fa", "--meta", tmp + "/meta.tsv", "--min_mq", "60",
                        "--tmp_dir", tmp + "/t"] + script,
                       env=dict(os.environ, PYTHONPATH=ROOT), stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
    wall = time.time() - t0
    assert r.returncode == 0, r.stderr[-3000:]
    t = json.loads([l for l in r.stderr.splitlines() if l.startswith("[timing] ")][0][9:])
    long_path = prefix + ".hccv.tsv" if hccv else prefix + ".SingleCellGenotype.tsv"
    row = dict(script="HCCVSingleCellGenotype" if hccv else "SingleCellGenotype", entries=len(keys) * n_meta,
               sites=len(keys), cells=n_meta, arm=arm, wall_s=round(wall, 2), long_table_s=round(t["long_table"], 2),
               long_mb=round(os.path.getsize(long_path) / 1e6, 1), peak_rss_gb=round(t["peak_rss_gb"], 3))
    ls = t.get("long_stats")
    if ls:
        row.update(text_ms=round(ls["ms_text"], 1), d2h_ms=round(ls["ms_copy"], 1), file_write_s=round(ls["write_s"], 2),
                   blocks=ls["blocks"], block_mb=round(ls["bytes"] / max(1, ls["blocks"]) / 1e6, 1),
                   text_ms_per_block=round(ls["ms_text"] / max(1, ls["blocks"]), 3))
    if not hccv:
        row.update(matrix_s=round(t.get("matrices", t.get("pandas", 0.0)), 2),
                   matrix_mb=round(sum(os.path.getsize(prefix + "." + k + ".tsv") for k in KINDS) / 1e6, 1))
        if arm != "pandas":
            row["rows_checked"] = check_sample(prefix)
    res.append(row)
    print(json.dumps(row), flush=True)
    return long_path


res = []
for size in sizes:
    n_sites = max(1, size // n_meta)
    keys = [all_keys[i] for i in np.sort(rng.choice(len(all_keys), min(n_sites, len(all_keys)), replace=False))]
    with open(tmp + "/cand.tsv", "w") as f:
        f.write("#CHROM\tStart\tEnd\tREF\tALT\n")
        for tid, p in keys:
            f.write("\t".join([d.contig_names[tid], str(p + 1), str(p + 1), "A", "ACGT"[p % 4], ".", "Cancer", ".", ".",
                               ".", ".", ".", ".", "3"]) + "\n")
    for hccv in ((False, True) if size == max(sizes) else (False,)):
        out = {}
        for arm in ["host", "device"] + (["pandas"] if size in pandas_sizes and not hccv else []):
            prefix = "%s/%s_%d" % (tmp, arm, size)
            out[arm] = (prefix, run(arm, hccv, prefix))
        assert same_bytes(out["host"][1], out["device"][1]), "long tables differ"
        floor = write_floor(os.path.getsize(out["device"][1]), tmp + "/floor.bin")
        print(json.dumps(dict(entries=len(keys) * n_meta, hccv=hccv, long_tables_identical=True,
                              write_floor_s=round(floor, 2))), flush=True)
        res.append(dict(entries=len(keys) * n_meta, hccv=hccv, write_floor_s=round(floor, 2)))
        if "pandas" in out:
            for k in KINDS:
                assert filecmp.cmp(out["device"][0] + "." + k + ".tsv", out["pandas"][0] + "." + k + ".tsv",
                                   shallow=False), k
            print("entries %d: device and pandas matrices identical" % (len(keys) * n_meta), flush=True)
        for arm, (prefix, long_path) in out.items():
            for path in [long_path] + ([prefix + "." + k + ".tsv" for k in KINDS] if not hccv else []):
                os.remove(path)
print(json.dumps({"cards": card, "scale": scale, "cells": n_meta, "runs": res}))
