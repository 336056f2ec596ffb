"""CPU-only checks: ABI surface, host restatement of the special functions vs scipy,
oracle vs hand-built pileup cases (SURVEY Appendix A corner cases)."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_abi_exports_every_declared_symbol(built):
    from longsom_b200 import _lib
    hdr = open(os.path.join(ROOT, "include", "longsom_b200.h")).read()
    declared = set(re.findall(r"\b(ls_[a-z0-9_]+)\s*\(", hdr))
    declared -= {"ls_ctx"}
    lib = C.CDLL(_lib.LIB_PATH)
    for name in sorted(declared):
        assert hasattr(lib, name), name
    assert declared == set(_lib.ABI_SYMBOLS)
    assert lib.ls_abi_version() == 1


def test_host_abi_exports_every_declared_symbol(built):
    """include/longsom_host.h <-> liblongsom_host.so (BAM decoder, TSV row writer, BAM splitter)."""
    from longsom_b200 import bamio
    hdr = open(os.path.join(ROOT, "include", "longsom_host.h")).read()
    body = hdr[hdr.index("extern \"C\""):]
    declared = set(re.findall(r"\b(ls_[a-z0-9_]+)\s*\(", body))
    assert len(declared) >= 15
    lib = bamio._load_host()
    for name in sorted(declared):
        assert hasattr(lib, name), name


def test_no_cuda_device_fails_loudly(built):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from longsom_b200._lib import LongSomError
    from longsom_b200.engine import Engine
    with pytest.raises(LongSomError):
        Engine(0)


def test_product_does_not_import_oracle():
    """The product package must never route through oracle/ (no CPU fallback)."""
    bad = []
    for base in ("longsom_b200", "workflow"):
        for dp, _, files in os.walk(os.path.join(ROOT, base)):
            for f in files:
                if f.endswith((".py", ".cu", ".cuh", ".h", ".c", ".cpp")):
                    src = open(os.path.join(dp, f), errors="ignore").read()
                    if re.search(r"^\s*(import|from)\s+oracle\b", src, re.M) or "liboracle" in src:
                        bad.append(os.path.join(dp, f))
    assert not bad, bad


@pytest.fixture(scope="module")
def cephes(built):
    so = os.path.join(ROOT, "tests", "support", "libcephes_host.so")
    src = os.path.join(ROOT, "tests", "support", "cephes_host.c")
    subprocess.check_call(["/usr/bin/gcc", "-O2", "-fPIC", "-shared", "-o", so, src, "-lm"])
    lib = C.CDLL(so)
    for f in ("h_lbeta", "h_lgam", "h_Gamma"):
        getattr(lib, f).restype = C.c_double
    lib.h_lbeta.argtypes = [C.c_double] * 2
    lib.h_lgam.argtypes = [C.c_double]
    lib.h_Gamma.argtypes = [C.c_double]
    lib.h_betabinom_sf.argtypes = [C.c_void_p, C.c_void_p, C.c_double, C.c_double, C.c_void_p, C.c_int64, C.c_void_p]
    return lib


def test_cephes_restatement_matches_scipy(cephes):
    import scipy.special as sp
    rng = np.random.default_rng(0)
    xs = np.concatenate([rng.uniform(0.01, 200, 5000), rng.uniform(100, 3e5, 5000), np.arange(1, 400, dtype=float)])
    g = np.array([cephes.h_lgam(x) for x in xs])
    assert np.array_equal(g, sp.gammaln(xs))
    xs2 = xs[xs < 171]
    assert np.array_equal(np.array([cephes.h_Gamma(x) for x in xs2]), sp.gamma(xs2))
    A = np.concatenate([rng.uniform(0.01, 300, 5000), rng.uniform(1, 2e5, 5000)])
    B = np.concatenate([rng.uniform(0.01, 300, 5000), rng.uniform(0.01, 2e5, 5000)])
    g = np.array([cephes.h_lbeta(a, b) for a, b in zip(A, B)])
    r = sp.betaln(A, B)
    assert np.max(np.abs(g - r) / np.maximum(1.0, np.abs(r))) < 5e-16


def test_host_sf_matches_scipy(cephes):
    from scipy.stats import betabinom
    rng = np.random.default_rng(1)
    n = np.concatenate([rng.integers(1, 300, 1500), rng.integers(300, 20000, 200), rng.integers(20000, 200000, 20)]).astype(np.int32)
    k = np.minimum((rng.random(len(n)) ** 3 * np.minimum(n, 3000)).astype(np.int32) + rng.integers(0, 3, len(n)).astype(np.int32), n + 1).astype(np.int32)
    p = np.zeros(len(n))
    scratch = np.zeros(300000)
    for a, b in [(0.260288007167716, 173.94711910763732), (0.08354121346569514, 103.47683488327257)]:
        cephes.h_betabinom_sf(k.ctypes.data, n.ctypes.data, a, b, p.ctypes.data, len(n), scratch.ctypes.data)
        ref = betabinom.sf(k - 0.1, n, a, b)
        assert np.max(np.abs(p - ref)) < 1e-14
        assert np.array_equal(np.round(p, 4), np.round(ref, 4))


def test_decoded_arrays_outlive_the_bam_object(built, tmp_path):
    """read_bam returns views into the native decoder's buffers: they must stay valid (and writable) after the
    BamData object is gone, and round-trip what write_bam wrote."""
    import gc
    import numpy as np
    from longsom_b200 import bamio, synth
    d = synth.generate(seed=3, contig_lens=[60000], n_genes=4, n_reads=400, n_cells=10)
    path = os.path.join(str(tmp_path), "x.bam")
    bamio.write_bam(path, d.contig_names, d.contig_lens, d.batch, lambda i: None if d.batch.cell[i] < 0 else "BC%d-1" % d.batch.cell[i])
    bd = bamio.read_bam(path, threads=3)
    b = bd.batch
    del bd
    gc.collect()
    for f in ("tid", "pos", "flag", "mapq", "cigar_off", "cigar", "l_qseq"):
        assert np.array_equal(getattr(b, f), getattr(d.batch, f)), f
    lq, bo, bo0 = b.l_qseq.astype(np.int64), b.base_off.astype(np.int64), d.batch.base_off.astype(np.int64)
    for i in (0, 1, b.n_reads // 2, b.n_reads - 1):
        assert np.array_equal(b.qual[bo[i]:bo[i] + lq[i]], d.batch.qual[bo0[i]:bo0[i] + lq[i]])
        assert not b.qual[bo[i] + lq[i]:bo[i + 1]].any()          # padding to 16 bases is zeroed
    b.qual[0] = 7   # writable view
    assert b.qual[0] == 7


def test_own_inflater_matches_zlib(built):
    """ls_inflate.h (the BGZF readers' DEFLATE decoder) against zlib on streams of every block type: random bytes
    (stored blocks), quality-like and base-like text (dynamic codes, short and long matches, period < 8), fixed-code
    streams, several blocks per stream; a wrong expected size, a truncated stream and garbage are refused."""
    import ctypes as C
    import zlib
    from longsom_b200 import bamio
    lib = bamio._load_host()
    lib.ls_inflate_raw.restype = C.c_int
    lib.ls_inflate_raw.argtypes = [C.c_char_p, C.c_int64, C.c_void_p, C.c_int64]
    rng = np.random.default_rng(3)

    def inflate(comp, n):
        out = np.full(n + 16, 0xEE, np.uint8)
        ok = lib.ls_inflate_raw(comp, len(comp), out.ctypes.data, n)
        assert (out[n:] == 0xEE).all(), "wrote past the end of the output"
        return ok, out[:n].tobytes()
    n_streams = 0
    for it in range(400):
        n = int(rng.integers(0, 65536)) if it % 25 else int(rng.integers(0, 50))
        mode = it % 6
        if mode == 0:
            d = rng.integers(0, 256, n, dtype=np.uint8)
        elif mode == 1:
            d = rng.integers(33, 74, n).astype(np.uint8)
        elif mode == 2:
            d = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, n)]
        elif mode == 3:
            d = np.where(rng.random(n) < 0.93, 65, rng.integers(0, 256, n)).astype(np.uint8)
        elif mode == 4:
            d = np.tile(rng.integers(0, 256, int(rng.integers(1, 12)), dtype=np.uint8), n + 1)[:n]
        else:
            d = (np.arange(n) * 7 % 251).astype(np.uint8)
        data = d.tobytes()
        strategy = [zlib.Z_DEFAULT_STRATEGY, zlib.Z_RLE, zlib.Z_HUFFMAN_ONLY, zlib.Z_FIXED][(it // 6) % 4]
        co = zlib.compressobj(it % 10, zlib.DEFLATED, -15, 8, strategy)
        comp = co.compress(data[:n // 2]) + (co.flush(zlib.Z_FULL_FLUSH) if it % 3 == 0 else b"") + co.compress(data[n // 2:]) + co.flush()
        ok, got = inflate(comp, n)
        assert ok == 1 and got == data, (it, n, mode)
        n_streams += 1
        if n > 4:
            assert inflate(comp, n - 1)[0] == 0
            assert inflate(comp, n + 1)[0] == 0
            assert inflate(comp[:-3], n)[0] == 0
    for it in range(2000):
        junk = rng.integers(0, 256, int(rng.integers(0, 200)), dtype=np.uint8).tobytes()
        inflate(junk, int(rng.integers(0, 70000)))   # must not crash or write out of bounds
    assert n_streams == 400


def test_numa_binding_helpers(built):
    """bind_near_gpu: the cpulist parser, and a silent no-op where there is no device / no NUMA information."""
    from longsom_b200.pipeline import _parse_cpulist, bind_near_gpu
    assert _parse_cpulist("0-3,8,10-11\n") == {0, 1, 2, 3, 8, 10, 11}
    assert _parse_cpulist("") == set()
    before = os.sched_getaffinity(0) if hasattr(os, "sched_getaffinity") else None
    import torch
    if not torch.cuda.is_available():
        assert bind_near_gpu(0) is None
        if before is not None:
            assert os.sched_getaffinity(0) == before


def test_early_cuda_warm_is_light_and_harmless(built):
    """_early.warm() must not pull the numeric stack in (its point is to run BESIDE those imports) and must swallow the
    absence of a device: the Engine created afterwards is what reports it."""
    import subprocess
    import sys
    code = ("import sys; sys.path.insert(0, %r)\n"
            "from longsom_b200 import _early\n"
            "t = _early.warm()\n"
            "assert 'numpy' not in sys.modules and 'pandas' not in sys.modules, sorted(sys.modules)\n"
            "t.join(60)\n"
            "assert not t.is_alive()\n"
            "import os; os.environ['LONGSOM_EARLY_CUDA'] = '0'\n"
            "assert _early.warm() is None\n"
            "os.environ['LONGSOM_GPUS'] = '3,1'; assert _early.first_device() == 3\n"
            "os.environ['LONGSOM_GPUS'] = '4'; assert _early.first_device() == 0\n"
            "print('ok')\n") % ROOT
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0 and r.stdout.strip() == "ok", r.stderr[-2000:]


def test_bench_dump_outputs_is_a_seeded_float64_sample(tmp_path, monkeypatch):
    """bench.py --dump-outputs: the same table gives the same files, the sampled rows are the rows site_index names,
    and counts_column_sums covers every row, not only the sample."""
    import bench
    from longsom_b200.batch import SiteCounts
    rng = np.random.default_rng(3)
    n = 1000
    s = SiteCounts(rng.integers(0, 3, n).astype(np.int32), np.sort(rng.integers(0, 1 << 30, n)).astype(np.int32),
                   rng.integers(0, 4, n).astype(np.uint8), rng.integers(0, 1 << 31, (n, 26)).astype(np.uint32))
    monkeypatch.setattr(bench, "DUMP_SITES", 100)
    bench.dump_outputs(str(tmp_path / "a"), s, 0, 1)
    bench.dump_outputs(str(tmp_path / "b"), s, 0, 1)
    names = ("site_index", "tid", "pos", "ref", "counts", "counts_column_sums")
    assert sorted(os.listdir(tmp_path / "a")) == sorted(x + ".npy" for x in names)
    got = {x: np.load(tmp_path / "a" / (x + ".npy")) for x in names}
    for x in names:
        assert got[x].dtype == np.float64
        assert np.array_equal(got[x], np.load(tmp_path / "b" / (x + ".npy")))
    idx = got["site_index"].astype(np.int64)
    assert idx.shape == (100,) and np.all(np.diff(idx) > 0)
    assert np.array_equal(got["pos"], s.pos[idx]) and np.array_equal(got["counts"], s.counts[idx])
    assert np.array_equal(got["counts_column_sums"], s.counts.sum(axis=0, dtype=np.uint64).astype(np.float64))
    bench.dump_outputs(str(tmp_path / "r"), s, 1, 2)
    assert np.load(tmp_path / "r" / "rank1_counts.npy").shape == (50, 26)
