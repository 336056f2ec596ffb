"""Paths that a fresh upload followed by one call never reaches, each compared with the CPU oracle or scipy:
replayed pileup runs on one upload (the path a steady stream of batches and bench.py take), the branches of sparse
genotyping (depth cap, hit-key width, deep pairs, the shallow-pair table, empty slots) and the chunked host entry of
the beta-binomial tail kernel."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from longsom_b200 import synth
from longsom_b200._lib import CLASS_ID
from longsom_b200.batch import ReadBatch, Windows, make_windows
from longsom_b200.engine import CountParams
from test_pileup_gpu import CASES, _compare

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
AB = (0.2474528917555431, 162.03696139428595)  # alpha / beta of a genotype run (as in test_configs_gpu)
TABLE_MIN_TUPLES = 4 * 65 * 65  # above this many tuples the sparse path looks shallow pairs up in a (k, n) <= 64 table
STAGED_CHUNK_TERMS = 1 << 26    # pmf terms per chunk of ls_betabinom_sf's staged path


def _windows(d):
    return Windows.from_intervals(make_windows(d.contig_lens, 50000), d.contig_seqs())


def _with_cells(b, cell):
    return ReadBatch(b.tid, b.pos, b.flag, b.mapq, np.asarray(cell, np.int32), b.cigar_off, b.cigar, b.base_off,
                     b.l_qseq, b.seq4, b.qual)


def _oracle_sites(d, n, seed):
    """n random covered sites (sorted), from the oracle's pileup table, with their upper-case reference bases."""
    import oracle
    sc = oracle.pileup_count(d.batch, _windows(d), CountParams(min_bq=20, min_mq=60, min_dp=1, min_cc=1), threads=8)[0]
    rng = np.random.default_rng(seed)
    idx = np.sort(rng.choice(sc.n_sites, size=min(n, sc.n_sites), replace=False))
    return sc.tid[idx], sc.pos[idx], sc.ref[idx]


def _ref_class(ref):
    return np.array([CLASS_ID[chr(r)] for r in ref], np.uint8)


# ---- A. pileup replay: one upload, several runs ----------------------------------------------------------------------

def _run(engine, prm):
    """One step as bench.py times it (run + compact), then the sites.  A replayed run compacts inside run(), so only
    a replay reports a compaction time from run()."""
    n = engine.run(prm)
    replayed = engine.last_stats["ms_compact"] > 0
    engine.compact()
    stats = dict(engine.last_stats)
    return engine.fetch(n), replayed, stats


FEW_CELLS = dict(seed=8, contig_lens=[100000], n_genes=3, n_reads=20000, n_cells=3, n_extra_cells=1, n_hot_genes=1,
                 hot_fraction=0.9)
REPLAY = [
    (CASES[0], dict(min_bq=20, min_mq=60)),                       # chrM, 200 cells
    (CASES[2], dict(min_bq=20, min_mq=60, min_ac=2)),             # hot genes, multi-part tiles, uncounted-read buffer
    (CASES[5], dict(min_bq=30, min_mq=0, min_dp=1, min_cc=1)),    # 6 kb reads: the cold run relaunches the builder
    (FEW_CELLS, dict(min_bq=20, min_mq=60, min_dp=5, min_cc=2)),  # 3 cells: unpacked counters
]


@pytest.mark.parametrize("case", range(len(REPLAY)))
def test_replayed_runs_match_oracle(engine, monkeypatch, case):
    import oracle
    cfg, prm = REPLAY[case]
    d = synth.generate(**cfg)
    w = _windows(d)
    p = CountParams(**prm)
    want, nal = oracle.pileup_count(d.batch, w, p, threads=8)
    assert want.n_sites > 0
    engine.upload(d.batch, w)
    for i in range(3):
        got, replayed, st = _run(engine, p)
        assert replayed == (i > 0), i
        _compare(got, want)
        assert st["n_aligned"] == nal
    monkeypatch.setenv("LS_NO_REPLAY", "1")
    got, replayed, _ = _run(engine, p)
    assert not replayed
    _compare(got, want)
    monkeypatch.delenv("LS_NO_REPLAY")
    got, replayed, _ = _run(engine, p)
    assert replayed
    _compare(got, want)


def test_replay_after_a_capped_run(engine):
    """P1 (nothing dropped: its sizes are cached), P2 (the depth cap drops reads: fewer segments and pieces), P1 again.
    The runs after P2 must size the segment builder for P1, not for what P2 left behind."""
    import oracle
    d = synth.generate(seed=5, contig_lens=[120000], n_genes=4, n_reads=20000, n_cells=300, n_hot_genes=1,
                       hot_fraction=0.8)
    w = _windows(d)
    p1 = CountParams(min_bq=20, min_mq=0)
    p2 = CountParams(min_bq=20, min_mq=60, max_depth=50)
    want1 = oracle.pileup_count(d.batch, w, p1, threads=8)[0]
    want2 = oracle.pileup_count(d.batch, w, p2, threads=8)[0]
    uncapped2 = oracle.pileup_count(d.batch, w, CountParams(min_bq=20, min_mq=60, max_depth=0), threads=8)[0]
    assert uncapped2.counts[:, 0].sum() > want2.counts[:, 0].sum()  # P2's cap really drops reads
    engine.upload(d.batch, w)
    got, _, st1 = _run(engine, p1)
    _compare(got, want1)
    got, _, st2 = _run(engine, p2)
    _compare(got, want2)
    assert st2["n_segments"] < st1["n_segments"]
    for _ in range(2):
        got, replayed, st = _run(engine, p1)
        _compare(got, want1)
        assert st["n_segments"] == st1["n_segments"]
    assert replayed  # P1 is replayed again, at the latest on its second run after P2


def test_replay_survives_other_kernels(engine):
    """Genotyping (dense and sparse, depth cap 100), beta-binomial tails (staged path) and site masks share
    counters, scan scratch, sort histograms and the genotype buffers with the pileup: a replay after them is still a
    replay and gives the same sites."""
    import oracle
    d = synth.generate(**CASES[0])
    w = _windows(d)
    p = CountParams(min_bq=20, min_mq=60)
    engine.upload(d.batch, w)
    first, _, _ = _run(engine, p)
    got, replayed, _ = _run(engine, p)
    assert replayed
    _compare(got, first)
    rng = np.random.default_rng(3)
    st, sp = first.tid[::5], first.pos[::5]
    alt = rng.integers(0, 4, st.shape[0]).astype(np.uint8)
    engine.genotype_sparse(st, sp, alt, d.n_cells, *AB, min_bq=30, min_mq=60, max_depth=100)
    engine.genotype_count(st, sp, alt, d.n_cells, min_bq=30, min_mq=60, max_depth=100)
    engine.betabinom_sf(np.array([5, 150000, 3000, 170000], np.int32), np.array([40, 200000, 9000, 200000], np.int32),
                        *AB)
    keys = (first.tid.astype(np.uint64) << np.uint64(32)) | first.pos.astype(np.uint64)
    assert engine.site_mask(keys, keys[::3]).all()
    got, replayed, _ = _run(engine, p)
    assert replayed
    _compare(got, first)
    _compare(got, oracle.pileup_count(d.batch, w, p, threads=8)[0])


# ---- B. sparse genotyping against the oracle's dense tensors ---------------------------------------------------------

def _check_tuples(engine, tup, odp, oal, skip=None, cell_map=None):
    """The tuples are the non-zero entries of the dense oracle tensors in (site, cell) order (cells through cell_map);
    p is what ls_betabinom_sf gives for the same (Alt, Dp), bit for bit, NaN where no tail is needed, and within
    1e-9 p + 1e-12 of scipy.  Returns the query mask."""
    from scipy.stats import betabinom
    site, cell, sdp, sal, p = tup
    ri, ci = np.nonzero(odp > 0)
    assert site.shape[0] == ri.shape[0], (site.shape[0], ri.shape[0])
    assert np.array_equal(site, ri)
    assert np.array_equal(cell, ci if cell_map is None else cell_map[ci])
    assert np.array_equal(sdp, odp[ri, ci]) and np.array_equal(sal, oal[ri, ci])
    q = sal > 0
    if skip is not None:
        q &= skip[site] == 0
    assert np.all(np.isnan(p[~q]))
    if q.any():
        want = engine.betabinom_sf(sal[q], sdp[q], *AB)
        assert np.array_equal(p[q], want), np.nonzero(p[q] != want)[0][:10]
        ref = betabinom.sf(sal[q] - 0.001, sdp[q], *AB)
        assert np.all(np.abs(p[q] - ref) <= 1e-9 * ref + 1e-12), np.abs(p[q] - ref).max()
    return q


HOT = dict(seed=22, contig_lens=[120000], n_genes=4, n_reads=15000, n_cells=100, n_hot_genes=1, hot_fraction=0.8)


@pytest.mark.parametrize("alt_only", [False, True])
def test_sparse_depth_cap(engine, alt_only):
    """The depth cap fires in the sparse path (slot counts and drops from the same walk over the CIGARs)."""
    import oracle
    d = synth.generate(**HOT)
    st, sp, _ = _oracle_sites(d, 500, 1)
    alt = np.random.default_rng(2).integers(0, 9, st.shape[0]).astype(np.uint8)  # includes O (7) and NA (8)
    kw = dict(min_bq=30, min_mq=60, alt_only=alt_only)
    udp, _ = oracle.genotype_count(d.batch, st, sp, alt, d.n_cells, max_depth=0, **kw)
    engine.upload(d.batch)
    for cap in (100, 2000):
        odp, oal = oracle.genotype_count(d.batch, st, sp, alt, d.n_cells, max_depth=cap, **kw)
        assert udp.sum() > odp.sum(), cap  # the cap fired
        tup = engine.genotype_sparse(st, sp, alt, d.n_cells, *AB, max_depth=cap, **kw)
        _check_tuples(engine, tup, odp, oal)


def _wide_cell_case():
    """60 barcoded cells, 1000 covered sites, and the oracle's tuples.  Every tenth barcoded read is given cell id 60 or
    67 (and the synthetic extra barcodes 60..62 stay): outside the 60 cells, so they must not count.  The last site is
    covered by cell 59 with reads of its alt class, so (999, 59) is the last tuple and carries the largest key."""
    import oracle
    C0 = 60
    d = synth.generate(seed=31, contig_lens=[90000], n_genes=6, n_reads=6000, n_cells=C0, n_extra_cells=3)
    cell = d.batch.cell.copy()
    own = np.nonzero((cell >= 0) & (cell < C0))[0]
    cell[own[0::20]] = C0
    cell[own[10::20]] = C0 + 7
    b = _with_cells(d.batch, cell)
    st, sp, ref = _oracle_sites(d, 3000, 4)
    odp, _ = oracle.genotype_count(b, st, sp, np.zeros(st.shape[0], np.uint8), C0, min_bq=30, min_mq=60)
    keep = np.nonzero(odp.sum(axis=1) > 0)[0][:1000]
    assert keep.shape[0] == 1000
    st, sp, ref = st[keep], sp[keep], ref[keep]
    alt = np.random.default_rng(5).integers(0, 4, 1000).astype(np.uint8)
    alt[-1] = _ref_class(ref[-1:])[0]
    dp, al = oracle.genotype_count(b, st, sp, alt, C0, min_bq=30, min_mq=60)
    c = int(np.nonzero(al[-1] > 0)[0][-1])  # a cell with alt reads at the last site becomes cell C0 - 1
    swap = np.arange(C0 + 8, dtype=np.int32)
    swap[c], swap[C0 - 1] = C0 - 1, c
    b = _with_cells(b, np.where(cell >= 0, swap[np.maximum(cell, 0)], -1))
    dp, al = oracle.genotype_count(b, st, sp, alt, C0, min_bq=30, min_mq=60)
    assert dp[-1, C0 - 1] > 0 and al[-1, C0 - 1] > 0
    return b, st, sp, alt, dp, al, C0


@pytest.mark.parametrize("n_cells", [2_147_483, 2_147_484])
def test_sparse_hit_keys_at_2_32(engine, n_cells):
    """1000 sites x n_cells x 2 is just below 2^32 (32-bit hit keys, all 32 bits used) or just above (64-bit keys).
    The batch's 60 cells are spread over [0, n_cells) by an increasing map that sends the last one to n_cells - 1;
    ids n_cells and n_cells + 7 lie outside and are dropped."""
    b, st, sp, alt, dp, al, C0 = _wide_cell_case()
    key_span = 1000 * n_cells * 2
    assert (key_span < 2 ** 32) == (n_cells == 2_147_483)
    rng = np.random.default_rng(6)
    cmap = np.concatenate([np.sort(rng.choice(n_cells - 1, C0 - 1, replace=False)), [n_cells - 1]]).astype(np.int64)
    lut = np.concatenate([cmap, n_cells + np.arange(8)])  # ids C0..C0 + 7 -> n_cells..n_cells + 7: past the last cell
    wide = np.where(b.cell < 0, -1, lut[np.maximum(b.cell, 0)])
    assert (wide == n_cells).any() and (wide == n_cells + 7).any()
    engine.upload(_with_cells(b, wide))
    tup = engine.genotype_sparse(st, sp, alt, n_cells, *AB, min_bq=30, min_mq=60)
    _check_tuples(engine, tup, dp, al, cell_map=cmap)
    site, cell, _, sal, _ = tup
    assert (site[-1], cell[-1]) == (999, n_cells - 1) and sal[-1] > 0  # key (key_span - 2) | 1: the largest real key


def test_sparse_forced_64bit_keys_identical(engine, monkeypatch):
    """LS_GENO_KEYS64=1 sorts 64-bit hit keys where 32 bits would do: the tuples must not change."""
    d = synth.generate(**HOT)
    st, sp, _ = _oracle_sites(d, 800, 7)
    alt = np.random.default_rng(8).integers(0, 4, st.shape[0]).astype(np.uint8)
    engine.upload(d.batch)
    a = engine.genotype_sparse(st, sp, alt, d.n_cells, *AB, min_bq=30, min_mq=60)
    monkeypatch.setenv("LS_GENO_KEYS64", "1")
    b = engine.genotype_sparse(st, sp, alt, d.n_cells, *AB, min_bq=30, min_mq=60)
    assert a[0].shape[0] > 1000
    for x, y in zip(a, b):
        assert np.array_equal(x, y, equal_nan=True)


def test_sparse_deep_pairs(engine):
    """3 cells on a hot gene, half the sites asking for the reference base: Alt ~ Dp in the hundreds to thousands.
    Pairs with Alt > 128 leave the in-register kernel (p = -1 on the device) and are finished by the fetch through
    the staged path; pairs with Dp in 65..128 are past the shallow-pair table."""
    import oracle
    d = synth.generate(**FEW_CELLS)
    st, sp, ref = _oracle_sites(d, 400, 9)
    rng = np.random.default_rng(10)
    alt = rng.integers(0, 4, st.shape[0]).astype(np.uint8)
    alt[0::2] = _ref_class(ref[0::2])
    skip = (np.arange(st.shape[0]) % 5 == 3).astype(np.uint8)
    odp, oal = oracle.genotype_count(d.batch, st, sp, alt, d.n_cells, min_bq=30, min_mq=60)
    engine.upload(d.batch)
    tup = engine.genotype_sparse(st, sp, alt, d.n_cells, *AB, skip_p=skip, min_bq=30, min_mq=60)
    q = _check_tuples(engine, tup, odp, oal, skip=skip)
    _, _, sdp, sal, _ = tup
    assert (sal[q] > 128).sum() > 10
    assert ((sdp[q] >= 65) & (sdp[q] <= 128)).any()


def test_sparse_table_and_no_table_agree(engine):
    """The same pairs, once in a call small enough to evaluate every tail in registers and once in a call that looks
    shallow pairs up in the (k, n) <= 64 table: every (Alt, Dp) gets one p, the one ls_betabinom_sf gives."""
    import oracle
    cfg = synth.config("C5", scale=0.02)
    cfg["n_cells"] = 200
    d = synth.generate(**cfg)
    st, sp, ref = _oracle_sites(d, 5000, 11)
    alt = np.random.default_rng(12).integers(0, 4, st.shape[0]).astype(np.uint8)
    alt[0::3] = _ref_class(ref[0::3])  # Alt = Dp at a third of the sites, a few mismatches elsewhere
    odp, oal = oracle.genotype_count(d.batch, st, sp, alt, d.n_cells, min_bq=30, min_mq=60)
    engine.upload(d.batch)
    full = engine.genotype_sparse(st, sp, alt, d.n_cells, *AB, min_bq=30, min_mq=60)
    assert full[0].shape[0] > TABLE_MIN_TUPLES
    qf = _check_tuples(engine, full, odp, oal)
    few = engine.genotype_sparse(st[:300], sp[:300], alt[:300], d.n_cells, *AB, min_bq=30, min_mq=60)
    assert 0 < few[0].shape[0] <= TABLE_MIN_TUPLES
    qs = _check_tuples(engine, few, odp[:300], oal[:300])
    # the small call's shallow pairs are among the large call's
    shallow = lambda t, q: set(zip(t[3][q & (t[2] <= 64)].tolist(), t[2][q & (t[2] <= 64)].tolist()))
    assert len(shallow(few, qs)) > 20 and shallow(few, qs) <= shallow(full, qf)
    pf = {(a, n): x for a, n, x in zip(full[3][qf].tolist(), full[2][qf].tolist(), full[4][qf].tolist())}
    for a, n, x in zip(few[3][qs].tolist(), few[2][qs].tolist(), few[4][qs].tolist()):
        assert pf[(a, n)] == x, (a, n)


def test_sparse_mostly_empty_slots(engine):
    """n_cells below the batch's largest cell id, --alt_flag Alt, chrM-style skipped sites and min_bq 40: most slots
    sized by the candidate walk receive no hit and stay sentinels."""
    import oracle
    d = synth.generate(**CASES[0])
    st, sp, _ = _oracle_sites(d, 2000, 13)
    alt = np.random.default_rng(14).integers(0, 9, st.shape[0]).astype(np.uint8)
    skip = (np.arange(st.shape[0]) % 4 == 1).astype(np.uint8)
    n_cells = 90
    assert d.batch.cell.max() >= 2 * n_cells
    kw = dict(min_bq=40, min_mq=60, alt_only=True)
    odp, oal = oracle.genotype_count(d.batch, st, sp, alt, n_cells, **kw)
    # every read entry of an in-range cell at a site, whatever its base and quality: fewer than the slots
    every, _ = oracle.genotype_count(d.batch, st, sp, alt, n_cells, min_bq=0, min_mq=60)
    engine.upload(d.batch)
    tup = engine.genotype_sparse(st, sp, alt, n_cells, *AB, skip_p=skip, **kw)
    hits = engine.last_stats["n_events"]
    _check_tuples(engine, tup, odp, oal, skip=skip)
    assert tup[0].shape[0] > 0
    assert hits == odp.sum() and hits < 0.2 * every.sum()


# ---- C. K2 host entry ------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def cephes(built, tmp_path_factory):
    """Host build of the restated special functions and the pairwise summation (tests/support/cephes_host.c)."""
    so = str(tmp_path_factory.mktemp("cephes") / "libcephes_host.so")
    subprocess.check_call(["/usr/bin/gcc", "-O2", "-fPIC", "-shared", "-o", so,
                           os.path.join(ROOT, "tests", "support", "cephes_host.c"), "-lm"])
    lib = C.CDLL(so)
    lib.h_betabinom_sf.argtypes = [C.c_void_p, C.c_void_p, C.c_double, C.c_double, C.c_void_p, C.c_int64, C.c_void_p]
    return lib


def _host_sf(cephes, k, n):
    k = np.ascontiguousarray(k, np.int32)
    n = np.ascontiguousarray(n, np.int32)
    p = np.zeros(k.shape[0])
    scratch = np.zeros(int(max(1, k.max())))
    cephes.h_betabinom_sf(k.ctypes.data, n.ctypes.data, AB[0], AB[1], p.ctypes.data, k.shape[0], scratch.ctypes.data)
    return p


def test_betabinom_staged_chunks(engine, cephes):
    """More than 1.5 x 2^26 pmf terms in one call: the staged path runs several chunks.  The result must not depend on
    how the queries are grouped into chunks."""
    from scipy.stats import betabinom
    rng = np.random.default_rng(15)
    nb, ns = 600, 2000
    n = np.concatenate([np.full(nb, 200000), rng.integers(1, 5000, ns)]).astype(np.int32)
    k = np.concatenate([rng.integers(150000, 200001, nb),
                        np.minimum(rng.integers(0, 400, ns), n[nb:] + 1)]).astype(np.int32)
    perm = rng.permutation(nb + ns)
    k, n = k[perm], n[perm]
    big = (k > 128) & (k <= n)
    assert k[big].astype(np.int64).sum() > 1.5 * STAGED_CHUNK_TERMS
    p = engine.betabinom_sf(k, n, *AB)
    g = 40
    parts = np.concatenate([engine.betabinom_sf(k[i:i + g], n[i:i + g], *AB) for i in range(0, k.shape[0], g)])
    assert np.array_equal(p, parts), np.nonzero(p != parts)[0][:10]
    host = np.concatenate([rng.choice(np.nonzero(big & (n == 200000))[0], 30, replace=False),
                           rng.choice(np.nonzero(n < 200000)[0], 20, replace=False)])
    hp = _host_sf(cephes, k[host], n[host])
    assert np.all(np.abs(p[host] - hp) <= 1e-9 * hp + 1e-12), np.abs(p[host] - hp).max()
    sci = np.concatenate([rng.choice(np.nonzero(big & (n == 200000))[0], 10, replace=False),
                          rng.choice(np.nonzero(big & (n < 200000))[0], 10, replace=False)])
    ref = betabinom.sf(k[sci] - 0.001, n[sci], *AB)
    assert np.all(np.abs(p[sci] - ref) <= 1e-9 * ref + 1e-12), np.abs(p[sci] - ref).max()


def test_betabinom_edges_land_at_their_index(engine):
    """k at the in-register limit (127 / 128 / 129), k = n, k > n, n = 0, k = 0 and n < 0 in one mixed call: every
    result lands at its own index, whichever path computed it."""
    from scipy.stats import betabinom
    edges = [(127, 5000), (128, 5000), (129, 5000), (5000, 5000), (5001, 5000), (5005, 5000), (128, 128), (129, 129),
             (130, 129), (0, 0), (1, 0), (0, 5000), (0, 129), (5, -1), (300, -2), (1, 1), (200, 20000), (129, 300)]
    rng = np.random.default_rng(16)
    fill_n = rng.integers(1, 3000, 200)
    fill = list(zip(np.minimum(rng.integers(0, 500, 200), fill_n).tolist(), fill_n.tolist()))
    qs = edges * 3 + fill
    order = rng.permutation(len(qs))
    k = np.array([qs[i][0] for i in order], np.int32)
    n = np.array([qs[i][1] for i in order], np.int32)
    p = engine.betabinom_sf(k, n, *AB)
    assert np.array_equal(p, engine.betabinom_sf(k[::-1], n[::-1], *AB)[::-1], equal_nan=True)
    for e in edges:
        i = np.nonzero((k == e[0]) & (n == e[1]))[0]
        one = engine.betabinom_sf(np.array([e[0]], np.int32), np.array([e[1]], np.int32), *AB)
        assert np.array_equal(p[i], np.repeat(one, i.shape[0]), equal_nan=True), e
    assert np.all(np.isnan(p[n < 0]))
    assert np.all(p[(n >= 0) & (k == 0)] == 1.0)
    assert np.all(p[(n >= 0) & (k > n)] == 0.0)
    v = (n >= 0) & (k > 0) & (k <= n)
    ref = betabinom.sf(k[v] - 0.001, n[v], *AB)
    assert np.all(np.abs(p[v] - ref) <= 1e-9 * ref + 1e-12), np.abs(p[v] - ref).max()
