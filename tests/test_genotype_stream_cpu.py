"""The chunk planner of the streamed genotype scripts (pipeline.plan_genotype_chunk) on hand-built reads, and the whole
streamed source (pipeline.stream_genotype) with the CPU oracle in place of the engine: every bin must receive, in the
chunk that completes it, exactly the reads that overlap its region, once, so that each chunk's pileup() calls see the
records the whole-file call sees."""
import numpy as np
import pytest

from longsom_b200 import bamio, pipeline, synth
from longsom_b200.cli.genotype import build_dict_variants, candidate_sites
from longsom_b200.pipeline import genotype_bins, plan_genotype_chunk


def keys(reads):
    """reads: [(tid, pos, end)] -> read_keys() of them."""
    t = np.array([r[0] for r in reads], np.int64) << 32
    p = np.array([r[1] for r in reads], np.int64)
    e = np.array([r[2] for r in reads], np.int64)
    return t | p, t | np.maximum(e, p + 1)


def bins_of(sites, bin_size=50000):
    """sites: [(tid, pos0)] sorted -> genotype_bins()."""
    return genotype_bins(np.array([s[0] for s in sites], np.int32), np.array([s[1] for s in sites], np.int32), bin_size)


def stream(reads, sites, cuts, bin_size=50000):
    """Feed reads (coordinate order) in chunks that end before the indices in `cuts`, carrying reads between chunks as
    stream_genotype's decoder does.  Returns {bin: ids of the reads sent with the chunk that completed it}."""
    rs, re_ = keys(reads)
    _, bs, be = bins_of(sites, bin_size)
    got, bi, carry = {}, 0, np.zeros(0, np.int64)
    edges = [0] + sorted(set(cuts) - {0}) + [len(reads)]
    chunks = [np.arange(a, c) for a, c in zip(edges[:-1], edges[1:]) if c > a] + [None]  # None: the end of the file
    for new in chunks:
        if bi >= be.shape[0] or (new is None and carry.shape[0] == 0):
            break
        if new is None:
            ids, last = carry, None
        else:
            ids = np.concatenate([carry, new])
            last = None if reads[new[-1]][0] < 0 else int(rs[new[-1]])
        done, send, keep = plan_genotype_chunk(rs[ids], re_[ids], bs, be, bi, last)
        assert np.unique(send).shape[0] == send.shape[0]
        for b in range(bi, done):
            assert b not in got, "bin %d completed twice" % b
            got[b] = ids[send]
        carry, bi = ids[keep], done
        if last is None:
            break
    assert bi == be.shape[0], "bins left incomplete"
    return got


def check(reads, sites, cuts, bin_size=50000):
    """Every bin gets exactly its overlapping reads; returns what stream() returned."""
    got = stream(reads, sites, cuts, bin_size)
    rs, re_ = keys(reads)
    _, bs, be = bins_of(sites, bin_size)
    for b in range(be.shape[0]):
        want = np.nonzero((rs < be[b]) & (re_ > bs[b]))[0]
        mine = got[b][(rs[got[b]] < be[b]) & (re_[got[b]] > bs[b])]
        assert np.array_equal(np.sort(mine), want), (b, mine, want)
        # nothing is sent that overlaps no complete bin of its chunk
        assert all(((rs[r] < be) & (re_[r] > bs)).any() for r in got[b])
    return got


def test_read_spanning_two_bins_completes_in_two_chunks():
    # bins [99, 101) and [50099, 50101) on contig 0; read 0 is spliced across both
    sites = [(0, 100), (0, 50100)]
    reads = [(0, 50, 60000), (0, 90, 300), (0, 200, 400), (0, 50090, 50200), (0, 60000, 60100)]
    got = check(reads, sites, cuts=[3])
    assert 0 in got[0] and 0 in got[1]  # sent once with each chunk
    assert sorted(got[0].tolist()) == [0, 1]
    assert sorted(got[1].tolist()) == [0, 3]


def test_region_ending_at_the_last_read_start_is_complete():
    # bin [99, 101): the chunk's last read starts at 101, so no later read can reach the region
    sites = [(0, 100), (0, 70000)]
    reads = [(0, 95, 99), (0, 100, 150), (0, 101, 180), (0, 69990, 70010)]
    _, bs, be = bins_of(sites)
    rs, re_ = keys(reads[:3])
    done, send, carry = plan_genotype_chunk(rs, re_, bs, be, 0, int(rs[2]))
    assert done == 1
    assert send.tolist() == [1]        # [95, 99) ends at the region start, [101, 180) starts at its end
    assert carry.tolist() == []        # none reaches the second bin
    done, _, _ = plan_genotype_chunk(rs[:2], re_[:2], bs, be, 0, int(rs[1]))
    assert done == 0                   # a read starting at 100 can still be followed by one at 100
    check(reads, sites, cuts=[3])
    check(reads, sites, cuts=[2])


def test_bins_on_contigs_listed_out_of_header_order(tmp_path):
    # the variant file lists chr10 first and chr1 last; the header order is chr1, chr2, chr10
    header = ["chr1", "chr2", "chr10"]
    tsv = tmp_path / "cand.tsv"
    rows = [("chr10", 501), ("chr10", 120001), ("chr2", 7001), ("chr1", 60001), ("chr1", 11)]
    with open(tsv, "w") as f:
        f.write("Chr\tPos\n")
        for c, p in rows:
            f.write("\t".join([c, str(p), ".", "A", "C"] + ["x"] * 9) + "\n")
    bin_info, keys_, site_tid, site_pos, _ = candidate_sites(build_dict_variants(str(tsv), 50000), header)
    assert [b[0] for b in bin_info] == ["chr10", "chr10", "chr2", "chr1", "chr1"]  # file order, for the rows
    assert keys_ == [(0, 10), (0, 60000), (1, 7000), (2, 500), (2, 120000)]
    first, bs, be = genotype_bins(site_tid, site_pos, 50000)
    assert first.tolist() == [0, 1, 2, 3, 4, 5] and np.all(np.diff(be) > 0)
    reads = [(0, 0, 100), (0, 59990, 61000), (1, 6000, 7500), (2, 400, 600), (2, 119000, 121000), (-1, -1, -1)]
    for cuts in ([1], [2, 3], [1, 2, 3, 4, 5], []):
        check(reads, [tuple(k) for k in keys_], cuts)


def test_contig_with_sites_and_no_reads():
    # contig 1 has a site and no read; contig 3 has a site and comes after the last read
    sites = [(0, 1000), (1, 500), (2, 300), (3, 10)]
    reads = [(0, 900, 1100), (0, 1001, 1010), (2, 250, 400), (2, 280, 290)]
    check(reads, sites, cuts=[2])
    _, bs, be = bins_of(sites)
    rs, re_ = keys(reads[:2])
    done, send, _ = plan_genotype_chunk(rs, re_, bs, be, 0, int(rs[1]))
    assert done == 1 and send.tolist() == [0]
    rs, re_ = keys(reads[2:])
    done, send, carry = plan_genotype_chunk(rs, re_, bs, be, 1, int(rs[1]))
    assert done == 2 and send.tolist() == [] and carry.tolist() == [0]  # contig 1 completes without reads
    done, send, carry = plan_genotype_chunk(rs[carry], re_[carry], bs, be, 2, None)  # end of file: contigs 2 and 3
    assert done == 4 and send.tolist() == [0] and carry.tolist() == []


def test_empty_site_list():
    first, bs, be = genotype_bins(np.zeros(0, np.int32), np.zeros(0, np.int32), 50000)
    assert first.tolist() == [0] and bs.shape[0] == 0 and be.shape[0] == 0
    rs, re_ = keys([(0, 5, 50), (0, 7, 9)])
    for last in (int(rs[-1]), None):
        done, send, carry = plan_genotype_chunk(rs, re_, bs, be, 0, last)
        assert done == 0 and send.shape[0] == 0 and carry.shape[0] == 0
    out = pipeline.stream_genotype("/nonexistent.bam", (np.zeros(0), np.zeros(0), np.zeros(0)), 50000, 3, lambda b: 0,
                                   {}, 0.2, 100.0, None, [0])
    assert [a.shape[0] for a in out] == [0] * 5


@pytest.mark.parametrize("seed", range(6))
def test_random_reads_bins_and_cuts(seed):
    rng = np.random.default_rng(seed)
    reads = []
    for t in range(3):
        pos = np.sort(rng.integers(0, 200000, 300))
        reads += [(t, int(p), int(p + rng.choice([0, 50, 900, 30000]))) for p in pos]
    reads += [(-1, -1, -1)] * 3
    sites = sorted({(int(rng.integers(0, 4)), int(rng.integers(0, 210000))) for _ in range(40)})
    cuts = np.sort(rng.choice(np.arange(1, len(reads)), size=int(rng.integers(1, 40)), replace=False)).tolist()
    check(reads, sites, cuts, bin_size=int(rng.choice([1000, 50000])))


# ---- the whole streamed source, the CPU oracle standing in for the engine -------------------------------------------
class OracleEngine:
    """Engine.upload / genotype_sparse with the CPU oracle's counts (p is not evaluated: NaN)."""

    def __init__(self, device):
        self.device, self.last_stats, self.batch = device, {}, None

    def upload(self, batch, windows):
        self.batch = batch

    def genotype_sparse(self, st, sp, alt, n_cells, alpha, beta, skip_p=None, bin_size=50000, **kw):
        import oracle
        dp, al = oracle.genotype_count(self.batch, st, sp, alt, n_cells, bin_size=bin_size, **kw)
        site, cell = np.nonzero(dp > 0)
        return (site.astype(np.int32), cell.astype(np.int32), dp[site, cell], al[site, cell],
                np.full(site.shape[0], np.nan))

    def close(self):
        pass


def test_stream_genotype_matches_one_whole_file_call(tmp_path, monkeypatch):
    import oracle
    d = synth.generate(seed=41, contig_lens=[120000, 16600], chrm=True, n_genes=5, n_reads=4000, n_cells=40,
                       n_hot_genes=1, hot_fraction=0.5)
    b = d.batch
    bam = str(tmp_path / "x.bam")
    bamio.write_bam(bam, d.contig_names, d.contig_lens, b, lambda i: None if b.cell[i] < 0 else synth.barcode_of(int(b.cell[i])) + "-1")
    rng = np.random.default_rng(3)
    pick = rng.choice(b.n_reads, 600, replace=False)
    keys_ = sorted({(int(b.tid[i]), int(b.pos[i]) + int(rng.integers(0, 400))) for i in pick})
    st = np.array([k[0] for k in keys_], np.int32)
    sp = np.array([k[1] for k in keys_], np.int32)
    alt = rng.integers(0, 4, st.shape[0]).astype(np.uint8)
    n_cells = 30  # barcodes of cells 30.. are not in the table
    kw = dict(min_bq=30, min_mq=60, max_depth=60, alt_only=False)
    cells = np.where((b.cell >= 0) & (b.cell < n_cells), b.cell, -1)
    whole = b.select(np.arange(b.n_reads))
    whole.cell = cells.astype(np.int32)
    dp, al = oracle.genotype_count(whole, st, sp, alt, n_cells, bin_size=5000, **kw)
    udp, _ = oracle.genotype_count(whole, st, sp, alt, n_cells, bin_size=5000, **dict(kw, max_depth=0))
    assert udp.sum() > dp.sum()  # the cap fires
    monkeypatch.setattr(pipeline, "take_engine", OracleEngine)
    col = {synth.barcode_of(c): c for c in range(n_cells)}
    stats = []
    site, cell, sdp, sal, _ = pipeline.stream_genotype(bam, (st, sp, alt), 5000, n_cells,
                                                       lambda t: col.get(t.split("-")[0], -1), kw, 0.2, 100.0, None,
                                                       [0, 0, 0], chunk_bytes=200_000, stats_out=stats)
    ri, ci = np.nonzero(dp > 0)
    assert np.array_equal(site, ri) and np.array_equal(cell, ci)
    assert np.array_equal(sdp, dp[ri, ci]) and np.array_equal(sal, al[ri, ci])
    # a chunk that completes the hot gene's bin holds all its reads: half the file
    assert len(stats) >= 8 and max(s["n_reads"] for s in stats) < 0.6 * b.n_reads
    assert max(s["n_carried"] for s in stats) > kw["max_depth"]  # capped bins were cut by chunk boundaries
