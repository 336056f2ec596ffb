"""K1' (genotype pileup), K2 (beta-binomial tails) and K3 (site masks) vs their oracles."""
import numpy as np
import pytest

from longsom_b200 import synth
from longsom_b200._lib import CLASS_ID, LS_CLASS_NA
from longsom_b200.batch import Windows, make_windows
from longsom_b200.engine import CountParams

pytestmark = pytest.mark.gpu

# alpha/beta shipped by the reference (config/config.yaml:52-55,87-90; step1.py:600-603)
AB = [(0.260288007167716, 173.94711910763732), (0.08354121346569514, 103.47683488327257),
      (0.21356058558983, 104.95768503076), (0.20314940430280, 162.03800230194)]


def _sites_from_counts(sc, n):
    rng = np.random.default_rng(7)
    idx = np.sort(rng.choice(sc.n_sites, size=min(n, sc.n_sites), replace=False))
    alt = rng.integers(0, 9, size=idx.shape[0]).astype(np.uint8)  # includes O (7) and NA (8)
    return sc.tid[idx], sc.pos[idx], alt


@pytest.mark.parametrize("alt_only", [False, True])
@pytest.mark.parametrize("min_bq,min_mq", [(30, 60), (0, 0)])
def test_genotype_parity(engine, alt_only, min_bq, min_mq):
    import oracle
    d = synth.generate(seed=21, contig_lens=[250000, 120000, 16600], chrm=True, n_genes=25, n_reads=25000, n_cells=300)
    w = Windows.from_intervals(make_windows(d.contig_lens, 50000), d.contig_seqs())
    sc = engine.pileup_count(d.batch, w, CountParams(min_mq=60))
    st, sp, alt = _sites_from_counts(sc, 3000)
    dp, al = engine.genotype_count(st, sp, alt, d.n_cells, min_bq=min_bq, min_mq=min_mq, alt_only=alt_only)
    odp, oal = oracle.genotype_count(d.batch, st, sp, alt, d.n_cells, min_bq=min_bq, min_mq=min_mq, alt_only=alt_only)
    assert np.array_equal(dp, odp)
    assert np.array_equal(al, oal)
    assert dp.sum() > 0 and (alt_only or al.sum() > 0)


def test_genotype_depth_cap(engine):
    import oracle
    d = synth.generate(seed=22, contig_lens=[120000], n_genes=4, n_reads=15000, n_cells=100, n_hot_genes=1,
                       hot_fraction=0.8)
    w = Windows.from_intervals(make_windows(d.contig_lens, 50000), d.contig_seqs())
    sc = engine.pileup_count(d.batch, w, CountParams(min_mq=60))
    st, sp, alt = _sites_from_counts(sc, 500)
    for cap in (100, 2000):
        dp, al = engine.genotype_count(st, sp, alt, d.n_cells, min_bq=30, min_mq=60, max_depth=cap)
        odp, oal = oracle.genotype_count(d.batch, st, sp, alt, d.n_cells, min_bq=30, min_mq=60, max_depth=cap)
        assert np.array_equal(dp, odp) and np.array_equal(al, oal)


def _bb_grid():
    rng = np.random.default_rng(3)
    n = np.concatenate([np.arange(0, 40), rng.integers(1, 300, 4000), rng.integers(300, 20000, 600),
                        rng.integers(20000, 200001, 40), [200000, 170, 171, 172]]).astype(np.int32)
    k = np.minimum((rng.random(n.shape[0]) ** 3 * np.minimum(n, 2500)).astype(np.int32) +
                   rng.integers(0, 3, n.shape[0]).astype(np.int32), n + 1).astype(np.int32)
    k[:8] = [0, 1, 2, 0, 5, 7, 1, 1]  # includes k > n and k == 0
    return k, n


@pytest.mark.parametrize("ab", AB)
def test_betabinom_sf_vs_scipy(engine, ab):
    from scipy.stats import betabinom
    a, b = ab
    k, n = _bb_grid()
    p = engine.betabinom_sf(k, n, a, b)
    for eps in (0.1, 0.001):
        ref = betabinom.sf(k - eps, n, a, b)
        # tolerance of SURVEY.md 8(c): |dp| <= 1e-9*p + 1e-12 for every query, n > 1e4 included (scipy itself
        # carries 1e-13..1e-16 absolute cancellation noise in 1-cdf)
        dev = np.abs(p - ref)
        bad = np.nonzero(dev > 1e-9 * ref + 1e-12)[0]
        assert bad.size == 0, [(int(k[i]), int(n[i]), float(dev[i])) for i in bad[:10]]
        assert np.array_equal(np.round(p, 4), np.round(ref, 4))


def test_betabinom_one_minus_cdf(engine):
    """step1's noise test uses 1 - cdf(x - 0.1, n, a, b) (step1.py:329-330) == sf for valid n."""
    from scipy.stats import betabinom
    a, b = AB[0]
    k = np.array([1, 3, 10, 50, 2], np.int32)
    n = np.array([30, 200, 1000, 5000, 2], np.int32)
    p = engine.betabinom_sf(k, n, a, b)
    ref = 1 - betabinom.cdf(k - 0.1, n, a, b)
    assert np.allclose(p, ref, rtol=1e-9, atol=1e-12)


def test_site_mask(engine):
    rng = np.random.default_rng(5)
    keys = (rng.integers(0, 25, 200000).astype(np.uint64) << np.uint64(32)) | rng.integers(0, 3_000_000, 200000).astype(np.uint64)
    q = np.concatenate([keys[rng.integers(0, keys.shape[0], 5000)],
                        (rng.integers(0, 25, 5000).astype(np.uint64) << np.uint64(32)) | rng.integers(0, 3_000_000, 5000).astype(np.uint64)])
    hit = engine.site_mask(keys, q)
    want = np.isin(q, keys).astype(np.uint8)
    assert np.array_equal(hit, want)
    assert hit[:5000].all()
    assert engine.site_mask(np.zeros(0, np.uint64), q).sum() == 0


def test_site_tables_stay_resident(engine):
    """K3 in two steps (step2 keeps its three site lists for the whole run, BaseCellCalling.step2.py:197-221): tables
    sorted once into resident slots, several lookups against each, slots independent, reload replaces, an empty slot
    is a state error."""
    rng = np.random.default_rng(6)

    def table(n, seed):
        r = np.random.default_rng(seed)
        return (r.integers(0, 90, n).astype(np.uint64) << np.uint64(32)) | r.integers(0, 250_000_000, n).astype(np.uint64)
    t0, t1 = table(1_000_000, 1), table(30_000, 2)
    engine.site_table_load(0, t0)
    engine.site_table_load(1, t1)
    for rep in range(3):
        q = np.concatenate([t0[rng.integers(0, t0.shape[0], 20000)], t1[rng.integers(0, t1.shape[0], 20000)], table(20000, 10 + rep)])
        assert np.array_equal(engine.site_table_lookup(0, q), np.isin(q, t0).astype(np.uint8))
        assert np.array_equal(engine.site_table_lookup(1, q), np.isin(q, t1).astype(np.uint8))
        # the one-shot call uses its own scratch slot: the resident tables survive it
        assert np.array_equal(engine.site_mask(t1, q), np.isin(q, t1).astype(np.uint8))
    engine.site_table_load(0, t1)
    q = np.concatenate([t0[:1000], t1[:1000]])
    assert np.array_equal(engine.site_table_lookup(0, q), np.isin(q, t1).astype(np.uint8))
    engine.site_table_load(2, np.zeros(0, np.uint64))
    assert engine.site_table_lookup(2, q).sum() == 0
    with pytest.raises(RuntimeError):
        engine.site_table_lookup(3, q)
