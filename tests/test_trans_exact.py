"""The TransCluster likelihood (log p0 and E[K] = sum_k k P(k | N, delta)) against an arbitrary-precision evaluation of the
series (tests/golden/make_trans_exact.py -> trans_exact.json), on the standalone kernel and on every device path that
produces the p0_log / eK / datediff columns.

Every fused path must give bitwise what the standalone trans_dist gives for the same (N, delta): they all run the same
trans_eval, so the standalone kernel is checked against the exact values and the paths against it. Day spans are decades
with negative days, where the reference's stopping rule collapses (SURVEY F7)."""
import importlib.util
import json
import math
import os

import numpy as np
import pytest

import tracs_b200
from tracs_b200 import api

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
FIX = json.load(open(os.path.join(GOLD, "trans_exact.json")))
CASES = FIX["cases"]
Y = 31556952.0
RATES = [(29.903, 73.0), (5.3, 6.0), (0.5, 2.0), (1.0, 100.0)]
TABLE_EAGER_MAX = 16384          # TransLut::EAGER_MAX: the table is computed in full, under the ingest
TABLE_MAX = 1 << 24              # TransLut::setup: larger (distance, day) tables go to the host unique-key path


def _gen():
    spec = importlib.util.spec_from_file_location("make_trans_exact", os.path.join(GOLD, "make_trans_exact.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def _delta(days):
    return (np.asarray(days, dtype=np.float64) * 86400.0) / Y


def _fixture(lamb, beta):
    return {(c["N"], c["days"]): c for c in CASES if (c["lamb"], c["beta"]) == (lamb, beta)}


# ---- the fixture itself (CPU) ----------------------------------------------------------------------------------------

def test_fixture_covers_the_grid():
    g = _gen()
    keys = {(c["N"], c["days"], c["lamb"], c["beta"]) for c in CASES}
    assert keys == {(N, d, la, be) for N in g.N_GRID for d in g.DAYS_GRID for la, be in g.RATES}
    assert max(g.N_GRID) == 2047 and max(g.DAYS_GRID) == 36500 and min(g.DAYS_GRID) == 0
    assert all(math.isfinite(c["log_p0"]) and math.isfinite(c["eK"]) and c["eK"] > 0 for c in CASES)


def test_fixture_delta0_is_the_closed_form():
    """delta = 0: P(k) is the negative binomial with p0 = (lamb / (lamb+beta))^(N+1) and mean (N+1) beta / lamb."""
    z = [c for c in CASES if c["days"] == 0]
    assert len(z) == 12 * 4
    for c in z:
        la, be, N = c["lamb"], c["beta"], c["N"]
        assert c["eK"] == pytest.approx((N + 1) * be / la, rel=1e-15)
        assert c["log_p0"] == pytest.approx((N + 1) * math.log(la / (la + be)), rel=1e-14)


@pytest.mark.parametrize("N,lamb,beta", [(0, 29.903, 73.0), (5, 29.903, 73.0), (2, 5.3, 6.0)])
def test_fixture_delta0_summed(N, lamb, beta):
    """The delta = 0 closed forms against the series itself: sum_k k P(k) of the pmf written out with factorials."""
    mpmath = pytest.importorskip("mpmath")
    with mpmath.workdps(40):
        la, be = mpmath.mpf(lamb), mpmath.mpf(beta)
        P = [la ** (N + 1) * be ** k * mpmath.binomial(N + k, k) / (la + be) ** (N + k + 1) for k in range(400)]
        assert abs(mpmath.fsum(P) - 1) < mpmath.mpf("1e-20")
        eK = mpmath.fsum(k * p for k, p in enumerate(P))
    c = _fixture(lamb, beta)[(N, 0)]
    assert float(eK) == pytest.approx(c["eK"], rel=1e-15)
    assert float(mpmath.log(P[0])) == pytest.approx(c["log_p0"], rel=1e-15)


@pytest.mark.parametrize("key", [(1, 730, 29.903, 73.0), (5, 3650, 5.3, 6.0), (2, 1000, 0.5, 2.0), (0, 90, 29.903, 73.0)])
def test_fixture_eK_summed_directly(key):
    """E[K] of a few keys from P(k | N, delta) written out term by term with factorials, without the generator's stepping:
    every P(k) recomputed from the definition, summed until the terms are past the mode and below 1e-30."""
    mpmath = pytest.importorskip("mpmath")
    N, days, lamb, beta = key
    with mpmath.workdps(40):
        d = mpmath.mpf((days * 86400.0) / Y)
        la, be = mpmath.mpf(lamb), mpmath.mpf(beta)
        pois = mpmath.fsum((la * d) ** i / mpmath.factorial(i) for i in range(N + 1))

        def P(k):
            M = N + k
            integ = mpmath.fsum(d ** (M - i) / mpmath.factorial(M - i) / (la + be) ** (i + 1) for i in range(M + 1))
            return la ** (N + 1) * be ** k * mpmath.factorial(M) / (mpmath.factorial(N) * mpmath.factorial(k)) * mpmath.exp(-d * be) / pois * integ

        total, eK, prev, k = mpmath.mpf(0), mpmath.mpf(0), mpmath.mpf(0), 0
        while True:
            p = P(k)
            total += p
            eK += k * p
            if k > 0 and p < prev and p < mpmath.mpf("1e-30"):
                break
            prev, k = p, k + 1
    c = _fixture(lamb, beta)[(N, days)]
    assert abs(total - 1) < mpmath.mpf("1e-20")
    assert float(eK) == pytest.approx(c["eK"], rel=1e-14)


@pytest.mark.parametrize("key", [(1, 730, 29.903, 73.0), (0, 1000, 29.903, 73.0), (5, 1461, 29.903, 73.0), (20, 90, 5.3, 6.0),
                                 (100, 3650, 0.5, 2.0), (2, 7300, 1.0, 100.0), (0, 36500, 29.903, 73.0), (40, 1, 1.0, 100.0)])
def test_fixture_rederived(key):
    """A few keys evaluated again, at a different precision, so that the committed values are not taken on trust; the
    series must sum to 1 and its k = 0 term must match the sum's own definition at k = 0."""
    mpmath = pytest.importorskip("mpmath")
    g = _gen()
    N, days, la, be = key
    lp0, eK, total = g.exact(N, g.delta_of(days), la, be, dps=60)
    c = _fixture(la, be)[(N, days)]
    assert abs(total - 1) < mpmath.mpf("1e-15")
    assert float(lp0) == pytest.approx(c["log_p0"], rel=1e-14)
    assert float(eK) == pytest.approx(c["eK"], rel=1e-14)
    # log p0 straight from the three factors at k = 0, no stepping
    with mpmath.workdps(60):
        d, L, B = mpmath.mpf(g.delta_of(days)), mpmath.mpf(la), mpmath.mpf(be)
        pois = mpmath.fsum((L * d) ** i / mpmath.factorial(i) for i in range(N + 1))
        integ = mpmath.fsum(d ** (N - i) / mpmath.factorial(N - i) / (L + B) ** (i + 1) for i in range(N + 1))
        direct = (N + 1) * mpmath.log(L) - d * B - mpmath.log(pois) + mpmath.log(integ)
    assert float(direct) == pytest.approx(c["log_p0"], rel=1e-14)


# ---- the standalone kernel against the exact values (GPU) ------------------------------------------------------------

def _check_exact(N, days, lamb, beta, thr, p0, eK):
    fx = _fixture(lamb, beta)
    ex_p0 = np.array([fx[(n, d)]["log_p0"] for n, d in zip(N, days)])
    ex_eK = np.array([fx[(n, d)]["eK"] for n, d in zip(N, days)])
    assert np.allclose(p0, ex_p0, rtol=1e-9, atol=0)
    assert not np.isnan(eK).any()
    # E[K] = +inf: the series had not provably converged by k = 10 000. Only allowed where E[K] is large.
    inf = np.isinf(eK)
    assert (eK[inf] > 0).all() and (ex_eK[inf] > 1000).all(), [(n, d) for n, d, i in zip(N, days, inf) if i and fx[(n, d)]["eK"] <= 1000]
    # the truncated tail is at most thr; the rounding of the sum (up to ~1e-10 relative, test_trans_dist_threshold_zero)
    # has to fit in the same allowance, plus 1e-12 exact
    err = np.abs(eK - ex_eK)
    bad = ~inf & ~(err <= thr + 1e-12 * ex_eK)
    assert not bad.any(), [(int(n), int(d), float(a), float(b)) for n, d, a, b in zip(N[bad], days[bad], eK[bad], ex_eK[bad])][:10]
    return inf


@pytest.mark.gpu
@pytest.mark.parametrize("thr", [0.01, 1e-6, 1.0])
@pytest.mark.parametrize("lamb,beta", RATES)
def test_trans_dist_exact(lamb, beta, thr):
    fx = _fixture(lamb, beta)
    N = np.array([k[0] for k in fx], np.int32)
    days = np.array([k[1] for k in fx], np.int64)
    p0, eK = api.trans_dist_np(N, _delta(days), lamb, beta, thr)
    inf = _check_exact(N, days, lamb, beta, thr, p0, eK)
    if (lamb, beta) != (1.0, 100.0):
        # every exact E[K] of these rates is below 8 200, far enough inside k < 10 000 that no key may stop at the cap
        assert not inf.any()


@pytest.mark.gpu
def test_trans_dist_threshold_zero():
    """thr = 0 asks for E[K] to working precision; a negative or NaN threshold asks for the same. The log of each term is a
    sum of parts as large as lgamma(N + k + 1) <= 1.1e5, each rounded to 2^-52 of its size (1.5e-11), so every term, and
    with it the sum, carries up to ~1e-10 relative error: that, not 1e-12, is the allowance here."""
    N = np.array([c["N"] for c in CASES], np.int32)
    days = np.array([c["days"] for c in CASES], np.int64)
    ex = np.array([c["eK"] for c in CASES])
    for lamb, beta in RATES:
        m = np.array([(c["lamb"], c["beta"]) == (lamb, beta) for c in CASES])
        p0, eK = api.trans_dist_np(N[m], _delta(days[m]), lamb, beta, 0.0)
        for thr in (-1.0, float("nan")):
            p0_t, eK_t = api.trans_dist_np(N[m], _delta(days[m]), lamb, beta, thr)
            assert np.array_equal(p0_t, p0) and np.array_equal(eK_t, eK), thr
        assert not np.isnan(eK).any()
        inf = np.isinf(eK)
        assert (ex[m][inf] > 1000).all()
        if (lamb, beta) != (1.0, 100.0):
            assert not inf.any()
        assert np.allclose(eK[~inf], ex[m][~inf], rtol=1e-10, atol=0)
    # a threshold of 0 once returned the converged series on these keys, and must still
    p0, eK = api.trans_dist_np(np.array([0, 2], np.int32), _delta([1, 30]), 29.903, 73.0, 0.0)
    fx = _fixture(29.903, 73.0)
    assert np.allclose(eK, [fx[(0, 1)]["eK"], fx[(2, 30)]["eK"]], rtol=1e-13, atol=0)


@pytest.mark.gpu
def test_trans_dist_samples_years_apart():
    """The keys where the reference's stopping rule gives E[K] ~ 0 for samples a few years apart (default rates)."""
    keys = [(1, 730, 148.38), (0, 1000, 202.31), (5, 548, 112.26), (5, 1461, 294.55), (20, 1461, 294.93), (0, 2000, 402.18),
            (0, 36500, 7297.6)]
    N = np.array([k[0] for k in keys], np.int32)
    days = np.array([k[1] for k in keys])
    p0, eK = api.trans_dist_np(N, _delta(days), 29.903, 73.0, 0.01)
    assert np.allclose(eK, [k[2] for k in keys], rtol=0, atol=0.02), eK.tolist()
    # lamb = 5.3, beta = 6, ten years; lamb = 1, beta = 100 does not converge by k = 10 000 (E[K] = 20 100)
    p0, eK = api.trans_dist_np(np.array([1], np.int32), _delta([3650]), 5.3, 6.0, 0.01)
    assert abs(eK[0] - 61.11) < 0.02
    p0, eK = api.trans_dist_np(np.array([200], np.int32), _delta([1]), 1.0, 100.0, 0.01)
    assert eK[0] == math.inf


# ---- every other device path: bitwise the standalone kernel (GPU) ----------------------------------------------------

def _days(n, span, seed):
    """n sampling days over [-span/2, span/2] (negative days included), both ends present."""
    d = np.random.default_rng(seed).integers(-(span // 2), span - span // 2, size=n).astype(np.int32)
    d[0], d[-1] = -(span // 2), span - span // 2 - 1
    return d


def _same_as_standalone(res, days, src, lamb=29.903, beta=73.0, thr=0.01):
    """p0_log / eK bitwise trans_dist of (src, |day_i - day_j| in years); datediff = |dday| * 86400 / 31556952."""
    r = np.asarray(res["rows"]).astype(np.int64)
    c = np.asarray(res["cols"]).astype(np.int64)
    assert len(r) > 0
    dd = np.abs(days[r].astype(np.int64) - days[c].astype(np.int64))
    dt = _delta(dd)
    assert np.array_equal(res["datediff"], dt)
    p0, eK = api.trans_dist_np(np.asarray(src).astype(np.int32), dt, lamb, beta, thr)
    assert np.array_equal(res["p0_log"], p0)
    assert np.array_equal(res["eK"], eK)
    return dd


def _alignment(n, L, seed, p_var=0.05, mu=3):
    from tracs_b200 import synth
    return synth.generate(n, L, p_var=p_var, n_clusters=4, mu=mu, p_N=0.01, seed=seed)


@pytest.mark.gpu
def test_fused_eager_table():
    # dist 10 -> d_top = 11 distances; 1 481 day differences: 11 * 1 481 = 16 291 <= 16 384 entries (eager table)
    s = _alignment(300, 3000, 1)
    days = _days(300, 1481, 2)
    res = tracs_b200.pairsnp_matrix(s, dist=10, days=days)
    assert tracs_b200.last_stats()["n_words"] * 32 >= 10
    assert 11 * (int(days.max()) - int(days.min()) + 1) <= TABLE_EAGER_MAX
    dd = _same_as_standalone(res, days, res["dist"])
    assert dd.max() > 1000


@pytest.mark.gpu
def test_fused_marked_table():
    # dist 30 -> 31 distances; 30 years = 10 958 day differences: 31 * 10 958 = 339 698 entries, between 16 384 and 2^24
    s = _alignment(400, 4000, 3)
    days = _days(400, 10958, 4)
    res = tracs_b200.pairsnp_matrix(s, dist=30, days=days)
    assert tracs_b200.last_stats()["n_words"] * 32 >= 30
    assert TABLE_EAGER_MAX < 31 * (int(days.max()) - int(days.min()) + 1) <= TABLE_MAX
    dd = _same_as_standalone(res, days, res["dist"])
    assert dd.max() > 5000
    res = tracs_b200.pairsnp_matrix(s, dist=30, days=days, threshold_Ek=0.0)
    _same_as_standalone(res, days, res["dist"], thr=0.0)


@pytest.mark.gpu
def test_host_unique_key_path():
    # dist 2000 with >= 2 000 variable sites -> 2 001 distances; 30 years = 10 958 day differences:
    # 2 001 * 10 958 = 21.9 M entries > 2^24 = 16.8 M, so the unique (N, delta) keys are evaluated from the host side
    s = _alignment(200, 20000, 5, p_var=0.2, mu=20)
    days = _days(200, 10958, 6)
    res = tracs_b200.pairsnp_matrix(s, dist=2000, days=days)
    assert tracs_b200.last_stats()["n_words"] * 32 >= 2000
    assert 2001 * (int(days.max()) - int(days.min()) + 1) > TABLE_MAX
    _same_as_standalone(res, days, res["dist"])


@pytest.mark.gpu
def test_filtered_distance_feeds_the_likelihood():
    # filter=True: the likelihood takes the filtered distance. dist 200 -> 201 * 10 958 = 2.2 M entries (marked table)
    s = _alignment(60, 30_000, 7, p_var=0.03, mu=5)
    days = _days(60, 10958, 8)
    res = tracs_b200.pairsnp_matrix(s, dist=200, filter=True, days=days)
    assert TABLE_EAGER_MAX < 201 * (int(days.max()) - int(days.min()) + 1) <= TABLE_MAX
    _same_as_standalone(res, days, res["filt"])


@pytest.mark.gpu
def test_query_db_ranges_and_database():
    # days: the queries first, then the database. dist 25 -> 26 * 7 300 = 189 800 entries (marked table)
    s = _alignment(500, 3000, 9)
    nq = 37
    days = _days(500, 7300, 10)
    res = tracs_b200.pairsnp_matrix(s, dist=25, i_end=nq, j_start=nq, days=days)
    assert (res["rows"] < nq).all() and (res["cols"] >= nq).all()
    _same_as_standalone(res, days, res["dist"])
    with tracs_b200.Database(s[nq:]) as db:
        got = db.query(s[:nq], dist=25, days=days)
    for k in ("rows", "cols", "dist", "p0_log", "eK", "datediff"):
        assert np.array_equal(got[k], res[k]), k


def _sites_input(torch):
    """Pairs at distance 0 and 1 (copied rows, one substituted site) in an alignment long enough for the site shard."""
    from tracs_b200 import synth
    s = synth.generate(400, 150_000, p_var=0.06, n_clusters=60, mu=4, p_N=0.002, seed=81)
    s[200:300] = s[0:100]
    s[300:400] = s[100:200]
    for r in range(300, 400):
        c = int(np.nonzero(s[r] == ord("A"))[0][r])
        s[r, c] = ord("C")
    n, L = s.shape
    pitch = (L + 127) // 128 * 128
    buf = torch.full((n, pitch), ord("N"), dtype=torch.uint8, device="cuda")
    buf[:, :L] = torch.from_numpy(s).cuda()
    return s, buf, pitch


@pytest.mark.gpu
def test_site_sharded_world1():
    """sites.sweep at world 1. dist 1 -> 2 distances; 8 192 day differences (22 years): 2 * 8 192 = 16 384 entries, an eager
    table. prepare() gives the days to open(), which computes the table under the ingest; without it the finish step
    builds the table when it emits the edges. The finish step of the prepared run must therefore launch exactly one
    kernel fewer (it found the table built at open and did not build its own)."""
    import torch
    from tracs_b200 import sites

    class Backend(sites.LibBackend):
        def finish(self, *a):
            res, st = super().finish(*a)
            self.finish_stats = st
            return res, st

    s, buf, pitch = _sites_input(torch)
    n, L = s.shape
    days = _days(n, 8192, 11)
    assert 2 * (int(days.max()) - int(days.min()) + 1) == TABLE_EAGER_MAX
    ref = tracs_b200.pairsnp_matrix(s, dist=1, days=days)
    launches = {}
    for prepared in (False, True):
        be = Backend(torch, torch.device("cuda"), buf.data_ptr(), n, L, pitch)
        if prepared:
            be.prepare(days, 29.903, 73.0, 0.01)
        res, st = sites.sweep(torch, None, torch.device("cuda"), 0, 1, buf.data_ptr(), n, L, pitch, L, 1, days=days, backend=be)
        launches[prepared] = be.finish_stats["kernel_launches"]
        assert res["eK"] is not None
        assert (res["dist"] == 0).sum() >= 100 and (res["dist"] == 1).sum() >= 100
        dd = _same_as_standalone(res, days, res["dist"])
        assert dd.max() > 2000
        for k in ("rows", "cols", "dist", "p0_log", "eK", "datediff"):
            assert np.array_equal(np.asarray(res[k]), ref[k]), k
    assert launches[True] == launches[False] - 1, launches


# ---- the distance command line, dates years apart (GPU) --------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("native", [False, True])
def test_distance_cli_years_apart(tmp_path, native):
    """Two runs of the distance stage: default rates, pairs 1 000 days (N = 0) and 730 days (N = 1) apart, where E[K] must
    match the exact value to within the precision; and clock rate 1 / transmission rate 100 with N = 200 one day apart,
    whose series does not converge by k = 10 000 and is written as Python writes float('inf')."""
    from tracs_b200 import distance, synth
    rng = np.random.default_rng(12)
    base = rng.choice(np.frombuffer(b"ACGT", np.uint8), size=600)
    a = base.copy()
    b = base.copy()
    c = base.copy()
    c[5] = ord("A") if c[5] != ord("A") else ord("C")
    msa = str(tmp_path / "years.fasta")
    synth.write_fasta(msa, np.stack([a, b, c]), names=["a", "b", "c"])
    meta = str(tmp_path / "years.csv")
    # a-b: 1 000 days, N = 0; a-c: 730 days (2020 is a leap year), N = 1; b-c: 270 days, N = 1
    open(meta, "w").write("sample,date\na,2020-01-01\nb,2022-09-27\nc,2021-12-31\n")
    out = str(tmp_path / "out.csv")
    distance.distance([msa], out, metadata=meta, precision=0.01, native_csv=native)
    rows = {(r[0], r[1]): r for r in (ln.rstrip("\n").split(",") for ln in open(out).readlines()[1:])}
    fx = _fixture(29.903, 73.0)
    assert rows[("a", "b")][3] == "0" and abs(float(rows[("a", "b")][5]) - fx[(0, 1000)]["eK"]) <= 0.01
    assert rows[("a", "c")][3] == "1" and abs(float(rows[("a", "c")][5]) - fx[(1, 730)]["eK"]) <= 0.01
    assert float(rows[("a", "b")][2]) == 1000 * 86400 / Y
    # the series that does not converge by the cap
    d = base.copy()
    d[:200] = np.where(d[:200] == ord("A"), ord("C"), ord("A"))
    msa2 = str(tmp_path / "cap.fasta")
    synth.write_fasta(msa2, np.stack([a, d]), names=["a", "b"])
    meta2 = str(tmp_path / "cap.csv")
    open(meta2, "w").write("sample,date\na,2020-01-01\nb,2020-01-02\n")
    out2 = str(tmp_path / "cap_out.csv")
    distance.distance([msa2], out2, metadata=meta2, clock_rate=1.0, trans_rate=100.0, precision=0.01, native_csv=native)
    r = open(out2).readlines()[1].rstrip("\n").split(",")
    assert r[3] == "200" and r[5] == str(math.inf) == "inf"
