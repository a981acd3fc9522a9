"""CPU: pins the oracle (oracle/tracs_oracle.c) against the reference's known-answer tests, the
committed golden fixtures (generated from the unmodified reference by tests/golden/make_golden.py)
and -- when oracle/_ref is present -- the reference module itself, live."""
import json
import os

import numpy as np
import pytest
from scipy.special import gammaln

from tracs_b200 import synth

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
G = json.load(open(os.path.join(GOLD, "golden.json")))
IMAX = 2147483647


def test_kat_lprob_k_given_N(oracle_mod):
    # reference tests/test_llk.py:21-29 (value derived from a Sage integral)
    lp, lhs = oracle_mod.lprob_k_given_N(7, 4, 0.16963, 3, 52, gammaln(range(20)))
    assert abs(lp + 17.9565184209608) < 1e-6
    assert abs(lhs - 12.0861694243766) < 1e-6


def test_kat_trans_distance(oracle_mod):
    # reference tests/test_trans_distance.py:29-42: delta = exactly one day, CLI default rates
    d = 86400 / 31556952.0
    assert abs(d - 0.002737907006988508) < 1e-15
    p0, eK = oracle_mod.trans_dist([0, 2], [d, d], 29.903, 73.0, 0.01)
    assert abs(np.exp(p0[0]) - 0.23794988406662973) < 1e-6
    assert abs(np.exp(p0[1]) - 0.024467137572328577) < 1e-6
    assert abs(eK[0] - 2.6335200453700187) < 1e-6
    assert abs(eK[1] - 7.315670110063259) < 1e-6


def test_kat_pairsnp_ordering(oracle_mod, tmp_path):
    # reference tests/test_pairsnp.py:7-8 pins (row, col) ordering and list types for 5 sequences
    s = synth.generate(5, 50, p_var=0.2, n_clusters=2, mu=1, p_N=0.0, seed=1, gaps=0)
    p = str(tmp_path / "five.aln")
    synth.write_fasta(p, s)
    r = oracle_mod.pairsnp([p], dist=IMAX)
    assert r[0] == [0, 0, 0, 0, 1, 1, 1, 2, 2, 3]
    assert r[1] == [1, 2, 3, 4, 2, 3, 4, 3, 4, 4]
    assert isinstance(r[2], list) and r[4] == [0] * 10


@pytest.mark.parametrize("case", G["pairsnp"], ids=lambda c: c["fasta"])
def test_golden_pairsnp(oracle_mod, case):
    r = oracle_mod.pairsnp([os.path.join(GOLD, case["fasta"])], n_threads=2, dist=case["dist"])
    assert r[0] == case["rows"] and r[1] == case["cols"] and r[2] == case["d"]
    assert r[3] == case["names"] and r[4] == case["filt"] and r[5] == case["ncomp"]


def test_golden_two_file(oracle_mod):
    case = G["two_file"][0]
    r = oracle_mod.pairsnp([os.path.join(GOLD, f) for f in case["fasta"]], dist=case["dist"])
    assert r[0] == case["rows"] and r[1] == case["cols"] and r[2] == case["d"] and r[3] == case["names"] and r[5] == case["ncomp"]


@pytest.mark.parametrize("case", G["filter"], ids=lambda c: c["fasta"])
def test_golden_filter(oracle_mod, case):
    r = oracle_mod.pairsnp([os.path.join(GOLD, case["fasta"])], dist=case["dist"], filter=True)
    assert r[0] == case["rows"] and r[2] == case["d"] and r[4] == case["filt"]


@pytest.mark.parametrize("k", range(len(G["trans_dist"]["cases"])))
def test_golden_trans_dist(oracle_mod, k):
    c = G["trans_dist"]["cases"][k]
    dt = np.array(c["days"]) * 86400.0 / 31556952.0
    p0, eK = oracle_mod.trans_dist(c["N"], dt, c["lamb"], c["beta"], c["thr"])
    assert np.allclose(p0, c["p0_log"], rtol=1e-9, atol=0)
    assert np.allclose(eK, c["eK"], rtol=1e-9, atol=0)


def test_golden_lprob(oracle_mod):
    for c in G["lprob_k_given_N"]:
        N, k, delta, lamb, beta = c["args"]
        out = oracle_mod.lprob_k_given_N(int(N), int(k), delta, lamb, beta, gammaln(range(40)))
        assert np.allclose(out, c["out"], rtol=1e-12)


def test_numpy_cross_check(oracle_mod):
    for seed in range(6):
        s = synth.generate(11 + seed, 97 + 13 * seed, p_var=0.3, n_clusters=3, mu=2, p_N=0.05, p_amb=0.2, seed=seed, three_base=True,
                           lowercase=0.1, odd_chars=0.03)
        for dist in (0, 5, IMAX):
            a = oracle_mod.pairsnp_ascii(s, dist=dist, n_threads=2)
            b = oracle_mod.pairsnp_numpy(s, dist=dist)
            assert a[0].tolist() == b[0].tolist() and a[1].tolist() == b[1].tolist()
            assert a[2].tolist() == b[2].tolist() and a[4].tolist() == b[3].tolist()
        a = oracle_mod.pairsnp_ascii(s, i_end=4, j_start=4, dist=IMAX)
        b = oracle_mod.pairsnp_numpy(s, i_end=4, j_start=4, dist=IMAX)
        assert a[1].tolist() == b[1].tolist() and a[2].tolist() == b[2].tolist()


def test_site_drop_rule_preserves_distances(oracle_mod):
    # SURVEY A.4: a site whose masks share a base across ALL samples contributes to no pair
    s = synth.generate(20, 600, p_var=0.1, n_clusters=3, mu=2, p_N=0.05, p_amb=0.1, seed=4)
    m = oracle_mod.masks_of(s)
    keep = np.bitwise_and.reduce(m, axis=0) == 0
    a = oracle_mod.pairsnp_ascii(s, dist=IMAX)
    b = oracle_mod.pairsnp_ascii(s[:, keep], dist=IMAX)
    assert 0 < keep.sum() < s.shape[1]
    assert a[2].tolist() == b[2].tolist()


def _golden_alignment(name):
    """Names and ASCII rows of a golden alignment (one header line per record, as synth.write_fasta writes it)."""
    import gzip
    names, rows = [], []
    for ln in (gzip.open if name.endswith(".gz") else open)(os.path.join(GOLD, name), "rb"):
        ln = ln.rstrip(b"\r\n")
        if ln.startswith(b">"):
            names.append(ln[1:].split()[0].decode())
            rows.append([])
        else:
            rows[-1].append(ln)
    return names, np.array([np.frombuffer(b"".join(r), np.uint8) for r in rows])


def _local_reference():
    """The unmodified reference module when a local build of it exists in oracle/_ref/ (not part of the repository), else None."""
    from oracle import refmod
    return refmod.load()[0] if refmod.available() else None


def test_live_reference(oracle_mod, tmp_path):
    """The oracle against the reference. Always: against the reference's outputs stored in golden.json (pairsnp at the
    stored thresholds and with filter=True; the trans_dist grid, delta == 0 included, is compared in test_golden_trans_dist),
    with every stored alignment re-written in each format the live comparison draws -- plain or gz, with or without header
    descriptions, line width 0 / 60 / 7 -- and read with 1 to 3 threads. With a local build of the reference: also live, on
    seeded random alignments."""
    for filt, cases in ((False, G["pairsnp"]), (True, G["filter"])):
        for case in cases:
            names, s = _golden_alignment(case["fasta"])
            exp = [case.get(k) for k in ("rows", "cols", "d", "names", "filt", "ncomp")]
            for k in range(6):
                p = str(tmp_path / ("k%d.fa%s" % (k, ".gz" if k % 2 else "")))
                synth.write_fasta(p, s, names=names, width=[0, 60, 7][k % 3], descriptions=bool(k % 2))
                r = oracle_mod.pairsnp([p], n_threads=1 + k % 3, dist=case["dist"], filter=filt)
                assert all(e is None or r[t] == e for t, e in enumerate(exp)), (case["fasta"], k)
    ref_mod = _local_reference()
    if ref_mod is None:
        return
    for trial in range(8):
        rng = np.random.default_rng(100 + trial)
        n, L = int(rng.integers(2, 30)), int(rng.integers(1, 700))
        s = synth.generate(n, L, p_var=0.2, n_clusters=3, mu=2, p_N=0.05, p_amb=0.1, seed=trial, lowercase=0.1, odd_chars=0.02,
                           three_base=True)
        p = str(tmp_path / ("t%d.fa%s" % (trial, ".gz" if trial % 2 else "")))
        synth.write_fasta(p, s, width=[0, 60, 7][trial % 3], descriptions=bool(trial % 2))
        for dist, filt in ((3, False), (IMAX, False), (IMAX, True)):
            # filter=True is only safe single-threaded in the reference: cached_binomial_cdf (src/pairsnp.hpp:40-58) keeps a
            # function-static std::map that the OpenMP pair loop (:380-432) inserts into without a lock -- with more
            # threads the run corrupts the heap now and then (seen here as a crash at interpreter exit)
            a = ref_mod.pairsnp(fasta=[p], n_threads=1 if filt else 1 + trial % 3, dist=dist, filter=filt)
            b = oracle_mod.pairsnp([p], n_threads=2, dist=dist, filter=filt)
            assert all(list(a[t]) == b[t] for t in range(6))
    N = np.repeat(np.arange(0, 30), 10)
    dt = np.tile(np.arange(0, 10) * 17, 30) * 86400.0 / 31556952.0
    a = ref_mod.trans_dist(N.tolist(), dt.tolist(), 29.903, 73.0, 0.01)
    b = oracle_mod.trans_dist(N, dt, 29.903, 73.0, 0.01)
    assert np.allclose(a[0], b[0], rtol=1e-9)
    # delta == 0: the reference reads past its 10000-entry lgamma table (UB: (N+1)*beta/lamb for small N,
    # inf for larger N in this build; SURVEY F6). The oracle defines it as the converged series.
    pos = dt > 0
    assert np.allclose(np.array(a[1])[pos], b[1][pos], rtol=1e-9)
    z = (~pos) & np.isfinite(np.array(a[1]))
    assert z.sum() > 0 and np.allclose(np.array(a[1])[z], b[1][z], rtol=1e-6)
    assert np.allclose(b[1][~pos], (N[~pos] + 1) * 73.0 / 29.903, rtol=1e-9)


def test_reconstructed_reference_fixture(oracle_mod):
    """tests/golden/ref_fixture/ambig.aln stands in for the absent fixture of the reference's tests/test_pairsnp.py:5-9: it
    gives exactly the vectors that test asserts, on the oracle (held to the reference's stored outputs above) and, with a local
    build of the reference, on the UNMODIFIED reference module itself."""
    p = os.path.join(GOLD, "ref_fixture", "ambig.aln")
    mods = [lambda: oracle_mod.pairsnp([p], n_threads=1, dist=10)]
    ref_mod = _local_reference()
    if ref_mod is not None:
        mods.append(lambda: ref_mod.pairsnp(fasta=[p], n_threads=1, dist=10, filter=False))
    for run in mods:
        r = run()
        assert list(r[0]) == [0, 0, 0, 0, 1, 1, 1, 2, 2, 3]
        assert list(r[1]) == [1, 2, 3, 4, 2, 3, 4, 3, 4, 4]
        assert list(r[2]) == [0, 2, 1, 1, 2, 2, 2, 3, 3, 0]
