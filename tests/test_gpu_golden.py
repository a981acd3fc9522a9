"""GPU: the CUDA path through the drop-in `TRACS` module and the distance driver against the golden
fixtures generated from the unmodified reference (tests/golden/make_golden.py)."""
import json
import os

import numpy as np
import pytest

import tracs_b200

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
G = json.load(open(os.path.join(GOLD, "golden.json")))


@pytest.mark.parametrize("case", G["pairsnp"], ids=lambda c: c["fasta"])
def test_golden_pairsnp(case):
    T = tracs_b200.install_dropin()
    r = T.pairsnp(fasta=[os.path.join(GOLD, case["fasta"])], n_threads=1, dist=case["dist"], filter=False)
    assert isinstance(r, tuple) and len(r) == 6 and all(isinstance(x, list) for x in r)
    assert r[0] == case["rows"] and r[1] == case["cols"] and r[2] == case["d"]
    assert r[3] == case["names"] and r[4] == case["filt"] and r[5] == case["ncomp"]


def test_golden_two_file():
    T = tracs_b200.install_dropin()
    case = G["two_file"][0]
    r = T.pairsnp(fasta=[os.path.join(GOLD, f) for f in case["fasta"]], n_threads=2, dist=case["dist"], filter=False)
    assert r[0] == case["rows"] and r[1] == case["cols"] and r[2] == case["d"] and r[3] == case["names"] and r[5] == case["ncomp"]


@pytest.mark.parametrize("k", range(len(G["trans_dist"]["cases"])))
def test_golden_trans_dist(k):
    T = tracs_b200.install_dropin()
    c = G["trans_dist"]["cases"][k]
    days = np.array(c["days"])
    dt = days * 86400.0 / 31556952.0
    p0, eK = T.trans_dist(np.array(c["N"]), dt, c["lamb"], c["beta"], c["thr"])
    assert isinstance(p0, list) and isinstance(eK, list)
    assert np.allclose(p0, c["p0_log"], rtol=1e-6, atol=0)
    ref_eK = np.array(c["eK"])
    pos = (days > 0) & np.isfinite(ref_eK)          # delta == 0 is UB in the reference (SURVEY F6)
    assert np.allclose(np.array(eK)[pos], ref_eK[pos], rtol=1e-6, atol=0)
    z = days == 0
    assert np.allclose(np.array(eK)[z], (np.array(c["N"])[z] + 1) * c["beta"] / c["lamb"], rtol=1e-12)


def _rows(path):
    return [ln.rstrip("\n").split(",") for ln in open(path)]


@pytest.mark.parametrize("tag,extra", [("meta", dict(metadata=os.path.join(GOLD, "cli_dates.csv"), trans_threshold=100.0)), ("nometa", {})])
def test_distance_cli_csv(tmp_path, tag, extra):
    from tracs_b200 import distance
    out = str(tmp_path / "d.csv")
    distance.distance([os.path.join(GOLD, "cli_combined.fasta.gz")], out, snp_threshold=40, n_cpu=2, **extra)
    got, exp = _rows(out), _rows(os.path.join(GOLD, "cli_%s.csv" % tag))
    assert got[0] == exp[0] and len(got) == len(exp)
    for g, e in zip(got[1:], exp[1:]):
        assert g[0] == e[0] and g[1] == e[1] and g[3] == e[3] and g[6] == e[6] and g[7] == e[7] and g[8] == e[8]
        if tag == "meta":
            assert g[2] == e[2]
            assert abs(float(g[4]) - float(e[4])) <= 1e-6 * abs(float(e[4]))
            if float(e[2]) > 0:
                assert abs(float(g[5]) - float(e[5])) <= 1e-6 * abs(float(e[5]))
        else:
            assert g[2] == "NA" and g[4] == "NA" and g[5] == "NA"


def test_reference_kat_csv(tmp_path):
    # the reference's tests/test_trans_distance.py values, through the whole driver
    from tracs_b200 import distance
    out = str(tmp_path / "kat.csv")
    distance.distance([os.path.join(GOLD, "kat.fasta")], out, metadata=os.path.join(GOLD, "kat_dates.csv"), trans_threshold=10.0,
                      snp_threshold=5)
    rows = _rows(out)
    l1, l2 = rows[1], rows[2]
    assert abs(float(l1[2]) - 0.002737907006988508) < 1e-6 and abs(float(l2[2]) - 0.002737907006988508) < 1e-6
    assert int(l1[3]) == 0 and int(l2[3]) == 2
    assert abs(float(l1[4]) - 0.23794988406662973) < 1e-6 and abs(float(l2[4]) - 0.024467137572328577) < 1e-6
    assert abs(float(l1[5]) - 2.6335200453700187) < 1e-6 and abs(float(l2[5]) - 7.315670110063259) < 1e-6
    assert rows[3][:4] == ["seq2", "seq3", "0.0", "1"] and rows[3][6:] == ["NA", "9", "kat"]


def test_reference_test_assertions_on_reconstructed_fixture(tmp_path):
    """The known answers of the reference's tests/test_llk.py, tests/test_pairsnp.py::test_pairsnp and
    tests/test_trans_distance.py (the last two on their fixtures ambig.aln / dates_ambig.csv, reconstructed in
    golden/ref_fixture/), through the drop-in module and the driver."""
    from scipy.special import gammaln
    from tracs_b200 import distance
    fx = os.path.join(GOLD, "ref_fixture")
    T = tracs_b200.install_dropin()
    lp, lhs = T.lprob_k_given_N(N=7, k=4, delta=0.16963, lamb=3, beta=52, lgamma=gammaln(range(20)))
    assert abs(lp + 17.9565184209608) < 1e-6 and abs(lhs - 12.0861694243766) < 1e-6
    r = T.pairsnp(fasta=[os.path.join(fx, "ambig.aln")], n_threads=1, dist=10, filter=False)
    assert all(isinstance(x, list) for x in r)
    assert r[0] == [0, 0, 0, 0, 1, 1, 1, 2, 2, 3] and r[1] == [1, 2, 3, 4, 2, 3, 4, 3, 4, 4] and r[2] == [0, 2, 1, 1, 2, 2, 2, 3, 3, 0]
    out = str(tmp_path / "ambig.csv")
    distance.distance([os.path.join(fx, "ambig.aln")], out, metadata=os.path.join(fx, "dates_ambig.csv"), trans_threshold=10.0,
                      snp_threshold=5)
    l1, l2 = _rows(out)[1:3]
    assert l1[:2] == ["seq1", "seq2"] and l2[:2] == ["seq1", "seq3"]
    assert abs(float(l1[2]) - 0.002737907006988508) < 1e-6 and int(l1[3]) == 0 and int(l2[3]) == 2
    assert abs(float(l1[4]) - 0.23794988406662973) < 1e-6 and abs(float(l2[4]) - 0.024467137572328577) < 1e-6
    assert abs(float(l1[5]) - 2.6335200453700187) < 1e-6 and abs(float(l2[5]) - 7.315670110063259) < 1e-6


def test_distance_cli_with_filter(tmp_path, ):
    # --filter: filtered column carries numbers, likelihood uses them; compare with the CPU oracle pipeline
    from oracle import oracle
    from tracs_b200 import distance
    out = str(tmp_path / "f.csv")
    msa = os.path.join(GOLD, "cli_combined.fasta.gz")
    distance.distance([msa], out, snp_threshold=40, recomb_filter=True, metadata=os.path.join(GOLD, "cli_dates.csv"), trans_threshold=1e9)
    rows = _rows(out)[1:]
    exp = oracle.pairsnp([msa], dist=40, filter=True)
    assert [int(r[6]) for r in rows] == exp[4] and [int(r[3]) for r in rows] == exp[2]


def test_config4_min_over_references(tmp_path):
    """BASELINE.json configs[3] in miniature: several reference MSAs over overlapping sample subsets with
    IUPAC codes and many N's; per-MSA sweeps, then min over references per unordered name pair.
    Checked against the CPU oracle + a plain dict group-by-min, and clustering invariance
    (connected components of `any row <= thr` == components of `min <= thr`, tracs/cluster.py:104-129)."""
    from oracle import oracle
    from scipy.sparse import csr_matrix
    from scipy.sparse.csgraph import connected_components
    from tracs_b200 import distance, synth
    rng = np.random.default_rng(7)
    all_names = ["smp%03d" % i for i in range(120)]
    per_msa, expect, any_rows = [], {}, []
    for r in range(4):
        members = np.sort(rng.choice(120, size=int(rng.integers(70, 120)), replace=False))
        L = int(rng.integers(20_000, 30_000))
        s = synth.generate(len(members), L, p_var=0.02, n_clusters=6, mu=4, p_N=0.3, p_amb=0.05, seed=40 + r, three_base=True)
        names = [all_names[m] for m in members]
        p = str(tmp_path / ("ref%d_combined.fasta.gz" % r))
        synth.write_fasta(p, s, names=names)
        got = tracs_b200.pairsnp(fasta=[p], n_threads=1, dist=100, filter=False)
        exp = oracle.pairsnp([p], dist=100)
        assert got[0] == exp[0] and got[1] == exp[1] and got[2] == exp[2] and got[5] == exp[5] and got[3] == names
        per_msa.append((got[3], got[0], got[1], got[2]))
        for i, j, d in zip(exp[0], exp[1], exp[2]):
            a, b = names[i], names[j]
            key = (a, b) if all_names.index(a) < all_names.index(b) else (b, a)
            expect[key] = min(expect.get(key, 1e300), d)
            any_rows.append((key, d))
    A, B, V = distance.min_over_references(per_msa)
    got_map = {}
    for a, b, v in zip(A, B, V):
        key = (a, b) if all_names.index(a) < all_names.index(b) else (b, a)
        assert key not in got_map
        got_map[key] = v
    assert got_map == {k: float(v) for k, v in expect.items()}
    # clustering is invariant under the combine
    idx = {nm: k for k, nm in enumerate(all_names)}
    for thr in (5, 20):
        def comps(pairs):
            if not pairs:
                return np.arange(120)
            r_ = [idx[a] for a, _ in pairs]
            c_ = [idx[b] for _, b in pairs]
            g = csr_matrix((np.ones(len(r_)), (r_, c_)), shape=(120, 120))
            return connected_components(g, directed=False)[1]
        c_any = comps([k for k, d in any_rows if d <= thr])
        c_min = comps([k for k, v in got_map.items() if v <= thr])
        assert np.array_equal(c_any, c_min)


def test_connected_components_match_scipy():
    from scipy.sparse import csr_matrix
    from scipy.sparse.csgraph import connected_components
    rng = np.random.default_rng(11)
    for n, m in ((1, 0), (10, 0), (50, 30), (2000, 1500), (20000, 30000), (5000, 200000)):
        a = rng.integers(0, n, m).astype(np.uint64)
        b = rng.integers(0, n, m).astype(np.uint64)
        nc, lab = tracs_b200.connected_components(a, b, n)
        g = csr_matrix((np.ones(m), (a.astype(np.int64), b.astype(np.int64))), shape=(n, n))
        enc, elab = connected_components(g, directed=False)
        assert nc == enc and lab.tolist() == elab.tolist()
    with pytest.raises(IndexError):
        tracs_b200.connected_components(np.array([5], np.uint64), np.array([1], np.uint64), 3)


@pytest.mark.parametrize("tag,thr,dist", [("snp10", 10, "snp"), ("ek5", 5, "expectedK"), ("direct", 0.05, "direct")])
def test_cluster_stage_matches_reference(tmp_path, tag, thr, dist):
    # distances by our driver on the GPU, clusters by our cluster stage; golden = reference tracs/cluster.py on the reference CSV
    from tracs_b200 import cluster, distance
    dcsv, ccsv = str(tmp_path / "d.csv"), str(tmp_path / "c.csv")
    distance.distance([os.path.join(GOLD, "cli_combined.fasta.gz")], dcsv, snp_threshold=40, n_cpu=1,
                      metadata=os.path.join(GOLD, "cli_dates.csv"), trans_threshold=100.0)
    cluster.cluster(dcsv, ccsv, thr, dist)
    assert open(ccsv).read() == open(os.path.join(GOLD, "cluster_%s.csv" % tag)).read()


@pytest.mark.parametrize("tag,extra", [("meta", dict(metadata=os.path.join(GOLD, "cli_dates.csv"), trans_threshold=100.0)), ("nometa", {})])
def test_distance_cli_native_csv(tmp_path, tag, extra):
    # the C writer produces the same file as the Python loop of the mirror (and hence as the reference, see above)
    from tracs_b200 import distance
    a, b = str(tmp_path / "py.csv"), str(tmp_path / "native.csv")
    distance.distance([os.path.join(GOLD, "cli_combined.fasta.gz")], a, snp_threshold=40, **extra)
    distance.distance([os.path.join(GOLD, "cli_combined.fasta.gz")], b, snp_threshold=40, native_csv=True, **extra)
    ra, rb = _rows(a), _rows(b)
    assert len(ra) == len(rb) and ra[0] == rb[0]
    for x, y in zip(ra[1:], rb[1:]):
        assert x[:4] == y[:4] and x[5:] == y[5:]
        if x[4] != "NA":   # exp() of numpy vs libm may differ in the last printed digit
            assert abs(float(x[4]) - float(y[4])) <= 1e-15 * abs(float(x[4]))
