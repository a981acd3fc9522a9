"""GPU parity: the CUDA path through the C ABI vs the CPU oracle, bit-exact for edges."""
import os

import numpy as np
import pytest

import tracs_b200
from tracs_b200 import synth

pytestmark = pytest.mark.gpu
IMAX = 2147483647


def _cmp(res, orc):
    r, c, d, f, nn = orc
    assert res["rows"].tolist() == r.tolist()
    assert res["cols"].tolist() == c.tolist()
    assert res["dist"].tolist() == d.tolist()
    assert res["ncomp"].tolist() == nn.tolist()


@pytest.mark.parametrize("n,L,dist", [(2, 1, IMAX), (5, 31, IMAX), (7, 32, 3), (33, 33, IMAX), (128, 1000, 40), (129, 4097, 25),
                                      (300, 20000, 30), (257, 1023, 0), (64, 5000, IMAX), (3, 70000, IMAX)])
def test_matrix_parity(oracle_mod, n, L, dist):
    s = synth.generate(n, L, p_var=0.05, n_clusters=4, mu=3, p_N=0.02, p_amb=0.05, seed=n * 7 + L, lowercase=0.05,
                       odd_chars=0.01, three_base=True)
    res = tracs_b200.pairsnp_matrix(s, dist=dist)
    _cmp(res, oracle_mod.pairsnp_ascii(s, dist=dist, n_threads=4))


def test_every_byte_value(oracle_mod):
    """k_pack decodes the plain alphabet arithmetically and repairs every other byte from the exact table:
    all 256 byte values (single-bit neighbours of A/C/G/T/N/- included) must give the reference's masks."""
    rng = np.random.default_rng(5)
    s = synth.generate(40, 4096, p_var=0.05, n_clusters=3, mu=3, p_N=0.01, seed=77)
    for c in range(4096):
        s[(c // 256 + c) % 40, c] = c % 256
    _cmp(tracs_b200.pairsnp_matrix(s, dist=IMAX), oracle_mod.pairsnp_ascii(s, dist=IMAX, n_threads=4))
    r = rng.integers(0, 256, size=(20, 3001), dtype=np.uint8)
    _cmp(tracs_b200.pairsnp_matrix(r, dist=IMAX), oracle_mod.pairsnp_ascii(r, dist=IMAX, n_threads=4))
    # near misses only: one flipped bit of a plain base
    base = np.frombuffer(b"ACGTN-acgtn", dtype=np.uint8)
    t = base[rng.integers(0, len(base), size=(24, 2000))] ^ (1 << rng.integers(0, 8, size=(24, 2000))).astype(np.uint8)
    _cmp(tracs_b200.pairsnp_matrix(t, dist=IMAX), oracle_mod.pairsnp_ascii(t, dist=IMAX, n_threads=4))


def test_pageable_source_is_staged(oracle_mod, monkeypatch):
    """A large pageable host matrix goes through the multi-threaded staging copy: same result as the direct copy."""
    s = synth.generate(600, 200_003, p_var=0.02, n_clusters=5, mu=3, p_N=0.01, seed=13)
    monkeypatch.setenv("TRACS_H2D_STAGE_MIN", "0")
    a = tracs_b200.pairsnp_matrix(s, dist=60)
    monkeypatch.setenv("TRACS_H2D_STAGE_MIN", str(1 << 40))
    b = tracs_b200.pairsnp_matrix(s, dist=60)
    for k in ("rows", "cols", "dist", "ncomp"):
        assert a[k].tolist() == b[k].tolist()
    _cmp(a, oracle_mod.pairsnp_ascii(s, dist=60, n_threads=8))


@pytest.mark.parametrize("n,L,p_var", [(600, 20000, 0.03), (300, 70001, 0.02), (1100, 9000, 0.04), (257, 4096, 0.01), (900, 33000, 0.2)])
def test_early_extraction_ingest_matches_oracle(oracle_mod, monkeypatch, n, L, p_var):
    """k_pack with the extracting warp (sites listed from the first 256 samples) + late gather + k_slice must give
    the planes of the two-pass ingest: forced on small inputs, compared with the oracle and with TRACS_INGEST=split."""
    s = synth.generate(n, L, p_var=p_var, n_clusters=6, mu=3, p_N=0.02, p_amb=0.05, seed=n + L, lowercase=0.05,
                       odd_chars=0.01, three_base=True)
    # sites that only start to vary after the first chunk of samples
    rng = np.random.default_rng(n)
    for c in rng.integers(0, L, size=40):
        s[:, c] = ord("A")
        s[rng.integers(256, n), c] = ord("T")
    dist = IMAX if n < 1000 else 60
    orc = oracle_mod.pairsnp_ascii(s, dist=dist, n_threads=4)
    monkeypatch.setenv("TRACS_INGEST", "early")
    res = tracs_b200.pairsnp_matrix(s, dist=dist)
    st_early = tracs_b200.last_stats()
    _cmp(res, orc)
    monkeypatch.setenv("TRACS_INGEST", "split")
    _cmp(tracs_b200.pairsnp_matrix(s, dist=dist), orc)
    assert tracs_b200.last_stats()["n_variable_sites"] == st_early["n_variable_sites"]


@pytest.mark.parametrize("n_clusters,dist,expect", [(60, 20, "refine"), (3, 20, "fallback"), (60, 0, "refine"), (3, 2047, "any"),
                                                    (60, 100, "any"), (60, 300, "any")])
def test_prefilter_refine_and_fallback(oracle_mod, n_clusters, dist, expect):
    # long enough (>= 256 words of variable sites) for the filter-and-refine path to engage
    s = synth.generate(300, 200_000, p_var=0.06, n_clusters=n_clusters, mu=4, p_N=0.002, p_amb=0.01, seed=41 + n_clusters)
    res = tracs_b200.pairsnp_matrix(s, dist=dist)
    st = tracs_b200.last_stats()
    _cmp(res, oracle_mod.pairsnp_ascii(s, dist=dist, n_threads=4))
    assert st["n_words"] >= 256
    if expect == "refine":
        # dist 0 / 20: the first window (4 words = 128 variable sites) is enough
        assert st["ms_refine"] > 0 and st["swept_wordpairs"] == st["n_pairs"] * 4
    elif expect == "fallback":
        # too many pairs survive the 4-, 8-, 16- and 64-word windows: four attempts, then the full-length sweep
        assert st["ms_refine"] == 0 and st["n_candidates"] > 0 and st["swept_wordpairs"] > st["n_pairs"] * (4 + 8 + 16 + 64)
    full = tracs_b200.pairsnp_matrix(s, dist=dist, full_sweep=True)
    st2 = tracs_b200.last_stats()
    assert st2["n_candidates"] == 0 and st2["ms_refine"] == 0
    for k in ("rows", "cols", "dist", "ncomp"):
        assert full[k].tolist() == res[k].tolist()


def test_identical_and_allN(oracle_mod):
    s = synth.generate(40, 500, p_var=0.0, p_N=0.0, gaps=0, seed=3)
    s[7, :] = ord("N")
    s[9, :] = ord("-")
    res = tracs_b200.pairsnp_matrix(s, dist=0)
    _cmp(res, oracle_mod.pairsnp_ascii(s, dist=0))
    assert len(res["rows"]) == 40 * 39 // 2


def test_negative_dist_and_empty(oracle_mod):
    s = synth.generate(10, 100, p_var=0.3, seed=5)
    res = tracs_b200.pairsnp_matrix(s, dist=-1)
    assert len(res["rows"]) == 0


def test_two_file_ranges(oracle_mod):
    s = synth.generate(300, 3000, p_var=0.05, n_clusters=3, mu=4, p_N=0.01, p_amb=0.02, seed=11)
    for n1 in (1, 100, 128, 299):
        res = tracs_b200.pairsnp_matrix(s, dist=60, i_end=n1, j_start=n1)
        _cmp(res, oracle_mod.pairsnp_ascii(s, i_end=n1, j_start=n1, dist=60, n_threads=4))


def test_sharded_equals_single(oracle_mod):
    s = synth.generate(700, 4000, p_var=0.05, n_clusters=5, mu=4, p_N=0.01, seed=12)
    full = tracs_b200.pairsnp_matrix(s, dist=80)
    for world in (2, 3, 8):
        parts = [tracs_b200.pairsnp_matrix(s, dist=80, shard_rank=r, shard_world=world) for r in range(world)]
        key = np.concatenate([(p["rows"] << np.uint64(32)) | p["cols"] for p in parts])
        order = np.argsort(key, kind="stable")
        for k in ("rows", "cols", "dist", "ncomp"):
            assert np.concatenate([p[k] for p in parts])[order].tolist() == full[k].tolist()


def test_fasta_entry_point(oracle_mod, tmp_path):
    s = synth.generate(37, 2500, p_var=0.05, n_clusters=3, mu=3, p_N=0.02, p_amb=0.05, seed=21, lowercase=0.1, odd_chars=0.01)
    for k, (gz, width, desc) in enumerate([(False, 0, False), (True, 60, True), (False, 7, True)]):
        p = str(tmp_path / ("a%d.fa%s" % (k, ".gz" if gz else "")))
        synth.write_fasta(p, s, width=width, descriptions=desc)
        got = tracs_b200.pairsnp(fasta=[p], n_threads=2, dist=50, filter=False)
        exp = oracle_mod.pairsnp([p], n_threads=2, dist=50)
        assert isinstance(got[0], list) and isinstance(got[3], list)
        for t in range(6):
            assert got[t] == exp[t]
    p1, p2 = str(tmp_path / "q.fa"), str(tmp_path / "db.fa.gz")
    synth.write_fasta(p1, s[:10], names=["q%d" % i for i in range(10)])
    synth.write_fasta(p2, s[10:], names=["d%d" % i for i in range(27)])
    got = tracs_b200.pairsnp(fasta=[p1, p2], n_threads=1, dist=IMAX, filter=False)
    exp = oracle_mod.pairsnp([p1, p2], dist=IMAX)
    for t in range(6):
        assert got[t] == exp[t]


def test_fasta_errors(tmp_path):
    p = str(tmp_path / "ragged.fa")
    open(p, "w").write(">a\nACGT\n>b\nACG\n")
    with pytest.raises(RuntimeError, match="variable sequence lengths"):
        tracs_b200.pairsnp(fasta=[p], n_threads=1, dist=10, filter=False)
    with pytest.raises(RuntimeError, match="Invalid number of fasta files"):
        tracs_b200.pairsnp(fasta=[p, p, p], n_threads=1, dist=10, filter=False)


def test_trans_dist_kat_and_grid(oracle_mod):
    # reference tests/test_trans_distance.py:29-42 (delta = one day, CLI default rates)
    d = 86400 / 31556952.0
    p0, eK = tracs_b200.trans_dist(np.array([0, 2]), np.array([d, d]), 29.903, 73.0, 0.01)
    assert abs(np.exp(p0[0]) - 0.23794988406662973) < 1e-6 and abs(np.exp(p0[1]) - 0.024467137572328577) < 1e-6
    assert abs(eK[0] - 2.6335200453700187) < 1e-6 and abs(eK[1] - 7.315670110063259) < 1e-6
    for lamb, beta in ((29.903, 73.0), (5.3, 6.0)):
        for thr in (0.01, 1e-6):
            N = np.repeat(np.arange(0, 41), 60).astype(np.int32)
            days = np.tile(np.arange(0, 180, 3), 41)
            dt = days * 86400.0 / 31556952.0
            p0, eK = tracs_b200.trans_dist(N, dt, lamb, beta, thr)
            op0, oeK, ke = oracle_mod.trans_dist(N, dt, lamb, beta, thr, with_k_exit=True)
            p0, eK = np.array(p0), np.array(eK)
            assert np.allclose(p0, op0, rtol=1e-6, atol=0)
            dom = np.isfinite(oeK) & ((N + ke + 1 < 10000) | (dt == 0))
            assert dom.sum() > 0.9 * dom.size
            assert np.allclose(eK[dom], oeK[dom], rtol=1e-6, atol=0)


def test_fused_trans(oracle_mod):
    s = synth.generate(200, 3000, p_var=0.05, n_clusters=4, mu=3, p_N=0.01, seed=31)
    days = np.random.default_rng(1).integers(0, 120, size=200).astype(np.int32)
    res = tracs_b200.pairsnp_matrix(s, dist=30, days=days, lamb=29.903, beta=73.0, threshold_Ek=0.01)
    r, c, d, f, nn = oracle_mod.pairsnp_ascii(s, dist=30)
    assert res["rows"].tolist() == r.tolist() and res["dist"].tolist() == d.tolist()
    dt = np.abs(days[r.astype(int)] * 86400.0 - days[c.astype(int)] * 86400.0) / 31556952.0
    assert res["datediff"].tolist() == dt.tolist()
    op0, oeK = oracle_mod.trans_dist(d.astype(np.int32), dt, 29.903, 73.0, 0.01)
    assert np.allclose(res["p0_log"], op0, rtol=1e-6, atol=0)
    assert np.allclose(res["eK"], oeK, rtol=1e-6, atol=0)


def test_min_over_refs():
    rng = np.random.default_rng(5)
    a = rng.integers(0, 50, 5000).astype(np.uint64)
    b = rng.integers(0, 50, 5000).astype(np.uint64)
    v = rng.integers(0, 100, 5000).astype(np.float64)
    oa, ob, ov = tracs_b200.min_over_refs(a, b, v)
    exp = {}
    for x, y, z in zip(a.tolist(), b.tolist(), v.tolist()):
        k = (min(x, y), max(x, y))
        exp[k] = min(exp.get(k, 1e300), z)
    ks = sorted(exp)
    assert list(zip(oa.tolist(), ob.tolist())) == ks
    assert ov.tolist() == [exp[k] for k in ks]


def test_recombination_filter(oracle_mod):
    # filter=True (src/pairsnp.hpp:251-318): scattered SNPs plus a dense block that must be removed
    s = synth.generate(24, 60_000, p_var=0.02, n_clusters=3, mu=6, p_N=0.002, p_amb=0.01, seed=51)
    rng = np.random.default_rng(2)
    for k in range(0, 24, 3):                      # recombination-like blocks: 30 substitutions inside 400 bp
        start = int(rng.integers(1000, 59000))
        sites = start + rng.choice(400, size=30, replace=False)
        s[k, sites] = np.where(s[k, sites] == ord("A"), ord("C"), ord("A"))
    for dist in (IMAX, 150):
        res = tracs_b200.pairsnp_matrix(s, dist=dist, filter=True)
        r, c, d, f, nn = oracle_mod.pairsnp_ascii(s, dist=dist, filter=True, n_threads=4)
        assert res["rows"].tolist() == r.tolist() and res["dist"].tolist() == d.tolist()
        assert res["filt"].tolist() == f.tolist()
        assert (f < d).any() and res["ncomp"].tolist() == nn.tolist()


def test_recombination_filter_on_early_extraction_ingest(oracle_mod, monkeypatch):
    """The filter walks each pair's SNP positions in ascending order: the planes built by the early-extraction ingest
    (early list merged with late sites) must keep that order. n > 256 so that the path can be forced."""
    s = synth.generate(300, 40_000, p_var=0.02, n_clusters=30, mu=6, p_N=0.002, p_amb=0.01, seed=52)
    rng = np.random.default_rng(3)
    for k in range(0, 300, 7):
        start = int(rng.integers(1000, 39000))
        sites = start + rng.choice(400, size=30, replace=False)
        s[k, sites] = np.where(s[k, sites] == ord("A"), ord("C"), ord("A"))
    for c in rng.integers(0, 40_000, size=30):      # sites that only vary after the first 256 samples
        s[:, c] = ord("G")
        s[rng.integers(256, 300), c] = ord("T")
    monkeypatch.setenv("TRACS_INGEST", "early")
    res = tracs_b200.pairsnp_matrix(s, dist=150, filter=True)
    assert tracs_b200.last_stats()["n_early_sites"] > 0
    r, c, d, f, nn = oracle_mod.pairsnp_ascii(s, dist=150, filter=True, n_threads=8)
    assert res["rows"].tolist() == r.tolist() and res["cols"].tolist() == c.tolist() and res["dist"].tolist() == d.tolist()
    assert res["filt"].tolist() == f.tolist() and (f < d).any() and res["ncomp"].tolist() == nn.tolist()


def test_filter_golden_and_fused_trans(oracle_mod):
    import json
    gold = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
    G = json.load(open(os.path.join(gold, "golden.json")))
    for case in G["filter"]:
        r = tracs_b200.pairsnp(fasta=[os.path.join(gold, case["fasta"])], n_threads=1, dist=case["dist"], filter=True)
        assert r[0] == case["rows"] and r[2] == case["d"] and r[4] == case["filt"]
    # fused likelihood is fed the FILTERED distance when the filter is on (tracs/distance.py:182-192)
    s = synth.generate(60, 30_000, p_var=0.03, n_clusters=4, mu=5, p_N=0.002, seed=52)
    days = np.random.default_rng(3).integers(0, 100, size=60).astype(np.int32)
    res = tracs_b200.pairsnp_matrix(s, dist=200, filter=True, days=days)
    r, c, d, f, nn = oracle_mod.pairsnp_ascii(s, dist=200, filter=True)
    assert res["filt"].tolist() == f.tolist()
    dt = np.abs(days[r.astype(int)] * 86400.0 - days[c.astype(int)] * 86400.0) / 31556952.0
    op0, oeK = oracle_mod.trans_dist(f.astype(np.int32), dt, 29.903, 73.0, 0.01)
    assert np.allclose(res["p0_log"], op0, rtol=1e-6, atol=0)
    pos = dt > 0
    assert np.allclose(res["eK"][pos], oeK[pos], rtol=1e-6, atol=0)


def test_device_packed_columns_match_host():
    import torch
    from tracs_b200.multi import _DevBytes, _sections, DEV_COLUMNS, _DEV_DTYPES
    s = synth.generate(300, 4000, p_var=0.05, n_clusters=4, mu=3, p_N=0.01, seed=61)
    days = np.random.default_rng(1).integers(0, 50, size=300).astype(np.int32)
    res = tracs_b200.pairsnp_matrix(s, dist=60, days=days, copy=False, keep_on_device=True)
    ptr, nbytes = res["dev_packed"]
    E = len(res["rows"])
    assert nbytes == 32 * E and E > 0
    host = torch.as_tensor(_DevBytes(ptr, nbytes), device="cuda").cpu().numpy()
    secs = dict(zip(DEV_COLUMNS, _sections(host, E, _DEV_DTYPES)))
    for c in ("rows", "cols", "dist", "ncomp"):
        assert secs[c].astype(np.uint64).tolist() == res[c].tolist()
    assert np.array_equal(secs["p0_log"], res["p0_log"]) and np.array_equal(secs["eK"], res["eK"])


def _site_sharded_local(torch, s, world, dist):
    """Emulates R ranks of the site-sharded sweep on one GPU (collectives replaced by torch ops)."""
    import ctypes as C
    from tracs_b200 import sites, _lib
    n, L = s.shape
    dev = torch.device("cuda")
    slabs, handles, cands = [], [], []
    for r in range(world):
        lo, hi = sites.slab_bounds(L, r, world)
        Ls = hi - lo
        pitch = max(128, (Ls + 127) // 128 * 128)
        buf = torch.full((n, pitch), ord("N"), dtype=torch.uint8, device=dev)
        if Ls:
            buf[:, :Ls] = torch.from_numpy(np.ascontiguousarray(s[:, lo:hi])).to(dev)
        slabs.append(buf)
        h, kptr, cnt, st = sites.open_shard(buf.data_ptr(), n, Ls, pitch, dist, r, world)
        handles.append(h)
        cands.append(torch.as_tensor(sites._Dev(kptr, cnt * 8), device=dev).view(torch.int64).clone() if cnt
                     else torch.empty(0, dtype=torch.int64, device=dev))
    keys, _ = torch.sort(torch.cat(cands))
    E = keys.numel()
    d = torch.zeros(max(E, 1), dtype=torch.int32, device=dev)
    u = torch.zeros(max(E, 1), dtype=torch.int32, device=dev)
    for h in handles:
        dr, ur = torch.zeros_like(d), torch.zeros_like(u)
        if E:
            _lib.check(_lib.lib().tracs_site_shard_partials(h, C.c_void_p(keys.data_ptr()), E, C.c_void_p(dr.data_ptr()), C.c_void_p(ur.data_ptr())))
        d += dr
        u += ur
        _lib.lib().tracs_site_shard_close(h)
    keep = d[:E] <= dist
    k = keys[:E][keep].cpu().numpy().astype(np.uint64)
    return (k >> np.uint64(32), k & np.uint64(0xFFFFFFFF), d[:E][keep].cpu().numpy().astype(np.uint64),
            (L - u[:E][keep].cpu().numpy().astype(np.int64)).astype(np.uint64), E)


@pytest.mark.parametrize("world", [1, 2, 5])
def test_site_sharded_equals_oracle(oracle_mod, world):
    import torch
    s = synth.generate(420, 150_000, p_var=0.06, n_clusters=50, mu=4, p_N=0.002, p_amb=0.01, seed=71)
    for dist in (0, 25):
        rows, cols, d, nn, n_cand = _site_sharded_local(torch, s, world, dist)
        r, c, od, f, onn = oracle_mod.pairsnp_ascii(s, dist=dist, n_threads=4)
        assert rows.tolist() == r.tolist() and cols.tolist() == c.tolist()
        assert d.tolist() == od.tolist() and nn.tolist() == onn.tolist()
        assert n_cand < 0.2 * 420 * 419 / 2


def test_synth_slabs_are_columns_of_the_whole():
    import torch
    n, L = 64, 10_000
    kw = dict(seed=5, p_var=0.05, n_clusters=4, mu=3.0, p_N=0.01, p_amb=0.02, gc=0.4)
    whole = torch.empty((n, 10_112), dtype=torch.uint8, device="cuda")
    tracs_b200.synth_device(whole.data_ptr(), n, L, 10_112, **kw)
    for lo, hi in ((0, 3840), (3840, 7680), (7680, 10_000)):
        pitch = (hi - lo + 127) // 128 * 128
        slab = torch.empty((n, pitch), dtype=torch.uint8, device="cuda")
        tracs_b200.synth_device(slab.data_ptr(), n, hi - lo, pitch, site_offset=lo, L_total=L, **kw)
        assert torch.equal(slab[:, :hi - lo], whole[:, lo:hi])


def test_sites_driver_world1_matches_fused_path():
    import torch
    from tracs_b200 import sites
    s = synth.generate(500, 150_000, p_var=0.06, n_clusters=60, mu=4, p_N=0.002, seed=81)
    days = np.random.default_rng(4).integers(0, 150, size=500).astype(np.int32)
    n, L = s.shape
    pitch = (L + 127) // 128 * 128
    buf = torch.full((n, pitch), ord("N"), dtype=torch.uint8, device="cuda")
    buf[:, :L] = torch.from_numpy(s).cuda()
    res, st = sites.sweep(torch, None, torch.device("cuda"), 0, 1, buf.data_ptr(), n, L, pitch, L, 20, days=days)
    ref = tracs_b200.pairsnp_matrix(s, dist=20, days=days)
    for k in ("rows", "cols", "dist", "ncomp"):
        assert res[k].tolist() == ref[k].tolist()
    assert np.array_equal(res["datediff"], ref["datediff"])
    assert np.allclose(res["p0_log"], ref["p0_log"], rtol=1e-12) and np.allclose(res["eK"], ref["eK"], rtol=1e-12)


@pytest.mark.parametrize("n,L,dist", [(100, 3000, IMAX), (300, 20000, 30), (129, 40000, 2000), (513, 9000, IMAX)])
def test_tensor_core_sweep_matches_oracle(oracle_mod, n, L, dist):
    # K1': tcgen05 int8 one-hot GEMM with the N-column correction; single bases, N, gaps, lower case -- no 2-/3-base codes
    s = synth.generate(n, L, p_var=0.08, n_clusters=5, mu=4, p_N=0.05, p_amb=0.0, seed=n + L, lowercase=0.05, odd_chars=0.01)
    res = tracs_b200.pairsnp_matrix(s, dist=dist, full_sweep="tc")
    _cmp(res, oracle_mod.pairsnp_ascii(s, dist=dist, n_threads=4))
    st = tracs_b200.last_stats()
    assert st["ms_refine"] == 0 and st["n_candidates"] == 0


def test_tensor_core_sweep_refuses_partial_ambiguity():
    s = synth.generate(64, 2000, p_var=0.1, n_clusters=3, mu=3, p_N=0.01, p_amb=0.2, seed=9)
    with pytest.raises(RuntimeError, match="IUPAC"):
        tracs_b200.pairsnp_matrix(s, dist=50, full_sweep="tc")
    tracs_b200.pairsnp_matrix(s, dist=50)  # the LOP3/POPC path takes it


def test_tensor_core_sweep_modes(oracle_mod):
    # query x db ranges, row-block shards and the automatic choice (unthresholded => full-length => tensor cores)
    s = synth.generate(700, 6000, p_var=0.08, n_clusters=6, mu=4, p_N=0.03, seed=91)
    for n1 in (100, 300):
        res = tracs_b200.pairsnp_matrix(s, dist=200, i_end=n1, j_start=n1, full_sweep="tc")
        _cmp(res, oracle_mod.pairsnp_ascii(s, i_end=n1, j_start=n1, dist=200, n_threads=4))
    full = tracs_b200.pairsnp_matrix(s, dist=IMAX)            # auto: no prefilter possible -> k_sweep_tc3
    _cmp(full, oracle_mod.pairsnp_ascii(s, dist=IMAX, n_threads=4))
    pop = tracs_b200.pairsnp_matrix(s, dist=IMAX, full_sweep=True)   # forced LOP3/POPC kernel
    for k in ("rows", "cols", "dist", "ncomp"):
        assert pop[k].tolist() == full[k].tolist()
    parts = [tracs_b200.pairsnp_matrix(s, dist=150, shard_rank=r, shard_world=3, full_sweep="tc") for r in range(3)]
    one = tracs_b200.pairsnp_matrix(s, dist=150, full_sweep=True)
    key = np.concatenate([(p["rows"] << np.uint64(32)) | p["cols"] for p in parts])
    order = np.argsort(key, kind="stable")
    for k in ("rows", "cols", "dist", "ncomp"):
        assert np.concatenate([p[k] for p in parts])[order].tolist() == one[k].tolist()


def test_filter_decisions_match_incomplete_beta_cdf():
    """k_filter_recomb sums the binomial pmf term by term; Boost (what the reference links) evaluates the regularised
    incomplete beta function. On near-threshold SNP layouts the kernel's filt must equal the windowing restated in
    Python with scipy.stats.binom (an incomplete-beta implementation) -- see tests/test_filter_pin.py for the margins."""
    from scipy import stats
    from oracle import binom_check as bc
    rng = np.random.default_rng(11)
    L, n = 200_000, 161
    base = np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, size=L)]
    s = np.repeat(base[None, :], n, axis=0)
    layouts = [None]
    for k in range(1, n):
        snp = set(rng.choice(L, size=int(rng.integers(3, 60)), replace=False).tolist())
        start, width = int(rng.integers(1000, L - 6000)), int(rng.integers(20, 5000))
        snp |= set((start + rng.choice(width, size=min(int(rng.integers(2, 12)), width), replace=False)).tolist())
        snp = np.array(sorted(snp))
        s[k, snp] = np.where(base[snp] == ord("A"), ord("C"), ord("A"))
        layouts.append(snp.tolist())
    res = tracs_b200.pairsnp_matrix(s, dist=IMAX, filter=True, want_ncomp=False)
    first = {int(c): (int(d), int(f)) for r, c, d, f in zip(res["rows"], res["cols"], res["dist"], res["filt"]) if r == 0}
    cdf = lambda nn, p, k: 1.0 if k >= nn else float(stats.binom.cdf(k, nn, p))
    for k in range(1, n):
        d, f = first[k]
        assert d == len(layouts[k])
        assert f == bc.filtered_distance(layouts[k], L, cdf)[0], k


@pytest.mark.parametrize("n,L,dist,p_N", [(100, 3000, IMAX, 0.0), (300, 20000, 30, 0.0), (513, 9000, IMAX, 0.0), (257, 33000, 500, 0.2),
                                          (130, 70001, IMAX, 0.01), (1100, 6000, 40, 0.0), (900, 5000, 60, 0.05)])
def test_tensor_core_sweep_planes(oracle_mod, n, L, dist, p_N):
    """k_sweep_tc3: three +-1 planes when no variable site holds an N (NP = 3), plus the N plane and the per-sample N
    counts otherwise (NP = 4); against the oracle."""
    s = synth.generate(n, L, p_var=0.08, n_clusters=5, mu=4, p_N=p_N, p_amb=0.0, seed=n + L, lowercase=0.05, gaps=0 if p_N == 0 else 2)
    orc = oracle_mod.pairsnp_ascii(s, dist=dist, n_threads=4)
    res = tracs_b200.pairsnp_matrix(s, dist=dist, full_sweep="tc")      # k_sweep_tc3: 128 x 512 super-tiles
    assert tracs_b200.last_stats()["tc_sweep"] in (33.0, 34.0)          # generation 3, three or four operand planes
    _cmp(res, orc)
    for n1 in (n // 3, n - 1):                                           # query x db ranges cut super-tiles short
        _cmp(tracs_b200.pairsnp_matrix(s, dist=dist, i_end=n1, j_start=n1, full_sweep="tc"),
             oracle_mod.pairsnp_ascii(s, i_end=n1, j_start=n1, dist=dist, n_threads=4))
