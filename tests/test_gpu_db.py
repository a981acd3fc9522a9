"""GPU: the resident sample database (tracs_b200.Database, tracs_db_*) returns exactly the two-file call on [q; db] with
i_end = j_start = nq: every column, the same order, the same indices, over shapes, options, input forms, ingest paths,
newly variable sites, repeated and interrupted queries, the likelihood columns, the golden files and the command line."""
import os
import subprocess
import sys

import numpy as np
import pytest

import tracs_b200
from tracs_b200 import synth

pytestmark = pytest.mark.gpu
IMAX = 2147483647
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")
COLS = ("rows", "cols", "dist", "ncomp", "p0_log", "eK", "datediff")


def _two_file(q, db, **kw):
    nq = q.shape[0]
    return tracs_b200.pairsnp_matrix(np.concatenate([q, db]), i_end=nq, j_start=nq, **kw)


def _same(got, want):
    for k in COLS:
        a, b = got[k], want[k]
        assert (a is None) == (b is None), k
        if a is not None:
            assert a.dtype == b.dtype and a.shape == b.shape, (k, a.shape, b.shape)
            assert np.array_equal(a, b), (k, np.argwhere(a != b)[:5])


def _pair(n, L, seed, **kw):
    args = dict(p_var=0.05, n_clusters=5, mu=3, p_N=0.01, p_amb=0.02, seed=seed)
    args.update(kw)
    return synth.generate(n, L, **args)


@pytest.mark.parametrize("n_db,nq,L", [(1, 1, 31), (1, 129, 32), (127, 2, 4097), (128, 128, 4097), (129, 127, 31), (129, 1, 4097),
                                       (1000, 129, 4097), (1000, 128, 70000), (3000, 2, 4097), (300, 4200, 4097), (3000, 129, 32)])
def test_shapes_match_the_two_file_call(oracle_mod, n_db, nq, L):
    s = _pair(n_db + nq, L, seed=n_db * 31 + nq * 7 + L)
    q, db = s[:nq], s[nq:]
    with tracs_b200.Database(db) as d:
        for dist in (20, IMAX):
            got = d.query(q, dist=dist)
            _same(got, _two_file(q, db, dist=dist))
            assert tracs_b200.last_stats()["n_pairs"] == nq * n_db
    if (n_db + nq) * L <= 3_000_000:
        r, c, dd, _, nn = oracle_mod.pairsnp_ascii(s, i_end=nq, j_start=nq, dist=20, n_threads=8)
        with tracs_b200.Database(db) as d:
            got = d.query(q, dist=20)
        assert got["rows"].tolist() == r.tolist() and got["cols"].tolist() == c.tolist()
        assert got["dist"].tolist() == dd.tolist() and got["ncomp"].tolist() == nn.tolist()


@pytest.mark.parametrize("dist", [0, 1, 20, 100, IMAX])
def test_options(dist):
    s = _pair(700, 9000, seed=dist % 997, p_amb=0.0)
    q, db = s[:150], s[150:]
    with tracs_b200.Database(db) as d:
        for want_ncomp in (True, False):
            for fs in (False, True, "tc"):
                kw = dict(dist=dist, want_ncomp=want_ncomp, full_sweep=fs)
                _same(d.query(q, **kw), _two_file(q, db, **kw))


def test_input_forms():
    import torch
    n_db, nq, L = 600, 140, 9000
    s = _pair(n_db + nq, L, seed=11)
    q, db = s[:nq], s[nq:]
    want = _two_file(q, db, dist=30)
    pitch = (L + 31) // 32 * 32
    nib_db, p4 = tracs_b200.pack_nibbles(db)
    nib_q, _ = tracs_b200.pack_nibbles(q)

    def dev_ascii(a):
        t = torch.full((a.shape[0], pitch), ord("N"), dtype=torch.uint8)
        t[:, :L] = torch.from_numpy(a)
        return t.cuda()

    dq, dq4 = dev_ascii(q), torch.from_numpy(nib_q).cuda()
    ddb, ddb4 = dev_ascii(db), torch.from_numpy(nib_db).cuda()
    dbs = [tracs_b200.Database(db), tracs_b200.Database(nib_db, packed=True, L=L),
           tracs_b200.Database.from_device(ddb.data_ptr(), n_db, L, pitch), tracs_b200.Database.from_device(ddb4.data_ptr(), n_db, L, p4, packed=True)]
    for d in dbs:
        _same(d.query(q, dist=30), want)
        _same(d.query(nib_q, dist=30, packed=True, L=L), want)
        _same(d.query_device(dq.data_ptr(), nq, pitch, dist=30), want)
        _same(d.query_device(dq4.data_ptr(), nq, p4, dist=30, packed=True), want)
        d.close()
        d.close()


def test_early_extraction_and_n_plane_paths(monkeypatch):
    import torch
    n_db, nq, L = 1100, 60, 70000
    p4 = (L + 31) // 32 * 16
    buf = torch.empty((n_db + nq) * p4, dtype=torch.uint8, device="cuda")
    tracs_b200.synth_device(buf.data_ptr(), n_db + nq, L, p4, seed=3, p_var=0.01, n_clusters=20, mu=5.0, p_N=1e-3, gaps=2, packed=True)
    host = buf.view(n_db + nq, p4).cpu().numpy()
    for env in ({}, {"TRACS_NBLOCKS": "dense"}, {"TRACS_NPLANE": "always"}, {"TRACS_NPLANE": "sparse"}, {"TRACS_PAIRS": "sparse"},
                {"TRACS_PAIRS": "dense"}):
        for k in ("TRACS_NBLOCKS", "TRACS_NPLANE", "TRACS_PAIRS"):
            monkeypatch.delenv(k, raising=False)
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        want = tracs_b200.pairsnp_packed(buf.data_ptr(), n_db + nq, L, p4, i_end=nq, j_start=nq, dist=20)
        with tracs_b200.Database.from_device(buf.data_ptr() + nq * p4, n_db, L, p4, packed=True) as d:
            open_stats = tracs_b200.last_stats()
            assert open_stats["n_early_sites"] > 0
            _same(d.query_device(buf.data_ptr(), nq, p4, dist=20, packed=True), want)
            _same(d.query(host[:nq], packed=True, L=L, dist=20), want)


def _built_new_sites():
    """A database with invariant sites (some with N / a code containing the base) and queries that make them variable."""
    rng = np.random.default_rng(17)
    n_db, nq, L = 400, 40, 3000
    db = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, L)][None, :].repeat(n_db, 0).copy()
    var = rng.choice(L, 100, replace=False)
    db[rng.integers(0, n_db, 300), var[rng.integers(0, 100, 300)]] = ord("T")
    inv = np.setdiff1d(np.arange(L), var)[:400]
    db[5, inv[:50]] = ord("N")
    code_with = {ord("A"): "R", ord("C"): "M", ord("G"): "S", ord("T"): "W"}  # 2-base codes containing the base
    disjoint = {ord("A"): "Y", ord("C"): "R", ord("G"): "W", ord("T"): "S"}  # 2-base codes without it
    for s in inv[50:100]:
        db[7, s] = ord(code_with[db[0, s]])
    q = db[:nq].copy()
    q[:, :] = db[0]
    q[1:, var] = db[1:nq, var]
    for k, s in enumerate(inv[:100]):
        q[k % nq, s] = ord("C") if db[0, s] != ord("C") else ord("G")        # a different base
    for k, s in enumerate(inv[100:150]):
        q[k % nq, s] = ord(disjoint[db[0, s]])                               # a 2-base code disjoint from it
    for k, s in enumerate(inv[150:200]):
        q[k % nq, s] = ord(code_with[db[0, s]])                              # a code that contains it (not new)
    for k, s in enumerate(inv[200:250]):
        q[k % nq, s] = ord("N")                                              # N (not new)
    for s in inv[250:300]:
        q[0, s] = ord("C") if db[0, s] != ord("C") else ord("G")             # varies only inside the batch
    return q, db


def test_newly_variable_sites(oracle_mod):
    q, db = _built_new_sites()
    nq = q.shape[0]
    with tracs_b200.Database(db) as d:
        v_db = d.info()["n_variable_sites"]
        for fs in (False, True):
            got = d.query(q, dist=IMAX, full_sweep=fs)
            _same(got, _two_file(q, db, dist=IMAX, full_sweep=fs))
        info = d.info()
        assert info["new_sites"] > 0 and v_db > 0
        assert v_db + info["new_sites"] == tracs_b200.last_stats()["n_variable_sites"]
    r, c, dd, _, nn = oracle_mod.pairsnp_ascii(np.concatenate([q, db]), i_end=nq, j_start=nq, dist=IMAX, n_threads=8)
    assert got["dist"].tolist() == dd.tolist() and got["ncomp"].tolist() == nn.tolist() and got["cols"].tolist() == c.tolist()


def test_no_state_leaks_between_queries():
    qa, db = _built_new_sites()
    s = _pair(db.shape[0] + 300, db.shape[1], seed=5)
    qb = s[:300]  # unrelated samples: most sites newly variable
    with tracs_b200.Database(db) as d:
        ra = d.query(qa, dist=IMAX)
        na = d.info()["new_sites"]
        rb = d.query(qb, dist=50)
        nb = d.info()["new_sites"]
        ra2 = d.query(qa, dist=IMAX)
        assert na != nb and d.info()["new_sites"] == na
    _same(ra, _two_file(qa, db, dist=IMAX))
    _same(rb, _two_file(qb, db, dist=50))
    _same(ra2, ra)


def test_likelihood_columns():
    n_db, nq, L = 900, 4300, 6000  # two query chunks
    s = _pair(n_db + nq, L, seed=23, p_amb=0.0)
    days = (np.arange(n_db + nq) * 13 % 200).astype(np.int32)
    q, db = s[:nq], s[nq:]
    with tracs_b200.Database(db) as d:
        for dist in (20, 200):
            got = d.query(q, dist=dist, days=days)
            assert got["p0_log"] is not None
            _same(got, _two_file(q, db, dist=dist, days=days))


def test_two_file_golden_through_from_fasta(oracle_mod):
    qp, dbp = os.path.join(GOLD, "query.fasta"), os.path.join(GOLD, "db.fasta.gz")
    with tracs_b200.Database.from_fasta(dbp, n_threads=2) as d:
        qs, qn = tracs_b200.read_fasta(qp)
        got = d.query(qs)
        names = qn + d.names
    r, c, dd, nm, _, nn = oracle_mod.pairsnp(fasta=[qp, dbp], n_threads=2, dist=IMAX)
    assert names == nm
    assert got["rows"].tolist() == list(r) and got["cols"].tolist() == list(c)
    assert got["dist"].tolist() == list(dd) and got["ncomp"].tolist() == list(nn)


def test_borrowed_buffer_is_never_written():
    import torch
    n_db, nq, L = 800, 200, 20000
    p4 = (L + 31) // 32 * 16
    buf = torch.empty(n_db * p4, dtype=torch.uint8, device="cuda")
    tracs_b200.synth_device(buf.data_ptr(), n_db, L, p4, seed=8, p_var=0.02, n_clusters=10, mu=4.0, packed=True)
    before = buf.clone()
    qs = _pair(nq, L, seed=9)
    with tracs_b200.Database.from_device(buf.data_ptr(), n_db, L, p4, packed=True) as d:
        for dist in (5, IMAX):
            d.query(qs, dist=dist)
        d.query(qs[:1], dist=IMAX, full_sweep=True)
    assert torch.equal(buf, before)


def test_too_many_new_sites_fails_with_size_and_the_handle_stays_usable():
    import torch
    n_db, L = 2000, 200_000
    db = _pair(n_db, L, seed=12, p_var=0.001, p_amb=0.0)
    rng = np.random.default_rng(1)
    q = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, (1000, L))]  # unrelated: most sites become variable
    nib_q, p4 = tracs_b200.pack_nibbles(q)
    dq = torch.from_numpy(nib_q).cuda()
    with tracs_b200.Database(db) as d:
        small = d.query(db[:3], dist=5)
        tracs_b200.api._lib.lib().tracs_trim()
        torch.cuda.empty_cache()
        free, _ = torch.cuda.mem_get_info()
        # the query's bit-planes (~0.6 GB: 3000 samples x ~6250 words, two layouts) cannot fit next to this
        hog = torch.empty(free - (400 << 20), dtype=torch.uint8, device="cuda")
        try:
            with pytest.raises(RuntimeError, match=r"take 0\.\d GB and do not fit in device memory next to the database"):
                d.query_device(dq.data_ptr(), 1000, p4, dist=20, packed=True)
        finally:
            del hog
            torch.cuda.empty_cache()
        _same(d.query(db[:3], dist=5), small)
        _same(d.query(q[:50], dist=20), _two_file(q[:50], db, dist=20))


def test_sigint_between_chunks_leaves_the_handle_usable():
    code = r'''
import os, signal, sys, threading, time, torch
import numpy as np
sys.path.insert(0, %r)
import tracs_b200
n_db, nq, L = 60000, 16384, 40000
p4 = L // 2
buf = torch.empty((n_db + nq) * p4, dtype=torch.uint8, device="cuda")
tracs_b200.synth_device(buf.data_ptr(), n_db + nq, L, p4, seed=9, p_var=1.0, n_clusters=n_db, mu=0.0, p_N=0.0, gc=0.5, gaps=0, packed=True)
d = tracs_b200.Database.from_device(buf.data_ptr() + nq * p4, n_db, L, p4, packed=True)
d.query_device(buf.data_ptr(), 64, p4, dist=10, packed=True, full_sweep=True)   # warm-up
t0 = time.perf_counter()
d.query_device(buf.data_ptr(), nq, p4, dist=10, packed=True, full_sweep=True)
t_full = time.perf_counter() - t0
threading.Timer(t_full / 4, lambda: os.kill(os.getpid(), signal.SIGINT)).start()
try:
    d.query_device(buf.data_ptr(), nq, p4, dist=10, packed=True, full_sweep=True)
    print("NOT-INTERRUPTED")
except KeyboardInterrupt as ex:
    print("INTERRUPTED", str(ex))
assert signal.getsignal(signal.SIGINT) is signal.default_int_handler
a = d.query_device(buf.data_ptr() + (nq - 300) * p4, 300, p4, dist=500, packed=True)
b = tracs_b200.pairsnp_packed(buf.data_ptr() + (nq - 300) * p4, 300 + n_db, L, p4, i_end=300, j_start=300, dist=500)
assert all(np.array_equal(a[k], b[k]) for k in ("rows", "cols", "dist", "ncomp"))
print("AFTER", len(a["rows"]))
''' % ROOT
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600)
    assert "INTERRUPTED Interrupted by user!" in out.stdout and "AFTER" in out.stdout, out.stdout + out.stderr


def test_after_interrupt_results_equal_a_fresh_call():
    # the query rows a stopped query left behind are cleared by the next one: simulate the leftovers with a larger batch
    s = _pair(1500, 5000, seed=41)
    db = s[500:]
    with tracs_b200.Database(db) as d:
        d.query(s[:500], dist=IMAX)
        got = d.query(s[:3], dist=IMAX)
    _same(got, _two_file(s[:3], db, dist=IMAX))


@pytest.mark.parametrize("meta", [False, True])
@pytest.mark.parametrize("K", [None, "5"])
def test_command_line_matches_distance_msa_db(tmp_path, meta, K):
    # the golden two-file pair, and a synthetic database with two query files
    s = _pair(260, 3000, seed=77)
    sdb, sq1, sq2 = tmp_path / "sdb.fasta", tmp_path / "sq1.fasta", tmp_path / "sq2.fasta"
    for path, rows, tag in ((sdb, s[60:], "d"), (sq1, s[:30], "a"), (sq2, s[30:60], "b")):
        path.write_text("".join(">%s%d\n%s\n" % (tag, i, r.tobytes().decode()) for i, r in enumerate(rows)))
    dates = tmp_path / "dates.csv"
    names = ["q%d" % i for i in range(300)] + ["d%d" % i for i in range(300)] + ["a%d" % i for i in range(30)] + ["b%d" % i for i in range(30)]
    dates.write_text("sample,date\n" + "".join("%s,2020-%02d-%02d\n" % (nm, 1 + i % 12, 1 + i * 7 % 28) for i, nm in enumerate(names)))
    opts = (["--meta", str(dates)] if meta else []) + (["-K", K] if K else [])
    for db, msas in ((os.path.join(GOLD, "db.fasta.gz"), [os.path.join(GOLD, "query.fasta")]), (str(sdb), [str(sq1), str(sq2)])):
        a, b = str(tmp_path / "query.csv"), str(tmp_path / "distance.csv")
        subprocess.run([sys.executable, "-m", "tracs_b200.query", "--db", db, "--msa"] + msas + ["-o", a, "-D", "20"] + opts, cwd=ROOT, check=True)
        subprocess.run([sys.executable, "-m", "tracs_b200.distance", "--msa"] + msas + ["--msa-db", db, "-o", b, "-D", "20"] + opts, cwd=ROOT,
                       check=True)
        assert open(a, "rb").read() == open(b, "rb").read()
        assert K is not None or open(a).read().count("\n") > 1
