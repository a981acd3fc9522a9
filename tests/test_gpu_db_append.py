"""GPU: appending to the resident sample database (Database.append, tracs_db_append_*) returns exactly the one-shot call on
[db; b] with j_start = n_db (every pair with a sample in the batch), and leaves a database that behaves as one opened on
[db; b] from scratch: over shapes, options, sequences of appends that grow the buffers, newly variable sites, input forms,
ingest paths, the likelihood columns, the borrowed buffer, failures and interrupts, and the command line."""
import csv
import io
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


def _one_shot(s, n_db, **kw):
    return tracs_b200.pairsnp_matrix(s, j_start=n_db, **kw)


@pytest.mark.parametrize("n_db,m,L,kw", [
    (100, 29, 4097, dict(dist=0)),
    (129, 130, 4097, dict(dist=20)),
    (257, 3, 31, dict(dist=IMAX)),
    (300, 77, 70000, dict(dist=20)),                          # prefilter (V > 8 000 sites)
    (300, 77, 70000, dict(dist=20, full_sweep=True)),
    (300, 77, 70000, dict(dist=IMAX, full_sweep="tc")),
    (1, 200, 4097, dict(dist=IMAX, full_sweep=True)),
])
def test_one_shot_batch_range_matches_oracle(oracle_mod, n_db, m, L, kw):
    # i_end = n with j_start = n_db: the pairs of an append, as the one-shot call computes them
    s = _pair(n_db + m, L, seed=n_db + 7 * m + L, p_var=0.15 if L == 70000 else 0.05, p_amb=0.0 if kw.get("full_sweep") == "tc" else 0.02)
    got = _one_shot(s, n_db, **kw)
    st = tracs_b200.last_stats()
    assert st["n_pairs"] == n_db * m + m * (m - 1) // 2
    if L == 70000 and not kw.get("full_sweep") and kw["dist"] == 20:
        assert st["n_candidates"] > 0  # the prefilter ran
    r, c, dd, _, nn = oracle_mod.pairsnp_ascii(s, i_end=n_db + m, j_start=n_db, dist=kw["dist"], n_threads=8)
    assert got["rows"].tolist() == r.tolist() and got["cols"].tolist() == c.tolist()
    assert got["dist"].tolist() == dd.tolist() and got["ncomp"].tolist() == nn.tolist()


@pytest.mark.parametrize("n_db,m,L", [(1, 1, 31), (1, 129, 4097), (127, 128, 4097), (129, 127, 31), (1000, 1, 4097), (128, 129, 70000),
                                      (300, 4200, 4097), (2000, 300, 32)])
def test_append_equals_the_one_shot_call(n_db, m, L):
    s = _pair(n_db + m, L, seed=n_db * 31 + m * 7 + L)
    for dist in (20, IMAX):
        with tracs_b200.Database(s[:n_db]) as d:
            got = d.append(s[n_db:], dist=dist)
            assert tracs_b200.last_stats()["n_pairs"] == n_db * m + m * (m - 1) // 2
            assert d.n == n_db + m and d.info()["n"] == n_db + m
        _same(got, _one_shot(s, n_db, dist=dist))


@pytest.mark.parametrize("dist", [0, 20, IMAX])
def test_options(dist):
    s = _pair(850, 9000, seed=dist % 997, p_amb=0.0)
    n_db = 700
    for want_ncomp in (True, False):
        for fs in (False, True, "tc"):
            kw = dict(dist=dist, want_ncomp=want_ncomp, full_sweep=fs)
            with tracs_b200.Database(s[:n_db]) as d:
                _same(d.append(s[n_db:], **kw), _one_shot(s, n_db, **kw))


def test_sequence_of_appends_is_the_grown_collection():
    L = 5000
    s = _pair(2700, L, seed=5, p_var=0.03)
    q = s[2400:]                      # never appended: queried at the end
    sizes = [1, 2, 70, 128, 300, 5, 900, 1, 600, 93]
    n0, results = 300, []
    with tracs_b200.Database(s[:n0]) as d:
        held = [d.info()["bytes_held"]]
        n = n0
        for m in sizes:
            got = d.append(s[n:n + m], dist=IMAX)
            _same(got, _one_shot(s[:n + m], n, dist=IMAX))
            results.append(got)
            n += m
            held.append(d.info()["bytes_held"])
        assert n == 2400 and d.n == n
        assert len(set(held)) >= 4
        fresh = tracs_b200.Database(s[:n])
        for k in ("n", "n_variable_sites"):
            assert d.info()[k] == fresh.info()[k], k
        got = d.query(q, dist=40)
        words = tracs_b200.last_stats()["n_words"]
        want = fresh.query(q, dist=40)
        assert tracs_b200.last_stats()["n_words"] == words
        fresh.close()
    _same(got, want)
    _same(got, tracs_b200.pairsnp_matrix(np.concatenate([q, s[:n]]), i_end=len(q), j_start=len(q), dist=40))
    first = tracs_b200.pairsnp_matrix(s[:n0], dist=IMAX)
    full = tracs_b200.pairsnp_matrix(s[:n], dist=IMAX)
    rows = np.concatenate([first["rows"]] + [r["rows"] for r in results])
    cols = np.concatenate([first["cols"]] + [r["cols"] for r in results])
    order = np.lexsort((cols, rows))
    for k in ("rows", "cols", "dist", "ncomp"):
        assert np.array_equal(np.concatenate([first[k]] + [r[k] for r in results])[order], full[k]), k


def _built_new_sites_batches(n_db=400, L=3000, n_batches=150, seed=17):
    """A database with many invariant sites (some with N or a code containing the base), then small batches of samples that
    each make a few of them variable (a different base, a disjoint 2-base code), or touch them without making them variable
    (a code containing the base, N)."""
    rng = np.random.default_rng(seed)
    ref = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, L)]
    db = ref[None, :].repeat(n_db, 0).copy()
    var = rng.choice(L, 100, replace=False)
    db[rng.integers(0, n_db, 300), var[rng.integers(0, 100, 300)]] = ord("T")
    inv = rng.permutation(np.setdiff1d(np.arange(L), var))
    db[5, inv[:40]] = ord("N")
    code_with = {ord("A"): "R", ord("C"): "M", ord("G"): "S", ord("T"): "W"}
    disjoint = {ord("A"): "Y", ord("C"): "R", ord("G"): "W", ord("T"): "S"}
    batches, k = [], 40
    for b in range(n_batches):
        m = 1 + b % 3
        x = db[rng.integers(0, n_db, m)].copy()
        for r in range(m):
            for _ in range(rng.integers(0, 3)):  # newly variable
                s_ = inv[k]
                k += 1
                x[r, s_] = ord("C") if ref[s_] != ord("C") else ord("G")
            if rng.random() < 0.3:
                x[r, inv[k]] = ord(disjoint[ref[inv[k]]])
                k += 1
            t = inv[rng.integers(40, 2000)]
            x[r, t] = ord(code_with[ref[t]]) if rng.random() < 0.5 else ord("N")
        batches.append(x)
    return db, batches


def test_many_small_appends_that_make_new_sites():
    db, batches = _built_new_sites_batches()
    alln = np.concatenate([db] + batches)
    n = db.shape[0]
    tracs_b200.pairsnp_matrix(db, dist=IMAX)
    v_prev = tracs_b200.last_stats()["n_variable_sites"]
    grew = 0
    with tracs_b200.Database(db) as d:
        for b in batches:
            m = b.shape[0]
            got = d.append(b, dist=IMAX)
            want = _one_shot(alln[:n + m], n, dist=IMAX)
            v = tracs_b200.last_stats()["n_variable_sites"]
            _same(got, want)
            assert d.info()["new_sites"] == v - v_prev and d.info()["n_variable_sites"] == v
            grew += v > v_prev
            v_prev = v
            n += m
        q = alln[:5]
        got = d.query(q, dist=IMAX)
        words = tracs_b200.last_stats()["n_words"]
    assert grew > 50
    with tracs_b200.Database(alln) as fresh:
        want = fresh.query(q, dist=IMAX)
        assert tracs_b200.last_stats()["n_words"] == words
    _same(got, want)


def test_input_forms_and_open_paths():
    import torch
    n_db, L = 600, 9000
    s = _pair(n_db + 4 * 70, L, seed=11)
    pitch = (L + 31) // 32 * 32
    nib, p4 = tracs_b200.pack_nibbles(s)

    def dev_ascii(a):
        t = torch.full((a.shape[0], pitch), ord("N"), dtype=torch.uint8)
        t[:, :L] = torch.from_numpy(a)
        return t.cuda()

    ddb, ddb4 = dev_ascii(s[:n_db]), torch.from_numpy(nib[:n_db]).cuda()
    before = ddb4.clone()
    dbs = [tracs_b200.Database(s[:n_db]), tracs_b200.Database(nib[:n_db], packed=True, L=L),
           tracs_b200.Database.from_device(ddb.data_ptr(), n_db, L, pitch), tracs_b200.Database.from_device(ddb4.data_ptr(), n_db, L, p4, packed=True)]
    for d in dbs:
        n = n_db
        for form in range(4):
            b = slice(n, n + 70)
            if form == 0:
                got = d.append(s[b], dist=30)
            elif form == 1:
                got = d.append(nib[b], dist=30, packed=True, L=L)
            elif form == 2:
                t = dev_ascii(s[b])
                got = d.append_device(t.data_ptr(), 70, pitch, dist=30)
            else:
                t = torch.from_numpy(nib[b]).cuda()
                got = d.append_device(t.data_ptr(), 70, p4, dist=30, packed=True)
                del t  # the rows were copied: the buffer is not kept
                torch.cuda.synchronize()
            _same(got, _one_shot(s[:n + 70], n, dist=30))
            n += 70
        _same(d.query(s[:40], dist=30), _one_shot(np.concatenate([s[:40], s[:n]]), 40, i_end=40, dist=30))
        d.close()
    assert torch.equal(ddb4, before)


def test_early_extraction_and_n_plane_paths(monkeypatch):
    import torch
    n_db, L = 1100, 70000
    sizes = [60, 300, 5]  # the first append and the second grow the N buffers; rows of a sparse N-plane are copied
    n_all = n_db + sum(sizes) + 40
    p4 = (L + 31) // 32 * 16
    buf = torch.empty(n_all * p4, dtype=torch.uint8, device="cuda")
    tracs_b200.synth_device(buf.data_ptr(), n_all, L, p4, seed=3, p_var=0.01, n_clusters=20, mu=5.0, p_N=1e-3, gaps=2, packed=True)
    host = buf.view(n_all, p4).cpu().numpy()
    for env in ({}, {"TRACS_NBLOCKS": "dense"}, {"TRACS_NPLANE": "always"}, {"TRACS_NPLANE": "sparse"}, {"TRACS_PAIRS": "sparse"},
                {"TRACS_PAIRS": "dense"}):
        for k in ("TRACS_NBLOCKS", "TRACS_NPLANE", "TRACS_PAIRS"):
            monkeypatch.delenv(k, raising=False)
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        with tracs_b200.Database.from_device(buf.data_ptr(), n_db, L, p4, packed=True) as d:
            assert tracs_b200.last_stats()["n_early_sites"] > 0
            n = n_db
            for i, m in enumerate(sizes):
                want = tracs_b200.pairsnp_packed(buf.data_ptr(), n + m, L, p4, j_start=n, dist=20)
                if i % 2:
                    got = d.append(host[n:n + m], packed=True, L=L, dist=20)
                else:
                    got = d.append_device(buf.data_ptr() + n * p4, m, p4, packed=True, dist=20)
                _same(got, want)
                n += m
            nq = n_all - n
            # the query rows sit right after the collection in the buffer: the two-file call needs them in front
            qbuf = torch.cat([buf[n * p4:], buf[:n * p4]])
            want = tracs_b200.pairsnp_packed(qbuf.data_ptr(), n_all, L, p4, i_end=nq, j_start=nq, dist=20)
            _same(d.query_device(buf.data_ptr() + n * p4, nq, p4, packed=True, dist=20), want)


def test_likelihood_columns():
    n_db, L = 900, 6000
    s = _pair(n_db + 4300 + 200, L, seed=23, p_amb=0.0)
    days = (np.arange(s.shape[0]) * 13 % 200).astype(np.int32)
    for dist in (20, 200):
        with tracs_b200.Database(s[:n_db]) as d:
            n = n_db
            for m in (200, 4300):
                got = d.append(s[n:n + m], dist=dist, days=days[:n + m])
                assert got["p0_log"] is not None
                _same(got, _one_shot(s[:n + m], n, dist=dist, days=days[:n + m]))
                n += m
            with pytest.raises(ValueError, match="days must hold"):
                d.append(s[:3], days=days[:n])


def test_from_fasta_then_append_with_names(oracle_mod):
    qp, dbp = os.path.join(GOLD, "query.fasta"), os.path.join(GOLD, "db.fasta.gz")
    dbs, dbn = tracs_b200.read_fasta(dbp)
    qs, qn = tracs_b200.read_fasta(qp)
    with tracs_b200.Database.from_fasta(dbp, n_threads=2) as d:
        with pytest.raises(ValueError, match="one name per appended sample"):
            d.append(qs)
        assert d.n == len(dbn)
        got = d.append(qs, names=qn)
        assert d.names == dbn + qn and d.n == len(dbn) + len(qn)
    s = np.concatenate([dbs, qs])
    _same(got, _one_shot(s, len(dbn), dist=IMAX))
    r, c, dd, _, nn = oracle_mod.pairsnp_ascii(s, i_end=len(s), j_start=len(dbn), dist=IMAX, n_threads=8)
    assert got["rows"].tolist() == r.tolist() and got["cols"].tolist() == c.tolist()
    assert got["dist"].tolist() == dd.tolist() and got["ncomp"].tolist() == nn.tolist()


def test_borrowed_buffer_is_never_written():
    import torch
    n_db, L = 800, 20000
    p4 = (L + 31) // 32 * 16
    buf = torch.empty(n_db * p4, dtype=torch.uint8, device="cuda")
    tracs_b200.synth_device(buf.data_ptr(), n_db, L, p4, seed=8, p_var=0.02, n_clusters=10, mu=4.0, packed=True)
    before = buf.clone()
    s = _pair(700, L, seed=9)
    with tracs_b200.Database.from_device(buf.data_ptr(), n_db, L, p4, packed=True) as d:
        for k, dist in enumerate((5, IMAX, 5)):
            d.append(s[200 * k:200 * (k + 1)], dist=dist)
            d.query(s[600:], dist=dist)
        d.append(s[690:], dist=IMAX, full_sweep=True)
        assert d.n == n_db + 610
    assert torch.equal(buf, before)


def test_bad_pitch_is_refused():
    s = _pair(40, 100, seed=1)
    with tracs_b200.Database(s[:30]) as d:
        with pytest.raises(RuntimeError, match=r"database append: pitch \(99\) must be >= L"):
            tracs_b200.api._lib.check(tracs_b200.api._lib.lib().tracs_db_append_host(
                tracs_b200.api.C.c_void_p(d._h), s.ctypes.data, 2, 99, None, tracs_b200.api.C.byref(tracs_b200.api.Edges())))
        with pytest.raises(RuntimeError, match="database append: pitch"):
            d.append_device(0, 2, 40, packed=True)
        assert d.info()["n"] == 30


@pytest.mark.parametrize("left_mb", [400, 40])
def test_append_that_does_not_fit_fails_with_size_and_leaves_the_database(left_mb):
    # 400 MB left: the N buffers grow (~0.3 GB), the bit-planes (~0.6 GB) do not fit; 40 MB left: the growth does not fit
    import torch
    n_db, L = 2000, 200_000
    db = _pair(n_db, L, seed=12, p_var=0.001, p_amb=0.0)
    rng = np.random.default_rng(1)
    b = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, (1000, L))]  # unrelated: most sites become variable
    nib_b, p4 = tracs_b200.pack_nibbles(b)
    db_b = torch.from_numpy(nib_b).cuda()
    with tracs_b200.Database(db) as d:
        info0 = d.info()
        small = d.query(db[:3], dist=5)
        tracs_b200.api._lib.lib().tracs_trim()
        torch.cuda.empty_cache()
        free, _ = torch.cuda.mem_get_info()
        hog = torch.empty(free - (left_mb << 20), dtype=torch.uint8, device="cuda")
        try:
            with pytest.raises(RuntimeError, match=r"database append: .* take \d+\.\d GB and do not fit in device memory next to the database"):
                d.append_device(db_b.data_ptr(), 1000, p4, dist=20, packed=True)
        finally:
            del hog
            torch.cuda.empty_cache()
        assert d.n == n_db
        for k in ("n", "n_variable_sites"):
            assert d.info()[k] == info0[k], k
        _same(d.query(db[:3], dist=5), small)
        _same(d.query(b[:50], dist=20), _one_shot(np.concatenate([b[:50], db]), 50, i_end=50, dist=20))
        got = d.append(b[:30], dist=20)
    _same(got, _one_shot(np.concatenate([db, b[:30]]), n_db, dist=20))


def test_sigint_during_an_append_leaves_the_database_unchanged():
    code = r'''
import os, signal, sys, threading, time, torch
import numpy as np
sys.path.insert(0, %r)
import tracs_b200
n_db, m, L = 60000, 16384, 40000
p4 = L // 2
n_all = n_db + m + 300
buf = torch.empty(n_all * p4, dtype=torch.uint8, device="cuda")
tracs_b200.synth_device(buf.data_ptr(), n_all, L, p4, seed=9, p_var=1.0, n_clusters=n_all, mu=0.0, p_N=0.0, gc=0.5, gaps=0, packed=True)
d = tracs_b200.Database.from_device(buf.data_ptr(), n_db, L, p4, packed=True)
d.query_device(buf.data_ptr() + n_db * p4, 64, p4, dist=10, packed=True, full_sweep=True)   # warm-up
t0 = time.perf_counter()
d.query_device(buf.data_ptr() + n_db * p4, m, p4, dist=10, packed=True, full_sweep=True)  # about the append's work
t_full = time.perf_counter() - t0
info0 = d.info()
threading.Timer(t_full / 4, lambda: os.kill(os.getpid(), signal.SIGINT)).start()
try:
    d.append_device(buf.data_ptr() + n_db * p4, m, p4, dist=10, packed=True, full_sweep=True)
    print("NOT-INTERRUPTED")
except KeyboardInterrupt as ex:
    print("INTERRUPTED", str(ex))
assert signal.getsignal(signal.SIGINT) is signal.default_int_handler
assert d.n == n_db and all(d.info()[k] == info0[k] for k in ("n", "n_variable_sites")), d.info()
same = lambda a, b: all(np.array_equal(a[k], b[k]) for k in ("rows", "cols", "dist", "ncomp"))
q0 = n_all - 300
qbuf = torch.cat([buf[q0 * p4:], buf[:n_db * p4]])
a = d.query_device(buf.data_ptr() + q0 * p4, 300, p4, dist=500, packed=True)
assert same(a, tracs_b200.pairsnp_packed(qbuf.data_ptr(), 300 + n_db, L, p4, i_end=300, j_start=300, dist=500))
a = d.append_device(buf.data_ptr() + n_db * p4, 300, p4, dist=500, packed=True)
assert same(a, tracs_b200.pairsnp_packed(buf.data_ptr(), n_db + 300, L, p4, j_start=n_db, dist=500))
print("AFTER", len(a["rows"]), d.n)
''' % ROOT
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600)
    assert "INTERRUPTED Interrupted by user!" in out.stdout and "AFTER" in out.stdout, out.stdout + out.stderr


@pytest.mark.parametrize("meta", [False, True])
def test_command_line_append(tmp_path, meta):
    s = _pair(330, 3000, seed=77)
    sdb, sq1, sq2, comb = tmp_path / "sdb.fasta", tmp_path / "sq1.fasta", tmp_path / "sq2.fasta", tmp_path / "comb.fasta"
    parts = ((sdb, s[:260], "d"), (sq1, s[260:290], "a"), (sq2, s[290:], "b"))
    for path, rows, tag in parts:
        path.write_text("".join(">%s%d\n%s\n" % (tag, i, r.tobytes().decode()) for i, r in enumerate(rows)))
    comb.write_text(sdb.read_text() + sq1.read_text() + sq2.read_text())
    opts = []
    if meta:
        dates = tmp_path / "dates.csv"
        names = ["d%d" % i for i in range(260)] + ["a%d" % i for i in range(30)] + ["b%d" % i for i in range(40)]
        dates.write_text("sample,date\n" + "".join("%s,2020-%02d-%02d\n" % (nm, 1 + i % 12, 1 + i * 7 % 28) for i, nm in enumerate(names)))
        opts = ["--meta", str(dates)]
    a, b = str(tmp_path / "append.csv"), str(tmp_path / "distance.csv")
    subprocess.run([sys.executable, "-m", "tracs_b200.query", "--db", str(sdb), "--msa", str(sq1), str(sq2), "--append", "-o", a, "-D", "25"] + opts,
                   cwd=ROOT, check=True)
    subprocess.run([sys.executable, "-m", "tracs_b200.distance", "--msa", str(comb), "-o", b, "-D", "25"] + opts, cwd=ROOT, check=True)
    got = list(csv.reader(io.StringIO(open(a).read())))
    want = list(csv.reader(io.StringIO(open(b).read())))
    assert got[0] == want[0]
    for tag, label in (("a", "sq1"), ("b", "sq2")):
        g = [r[:-1] for r in got[1:] if r[-1] == label]
        w = [r[:-1] for r in want[1:] if r[1].startswith(tag)]
        assert g == w and len(g) > 0, label
    assert len(got) == sum(1 for r in want[1:] if r[1][0] in "ab") + 1
