"""GPU: the dense all-pairs distance matrix (tracs_distance_matrix_*, k_sweep<true>, k_sweep_tc3<NP, true>) against the
CPU oracle and against the thresholded pair list, on both kernels, every input form and both shapes."""
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


def _square_from_edges(n, rows, cols, dist):
    m = np.zeros((n, n), np.int64)
    r, c = np.asarray(rows, np.int64), np.asarray(cols, np.int64)
    m[r, c] = np.asarray(dist, np.int64)
    m[c, r] = np.asarray(dist, np.int64)
    return m


def _oracle_square(oracle_mod, s):
    r, c, d, _, _ = oracle_mod.pairsnp_ascii(s, dist=IMAX, n_threads=8)
    return _square_from_edges(s.shape[0], r, c, d)


def _oracle_rect(oracle_mod, s, q):
    n = s.shape[0]
    r, c, d, _, _ = oracle_mod.pairsnp_ascii(s, i_end=q, j_start=q, dist=IMAX, n_threads=8)
    m = np.full((q, n - q), -1, np.int64)
    m[r.astype(np.int64), c.astype(np.int64) - q] = d
    return m


def _check_square(m, want):
    assert m.dtype == np.int32 and m.shape == want.shape
    assert (np.diag(m) == 0).all()
    assert (m == m.T).all()
    assert (m.astype(np.int64) == want).all(), np.argwhere(m != want)[:5]


@pytest.mark.parametrize("n,L", [(2, 1), (5, 31), (7, 32), (33, 33), (128, 1000), (129, 4097), (300, 20000), (257, 1023), (64, 5000),
                                 (3, 70000)])
def test_parity_with_oracle(oracle_mod, n, L):
    s = synth.generate(n, L, p_var=0.05, n_clusters=4, mu=3, p_N=0.02, p_amb=0.05, seed=n * 7 + L, lowercase=0.05, odd_chars=0.01,
                       three_base=True)
    _check_square(tracs_b200.distance_matrix(s), _oracle_square(oracle_mod, s))


def test_every_byte_value(oracle_mod):
    s = synth.generate(40, 4096, p_var=0.05, n_clusters=3, mu=3, p_N=0.01, seed=77)
    for c in range(4096):
        s[(c // 256 + c) % 40, c] = c % 256
    _check_square(tracs_b200.distance_matrix(s), _oracle_square(oracle_mod, s))
    r = np.random.default_rng(5).integers(0, 256, size=(20, 3001), dtype=np.uint8)
    _check_square(tracs_b200.distance_matrix(r), _oracle_square(oracle_mod, r))


@pytest.mark.parametrize("n", [1, 2, 127, 128, 129, 255, 256, 257, 511, 512, 513, 640, 641])
def test_tile_and_super_tile_edges(oracle_mod, n):
    # single-base codes (tensor cores allowed), N and gaps: super-tiles of 1-4 column blocks and partial blocks
    s = synth.generate(n, 3000, p_var=0.05, n_clusters=5, mu=4, p_N=0.01, seed=1000 + n)
    want = _oracle_square(oracle_mod, s)
    tc = tracs_b200.distance_matrix(s)
    assert tracs_b200.last_stats()["tc_sweep"] in (33, 34)  # <3> when no sample happens to hold an N at a variable site
    _check_square(tc, want)
    lop = tracs_b200.distance_matrix(s, full_sweep=True)
    assert tracs_b200.last_stats()["tc_sweep"] == 0
    _check_square(lop, want)


@pytest.mark.parametrize("p_N,code", [(0.01, 34), (0.0, 33)])
def test_kernel_selection(oracle_mod, p_N, code):
    s = synth.generate(300, 5000, p_var=0.05, n_clusters=4, mu=3, p_N=p_N, gaps=2 if p_N else 0, seed=21)
    want = _oracle_square(oracle_mod, s)
    m0 = tracs_b200.distance_matrix(s)
    st = tracs_b200.last_stats()
    assert st["tc_sweep"] == code
    assert st["n_pairs"] == 300 * 299 // 2 and st["n_edges"] == 0 and st["n_candidates"] == 0 and st["ms_sort"] == 0
    assert st["ms_ncomp"] == 0 and st["n_tiles"] > 0 and st["kernel_launches"] > 0 and st["d2h_bytes"] == 300 * 300 * 4
    m2 = tracs_b200.distance_matrix(s, full_sweep="tc")
    assert tracs_b200.last_stats()["tc_sweep"] == code
    m1 = tracs_b200.distance_matrix(s, full_sweep=True)
    assert tracs_b200.last_stats()["tc_sweep"] == 0
    assert (m0 == m1).all() and (m0 == m2).all()
    _check_square(m0, want)


def test_tensor_cores_required_refuses_partial_ambiguity():
    s = synth.generate(100, 2000, p_var=0.05, n_clusters=3, mu=3, p_amb=0.05, seed=3, three_base=True)
    with pytest.raises(RuntimeError, match="tensor-core sweep requested but the alignment has 2-/3-base IUPAC codes"):
        tracs_b200.distance_matrix(s, full_sweep="tc")
    tracs_b200.distance_matrix(s)  # variant 0 falls back to the LOP3/POPC kernel
    assert tracs_b200.last_stats()["tc_sweep"] == 0


@pytest.mark.parametrize("q", [1, 100, 128, 129, 300])
def test_query_x_db(oracle_mod, q):
    s = synth.generate(400, 6000, p_var=0.05, n_clusters=5, mu=3, p_N=0.01, seed=400 + q)
    full = tracs_b200.distance_matrix(s)
    for fs in (False, True):
        rect = tracs_b200.distance_matrix(s, n_query=q, full_sweep=fs)
        assert rect.shape == (q, 400 - q)
        assert (rect == full[:q, q:]).all()
        assert (rect.astype(np.int64) == _oracle_rect(oracle_mod, s, q)).all()


def test_input_forms_agree():
    import torch
    n, L = 700, 9000
    pitch = (L + 31) // 32 * 32
    pitch4 = max(16, (L + 31) // 32 * 16)
    a = torch.empty(n * pitch, dtype=torch.uint8, device="cuda")
    p = torch.empty(n * pitch4, dtype=torch.uint8, device="cuda")
    kw = dict(seed=5, p_var=0.05, n_clusters=6, mu=4, p_N=0.01)
    tracs_b200.synth_device(a.data_ptr(), n, L, pitch, **kw)
    tracs_b200.synth_device(p.data_ptr(), n, L, pitch4, packed=True, **kw)
    host = a.view(n, pitch)[:, :L].cpu().numpy()
    nib, _ = tracs_b200.pack_nibbles(host)
    outs = {"host_ascii": tracs_b200.distance_matrix(host), "host_packed": tracs_b200.distance_matrix(nib, packed=True, L=L)}
    for name, buf, pt, packed in (("dev_ascii", a, pitch, False), ("dev_packed", p, pitch4, True)):
        o = torch.empty((n, n), dtype=torch.int32, device="cuda")
        tracs_b200.distance_matrix_device(buf.data_ptr(), n, L, pt, o.data_ptr(), n, packed=packed)
        outs[name] = o.cpu().numpy()
    for k, v in outs.items():
        assert (v == outs["host_ascii"]).all(), k
    r = tracs_b200.pairsnp_matrix(host, dist=IMAX, want_ncomp=False)
    assert (outs["host_ascii"].astype(np.int64) == _square_from_edges(n, r["rows"], r["cols"], r["dist"])).all()


@pytest.mark.parametrize("q", [None, 200])
@pytest.mark.parametrize("fs", [False, True])
def test_padding_columns_untouched(q, fs):
    import torch
    n, L = 520, 7000
    s = synth.generate(n, L, p_var=0.05, n_clusters=4, mu=3, p_N=0.01, seed=99)
    want = tracs_b200.distance_matrix(s, n_query=q, full_sweep=fs)
    rows, cols = want.shape
    ld = cols + 37
    pitch = (L + 31) // 32 * 32
    dev = torch.full((n, pitch), ord("N"), dtype=torch.uint8)
    dev[:, :L] = torch.from_numpy(s)
    dev = dev.cuda()
    out = torch.full((rows, ld), -7, dtype=torch.int32, device="cuda")
    tracs_b200.distance_matrix_device(dev.data_ptr(), n, L, pitch, out.data_ptr(), ld, n_query=q, full_sweep=fs)
    o = out.cpu().numpy()
    assert (o[:, cols:] == -7).all()
    assert (o[:, :cols] == want).all()


@pytest.mark.parametrize("p_N,gaps", [(0.0, 0), (0.02, 2)])
def test_matches_the_pair_list_beyond_the_oracle(p_N, gaps):
    import torch
    n, L = 3000, 200_000
    pitch4 = (L + 31) // 32 * 16
    buf = torch.empty(n * pitch4, dtype=torch.uint8, device="cuda")
    tracs_b200.synth_device(buf.data_ptr(), n, L, pitch4, seed=31, p_var=1.0, n_clusters=30, mu=20.0, p_N=p_N, gaps=gaps, packed=True)
    for fs in ("tc", True):
        out = torch.empty((n, n), dtype=torch.int32, device="cuda")
        tracs_b200.distance_matrix_device(buf.data_ptr(), n, L, pitch4, out.data_ptr(), n, packed=True, full_sweep=fs)
        st = tracs_b200.last_stats()
        assert st["tc_sweep"] == (0 if fs is True else (34 if p_N else 33))
        e = tracs_b200.pairsnp_packed(buf.data_ptr(), n, L, pitch4, dist=IMAX, full_sweep=fs, want_ncomp=False)
        assert len(e["rows"]) == n * (n - 1) // 2
        m = out.cpu().numpy()
        assert (m.astype(np.int64) == _square_from_edges(n, e["rows"], e["cols"], e["dist"])).all()
        assert (np.diag(m) == 0).all()


def test_too_large_fails_cleanly_and_the_library_stays_usable():
    import ctypes as C
    from tracs_b200 import _lib, api
    n, L = 250_000, 64
    seqs = np.full((n, L), ord("A"), np.uint8)
    seqs[::7, 3] = ord("C")
    o, _ = api.make_opts()
    out = np.zeros(16, np.int32)  # never written: the call fails before any result exists
    rc = _lib.lib().tracs_distance_matrix_host(seqs.ctypes.data, n, L, L, C.byref(o), out.ctypes.data, n)
    msg = _lib.lib().tracs_last_error().decode()
    assert rc == 1 and "do not fit in device memory" in msg and "250.0 GB" in msg and "thresholded pair list" in msg, msg
    small = tracs_b200.distance_matrix(seqs[:300])
    assert small.shape == (300, 300) and small.max() == 1


def test_sigint_between_bands_unwinds_the_call():
    code = r'''
import os, signal, sys, threading, time, torch
sys.path.insert(0, %r)
import tracs_b200
n, L = 60000, 40000
pitch = L // 2
buf = torch.empty(n * pitch, dtype=torch.uint8, device="cuda")
out = torch.empty((n, n), dtype=torch.int32, device="cuda")
tracs_b200.synth_device(buf.data_ptr(), n, L, pitch, seed=9, p_var=1.0, n_clusters=n, mu=0.0, p_N=0.0, gc=0.5, gaps=0, packed=True)
tracs_b200.distance_matrix_device(buf.data_ptr(), 2000, L, pitch, out.data_ptr(), 2000, packed=True)   # warm-up
t0 = time.perf_counter()
tracs_b200.distance_matrix_device(buf.data_ptr(), n, L, pitch, out.data_ptr(), n, packed=True, full_sweep=True)
t_full = time.perf_counter() - t0
threading.Timer(min(0.15, t_full / 4), lambda: os.kill(os.getpid(), signal.SIGINT)).start()
t0 = time.perf_counter()
try:
    tracs_b200.distance_matrix_device(buf.data_ptr(), n, L, pitch, out.data_ptr(), n, packed=True, full_sweep=True)
    print("NOT-INTERRUPTED")
except KeyboardInterrupt as ex:
    print("INTERRUPTED", str(ex), "%%.3f %%.3f" %% (time.perf_counter() - t0, t_full))
assert signal.getsignal(signal.SIGINT) is signal.default_int_handler
tracs_b200.distance_matrix_device(buf.data_ptr(), 3000, L, pitch, out.data_ptr(), 3000, packed=True)   # usable afterwards
print("AFTER", int(out.view(-1)[:3000 * 3000].view(3000, 3000).diagonal().abs().sum()))
''' % ROOT
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300)
    assert "INTERRUPTED Interrupted by user!" in out.stdout and "AFTER 0" in out.stdout, out.stdout + out.stderr
    took, full = map(float, out.stdout.split("INTERRUPTED Interrupted by user!")[1].split()[:2])
    assert took < full, (took, full)


def _read_table(path, sep):
    lines = open(path).read().split("\n")
    assert lines[-1] == ""
    head = lines[0].split(sep)
    assert head[0] == ""
    rows = [ln.split(sep) for ln in lines[1:-1]]
    return head[1:], [r[0] for r in rows], np.array([[int(x) for x in r[1:]] for r in rows], np.int64).reshape(len(rows), len(head) - 1)


@pytest.mark.parametrize("files", [["aln0.fasta"], ["aln1.fasta.gz"], ["aln2.fasta"], ["aln3.fasta.gz"], ["aln4.fasta"],
                                   ["query.fasta", "db.fasta.gz"]])
def test_dists_command_line(oracle_mod, tmp_path, files):
    paths = [os.path.join(GOLD, f) for f in files]
    tsv, csv = str(tmp_path / "out.tsv"), str(tmp_path / "out.csv")
    args = [sys.executable, "-m", "tracs_b200.dists", "--msa", paths[0]] + (["--msa-db", paths[1]] if len(paths) > 1 else [])
    subprocess.run(args + ["-o", tsv, "-t", "3"], cwd=ROOT, check=True)
    subprocess.run(args + ["-o", csv, "--csv"], cwd=ROOT, check=True)
    assert open(csv).read() == open(tsv).read().replace("\t", ",")
    cols, rows, m = _read_table(tsv, "\t")
    r, c, d, names, _, _ = oracle_mod.pairsnp(fasta=paths, n_threads=2, dist=IMAX)
    n = len(names)
    full = _square_from_edges(n, r, c, d)
    if len(paths) == 1:
        assert rows == names and cols == names
        assert (m == full).all()
    else:
        nq = len(tracs_b200.read_fasta(paths[0])[1])
        assert rows == names[:nq] and cols == names[nq:]
        assert (m == full[:nq, nq:]).all()
