"""CPU: the C-ABI library loads, exports every symbol include/tracs_b200.h declares, fails loudly
without a GPU, and its host-only entry points (FASTA loader, lprob_k_given_N, calculate_posteriors,
shard dealing) match the oracle / golden fixtures."""
import ctypes as C
import json
import os
import re

import numpy as np
import pytest
from scipy.special import gammaln

import tracs_b200
from tracs_b200 import _lib, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")
G = json.load(open(os.path.join(GOLD, "golden.json")))


def test_exports_match_header():
    hdr = open(os.path.join(ROOT, "include", "tracs_b200.h")).read()
    declared = set(re.findall(r"\b(tracs_[a-z0-9_]+)\s*\(", hdr, flags=re.I))
    declared = {d for d in declared if not d.endswith("_t")}
    assert len(declared) >= 20
    lib = C.CDLL(_lib.LIB_PATH)
    for sym in sorted(declared):
        assert hasattr(lib, sym), "missing export: " + sym
    assert declared == set(_lib.SYMBOLS), declared ^ set(_lib.SYMBOLS)


def test_struct_layouts_match_c(tmp_path):
    """sizeof / offsetof of every struct in include/tracs_b200.h as gcc lays them out == the ctypes mirrors."""
    import subprocess
    structs = {"tracs_edges_t": _lib.Edges, "tracs_stats_t": _lib.Stats, "tracs_opts_t": _lib.Opts, "tracs_synth_t": _lib.Synth}
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "tracs_b200.h"', 'int main(void) {']
    for cname, cls in structs.items():
        lines.append('printf("%s %%zu\\n", sizeof(%s));' % (cname, cname))
        for f, _ in cls._fields_:
            lines.append('printf("%s.%s %%zu\\n", offsetof(%s, %s));' % (cname, f, cname, f))
    lines.append("return 0; }")
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = dict(l.split() for l in subprocess.check_output([str(exe)]).decode().splitlines())
    for cname, cls in structs.items():
        assert int(got[cname]) == C.sizeof(cls), cname
        for f, _ in cls._fields_:
            assert int(got["%s.%s" % (cname, f)]) == getattr(cls, f).offset, (cname, f)


def test_no_gpu_fails_loudly():
    if _lib.lib().tracs_device_count() > 0:
        pytest.skip("GPU present")
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        tracs_b200.trans_dist([1], [0.1], 29.9, 73.0, 0.01)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        tracs_b200.pairsnp_matrix(np.full((2, 4), 65, np.uint8))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        tracs_b200.pairsnp(fasta=[os.path.join(GOLD, "kat.fasta")], n_threads=1, dist=5, filter=False)


def test_product_does_not_import_oracle():
    import subprocess, sys
    code = "import sys; import tracs_b200, tracs_b200.distance, tracs_b200.multi; tracs_b200.install_dropin(); " \
           "assert not [m for m in sys.modules if m.startswith('oracle')], 'oracle imported by product'"
    subprocess.check_call([sys.executable, "-c", code], cwd=ROOT)
    for dirpath, _, files in os.walk(os.path.join(ROOT, "tracs_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".cpp")):
                src = open(os.path.join(dirpath, f)).read()
                assert "liboracle" not in src and "from oracle" not in src and "import oracle" not in src, f


def test_dropin_module_surface():
    T = tracs_b200.install_dropin()
    for name in ("pairsnp", "trans_dist", "lprob_k_given_N", "calculate_posteriors"):
        assert callable(getattr(T, name))
    # keyword names of src/python_bindings.cpp:12-25
    import inspect
    assert list(inspect.signature(T.pairsnp).parameters) == ["fasta", "n_threads", "dist", "filter"]
    assert list(inspect.signature(T.trans_dist).parameters) == ["snpdiff", "datediff", "lamb", "beta", "threshold_Ek"]
    assert list(inspect.signature(T.lprob_k_given_N).parameters) == ["N", "k", "delta", "lamb", "beta", "lgamma"]
    assert list(inspect.signature(T.calculate_posteriors).parameters) == ["counts", "alphas", "keep", "threshold"]


def test_lprob_k_given_N_kat_and_golden():
    lp, lhs = tracs_b200.lprob_k_given_N(7, 4, 0.16963, 3, 52, gammaln(range(20)))  # reference tests/test_llk.py:21-29
    assert abs(lp + 17.9565184209608) < 1e-6 and abs(lhs - 12.0861694243766) < 1e-6
    for c in G["lprob_k_given_N"]:
        N, k, delta, lamb, beta = c["args"]
        assert np.allclose(tracs_b200.lprob_k_given_N(int(N), int(k), delta, lamb, beta, gammaln(range(40))), c["out"], rtol=1e-12)
    with pytest.raises(IndexError):
        tracs_b200.lprob_k_given_N(7, 4, 0.1, 3, 52, gammaln(range(5)))


def test_calculate_posteriors_golden():
    for c in G["calculate_posteriors"]:
        out = tracs_b200.calculate_posteriors(np.array(c["counts"]), c["alphas"], c["keep"], c["threshold"])
        assert out.shape == np.array(c["counts"]).shape
        assert np.allclose(out, c["out"], rtol=1e-14, atol=0)


@pytest.mark.parametrize("name", ["aln0.fasta", "aln1.fasta.gz", "aln2.fasta", "aln3.fasta.gz", "aln4.fasta", "query.fasta", "db.fasta.gz"])
def test_fasta_loader_golden(oracle_mod, name):
    a, names = tracs_b200.read_fasta(os.path.join(GOLD, name))
    exp = oracle_mod.pairsnp([os.path.join(GOLD, name)], dist=-1)
    assert names == exp[3]
    m = oracle_mod.masks_of(a)
    assert m.shape[0] == len(names)


def test_fasta_loader_record_semantics(oracle_mod, tmp_path):
    # kseq semantics (reference src/kseq.h:170-208): junk before the first header, names end at
    # whitespace, '>'/'@'/'+' end a sequence anywhere, blank lines / CRLF / spaces dropped, FASTQ blocks.
    cases = {
        "plain": b">a desc here\nACGT\nAC\n>b\nAC-NNT\n",
        "junk_crlf": b"junk line\r\n>a\tx\r\nAC GT\r\n\r\nAC\r\n>b\r\nACGTAC\r\n",
        "no_trailing_newline": b">a\nACGT\n>b\nACGA",
        "fastq": b"@r1 d\nACGT\n+\nIIII\n@r2\nACGA\n+r2\nII!I\n",
        "fastq_multi": b"@r1\nAC\nGT\n+\nII\nII\n@r2\nACGA\n+\nIIII\n",
        "gt_inside": b">a\nAC>b\nGT\n",
        "empty_seq": b">a\n>b\n",
        "single": b">only\nACGTNNNN",
        "lower_iupac": b">a\nacgtmrwsykvhdbn-x?.\n>b\nACGTMRWSYKVHDBN-X?.\n",
    }
    for tag, data in cases.items():
        p = str(tmp_path / (tag + ".fa"))
        open(p, "wb").write(data)
        a, names = tracs_b200.read_fasta(p)
        exp = oracle_mod.pairsnp([p], dist=2147483647)
        assert names == exp[3], tag
        if len(names) >= 2 and a.shape[1] > 0:
            got = oracle_mod.pairsnp_ascii(a, dist=2147483647)
            assert got[2].tolist() == exp[2] and got[4].tolist() == exp[5], tag
    p = str(tmp_path / "ragged.fa")
    open(p, "wb").write(b">a\nACGT\n>b\nACG\n")
    with pytest.raises(RuntimeError, match="variable sequence lengths"):
        tracs_b200.read_fasta(p)
    p = str(tmp_path / "trunc.fq")
    open(p, "wb").write(b"@r1\nACGT\n+\nII")
    with pytest.raises(RuntimeError, match="Error reading FASTA"):
        tracs_b200.read_fasta(p)
    with pytest.raises(RuntimeError, match="Error reading FASTA"):
        tracs_b200.read_fasta(str(tmp_path / "does_not_exist.fa"))


def test_fasta_loader_live_reference_errors(oracle_mod, tmp_path):
    """Ragged input: the reference's error, from the loader, the oracle and, where a local build of the reference exists
    in oracle/_ref/ (not part of the repository), the unmodified reference module."""
    from oracle import refmod
    p = str(tmp_path / "ragged.fa")
    open(p, "wb").write(b">a\nACGT\n>b\nACG\n")
    calls = [lambda: tracs_b200.read_fasta(p), lambda: oracle_mod.pairsnp([p], dist=1)]
    if refmod.available():
        calls.append(lambda: refmod.load()[0].pairsnp(fasta=[p], n_threads=1, dist=1, filter=False))
    for call in calls:
        with pytest.raises(RuntimeError, match="variable sequence lengths"):
            call()


def test_fasta_loader_large_roundtrip(tmp_path):
    s = synth.generate(50, 30011, p_var=0.02, seed=8, lowercase=0.05)
    for gz, width in ((False, 0), (True, 61)):
        p = str(tmp_path / ("big.fa" + (".gz" if gz else "")))
        synth.write_fasta(p, s, width=width, descriptions=True)
        a, names = tracs_b200.read_fasta(p)
        assert names == ["s%d" % i for i in range(50)] and np.array_equal(a, s)


def _read_both(p):
    """(sequential result or error text, 4-thread result or error text) of the loader on one file."""
    out = []
    for nt in (1, 4):
        try:
            a, names = tracs_b200.read_fasta(p, n_threads=nt)
            out.append((names, a.shape, a.tobytes()))
        except RuntimeError as e:
            out.append(str(e))
    return out


def test_fasta_loader_threads_equal_sequential(tmp_path, monkeypatch):
    # the multi-threaded reader of plain files must be indistinguishable from the sequential state machine:
    # same names, order, bases -- and the same error -- also where it has to hand the file back
    monkeypatch.setenv("TRACS_FASTA_PAR_MIN", "0")
    monkeypatch.setenv("TRACS_FASTA_SINK_CHECK", "1")   # the rows streamed to a sink while parsing == the finished matrix
    cases = {
        "plain": b">a desc here\nACGT\nAC\n>b\nAC-NNT\n>c\nACGTAC\n",
        "crlf": b">a\tx\r\nAC GT\r\n\r\nAC\r\n>b\r\nACGTAC\r\n>c x\r\nACGTAC",
        "junk_first": b"junk line\n>a\nACGT\n>b\nACGA\n",
        "gt_in_header": b">a > b >c\nACGT\n>b>x\nACGA\n>c\nAAAA\n",
        "gt_inside_seq": b">a\nACGT\n>b\nAC>x\nGT\n>c\nACGT\n",
        "at_inside_seq": b">a\nACGT\n>b\nAC@x\nGT\n>c\nACGT\n",
        "plus_inside_seq": b">a\nACGT\n>b\nACGT\n+\nIIII\n>c\nACGT\n",
        "fastq": b"@r1 d\nACGT\n+\nIIII\n@r2\nACGA\n+r2\nII!I\n",
        "fastq_after_fasta": b">a\nACGT\n>b\nACGT\n@r\nACGA\n+\nIIII\n",
        "empty_seqs": b">a\n>b\n>c\n",
        "last_header_only": b">a\nACGT\n>b\nACGT\n>c",
        "last_gt_only": b">a\nACGT\n>b\nACGT\n>",
        "last_no_newline": b">a\nACGT\n>b\nACGT\n>c\nACGA",
        "ragged_middle": b">a\nACGT\n>b\nACG\n>c\nACGT\n",
        "ragged_last": b">a\nACGT\n>b\nACGT\n>c\nACG\n",
        "ragged_long": b">a\nACGT\n>b\nACGTACGTACGTACGTACGTACGTACGTACGTAAA\n>c\nACGT\n",
        "ragged_then_truncated_fastq": b">a\nACGT\n>b\nACG\n@c\nACGT\n+\nII",
        "truncated_fastq_tail": b">a\nACGT\n>b\nACGT\n@c\nACGT\n+\nII",
        "blank_lines": b">a\n\n\nAC\n\nGT\n\n>b\n\nACGT\n\n\n>c\nACGT\n\n",
        "long_lines": b"".join(b">s%d\n" % i + b"ACGTNacgtn-" * 37 + b"\n" + b"MRWSYKVHDB" * 11 + b"\n" for i in range(9)),
    }
    for tag, data in cases.items():
        p = str(tmp_path / (tag + ".fa"))
        open(p, "wb").write(data)
        seq, par = _read_both(p)
        assert seq == par, tag
    s = synth.generate(64, 30011, p_var=0.02, seed=9, lowercase=0.05)
    for width in (0, 61):
        p = str(tmp_path / ("big%d.fa" % width))
        synth.write_fasta(p, s, width=width, descriptions=True)
        a, names = tracs_b200.read_fasta(p, n_threads=8)
        assert names == ["s%d" % i for i in range(64)] and np.array_equal(a, s)
    # many ~32 MB sink chunks: 600 records x 200 kb through the parallel reader, and gzip through the sequential one
    s = synth.generate(600, 200_000, p_var=0.01, seed=10)
    for nm in ("chunks.fa", "chunks.fa.gz"):
        p = str(tmp_path / nm)
        synth.write_fasta(p, s if nm.endswith(".fa") else s[:120])
        a, names = tracs_b200.read_fasta(p, n_threads=8)
        assert np.array_equal(a, s[:len(a)]) and len(a) == (600 if nm.endswith(".fa") else 120)


def test_shard_dealing_covers_and_balances():
    for n_rb, world in ((1, 1), (7, 2), (79, 8), (782, 8), (5, 8), (16, 4)):
        parts = [tracs_b200.shard_rowblocks(n_rb, world, r) for r in range(world)]
        allrb = np.sort(np.concatenate(parts))
        assert allrb.tolist() == list(range(n_rb))
        # triangle work of row-block rb ~ (n_rb - rb) tiles; boustrophedon keeps shards within one round of each other
        work = [sum(n_rb - int(rb) for rb in p) for p in parts]
        if n_rb >= 4 * world:
            assert max(work) - min(work) <= 2 * world + n_rb % (2 * world) * world


def test_float_repr_matches_python():
    import math, random, struct
    L = _lib.lib()
    buf = C.create_string_buffer(64)

    def r(v):
        L.tracs_float_repr(v, buf)
        return buf.value.decode()

    for v in [0.0, -0.0, 1.0, 0.1, 1e-4, 1e-5, 1.5e-5, 1e15, 1e16, 1.5e16, 1e22, 0.002737907006988508, float("inf"), -float("inf"),
              5e-324, 1.7976931348623157e308, 100.0, 12345.678, 0.23794988406662973]:
        assert r(v) == repr(v)
    assert r(float("nan")) == "nan"
    random.seed(3)
    for _ in range(20000):
        v = struct.unpack("d", struct.pack("Q", random.getrandbits(64)))[0]
        if not math.isnan(v):
            assert r(v) == repr(v)
        w = random.random() * 10 ** random.randint(-8, 18)
        assert r(w) == repr(w)


def test_native_csv_writer_layout(tmp_path):
    # host-only: build an edge table by hand and check every quirk of tracs/distance.py:206-258
    e = _lib.Edges()
    n = 3
    rows = (C.c_uint64 * n)(0, 0, 1)
    cols = (C.c_uint64 * n)(1, 2, 2)
    dist = (C.c_uint64 * n)(0, 2, 1)
    filt = (C.c_uint64 * n)(0, 1, 1)
    ncomp = (C.c_uint64 * n)(9, 10, 9)
    import math
    lp = [math.log(0.25), math.log(0.5), math.log(0.125)]
    p0 = (C.c_double * n)(*lp)
    eK = (C.c_double * n)(2.5, 12.0, 4.0)
    dt = (C.c_double * n)(0.002737907006988508, 0.002737907006988508, 0.0)
    names = (C.c_char_p * 3)(b"seq1", b"seq2", b"seq3")
    e.n_edges, e.rows, e.cols, e.dist, e.filt, e.ncomp = n, rows, cols, dist, filt, ncomp
    e.p0_log, e.eK, e.datediff = p0, eK, dt
    out = str(tmp_path / "o.csv")
    w = C.c_size_t(0)
    L = _lib.lib()
    _lib.check(L.tracs_write_distance_csv(out.encode(), 0, C.byref(e), names, 3, b"kat", 1, 0, 1, 10.0, C.byref(w)))
    lines = open(out).read().splitlines()
    assert w.value == 2 and lines[0].startswith("sampleA,sampleB,date difference,SNP distance")
    assert lines[1] == "seq1,seq2,0.002737907006988508,0,%r,2.5,NA,9,kat" % math.exp(lp[0])  # NA: metadata, no filter
    assert lines[2] == "seq2,seq3,0.0,1,%r,4.0,NA,9,kat" % math.exp(lp[2])                   # eK = 12 > K = 10 dropped
    _lib.check(L.tracs_write_distance_csv(out.encode(), 1, C.byref(e), names, 3, b"k2", 0, 0, 0, 0.0, C.byref(w)))
    lines = open(out).read().splitlines()
    assert w.value == 3 and lines[3] == "seq1,seq2,NA,0,NA,NA,0,9,k2"             # no metadata: NA columns, filtered column = 0


def test_compiled_pybind_module_surface(tmp_path):
    """The compiled `TRACS` extension (tracs_b200/dropin_native/, pybind11 over the C ABI; INTEGRATION.md option B):
    same four names and keywords as src/python_bindings.cpp:12-25, host-side entries work without a GPU, device
    entries fail loudly; the reference's own tests/test_llk.py passes on it when staged."""
    import subprocess, sys
    from tracs_b200 import build
    path = build.build_pybind()
    d = os.path.dirname(path)
    code = ("import TRACS, inspect, numpy as np\n"
            "from scipy.special import gammaln\n"
            "assert TRACS.__file__.endswith('.so') and TRACS.__doc__ == 'Meta Transmission Clustering'\n"
            "assert sorted(n for n in dir(TRACS) if not n.startswith('_')) == ['calculate_posteriors', 'lprob_k_given_N', 'pairsnp', 'trans_dist']\n"
            "r = TRACS.lprob_k_given_N(N=7, k=4, delta=0.16963, lamb=3, beta=52, lgamma=gammaln(range(20)))\n"
            "assert abs(r[0] + 17.9565184209608) < 1e-6 and abs(r[1] - 12.0861694243766) < 1e-6\n"
            "try:\n    TRACS.lprob_k_given_N(7, 4, 0.1, 3, 52, [0.0] * 5)\n    raise SystemExit(2)\nexcept IndexError:\n    pass\n"
            "p = TRACS.calculate_posteriors(counts=np.array([[1., 2.], [0., 0.]]), alphas=[0.5, 0.2], keep=True, threshold=0.05)\n"
            "assert p.shape == (2, 2) and p.dtype == np.float64\n"
            "try:\n    TRACS.pairsnp(fasta=['a', 'b', 'c'], n_threads=1, dist=1, filter=False)\n    raise SystemExit(3)\n"
            "except RuntimeError as e:\n    assert 'Invalid number of fasta files' in str(e)\n")
    env = dict(os.environ, PYTHONPATH=d)
    subprocess.check_call([sys.executable, "-c", code], env=env, cwd=str(tmp_path))
    t = os.path.join(ROOT, "oracle", "_ref", "py", "ref_tests")
    if os.path.exists(os.path.join(t, "test_llk.py")):
        r = subprocess.run([sys.executable, "-m", "pytest", "-q", "-p", "no:cacheprovider", "--rootdir", t, os.path.join(t, "test_llk.py")],
                           env=env, cwd=str(tmp_path), capture_output=True, text=True)
        assert r.returncode == 0 and "1 passed" in r.stdout, r.stdout + r.stderr
