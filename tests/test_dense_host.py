"""CPU: the dense distance-matrix surface without a device -- the native text writer's exact bytes, every argument
error of tracs_distance_matrix_* (raised before any device call), the missing-device error of the Python entries and
the dists command line."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

import tracs_b200
from tracs_b200 import _lib, api

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
IMAX = 2147483647


def _expected_text(m, row_names, col_names, sep):
    lines = [sep.join([""] + list(col_names))]
    for name, row in zip(row_names, np.asarray(m)):
        lines.append(sep.join([name] + [str(int(v)) for v in row]))
    return ("\n".join(lines) + "\n").encode()


@pytest.mark.parametrize("sep", ["\t", ","])
def test_writer_bytes_square_and_rectangle(tmp_path, sep):
    sq = np.array([[0, 3, 12], [3, 0, 7], [12, 7, 0]], np.int32)
    names = ["s1", "sample_two", "x"]
    p = tmp_path / "sq.txt"
    tracs_b200.write_distance_matrix(p, sq, names, names, sep=sep)
    want = (sep + "s1" + sep + "sample_two" + sep + "x\n" + "s1" + sep + "0" + sep + "3" + sep + "12\n" +
            "sample_two" + sep + "3" + sep + "0" + sep + "7\n" + "x" + sep + "12" + sep + "7" + sep + "0\n").encode()
    assert p.read_bytes() == want
    # a rectangle with other row and column names, read through a row-strided view (ld > cols) of a larger buffer
    big = np.full((2, 7), -99, np.int32)
    big[:, :3] = [[5, 0, 2147483647], [1, -4, 10]]
    rect = big[:, :3]
    assert rect.strides[0] == 7 * 4
    tracs_b200.write_distance_matrix(p, rect, ["q0", "q1"], ["d0", "d1", "d2"], sep=sep)
    assert p.read_bytes() == _expected_text(rect, ["q0", "q1"], ["d0", "d1", "d2"], sep)
    # the C entry with an explicit ld
    rn = (C.c_char_p * 2)(b"q0", b"q1")
    cn = (C.c_char_p * 3)(b"d0", b"d1", b"d2")
    _lib.check(_lib.lib().tracs_write_distance_matrix(os.fsencode(str(p)), big.ctypes.data, 2, 3, 7, rn, cn, sep.encode()))
    assert p.read_bytes() == _expected_text(rect, ["q0", "q1"], ["d0", "d1", "d2"], sep)


def test_writer_output_does_not_depend_on_threads(tmp_path):
    # enough rows for many formatting ranges (about 4 MB of text each), so that 8 threads all take part
    rng = np.random.default_rng(3)
    m = rng.integers(-5, 2_000_000, size=(3001, 1000), dtype=np.int32)
    rows = ["r%d" % i for i in range(m.shape[0])]
    cols = ["c%d" % j for j in range(m.shape[1])]
    out = {}
    for t in (1, 8):
        p = tmp_path / ("t%d.tsv" % t)
        tracs_b200.write_distance_matrix(p, m, rows, cols, n_threads=t)
        out[t] = p.read_bytes()
    assert out[1] == out[8]
    assert out[1] == _expected_text(m, rows, cols, "\t")


def test_writer_argument_errors(tmp_path):
    m = np.zeros((2, 2), np.int32)
    with pytest.raises(RuntimeError, match="sep"):
        tracs_b200.write_distance_matrix(tmp_path / "x", m, ["a", "b"], ["a", "b"], sep=";")
    with pytest.raises(ValueError, match="one name per row"):
        tracs_b200.write_distance_matrix(tmp_path / "x", m, ["a"], ["a", "b"])
    names = (C.c_char_p * 2)(b"a", b"b")
    with pytest.raises(RuntimeError, match="ld"):
        _lib.check(_lib.lib().tracs_write_distance_matrix(os.fsencode(str(tmp_path / "x")), m.ctypes.data, 2, 2, 1, names, names, b"\t"))


def _opts(**kw):
    o, keep = api.make_opts(**kw)
    return o, keep


def _host_call(seqs, o, out, ld, L=None, pitch=None):
    n = seqs.shape[0]
    L = seqs.shape[1] if L is None else L
    pitch = seqs.shape[1] if pitch is None else pitch
    return _lib.lib().tracs_distance_matrix_host(seqs.ctypes.data, n, L, pitch, C.byref(o), out.ctypes.data if out is not None else None, ld)


@pytest.mark.parametrize("kw,field", [
    (dict(dist=20), "opts->dist"),
    (dict(filter=True), "opts->filter"),
    (dict(days=np.zeros(10, np.int32)), "opts->want_trans"),
    (dict(keep_on_device=True), "opts->keep_on_device"),
    (dict(shard_world=2), "opts->shard_world"),
    (dict(i_end=5), "opts->i_end"),               # neither square nor a rectangle
    (dict(i_end=5, j_start=3), "opts->i_end"),    # j_start < i_end
    (dict(i_end=5, j_start=10), "opts->i_end"),   # j_start >= n
    (dict(i_end=11), "opts->i_end"),              # i_end > n
    (dict(j_start=4), "opts->i_end"),             # i_end = 0 means n, and j_start < n
])
def test_validation_errors_without_a_device(kw, field):
    seqs = np.full((10, 64), ord("A"), np.uint8)
    out = np.zeros((10, 10), np.int32)
    o, keep = _opts(**kw)
    rc = _host_call(seqs, o, out, 10)
    assert rc == 1
    msg = _lib.lib().tracs_last_error().decode()
    assert field in msg and "no CPU fallback" not in msg, msg
    # the device entry checks the same things first
    rc = _lib.lib().tracs_distance_matrix_device(C.c_void_p(1 << 20), 10, 64, 64, C.byref(o), C.c_void_p(1 << 21), 10)
    assert rc == 1 and field in _lib.lib().tracs_last_error().decode()


def test_validation_errors_of_shape_and_pitch():
    lib = _lib.lib()
    seqs = np.full((10, 64), ord("A"), np.uint8)
    out = np.zeros((10, 10), np.int32)

    def err(rc):
        assert rc == 1
        return lib.tracs_last_error().decode()

    o, _ = _opts()
    assert "ld (9)" in err(_host_call(seqs, o, out, 9))
    assert "out is NULL" in err(_host_call(seqs, o, None, 10))
    assert "pitch" in err(_host_call(seqs, o, out, 10, L=64, pitch=63))
    o.sweep_variant = 3
    assert "opts->sweep_variant" in err(_host_call(seqs, o, out, 10))
    # rectangle 4 x 6: ld counts columns of the rectangle
    o, _ = _opts(i_end=4, j_start=4)
    assert "ld (5)" in err(_host_call(seqs, o, out, 5))
    op, _ = _opts(packed=True)
    assert "pitch" in err(_host_call(seqs, op, out, 10, L=200, pitch=64))  # 64 bytes cannot hold 200 sites
    # device input: ASCII pitch a multiple of 32, packed pitch a multiple of 16 bytes
    assert "pitch" in err(lib.tracs_distance_matrix_device(C.c_void_p(1 << 20), 10, 64, 80, C.byref(o), C.c_void_p(1 << 21), 6))
    assert "pitch" in err(lib.tracs_distance_matrix_device(C.c_void_p(1 << 20), 10, 64, 24, C.byref(op), C.c_void_p(1 << 21), 10))


def test_python_entry_shape_errors():
    with pytest.raises(ValueError, match="n_query"):
        tracs_b200.distance_matrix(np.full((4, 8), ord("A"), np.uint8), n_query=4)
    with pytest.raises(ValueError, match="n_query"):
        tracs_b200.distance_matrix(np.full((4, 8), ord("A"), np.uint8), n_query=0)
    with pytest.raises(ValueError, match="L"):
        tracs_b200.distance_matrix(np.zeros((4, 16), np.uint8), packed=True)


def test_no_gpu_fails_loudly():
    if _lib.lib().tracs_device_count() > 0:
        pytest.skip("GPU present")
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        tracs_b200.distance_matrix(np.full((3, 40), ord("A"), np.uint8))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        tracs_b200.distance_matrix(np.full((5, 40), ord("A"), np.uint8), n_query=2)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        tracs_b200.distance_matrix_device(1 << 20, 3, 40, 64, 1 << 21, 3)


def test_dists_help_runs():
    out = subprocess.run([sys.executable, "-m", "tracs_b200.dists", "--help"], cwd=ROOT, capture_output=True, text=True, check=True)
    assert "--msa-db" in out.stdout and "--csv" in out.stdout


def test_dists_refuses_files_of_unequal_length(tmp_path):
    from tracs_b200 import dists
    (tmp_path / "q.fa").write_text(">a\nACGTACGT\n")
    (tmp_path / "d.fa").write_text(">b\nACGTACG\n")
    with pytest.raises(RuntimeError, match="Error reading FASTA, variable sequence lengths!"):
        dists.dists(str(tmp_path / "q.fa"), str(tmp_path / "o.tsv"), msa_db=str(tmp_path / "d.fa"))
