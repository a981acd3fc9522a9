"""CPU: appending to the resident sample database (tracs_db_append_*, Database.append) refuses bad arguments before any
device call, naming the field, and fails loudly without a GPU."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from tracs_b200 import _lib, api

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _err(rc):
    assert rc != 0
    return _lib.lib().tracs_last_error().decode()


@pytest.mark.parametrize("handle", [None, 0x1234560, 0x7f00dead0000])
def test_bad_handles_are_refused(handle):
    lib = _lib.lib()
    h = C.c_void_p(handle)
    o, _ = api.make_opts()
    b = np.full((2, 8), 65, np.uint8)
    for rc in (lib.tracs_db_append_host(h, b.ctypes.data, 2, 8, C.byref(o), C.byref(_lib.Edges())),
               lib.tracs_db_append_device(h, None, 0, 32, C.byref(o), C.byref(_lib.Edges()))):
        assert "handle is NULL, closed, or was never opened" in _err(rc)


@pytest.mark.parametrize("kw,msg", [
    (dict(filter=True), "database append: opts->filter"),
    (dict(keep_on_device=True), "database append: opts->keep_on_device"),
    (dict(shard_world=2), "database append: opts->shard_world > 1"),
    (dict(i_end=1), "database append: opts->i_end / opts->j_start must be 0"),
    (dict(j_start=1), "database append: opts->i_end / opts->j_start must be 0"),
])
def test_option_errors_need_no_device(kw, msg):
    o, _ = api.make_opts(**kw)
    b = np.full((2, 8), 65, np.uint8)
    assert msg in _err(_lib.lib().tracs_db_append_host(None, b.ctypes.data, 2, 8, C.byref(o), C.byref(_lib.Edges())))
    assert msg in _err(_lib.lib().tracs_db_append_device(None, None, 2, 32, C.byref(o), C.byref(_lib.Edges())))
    assert "database append: out is NULL" in _err(_lib.lib().tracs_db_append_host(None, b.ctypes.data, 2, 8, C.byref(o), None))


def _fake(n=5, L=8, names=None):
    """A Python handle that never reaches the library: the checks below run before any call."""
    db = api.Database.__new__(api.Database)
    db._h, db._keep, db.n, db.L, db.names = 0xdead, None, n, L, names
    return db


def test_python_argument_errors():
    b = np.full((2, 8), 65, np.uint8)
    with pytest.raises(ValueError, match=r"days must hold n_db \+ m = 7 values"):
        _fake().append(b, days=np.zeros(2, np.int32))
    with pytest.raises(ValueError, match=r"days must hold n_db \+ m = 7 values"):
        _fake().append_device(0, 2, 32, days=np.zeros(5, np.int32))
    with pytest.raises(ValueError, match="one name per appended sample"):
        _fake(names=["a"] * 5).append(b)
    with pytest.raises(ValueError, match="one name per appended sample"):
        _fake(names=["a"] * 5).append(b, names=["x"])
    with pytest.raises(ValueError, match="no sample names"):
        _fake().append(b, names=["x", "y"])
    with pytest.raises(ValueError, match="differs from the database's L"):
        _fake().append(np.full((2, 9), 65, np.uint8))
    with pytest.raises(ValueError, match="2-D"):
        _fake().append(np.zeros(8, np.uint8))
    closed = _fake()
    closed._h = None
    with pytest.raises(RuntimeError, match="handle is closed"):
        closed.append(b)


def test_append_without_gpu_fails_loudly(tmp_path):
    if _lib.lib().tracs_device_count() > 0:
        pytest.skip("GPU present")
    db, q = tmp_path / "db.fasta", tmp_path / "q.fasta"
    db.write_text(">a\nACGTACGT\n>b\nACGTACGA\n")
    q.write_text(">c\nACGTACGG\n")
    out = subprocess.run([sys.executable, "-m", "tracs_b200.query", "--db", str(db), "--msa", str(q), "--append", "-o", str(tmp_path / "o.csv")],
                         cwd=ROOT, capture_output=True, text=True)
    assert out.returncode != 0 and "no CPU fallback" in out.stderr, out.stderr


def test_command_line_help():
    out = subprocess.run([sys.executable, "-m", "tracs_b200.query", "--help"], cwd=ROOT, capture_output=True, text=True)
    assert out.returncode == 0 and "--append" in out.stdout
