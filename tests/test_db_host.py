"""CPU: the resident sample database (tracs_db_*) refuses bad arguments before any device call, fails loudly without a GPU,
refuses NULL / closed / unknown handles without touching them, and its command line parses."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

import tracs_b200
from tracs_b200 import _lib, api

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _err(rc):
    assert rc != 0
    return _lib.lib().tracs_last_error().decode()


def test_info_struct_layout_matches_c(tmp_path):
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "tracs_b200.h"', 'int main(void) {',
             'printf("size %zu\\n", sizeof(tracs_db_info_t));']
    for f, _ in _lib.DbInfo._fields_:
        lines.append('printf("%s %%zu\\n", offsetof(tracs_db_info_t, %s));' % (f, f))
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines + ["return 0; }"]))
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(tmp_path / "layout")])
    got = dict(l.split() for l in subprocess.check_output([str(tmp_path / "layout")]).decode().splitlines())
    assert int(got["size"]) == C.sizeof(_lib.DbInfo)
    for f, _ in _lib.DbInfo._fields_:
        assert int(got[f]) == getattr(_lib.DbInfo, f).offset, f


@pytest.mark.parametrize("handle", [None, 0x1234560, "closed-like"])
def test_bad_handles_are_refused(handle):
    lib = _lib.lib()
    h = C.c_void_p(0x7f00dead0000 if handle == "closed-like" else handle)
    e = _lib.Edges()
    q = np.full((2, 8), 65, np.uint8)
    o, _ = api.make_opts()
    for rc in (lib.tracs_db_query_host(h, q.ctypes.data, 2, 8, C.byref(o), C.byref(e)),
               lib.tracs_db_query_device(h, None, 0, 32, C.byref(o), C.byref(e)),
               lib.tracs_db_info(h, C.byref(_lib.DbInfo())),
               lib.tracs_db_close(h)):
        assert "handle is NULL, closed, or was never opened" in _err(rc)


def test_closed_python_handle():
    db = api.Database.__new__(api.Database)
    db._h = None
    db.close()  # closing twice is harmless in Python
    with pytest.raises(RuntimeError, match="handle is closed"):
        db.info()


@pytest.mark.parametrize("field,kw,msg", [
    ("filter", dict(filter=True), "opts->filter"),
    ("keep_on_device", dict(keep_on_device=True), "opts->keep_on_device"),
    ("shard_world", dict(shard_world=2), "opts->shard_world > 1"),
    ("i_end", dict(i_end=1), "opts->i_end / opts->j_start must be 0"),
    ("j_start", dict(j_start=1), "opts->i_end / opts->j_start must be 0"),
])
def test_query_option_errors_need_no_device(field, kw, msg):
    o, _ = api.make_opts(**kw)
    e = _lib.Edges()
    q = np.full((2, 8), 65, np.uint8)
    assert msg in _err(_lib.lib().tracs_db_query_host(None, q.ctypes.data, 2, 8, C.byref(o), C.byref(e)))
    assert msg in _err(_lib.lib().tracs_db_query_device(None, None, 2, 32, C.byref(o), C.byref(e)))


def test_open_argument_errors_need_no_device():
    lib = _lib.lib()
    s = np.full((3, 100), 65, np.uint8)
    h = C.c_void_p()
    o, _ = api.make_opts()
    assert "n must be at least 1" in _err(lib.tracs_db_open_host(s.ctypes.data, 0, 100, 100, C.byref(o), C.byref(h)))
    assert "pitch (99) must be >= L" in _err(lib.tracs_db_open_host(s.ctypes.data, 3, 100, 99, C.byref(o), C.byref(h)))
    assert "handle's address) is NULL" in _err(lib.tracs_db_open_host(s.ctypes.data, 3, 100, 100, C.byref(o), None))
    assert "must be a multiple of 32" in _err(lib.tracs_db_open_device(None, 3, 100, 100, C.byref(o), C.byref(h)))
    op, _ = api.make_opts(packed=True)
    assert "multiple of 16 bytes" in _err(lib.tracs_db_open_device(None, 3, 100, 40, C.byref(op), C.byref(h)))
    assert h.value is None


def test_python_argument_errors():
    with pytest.raises(ValueError, match="L \\(sites\\) is required"):
        tracs_b200.Database(np.zeros((2, 16), np.uint8), packed=True)
    with pytest.raises(ValueError, match="2-D"):
        tracs_b200.Database(np.zeros(16, np.uint8))


def test_open_without_gpu_fails_loudly():
    if _lib.lib().tracs_device_count() > 0:
        pytest.skip("GPU present")
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        tracs_b200.Database(np.full((2, 40), 65, np.uint8))
    h = C.c_void_p()
    o, _ = api.make_opts()
    assert "no CPU fallback" in _err(_lib.lib().tracs_db_open_device(None, 2, 40, 64, C.byref(o), C.byref(h)))


def test_command_line_help_and_unequal_lengths(tmp_path):
    out = subprocess.run([sys.executable, "-m", "tracs_b200.query", "--help"], cwd=ROOT, capture_output=True, text=True)
    assert out.returncode == 0 and "--db" in out.stdout and "--msa" in out.stdout and "--filter" not in out.stdout
    db, q = tmp_path / "db.fasta", tmp_path / "q.fasta"
    db.write_text(">a\nACGTACGT\n>b\nACGTACGA\n")
    q.write_text(">c\nACGTAC\n")
    out = subprocess.run([sys.executable, "-m", "tracs_b200.query", "--db", str(db), "--msa", str(q), "-o", str(tmp_path / "o.csv")],
                         cwd=ROOT, capture_output=True, text=True)
    assert out.returncode != 0
    if _lib.lib().tracs_device_count() > 0:
        assert "the alignments must have the same length" in out.stderr, out.stderr
    else:
        assert "no CPU fallback" in out.stderr, out.stderr
