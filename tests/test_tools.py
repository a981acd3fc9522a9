"""CPU checks of the small helper scripts that produce committed evidence."""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_launch_summary_reads_the_committed_launch_list():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "launch_summary.py"),
                          os.path.join(ROOT, "profiles", "r1_launches.csv")], capture_output=True, text=True, check=True).stdout
    assert out.startswith("One step = ")
    rows = [ln for ln in out.splitlines() if ln.startswith("| tracs::")]
    names = [ln.split("|")[1].strip() for ln in rows]
    # the dominant kernels of the default (filter-and-refine) step, largest first
    assert names[0] in ("tracs::k_pack_x", "tracs::k_pack") and "tracs::k_refine" in names and "tracs::k_ncomp" in names
    shares = [float(ln.split("|")[4]) for ln in rows]
    assert shares == sorted(shares, reverse=True) and 0.99 < sum(float(ln.split("|")[4]) for ln in out.splitlines()
                                                                 if ln.startswith("| ") and not ln.startswith("| kernel")) < 1.01


def test_launch_summary_round2_list_and_traffic_table_agree():
    """The round-2 launch list (packed C3 step, two-parameter kernel templates, DRAM byte columns) and the per-config traffic
    table bench.py reads: the dominant kernel's DRAM bytes per launch are the same number in both."""
    import json
    out = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "launch_summary.py"),
                          os.path.join(ROOT, "profiles", "r2_launches.csv")], capture_output=True, text=True, check=True).stdout
    rows = [ln.split("|") for ln in out.splitlines() if ln.startswith("| tracs::")]
    names = [r[1].strip() for r in rows]
    assert names[0].startswith("tracs::k_pack4<1") and "tracs::k_sweep" in names[:3] and "tracs::k_block_n" in names[:4]
    pack_gb = float(rows[0][5])
    traffic = json.load(open(os.path.join(ROOT, "profiles", "kernel_traffic.json")))["C3"]
    assert abs(traffic["k_pack4<true>"] / 1e9 - pack_gb) < 0.5
    assert abs(traffic["k_block_n"] / 1e9 - float(rows[names.index("tracs::k_block_n")][5])) < 0.5


def test_bench_traffic_lookup_is_keyed_by_config():
    sys.path.insert(0, ROOT)
    import bench
    assert bench.kernel_traffic("C3").get("k_pack4<true>", 0) > 1e11
    assert "k_pack4<true>" not in bench.kernel_traffic("C2") and bench.kernel_traffic("C2").get("k_pack_x", 0) > 5e10
    assert bench.kernel_traffic(None) == {} and bench.kernel_traffic("C9") == {}
    r = bench.tc_roof(1e9, 10.0, "x", {"tops": 4500.0, "source": "t"}, 4.6e12, code=34)
    assert r["kernel"] == "k_sweep_tc3<4>" and r["executed_planes_per_site"] == 4 and abs(r["executed_tops"] - r["achieved"]) < 1e-9
    assert bench.tc_roof(1e9, 10.0, "x", None, 4.6e12, code=15)["kernel"] == "k_sweep_tc"


def test_bench_dump_outputs_writes_float_columns_and_a_seeded_sample(tmp_path, monkeypatch):
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    n = 5000
    cols = {"rows": np.arange(n, dtype=np.uint64), "cols": np.arange(n, dtype=np.uint64) + np.uint64(2**40),
            "filt": np.broadcast_to(np.uint64(0), (n,)), "p0_log": -np.linspace(0.0, 3.0, n), "eK": None}
    bench.dump_outputs(str(tmp_path / "all"), cols)
    got = {k: np.load(str(tmp_path / "all" / (k + ".npy"))) for k in ("rows", "cols", "filt", "p0_log", "edge_index")}
    assert not (tmp_path / "all" / "eK.npy").exists()
    assert all(v.dtype == np.float64 and v.shape == (n,) for v in got.values())
    assert np.array_equal(got["cols"].astype(np.uint64), cols["cols"]) and np.array_equal(got["edge_index"], np.arange(n))
    monkeypatch.setattr(bench, "DUMP_BYTES", 100_000)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), cols)
    files = sorted(os.listdir(str(tmp_path / "a")))
    assert sum(os.path.getsize(str(tmp_path / "a" / f)) for f in files) <= 100_000
    idx = np.load(str(tmp_path / "a" / "edge_index.npy")).astype(np.int64)
    assert 0 < len(idx) < n and np.all(np.diff(idx) > 0)
    for f in files:
        a, b = np.load(str(tmp_path / "a" / f)), np.load(str(tmp_path / "b" / f))
        assert np.array_equal(a, b) and len(a) == len(idx)
    assert np.array_equal(np.load(str(tmp_path / "a" / "p0_log.npy")), cols["p0_log"][idx])


def test_bench_edge_columns_of_single_and_multi_gpu_results(tmp_path):
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    from tracs_b200 import sites
    n = 7
    shared = {c: np.arange(n, dtype=dt) for c, dt in sites.SharedEdgeTable.COLS}     # what sites.sweep returns on rank 0
    single = dict(shared, filt=np.broadcast_to(np.uint64(0), (n,)), seq_length=100, names=[], dev_packed=None)
    for res, files in ((shared, 8), (single, 9)):
        d = tmp_path / str(files)
        bench.dump_outputs(str(d), bench.edge_columns(res))
        assert len(os.listdir(str(d))) == files and np.array_equal(np.load(str(d / "eK.npy")), np.arange(n, dtype=np.float64))
