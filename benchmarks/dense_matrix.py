"""Dense all-pairs distance matrix (tracs_distance_matrix_device) at the shapes of bench.py's configurations. One JSON
line per case on stdout, each with the card's name and power limit (read-only nvidia-smi query):

  C5  50 000 x 1 Mb packed, every site variable, 10 GB square in a torch int32 tensor. Variant 0 (tensor cores) and
      variant 1 (LOP3/POPC): ms_total / ms_sweep of the dense call, alternated in the same process with the thresholded
      full-length sweep of the same kernel (dist = 20, full_sweep = "tc" / True: what bench.py's C5 line times).
  C2  10 000 x 5 Mb ASCII: the dense call vs pairsnp_device(dist = INT32_MAX), the existing way to get every pair (time,
      host bytes, agreement at every pair).
  C3  100 000 x 2 Mb packed: does the 40 GB square fit next to the 100 GB input and the ingest (free device memory
      before / after); the time if it does, the error if it does not.

Every case re-derives >= 10 000 random matrix entries per site in NumPy (spot_checks).

    python benchmarks/dense_matrix.py [--cases C5,C2,C3] [--reps 2]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np

import bench
from bench import CONFIGS, Input, Clocks

IMAX = 2147483647
POP8 = np.array([bin(x).count("1") for x in range(256)], np.uint16)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                       text=True)
    name, power, clk = [x.strip() for x in q.stdout.splitlines()[0].split(",")]
    return {"name": name, "power_limit": power, "clocks_max_sm": clk}


def spot_checks(inp, mat, n_rows=100, n_cols=100, seed=0, col0=0):
    """n_rows x n_cols random entries of `mat` (torch device tensor, row i, column j - col0) re-derived per site in NumPy:
    d = #{s: m_i[s] & m_j[s] == 0} (src/pairsnp.hpp:398-403). Sites where every sampled row shares a base are matches for
    every sampled pair and are dropped first; the rest is counted on packed bit-planes."""
    import torch
    rng = np.random.default_rng(seed)
    I = np.sort(rng.choice(min(inp.n, mat.shape[0]), size=n_rows, replace=False))
    J = np.sort(rng.choice(mat.shape[1], size=n_cols, replace=False)) + col0
    got = mat[torch.as_tensor(I, device=mat.device)][:, torch.as_tensor(J - col0, device=mat.device)].cpu().numpy().astype(np.int64)
    M = np.stack([inp.row_masks(int(x)) for x in np.concatenate([I, J])])
    keep = np.bitwise_and.reduce(M, axis=0) == 0
    M = M[:, keep]
    planes = [np.packbits(((M >> b) & 1).astype(np.uint8), axis=1) for b in range(4)]
    K = M.shape[1]
    want = np.empty((n_rows, n_cols), np.int64)
    for a in range(n_rows):
        anyb = np.zeros((n_cols, planes[0].shape[1]), np.uint8)
        for P in planes:
            anyb |= P[a] & P[n_rows:]
        want[a] = K - POP8[anyb].sum(axis=1, dtype=np.int64)
    bad = int((got != want).sum())
    return {"entries_checked": int(got.size), "mismatches": bad, "ok": bad == 0, "sites_kept": int(K),
            "method": "per-site NumPy definition on the sampled rows (sites shared by every sampled row dropped)"}


def stats():
    import tracs_b200
    return tracs_b200.last_stats()


def trim():
    import torch
    from tracs_b200 import _lib
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    _lib.lib().tracs_trim()


def case_c5(args, torch, tracs_b200, info):
    w = CONFIGS["C5"]
    inp = Input(torch, tracs_b200, "cuda", w)
    n, L = inp.n, inp.Ls
    peak = tracs_b200.int_peak()
    tc = tracs_b200.tc_peak_sustained(2.0)
    peak_wp = min(peak["lop3_per_s"] / 4.0, peak["popc_per_s"])
    out = torch.empty((n, n), dtype=torch.int32, device="cuda")
    # warm-up of every kernel the timed calls use (module load, function attributes)
    for fs in (False, True):
        tracs_b200.distance_matrix_device(inp.buf.data_ptr(), 2048, L, inp.pitch, out.data_ptr(), 2048, packed=True, full_sweep=fs)
        tracs_b200.pairsnp_packed(inp.buf.data_ptr(), 2048, L, inp.pitch, dist=20, full_sweep=fs or "tc")
    for variant in (0, 1):
        fs_dense, fs_thr = (False, "tc") if variant == 0 else (True, True)
        clocks = Clocks(0)
        clocks.start()
        clocks.mark()
        dense, thr = [], []
        for _ in range(args.reps):
            tracs_b200.distance_matrix_device(inp.buf.data_ptr(), n, L, inp.pitch, out.data_ptr(), n, packed=True, full_sweep=fs_dense)
            dense.append(stats())
            tracs_b200.pairsnp_packed(inp.buf.data_ptr(), n, L, inp.pitch, dist=20, full_sweep=fs_thr)
            thr.append(stats())
        clk = clocks.stop()
        d_sweep = float(np.median([s["ms_sweep"] for s in dense]))
        t_sweep = float(np.median([s["ms_sweep"] for s in thr]))
        d_total = float(np.median([s["ms_total"] for s in dense]))
        s0 = dense[0]
        wp = s0["swept_wordpairs"]
        if s0["tc_sweep"] > 0.5:
            roof = bench.tc_roof(wp, d_sweep, "dense full-length sweep", tc, peak_wp, code=int(round(s0["tc_sweep"])))
        else:
            roof = bench.int_roof(wp, d_sweep, "full-length sweep (dense epilogue)", peak, {})
        code = int(round(s0["tc_sweep"]))
        bench_line = {"case": "C5", "variant": variant, "kernel": ("k_sweep_tc3<%d, true>" % (code % 10)) if code else "k_sweep<true>",
                      "n": n, "L": L, "n_pairs": s0["n_pairs"], "matrix_gb": n * n * 4 / 1e9,
                      "dense_ms_total": [s["ms_total"] for s in dense], "dense_ms_sweep": [s["ms_sweep"] for s in dense],
                      "thresholded_ms_sweep": [s["ms_sweep"] for s in thr], "thresholded_kernel_code": thr[0]["tc_sweep"],
                      "dense_code": s0["tc_sweep"], "sweep_ratio_dense_over_thresholded": d_sweep / t_sweep,
                      "within_10_percent": d_sweep <= 1.10 * t_sweep,
                      "site_pairs_per_s_sweep": s0["n_pairs"] * L / (d_sweep * 1e-3),
                      "site_pairs_per_s_total": s0["n_pairs"] * L / (d_total * 1e-3),
                      "roofline": roof, "clocks": clk, "card": info,
                      "spot_checks": spot_checks(inp, out, seed=variant)}
        print(json.dumps(bench_line), flush=True)
    del out, inp
    trim()


def case_c2(args, torch, tracs_b200, info):
    w = CONFIGS["C2"]
    inp = Input(torch, tracs_b200, "cuda", w)
    n, L = inp.n, inp.Ls
    out = torch.empty((n, n), dtype=torch.int32, device="cuda")
    tracs_b200.distance_matrix_device(inp.buf.data_ptr(), 512, L, inp.pitch, out.data_ptr(), 512)  # warm-up
    dense, sparse, wall_d, wall_s, d2h = [], [], [], [], []
    e = None
    for _ in range(args.reps):
        t0 = time.perf_counter()
        tracs_b200.distance_matrix_device(inp.buf.data_ptr(), n, L, inp.pitch, out.data_ptr(), n)
        torch.cuda.synchronize()
        wall_d.append((time.perf_counter() - t0) * 1e3)
        dense.append(stats())
        t0 = time.perf_counter()
        host = out.cpu()
        d2h.append((time.perf_counter() - t0) * 1e3)
        e = None
        t0 = time.perf_counter()
        e = tracs_b200.pairsnp_device(inp.buf.data_ptr(), n, L, inp.pitch, dist=IMAX)
        wall_s.append((time.perf_counter() - t0) * 1e3)
        sparse.append(stats())
    m = host.numpy()
    rows, cols = e["rows"].astype(np.int64), e["cols"].astype(np.int64)
    agree = bool(len(rows) == n * (n - 1) // 2 and (m[rows, cols] == e["dist"]).all() and (m[cols, rows] == e["dist"]).all()
                 and (np.diag(m) == 0).all())
    line = {"case": "C2", "n": n, "L": L, "n_pairs": dense[0]["n_pairs"], "dense_kernel_code": dense[0]["tc_sweep"],
            "dense_ms_total": [s["ms_total"] for s in dense], "dense_ms_sweep": [s["ms_sweep"] for s in dense], "dense_wall_ms": wall_d,
            "dense_host_bytes": 0, "dense_matrix_bytes": n * n * 4, "matrix_to_host_ms (torch .cpu(), pageable)": d2h,
            "pairs_ms_total": [s["ms_total"] for s in sparse], "pairs_ms_sweep": [s["ms_sweep"] for s in sparse], "pairs_wall_ms": wall_s,
            "pairs_d2h_bytes": sparse[0]["d2h_bytes"], "pairs_host_bytes_per_edge": 56, "pairs_edges": int(len(rows)),
            "agree_at_every_pair": agree, "card": info, "spot_checks": spot_checks(inp, out)}
    print(json.dumps(line), flush=True)
    del out, inp, e, host, m
    trim()


def case_c3(args, torch, tracs_b200, info):
    w = CONFIGS["C3"]
    free0, total = torch.cuda.mem_get_info()
    inp = Input(torch, tracs_b200, "cuda", w)
    n, L = inp.n, inp.Ls
    free1, _ = torch.cuda.mem_get_info()
    line = {"case": "C3", "n": n, "L": L, "matrix_gb": n * n * 4 / 1e9, "input_gb": inp.bytes / 1e9, "device_total_gb": total / 1e9,
            "free_gb_before_input": free0 / 1e9, "free_gb_after_input": free1 / 1e9, "card": info}
    try:
        out = torch.empty((n, n), dtype=torch.int32, device="cuda")
    except Exception as ex:
        line.update({"fits": False, "error": "torch could not allocate the square next to the input: " + str(ex).splitlines()[0]})
        print(json.dumps(line), flush=True)
        return
    line["free_gb_after_matrix"] = torch.cuda.mem_get_info()[0] / 1e9
    try:
        t0 = time.perf_counter()
        tracs_b200.distance_matrix_device(inp.buf.data_ptr(), n, L, inp.pitch, out.data_ptr(), n, packed=True)
        torch.cuda.synchronize()
        s = stats()
        line.update({"fits": True, "wall_ms": (time.perf_counter() - t0) * 1e3, "ms_total": s["ms_total"], "ms_sweep": s["ms_sweep"],
                     "ms_pack": s["ms_pack"], "ms_compact": s["ms_compact"], "kernel_code": s["tc_sweep"], "n_pairs": s["n_pairs"],
                     "spot_checks": spot_checks(inp, out)})
    except RuntimeError as ex:
        line.update({"fits": False, "error": str(ex)})
    line["free_gb_after_call"] = torch.cuda.mem_get_info()[0] / 1e9
    print(json.dumps(line), flush=True)
    del out, inp
    trim()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cases", default="C5,C2,C3")
    ap.add_argument("--reps", type=int, default=2)
    args = ap.parse_args()
    import torch
    import tracs_b200
    if not torch.cuda.is_available():
        raise SystemExit("dense_matrix.py measures on a CUDA device; none is available")
    info = card()
    for c in args.cases.split(","):
        {"C5": case_c5, "C2": case_c2, "C3": case_c3}[c](args, torch, tracs_b200, info)


if __name__ == "__main__":
    main()
