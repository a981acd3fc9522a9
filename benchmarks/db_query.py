"""Resident sample database against the two-file call, on the C3 alignment (100 000 x 2 Mb, packed, on the device).

The database is rows [10 000, 100 000) of one buffer, opened by borrowing it (a pointer offset); a query batch of nq samples
is rows [10 000 - nq, 10 000), with dist 20 and sampling days. The baseline is the two-file call
pairsnp_packed(i_end = j_start = nq) on rows [10 000 - nq, 100 000) of the same buffer, which ingests the database again on
every call. The baselines run first (their host columns are kept), then tracs_trim() hands their scratch back before the
database is opened: 100 GB of input, the handle and a baseline ingest do not all fit at once.

Prints one JSON line per batch size (and one for the open) and checks in the run that every query returns columns
byte-identical to its baseline. Usage: python benchmarks/db_query.py [--reps 5] [--batches 1,100,1000,10000] [--n 100000]"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

COLS = ("rows", "cols", "dist", "ncomp", "p0_log", "eK", "datediff")


def card():
    try:
        return subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], text=True).strip()
    except Exception as e:  # noqa: BLE001
        return "unknown (%s)" % e


def timed(f, reps):
    import torch
    ts, out = [], None
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = f()
        torch.cuda.synchronize()
        ts.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(ts)), ts, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--batches", default="1,100,1000,10000")
    ap.add_argument("--n", type=int, default=100_000)
    ap.add_argument("--L", type=int, default=2_000_000)
    ap.add_argument("--split", type=int, default=10_000, help="first database row")
    a = ap.parse_args()
    import torch
    import tracs_b200
    print(json.dumps({"card": card()}), flush=True)
    n, L, split = a.n, a.L, a.split
    p4 = (L + 31) // 32 * 16
    buf = torch.empty(n * p4, dtype=torch.uint8, device="cuda")
    d_days = torch.empty(n, dtype=torch.int32, device="cuda")
    tracs_b200.synth_device(buf.data_ptr(), n, L, p4, seed=3, p_var=0.01, n_clusters=2000, mu=5.0, p_N=1e-3, p_amb=0.0, gc=0.5, n_days=180,
                            gaps=2, dev_days=d_days.data_ptr(), packed=True)
    days = d_days.cpu().numpy()
    batches = [int(x) for x in a.batches.split(",")]
    kw = dict(dist=20, lamb=29.903, beta=73.0, threshold_Ek=0.01)
    base = {}
    for nq in batches:
        lo = split - nq
        f = lambda: tracs_b200.pairsnp_packed(buf.data_ptr() + lo * p4, n - lo, L, p4, i_end=nq, j_start=nq, days=days[lo:], **kw)  # noqa: E731
        f()  # warm-up
        ms, ts, out = timed(f, a.reps)
        base[nq] = (ms, ts, out, tracs_b200.last_stats())
    tracs_b200.api._lib.lib().tracs_trim()
    t0 = time.perf_counter()
    db = tracs_b200.Database.from_device(buf.data_ptr() + split * p4, n - split, L, p4, packed=True)
    torch.cuda.synchronize()
    open_ms = (time.perf_counter() - t0) * 1e3
    info = db.info()
    print(json.dumps({"open_ms": open_ms, "open_stats": tracs_b200.last_stats(), "info": info}), flush=True)
    for nq in batches:
        lo = split - nq
        qdays = np.concatenate([days[lo:split], days[split:]])
        fd = lambda: db.query_device(buf.data_ptr() + lo * p4, nq, p4, days=qdays, packed=True, **{"dist": 20})  # noqa: E731
        fd()
        ms_dev, ts_dev, out_dev = timed(fd, a.reps)
        st = tracs_b200.last_stats()
        new_sites = db.info()["new_sites"]
        host_q = buf[lo * p4:split * p4].view(nq, p4).cpu().numpy()
        fh = lambda: db.query(host_q, days=qdays, packed=True, L=L, dist=20)  # noqa: E731
        fh()
        ms_host, ts_host, out_host = timed(fh, a.reps)
        b_ms, b_ts, b_out, b_st = base[nq]
        same = all((out_dev[k] is None and b_out[k] is None) or (out_dev[k] is not None and b_out[k] is not None and
                                                                  out_dev[k].dtype == b_out[k].dtype and
                                                                  out_dev[k].tobytes() == b_out[k].tobytes()) for k in COLS)
        same_host = all((out_host[k] is None) == (b_out[k] is None) and (out_host[k] is None or out_host[k].tobytes() == b_out[k].tobytes())
                        for k in COLS)
        print(json.dumps({"nq": nq, "n_db": n - split, "edges": int(len(out_dev["rows"])), "query_device_ms": ms_dev, "query_host_ms": ms_host,
                          "two_file_ms": b_ms, "speedup_device": b_ms / ms_dev, "speedup_host": b_ms / ms_host, "new_sites": new_sites,
                          "identical_device": same, "identical_host": same_host, "ts_device": ts_dev, "ts_host": ts_host, "ts_two_file": b_ts,
                          "query_stats": st, "two_file_stats": b_st}), flush=True)
        assert same and same_host, nq
    db.close()
    print(json.dumps({"card": card()}), flush=True)


if __name__ == "__main__":
    main()
