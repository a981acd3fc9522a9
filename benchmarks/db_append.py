"""Appending to the resident sample database against the one-shot call, on the C3 alignment (100 000 x 2 Mb, packed, on the
device, with sampling days).

The database is rows [0, 90 000) of one buffer, opened by borrowing it. Batches of 1, 10, 100, 1 000, 4 000 and 1 samples,
the rows right after it, are appended in turn (dist 20, days). What a caller runs without the append is the one-shot call
pairsnp_packed(n_db + m rows, j_start = n_db) on the same prefix of the buffer, which ingests the whole prefix again; every
append must return columns byte-identical to it (checked in the run). The baselines run first and tracs_trim() hands their
scratch back before the database is opened: 100 GB of input, the handle (with its N-plane growth) and a one-shot ingest do
not all fit at once. The appends cannot be repeated on one handle, so each of --reps sequences opens the database anew.

Then a query of 1 000 samples (the rows after the last batch) on the grown handle against the same query on a handle
freshly opened on the same rows. Prints JSON lines; the card's name and power limit are read first and last.
Usage: python benchmarks/db_append.py [--reps 5] [--batches 1,10,100,1000,4000,1]"""
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


def identical(a, b):
    return all((a[k] is None) == (b[k] is None) and (a[k] is None or (a[k].dtype == b[k].dtype and a[k].tobytes() == b[k].tobytes()))
               for k in COLS)


def timed(f):
    import torch
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = f()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--batches", default="1,10,100,1000,4000,1")
    ap.add_argument("--n", type=int, default=100_000)
    ap.add_argument("--L", type=int, default=2_000_000)
    ap.add_argument("--n-db", dest="n_db", type=int, default=90_000)
    ap.add_argument("--nq", type=int, default=1000, help="query batch on the grown and on a fresh handle")
    a = ap.parse_args()
    import torch
    import tracs_b200
    print(json.dumps({"card": card()}), flush=True)
    n, L, n_db = a.n, a.L, a.n_db
    p4 = (L + 31) // 32 * 16
    buf = torch.empty(n * p4, dtype=torch.uint8, device="cuda")
    d_days = torch.empty(n, dtype=torch.int32, device="cuda")
    tracs_b200.synth_device(buf.data_ptr(), n, L, p4, seed=3, p_var=0.01, n_clusters=2000, mu=5.0, p_N=1e-3, p_amb=0.0, gc=0.5, n_days=180,
                            gaps=2, dev_days=d_days.data_ptr(), packed=True)
    days = d_days.cpu().numpy()
    batches = [int(x) for x in a.batches.split(",")]
    starts = [int(x) for x in np.cumsum([n_db] + batches[:-1])]
    n_end = starts[-1] + batches[-1]
    assert n_end + a.nq <= n
    kw = dict(dist=20)  # default likelihood rates

    # ---- the one-shot call on each prefix ----------------------------------------------------------------------------------
    base = []
    for s0, m in zip(starts, batches):
        f = lambda: tracs_b200.pairsnp_packed(buf.data_ptr(), s0 + m, L, p4, j_start=s0, days=days[:s0 + m], **kw)  # noqa: E731
        f()  # warm-up
        ts, out = [], None
        for _ in range(a.reps):
            ms, out = timed(f)
            ts.append(ms)
        base.append((ts, out, tracs_b200.last_stats()))
    tracs_b200.api._lib.lib().tracs_trim()

    # ---- appends: one sequence per rep, each on a freshly opened handle ------------------------------------------------------
    app = [[] for _ in batches]
    db = None
    for rep in range(a.reps):
        if db is not None:
            db.close()
            tracs_b200.api._lib.lib().tracs_trim()
        open_ms, db = timed(lambda: tracs_b200.Database.from_device(buf.data_ptr(), n_db, L, p4, packed=True))
        if rep == 0:
            print(json.dumps({"open_ms": open_ms, "info": db.info()}), flush=True)
        cap = n_db  # the handle's rule (DESIGN 4.5): N buffers hold the database's rows at open, grow to max(n + m, 1.25 n)
        for k, (s0, m) in enumerate(zip(starts, batches)):
            held0 = db.info()["bytes_held"]
            ms, out = timed(lambda: db.append_device(buf.data_ptr() + s0 * p4, m, p4, days=days[:s0 + m], packed=True, **kw))
            grew = s0 + m > cap
            if grew:
                cap = max(s0 + m, s0 + s0 // 4)
            same = identical(out, base[k][1])
            app[k].append((ms, same, grew, tracs_b200.last_stats(), db.info(), held0))
            assert same, (rep, m)
    for k, (s0, m) in enumerate(zip(starts, batches)):
        ts_b, out_b, st_b = base[k]
        ts_a = [x[0] for x in app[k]]
        ms_a, ms_b = float(np.median(ts_a)), float(np.median(ts_b))
        _, _, grew, st_a, info, held0 = app[k][-1]
        print(json.dumps({"m": m, "n_db": int(s0), "pairs": int(s0) * m + m * (m - 1) // 2, "edges": int(len(out_b["rows"])),
                          "grew_n_buffers": grew, "append_ms": ms_a, "one_shot_ms": ms_b, "speedup": ms_b / ms_a,
                          "identical": all(x[1] for x in app[k]), "new_sites": info["new_sites"], "bytes_held_before": held0,
                          "bytes_held_after": info["bytes_held"], "ts_append": ts_a, "ts_one_shot": ts_b, "append_stats": st_a,
                          "one_shot_stats": st_b}), flush=True)

    # ---- a query on the grown handle against one on a fresh handle of the same rows -----------------------------------------
    nq = a.nq
    qdays = np.concatenate([days[n_end:n_end + nq], days[:n_end]])
    qptr = buf.data_ptr() + n_end * p4
    res = {}
    for name in ("grown", "fresh"):
        if name == "fresh":
            db.close()
            tracs_b200.api._lib.lib().tracs_trim()
            db = tracs_b200.Database.from_device(buf.data_ptr(), n_end, L, p4, packed=True)
        q = lambda: db.query_device(qptr, nq, p4, days=qdays, packed=True, **kw)  # noqa: E731
        q()
        ts, out = [], None
        for _ in range(a.reps):
            ms, out = timed(q)
            ts.append(ms)
        res[name] = (ts, out, tracs_b200.last_stats(), db.info())
    db.close()
    same = identical(res["grown"][1], res["fresh"][1])
    print(json.dumps({"query_nq": nq, "n_db": int(n_end), "grown_ms": float(np.median(res["grown"][0])),
                      "fresh_ms": float(np.median(res["fresh"][0])), "identical": same, "ts_grown": res["grown"][0],
                      "ts_fresh": res["fresh"][0], "grown_stats": res["grown"][2], "fresh_stats": res["fresh"][2],
                      "grown_info": res["grown"][3], "fresh_info": res["fresh"][3]}), flush=True)
    assert same
    print(json.dumps({"card": card()}), flush=True)


if __name__ == "__main__":
    main()
