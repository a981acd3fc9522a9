"""bench.py --config C1 | C4 | C5: the other shapes BASELINE.json names, each as one JSON line with `roofline`,
`cpu_baseline` and in-run parity spot checks (same contract as the default C3 line; single GPU).

  C1  1,000 x 2.8 Mb through the reference's entry point TRACS.pairsnp(fasta=[...]) on a FASTA file in /dev/shm --
      the one shape the reference runs in full (bench.py --impl reference --config C1), so the two arms have the
      SAME config; `value` is the device-resident number, `e2e` the file-to-lists number.
  C4  20 per-reference alignments of up to 2,000 samples (ambiguity codes, 30 % N), dist <= 100, one sweep per MSA
      (tracs/distance.py:159 loop) + device min-over-references (tracs_min_over_refs).
  C5  50,000 x 1 Mb, every site variable: the full-length tile sweep forced on the LOP3/POPC kernel and on the
      tcgen05 int8 one-hot GEMM, head to head."""
import ctypes as C
import os
import tempfile
import time

import numpy as np


def _setup(args, B):
    import torch
    import tracs_b200
    from tracs_b200 import _lib
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; this framework has no CPU path")
    torch.cuda.set_device(0)
    _lib.check(_lib.lib().tracs_set_device(0))
    return torch, tracs_b200, _lib, torch.device("cuda", 0)


def _cpu_baseline(args, B, w):
    if args.no_cpu:
        return {"value": None, "note": "skipped (--no-cpu)"}
    try:
        mod, kind, what = B.load_reference()
        smp = B.RefSample(w)
        try:
            r = smp.step(mod, B.n_cores())
        finally:
            smp.cleanup()
        return {"value": r["value"], "unit": "site-pairs/s", "cores": B.n_cores(), "kind": kind, "sample": smp.desc, "what": what,
                "projected": True, "pair_stage_site_pairs_per_s": r["pair_rate"], "load_bases_per_s": r["load_rate"]}
    except Exception as ex:
        return {"value": None, "error": repr(ex)}


def _timed(torch, fn, steps, warmup):
    out = None
    for _ in range(warmup + 1):   # + 1: the result-buffer caches need two live result sets before the clock starts
        out = fn()                # (one set stays referenced while the next call runs, as in the timed loop)
    out = out[0]
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    stats = []
    ev0.record()
    for _ in range(steps):
        t0 = time.perf_counter()
        out, st = fn()
        st = dict(st)
        st["wall_ms"] = 1e3 * (time.perf_counter() - t0)
        stats.append(st)
    ev1.record()
    torch.cuda.synchronize()
    return ev0.elapsed_time(ev1) / steps, out, stats


def _base_line(B, args, w, cfg, value, ms, steps, warmup, clk, launches):
    return {"metric": B.METRIC, "value": value, "unit": "site-pairs/s", "n_gpus": 1, "steps": steps, "warmup": warmup, "ms_per_step": ms,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": B.DTYPE,
            "data": "synthetic (device-generated alignment, seeded)", "config": B.config_block(w, cfg, 1), "clocks": clk,
            "gpu_launches": launches}


# ------------------------------------------------------------------------------------------------ C1
def run_c1(args, saved_stdout, B):
    torch, tracs_b200, _lib, device = _setup(args, B)
    w = dict(B.CONFIGS["C1"], fmt="ascii")
    n, L = w["n"], w["L"]
    P = n * (n - 1) // 2
    inp = B.Input(torch, tracs_b200, device, w)
    peak = tracs_b200.int_peak()
    tc_peak = B.measured_tc_peak(tracs_b200)
    kw = dict(dist=w["dist"])
    clocks = B.Clocks(0)
    clocks.start()

    def step():
        return tracs_b200.pairsnp_device(inp.buf.data_ptr(), n, L, inp.pitch, copy=False, **kw), tracs_b200.last_stats()
    clocks.mark()
    ms, res, stats = _timed(torch, step, args.steps, args.warmup)
    clk = clocks.stop()
    if args.dump_outputs:
        B.dump_outputs(args.dump_outputs, B.edge_columns(res))
    roof_pack, roof_sweep, pack_kernel = B.rooflines(tracs_b200, w, stats, peak, n, L, tc_peak, config=args.config if not (args.n or args.L) else None)
    line = _base_line(B, args, B.CONFIGS["C1"], "C1", P * L / (ms * 1e-3), ms, args.steps, args.warmup, clk,
                      int(sum(s["kernel_launches"] for s in stats)))
    line["roofline"] = roof_pack
    line["roofline_kernels"] = {pack_kernel: roof_pack, "tile_sweep_as_launched": roof_sweep}
    line["details"] = {"edges": int(len(res["rows"])), "variable_sites": int(stats[-1]["n_variable_sites"])}
    line["stages_ms"] = {k: float(np.mean([s[k] for s in stats])) for k in ("ms_pack", "ms_compact", "ms_sweep", "ms_refine", "ms_sort",
                                                                               "ms_ncomp", "ms_trans", "ms_d2h", "ms_total")}
    line["parity_spot_checks"] = B.spot_checks(inp, res, w["dist"])
    # ---- e2e: the reference's entry point on a FASTA file ---------------------------------------------------------
    e2e = {"value": None, "unit": "site-pairs/s", "h2d_bytes_per_step": n * L, "d2h_bytes_per_step": None}
    if not args.no_e2e:
        d = tempfile.mkdtemp(prefix="tracs_c1_", dir="/dev/shm" if os.path.isdir("/dev/shm") else None)
        try:
            path = os.path.join(d, "c1.fasta")
            host = inp.buf.view(n, inp.pitch)[:, :L].cpu().numpy()
            with open(path, "wb") as f:
                for i in range(n):
                    f.write(b">s%d\n" % i)
                    f.write(host[i].tobytes())
                    f.write(b"\n")
            del host
            T = tracs_b200.install_dropin()
            cores = B.n_cores()
            T.pairsnp(fasta=[path], n_threads=cores, dist=w["dist"], filter=False)   # warm-up (page cache, buffer caches)
            ts = []
            for _ in range(max(1, args.e2e_steps)):
                t0 = time.perf_counter()
                r = T.pairsnp(fasta=[path], n_threads=cores, dist=w["dist"], filter=False)
                ts.append(time.perf_counter() - t0)
            st = tracs_b200.last_stats()
            te = float(np.median(ts))
            e2e.update({"value": P * L / te, "ms_per_step": 1e3 * te, "steps": len(ts), "d2h_bytes_per_step": int(st["d2h_bytes"]),
                        "api": "TRACS.pairsnp(fasta=[plain FASTA in /dev/shm], n_threads=%d, dist=20, filter=False) -> 6-tuple of lists" % cores,
                        "file_bytes": os.path.getsize(path),
                        "edges_equal_device_path": bool(r[0] == res["rows"].tolist() and r[2] == res["dist"].tolist() and r[5] == res["ncomp"].tolist())})
            # the same file gzip-compressed (what tracs/combine.py:220-239 writes), on a 10 % subsample: single-stream inflate bound
            import gzip
            gz = os.path.join(d, "c1_sub.fasta.gz")
            sub = max(2, n // 10)
            with open(path, "rb") as fi, gzip.open(gz, "wb", compresslevel=1) as fo:
                for _ in range(2 * sub):
                    fo.write(fi.readline())
            t0 = time.perf_counter()
            T.pairsnp(fasta=[gz], n_threads=cores, dist=w["dist"], filter=False)
            tg = time.perf_counter() - t0
            e2e["gz_subsample"] = {"seqs": sub, "seconds": tg, "bases_per_s": sub * L / tg,
                                   "note": "single-member .gz is bound by one zlib inflate stream; parse and copies overlap it"}
        except Exception as ex:
            e2e["error"] = repr(ex)
        finally:
            import shutil
            shutil.rmtree(d, ignore_errors=True)
    line["e2e"] = e2e
    line["cpu_baseline"] = _cpu_baseline(args, B, B.CONFIGS["C1"])
    B._emit(saved_stdout, line)
    return 0


# ------------------------------------------------------------------------------------------------ C5
def run_c5(args, saved_stdout, B):
    torch, tracs_b200, _lib, device = _setup(args, B)
    w = B.CONFIGS["C5"]
    n, L = w["n"], w["L"]
    P = n * (n - 1) // 2
    inp = B.Input(torch, tracs_b200, device, w)
    peak = tracs_b200.int_peak()
    tc_peak = B.measured_tc_peak(tracs_b200)
    peak_wp = min(peak["lop3_per_s"] / 4.0, peak["popc_per_s"])
    kw = dict(dist=w["dist"])
    clocks = B.Clocks(0)
    clocks.start()
    kernels, results, launches = {}, {}, 0
    # the faster kernel is the line's value; the tensor-core kernel gets 3 warm-ups, the 11 s LOP3/POPC sweep one
    plan = {"k_sweep_full_length": (args.steps, 1), "k_sweep_tc_full_length": (args.steps, 3)}
    clocks.mark()
    for nm, variant in (("k_sweep_full_length", True), ("k_sweep_tc_full_length", "tc")):
        def step():
            return tracs_b200.pairsnp_packed(inp.buf.data_ptr(), n, L, inp.pitch, full_sweep=variant, copy=False, **kw), tracs_b200.last_stats()
        ms, res, stats = _timed(torch, step, *plan[nm])
        s = stats[-1]
        launches += int(sum(x["kernel_launches"] for x in stats))
        rf = (B.tc_roof(s["swept_wordpairs"], s["ms_sweep"], "full-length sweep, tcgen05.mma kind::i8, int32 accumulators in TMEM", tc_peak, peak_wp,
                        code=int(round(s["tc_sweep"])))
              if variant == "tc" else B.int_roof(s["swept_wordpairs"], s["ms_sweep"], "full-length sweep (LOP3 + POPC)", peak, {}))
        rf["whole_step_ms"] = ms
        kernels[nm] = rf
        results[nm] = (ms, res, stats)
    clk = clocks.stop()
    best = min(results, key=lambda k: results[k][0])
    ms, res, stats = results[best]
    other = results[[k for k in results if k != best][0]][1]
    if args.dump_outputs:
        B.dump_outputs(args.dump_outputs, B.edge_columns(res))
    # the thresholded default path on the same input (prefilter + component blocks), for reference
    def dstep():
        return tracs_b200.pairsnp_packed(inp.buf.data_ptr(), n, L, inp.pitch, copy=False, **kw), tracs_b200.last_stats()
    ms_def, res_def, st_def = _timed(torch, dstep, 2, 1)
    # The tensor-core sweep is ONE 3.5 s launch under the board's power cap: its denominator is the rate the same pipe
    # sustains over seconds (measured right here, probe held 2 s), not the 10 ms burst figure (kept as peak_burst).
    try:
        sus = tracs_b200.tc_peak_sustained(2.0)
        rf = kernels["k_sweep_tc_full_length"]
        rf["peak_burst"], rf["frac_of_burst_peak"] = rf["peak"], rf["frac"]
        rf["peak"], rf["frac"], rf["peak_source"] = sus["tops"], rf["achieved"] / sus["tops"], sus["source"]
    except Exception as ex:
        kernels["k_sweep_tc_full_length"]["sustained_peak_error"] = repr(ex)
    line = _base_line(B, args, w, "C5", P * L / (ms * 1e-3), ms, plan[best][0], plan[best][1], clk, launches)
    line["roofline"] = kernels[best]
    line["roofline_kernels"] = kernels
    line["details"] = {"edges": int(len(res["rows"])), "variable_sites": int(stats[-1]["n_variable_sites"]), "words": int(stats[-1]["n_words"]),
                       "step": "full-length tile sweep forced (no prefilter): what an unthresholded / dense run executes; value = the faster kernel",
                       "faster_kernel": best, "tc_speedup_vs_int_pipe": results["k_sweep_full_length"][0] / results["k_sweep_tc_full_length"][0],
                       "kernels_agree": bool(all(np.array_equal(res[k], other[k]) for k in ("rows", "cols", "dist", "ncomp"))),
                       "default_thresholded_path_ms": ms_def,
                       "default_path_agrees": bool(all(np.array_equal(res[k], res_def[k]) for k in ("rows", "cols", "dist", "ncomp")))}
    line["stages_ms"] = {k: float(stats[-1][k]) for k in ("ms_pack", "ms_compact", "ms_sweep", "ms_sort", "ms_ncomp", "ms_d2h", "ms_total")}
    line["parity_spot_checks"] = B.spot_checks(inp, res, w["dist"])
    line["e2e"] = {"value": None, "unit": "site-pairs/s", "h2d_bytes_per_step": None, "d2h_bytes_per_step": None,
                   "note": "kernel comparison config; host-buffer e2e is measured on the default (C3) and C1 lines"}
    line["cpu_baseline"] = _cpu_baseline(args, B, w)
    B._emit(saved_stdout, line)
    return 0


# ------------------------------------------------------------------------------------------------ C4
def run_c4(args, saved_stdout, B):
    torch, tracs_b200, _lib, device = _setup(args, B)
    w = B.CONFIGS["C4"]
    n_all, n_refs = w["n"], w["n_refs"]
    rng = np.random.default_rng(w["seed"])
    msas = []
    for r in range(n_refs):
        frac = rng.uniform(0.6, 1.0)
        subset = np.sort(rng.choice(n_all, size=int(round(frac * n_all)), replace=False))
        L_r = int(rng.integers(2_000_000, 3_000_001))
        wr = dict(w, n=len(subset), L=L_r, seed=w["seed"] + r, n_clusters=max(2, w["n_clusters"] * len(subset) // n_all))
        msas.append((subset.astype(np.uint64), B.Input(torch, tracs_b200, device, wr), wr))
    peak = tracs_b200.int_peak()
    tc_peak = B.measured_tc_peak(tracs_b200)
    work = sum(wr["n"] * (wr["n"] - 1) // 2 * wr["L"] for _, _, wr in msas)

    def step():
        a, b, v, per = [], [], [], []
        for subset, inp, wr in msas:       # tracs/distance.py:159: one sweep per reference MSA
            res = tracs_b200.pairsnp_device(inp.buf.data_ptr(), wr["n"], wr["L"], inp.pitch, copy=False, dist=w["dist"])
            per.append((res, tracs_b200.last_stats()))
            a.append(subset[res["rows"].astype(np.int64)])
            b.append(subset[res["cols"].astype(np.int64)])
            v.append(res["dist"].astype(np.float64))
        oa, ob, ov = tracs_b200.min_over_refs(np.concatenate(a), np.concatenate(b), np.concatenate(v))   # SURVEY A.6, on the device
        agg = {k: float(sum(s[k] for _, s in per)) for k in per[0][1] if k.startswith("ms_") or k in ("kernel_launches", "swept_wordpairs",
                                                                                                       "n_pairs", "n_candidates", "n_edges")}
        agg["tc_sweep"] = float(max(s["tc_sweep"] for _, s in per))
        agg["n_early_sites"] = float(np.mean([s["n_early_sites"] for _, s in per]))
        agg["n_variable_sites"] = float(sum(s["n_variable_sites"] for _, s in per))
        return (oa, ob, ov, per), agg
    clocks = B.Clocks(0)
    clocks.start()
    clocks.mark()
    steps = args.steps
    ms, out, stats = _timed(torch, step, steps, 2)
    clk = clocks.stop()
    oa, ob, ov, per = out
    if args.dump_outputs:   # what the step hands back: the pairs after the min over references, in sample ids
        B.dump_outputs(args.dump_outputs, {"rows": oa, "cols": ob, "dist": ov})
    line = _base_line(B, args, w, "C4", work / (ms * 1e-3), ms, steps, 2, clk, int(sum(s["kernel_launches"] for s in stats)))
    s = stats[-1]
    wp, t_sw = s["swept_wordpairs"], s["ms_sweep"]
    roof_sweep = (B.tc_roof(wp, t_sw, "all 20 MSAs, tile sweep as launched", tc_peak, min(peak["lop3_per_s"] / 4.0, peak["popc_per_s"]),
                            code=int(round(s["tc_sweep"])))
                  if s["tc_sweep"] > 0.5 else B.int_roof(wp, t_sw, "all 20 MSAs, tile sweep as launched (LOP3 + POPC: ambiguity codes)", peak, {}))
    hbm, hbm_src = B.hbm_peak()
    pack_bytes = sum(wr["n"] * wr["L"] * (1 + 1 / 8) for _, _, wr in msas)
    roof_pack = {"bound": "hbm", "kernel": "k_pack / k_pack_x", "achieved": pack_bytes / (s["ms_pack"] * 1e-3) / 1e9, "peak": hbm, "unit": "GB/s",
                 "frac": pack_bytes / (s["ms_pack"] * 1e-3) / 1e9 / hbm, "traffic": None, "ms_per_launch": s["ms_pack"] / n_refs,
                 "peak_source": hbm_src, "what": "all pack launches of the 20 MSAs (ASCII read + N-plane write)"}
    line["roofline"] = roof_pack if s["ms_pack"] >= s["ms_sweep"] else roof_sweep
    line["roofline_kernels"] = {"pack": roof_pack, "tile_sweep_as_launched": roof_sweep}
    line["details"] = {"msas": n_refs, "samples": n_all, "rows_before_combine": int(sum(len(p[0]["rows"]) for p in per)),
                       "pairs_after_min_over_refs": int(len(oa)), "site_pairs_per_step": int(work),
                       "sweep_kernel": "k_sweep_tc3" if s["tc_sweep"] > 0.5 else "k_sweep (2-/3-base IUPAC codes at variable sites rule out the one-hot GEMM)"}
    line["stages_ms"] = {k: s[k] for k in ("ms_pack", "ms_compact", "ms_sweep", "ms_refine", "ms_sort", "ms_ncomp", "ms_d2h", "ms_total")}
    line["stages_ms"]["per_step_wall_ms"] = [round(x["wall_ms"], 1) for x in stats]
    # parity spot checks on the first MSA + the combine against a dictionary
    subset, inp, wr = msas[0]
    line["parity_spot_checks"] = B.spot_checks(inp, per[0][0], w["dist"])
    best = {}
    for (res, _), (sub, _, _) in zip(per, msas):
        for i, j, d in zip(sub[res["rows"].astype(np.int64)][:20000].tolist(), sub[res["cols"].astype(np.int64)][:20000].tolist(), res["dist"][:20000].tolist()):
            best[(i, j)] = min(best.get((i, j), 1e300), d)
    got = {(int(x), int(y)): float(z) for x, y, z in zip(oa.tolist(), ob.tolist(), ov.tolist())}
    line["parity_spot_checks"]["min_over_refs_ok"] = bool(all(got.get(k, -1) <= v for k, v in list(best.items())[:5000]))
    line["e2e"] = {"value": None, "unit": "site-pairs/s", "h2d_bytes_per_step": None, "d2h_bytes_per_step": None,
                   "note": "host-buffer e2e is measured on the default (C3) and C1 lines"}
    line["cpu_baseline"] = _cpu_baseline(args, B, w)
    B._emit(saved_stdout, line)
    return 0
