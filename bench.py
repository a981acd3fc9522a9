#!/usr/bin/env python
"""bench.py -- pairwise SNP distance + transmission likelihood sweep on B200 (driver contract).

Metric: site-pair comparisons/s = P*L / t  (P = N(N-1)/2 pairs, L = nominal alignment length), the metric
BASELINE.json names. Default workload: BASELINE.json configs[2] ("C3") -- ONE alignment of 100,000 synthetic
sequences x 2 Mb, ~1% variable sites, SNP threshold 20, TransCluster likelihood with sampling dates -- the shape
the north star's target is quoted on. Held as 4-bit base masks (tracs_pairsnp_packed) it is 100 GB and fits one
B200, so it is the workload at EVERY GPU count:

  --gpus 1      the single-GPU path on the device-resident packed alignment.
  --gpus N      STRONG scaling of that one alignment ("scaling": "strong"): rank r holds the column slab
                [L*r/N, L*(r+1)/N) of every sequence (tracs_b200/sites.py): per-slab ingest + prefilter of the
                rank's triangle row-blocks, candidate all-gather, per-slab partial d / |N u N| for all candidates,
                reduce-scatter, native finish of one slice per rank into a shared page-locked host table.
                Collectives: NCCL all-gather + reduce-scatter, O(candidates).
  step          one whole pass of the hot path: packed alignment (resident in HBM) -> column masks + N planes ->
                variable-site bit-planes -> all-pairs tile sweep with fused threshold -> ordered edge list ->
                compared-site counts -> transmission likelihood -> edge columns on the host of rank 0.
  value         P*L / step time (CUDA events, max over ranks).
  e2e           same metric with the alignment in page-locked HOST memory when the clock starts: every step copies
                it host -> device (each rank its own slab over its own PCIe link) and the edge columns back.
  --config C2   BASELINE configs[1] (10,000 x 5 Mb, ASCII input, one GPU);   --config C1 / C4 / C5: the other
                named shapes (C1 through the FASTA entry point on both arms, C4 per-reference loop + device
                min-over-references, C5 dense full-length sweep: LOP3/POPC kernel vs tcgen05 int8 GEMM).
  --impl reference   the unmodified reference (oracle/_ref, built from /root/reference/src) timed on the host
                cores on a bounded, DRAM-resident sample of the same workload (C1: the whole workload).
  --steps K     the number of timed steps on every path. Lower it for --config C5 (each step runs both full-length sweeps,
                ~11 s + ~4 s on one B200) and for --impl reference --config C1 (~2 min per step).
  --dump-outputs DIR   the edge columns the last timed step returned, as DIR/<name>.npy: the inputs are seeded, so two builds
                run with the same arguments can be compared output for output.
"""
import argparse
import ctypes as C
import json
import os
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np

SECONDS_IN_YEAR = 31556952.0
COMMON = dict(p_amb=0.0, n_days=180, gaps=2, dist=20, lamb=29.903, beta=73.0, threshold_Ek=0.01, mu=5.0, p_N=1e-3)
CONFIGS = {
    "C1": dict(COMMON, name="C1: 1000 S. aureus-like seqs x 2.8 Mb, 1% variable sites, dist<=20, through the FASTA entry point",
               n=1000, L=2_800_000, p_var=0.01, n_clusters=20, gc=0.33, seed=1, fmt="fasta"),
    "C2": dict(COMMON, name="C2: 10000 seqs x 5 Mb E. coli-like, 1% variable sites, dist<=20, transcluster with dates",
               n=10000, L=5_000_000, p_var=0.01, n_clusters=100, gc=0.508, seed=2, fmt="ascii"),
    "C3": dict(COMMON, name="C3: 100000 seqs x 2 Mb sparse alignment, 1% variable sites, dist<=20, transcluster with dates",
               n=100000, L=2_000_000, p_var=0.01, n_clusters=2000, gc=0.5, seed=3, fmt="packed"),
    "C4": dict(COMMON, name="C4: metagenomic multi-strain, 2000 samples x 20 references, ambiguity codes, p_N 0.3, dist<=100, "
                            "min-over-references", n=2000, L=2_500_000, p_var=0.01, n_clusters=40, gc=0.5, seed=4, fmt="ascii",
               p_N=0.3, p_amb=0.05, dist=100, n_refs=20),
    "C5": dict(COMMON, name="C5: dense unambiguous 50000 seqs x 1 Mb, every site variable, full-length sweep: "
                            "LOP3/POPC kernel vs tcgen05 int8 one-hot GEMM", n=50000, L=1_000_000, p_var=1.0, n_clusters=500,
               gc=0.5, seed=5, fmt="packed", p_N=0.0, gaps=0),
}
METRIC = "site-pair comparisons/s (P*L/t)"
DTYPE = "u32 bit-planes (int32 counts), f64 likelihood"


def n_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def config_block(w, cfg_name, world):
    """The `config` object of the JSON line: a function of (--config, --gpus) only, so both arms print the same one."""
    n, L = w["n"], w["L"]
    if cfg_name == "C3" and world > 1:
        par = ("site-sharded strong scaling of ONE alignment: rank r ingests columns [L*r/%d, L*(r+1)/%d) of every sequence and "
               "prefilters its triangle row-blocks; candidates all-gathered, per-slab partial d and |N u N| reduce-scattered (NCCL), "
               "every rank finishes a slice of the edges and copies it into one shared page-locked host table" % (world, world))
    elif world > 1:
        par = "%d independent replicas of the workload, one per GPU (no exchange)" % world
    else:
        par = "1 GPU"
    gb = n * L / (2e9 if w["fmt"] == "packed" else 1e9)
    return {"workload": w["name"], "config": cfg_name, "n": n, "L": L, "pairs": n * (n - 1) // 2, "dist": w["dist"],
            "input": {"packed": "4-bit base masks resident in HBM", "ascii": "ASCII matrix resident in HBM",
                      "fasta": "FASTA file (page cache)"}[w["fmt"]],
            "parallelism": par, "l2": "inputs (%.1f GB) larger than L2; no flush needed" % gb}


# ------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the reference's own CPU implementation on a bounded sample
# ------------------------------------------------------------------------------------------------
class RefSample:
    """Bounded sample of the workload for the CPU reference: same generator, fewer / shorter sequences, large enough
    that the reference's bitsets (n_p * L_p / 2 bytes) do not fit the host's caches. The reference's serial loader is
    timed on its own through the empty-second-FASTA trick (pair loop empty: src/pairsnp.hpp:352-360,395)."""

    def __init__(self, w, n_p=1280, L_p=125_000, full=False):
        from tracs_b200 import synth
        if full:
            n_p, L_p = w["n"], w["L"]
        self.w, self.n_p, self.L_p, self.full = w, n_p, L_p, full
        self.dir = tempfile.mkdtemp(prefix="tracs_ref_", dir="/dev/shm" if os.path.isdir("/dev/shm") else None)
        seqs = synth.generate(n_p, L_p, p_var=w["p_var"], n_clusters=max(2, w["n_clusters"] * n_p // w["n"]), mu=w["mu"],
                              p_N=w["p_N"], p_amb=w["p_amb"], gc=w["gc"], seed=w["seed"], gaps=w["gaps"])
        self.msa = os.path.join(self.dir, "sample.fasta")
        synth.write_fasta(self.msa, seqs)
        del seqs
        self.empty = os.path.join(self.dir, "empty.fasta")
        open(self.empty, "w").close()
        self.t_load = None
        if full:
            self.desc = "the whole workload (%d seqs x %d bp FASTA in /dev/shm) through TRACS.pairsnp(fasta=...)" % (n_p, L_p)
        else:
            self.desc = ("reference pairsnp (oracle/_ref, unmodified src/pairsnp.hpp, -O3 -ffast-math) on %d seqs x %d bp of the same "
                         "generator (bitsets %d MB: DRAM-resident); loader timed alone once (empty second FASTA), pair stage = full "
                         "call - loader; value = projected whole-job rate at %d x %d: P*L / (N*L/load_rate + P*L/pair_rate)"
                         % (n_p, L_p, n_p * L_p // 2 // 1000000, w["n"], w["L"]))

    def cleanup(self):
        import shutil
        shutil.rmtree(self.dir, ignore_errors=True)

    def time_loader(self, mod, threads):
        t0 = time.perf_counter()
        mod.pairsnp(fasta=[self.msa, self.empty], n_threads=threads, dist=self.w["dist"], filter=False)
        self.t_load = time.perf_counter() - t0
        return self.t_load

    def step(self, mod, threads):
        w = self.w
        if self.t_load is None:
            self.time_loader(mod, threads)
        t0 = time.perf_counter()
        r = mod.pairsnp(fasta=[self.msa], n_threads=threads, dist=w["dist"], filter=False)
        t_full = time.perf_counter() - t0
        t_pairs = max(t_full - self.t_load, 1e-6)
        P_s = self.n_p * (self.n_p - 1) // 2
        pair_rate = P_s * self.L_p / t_pairs
        load_rate = self.n_p * self.L_p / self.t_load
        P = w["n"] * (w["n"] - 1) // 2
        if self.full:
            val = P_s * self.L_p / t_full
        else:
            val = P * w["L"] / (w["n"] * w["L"] / load_rate + P * w["L"] / pair_rate)
        return dict(t_step=t_full, pair_rate=pair_rate, load_rate=load_rate, value=val, edges=len(r[0]))


def load_reference():
    from oracle import refmod
    if refmod.available():
        mod, variant = refmod.load()
        return mod, "reference", "oracle/_ref/%s" % variant
    # the oracle port (plain C restatement) when the reference could not be compiled
    from oracle import oracle

    class _Port:
        @staticmethod
        def pairsnp(fasta, n_threads, dist, filter):
            return oracle.pairsnp(fasta, n_threads=n_threads, dist=dist, filter=filter, as_lists=False)
    return _Port, "port", "oracle/liboracle.so"


def run_reference(args, saved_stdout):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    w = CONFIGS[args.config]
    mod, kind, what = load_reference()
    cores = n_cores()
    full = args.config == "C1"
    smp = RefSample(w, full=full)
    try:
        steps = args.steps
        warm = 0 if full else args.warmup   # the whole C1 workload takes ~2 minutes per step: no warm-up steps
        smp.time_loader(mod, cores)
        for _ in range(warm):
            smp.step(mod, cores)
        t0 = time.perf_counter()
        rs = [smp.step(mod, cores) for _ in range(steps)]
        t = time.perf_counter() - t0
    finally:
        smp.cleanup()
    val = float(np.median([r["value"] for r in rs]))
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": "site-pairs/s",
        "n_gpus": args.gpus, "steps": steps, "warmup": warm, "ms_per_step": 1e3 * t / max(1, steps),
        "higher_is_better": True, "scaling": "strong" if args.config == "C3" else "weak", "vs_baseline": None, "dtype": "u64 bitset words",
        "data": "synthetic", "config": config_block(w, args.config, args.gpus),
        "cpu_baseline": {"value": val, "unit": "site-pairs/s", "cores": cores, "kind": kind, "sample": smp.desc, "what": what,
                         "projected": not full, "pair_stage_site_pairs_per_s": float(np.median([r["pair_rate"] for r in rs])),
                         "load_bases_per_s": float(np.median([r["load_rate"] for r in rs]))},
        "e2e": {"value": val, "unit": "site-pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    _emit(saved_stdout, line)
    return 0


# ------------------------------------------------------------------------------------------------
# clocks sampler
# ------------------------------------------------------------------------------------------------
class Clocks:
    """SM clock / throttle-reason sampler for the timed region. In-process NVML (nvidia_ml_py) polled from a
    thread: spawning `nvidia-smi -lms` inside a 250 ms timed region costs more than the region itself
    (its start-up holds driver locks and showed up as 50-200 ms stalls of single steps). The sampler is
    initialised before warm-up; only samples taken between mark() and stop() are reported."""
    REASONS = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}

    def __init__(self, index, period_s=0.02):
        self.index, self.period = index, period_s
        self.rows, self.t_mark = [], None
        self.ok, self.stop_flag = False, False
        try:
            import pynvml
            self.nv = pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[index]) if vis and vis.split(",")[index].isdigit() else index
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_sm = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.ok = True
        except Exception as ex:
            self.err = repr(ex)

    def start(self):
        if not self.ok:
            return
        self.t = threading.Thread(target=self._run, daemon=True)
        self.t.start()

    def mark(self):
        self.t_mark = time.perf_counter()

    def _run(self):
        nv = self.nv
        while not self.stop_flag:
            try:
                sm = float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    rs = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                except Exception:
                    rs = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                pw = nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0
                self.rows.append((time.perf_counter(), sm, rs, pw))
            except Exception:
                pass
            time.sleep(self.period)

    def stop(self):
        if not self.ok:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml unavailable: " + getattr(self, "err", "?")]}
        self.stop_flag = True
        self.t.join(timeout=2)
        rows = [r for r in self.rows if self.t_mark is None or r[0] >= self.t_mark]
        if not rows:
            rows = self.rows[-1:]
        reasons = sorted({nm for nm, bit in self.REASONS.items() for r in rows if r[2] & bit})
        return {"sm_mhz": float(np.median([r[1] for r in rows])) if rows else None, "sm_max_mhz": self.max_sm, "reasons": reasons,
                "samples": len(rows), "power_w_max": max([r[3] for r in rows]) if rows else None, "source": "nvml, 20 ms period"}


def _claim_stdout():
    """The contract is ONE JSON line on stdout. Libraries (NCCL's version banner, for one) print to fd 1,
    so fd 1 is pointed at stderr for the whole run and the JSON line goes to the saved descriptor."""
    sys.stdout.flush()
    saved = os.dup(1)
    os.dup2(2, 1)
    return saved


def _emit(saved_fd, line):
    sys.stdout.flush()
    os.write(saved_fd, (json.dumps(line) + "\n").encode())


DUMP_BYTES = 64_000_000


def dump_outputs(path, columns):
    """--dump-outputs: writes the edge columns the timed path returned in its last step as <path>/<name>.npy, float64 (exact
    for the integer columns), together with edge_index.npy, the position of each written edge in the full output. When all
    of it would exceed DUMP_BYTES, every column keeps the same sample of edges, drawn with a fixed seed from the edge count,
    so two builds run with the same arguments write files that can be compared one to one."""
    cols = {k: np.asarray(v) for k, v in columns.items() if v is not None}
    n = len(next(iter(cols.values())))
    per_edge = 8 * (len(cols) + 1)
    k = (DUMP_BYTES - 4096 * (len(cols) + 1)) // per_edge
    idx = np.arange(n) if n <= k else np.sort(np.random.default_rng(0).choice(n, size=k, replace=False))
    os.makedirs(path, exist_ok=True)
    for name, v in cols.items():
        np.save(os.path.join(path, name + ".npy"), v[idx].astype(np.float64))
    np.save(os.path.join(path, "edge_index.npy"), idx.astype(np.float64))


def edge_columns(res):
    """The per-edge numeric columns of an edge table (rows, cols, dist, filt, ncomp and, with dates, p0_log, eK, datediff).
    The shared table of a multi-GPU run has no filt column: columns a table lacks are left out."""
    return {k: res.get(k) for k in ("rows", "cols", "dist", "filt", "ncomp", "p0_log", "eK", "datediff")}


def hbm_peak():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"], "MEASURED_PEAKS.json hbm_gbs (measured copy bandwidth)"
    except Exception:
        return 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md); MEASURED_PEAKS.json absent"


def bind_to_gpu_numa_node(index):
    """One process per GPU: run on the CPUs next to that GPU (NVML's ideal affinity) BEFORE any page-locked host memory is
    allocated, so that every rank's host slab and result columns live on its GPU's NUMA node and the N concurrent
    host <-> device streams do not all cross the socket interconnect. Returns what was done (goes into the JSON line)."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        before = len(os.sched_getaffinity(0))
        pynvml.nvmlDeviceSetCpuAffinity(h)
        after = len(os.sched_getaffinity(0))
        return "nvml ideal cpu affinity (%d -> %d cpus)" % (before, after)
    except Exception as ex:   # containers may forbid it: measured as is
        return "unchanged (%s)" % type(ex).__name__


def pinned_on_gpu_node(index, nbytes, _lib):
    """A page-locked host buffer on the NUMA node the GPU hangs off (anonymous mmap + mbind + cudaHostRegister): with one
    process per GPU streaming its slab, buffers that all sit on the node the container's CPUs belong to make half of the
    GPUs read across the socket interconnect. Returns (uint8 numpy array or None, note)."""
    import ctypes
    import mmap
    try:
        import pynvml
        pynvml.nvmlInit()
        bus = pynvml.nvmlDeviceGetPciInfo(pynvml.nvmlDeviceGetHandleByIndex(index)).busId
        bus = (bus.decode() if isinstance(bus, bytes) else bus).lower()
        if len(bus.split(":")[0]) == 8:
            bus = bus[4:]
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % bus).read().strip())
        if node < 0:
            return None, "gpu numa node unknown"
        m = mmap.mmap(-1, nbytes)
        arr = np.frombuffer(m, dtype=np.uint8)
        mask = (ctypes.c_ulong * 2)(0, 0)
        mask[node // 64] = 1 << (node % 64)
        libc = ctypes.CDLL(None, use_errno=True)
        # SYS_mbind with MPOL_PREFERRED: pages come from the GPU's node while it has room and from elsewhere after that
        # (MPOL_BIND would fail the allocation instead)
        if libc.syscall(237, ctypes.c_void_p(arr.ctypes.data), ctypes.c_ulong(nbytes), 1, mask, ctypes.c_ulong(129), 0) != 0:
            return None, "mbind to node %d refused (errno %d)" % (node, ctypes.get_errno())
        _lib.check(_lib.lib().tracs_host_register(arr.ctypes.data, nbytes))
        return arr, "mmap + mbind(preferred node %d) + cudaHostRegister" % node
    except Exception as ex:
        return None, "unavailable (%s)" % type(ex).__name__


def kernel_traffic(config=None):
    """DRAM bytes per launch from the committed ncu captures (profiles/kernel_traffic.json), keyed by the config whose
    launch was captured: a figure is only attached to a launch of the same shape."""
    p = os.path.join(ROOT, "profiles", "kernel_traffic.json")
    try:
        return json.load(open(p)).get(config or "", {})
    except Exception:
        return {}


# ------------------------------------------------------------------------------------------------
# the device-resident input of one rank
# ------------------------------------------------------------------------------------------------
class Input:
    """Synthetic alignment (or one column slab of it) generated in device memory, ASCII or 4-bit packed."""

    def __init__(self, torch, tracs_b200, device, w, lo=0, hi=None, seed=None):
        self.torch, self.t, self.w = torch, tracs_b200, w
        n, L = w["n"], w["L"]
        hi = L if hi is None else hi
        self.n, self.L_total, self.lo, self.Ls = n, L, lo, hi - lo
        self.packed = w["fmt"] == "packed"
        if self.packed:
            self.pitch = max(16, (self.Ls + 31) // 32 * 16)
        else:
            self.pitch = max(128, (self.Ls + 127) // 128 * 128)
        self.buf = torch.empty(n * self.pitch, dtype=torch.uint8, device=device)
        d_days = torch.empty(n, dtype=torch.int32, device=device)
        tracs_b200.synth_device(self.buf.data_ptr(), n, self.Ls, self.pitch, seed=w["seed"] if seed is None else seed, p_var=w["p_var"],
                                n_clusters=w["n_clusters"], mu=w["mu"], p_N=w["p_N"], p_amb=w["p_amb"], gc=w["gc"], n_days=w["n_days"],
                                gaps=w["gaps"], dev_days=d_days.data_ptr(), site_offset=lo, L_total=L, packed=self.packed)
        self.days = d_days.cpu().numpy()
        self.bytes = n * self.pitch

    def row_masks(self, i):
        """4-bit masks of row i (host, numpy) -- for the in-bench parity spot checks."""
        row = self.buf[i * self.pitch:(i + 1) * self.pitch].cpu().numpy()
        if self.packed:
            m = np.empty(2 * row.size, np.uint8)
            m[0::2], m[1::2] = row & 15, row >> 4
            return m[:self.Ls]
        from tracs_b200.api import MASKS
        return MASKS[row[:self.Ls]]


def spot_checks(inp, res, dist, n_check=10, seed=0):
    """Parity evidence AT the benchmarked shape: some emitted edges and some random non-edges re-derived per site in
    NumPy from the two rows (d = #{s: m_i & m_j == 0}; compared sites = L - #{s: m_i or m_j is N}; src/pairsnp.hpp:398-419)."""
    rng = np.random.default_rng(seed)
    E = len(res["rows"])
    out = {"edges_checked": 0, "non_edges_checked": 0, "ok": True, "method": "per-site NumPy definition on the two rows"}
    if E == 0:
        return out
    key = (res["rows"].astype(np.uint64) << np.uint64(32)) | res["cols"].astype(np.uint64)
    for e in rng.integers(0, E, size=n_check).tolist():
        i, j = int(res["rows"][e]), int(res["cols"][e])
        mi, mj = inp.row_masks(i), inp.row_masks(j)
        d = int(((mi & mj) == 0).sum())
        nn = int(inp.Ls - ((mi == 15) | (mj == 15)).sum())
        good = d == int(res["dist"][e]) and nn == int(res["ncomp"][e]) and d <= dist
        out["ok"] = bool(out["ok"] and good)
        out["edges_checked"] += 1
    for _ in range(n_check):
        i, j = sorted(rng.integers(0, inp.n, size=2).tolist())
        if i == j:
            continue
        mi, mj = inp.row_masks(i), inp.row_masks(j)
        d = int(((mi & mj) == 0).sum())
        k = (np.uint64(i) << np.uint64(32)) | np.uint64(j)
        pos = int(np.searchsorted(key, k))
        listed = pos < E and key[pos] == k
        out["ok"] = bool(out["ok"] and (listed == (d <= dist)) and (not listed or int(res["dist"][pos]) == d))
        out["non_edges_checked"] += 1
    return out


# ------------------------------------------------------------------------------------------------
# rooflines
# ------------------------------------------------------------------------------------------------
def rooflines(tracs_b200, w, stats, peak, n_rows, L_slab, tc_peak, config=None, whole=True):
    """Per-kernel roofline entries from the library's stage timers (CUDA events on the call's stream)."""
    def avg(k):
        return float(np.mean([s[k] for s in stats]))
    hbm, hbm_src = hbm_peak()
    traffic = kernel_traffic(config) if whole else {}   # per-launch DRAM bytes only apply to the whole-alignment launch
    peak_wp = min(peak["lop3_per_s"] / 4.0, peak["popc_per_s"])
    packed = w["fmt"] == "packed"
    npitch_words = max(32, ((L_slab + 31) // 32 + 31) // 32 * 32)
    n_early = int(round(avg("n_early_sites")))
    n_main = n_rows - 256 if n_early else n_rows
    fam = "k_pack4" if packed else "k_pack"
    pack_kernel = (fam + ("<true>" if packed else "_x")) if n_early else (fam + ("<false>" if packed else ""))
    # algorithmic bytes (DESIGN 4): per base 1 B (ASCII) or 1/2 B (packed) read + 1/8 B N-plane write (+ summary byte per
    # 1024 sites); the extracting variant also writes one byte per (sample, early site)
    in_bytes = n_main * (L_slab // 2 if packed else L_slab)
    nplane_bytes = n_main * npitch_words * 4
    sparse_n = avg("sparse_nplane") > 0.5
    if sparse_n:
        # sparse N: only the 128-site blocks that hold an N are algorithmic output (16 B each; the kernel stores whole 32-byte
        # sectors). Expected share from the generator: i.i.d. N at p_N plus `gaps` runs of L/1000 sites per sample
        blocks = max(1, (L_slab + 127) // 128)
        f = 1.0 - (1.0 - w["p_N"]) ** 128
        f = min(1.0, f + w.get("gaps", 0) * ((w["L"] // 1000) / 128.0 + 1.0) / blocks)
        nplane_bytes = int(nplane_bytes * f)
    pack_bytes = in_bytes + nplane_bytes + n_main * (npitch_words // 32) + n_main * n_early
    ms_main = avg("ms_pack_main")
    roof_pack = {"bound": "hbm", "kernel": pack_kernel, "achieved": pack_bytes / (ms_main * 1e-3) / 1e9, "peak": hbm, "unit": "GB/s",
                 "frac": pack_bytes / (ms_main * 1e-3) / 1e9 / hbm, "traffic": traffic.get(pack_kernel),
                 "ms_per_launch": ms_main, "algorithmic_bytes": pack_bytes, "samples_in_launch": n_main, "early_sites": n_early,
                 "n_plane": "sparse stores (blocks that hold an N)" if sparse_n else "every word stored", "peak_source": hbm_src}
    wp = avg("swept_wordpairs")
    ms_sw = avg("ms_sweep")
    pf_words = int(round(wp / max(1.0, avg("n_pairs"))))
    prefiltered = (avg("n_candidates") > 0 or avg("ms_refine") > 0) and pf_words < int(round(avg("n_words")))
    what = "prefilter launch (first %d words of every pair)" % pf_words if prefiltered else "full-length sweep (%d words)" % pf_words
    if avg("tc_sweep") > 0.5:
        roof_sweep = tc_roof(wp, ms_sw, what, tc_peak, peak_wp, code=int(round(avg("tc_sweep"))))
    else:
        roof_sweep = int_roof(wp, ms_sw, what, peak, traffic)
    return roof_pack, roof_sweep, pack_kernel


TC_KERNELS = {1: "k_sweep_tc", 2: "k_sweep_tc2", 3: "k_sweep_tc3"}


def tc_roof(wordpairs, ms, what, tc_peak, peak_wp, code=33):
    """`code` = tracs_stats_t.tc_sweep: 10 * kernel generation + int8 operand planes executed per site."""
    macs = wordpairs * 32 * 4          # algorithmic: one-hot K = 4 per site (SURVEY 8d)
    gen, planes = divmod(int(code), 10)
    kernel = TC_KERNELS.get(gen, "k_sweep_tc") + ("<%d>" % planes if gen >= 2 else "")
    pk = tc_peak["tops"] if tc_peak else 4500.0
    return {"bound": "tensor", "kernel": kernel, "what": what, "achieved": 2 * macs / (ms * 1e-3) / 1e12, "peak": pk,
            "unit": "TOP/s", "frac": 2 * macs / (ms * 1e-3) / 1e12 / pk, "traffic": None, "ms_per_launch": ms,
            "executed_planes_per_site": planes, "executed_tops": 2 * macs * (planes / 4.0) / (ms * 1e-3) / 1e12,
            "peak_source": (tc_peak["source"] if tc_peak else "NOMINAL dense int8 (4.5 POP/s)"),
            "equivalent_int_pipe_frac": (wordpairs / (ms * 1e-3)) / peak_wp}


def int_roof(wordpairs, ms, what, peak, traffic):
    peak_wp = min(peak["lop3_per_s"] / 4.0, peak["popc_per_s"])
    return {"bound": "int_pipe", "kernel": "k_sweep", "what": what, "achieved": wordpairs * 6 / (ms * 1e-3) / 1e9,
            "peak": peak_wp * 6 / 1e9, "unit": "Ginstr/s", "frac": (wordpairs * 6 / (ms * 1e-3)) / (peak_wp * 6),
            "traffic": traffic.get("k_sweep_full_length") if what.startswith("full") else traffic.get("k_sweep_prefilter"),
            "achieved_wordpairs_per_s": wordpairs / (ms * 1e-3), "ms_per_launch": ms,
            "peak_source": "measured in this run (tracs_int_peak: register-resident LOP3 and POPC loops; a word-pair needs "
                           "4 LOP3 on the 64-lane ALU pipe and 1 POPC on the 16-lane XU pipe => min(lop3/4, popc) word-pairs/s)",
            "lop3_per_s": peak["lop3_per_s"], "popc_per_s": peak["popc_per_s"],
            "mix_wordpairs_per_s": peak["mix_wordpairs_per_s"], "mix_imad_wordpairs_per_s": peak["mix_imad_wordpairs_per_s"]}


def measured_tc_peak(tracs_b200):
    try:
        return tracs_b200.tc_peak()
    except Exception:
        return None


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
def main():
    saved_stdout = _claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="C3", choices=sorted(CONFIGS))
    ap.add_argument("--n", type=int, default=None, help="override sample count (debug only; invalidates the headline)")
    ap.add_argument("--L", type=int, default=None, help="override alignment length (debug only)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the forced full-length sweeps reported under roofline_kernels")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--profile-phases", action="store_true", help="N>1: one extra untimed step with per-phase host timers (stages_ms.phases_ms)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the edge columns of the last timed step as DIR/<name>.npy (float64, at most 64 MB: a seeded sample of "
                         "edges above that)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes what the CUDA path computed (--impl b200)")
    if args.n or args.L:
        for c in CONFIGS.values():
            if args.n:
                c["n_clusters"] = max(2, c["n_clusters"] * args.n // c["n"])
                c["n"] = args.n
            if args.L:
                c["L"] = args.L
    if args.impl == "reference":
        return run_reference(args, saved_stdout)
    args.warmup = max(args.warmup, 3)
    if args.config == "C1":
        from benchmarks import other_configs
        return other_configs.run_c1(args, saved_stdout, sys.modules[__name__])
    if args.config == "C4":
        from benchmarks import other_configs
        return other_configs.run_c4(args, saved_stdout, sys.modules[__name__])
    if args.config == "C5":
        from benchmarks import other_configs
        return other_configs.run_c5(args, saved_stdout, sys.modules[__name__])

    import torch
    import tracs_b200
    from tracs_b200 import _lib, sites

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; this framework has no CPU path")
    torch.cuda.set_device(local)
    _lib.check(_lib.lib().tracs_set_device(local))
    device = torch.device("cuda", local)
    cpu_affinity = bind_to_gpu_numa_node(local) if world > 1 else None
    dist_mod = None
    if world > 1:
        # keep NCCL's own banner / debug lines off stdout: the contract is ONE JSON line there
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        import torch.distributed as dist_mod
        dist_mod.init_process_group("nccl", device_id=device)

    w = CONFIGS[args.config]
    n, L = w["n"], w["L"]
    P = n * (n - 1) // 2
    strong = args.config == "C3" and world > 1
    replicas = world if (world > 1 and not strong) else 1

    # ---- synthetic input, generated in device memory ------------------------------------------
    if strong:
        lo, hi = sites.slab_bounds(L, rank, world)
        inp = Input(torch, tracs_b200, device, w, lo, hi)
    else:
        inp = Input(torch, tracs_b200, device, w, seed=w["seed"] + 1000 * rank if replicas > 1 else None)
    kw = dict(dist=w["dist"], days=inp.days, lamb=w["lamb"], beta=w["beta"], threshold_Ek=w["threshold_Ek"])
    peak = tracs_b200.int_peak() if rank == 0 else None
    tc_peak = measured_tc_peak(tracs_b200) if rank == 0 else None

    def step():
        if strong:
            return sites.sweep(torch, dist_mod, device, rank, world, inp.buf.data_ptr(), n, inp.Ls, inp.pitch, L, w["dist"], days=inp.days,
                               lamb=w["lamb"], beta=w["beta"], threshold_Ek=w["threshold_Ek"], packed=inp.packed)
        if inp.packed:
            res = tracs_b200.pairsnp_packed(inp.buf.data_ptr(), n, L, inp.pitch, copy=False, **kw)
        else:
            res = tracs_b200.pairsnp_device(inp.buf.data_ptr(), n, L, inp.pitch, copy=False, **kw)
        return res, tracs_b200.last_stats()

    def sync():
        torch.cuda.synchronize()
        if world > 1:
            dist_mod.barrier()
            torch.cuda.synchronize()

    def timed(fn, steps):
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        stats, res = [], None
        res, _ = fn()   # untimed: this loop's own result slot (the previous result stays alive while a call runs)
        sync()
        t0 = time.perf_counter()
        ev0.record()
        for _ in range(steps):
            res, st = fn()
            stats.append(st)
        ev1.record()
        sync()
        t_wall = time.perf_counter() - t0
        t_ms = torch.tensor([ev0.elapsed_time(ev1)], dtype=torch.float64, device=device)
        if world > 1:
            dist_mod.all_reduce(t_ms, op=dist_mod.ReduceOp.MAX)
        return float(t_ms.item()) / steps, t_wall / steps, stats, res

    clocks = Clocks(local)
    if rank == 0:
        clocks.start()
    for _ in range(args.warmup):
        res = step()   # one result held while the next call runs, like in the timed loop: the page-locked result-buffer cache
        #                reaches its steady state (two sets of columns) before the clock starts
    del res
    clocks.mark()
    ms_per_step, wall_per_step, stats, res = timed(step, args.steps)
    clk = clocks.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, edge_columns(res))
    value = replicas * P * L / (ms_per_step * 1e-3)

    def avg(k):
        return float(np.mean([s.get(k, 0) for s in stats]))

    line = None
    if rank == 0:
        n_edges = len(res["rows"])
        launches = int(sum(s["kernel_launches"] for s in stats))
        roof_pack, roof_sweep, pack_kernel = rooflines(tracs_b200, w, stats, peak, n, inp.Ls, tc_peak, config=args.config if not (args.n or args.L) else None, whole=(world == 1))
        keys = ("ms_pack", "ms_pack_main", "ms_compact", "ms_sweep", "ms_refine", "ms_sort", "ms_ncomp", "ms_trans", "ms_d2h", "ms_total",
                "ms_finish")
        stages = {k: avg(k) for k in keys}
        stages["n_candidates"] = avg("n_candidates_all") if strong else avg("n_candidates")
        stages["per_step_ms_total"] = [round(s_["ms_total"], 2) for s_ in stats]
        roof = roof_pack if avg("ms_pack_main") >= avg("ms_sweep") else roof_sweep
        kernels = {pack_kernel: roof_pack, "tile_sweep_as_launched": roof_sweep}
        line = {
            "metric": METRIC, "value": value, "unit": "site-pairs/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong" if args.config == "C3" else "weak",
            "vs_baseline": None, "dtype": DTYPE, "data": "synthetic (device-generated alignment, seeded)",
            "config": config_block(w, args.config, world),
            "details": {"variable_sites": int(stats[-1]["n_variable_sites"]), "words": int(stats[-1]["n_words"]), "edges": int(n_edges),
                        "bytes_resident_per_gpu": int(inp.bytes),
                        "algorithm": "exact filter-and-refine: tile sweep over the first words of every pair, per-pair completion of the "
                                     "survivors; roofline_kernels.*_full_length give the forced full-length tile sweeps"},
            "clocks": clk, "gpu_launches": launches, "roofline": roof, "roofline_kernels": kernels, "stages_ms": stages,
            "wall_ms_per_step": 1e3 * wall_per_step,
            "parity_spot_checks": spot_checks(inp, res, w["dist"]) if not strong else None,
        }
        if strong:
            line["collectives"] = ["ncclAllGather (candidate counts + keys)", "ncclReduceScatter (partial d, |N u N|)",
                                   "ncclAllGather (edge counts per slice)", "barrier (slices landed in the shared host table)"]
    if strong and args.profile_phases:
        _, stp = sites.sweep(torch, dist_mod, device, rank, world, inp.buf.data_ptr(), n, inp.Ls, inp.pitch, L, w["dist"], days=inp.days,
                             lamb=w["lamb"], beta=w["beta"], threshold_Ek=w["threshold_Ek"], packed=inp.packed, profile=True)
        if rank == 0:
            line["stages_ms"]["phases_ms_rank0"] = stp.get("phases_ms")
    # ---- the same tile kernels forced over the full length (what an unthresholded / dense run executes) ----------
    if rank == 0 and world == 1 and not args.no_extra:
        if True:
            for nm, variant in (("k_sweep_full_length", True), ("k_sweep_tc_full_length", "tc")):
                try:
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    fn = tracs_b200.pairsnp_packed if inp.packed else tracs_b200.pairsnp_device
                    r2 = fn(inp.buf.data_ptr(), n, L, inp.pitch, full_sweep=variant, copy=False, **kw)
                    torch.cuda.synchronize()
                    t_full = time.perf_counter() - t0
                    s2 = tracs_b200.last_stats()
                    rf = (tc_roof(s2["swept_wordpairs"], s2["ms_sweep"], "full-length sweep, tcgen05.mma kind::i8, operands expanded from the "
                                  "bit-planes in shared memory, int32 accumulators in TMEM", tc_peak,
                                  min(peak["lop3_per_s"] / 4.0, peak["popc_per_s"]), code=int(round(s2["tc_sweep"]))) if variant == "tc" else
                          int_roof(s2["swept_wordpairs"], s2["ms_sweep"], "full-length sweep (prefilter disabled)", peak,
                                   kernel_traffic(args.config if not (args.n or args.L) else None)))
                    rf["whole_step_ms"] = 1e3 * t_full
                    rf["edges_equal_default_path"] = bool(all(np.array_equal(r2[k], res[k]) for k in ("rows", "cols", "dist", "ncomp")))
                    kernels[nm] = rf
                    del r2
                except Exception as ex:
                    kernels[nm] = {"error": repr(ex)}

    # ---- e2e: the alignment starts in page-locked HOST memory; H2D of every rank's share + edge D2H inside the timed region ----
    if not args.no_e2e:
        e2e = {"value": None, "unit": "site-pairs/s", "h2d_bytes_per_step": None, "d2h_bytes_per_step": None}
        try:
            host_arr, host_note = pinned_on_gpu_node(local, inp.bytes, _lib) if world > 1 else (None, None)
            host = None
            if host_arr is not None:
                try:   # a first small round trip through the buffer; anything odd -> the plain page-locked allocation
                    host = torch.from_numpy(host_arr)
                    host[:4096].copy_(inp.buf.view(-1)[:4096])
                    torch.cuda.synchronize()
                except Exception as ex:
                    host, host_note = None, "numa-placed buffer unusable (%s): cudaHostAlloc instead" % type(ex).__name__
                    try:
                        _lib.lib().tracs_host_unregister(host_arr.ctypes.data)
                    except Exception:
                        pass
                    host_arr = None
            if host is None:
                host = torch.empty(inp.bytes, dtype=torch.uint8, pin_memory=True)
            e2e["host_buffer"] = host_note or "cudaHostAlloc"
            host.copy_(inp.buf.view(-1))
            torch.cuda.synchronize()
            hp = host.numpy()
            width = (inp.Ls + 1) // 2 if inp.packed else inp.Ls
            if strong:
                def e2e_step():
                    inp.buf.copy_(host, non_blocking=True)     # this rank's slab over this GPU's PCIe link
                    return step()
                api = "tracs_b200.sites.sweep on per-rank page-locked host slabs (H2D of the slab, then tracs_site_shard_open/partials/finish)"
            else:
                del inp.buf
                torch.cuda.empty_cache()
                o, keep = tracs_b200.api.make_opts(packed=inp.packed, **kw)

                def e2e_step():
                    e = _lib.Edges()
                    _lib.check(_lib.lib().tracs_pairsnp_host(hp.ctypes.data, n, L, inp.pitch, C.byref(o), C.byref(e)))
                    return _lib.take_edges(e, names=False, copy=False), tracs_b200.last_stats()
                api = "tracs_pairsnp_host (C ABI, page-locked host %s matrix) incl. fused transmission likelihood" % ("packed" if inp.packed else "ASCII")
            e2e_step()
            ms_e, wall_e, st_e, r2 = timed(e2e_step, args.e2e_steps)
            if rank == 0:
                e2e.update({"value": replicas * P * L / (ms_e * 1e-3), "ms_per_step": ms_e, "wall_ms_per_step": 1e3 * wall_e, "steps": args.e2e_steps,
                            "h2d_bytes_per_step": int(n * ((L + 1) // 2 if inp.packed else L)) if strong else int(n * width * replicas),
                            "d2h_bytes_per_step": int(st_e[-1].get("d2h_bytes", 0)), "host_memory": "pinned", "api": api,
                            "edges_equal_device_path": bool(all(np.array_equal(r2[k], res[k]) for k in ("rows", "cols", "dist", "ncomp")))})
            if host_arr is not None:
                try:
                    torch.cuda.synchronize()
                    _lib.lib().tracs_host_unregister(host_arr.ctypes.data)
                except Exception:
                    pass
            del host
        except Exception as ex:  # report, never fake
            e2e["error"] = repr(ex)
        if rank == 0:
            line["e2e"] = e2e
    elif rank == 0:
        line["e2e"] = {"value": None, "unit": "site-pairs/s", "h2d_bytes_per_step": None, "d2h_bytes_per_step": None, "note": "skipped (--no-e2e)"}

    # ---- cpu baseline beside it (rank 0, N=1) -----------------------------------------------------
    if rank == 0 and world == 1 and not args.no_cpu:
        try:
            mod, kind, what = load_reference()
            smp = RefSample(w)
            try:
                r = smp.step(mod, n_cores())
            finally:
                smp.cleanup()
            line["cpu_baseline"] = {"value": r["value"], "unit": "site-pairs/s", "cores": n_cores(), "kind": kind, "sample": smp.desc,
                                    "what": what, "projected": True, "pair_stage_site_pairs_per_s": r["pair_rate"],
                                    "load_bases_per_s": r["load_rate"]}
        except Exception as ex:
            line["cpu_baseline"] = {"value": None, "error": repr(ex)}
    elif rank == 0:
        line["cpu_baseline"] = {"value": None, "note": "timed at N=1 only"}

    if rank == 0:
        if cpu_affinity:
            line["cpu_affinity"] = cpu_affinity
        _emit(saved_stdout, line)
    if world > 1:
        dist_mod.barrier()
        dist_mod.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
