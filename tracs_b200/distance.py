"""Host-side mirror of the reference's `tracs distance` stage for the hot path: one pair sweep per
MSA (+ optional query-vs-database FASTA), optional TransCluster likelihood from sampling dates, one
CSV row per kept edge. Same options, column order and quirks as gtonkinhill/tracs
tracs/distance.py:15-259 (cited inline), written against the drop-in module's entry points so a
GPU box without the reference checkout can produce byte-comparable CSVs.

The reference's own tracs/distance.py also runs unchanged on top of tracs_b200/dropin/TRACS.py;
this module exists so the parity tests do not need /root/reference at run time."""
import argparse
import os
from datetime import date

import numpy as np

from . import api

SECONDS_IN_YEAR = 31556952.0  # tracs/transcluster.py:5
HEADER = ("sampleA,sampleB,date difference,SNP distance,transmission distance,expected K,"
          "filtered SNP distance,sites considered,MSA file\n")  # tracs/distance.py:156-158


def read_dates(path):
    """tracs/distance.py:145-151: skip the header line; column 0 = sample, column 1 = ISO date."""
    dates = {}
    with open(path) as f:
        next(f)
        for line in f:
            parts = line.strip().split(",")
            dates[parts[0]] = date.fromisoformat(parts[1])
    return dates


def date_differences(rows, cols, names, dates):
    """tracs/transcluster.py:26-33: seconds since 1970-01-01 for samples 0..max index (KeyError if
    one has no date), |t_i - t_j| / SECONDS_IN_YEAR."""
    epoch = date.fromisoformat("1970-01-01")
    top = int(max(max(rows), max(cols)))
    t = np.array([(dates[names[s]] - epoch).total_seconds() for s in range(top + 1)])
    return np.abs(t[np.asarray(rows, dtype=np.int64)] - t[np.asarray(cols, dtype=np.int64)]) / SECONDS_IN_YEAR


def _distance_native(msa_files, output_file, msa_db, dates, snp_threshold, recomb_filter, clock_rate, trans_rate, trans_threshold,
                     precision, n_cpu):
    """Same stage with the edge columns kept in C arrays end to end: tracs_pairsnp -> tracs_trans_dist ->
    tracs_write_distance_csv (no per-edge Python objects)."""
    import ctypes as C
    from . import _lib
    L = _lib.lib()
    for k, msa in enumerate(msa_files):
        fastas = [os.fspath(msa)] + ([os.fspath(msa_db)] if msa_db is not None else [])
        paths = (C.c_char_p * len(fastas))(*[os.fsencode(p) for p in fastas])
        e = _lib.Edges()
        _lib.check(L.tracs_pairsnp(paths, len(fastas), int(n_cpu), int(snp_threshold), int(bool(recomb_filter)), C.byref(e)))
        keep = []
        try:
            n = e.n_edges
            names = [e.names[i].decode() for i in range(e.n_names)]
            has_trans = dates is not None and n > 0
            if has_trans:
                rows = np.ctypeslib.as_array(e.rows, shape=(n,))
                cols = np.ctypeslib.as_array(e.cols, shape=(n,))
                src = np.ctypeslib.as_array(e.filt if recomb_filter else e.dist, shape=(n,))
                dt = np.ascontiguousarray(date_differences(rows, cols, names, dates), dtype=np.float64)
                p0, eK = api.trans_dist_np(src.astype(np.int32), dt, clock_rate, trans_rate, precision)
                keep = [dt, p0, eK]
                e.datediff = dt.ctypes.data_as(C.POINTER(C.c_double))
                e.p0_log = p0.ctypes.data_as(C.POINTER(C.c_double))
                e.eK = eK.ctypes.data_as(C.POINTER(C.c_double))
            ref = os.path.basename(msa).split(".")[0].replace("_combined", "")
            written = C.c_size_t(0)
            _lib.check(L.tracs_write_distance_csv(os.fsencode(output_file), int(k > 0), C.byref(e), e.names, e.n_names, ref.encode(),
                                                  int(has_trans), int(bool(recomb_filter)), int(trans_threshold is not None),
                                                  float(trans_threshold if trans_threshold is not None else 0.0), C.byref(written)))
        finally:
            # the likelihood columns are NumPy-owned: detach them before the library frees its own arrays
            e.datediff = e.p0_log = e.eK = C.POINTER(C.c_double)()
            L.tracs_edges_free(C.byref(e))
            del keep


def distance(msa_files, output_file, msa_db=None, metadata=None, snp_threshold=2147483647, recomb_filter=False,
             clock_rate=1e-3 * 29903, trans_rate=73.0, trans_threshold=None, precision=0.01, n_cpu=1, native_csv=False):
    dates = read_dates(metadata) if metadata is not None else None
    if native_csv:
        return _distance_native(msa_files, output_file, msa_db, dates, snp_threshold, recomb_filter, clock_rate, trans_rate,
                                trans_threshold, precision, n_cpu)
    with open(output_file, "w") as out:
        out.write(HEADER)
        for msa in msa_files:
            fastas = [msa, msa_db] if msa_db is not None else [msa]
            rows, cols, snp, names, filt, ncomp = api.pairsnp(fasta=fastas, n_threads=n_cpu, dist=snp_threshold, filter=recomb_filter)
            write_rows(out, msa, rows, cols, snp, names, filt, ncomp, dates, recomb_filter, clock_rate, trans_rate, trans_threshold,
                       precision)


def write_rows(out, msa, rows, cols, snp, names, filt, ncomp, dates, recomb_filter, clock_rate, trans_rate, trans_threshold, precision):
    """The CSV rows of one MSA's edge lists (lists, in (row, col) order; names indexed by rows / cols) into the open file."""
    ref = os.path.basename(msa).split(".")[0].replace("_combined", "")  # tracs/distance.py:208-209
    if dates is not None and len(rows) > 0:
        dt = date_differences(rows, cols, names, dates)
        # with the filter on, the likelihood is fed the filtered distance (tracs/distance.py:182-192)
        p0, eK = api.trans_dist(filt if recomb_filter else snp, dt, clock_rate, trans_rate, precision)
        p0 = np.exp(np.asarray(p0))  # tracs/transcluster.py:38-39
        filt_col = filt if recomb_filter else ["NA"] * len(rows)  # tracs/distance.py:204
        for e in range(len(rows)):
            if trans_threshold is None or trans_threshold >= eK[e]:  # tracs/distance.py:222
                out.write(",".join([names[rows[e]], names[cols[e]], str(dt[e]), str(int(snp[e])), str(p0[e]), str(eK[e]),
                                    str(filt_col[e]), str(ncomp[e]), ref]) + "\n")
    else:
        for e in range(len(rows)):  # tracs/distance.py:239-258
            out.write(",".join([names[rows[e]], names[cols[e]], "NA", str(int(snp[e])), "NA", "NA", str(filt[e]), str(ncomp[e]),
                                ref]) + "\n")


def main(argv=None):
    ap = argparse.ArgumentParser(description="Pairwise SNP and transmission distances (B200)")
    ap.add_argument("--msa", dest="msa_files", required=True, nargs="+")
    ap.add_argument("--msa-db", dest="msa_db", default=None)
    ap.add_argument("--meta", dest="metadata", default=None)
    ap.add_argument("-o", "--output", dest="output_file", required=True)
    ap.add_argument("-D", "--snp_threshold", type=int, default=2147483647)
    ap.add_argument("--filter", dest="recomb_filter", action="store_true")
    ap.add_argument("--clock_rate", type=float, default=1e-3 * 29903)
    ap.add_argument("--trans_rate", type=float, default=73.0)
    ap.add_argument("-K", "--trans_threshold", type=float, default=None)
    ap.add_argument("--precision", type=float, default=0.01)
    ap.add_argument("-t", "--threads", dest="n_cpu", type=int, default=1)
    ap.add_argument("--native-csv", dest="native_csv", action="store_true", help="write the CSV from C (no per-edge Python objects)")
    a = ap.parse_args(argv)
    distance(**vars(a))


if __name__ == "__main__":
    main()


def min_over_references(per_msa, column="dist"):
    """Min-over-references combine (SURVEY A.6). The reference only realises it implicitly: one CSV row
    per (pair, MSA) (tracs/distance.py:159-258) and tracs/cluster.py:104-113 links a pair if ANY row is
    under the threshold, i.e. min over MSAs <= threshold.

    per_msa: iterable of (names, rows, cols, values) per reference MSA (indices into that MSA's names).
    Returns (nameA, nameB, value) lists: one entry per unordered sample-name pair, value = min over the
    MSAs that contain the pair, sorted by the order names were first seen. Runs on the GPU
    (tracs_min_over_refs: radix sort + reduce-by-key)."""
    ids = {}
    a_all, b_all, v_all = [], [], []
    for names, rows, cols, values in per_msa:
        gid = np.array([ids.setdefault(nm, len(ids)) for nm in names], dtype=np.uint64)
        if len(rows):
            a_all.append(gid[np.asarray(rows, dtype=np.int64)])
            b_all.append(gid[np.asarray(cols, dtype=np.int64)])
            v_all.append(np.asarray(values, dtype=np.float64))
    if not a_all:
        return [], [], []
    oa, ob, ov = api.min_over_refs(np.concatenate(a_all), np.concatenate(b_all), np.concatenate(v_all))
    inv = [None] * len(ids)
    for nm, k in ids.items():
        inv[k] = nm
    return [inv[int(x)] for x in oa], [inv[int(x)] for x in ob], ov.tolist()
