"""Host-side mirror of the reference's native interface for the pairwise-distance hot path.

Same names, argument meaning and error behaviour as the pybind11 module `TRACS` of
gtonkinhill/tracs (src/python_bindings.cpp:8-26); everything executes in libtracs_b200.so."""
import ctypes as C
import os

import numpy as np

from . import _lib
from ._lib import INT32_MAX, Opts, Edges


def pairsnp(fasta, n_threads, dist, filter):
    """TRACS.pairsnp (src/python_bindings.cpp:12-13; src/pairsnp.hpp:320-458).

    fasta: list of 1 or 2 FASTA(.gz) paths; returns the 6-tuple of Python lists
    (rows, cols, distances, seq_names, filt_distances, n_compared_sites) in (row, col) order."""
    fasta = [os.fspath(p) for p in fasta]
    paths = (C.c_char_p * max(1, len(fasta)))(*[os.fsencode(p) for p in fasta])
    e = Edges()
    try:
        _lib.check(_lib.lib().tracs_pairsnp(paths, len(fasta), int(n_threads), int(dist), int(bool(filter)), C.byref(e)))
    except KeyboardInterrupt:
        # the reference prints this and calls exit(1) from inside the extension (src/pairsnp.hpp:207-214, 434-441)
        import sys
        sys.stderr.write("Interrupted by user!\n")
        raise SystemExit(1)
    r = _lib.take_edges(e, as_lists=True)
    return (r["rows"], r["cols"], r["dist"], r["names"], r["filt"], r["ncomp"])


def trans_dist(snpdiff, datediff, lamb, beta, threshold_Ek):
    """TRACS.trans_dist (src/python_bindings.cpp:19-21; src/transcluster.hpp:240-287).
    Returns (log p0 list, E[K] list)."""
    p0, eK = trans_dist_np(snpdiff, datediff, lamb, beta, threshold_Ek)
    return p0.tolist(), eK.tolist()


def trans_dist_np(snpdiff, datediff, lamb, beta, threshold_Ek):
    """trans_dist returning NumPy arrays (no list conversion)."""
    snp = np.ascontiguousarray(snpdiff, dtype=np.int32)
    dt = np.ascontiguousarray(datediff, dtype=np.float64)
    if snp.shape != dt.shape:
        # the reference indexes datediff[i] for i < len(snpdiff) (src/transcluster.hpp:263-265)
        raise IndexError("snpdiff and datediff must have the same length")
    n = snp.size
    p0 = np.empty(n, np.float64)
    eK = np.empty(n, np.float64)
    _lib.check(_lib.lib().tracs_trans_dist(snp.ctypes.data, dt.ctypes.data, n, float(lamb), float(beta), float(threshold_Ek),
                                          p0.ctypes.data, eK.ctypes.data))
    return p0, eK


def lprob_k_given_N(N, k, delta, lamb, beta, lgamma):
    """TRACS.lprob_k_given_N (src/python_bindings.cpp:15-17; src/transcluster.hpp:90-129)."""
    lg = np.ascontiguousarray(lgamma, dtype=np.float64)
    out = np.empty(2, np.float64)
    _lib.check(_lib.lib().tracs_lprob_k_given_N(int(N), int(k), float(delta), float(lamb), float(beta), lg.ctypes.data, lg.size,
                                               out.ctypes.data))
    return float(out[0]), float(out[1])


def calculate_posteriors(counts, alphas, keep, threshold):
    """TRACS.calculate_posteriors (src/python_bindings.cpp:23-25; src/dmultinomial.hpp:8-86)."""
    c = np.ascontiguousarray(counts, dtype=np.float64)
    if c.ndim != 2:
        raise RuntimeError("counts must be a 2-D array")
    a = np.ascontiguousarray(alphas, dtype=np.float64)
    out = np.empty_like(c)
    _lib.check(_lib.lib().tracs_calculate_posteriors(c.ctypes.data, c.shape[0], c.shape[1], a.ctypes.data, a.size, int(bool(keep)),
                                                    float(threshold), out.ctypes.data))
    return out


# ---- extras (not in the reference module) ------------------------------------------------------

def make_opts(dist=INT32_MAX, i_end=0, j_start=0, shard_rank=0, shard_world=1, want_ncomp=True, days=None, lamb=29.903,
              beta=73.0, threshold_Ek=0.01, filter=False, full_sweep=False, keep_on_device=False, packed=False):
    o = Opts()
    o.dist = int(dist)
    o.filter = int(bool(filter))
    o.i_end = int(i_end)
    o.j_start = int(j_start)
    o.shard_rank = int(shard_rank)
    o.shard_world = int(shard_world)
    o.want_ncomp = int(bool(want_ncomp))
    o.sweep_variant = 2 if full_sweep == "tc" else (1 if full_sweep else 0)
    o.keep_on_device = int(bool(keep_on_device))
    o.packed_input = int(bool(packed))
    keep = None
    if days is not None:
        keep = np.ascontiguousarray(days, dtype=np.int32)
        o.days = keep.ctypes.data_as(C.POINTER(C.c_int32))
        o.want_trans = 1
    o.lamb, o.beta, o.threshold_Ek = float(lamb), float(beta), float(threshold_Ek)
    return o, keep


def pairsnp_matrix(seqs, copy=True, **kw):
    """Pair sweep on a HOST ASCII matrix uint8[n][L] (the bytes load_seqs holds per record);
    H2D copy included. Returns a dict of numpy arrays (rows, cols, dist, ncomp[, p0_log, eK, datediff])."""
    seqs = np.ascontiguousarray(seqs, dtype=np.uint8)
    n, L = seqs.shape
    o, keep = make_opts(**kw)
    e = Edges()
    _lib.check(_lib.lib().tracs_pairsnp_host(seqs.ctypes.data, n, L, L, C.byref(o), C.byref(e)))
    return _lib.take_edges(e, names=False, copy=copy)


def pairsnp_device(dev_ptr, n, L, pitch, copy=True, **kw):
    """Pair sweep on a DEVICE-resident ASCII matrix (raw device pointer as int)."""
    o, keep = make_opts(**kw)
    e = Edges()
    _lib.check(_lib.lib().tracs_pairsnp_device(C.c_void_p(dev_ptr), n, L, pitch, C.byref(o), C.byref(e)))
    return _lib.take_edges(e, names=False, copy=copy)


MASKS = np.full(256, 15, np.uint8)
for _c, _m in zip("ACGTMRWSYKVHDB", (1, 2, 4, 8, 3, 5, 9, 6, 10, 12, 7, 11, 13, 14)):
    MASKS[ord(_c)] = MASKS[ord(_c.lower())] = _m


def pack_nibbles(seqs):
    """Host helper: ASCII matrix uint8[n][L] -> 4-bit packed rows uint8[n][pitch] in the layout
    tracs_pairsnp_packed takes (site s in byte s >> 1, low nibble first; pitch a multiple of 16 bytes holding L rounded
    up to 32 sites; padding sites = 1111). The nibble is the base mask of src/pairsnp.hpp:107-199."""
    seqs = np.ascontiguousarray(seqs, dtype=np.uint8)
    n, L = seqs.shape
    pitch = max(16, (L + 31) // 32 * 16)
    m = np.full((n, pitch * 2), 15, np.uint8)
    m[:, :L] = MASKS[seqs]
    return (m[:, 0::2] | (m[:, 1::2] << 4)).astype(np.uint8), pitch


def pairsnp_packed_host(nib, L, copy=True, **kw):
    """Pair sweep on a HOST matrix of 4-bit packed rows (pack_nibbles layout); H2D copy included."""
    nib = np.ascontiguousarray(nib, dtype=np.uint8)
    n, pitch = nib.shape
    o, keep = make_opts(packed=True, **kw)
    e = Edges()
    _lib.check(_lib.lib().tracs_pairsnp_host(nib.ctypes.data, n, L, pitch, C.byref(o), C.byref(e)))
    return _lib.take_edges(e, names=False, copy=copy)


def pairsnp_packed(dev_ptr, n, L, pitch_bytes, copy=True, **kw):
    """Pair sweep on a DEVICE-resident 4-bit packed alignment (raw device pointer as int)."""
    o, keep = make_opts(**kw)
    e = Edges()
    _lib.check(_lib.lib().tracs_pairsnp_packed(C.c_void_p(dev_ptr), n, L, pitch_bytes, C.byref(o), C.byref(e)))
    return _lib.take_edges(e, names=False, copy=copy)


def _dense_opts(n, n_query, packed, full_sweep):
    """Options of the dense entry points: the square n x n matrix, or with n_query = q the q x (n - q) rectangle
    (rows = samples [0, q), columns = samples [q, n)). Returns (opts, rows, cols)."""
    if n_query is None:
        return make_opts(packed=packed, full_sweep=full_sweep)[0], n, n
    q = int(n_query)
    if not 0 < q < n:
        raise ValueError("n_query must satisfy 0 < n_query < n (rows = samples [0, n_query), columns = samples [n_query, n))")
    return make_opts(i_end=q, j_start=q, packed=packed, full_sweep=full_sweep)[0], q, n - q


def distance_matrix(seqs, n_query=None, packed=False, L=None, full_sweep=False):
    """All-pairs SNP distances of a HOST alignment as a numpy int32 matrix: the `dist` column of pairsnp_* with
    dist = INT32_MAX, for every pair. seqs: ASCII uint8[n][L], or with packed=True pack_nibbles rows (then L is
    required). Square n x n (symmetric, zero diagonal), or with n_query = q the q x (n - q) query x db rectangle.
    full_sweep: 0/False = tensor cores when the masks allow them, True = LOP3/POPC kernel, "tc" = tensor cores required."""
    seqs = np.ascontiguousarray(seqs, dtype=np.uint8)
    if seqs.ndim != 2:
        raise ValueError("seqs must be a 2-D uint8 matrix")
    n, width = seqs.shape
    if packed and L is None:
        raise ValueError("L (sites) is required with packed=True")
    L = width if L is None else int(L)
    o, rows, cols = _dense_opts(n, n_query, packed, full_sweep)
    out = np.empty((rows, cols), np.int32)
    _lib.check(_lib.lib().tracs_distance_matrix_host(seqs.ctypes.data, n, L, width, C.byref(o), out.ctypes.data, cols))
    return out


def distance_matrix_device(dev_ptr, n, L, pitch, out_ptr, ld, n_query=None, packed=False, full_sweep=False):
    """All-pairs SNP distances of a DEVICE-resident alignment (ASCII, or 4-bit packed with packed=True) written into a
    caller's device int32 buffer out_ptr (row r at out_ptr + 4 * r * ld), e.g. a torch int32 tensor's data_ptr().
    Shapes as distance_matrix; padding columns (ld > cols) are not written."""
    o, _, _ = _dense_opts(int(n), n_query, packed, full_sweep)
    _lib.check(_lib.lib().tracs_distance_matrix_device(C.c_void_p(dev_ptr), int(n), int(L), int(pitch), C.byref(o), C.c_void_p(out_ptr),
                                                       int(ld)))


def write_distance_matrix(path, m, row_names, col_names, sep="\t", n_threads=None):
    """Writes an int32 matrix as text through the native writer: a header line (an empty cell, then the column names),
    then one line per row (its name, then the values). sep is "\\t" or ","; names are written as given. A row-strided
    view (m = big[:, :cols]) is written without a copy. n_threads: formatting threads (the output does not depend on it)."""
    m = np.asarray(m)
    if m.ndim != 2:
        raise ValueError("m must be a 2-D matrix")
    if m.dtype != np.int32 or m.strides[1] != 4 or m.strides[0] % 4 or m.strides[0] < 4 * m.shape[1]:
        m = np.ascontiguousarray(m, dtype=np.int32)
    rows, cols = m.shape
    ld = max(cols, m.strides[0] // 4) if rows > 1 else cols
    if len(row_names) != rows or len(col_names) != cols:
        raise ValueError("need one name per row (%d) and per column (%d)" % (rows, cols))
    rn = (C.c_char_p * max(1, rows))(*[str(s).encode() for s in row_names])
    cn = (C.c_char_p * max(1, cols))(*[str(s).encode() for s in col_names])
    old = os.environ.get("TRACS_WRITE_THREADS")
    if n_threads is not None:
        os.environ["TRACS_WRITE_THREADS"] = str(int(n_threads))
    try:
        _lib.check(_lib.lib().tracs_write_distance_matrix(os.fsencode(os.fspath(path)), m.ctypes.data, rows, cols, ld, rn, cn,
                                                          sep.encode()))
    finally:
        if n_threads is not None:
            if old is None:
                os.environ.pop("TRACS_WRITE_THREADS", None)
            else:
                os.environ["TRACS_WRITE_THREADS"] = old


class Database:
    """A sample collection ingested once and kept on the GPU, against which batches of new samples are placed: the two-file
    (query x db) mode of pairsnp without ingesting the database again on every call.

    query(q) returns exactly what pairsnp_matrix(concatenate([q, db]), i_end=nq, j_start=nq) returns: the same columns in the
    same order, rows = query index in [0, nq), cols = nq + database index. `days` (for the transmission likelihood) covers
    the queries first, then the database. Not supported: the recombination filter, query x query pairs.

    append(b) adds the batch to the database and returns exactly what pairsnp_matrix(concatenate([db, b]), j_start=n_db)
    returns: every pair with a sample in the batch, indexed in the grown collection (the batch is n_db .. n_db + m - 1).
    Afterwards the database is [db; b]; an append that raises leaves it as it was.

    Database(seqs) copies a host matrix (ASCII uint8[n][L], or pack_nibbles rows with packed=True and L) into device memory
    the handle owns. Use it as a context manager, or close() it, to release that memory."""

    def __init__(self, seqs=None, packed=False, L=None, _handle=None, _keep=None):
        self._h = None
        self._keep = _keep
        self.names = None
        if _handle is not None:
            self._h = _handle
        else:
            seqs = np.ascontiguousarray(seqs, dtype=np.uint8)
            if seqs.ndim != 2:
                raise ValueError("seqs must be a 2-D uint8 matrix")
            n, width = seqs.shape
            if packed and L is None:
                raise ValueError("L (sites) is required with packed=True")
            L = width if L is None else int(L)
            o, _ = make_opts(packed=packed)
            h = C.c_void_p()
            _lib.check(_lib.lib().tracs_db_open_host(seqs.ctypes.data, n, L, width, C.byref(o), C.byref(h)))
            self._h = h.value
        self.n, self.L = self.info()["n"], self.info()["L"]

    @classmethod
    def from_device(cls, ptr, n, L, pitch, packed=False):
        """A database over a DEVICE buffer (raw pointer as int; ASCII rows, or 4-bit rows with packed=True). A 4-bit buffer is
        BORROWED, not copied: it must stay allocated and unchanged until close(); the library never writes to it. ASCII rows are
        encoded once into 4-bit rows the handle owns, and the buffer is not kept."""
        o, _ = make_opts(packed=packed)
        h = C.c_void_p()
        _lib.check(_lib.lib().tracs_db_open_device(C.c_void_p(ptr), int(n), int(L), int(pitch), C.byref(o), C.byref(h)))
        return cls(_handle=h.value)

    @classmethod
    def from_fasta(cls, path, n_threads=1):
        """A database from a FASTA(.gz) file (read into host memory first with read_fasta); keeps the sample names."""
        seqs, names = read_fasta(path, n_threads)
        db = cls(seqs)
        db.names = names
        return db

    def _opts(self, dist, days, want_ncomp, full_sweep, packed, nq):
        if days is not None and len(days) != nq + self.n:
            raise ValueError("days must hold nq + n_db = %d values (queries first, then the database)" % (nq + self.n))
        return make_opts(dist=dist, days=days, want_ncomp=want_ncomp, full_sweep=full_sweep, packed=packed)

    def query(self, seqs, dist=INT32_MAX, days=None, want_ncomp=True, full_sweep=False, packed=False, L=None):
        """Edges between the HOST query rows (ASCII uint8[nq][L], or pack_nibbles rows with packed=True) and the database,
        as the dict of pairsnp_matrix."""
        seqs = np.ascontiguousarray(seqs, dtype=np.uint8)
        if seqs.ndim != 2:
            raise ValueError("seqs must be a 2-D uint8 matrix")
        nq, width = seqs.shape
        L = (width if not packed else self.L) if L is None else int(L)
        if L != self.L:
            raise ValueError("query L (%d sites) differs from the database's L (%d sites)" % (L, self.L))
        o, keep = self._opts(dist, days, want_ncomp, full_sweep, packed, nq)
        e = Edges()
        _lib.check(_lib.lib().tracs_db_query_host(C.c_void_p(self._handle()), seqs.ctypes.data, nq, width, C.byref(o), C.byref(e)))
        return _lib.take_edges(e, names=False)

    def query_device(self, ptr, nq, pitch, dist=INT32_MAX, days=None, want_ncomp=True, full_sweep=False, packed=False):
        """query() on DEVICE query rows (raw pointer as int; ASCII rows, or 4-bit rows with packed=True) of the database's L."""
        o, keep = self._opts(dist, days, want_ncomp, full_sweep, packed, int(nq))
        e = Edges()
        _lib.check(_lib.lib().tracs_db_query_device(C.c_void_p(self._handle()), C.c_void_p(ptr), int(nq), int(pitch), C.byref(o), C.byref(e)))
        return _lib.take_edges(e, names=False)

    def _append_opts(self, dist, days, want_ncomp, full_sweep, packed, m, names):
        if days is not None and len(days) != self.n + m:
            raise ValueError("days must hold n_db + m = %d values (the database first, then the batch)" % (self.n + m))
        if self.names is not None and (names is None or len(names) != m):
            raise ValueError("the database has sample names: give one name per appended sample (%d)" % m)
        if self.names is None and names is not None:
            raise ValueError("the database has no sample names to extend")
        return make_opts(dist=dist, days=days, want_ncomp=want_ncomp, full_sweep=full_sweep, packed=packed)

    def _appended(self, e, m, names):
        r = _lib.take_edges(e, names=False)
        self.n += m
        if names is not None:
            self.names = self.names + list(names)
        return r

    def append(self, seqs, dist=INT32_MAX, days=None, want_ncomp=True, full_sweep=False, packed=False, L=None, names=None):
        """Adds the HOST rows (ASCII uint8[m][L], or pack_nibbles rows with packed=True) to the database and returns the edges
        of every pair with a sample in the batch, as the dict of pairsnp_matrix, indexed in the grown collection. `days`:
        n_db + m values, the database first. `names`: one per appended sample, required when the database has names
        (from_fasta), which it then extends."""
        seqs = np.ascontiguousarray(seqs, dtype=np.uint8)
        if seqs.ndim != 2:
            raise ValueError("seqs must be a 2-D uint8 matrix")
        m, width = seqs.shape
        L = (width if not packed else self.L) if L is None else int(L)
        if L != self.L:
            raise ValueError("appended L (%d sites) differs from the database's L (%d sites)" % (L, self.L))
        o, keep = self._append_opts(dist, days, want_ncomp, full_sweep, packed, m, names)
        e = Edges()
        _lib.check(_lib.lib().tracs_db_append_host(C.c_void_p(self._handle()), seqs.ctypes.data, m, width, C.byref(o), C.byref(e)))
        return self._appended(e, m, names)

    def append_device(self, ptr, m, pitch, dist=INT32_MAX, days=None, want_ncomp=True, full_sweep=False, packed=False, names=None):
        """append() of DEVICE rows (raw pointer as int; ASCII rows, or 4-bit rows with packed=True) of the database's L. The
        rows are copied: the buffer is not kept."""
        o, keep = self._append_opts(dist, days, want_ncomp, full_sweep, packed, int(m), names)
        e = Edges()
        _lib.check(_lib.lib().tracs_db_append_device(C.c_void_p(self._handle()), C.c_void_p(ptr), int(m), int(pitch), C.byref(o), C.byref(e)))
        return self._appended(e, int(m), names)

    def info(self):
        """n, L, n_variable_sites (of the database), device, bytes_held, query_rows (swept at once) and new_sites (sites
        that the last query or appended batch made variable)."""
        i = _lib.DbInfo()
        _lib.check(_lib.lib().tracs_db_info(C.c_void_p(self._handle()), C.byref(i)))
        return i.as_dict()

    def _handle(self):
        if self._h is None:
            raise RuntimeError("database: the handle is closed")
        return self._h

    def close(self):
        """Releases the device memory the handle holds (a borrowed buffer stays the caller's). Closing twice is harmless."""
        if self._h is not None:
            h, self._h = self._h, None
            _lib.check(_lib.lib().tracs_db_close(C.c_void_p(h)))

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def min_over_refs(a, b, val):
    """Min-over-references combine (SURVEY A.6): unordered (a,b) -> min(val). Sorted by (lo, hi)."""
    a = np.ascontiguousarray(a, dtype=np.uint64)
    b = np.ascontiguousarray(b, dtype=np.uint64)
    v = np.ascontiguousarray(val, dtype=np.float64)
    n = a.size
    oa = np.empty(n, np.uint64)
    ob = np.empty(n, np.uint64)
    ov = np.empty(n, np.float64)
    m = C.c_size_t(0)
    _lib.check(_lib.lib().tracs_min_over_refs(a.ctypes.data, b.ctypes.data, v.ctypes.data, n, oa.ctypes.data, ob.ctypes.data,
                                             ov.ctypes.data, C.byref(m)))
    return oa[:m.value].copy(), ob[:m.value].copy(), ov[:m.value].copy()


def synth_device(dev_ptr, n, L, pitch, seed=1, p_var=0.01, n_clusters=20, mu=5.0, p_N=1e-3, p_amb=0.0, gc=0.5, n_days=180,
                 gaps=2, dev_days=None, site_offset=0, L_total=0, packed=False):
    """Seeded synthetic alignment written straight into device memory. With site_offset / L_total the
    buffer receives the column slab [site_offset, site_offset + L) of an L_total-site alignment
    (identical bytes to the corresponding columns of the whole alignment). packed=True writes 4-bit masks
    (tracs_pairsnp_packed layout; `pitch` = bytes per packed row) of the same alignment."""
    cfg = _lib.Synth(n, L, pitch, seed, p_var, n_clusters, mu, p_N, p_amb, gc, n_days, gaps, site_offset, L_total, int(bool(packed)), 0)
    _lib.check(_lib.lib().tracs_synth_device(C.byref(cfg), C.c_void_p(dev_ptr), C.c_void_p(dev_days) if dev_days else None))


def connected_components(a, b, n_nodes):
    """Labels of the connected components of an undirected edge list, numbered like
    scipy.sparse.csgraph.connected_components. Returns (n_components, labels uint32[n_nodes])."""
    a = np.ascontiguousarray(a, dtype=np.uint64)
    b = np.ascontiguousarray(b, dtype=np.uint64)
    labels = np.zeros(int(n_nodes), np.uint32)
    nc = C.c_size_t(0)
    _lib.check(_lib.lib().tracs_connected_components(a.ctypes.data, b.ctypes.data, a.size, int(n_nodes), labels.ctypes.data, C.byref(nc)))
    return nc.value, labels


def read_fasta(path, n_threads=1):
    """FASTA/FASTQ(.gz) -> (uint8[n][L] ASCII matrix, names). Host only (the loader half of pairsnp)."""
    seqs = C.POINTER(C.c_uint8)()
    names = C.POINTER(C.c_char_p)()
    n, L = C.c_size_t(0), C.c_size_t(0)
    _lib.check(_lib.lib().tracs_read_fasta(os.fsencode(os.fspath(path)), int(n_threads), C.byref(seqs), C.byref(n), C.byref(L), C.byref(names)))
    try:
        if n.value and L.value:
            a = np.ctypeslib.as_array(seqs, shape=(n.value * L.value,)).reshape(n.value, L.value).copy()
        else:
            a = np.zeros((n.value, L.value), np.uint8)
        nm = [names[i].decode() for i in range(n.value)]
    finally:
        _lib.lib().tracs_free_fasta(seqs, names, n.value)
    return a, nm


def shard_rowblocks(n_rowblocks, world, rank):
    out = np.zeros(max(1, n_rowblocks), np.uint32)
    k = C.c_uint32(0)
    _lib.check(_lib.lib().tracs_shard_rowblocks(n_rowblocks, world, rank, out.ctypes.data, C.byref(k)))
    return out[:k.value].copy()


def int_peak():
    out = np.zeros(8, np.float64)
    _lib.check(_lib.lib().tracs_int_peak(out.ctypes.data))
    return {"lop3_per_s": out[0], "popc_per_s": out[1], "iadd_per_s": out[2], "mix_wordpairs_per_s": out[3],
            "mix_imad_wordpairs_per_s": out[4], "n_sm": int(out[5])}


def tc_peak():
    """Measured int8 tensor-pipe peak (tracs_tc_peak): back-to-back tcgen05.mma kind::i8 on every SM."""
    out = np.zeros(4, np.float64)
    _lib.check(_lib.lib().tracs_tc_peak(out.ctypes.data))
    return {"tops": float(max(out[0], out[1])), "tops_n128": float(out[0]), "tops_n256": float(out[1]), "clk_per_mma_n128": float(out[2]),
            "clk_per_mma_n256": float(out[3]),
            "source": "measured in this run (tracs_tc_peak: back-to-back tcgen05.mma kind::i8 M128 K32 on all SMs, N = 128 / 256, best shape)"}


def tc_peak_sustained(seconds=2.0):
    """The tensor-pipe probe held for `seconds`: TOP/s over the second half of the run (power-capped steady state)."""
    out = np.zeros(2, np.float64)
    _lib.check(_lib.lib().tracs_tc_peak_sustained(C.c_double(seconds), out.ctypes.data))
    return {"tops": float(out[0]), "tops_whole_run": float(out[1]), "seconds": float(seconds),
            "source": "measured in this run (tracs_tc_peak_sustained: back-to-back tcgen05.mma kind::i8 M128 N256 K32 on all SMs "
                      "held for %.1f s, second half: the rate under the board's power cap)" % seconds}


def last_stats():
    return _lib.last_stats()
