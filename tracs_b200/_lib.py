"""ctypes binding of libtracs_b200.so (the C ABI declared in include/tracs_b200.h).

There is no CPU fallback: if the shared library is missing or no CUDA device is usable, the
compute entry points raise."""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libtracs_b200.so")

INT32_MAX = 2147483647


class Edges(C.Structure):
    _fields_ = [("n_edges", C.c_size_t), ("rows", C.POINTER(C.c_uint64)), ("cols", C.POINTER(C.c_uint64)),
                ("dist", C.POINTER(C.c_uint64)), ("filt", C.POINTER(C.c_uint64)), ("ncomp", C.POINTER(C.c_uint64)),
                ("p0_log", C.POINTER(C.c_double)), ("eK", C.POINTER(C.c_double)), ("datediff", C.POINTER(C.c_double)),
                ("n_names", C.c_size_t), ("names", C.POINTER(C.c_char_p)), ("seq_length", C.c_uint64),
                ("dev_packed", C.c_void_p), ("dev_packed_bytes", C.c_size_t)]


class Stats(C.Structure):
    _fields_ = [(k, C.c_uint64) for k in ("n_samples", "seq_length", "n_variable_sites", "n_words", "n_tiles", "n_pairs",
                                          "n_edges", "kernel_launches", "h2d_bytes", "d2h_bytes", "n_candidates",
                                          "swept_wordpairs", "n_early_sites")] + \
               [(k, C.c_float) for k in ("ms_pack", "ms_compact", "ms_sweep", "ms_refine", "ms_sort", "ms_ncomp", "ms_trans", "ms_total", "ms_d2h", "ms_filter", "tc_sweep", "ms_pack_main", "sparse_nplane", "reserved0")]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class Opts(C.Structure):
    _fields_ = [("dist", C.c_int32), ("filter", C.c_int32), ("i_end", C.c_uint64), ("j_start", C.c_uint64),
                ("shard_rank", C.c_int32), ("shard_world", C.c_int32), ("want_ncomp", C.c_int32),
                ("want_trans", C.c_int32), ("days", C.POINTER(C.c_int32)), ("lamb", C.c_double), ("beta", C.c_double),
                ("threshold_Ek", C.c_double), ("sweep_variant", C.c_int32), ("keep_on_device", C.c_int32),
                ("packed_input", C.c_int32), ("reserved0", C.c_int32)]


class DbInfo(C.Structure):
    _fields_ = [("n", C.c_uint64), ("L", C.c_uint64), ("n_variable_sites", C.c_uint64), ("device", C.c_int32), ("reserved0", C.c_int32),
                ("bytes_held", C.c_uint64), ("query_rows", C.c_uint64), ("new_sites", C.c_uint64)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class Synth(C.Structure):
    _fields_ = [("n", C.c_uint64), ("L", C.c_uint64), ("pitch", C.c_uint64), ("seed", C.c_uint64), ("p_var", C.c_double),
                ("n_clusters", C.c_uint32), ("mu", C.c_double), ("p_N", C.c_double), ("p_amb", C.c_double),
                ("gc", C.c_double), ("n_days", C.c_uint32), ("gaps", C.c_uint32), ("site_offset", C.c_uint64), ("L_total", C.c_uint64),
                ("packed", C.c_uint32), ("reserved0", C.c_uint32)]


# every symbol include/tracs_b200.h declares
SYMBOLS = ["tracs_pairsnp", "tracs_pairsnp_host", "tracs_pairsnp_device", "tracs_edges_free", "tracs_trans_dist",
           "tracs_lprob_k_given_N", "tracs_calculate_posteriors", "tracs_min_over_refs", "tracs_last_error",
           "tracs_last_stats", "tracs_device_count", "tracs_trim", "tracs_set_device", "tracs_synth_device", "tracs_dev_alloc",
           "tracs_dev_free", "tracs_host_alloc_pinned", "tracs_host_free_pinned", "tracs_memcpy_d2h",
           "tracs_memcpy_h2d", "tracs_int_peak", "tracs_read_fasta", "tracs_free_fasta", "tracs_shard_rowblocks",
           "tracs_site_shard_open", "tracs_site_shard_partials", "tracs_site_shard_close", "tracs_connected_components",
           "tracs_write_distance_csv", "tracs_float_repr", "tracs_pairsnp_packed", "tracs_encode_packed", "tracs_site_shard_finish", "tracs_tc_peak", "tracs_tc_peak_sustained", "tracs_site_shard_select", "tracs_site_shard_emit",
           "tracs_host_register", "tracs_host_unregister", "tracs_distance_matrix_device", "tracs_distance_matrix_host",
           "tracs_write_distance_matrix", "tracs_db_open_host", "tracs_db_open_device", "tracs_db_query_host", "tracs_db_query_device",
           "tracs_db_info", "tracs_db_close"]

_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError("tracs_b200: %s is not built (run `python -m tracs_b200.build`); there is no CPU fallback" % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        L.tracs_last_error.restype = C.c_char_p
        L.tracs_pairsnp.argtypes = [C.POINTER(C.c_char_p), C.c_int, C.c_int, C.c_int32, C.c_int, C.POINTER(Edges)]
        L.tracs_pairsnp_host.argtypes = [C.c_void_p, C.c_size_t, C.c_size_t, C.c_size_t, C.POINTER(Opts), C.POINTER(Edges)]
        L.tracs_pairsnp_device.argtypes = [C.c_void_p, C.c_size_t, C.c_size_t, C.c_size_t, C.POINTER(Opts), C.POINTER(Edges)]
        L.tracs_pairsnp_packed.argtypes = [C.c_void_p, C.c_size_t, C.c_size_t, C.c_size_t, C.POINTER(Opts), C.POINTER(Edges)]
        L.tracs_encode_packed.argtypes = [C.c_void_p, C.c_size_t, C.c_size_t, C.c_size_t, C.c_void_p, C.c_size_t]
        L.tracs_site_shard_finish.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_size_t, C.c_size_t, C.POINTER(Opts),
                                              C.POINTER(Edges)]
        L.tracs_site_shard_select.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_size_t, C.c_size_t, C.POINTER(Opts),
                                              C.POINTER(C.c_void_p), C.POINTER(C.c_size_t)]
        L.tracs_site_shard_emit.argtypes = [C.c_void_p, C.POINTER(Edges), C.c_size_t, C.POINTER(C.c_int)]
        L.tracs_host_register.argtypes = [C.c_void_p, C.c_size_t]
        L.tracs_host_unregister.argtypes = [C.c_void_p]
        L.tracs_edges_free.argtypes = [C.POINTER(Edges)]
        L.tracs_edges_free.restype = None
        L.tracs_trans_dist.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_double, C.c_double, C.c_double, C.c_void_p, C.c_void_p]
        L.tracs_lprob_k_given_N.argtypes = [C.c_size_t, C.c_size_t, C.c_double, C.c_double, C.c_double, C.c_void_p, C.c_size_t, C.c_void_p]
        L.tracs_calculate_posteriors.argtypes = [C.c_void_p, C.c_size_t, C.c_size_t, C.c_void_p, C.c_size_t, C.c_int, C.c_double, C.c_void_p]
        L.tracs_min_over_refs.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_size_t)]
        L.tracs_last_stats.argtypes = [C.POINTER(Stats)]
        L.tracs_set_device.argtypes = [C.c_int]
        L.tracs_synth_device.argtypes = [C.POINTER(Synth), C.c_void_p, C.c_void_p]
        L.tracs_dev_alloc.argtypes = [C.POINTER(C.c_void_p), C.c_size_t]
        L.tracs_dev_free.argtypes = [C.c_void_p]
        L.tracs_host_alloc_pinned.argtypes = [C.POINTER(C.c_void_p), C.c_size_t]
        L.tracs_host_free_pinned.argtypes = [C.c_void_p]
        L.tracs_memcpy_d2h.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t]
        L.tracs_memcpy_h2d.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t]
        L.tracs_int_peak.argtypes = [C.c_void_p]
        L.tracs_tc_peak.argtypes = [C.c_void_p]
        L.tracs_tc_peak_sustained.argtypes = [C.c_double, C.c_void_p]
        L.tracs_read_fasta.argtypes = [C.c_char_p, C.c_int, C.POINTER(C.POINTER(C.c_uint8)), C.POINTER(C.c_size_t), C.POINTER(C.c_size_t),
                                       C.POINTER(C.POINTER(C.c_char_p))]
        L.tracs_free_fasta.argtypes = [C.POINTER(C.c_uint8), C.POINTER(C.c_char_p), C.c_size_t]
        L.tracs_free_fasta.restype = None
        L.tracs_site_shard_open.argtypes = [C.c_void_p, C.c_size_t, C.c_size_t, C.c_size_t, C.POINTER(Opts), C.POINTER(C.c_void_p),
                                            C.POINTER(C.c_void_p), C.POINTER(C.c_size_t)]
        L.tracs_site_shard_partials.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p]
        L.tracs_site_shard_close.argtypes = [C.c_void_p]
        L.tracs_connected_components.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_size_t, C.c_void_p, C.POINTER(C.c_size_t)]
        L.tracs_write_distance_csv.argtypes = [C.c_char_p, C.c_int, C.POINTER(Edges), C.POINTER(C.c_char_p), C.c_size_t, C.c_char_p, C.c_int,
                                               C.c_int, C.c_int, C.c_double, C.POINTER(C.c_size_t)]
        L.tracs_float_repr.argtypes = [C.c_double, C.c_char_p]
        L.tracs_float_repr.restype = C.c_size_t
        L.tracs_shard_rowblocks.argtypes = [C.c_uint32, C.c_int32, C.c_int32, C.c_void_p, C.POINTER(C.c_uint32)]
        L.tracs_distance_matrix_device.argtypes = [C.c_void_p, C.c_size_t, C.c_size_t, C.c_size_t, C.POINTER(Opts), C.c_void_p, C.c_size_t]
        L.tracs_distance_matrix_host.argtypes = [C.c_void_p, C.c_size_t, C.c_size_t, C.c_size_t, C.POINTER(Opts), C.c_void_p, C.c_size_t]
        L.tracs_write_distance_matrix.argtypes = [C.c_char_p, C.c_void_p, C.c_size_t, C.c_size_t, C.c_size_t, C.POINTER(C.c_char_p),
                                                  C.POINTER(C.c_char_p), C.c_char]
        L.tracs_db_open_host.argtypes = [C.c_void_p, C.c_size_t, C.c_size_t, C.c_size_t, C.POINTER(Opts), C.POINTER(C.c_void_p)]
        L.tracs_db_open_device.argtypes = [C.c_void_p, C.c_size_t, C.c_size_t, C.c_size_t, C.POINTER(Opts), C.POINTER(C.c_void_p)]
        L.tracs_db_query_host.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_size_t, C.POINTER(Opts), C.POINTER(Edges)]
        L.tracs_db_query_device.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_size_t, C.POINTER(Opts), C.POINTER(Edges)]
        L.tracs_db_info.argtypes = [C.c_void_p, C.POINTER(DbInfo)]
        L.tracs_db_close.argtypes = [C.c_void_p]
        _lib = L
    return _lib


def check(rc):
    """Status code -> Python exception (RuntimeError like pybind11's std::runtime_error mapping,
    IndexError for std::out_of_range)."""
    if rc == 0:
        return
    msg = lib().tracs_last_error().decode(errors="replace")
    if rc == 3:
        raise IndexError(msg)
    if rc == 4:     # SIGINT arrived during the call (the library checks between bands / chunks)
        raise KeyboardInterrupt(msg)
    raise RuntimeError(msg)


def last_stats():
    s = Stats()
    lib().tracs_last_stats(C.byref(s))
    return s.as_dict()


class _EdgeOwner:
    """Keeps a tracs_edges_t alive while zero-copy numpy views of its columns exist."""

    def __init__(self, e):
        self.e = e

    def __del__(self):
        try:
            lib().tracs_edges_free(C.byref(self.e))
        except Exception:
            pass


class EdgeTable(dict):
    """dict of edge columns; with copy=False the arrays are views into library-owned memory that
    stays valid as long as this object is alive."""
    _owner = None


def take_edges(e, as_lists=False, names=True, copy=True):
    """tracs_edges_t -> EdgeTable of numpy arrays (or Python lists). copy=True copies and frees the
    struct at once; copy=False wraps the library's buffers without copying."""
    n = e.n_edges
    e_has_rows = bool(e.rows) or n == 0

    def arr(p, dt):
        if not p:
            return None
        if not n:
            return np.zeros(0, dt)
        a = np.ctypeslib.as_array(p, shape=(n,))
        return a.astype(dt, copy=True) if copy else a

    out = EdgeTable({"rows": arr(e.rows, np.uint64), "cols": arr(e.cols, np.uint64), "dist": arr(e.dist, np.uint64),
                     "filt": arr(e.filt, np.uint64), "ncomp": arr(e.ncomp, np.uint64), "p0_log": arr(e.p0_log, np.float64),
                     "eK": arr(e.eK, np.float64), "datediff": arr(e.datediff, np.float64), "seq_length": int(e.seq_length),
                     "names": [e.names[i].decode() for i in range(e.n_names)] if (names and e.names) else [],
                     "dev_packed": (int(e.dev_packed), int(e.dev_packed_bytes)) if (e.dev_packed and not copy) else None})
    if copy:
        lib().tracs_edges_free(C.byref(e))
    else:
        out._owner = _EdgeOwner(e)
    if out["filt"] is None and e_has_rows:
        # filter off: the reference returns a vector of zeros (src/pairsnp.hpp:452). A zero-stride read-only view: a real
        # 8 B x E array costs 1.4 - 4 ms per C3 call (glibc hands back recycled heap that calloc has to clear)
        out["filt"] = np.broadcast_to(np.uint64(0), (n,))
    if as_lists:
        for k in ("rows", "cols", "dist", "filt", "ncomp"):
            out[k] = out[k].tolist()
    return out
