/*
 * tracs_b200.h -- C ABI of libtracs_b200.so, the B200 (sm_100a) implementation of the TRACS
 * pairwise-distance hot path. Plain pointers and sizes only; no torch / pybind types.
 *
 * Each entry point names the reference interface it replaces (paths relative to the
 * gtonkinhill/tracs source tree). The Python module `TRACS` the reference callers import
 * (tracs/distance.py:8, tracs/transcluster.py:2, tracs/align.py:21) is a thin binding over these
 * calls: tracs_b200/dropin/TRACS.py (see INTEGRATION.md).
 *
 * Conventions
 *   - every function returns 0 on success, non-zero on failure; tracs_last_error() then holds a
 *     message (thread-local). CUDA errors are reported the same way. There is NO CPU fallback:
 *     without a usable CUDA device the compute entry points fail.
 *   - result arrays are allocated by the library and released with tracs_edges_free().
 *   - inputs are borrowed for the duration of the call only.
 *   - one call at a time per process (like the reference module, which holds the GIL and uses
 *     function-static caches: src/pairsnp.hpp:19,43).
 */
#ifndef TRACS_B200_H
#define TRACS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* Sparse (COO) result of a pair sweep == the 6-tuple returned by pairsnp()
 * (src/pairsnp.hpp:320-322,457): rows, cols, distances, seq_names, filt_distances,
 * n_compared_sites, all in (row, col) lexicographic order (src/pairsnp.hpp:395,450-457).
 * p0_log / eK are filled only by the fused entry points when sampling days are supplied
 * (what tracs/transcluster.py:8-41 + src/transcluster.hpp:240-287 compute per edge). */
typedef struct tracs_edges {
  size_t n_edges;
  uint64_t *rows;    /* sample index i                                   */
  uint64_t *cols;    /* sample index j                                   */
  uint64_t *dist;    /* SNP distance d(i,j)                              */
  uint64_t *filt;    /* recombination-filtered distance; NULL when the filter is off (= the reference's vector of zeros) */
  uint64_t *ncomp;   /* compared (non-N) sites                           */
  double *p0_log;    /* log P(direct transmission)   or NULL             */
  double *eK;        /* E[# intermediate hosts]       or NULL             */
  double *datediff;  /* |t_i - t_j| in years          or NULL             */
  size_t n_names;
  char **names;      /* n_names NUL-terminated strings, or NULL           */
  uint64_t seq_length;
  /* tracs_opts_t.keep_on_device: the same columns, still in DEVICE memory, packed column-wise as
   * u32 rows[n] | u32 cols[n] | u32 dist[n] (the raw SNP distance) | u32 ncomp[n] | f64 p0_log[n] | f64 eK[n]
   * (32 bytes per edge) so a multi-GPU caller can gather edge lists GPU-to-GPU. The filtered distance is not
   * part of the block (callers that ran the filter gather the host columns). NULL otherwise. */
  void *dev_packed;
  size_t dev_packed_bytes;
} tracs_edges_t;

/* Per-call statistics of the last sweep on this thread (for bench.py / roofline accounting). */
typedef struct tracs_stats {
  uint64_t n_samples, seq_length;
  uint64_t n_variable_sites; /* V_eff: sites kept by the exact drop rule (SURVEY A.4)     */
  uint64_t n_words;          /* ceil(V_eff/32) padded to the k-chunk                        */
  uint64_t n_tiles;          /* 128x128 pair tiles swept                                    */
  uint64_t n_pairs;          /* pairs in range (what the reference loop visits)             */
  uint64_t n_edges;
  uint64_t kernel_launches;  /* kernels of this library launched by the call                */
  uint64_t h2d_bytes, d2h_bytes;
  uint64_t n_candidates;     /* pairs that survived the prefilter sweep (0 if it did not run)       */
  uint64_t swept_wordpairs;  /* 32-site word-pairs the tile kernel actually evaluated               */
  uint64_t n_early_sites;    /* sites listed from the first sample chunk and extracted while packing (0: two-pass ingest) */
  float ms_pack;             /* ASCII -> column masks + N planes (K0a): all pack launches + early site list */
  float ms_compact;          /* variable-site selection + bit-plane gather (K0b)            */
  float ms_sweep;            /* pair tile sweep incl. threshold/compaction epilogue (K1)    */
  float ms_refine;           /* per-pair refinement of prefilter candidates (K1b)           */
  float ms_sort;             /* edge ordering                                               */
  float ms_ncomp;            /* compared-sites kernel (K2)                                  */
  float ms_trans;            /* transmission LUT + gather (K3)                              */
  float ms_total;            /* device time of the whole call (events on the call's stream) */
  float ms_d2h;              /* edge columns device -> host                                  */
  float ms_filter;           /* recombination filter (K4), only when filter != 0             */
  float tc_sweep;            /* 0: LOP3/POPC tile kernel; else 30 + int8 operand planes executed per site:
                                33 / 34 = k_sweep_tc3<3|4> */
  float ms_pack_main;        /* the main pack launch alone: k_pack_x over samples 256.. (early extraction) or k_pack over all */
  float sparse_nplane;       /* 1: sparse N (first-chunk estimate): the main ingest launch stored only the N-plane sectors that hold an N */
  float reserved0;
} tracs_stats_t;

/* Options shared by the matrix-input entry points. Zero-initialise, then set. */
typedef struct tracs_opts {
  int32_t dist;        /* keep pairs with d <= dist  (pairsnp arg `dist`, int; INT32_MAX = all) */
  int32_t filter;      /* pairsnp arg `filter` (recombination filter, src/pairsnp.hpp:251-318)  */
  uint64_t i_end;      /* rows are samples [0, i_end)              (src/pairsnp.hpp:348,382)    */
  uint64_t j_start;    /* cols are samples [max(j_start,i+1), n)   (src/pairsnp.hpp:354-358,395)*/
  int32_t shard_rank;  /* this process sweeps row-blocks dealt to shard_rank of shard_world       */
  int32_t shard_world; /* (0 or 1 = everything). No inter-GPU traffic inside the call.           */
  int32_t want_ncomp;  /* compute n_compared_sites (the reference always does)                   */
  int32_t want_trans;  /* fused transmission likelihood: needs days != NULL                      */
  const int32_t *days; /* host: sampling day number per sample (days since any epoch)            */
  double lamb, beta, threshold_Ek; /* trans_dist args (src/transcluster.hpp:241)                 */
  int32_t sweep_variant; /* 0 = prefilter + refine when the threshold allows; 1 = always the full-length LOP3/POPC
                          * tile sweep; 2 = full-length sweep on the tensor cores (tcgen05 int8 one-hot GEMM; needs
                          * single-base-or-N masks at the variable sites, else the call fails) */
  int32_t keep_on_device; /* also return the edge columns packed in device memory (tracs_edges_t.dev_packed) */
  int32_t packed_input;   /* the alignment is given as 4-bit base masks, two sites per byte (see tracs_pairsnp_packed),
                           * instead of ASCII: applies to tracs_pairsnp_host / _device and tracs_site_shard_open */
  int32_t reserved0;
} tracs_opts_t;

/* Replaces TRACS.pairsnp(fasta, n_threads, dist, filter) -- src/python_bindings.cpp:12-13,
 * src/pairsnp.hpp:320-458. paths: 1 or 2 FASTA(.gz) files (2 = query x db). n_threads sizes only
 * host-side parsing: a plain (uncompressed) file is parsed by n_threads workers whenever that is provably
 * identical to the sequential kseq semantics (checked while parsing, else the sequential reader runs). */
int tracs_pairsnp(const char *const *paths, int n_paths, int n_threads, int32_t dist, int filter,
                  tracs_edges_t *out);

/* Same sweep on an alignment already held as an ASCII matrix seqs[n][pitch] (the bytes
 * load_seqs keeps per record, src/pairsnp.hpp:99-110) in HOST memory; includes the H2D copy
 * (page-locked sources go to the copy engine directly; large pageable ones are staged by worker
 * threads through page-locked double buffers). */
int tracs_pairsnp_host(const uint8_t *seqs, size_t n, size_t L, size_t pitch, const tracs_opts_t *opts,
                       tracs_edges_t *out);

/* Same, with the ASCII matrix already resident in DEVICE memory (pitch % 16 == 0). */
int tracs_pairsnp_device(const uint8_t *dev_seqs, size_t n, size_t L, size_t pitch, const tracs_opts_t *opts,
                         tracs_edges_t *out);

/* Same sweep on an alignment held in DEVICE memory as 4-bit base masks: nib[n][pitch_bytes], site s of a sample in
 * byte s >> 1, bits [4 * (s & 1), +4); the nibble is the mask the reference's loader derives from the base
 * (src/pairsnp.hpp:107-199: bit0 A, bit1 C, bit2 G, bit3 T; N, '-', anything else = 1111). pitch_bytes % 16 == 0 and
 * 2 * pitch_bytes >= L rounded up to 32. Half the bytes of the ASCII matrix: 100 000 x 2 Mb is 100 GB and fits one
 * B200 (SURVEY 8b `tracs_pairsnp_packed`, 8d "packed 4-bit IUPAC masks directly on device"). */
int tracs_pairsnp_packed(const uint8_t *dev_nib, size_t n, size_t L, size_t pitch_bytes, const tracs_opts_t *opts,
                         tracs_edges_t *out);

/* All-pairs SNP distance as a dense int32 matrix. d(i, j) is the `dist` column of tracs_pairsnp_* with
 * dist = INT32_MAX: the number of sites where the two base masks share no base (src/pairsnp.hpp:393-403; N, gaps and
 * unknown bytes match everything, IUPAC codes are honoured). Two shapes, chosen by opts->i_end / opts->j_start:
 *   i_end = 0 or n, j_start = 0       -> n x n, symmetric, both triangles written, diagonal 0;
 *   0 < i_end <= j_start < n          -> i_end x (n - j_start): rows = samples [0, i_end), cols = samples [j_start, n)
 *                                        (the query x db mode of tracs_pairsnp with two files).
 * out[r * ld + c]; entries of the padding (ld > cols) are never written. opts may be NULL (square matrix).
 * opts->packed_input selects ASCII or 4-bit input as on the other entry points; opts->sweep_variant: 0 = tensor cores
 * when the masks allow them, else LOP3/POPC; 1 = LOP3/POPC; 2 = tensor cores required (fails on 2-/3-base codes at
 * variable sites). opts->want_ncomp is ignored. Errors, raised before any device call and naming the field: dist other
 * than INT32_MAX, filter, want_trans / days, keep_on_device, shard_world > 1, any other (i_end, j_start), ld smaller
 * than the column count, a bad pitch. A matrix that does not fit in device memory next to the ingest fails with a
 * message that gives its size (no partial result). Not computed: the compared-sites count of every pair (use the
 * thresholded pair list). */
int tracs_distance_matrix_device(const uint8_t *dev_seqs, size_t n, size_t L, size_t pitch, const tracs_opts_t *opts,
                                 int32_t *dev_out, size_t ld); /* device input (ASCII or packed), caller-owned device matrix */
int tracs_distance_matrix_host(const uint8_t *seqs, size_t n, size_t L, size_t pitch, const tracs_opts_t *opts, int32_t *out,
                               size_t ld); /* host input (streamed like tracs_pairsnp_host), host output */
/* Host only: the matrix as text. First line: an empty cell, then the column names; then one line per row: the row
 * name, then the values. sep = '\t' or ','. Names are written as given (no quoting, like tracs_write_distance_csv).
 * Rows are formatted by parallel threads (TRACS_WRITE_THREADS, default: the hardware threads, at most 16); the bytes
 * do not depend on their number. */
int tracs_write_distance_matrix(const char *path, const int32_t *m, size_t rows, size_t cols, size_t ld,
                                const char *const *row_names, const char *const *col_names, char sep);

/* ---- resident sample database (query x db without re-ingesting the database) ----------------------------------------
 * The two-file mode of pairsnp (rows = new samples, cols = a database) for callers that place batch after batch of new
 * samples against the same collection: the database is ingested once (N-plane, variable sites, bit-planes) and stays on the
 * device; each query pays for its own rows and its own pairs. For a database db (n_db samples, L sites) and a query batch
 * q (nq samples, the same L):
 *   tracs_db_query_*(db, q, opts)  returns exactly what  tracs_pairsnp_host([q; db], opts with i_end = j_start = nq)
 * returns: every column, the same (row, col) order, two-file indices (rows in [0, nq), cols in [nq, nq + n_db)).
 * opts as on the two-file call: dist, want_ncomp, sweep_variant, packed_input (of the query rows), want_trans / days (nq + n_db
 * days, queries first) / lamb / beta / threshold_Ek. Refused before any device call, naming the field: filter, keep_on_device,
 * shard_world > 1, i_end or j_start set, a bad pitch, a NULL or closed handle. nq = 0 returns no edges.
 * A query whose bit-planes do not fit in device memory fails with their size in GB; the handle stays usable.
 * tracs_last_stats after a query describes the query's own work (n_pairs = nq * n_db).
 *
 * open: opts may be NULL; only opts->packed_input is read (ASCII rows, or 4-bit rows as tracs_pairsnp_packed).
 *   _host copies the rows into device memory the library owns (streamed like tracs_pairsnp_host).
 *   _device with 4-bit rows BORROWS dev_seqs until tracs_db_close: unlike every other entry point, the buffer must stay allocated
 *   and unchanged while the handle is open (the library only reads it; a second copy of a 100 GB database would not fit).
 *   _device with ASCII rows encodes them once into 4-bit rows the library owns (half their size); dev_seqs is not kept.
 * The handle belongs to the device that was current at open; a query while another device is current fails. Closing a handle
 * twice, or passing one that was never opened, fails without touching memory. */
typedef struct tracs_db_info {
  uint64_t n;                /* database samples                                                   */
  uint64_t L;                /* sites                                                              */
  uint64_t n_variable_sites; /* variable sites of the database alone                               */
  int32_t device;            /* the device the handle belongs to                                   */
  int32_t reserved0;
  uint64_t bytes_held;       /* device bytes the handle holds (borrowed rows not counted)          */
  uint64_t query_rows;       /* query rows swept at once; larger batches go through in chunks       */
  uint64_t new_sites;        /* sites variable in [q; db] but not in db, for the last query batch  */
} tracs_db_info_t;
int tracs_db_open_host(const uint8_t *seqs, size_t n, size_t L, size_t pitch, const tracs_opts_t *opts, void **db);
int tracs_db_open_device(const uint8_t *dev_seqs, size_t n, size_t L, size_t pitch, const tracs_opts_t *opts, void **db);
int tracs_db_query_host(void *db, const uint8_t *seqs, size_t nq, size_t pitch, const tracs_opts_t *opts, tracs_edges_t *out);
int tracs_db_query_device(void *db, const uint8_t *dev_seqs, size_t nq, size_t pitch, const tracs_opts_t *opts, tracs_edges_t *out);
int tracs_db_info(void *db, tracs_db_info_t *out);
int tracs_db_close(void *db);

/* ASCII rows -> packed rows on the device (what the host-streaming path runs per chunk): dev_ascii[rows][pitch]
 * (pitch % 32 == 0, >= L rounded up to 32) -> dev_nib[rows][pitch_bytes]. Sites >= L become 1111. */
int tracs_encode_packed(const uint8_t *dev_ascii, size_t rows, size_t L, size_t pitch, uint8_t *dev_nib, size_t pitch_bytes);

void tracs_edges_free(tracs_edges_t *e);

/* The loader half of pairsnp on its own (src/pairsnp.hpp:62-220 + src/kseq.h:170-208 record
 * semantics): FASTA/FASTQ(.gz) -> ASCII matrix seqs[n][L] (malloc'ed, pitch == L) + names. Host only.
 * Errors like the reference: "Error reading FASTA!", "... variable sequence lengths!". */
int tracs_read_fasta(const char *path, int n_threads, uint8_t **seqs, size_t *n, size_t *L, char ***names);
void tracs_free_fasta(uint8_t *seqs, char **names, size_t n);

/* Row-blocks (128 samples each) that shard `rank` of `world` sweeps (boustrophedon deal).
 * out: caller-allocated, n_rowblocks entries. Host only. */
int tracs_shard_rowblocks(uint32_t n_rowblocks, int32_t world, int32_t rank, uint32_t *out, uint32_t *n_out);

/* Replaces TRACS.trans_dist(snpdiff, datediff, lamb, beta, threshold_Ek) --
 * src/python_bindings.cpp:19-21, src/transcluster.hpp:240-287. p0_log and eK: caller-allocated,
 * n doubles each. */
int tracs_trans_dist(const int32_t *snpdiff, const double *datediff, size_t n, double lamb, double beta,
                     double threshold_Ek, double *p0_log, double *eK);

/* Replaces TRACS.lprob_k_given_N(N, k, delta, lamb, beta, lgamma) -- src/python_bindings.cpp:15-17,
 * src/transcluster.hpp:90-129. Scalar, test-only entry in the reference; host arithmetic.
 * out[0] = lprob, out[1] = lhs. Fails (index error) if the table is shorter than N+k+2. */
int tracs_lprob_k_given_N(size_t N, size_t k, double delta, double lamb, double beta, const double *lgamma_tab,
                          size_t n_lgamma, double out[2]);

/* Replaces TRACS.calculate_posteriors(counts, alphas, keep, threshold) --
 * src/python_bindings.cpp:23-25, src/dmultinomial.hpp:8-86. Not on the hot path (align stage);
 * exported so `import tracs.align` keeps working. Host arithmetic. out: rows*cols doubles. */
int tracs_calculate_posteriors(const double *counts, size_t rows, size_t cols, const double *alphas, size_t n_alpha,
                               int keep, double threshold, double *out);

/* Min-over-references combine (SURVEY A.6; tracs/distance.py:159-258 + tracs/cluster.py:104-113
 * realise it implicitly): edges keyed by unordered (a,b) sample-id pair, value = min. Inputs are
 * concatenated per-MSA edge lists with GLOBAL sample ids. Outputs caller-allocated (n each);
 * *n_out receives the number of distinct pairs, sorted by (min id, max id). Runs on the device. */
int tracs_min_over_refs(const uint64_t *a, const uint64_t *b, const double *val, size_t n, uint64_t *out_a,
                        uint64_t *out_b, double *out_val, size_t *n_out);

/* ---- site-sharded multi-GPU sweep (alignments larger than one GPU) ------------------------------
 * d(i,j) and |N_i u N_j| are sums over disjoint site ranges, so rank r of R ingests only the column
 * slab [L*r/R, L*(r+1)/R) of every sequence (dev_slab[n][pitch], L_slab sites), prefilters its share
 * of the triangle row-blocks (opts->shard_rank/shard_world, opts->dist < 2048) and returns the
 * candidate pairs it could not reject (device array of keys i<<32|j, sorted; owned by the handle).
 * The caller all-gathers the candidate lists, calls tracs_site_shard_partials on every rank with the
 * full list (device pointers; outputs: this slab's mismatch count and |N_i u N_j| per candidate),
 * sums the two vectors over ranks (all-reduce) and keeps d <= dist; compared sites = L - union.
 * Same quantities as src/pairsnp.hpp:398-403,417-419. tracs_b200/sites.py drives this with NCCL. */
int tracs_site_shard_open(const uint8_t *dev_slab, size_t n, size_t L_slab, size_t pitch, const tracs_opts_t *opts,
                          void **handle, const uint64_t **dev_cand_keys, size_t *n_cand);
int tracs_site_shard_partials(void *handle, const uint64_t *dev_keys, size_t n_keys, uint32_t *dev_d, uint32_t *dev_union);
/* Last step of the site-sharded sweep, on ONE rank (the all-reduce leaves every rank with the summed vectors):
 * keeps the candidates with d <= opts->dist, compared sites = L_total - union, optional fused transmission
 * likelihood (opts->days of all n samples), columns to page-locked host memory. dev_keys sorted ascending
 * (i << 32 | j), dev_d / dev_union: the summed per-candidate vectors. `handle` may be NULL (nothing of the
 * shard is read). Output as tracs_pairsnp_device. */
int tracs_site_shard_finish(const uint64_t *dev_keys, const uint32_t *dev_d, const uint32_t *dev_union, size_t n_keys,
                            size_t n_samples, size_t L_total, const tracs_opts_t *opts, tracs_edges_t *out);
/* The same last step split in two, for N > 1: every rank takes a contiguous slice of the summed candidate vectors.
 * _select thresholds the slice and returns how many edges it holds (the selected columns stay on the device, owned by
 * *selection); the caller exchanges the counts (all-gather) to learn where each slice starts in the edge table;
 * _emit computes the likelihood columns and copies everything into the caller's HOST columns (dst->rows ... datediff:
 * page-locked or tracs_host_register'ed memory, e.g. one shared-memory segment mapped by all ranks) starting at
 * element `at`, then releases the selection. So each GPU delivers its share over its own PCIe link. dst->filt, names
 * and counts are not touched; dst->ncomp / p0_log / eK / datediff may be NULL when not wanted. */
int tracs_site_shard_select(const uint64_t *dev_keys, const uint32_t *dev_d, const uint32_t *dev_union, size_t n_keys,
                            size_t n_samples, size_t L_total, const tracs_opts_t *opts, void **selection, size_t *n_selected);
int tracs_site_shard_emit(void *selection, const tracs_edges_t *dst, size_t at, int *has_trans);
int tracs_site_shard_close(void *handle);

/* Single-linkage clusters of the thresholded edge list = connected components (what tracs/cluster.py:126-129
 * asks scipy for). a/b: edge endpoints (node ids < n_nodes), labels: n_nodes entries, numbered like
 * scipy.sparse.csgraph.connected_components (by the smallest node of each component). Runs on the device. */
int tracs_connected_components(const uint64_t *a, const uint64_t *b, size_t n_edges, size_t n_nodes, uint32_t *labels,
                               size_t *n_components);

/* Native writer of the distance CSV (the per-edge Python loop of tracs/distance.py:206-258): same header,
 * column order and quirks (NA columns without metadata, `NA` in the filtered column with metadata but no
 * filter, rows with expected K above the -K threshold dropped, floats printed like Python's repr).
 * e: edges of one MSA (p0_log/eK/datediff set when the likelihood was computed); names: sample names. Host only. */
int tracs_write_distance_csv(const char *path, int append, const tracs_edges_t *e, const char *const *names, size_t n_names,
                             const char *msa_label, int has_trans, int filter_on, int use_k_threshold, double k_threshold,
                             size_t *rows_written);
/* Python-repr formatting of a double (what the writer uses); buf >= 32 bytes; returns the length. */
size_t tracs_float_repr(double v, char *buf);

const char *tracs_last_error(void);
int tracs_last_stats(tracs_stats_t *out);
int tracs_device_count(void);
/* Device scratch blocks and page-locked result blocks are cached by the library between calls
 * (reused whole, by size); this returns the idle ones to the driver. */
int tracs_trim(void);
int tracs_set_device(int device);

/* ---- bench / test utilities (not in the reference) ------------------------------------------ */

/* Seeded synthetic alignment generated directly in device memory (SURVEY 8d generator G).
 * dev_seqs: device buffer n*pitch bytes. dev_days (optional, device, n int32): sampling days. */
typedef struct tracs_synth {
  uint64_t n, L, pitch, seed;
  double p_var;    /* fraction of variable sites                         */
  uint32_t n_clusters;
  double mu;       /* mean private substitutions per sample              */
  double p_N;      /* iid N probability per (sample, site)               */
  double p_amb;    /* ambiguity-code probability per (sample, var site)  */
  double gc;
  uint32_t n_days; /* days drawn uniformly from [0, n_days)              */
  uint32_t gaps;   /* number of '-' runs of length L/1000 per sample     */
  uint64_t site_offset; /* generate columns [site_offset, site_offset + L) of an alignment of L_total sites */
  uint64_t L_total;     /* 0 = L (whole alignment)                                                        */
  uint32_t packed;      /* 1: write 4-bit masks (tracs_pairsnp_packed layout), `pitch` = bytes per packed row */
  uint32_t reserved0;
} tracs_synth_t;
int tracs_synth_device(const tracs_synth_t *cfg, uint8_t *dev_seqs, int32_t *dev_days);

/* Device memory helpers so a host program can own device-resident inputs without a CUDA binding. */
int tracs_dev_alloc(void **p, size_t bytes);
int tracs_dev_free(void *p);
int tracs_host_alloc_pinned(void **p, size_t bytes);
int tracs_host_free_pinned(void *p);
/* page-locks an existing host range (e.g. a shared-memory mapping) for direct device copies / releases it */
int tracs_host_register(void *p, size_t bytes);
int tracs_host_unregister(void *p);
int tracs_memcpy_d2h(void *dst, const void *src, size_t bytes);
int tracs_memcpy_h2d(void *dst, const void *src, size_t bytes);

/* Measures the INT-pipe peak on the current device with register-resident loops.
 * out[0] = LOP3 lane-ops/s, out[1] = POPC lane-ops/s, out[2] = IADD lane-ops/s,
 * out[3] = word-pairs/s of the sweep's (4 LOP3 + POPC + ADD) mix, out[4] = same with the add
 * issued as IMAD (FMA pipe), out[5] = SM count. */
int tracs_int_peak(double out[8]);

/* Measures the int8 tensor-pipe peak on the current device: every SM issues back-to-back
 * tcgen05.mma.cta_group::1.kind::i8 (M = 128, K = 32) from shared-memory operands into TMEM.
 * out[0] = TOP/s with N = 128 (one 128 x 128 tile per MMA), out[1] = TOP/s with N = 256 (the shape k_sweep_tc3 issues),
 * out[2], out[3] = SM clock cycles per MMA for the two shapes. */
int tracs_tc_peak(double out[4]);
/* The same probe held for `seconds` (0.05 .. 10): out[0] = TOP/s over the second half of the run (what the pipe sustains under
 * the board's power cap: the denominator for multi-second tensor-core kernels), out[1] = over the whole run. */
int tracs_tc_peak_sustained(double seconds, double out[2]);

#ifdef __cplusplus
}
#endif
#endif
