// Shared declarations for libtracs_b200.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <sys/mman.h>
#include <memory>
#include <new>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/tracs_b200.h"

namespace tracs {

void set_error(const std::string &msg);
extern thread_local tracs_stats_t g_stats;

struct CudaError {
  std::string msg;
};

#define TRACS_CK(call)                                                                             \
  do {                                                                                             \
    cudaError_t e__ = (call);                                                                      \
    if (e__ != cudaSuccess) {                                                                      \
      char b__[512];                                                                               \
      snprintf(b__, sizeof b__, "CUDA error %s at %s:%d: %s", cudaGetErrorName(e__), __FILE__,     \
               __LINE__, cudaGetErrorString(e__));                                                 \
      throw tracs::CudaError{b__};                                                                 \
    }                                                                                              \
  } while (0)

// Device scratch comes from a block cache owned by the library: a freed block is kept whole and
// handed to the next request of (about) the same size, so the multi-GB buffers of one call are reused
// by the next one without fragmentation or driver calls (tracs_trim() releases the idle blocks).
// All work of a call is issued on one stream, so reuse is ordered by the stream.
void *dev_cache_alloc(size_t bytes);
void dev_cache_free(void *p);

void require_device();  // throws unless a CUDA device is usable (there is no CPU fallback)

// Ctrl-C during a long call (reference: PyErr_CheckSignals in its loops, then "Interrupted by user!" and exit(1),
// src/pairsnp.hpp:207-214, 434-441). The compute entry points install a SIGINT handler for their duration
// (InterruptScope) that only raises a flag; the sweep checks it between bands / chunks and unwinds with
// status 4, which the Python bindings turn into KeyboardInterrupt (drop-in pairsnp: message + exit code 1).
struct Interrupted {};
struct InterruptScope {
  InterruptScope();
  ~InterruptScope();
  InterruptScope(const InterruptScope &) = delete;
  InterruptScope &operator=(const InterruptScope &) = delete;
};
void check_interrupt();  // throws Interrupted if SIGINT arrived since the innermost scope began

// C-ABI status codes: 0 ok, 1 runtime error, 2 CUDA error, 3 index/range error, 4 interrupted (SIGINT)
template <typename F>
static int guarded(F &&f) {
  try {
    f();
    return 0;
  } catch (const Interrupted &) {
    set_error("Interrupted by user!");
    cudaDeviceSynchronize();
    return 4;
  } catch (const CudaError &e) {
    set_error(e.msg);
    cudaGetLastError();
    return 2;
  } catch (const std::out_of_range &e) {
    set_error(e.what());
    return 3;
  } catch (const std::exception &e) {
    set_error(e.what());
    return 1;
  }
}

// RAII device buffer
template <typename T>
struct DevBuf {
  T *p = nullptr;
  size_t n = 0;
  bool owned = true;
  DevBuf() {}
  explicit DevBuf(size_t count) { alloc(count); }
  DevBuf(const DevBuf &) = delete;
  DevBuf &operator=(const DevBuf &) = delete;
  void alloc(size_t count) {
    release();
    n = count;
    if (count) p = (T *)dev_cache_alloc(count * sizeof(T));
  }
  // a view of `count` elements of memory that something else owns: never freed through this object
  void borrow(T *q, size_t count) {
    release();
    p = q;
    n = count;
    owned = false;
  }
  void release() {
    if (p && owned) dev_cache_free(p);
    p = nullptr;
    n = 0;
    owned = true;
  }
  ~DevBuf() { release(); }
};

// One auxiliary stream per host thread and device (non-blocking: no implicit ordering with the legacy default stream
// the entry points run on): side work that overlaps the main stream -- the likelihood table under the ingest, the
// copies of finished edge columns under the compared-sites kernel. Ordering is by events only.
inline cudaStream_t aux_stream() {
  static thread_local cudaStream_t s[64] = {};
  int dev = 0;
  cudaGetDevice(&dev);
  dev &= 63;
  if (!s[dev]) cudaStreamCreateWithFlags(&s[dev], cudaStreamNonBlocking);
  return s[dev];
}

// Stage timers that do not stall the host: event pairs are recorded as the work is enqueued and read once at the end.
struct DeferredTimers {
  struct Item { cudaEvent_t a, b; float *acc; };
  std::vector<Item> items;
  cudaStream_t s;
  explicit DeferredTimers(cudaStream_t st) : s(st) {}
  void start(float *acc) {
    Item it{nullptr, nullptr, acc};
    cudaEventCreate(&it.a);
    cudaEventCreate(&it.b);
    cudaEventRecord(it.a, s);
    items.push_back(it);
  }
  void stop() { cudaEventRecord(items.back().b, s); }
  void resolve() {  // after the stream has been synchronised
    for (Item &it : items) {
      float ms = 0;
      if (cudaEventElapsedTime(&ms, it.a, it.b) == cudaSuccess) *it.acc += ms;
      else cudaGetLastError();  // unwinding after an error: the pair was never completed
      cudaEventDestroy(it.a);
      cudaEventDestroy(it.b);
    }
    items.clear();
  }
  ~DeferredTimers() { resolve(); }
};

struct Timer {
  cudaEvent_t a, b;
  cudaStream_t s;
  explicit Timer(cudaStream_t st) : s(st) {
    cudaEventCreate(&a);
    cudaEventCreate(&b);
  }
  ~Timer() {
    cudaEventDestroy(a);
    cudaEventDestroy(b);
  }
  void start() { cudaEventRecord(a, s); }
  float stop() {
    cudaEventRecord(b, s);
    cudaEventSynchronize(b);
    float ms = 0;
    cudaEventElapsedTime(&ms, a, b);
    return ms;
  }
};

// ------------------------------------------------------------------------------------------
// base-mask table: bit0=A bit1=C bit2=G bit3=T ; everything that is not an IUPAC code = 15
// ------------------------------------------------------------------------------------------
__host__ __device__ inline uint32_t base_mask(uint32_t c) {
  c &= 0xFFu;
  if (c >= 'a' && c <= 'z') c -= 32;
  switch (c) {
    case 'A': return 1;
    case 'C': return 2;
    case 'G': return 4;
    case 'T': return 8;
    case 'M': return 3;
    case 'R': return 5;
    case 'W': return 9;
    case 'S': return 6;
    case 'Y': return 10;
    case 'K': return 12;
    case 'V': return 7;
    case 'H': return 11;
    case 'D': return 13;
    case 'B': return 14;
    default: return 15;
  }
}

// ASCII rows -> 4-bit packed rows on the device (pack4.inl, k_encode)
void encode_rows_device(const uint8_t *dev_ascii, uint64_t rows, uint64_t L, uint64_t pitch, uint8_t *dev_nib, uint64_t pitch4,
                        cudaStream_t st);

// ---- geometry of the pair sweep ------------------------------------------------------------
constexpr int TILE = 128;  // samples per tile side
constexpr int KC = 8;      // 32-site words per pipeline stage
constexpr int STAGES = 3;  // shared-memory ring depth

// Growable byte buffer for parsed sequences: realloc growth (large blocks move by mremap, no copy),
// never zero-filled, and its storage can be handed to the caller (release()).
struct ByteBuf {
  uint8_t *p = nullptr;
  size_t len = 0, cap = 0;
  ByteBuf() {}
  ByteBuf(const ByteBuf &) = delete;
  ByteBuf &operator=(const ByteBuf &) = delete;
  ~ByteBuf() { free(p); }
  void reserve(size_t want) {
    if (want <= cap) return;
    size_t c = cap ? cap + cap / 2 : (size_t)1 << 20;
    if (c < want) c = want;
    uint8_t *q = (uint8_t *)realloc(p, c);
    if (!q) throw std::bad_alloc();
    p = q;
    cap = c;
#ifdef MADV_HUGEPAGE
    // multi-GB matrices written once by many parser threads: 2 MB pages cut the first-touch faults 512-fold
    if (c >= ((size_t)8 << 20)) madvise((void *)(((uintptr_t)q + 4095) & ~(uintptr_t)4095), (c - 4096) & ~(size_t)4095, MADV_HUGEPAGE);
#endif
  }
  uint8_t *data() { return p; }
  size_t size() const { return len; }
  uint8_t *release() {
    if (!p) p = (uint8_t *)malloc(1);
    uint8_t *q = p;
    p = nullptr;
    len = cap = 0;
    return q;
  }
};

// FASTA reader (fasta.cpp): kseq-compatible record semantics (reference src/kseq.h:170-208).
struct Alignment {
  std::vector<uint8_t> ascii;  // n * L bytes, row-major, pitch == L
  std::vector<std::string> names;
  uint64_t n = 0, L = 0;
};
// Consumer of parsed rows while the reader is still parsing (the FASTA entry point streams them to the device):
// rows() is called from the reader's coordinating thread, in row order, with a pointer to `count` complete rows of
// `L` bytes each; reset() tells the consumer to forget everything it was given (the parallel reader found out that
// the file needs the sequential state machine and starts over).
struct RowSink {
  virtual void expect(uint64_t total_rows, uint64_t L) = 0;  // optional hint, before the first rows()
  virtual void rows(const uint8_t *p, uint64_t first_row, uint64_t count, uint64_t L) = 0;
  virtual void reset() = 0;
  virtual ~RowSink() {}
};
// appends the records of `path`; returns number of records read; throws std::runtime_error. `sink` (optional) is fed
// the rows as they complete, numbered from `row0`.
uint64_t read_fasta(const char *path, int n_threads, ByteBuf &ascii, std::vector<std::string> &names, uint64_t &L,
                    RowSink *sink = nullptr, uint64_t row0 = 0);

// Static multi-GPU partition: row-blocks of 128 samples are dealt boustrophedon
// (0..w-1, w-1..0, ...) so every shard sweeps (nearly) the same triangle area.
inline int shard_owner(uint32_t row_block, int world) {
  const uint32_t round = row_block / (uint32_t)world, pos = row_block % (uint32_t)world;
  return (round & 1u) ? (world - 1 - (int)pos) : (int)pos;
}

// host-side edge columns produced by the sweep (sorted by (row, col))
// Result columns live in page-locked host blocks that are cached across calls (host_pool_*):
// the D2H copy runs at full PCIe rate into memory that is already mapped, and
// tracs_edges_free() hands the blocks back to the cache instead of the OS.
void *host_pool_alloc(size_t bytes);
void host_pool_free(void *p);

// pool-backed growable column: the D2H copy lands in the buffer that is handed to the caller
// (tracs_edges_t owns it afterwards), no zero-fill, no second host copy.
template <typename T>
struct HostCol {
  T *p = nullptr;
  size_t n = 0, cap = 0;
  HostCol() {}
  HostCol(const HostCol &) = delete;
  HostCol &operator=(const HostCol &) = delete;
  ~HostCol() { host_pool_free(p); }
  size_t size() const { return n; }
  T *data() { return p; }
  T &operator[](size_t i) { return p[i]; }
  void resize(size_t m) {
    if (m > cap) {
      size_t c = cap ? cap * 2 : 1024;
      if (c < m) c = m;
      T *q = (T *)host_pool_alloc(c * sizeof(T));
      if (n) memcpy(q, p, n * sizeof(T));
      host_pool_free(p);
      p = q;
      cap = c;
    }
    n = m;
  }
  T *release() {  // never returns NULL so callers can always free()/index
    if (!p) p = (T *)host_pool_alloc(sizeof(T));
    T *q = p;
    p = nullptr;
    n = cap = 0;
    return q;
  }
};
struct HostEdges {
  HostCol<uint64_t> rows, cols, dist, ncomp, filt;
  HostCol<double> p0_log, eK, datediff;  // filled when the fused transmission path ran on the device
  bool has_trans = false;
  void *dev_packed = nullptr;  // cudaMalloc'ed, see tracs_edges_t.dev_packed
  size_t dev_packed_bytes = 0;
  ~HostEdges() { if (dev_packed) cudaFree(dev_packed); }
};
std::shared_ptr<const std::vector<double>> lgamma_table(size_t n);  // lg[x] = lgamma(x), x < n; immutable snapshot
void sweep_device(const uint8_t *dev_seqs, uint64_t n, uint64_t L, uint64_t pitch, const tracs_opts_t &o,
                  HostEdges &out, cudaStream_t st);
// every pair's distance into a dense int32 device matrix (tracs_distance_matrix_device; arguments validated by the caller)
void distance_matrix_device(const uint8_t *dev_seqs, uint64_t n, uint64_t L, uint64_t pitch, const tracs_opts_t &o, int32_t *out,
                            uint64_t ld, cudaStream_t st);

// resident sample database (db.inl; arguments validated by the caller; database and query rows 4-bit). db_open takes over
// `adopt` (the rows it points into) when given; otherwise the rows stay the caller's.
struct ResidentDb;
ResidentDb *db_open(const uint8_t *dev_rows, uint64_t n, uint64_t L, uint64_t pitch, DevBuf<uint8_t> *adopt, cudaStream_t st);
void db_query(ResidentDb &db, const uint8_t *dev_q, uint64_t nq, uint64_t qpitch, const tracs_opts_t &o, HostEdges &out, cudaStream_t st);
void db_info(const ResidentDb &db, tracs_db_info_t &out);
void db_close(ResidentDb *db);

// last step of the site-sharded sweep (shard.inl): summed candidate vectors -> edge columns
void site_shard_finish_device(const uint64_t *dev_keys, const uint32_t *dev_d, const uint32_t *dev_union, uint64_t n_keys, uint64_t n,
                              uint64_t L_total, const tracs_opts_t &o, HostEdges &out, cudaStream_t st);

// transcluster on device (trans.cu)
void trans_dist_device(const int32_t *snp, const double *dt, size_t n, double lamb, double beta, double thr,
                       double *p0_log, double *eK, cudaStream_t st);

}  // namespace tracs
