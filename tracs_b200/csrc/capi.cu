// C ABI of libtracs_b200.so (see include/tracs_b200.h for the contract and reference citations).
#include <cub/cub.cuh>
#include <math.h>
#include <signal.h>
#include <string.h>

#include <algorithm>
#include <charconv>
#include <functional>
#include <numeric>
#include <map>
#include <set>
#include <mutex>
#include <stdexcept>
#include <string>
#include <thread>
#include <unordered_map>

#include "common.cuh"

namespace tracs {

thread_local std::string g_err;
thread_local tracs_stats_t g_stats;
void set_error(const std::string &msg) { g_err = msg; }

// ---- device block cache ------------------------------------------------------------------------------
namespace {
struct DevCache {
  std::mutex mu;
  std::unordered_map<void *, std::pair<size_t, int>> live;  // block -> (size, device)
  std::multimap<size_t, std::pair<void *, int>> idle;       // size -> (block, device)
};
DevCache &dev_cache() {
  static DevCache *dc = new DevCache();  // leaked on purpose (outlives CUDA teardown)
  return *dc;
}
constexpr size_t DEV_GRANULE = 1 << 16;
}  // namespace

void *dev_cache_alloc(size_t bytes) {
  const size_t want = (bytes + DEV_GRANULE - 1) / DEV_GRANULE * DEV_GRANULE;
  int dev = 0;
  TRACS_CK(cudaGetDevice(&dev));
  DevCache &dc = dev_cache();
  {
    std::lock_guard<std::mutex> g(dc.mu);
    // smallest idle block on this device that fits without wasting more than a quarter of it (multi-GB requests) or
    // more than the request itself (smaller ones: a run over alignments of different shapes, one MSA per reference,
    // would otherwise miss the cache on every call and pay a cudaMalloc per buffer)
    const size_t slack = want >= ((size_t)4 << 30) ? want / 4 : want;
    for (auto it = dc.idle.lower_bound(want); it != dc.idle.end() && it->first <= want + slack + DEV_GRANULE; ++it) {
      if (it->second.second != dev) continue;
      void *p = it->second.first;
      dc.live[p] = {it->first, dev};
      dc.idle.erase(it);
      return p;
    }
  }
  static const bool debug = getenv("TRACS_DEBUG_ALLOC") != nullptr;
  void *p = nullptr;
  cudaError_t e = cudaMalloc(&p, want);
  if (debug) fprintf(stderr, "[tracs alloc] cudaMalloc %zu MB -> %s\n", want >> 20, cudaGetErrorName(e));
  if (e == cudaErrorMemoryAllocation) {  // make room: drop every idle block of this device and retry once
    cudaGetLastError();
    std::vector<void *> drop;
    {
      std::lock_guard<std::mutex> g(dc.mu);
      for (auto it = dc.idle.begin(); it != dc.idle.end();) {
        if (it->second.second == dev) { drop.push_back(it->second.first); it = dc.idle.erase(it); } else ++it;
      }
    }
    for (void *q : drop) cudaFree(q);
    e = cudaMalloc(&p, want);
  }
  TRACS_CK(e);
  std::lock_guard<std::mutex> g(dc.mu);
  dc.live[p] = {want, dev};
  return p;
}

void dev_cache_free(void *p) {
  if (!p) return;
  DevCache &dc = dev_cache();
  std::lock_guard<std::mutex> g(dc.mu);
  auto it = dc.live.find(p);
  if (it == dc.live.end()) return;
  dc.idle.emplace(it->second.first, std::make_pair(p, it->second.second));
  dc.live.erase(it);
}

// ---- page-locked host block cache ----------------------------------------------------------------
namespace {
struct HostPool {
  std::mutex mu;
  std::unordered_map<void *, size_t> live;             // block -> size class (bytes)
  std::unordered_map<size_t, std::vector<void *>> idle;  // size class -> cached blocks
  size_t cached_bytes = 0;
};
HostPool &host_pool() {
  static HostPool *hp = new HostPool();  // leaked on purpose: outlives static destructors / CUDA teardown
  return *hp;
}
constexpr size_t HOST_POOL_MIN = 1 << 16;         // smaller requests use malloc
constexpr size_t HOST_POOL_MAX_CACHED = 8ull << 30;
}  // namespace

void *host_pool_alloc(size_t bytes) {
  if (bytes < HOST_POOL_MIN) {
    void *p = malloc(std::max<size_t>(bytes, 8));
    if (!p) throw std::bad_alloc();
    return p;
  }
  size_t cls = HOST_POOL_MIN;
  while (cls < bytes) cls <<= 1;
  HostPool &hp = host_pool();
  {
    std::lock_guard<std::mutex> g(hp.mu);
    auto it = hp.idle.find(cls);
    if (it != hp.idle.end() && !it->second.empty()) {
      void *p = it->second.back();
      it->second.pop_back();
      hp.cached_bytes -= cls;
      hp.live[p] = cls;
      return p;
    }
  }
  void *p = nullptr;
  if (cudaHostAlloc(&p, cls, cudaHostAllocDefault) != cudaSuccess) {
    cudaGetLastError();
    p = malloc(cls);  // still correct, just a slower copy
    if (!p) throw std::bad_alloc();
    return p;
  }
  std::lock_guard<std::mutex> g(hp.mu);
  hp.live[p] = cls;
  return p;
}

void host_pool_free(void *p) {
  if (!p) return;
  HostPool &hp = host_pool();
  {
    std::lock_guard<std::mutex> g(hp.mu);
    auto it = hp.live.find(p);
    if (it == hp.live.end()) {
      // not a pool block
    } else {
      const size_t cls = it->second;
      hp.live.erase(it);
      if (hp.cached_bytes + cls <= HOST_POOL_MAX_CACHED) {
        hp.idle[cls].push_back(p);
        hp.cached_bytes += cls;
      } else {
        cudaFreeHost(p);
      }
      return;
    }
  }
  free(p);
}

// ---- SIGINT during a call ---------------------------------------------------------------------------------
namespace {
volatile sig_atomic_t g_sigint = 0;
int g_scope_depth = 0;
struct sigaction g_prev_action;
void on_sigint(int) { g_sigint = 1; }
}  // namespace

InterruptScope::InterruptScope() {
  const char *env = getenv("TRACS_SIGINT");
  if (env && !strcmp(env, "0")) return;
  if (g_scope_depth++ == 0) {
    g_sigint = 0;
    struct sigaction sa;
    memset(&sa, 0, sizeof sa);
    sa.sa_handler = on_sigint;
    sigemptyset(&sa.sa_mask);
    sa.sa_flags = SA_RESTART;
    sigaction(SIGINT, &sa, &g_prev_action);
  }
}
InterruptScope::~InterruptScope() {
  const char *env = getenv("TRACS_SIGINT");
  if (env && !strcmp(env, "0")) return;
  if (--g_scope_depth == 0) sigaction(SIGINT, &g_prev_action, nullptr);
}
void check_interrupt() {
  if (g_sigint) throw Interrupted{};
}

void require_device() {
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0)
    throw std::runtime_error(std::string("tracs_b200: no CUDA device available (") + cudaGetErrorString(e) +
                             "); this library has no CPU fallback");
}

template <typename T>
static T *dup_array(const std::vector<T> &v) {
  T *p = (T *)host_pool_alloc(std::max<size_t>(1, v.size()) * sizeof(T));
  if (!v.empty()) memcpy(p, v.data(), v.size() * sizeof(T));
  return p;
}

static void finish_edges(HostEdges &he, const tracs_opts_t &o, uint64_t n, uint64_t L, tracs_edges_t *out,
                         cudaStream_t st) {
  const size_t E = he.rows.size();
  out->n_edges = E;
  const bool have_filt = o.filter && he.filt.size() == E;
  out->seq_length = L;
  if (he.ncomp.size() != E) {  // compared sites not requested: zeros
    he.ncomp.resize(E);
    if (E) memset(he.ncomp.data(), 0, E * sizeof(uint64_t));
  }
  if (o.want_trans && o.days && he.has_trans) {
    out->p0_log = he.p0_log.release();
    out->eK = he.eK.release();
    out->datediff = he.datediff.release();
  } else if (o.want_trans && o.days) {
    // key table too large for the device-side path: unique (N, delta) keys are collected on the host.
    // tracs/transcluster.py:26-36: seconds since epoch -> |dt| / SECONDS_IN_YEAR -> trans_dist
    std::vector<double> dt(E), p0(E), ek(E);
    std::vector<int32_t> d32(E);
    for (size_t e = 0; e < E; ++e) {
      const double ti = (double)o.days[he.rows[e]] * 86400.0, tj = (double)o.days[he.cols[e]] * 86400.0;
      dt[e] = fabs(ti - tj) / 31556952.0;
      d32[e] = (int32_t)(have_filt ? he.filt[e] : he.dist[e]);
    }
    trans_dist_device(d32.data(), dt.data(), E, o.lamb, o.beta, o.threshold_Ek, p0.data(), ek.data(), st);
    out->p0_log = dup_array(p0);
    out->eK = dup_array(ek);
    out->datediff = dup_array(dt);
  }
  // filter off: the reference's filt_distances is a vector of zeros (src/pairsnp.hpp:452); here the column is simply
  // absent (NULL) and the bindings synthesise the zeros -- zero-filling E x 8 bytes per call cost 2 ms at 2.5 M edges
  out->filt = have_filt ? he.filt.release() : nullptr;
  out->dev_packed = he.dev_packed;
  out->dev_packed_bytes = he.dev_packed_bytes;
  he.dev_packed = nullptr;
  out->rows = he.rows.release();
  out->cols = he.cols.release();
  out->dist = he.dist.release();
  out->ncomp = he.ncomp.release();
  (void)n;
}

// ---- synthetic alignment generator (SURVEY 8d, generator G; hash-based, seeded) ---------------
__device__ __forceinline__ uint64_t mix64(uint64_t x) {
  x ^= x >> 33; x *= 0xff51afd7ed558ccdull;
  x ^= x >> 33; x *= 0xc4ceb9fe1a85ec53ull;
  x ^= x >> 33;
  return x;
}
struct SynthDev {
  uint64_t n, L, pitch, seed;
  uint32_t thr_var24, thr_found16, thr_gc16, n_clusters;
  uint32_t thr_priv32, thr_N32, thr_amb16, n_days, gaps;
  uint64_t gap_len;
  uint64_t site_offset, L_total;  // this buffer holds columns [site_offset, site_offset + L) of L_total
  uint32_t packed;                // write 4-bit masks (two sites per byte) instead of ASCII
};
__global__ void k_synth(SynthDev c, uint8_t *__restrict__ seqs) {
  const uint64_t chunks = (c.packed ? c.pitch * 2 : c.pitch) / 16;  // 16 sites per thread
  const uint64_t gid = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (gid >= c.n * chunks) return;
  const uint64_t s = gid / chunks, ch = gid % chunks;
  const uint32_t cluster = (uint32_t)(mix64(c.seed * 0x100000001b3ull + 0x51ull + s) % c.n_clusters);
  uint64_t g0[4] = {~0ull, ~0ull, ~0ull, ~0ull};
  for (uint32_t r = 0; r < c.gaps && r < 4; ++r)
    if (c.L_total > c.gap_len) g0[r] = mix64(c.seed ^ (0xabcdefull + s * 8 + r)) % (c.L_total - c.gap_len);
  const char B[4] = {'A', 'C', 'G', 'T'};
  // 2-base IUPAC codes indexed [b][o]
  const char AMB[4][4] = {{'A', 'M', 'R', 'W'}, {'M', 'C', 'S', 'Y'}, {'R', 'S', 'G', 'K'}, {'W', 'Y', 'K', 'T'}};
  uint32_t outw[4];
  uint32_t nibw[2] = {0u, 0u};
  for (int q = 0; q < 4; ++q) {
    uint32_t w = 0;
    for (int t = 0; t < 4; ++t) {
      const uint64_t lsite = ch * 16 + q * 4 + t;
      const uint64_t site = c.site_offset + lsite;  // every random draw is keyed on the GLOBAL site
      char chv = 'N';
      if (lsite < c.L) {
        const uint64_t hs = mix64(c.seed * 0x9E3779B97F4A7C15ull + site);
        uint32_t b;
        if ((hs & 0xFFFFu) < c.thr_gc16) b = ((hs >> 60) & 1) ? 1u : 2u; else b = ((hs >> 60) & 1) ? 0u : 3u;
        const bool isvar = ((hs >> 16) & 0xFFFFFFu) < c.thr_var24;
        bool amb = false;
        uint32_t other = 0;
        if (isvar) {
          const uint64_t hc = mix64(hs ^ ((uint64_t)(cluster + 1) * 0xD6E8FEB86659FD93ull));
          if ((hc & 0xFFFFu) < c.thr_found16) b = (b + 1 + (uint32_t)((hc >> 16) % 3)) & 3u;
          const uint64_t hp = mix64(hs ^ ((s + 1) * 0xA24BAED4963EE407ull));
          if ((uint32_t)hp < c.thr_priv32) b = (b + 1 + (uint32_t)((hp >> 32) % 3)) & 3u;
          if (((hp >> 40) & 0xFFFFu) < c.thr_amb16) { amb = true; other = (b + 1 + (uint32_t)((hp >> 56) % 3)) & 3u; }
        }
        chv = amb ? AMB[b][other] : B[b];
        const uint64_t hn = mix64((c.seed + 0x7777ull) * 0xC2B2AE3D27D4EB4Full + s * c.L_total + site);
        if ((uint32_t)hn < c.thr_N32) chv = 'N';
        for (int r = 0; r < 4; ++r) if (site >= g0[r] && site - g0[r] < c.gap_len) chv = '-';
      }
      w |= (uint32_t)(uint8_t)chv << (8 * t);
      nibw[q >> 1] |= base_mask((uint32_t)(uint8_t)chv) << (4 * ((q & 1) * 4 + t));
    }
    outw[q] = w;
  }
  if (c.packed) *reinterpret_cast<uint2 *>(seqs + s * c.pitch + ch * 8) = make_uint2(nibw[0], nibw[1]);
  else *reinterpret_cast<uint4 *>(seqs + s * c.pitch + ch * 16) = make_uint4(outw[0], outw[1], outw[2], outw[3]);
}
__global__ void k_synth_days(uint64_t n, uint64_t seed, uint32_t n_days, int32_t *days) {
  uint64_t s = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (s < n) days[s] = (int32_t)(mix64(seed * 31ull + 0xDA7Eull + s) % (n_days ? n_days : 1));
}

// ---- INT pipe peak micro-benchmarks -------------------------------------------------------------
template <int MODE>
__global__ void __launch_bounds__(256) k_peak(uint32_t *out, int iters, long long *cycles) {
  uint32_t x[48];
#pragma unroll
  for (int i = 0; i < 48; ++i) x[i] = threadIdx.x * 2654435761u + i * 40503u + blockIdx.x;
  uint32_t acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  const long long t0 = clock64();
  for (int it = 0; it < iters; ++it) {
    if (MODE == 0) {  // LOP3 only: 16 independent chains
#pragma unroll
      for (int r = 0; r < 4; ++r)
#pragma unroll
        for (int i = 0; i < 16; ++i)
          asm volatile("lop3.b32 %0, %0, %1, %2, 0x96;" : "+r"(x[i]) : "r"(x[(i + 1) & 15]), "r"(x[(i + 5) & 15]));
    } else if (MODE == 1) {  // POPC only
#pragma unroll
      for (int r = 0; r < 4; ++r)
#pragma unroll
        for (int i = 0; i < 16; ++i) asm volatile("popc.b32 %0, %0;" : "+r"(x[i]));
    } else if (MODE == 2) {  // IADD only
#pragma unroll
      for (int r = 0; r < 4; ++r)
#pragma unroll
        for (int i = 0; i < 16; ++i) asm volatile("add.u32 %0, %0, %1;" : "+r"(x[i]) : "r"(x[(i + 3) & 15]));
    } else {
      // the sweep's per-word-pair mix on register operands: 8 row quads x 4 col quads = 32
      // distinct word-pairs per iteration (4 LOP3 + POPC + ADD each); every row quad changes each
      // iteration so nothing is loop-invariant or common between pairs.
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          uint32_t m;
          asm volatile("and.b32 %0, %1, %2;" : "=r"(m) : "r"(x[i * 4 + 0]), "r"(x[32 + j * 4 + 0]));
          asm volatile("lop3.b32 %0, %1, %2, %0, 0xEA;" : "+r"(m) : "r"(x[i * 4 + 1]), "r"(x[32 + j * 4 + 1]));
          asm volatile("lop3.b32 %0, %1, %2, %0, 0xEA;" : "+r"(m) : "r"(x[i * 4 + 2]), "r"(x[32 + j * 4 + 2]));
          asm volatile("lop3.b32 %0, %1, %2, %0, 0xEA;" : "+r"(m) : "r"(x[i * 4 + 3]), "r"(x[32 + j * 4 + 3]));
          uint32_t p;
          asm volatile("popc.b32 %0, %1;" : "=r"(p) : "r"(m));
          if (MODE == 3) acc[(i + j) & 7] += p;
          else asm volatile("mad.lo.u32 %0, %1, 1, %0;" : "+r"(acc[(i + j) & 7]) : "r"(p));
        }
#pragma unroll
      for (int i = 0; i < 8; ++i) x[i * 4] += acc[i] + it;
    }
  }
  const long long t1 = clock64();
  uint32_t s = 0;
#pragma unroll
  for (int i = 0; i < 48; ++i) s ^= x[i];
#pragma unroll
  for (int i = 0; i < 8; ++i) s += acc[i];
  out[blockIdx.x * blockDim.x + threadIdx.x] = s;
  if (threadIdx.x == 0 && blockIdx.x == 0) *cycles = t1 - t0;
}

}  // namespace tracs

using namespace tracs;

extern "C" {

const char *tracs_last_error(void) { return g_err.c_str(); }

int tracs_last_stats(tracs_stats_t *out) {
  *out = g_stats;
  return 0;
}

int tracs_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return n;
}

int tracs_set_device(int device) {
  return guarded([&] { TRACS_CK(cudaSetDevice(device)); });
}

void tracs_edges_free(tracs_edges_t *e) {
  if (!e) return;
  host_pool_free(e->rows); host_pool_free(e->cols); host_pool_free(e->dist); host_pool_free(e->filt); host_pool_free(e->ncomp);
  host_pool_free(e->p0_log); host_pool_free(e->eK); host_pool_free(e->datediff);
  if (e->dev_packed) cudaFree(e->dev_packed);
  if (e->names) {
    for (size_t i = 0; i < e->n_names; ++i) free(e->names[i]);
    free(e->names);
  }
  memset(e, 0, sizeof *e);
}

static tracs_opts_t normalise(const tracs_opts_t *opts, size_t n) {
  tracs_opts_t o;
  if (opts) o = *opts; else { memset(&o, 0, sizeof o); o.dist = INT32_MAX; o.want_ncomp = 1; }
  if (o.i_end == 0 || o.i_end > n) o.i_end = n;
  if (o.shard_world <= 0) { o.shard_world = 1; o.shard_rank = 0; }
  return o;
}

// Host -> device copy of a row-major byte matrix. Page-locked sources go to the copy engine directly. A large
// PAGEABLE source (numpy arrays, the FASTA reader's buffer) would be staged by the driver through one thread;
// here a few workers copy row chunks into their own page-locked double buffers and queue each chunk on their
// own stream, so the memcpy of one chunk overlaps the DMA of the others.
static void h2d_rows(uint8_t *dev, size_t dpitch, const uint8_t *src, size_t spitch, size_t width, size_t rows, cudaStream_t st) {
  cudaPointerAttributes attr;
  const bool pinned = cudaPointerGetAttributes(&attr, src) == cudaSuccess && attr.type != cudaMemoryTypeUnregistered;
  cudaGetLastError();
  const char *env_min = getenv("TRACS_H2D_STAGE_MIN");  // read per call: tests switch it
  const size_t min_bytes = env_min ? (size_t)strtoull(env_min, nullptr, 10) : ((size_t)256 << 20);
  if (pinned || width * rows < min_bytes) {
    TRACS_CK(cudaMemcpy2DAsync(dev, dpitch, src, spitch, width, rows, cudaMemcpyHostToDevice, st));
    return;
  }
  const size_t CH = (size_t)32 << 20;  // staging buffer
  if (width > CH) {                    // very long rows: leave it to the driver
    TRACS_CK(cudaMemcpy2DAsync(dev, dpitch, src, spitch, width, rows, cudaMemcpyHostToDevice, st));
    return;
  }
  TRACS_CK(cudaStreamSynchronize(st));  // work queued on `st` for the destination (padding fill) comes first
  const char *env_thr = getenv("TRACS_H2D_THREADS");
  const unsigned h2d_threads = env_thr ? (unsigned)std::max(1, atoi(env_thr)) : 12u;
  const size_t rows_per = std::max<size_t>(1, CH / width);
  const size_t n_chunks = (rows + rows_per - 1) / rows_per;
  const int T = (int)std::min<size_t>(n_chunks, std::max(1u, std::min(h2d_threads, std::thread::hardware_concurrency())));
  int devid = 0;
  TRACS_CK(cudaGetDevice(&devid));
  std::vector<std::string> errs((size_t)T);
  std::vector<std::thread> pool;
  for (int t = 0; t < T; ++t)
    pool.emplace_back([&, t] {
      cudaStream_t ws = nullptr;
      cudaEvent_t ev[2] = {nullptr, nullptr};
      uint8_t *buf[2] = {nullptr, nullptr};
      try {
        TRACS_CK(cudaSetDevice(devid));
        TRACS_CK(cudaStreamCreateWithFlags(&ws, cudaStreamNonBlocking));
        for (int b = 0; b < 2; ++b) {
          buf[b] = (uint8_t *)host_pool_alloc(CH);
          TRACS_CK(cudaEventCreateWithFlags(&ev[b], cudaEventDisableTiming));
        }
        int turn = 0;
        for (size_t c = (size_t)t; c < n_chunks; c += (size_t)T, turn ^= 1) {
          const size_t r0 = c * rows_per, nr = std::min(rows_per, rows - r0);
          TRACS_CK(cudaEventSynchronize(ev[turn]));  // the DMA that last read this buffer is done
          for (size_t r = 0; r < nr; ++r) memcpy(buf[turn] + r * width, src + (r0 + r) * spitch, width);
          TRACS_CK(cudaMemcpy2DAsync(dev + r0 * dpitch, dpitch, buf[turn], width, width, nr, cudaMemcpyHostToDevice, ws));
          TRACS_CK(cudaEventRecord(ev[turn], ws));
        }
        TRACS_CK(cudaStreamSynchronize(ws));
      } catch (const std::exception &e) {
        errs[t] = e.what();
      }
      for (int b = 0; b < 2; ++b) {
        if (ev[b]) cudaEventDestroy(ev[b]);
        if (buf[b]) host_pool_free(buf[b]);
      }
      if (ws) cudaStreamDestroy(ws);
    });
  for (auto &th : pool) th.join();
  for (auto &e : errs)
    if (!e.empty()) throw std::runtime_error("host to device staging: " + e);
  (void)st;  // the workers have synchronised their streams: the data is in place for any stream
}

// Host matrix -> device-resident PACKED alignment (pack4.inl layout), streamed in sample chunks: the copy of chunk
// c + 1 (copy stream) overlaps the ASCII -> nibble encode of chunk c (compute stream), and only two ASCII chunks are
// ever resident, so an alignment whose ASCII form exceeds the device (100 000 x 2 Mb = 200 GB) still goes through.
// A host matrix that is already packed is copied straight into place.
static size_t packed_pitch(size_t L) { return std::max<size_t>(16, (L + 31) / 32 * 16); }

static void stream_host_to_packed(const uint8_t *seqs, size_t n, size_t L, size_t hpitch, bool host_is_packed, DevBuf<uint8_t> &nib,
                                  size_t &pitch4, cudaStream_t st) {
  pitch4 = packed_pitch(L);
  nib.alloc(n * pitch4);
  if (n == 0 || L == 0) return;
  if (host_is_packed) {
    h2d_rows(nib.p, pitch4, seqs, hpitch, (L + 1) / 2, n, st);
    g_stats.h2d_bytes += (uint64_t)n * ((L + 1) / 2);
    return;
  }
  const size_t apitch = (L + 31) / 32 * 32;
  const char *env_ch = getenv("TRACS_STREAM_CHUNK_BYTES");  // tests shrink it to exercise many chunks
  const size_t chunk_bytes = env_ch ? (size_t)strtoull(env_ch, nullptr, 10) : ((size_t)256 << 20);
  const size_t R = std::min(n, std::max<size_t>(1, chunk_bytes / apitch));
  DevBuf<uint8_t> stage0(R * apitch), stage1(n > R ? R * apitch : 0);
  uint8_t *stage[2] = {stage0.p, stage1.p ? stage1.p : stage0.p};
  static thread_local cudaStream_t cp = nullptr;
  static thread_local cudaEvent_t ev_copied[2] = {nullptr, nullptr}, ev_free[2] = {nullptr, nullptr};
  static thread_local int cp_dev = -1;
  int dev = 0;
  TRACS_CK(cudaGetDevice(&dev));
  if (!cp || cp_dev != dev) {
    cp_dev = dev;
    TRACS_CK(cudaStreamCreateWithFlags(&cp, cudaStreamNonBlocking));
    for (int b = 0; b < 2; ++b) {
      TRACS_CK(cudaEventCreateWithFlags(&ev_copied[b], cudaEventDisableTiming));
      TRACS_CK(cudaEventCreateWithFlags(&ev_free[b], cudaEventDisableTiming));
    }
  }
  size_t c = 0;
  for (size_t r0 = 0; r0 < n; r0 += R, ++c) {
    const int b = (int)(c & 1);
    const size_t nr = std::min(R, n - r0);
    check_interrupt();
    if (c >= 2) TRACS_CK(cudaStreamWaitEvent(cp, ev_free[b], 0));  // the encode that last read this buffer is done
    h2d_rows(stage[b], apitch, seqs + r0 * hpitch, hpitch, L, nr, cp);
    TRACS_CK(cudaEventRecord(ev_copied[b], cp));
    TRACS_CK(cudaStreamWaitEvent(st, ev_copied[b], 0));
    encode_rows_device(stage[b], nr, L, apitch, nib.p + r0 * pitch4, pitch4, st);
    TRACS_CK(cudaEventRecord(ev_free[b], st));
  }
  TRACS_CK(cudaStreamSynchronize(st));  // the staging buffers go back to the cache
  g_stats.h2d_bytes += (uint64_t)n * L;
}

// RowSink of the FASTA entry point: rows arrive from the reader while it is still parsing; each batch is copied
// into a page-locked staging buffer, sent to the device on a copy stream and encoded into the resident packed
// alignment on the compute stream. Two staging slots: the host memcpy of batch k + 1 overlaps the DMA of batch k,
// the encode of batch k overlaps both. The packed alignment grows by doubling when the record count is not known
// up front (gz / sequential reader).
struct DeviceRowStreamer : RowSink {
  cudaStream_t st, cp = nullptr;
  cudaEvent_t ev_copied[2] = {nullptr, nullptr}, ev_free[2] = {nullptr, nullptr};
  bool used[2] = {false, false};
  uint8_t *hbuf[2] = {nullptr, nullptr};
  DevBuf<uint8_t> dbuf[2], nib;
  uint64_t L = 0, pitch4 = 0, apitch = 0, cap_rows = 0, n_rows = 0, hint_rows = 0;
  size_t slot_bytes = 0;
  unsigned turn = 0;
  explicit DeviceRowStreamer(cudaStream_t s) : st(s) {
    TRACS_CK(cudaStreamCreateWithFlags(&cp, cudaStreamNonBlocking));
    for (int b = 0; b < 2; ++b) {
      TRACS_CK(cudaEventCreateWithFlags(&ev_copied[b], cudaEventDisableTiming));
      TRACS_CK(cudaEventCreateWithFlags(&ev_free[b], cudaEventDisableTiming));
    }
  }
  ~DeviceRowStreamer() override {
    cudaStreamSynchronize(cp);
    cudaStreamSynchronize(st);
    for (int b = 0; b < 2; ++b) {
      if (hbuf[b]) host_pool_free(hbuf[b]);
      if (ev_copied[b]) cudaEventDestroy(ev_copied[b]);
      if (ev_free[b]) cudaEventDestroy(ev_free[b]);
    }
    if (cp) cudaStreamDestroy(cp);
  }
  void expect(uint64_t total_rows, uint64_t) override { hint_rows = std::max(hint_rows, total_rows); }
  void reset() override {
    TRACS_CK(cudaStreamSynchronize(cp));
    TRACS_CK(cudaStreamSynchronize(st));
    n_rows = 0;
  }
  void reserve_rows(uint64_t want) {
    if (want <= cap_rows) return;
    uint64_t c = std::max<uint64_t>(std::max(want, hint_rows), cap_rows * 2);
    DevBuf<uint8_t> bigger(c * pitch4);
    if (n_rows) {
      TRACS_CK(cudaStreamSynchronize(cp));
      TRACS_CK(cudaMemcpyAsync(bigger.p, nib.p, n_rows * pitch4, cudaMemcpyDeviceToDevice, st));
      TRACS_CK(cudaStreamSynchronize(st));
    }
    std::swap(nib.p, bigger.p);
    std::swap(nib.n, bigger.n);
    cap_rows = c;
  }
  void rows(const uint8_t *p, uint64_t first_row, uint64_t count, uint64_t Lr) override {
    if (count == 0) return;
    if (L == 0) {
      if (Lr == 0) return;
      L = Lr;
      pitch4 = std::max<uint64_t>(16, (L + 31) / 32 * 16);
      apitch = (L + 31) / 32 * 32;
      const char *env_ch = getenv("TRACS_STREAM_CHUNK_BYTES");
      slot_bytes = std::max<size_t>(apitch, env_ch ? (size_t)strtoull(env_ch, nullptr, 10) : ((size_t)32 << 20));
      for (int b = 0; b < 2; ++b) {
        hbuf[b] = (uint8_t *)host_pool_alloc(slot_bytes);
        dbuf[b].alloc(slot_bytes);
      }
    }
    if (Lr != L) throw std::runtime_error("Error reading FASTA, variable sequence lengths!");
    if (first_row != n_rows) throw std::runtime_error("internal error: rows streamed out of order");
    check_interrupt();
    reserve_rows(first_row + count);
    const uint64_t R = std::max<uint64_t>(1, slot_bytes / apitch);
    for (uint64_t r0 = 0; r0 < count; r0 += R) {
      const uint64_t nr = std::min(R, count - r0);
      const int b = (int)(turn++ & 1u);
      if (used[b]) TRACS_CK(cudaEventSynchronize(ev_free[b]));  // the encode that read this slot's device half is done (so is its DMA)
      for (uint64_t r = 0; r < nr; ++r) memcpy(hbuf[b] + r * L, p + (r0 + r) * L, L);
      TRACS_CK(cudaMemcpy2DAsync(dbuf[b].p, apitch, hbuf[b], L, L, nr, cudaMemcpyHostToDevice, cp));
      TRACS_CK(cudaEventRecord(ev_copied[b], cp));
      TRACS_CK(cudaStreamWaitEvent(st, ev_copied[b], 0));
      encode_rows_device(dbuf[b].p, nr, L, apitch, nib.p + (first_row + r0) * pitch4, pitch4, st);
      TRACS_CK(cudaEventRecord(ev_free[b], st));
      used[b] = true;
    }
    n_rows = first_row + count;
    g_stats.h2d_bytes += count * L;
  }
  void finish() {
    TRACS_CK(cudaStreamSynchronize(cp));
    TRACS_CK(cudaStreamSynchronize(st));
  }
};

int tracs_encode_packed(const uint8_t *dev_ascii, size_t rows, size_t L, size_t pitch, uint8_t *dev_nib, size_t pitch_bytes) {
  return guarded([&] {
    require_device();
    encode_rows_device(dev_ascii, rows, L, pitch, dev_nib, pitch_bytes, 0);
    TRACS_CK(cudaStreamSynchronize(0));
  });
}

int tracs_pairsnp_packed(const uint8_t *dev_nib, size_t n, size_t L, size_t pitch_bytes, const tracs_opts_t *opts,
                         tracs_edges_t *out) {
  memset(out, 0, sizeof *out);
  memset(&g_stats, 0, sizeof g_stats);
  return guarded([&] {
    require_device();
    InterruptScope sigint;
    tracs_opts_t o = normalise(opts, n);
    o.packed_input = 1;
    HostEdges he;
    sweep_device(dev_nib, n, L, pitch_bytes, o, he, 0);
    finish_edges(he, o, n, L, out, 0);
  });
}

int tracs_site_shard_finish(const uint64_t *dev_keys, const uint32_t *dev_d, const uint32_t *dev_union, size_t n_keys,
                            size_t n_samples, size_t L_total, const tracs_opts_t *opts, tracs_edges_t *out) {
  memset(out, 0, sizeof *out);
  memset(&g_stats, 0, sizeof g_stats);
  return guarded([&] {
    require_device();
    if (!opts) throw std::runtime_error("site shard: options required");
    tracs_opts_t o = normalise(opts, n_samples);
    o.filter = 0;
    HostEdges he;
    site_shard_finish_device(dev_keys, dev_d, dev_union, n_keys, n_samples, L_total, o, he, 0);
    finish_edges(he, o, n_samples, L_total, out, 0);
  });
}

int tracs_pairsnp_device(const uint8_t *dev_seqs, size_t n, size_t L, size_t pitch, const tracs_opts_t *opts,
                         tracs_edges_t *out) {
  memset(out, 0, sizeof *out);
  memset(&g_stats, 0, sizeof g_stats);
  return guarded([&] {
    require_device();
    InterruptScope sigint;
    tracs_opts_t o = normalise(opts, n);
    HostEdges he;
    sweep_device(dev_seqs, n, L, pitch, o, he, 0);
    finish_edges(he, o, n, L, out, 0);
  });
}

int tracs_pairsnp_host(const uint8_t *seqs, size_t n, size_t L, size_t pitch, const tracs_opts_t *opts,
                       tracs_edges_t *out) {
  memset(out, 0, sizeof *out);
  memset(&g_stats, 0, sizeof g_stats);
  return guarded([&] {
    require_device();
    InterruptScope sigint;
    tracs_opts_t o = normalise(opts, n);
    HostEdges he;
    const char *mode = getenv("TRACS_HOST_INGEST");  // "ascii": keep the ASCII matrix resident and pack it directly
    if (n > 0 && !o.packed_input && mode && !strcmp(mode, "ascii")) {
      const size_t dp = std::max<size_t>(32, (L + 31) / 32 * 32);
      DevBuf<uint8_t> d(n * dp);
      if (dp != L) TRACS_CK(cudaMemsetAsync(d.p, 'N', n * dp, 0));
      if (L > 0) h2d_rows(d.p, dp, seqs, pitch, L, n, 0);
      sweep_device(d.p, n, L, dp, o, he, 0);
      g_stats.h2d_bytes += (uint64_t)n * L;
    } else if (n > 0) {
      DevBuf<uint8_t> nib;
      size_t pitch4 = 0;
      stream_host_to_packed(seqs, n, L, pitch, o.packed_input != 0, nib, pitch4, 0);
      o.packed_input = 1;
      sweep_device(nib.p, n, L, pitch4, o, he, 0);  // adds to the counters of the call
    }
    finish_edges(he, o, n, L, out, 0);
  });
}

}  // extern "C"

// ---- dense distance matrix (tracs_distance_matrix_*) ----------------------------------------------------
namespace tracs {
struct DenseShape {
  uint64_t rows = 0, cols = 0;
};
// Pitch of an input matrix of n rows: host rows hold L ASCII bytes or (L + 1) / 2 packed bytes; device rows follow the
// ingest's alignment rules. Host code only.
static void check_pitch(const char *pre, size_t pitch, size_t L, bool packed, bool host_input, size_t n) {
  bool pitch_ok;
  if (host_input) pitch_ok = packed ? pitch >= (L + 1) / 2 : pitch >= L;
  else if (packed) pitch_ok = pitch % 16 == 0 && pitch * 2 >= std::max<size_t>(32, (L + 31) / 32 * 32);
  else pitch_ok = pitch % 32 == 0 && pitch >= (L + 31) / 32 * 32;
  if (!pitch_ok && n > 0)
    throw std::runtime_error(std::string(pre) + "pitch (" + std::to_string(pitch) + ") " +
                             (host_input ? (packed ? "must hold (L + 1) / 2 bytes" : "must be >= L")
                                         : (packed ? "must be a multiple of 16 bytes and hold L rounded up to 32 sites"
                                                   : "must be a multiple of 32 and >= L rounded up to 32")));
}
// Argument check of the dense entry points. Host code only (no device call), so it runs before require_device().
static DenseShape dense_check(const tracs_opts_t *opts, size_t n, size_t L, size_t pitch, size_t ld, const void *out, bool host_input) {
  const tracs_opts_t o = normalise(opts, n);
  const char *pre = "distance matrix: ";
  if (o.dist != INT32_MAX)
    throw std::runtime_error(std::string(pre) + "opts->dist must be INT32_MAX (every pair); a threshold is what tracs_pairsnp_* is for");
  if (o.filter) throw std::runtime_error(std::string(pre) + "opts->filter (recombination filter) applies to the thresholded pair list only");
  if (o.want_trans || o.days) throw std::runtime_error(std::string(pre) + "opts->want_trans / opts->days (transmission likelihood) apply to the thresholded pair list only");
  if (o.keep_on_device) throw std::runtime_error(std::string(pre) + "opts->keep_on_device applies to the edge list only");
  if (o.shard_world > 1) throw std::runtime_error(std::string(pre) + "opts->shard_world > 1: the dense matrix is computed on one GPU");
  if (o.sweep_variant < 0 || o.sweep_variant > 2) throw std::runtime_error(std::string(pre) + "opts->sweep_variant must be 0, 1 or 2");
  if (n >= (1ull << 31)) throw std::runtime_error(std::string(pre) + "n: too many samples");
  const uint64_t i_end = opts ? opts->i_end : 0, j_start = opts ? opts->j_start : 0;
  DenseShape sh;
  if ((i_end == 0 || i_end == n) && j_start == 0) {
    sh.rows = sh.cols = n;  // square
  } else if (i_end >= 1 && j_start >= i_end && j_start < n) {
    sh.rows = i_end;  // query x db rectangle
    sh.cols = n - j_start;
  } else {
    throw std::runtime_error(std::string(pre) + "opts->i_end / opts->j_start: either i_end = 0 or n with j_start = 0 (square matrix), or "
                             "0 < i_end <= j_start < n (rows [0, i_end) x cols [j_start, n))");
  }
  if (ld < sh.cols) throw std::runtime_error(std::string(pre) + "ld (" + std::to_string(ld) + ") is smaller than the column count (" + std::to_string(sh.cols) + ")");
  if (!out && sh.rows && sh.cols) throw std::runtime_error(std::string(pre) + "out is NULL");
  const bool packed = o.packed_input != 0;
  check_pitch(pre, pitch, L, packed, host_input, n);
  return sh;
}

static std::string dense_too_large(uint64_t rows, uint64_t cols) {
  size_t free_b = 0, total_b = 0;
  if (cudaMemGetInfo(&free_b, &total_b) != cudaSuccess) cudaGetLastError();
  char b[512];
  snprintf(b, sizeof b,
           "distance matrix: a %llu x %llu int32 matrix (%.1f GB) and the ingest of the alignment do not fit in device memory "
           "(%.1f GB on the device): for an alignment this large ask for the thresholded pair list (tracs_pairsnp_* with a finite dist)",
           (unsigned long long)rows, (unsigned long long)cols, (double)rows * (double)cols * 4.0 / 1e9, (double)total_b / 1e9);
  return b;
}

// a device allocation that fails inside the call becomes the "does not fit" message (the buffers already taken go back
// to the cache on the way out, so the library stays usable)
template <typename F>
static void dense_fit_guard(uint64_t rows, uint64_t cols, F &&f) {
  try {
    f();
  } catch (const CudaError &e) {
    if (e.msg.find("cudaErrorMemoryAllocation") == std::string::npos) throw;
    cudaGetLastError();
    throw std::runtime_error(dense_too_large(rows, cols));
  }
}
}  // namespace tracs

extern "C" {

int tracs_distance_matrix_device(const uint8_t *dev_seqs, size_t n, size_t L, size_t pitch, const tracs_opts_t *opts, int32_t *dev_out,
                                 size_t ld) {
  memset(&g_stats, 0, sizeof g_stats);
  return guarded([&] {
    const DenseShape sh = dense_check(opts, n, L, pitch, ld, dev_out, false);
    require_device();
    InterruptScope sigint;
    if (sh.rows == 0 || sh.cols == 0) return;
    const tracs_opts_t o = normalise(opts, n);
    dense_fit_guard(sh.rows, sh.cols, [&] { distance_matrix_device(dev_seqs, n, L, pitch, o, dev_out, ld, 0); });
  });
}

int tracs_distance_matrix_host(const uint8_t *seqs, size_t n, size_t L, size_t pitch, const tracs_opts_t *opts, int32_t *out,
                               size_t ld) {
  memset(&g_stats, 0, sizeof g_stats);
  return guarded([&] {
    const DenseShape sh = dense_check(opts, n, L, pitch, ld, out, true);
    require_device();
    InterruptScope sigint;
    if (sh.rows == 0 || sh.cols == 0) return;
    tracs_opts_t o = normalise(opts, n);
    const uint64_t m_bytes = sh.rows * sh.cols * 4, in_bytes = (uint64_t)n * std::max<uint64_t>(16, (L + 31) / 32 * 16);
    size_t free_b = 0, total_b = 0;
    TRACS_CK(cudaMemGetInfo(&free_b, &total_b));
    if (m_bytes + in_bytes > total_b) throw std::runtime_error(dense_too_large(sh.rows, sh.cols));
    dense_fit_guard(sh.rows, sh.cols, [&] {
      DevBuf<int32_t> m(sh.rows * sh.cols);  // library-owned, ld = cols
      {
        DevBuf<uint8_t> nib;
        size_t pitch4 = 0;
        stream_host_to_packed(seqs, n, L, pitch, o.packed_input != 0, nib, pitch4, 0);
        o.packed_input = 1;
        distance_matrix_device(nib.p, n, L, pitch4, o, m.p, sh.cols, 0);
      }
      Timer T(0);
      T.start();
      TRACS_CK(cudaMemcpy2DAsync(out, ld * 4, m.p, sh.cols * 4, sh.cols * 4, sh.rows, cudaMemcpyDeviceToHost, 0));
      TRACS_CK(cudaStreamSynchronize(0));
      g_stats.ms_d2h += T.stop();
      g_stats.ms_total += g_stats.ms_d2h;
      g_stats.d2h_bytes += m_bytes;
    });
  });
}

}  // extern "C"

// ---- resident sample database (tracs_db_*) ----------------------------------------------------------------------
namespace tracs {
namespace {
std::mutex g_db_mu;
std::set<ResidentDb *> g_db_live;  // handles between open and close: anything else is refused, never dereferenced
}  // namespace

static ResidentDb *db_lookup(void *h) {
  std::lock_guard<std::mutex> g(g_db_mu);
  auto it = g_db_live.find((ResidentDb *)h);
  if (!h || it == g_db_live.end()) throw std::runtime_error("database: the handle is NULL, closed, or was never opened");
  return *it;
}

static void db_register(ResidentDb *db) {
  std::lock_guard<std::mutex> g(g_db_mu);
  g_db_live.insert(db);
}

// Argument check of tracs_db_query_*. Host code only, so it runs before require_device().
static tracs_opts_t db_query_check(void *h, size_t nq, size_t pitch, const tracs_opts_t *opts, const tracs_edges_t *out, bool host_input,
                                   ResidentDb *&db, uint64_t &L) {
  const char *pre = "database query: ";
  if (!out) throw std::runtime_error(std::string(pre) + "out is NULL");
  tracs_opts_t o;
  if (opts) o = *opts; else { memset(&o, 0, sizeof o); o.dist = INT32_MAX; o.want_ncomp = 1; }
  if (o.filter) throw std::runtime_error(std::string(pre) + "opts->filter (recombination filter) is not supported against a database");
  if (o.keep_on_device) throw std::runtime_error(std::string(pre) + "opts->keep_on_device is not supported against a database");
  if (o.shard_world > 1) throw std::runtime_error(std::string(pre) + "opts->shard_world > 1: a database is swept on one GPU");
  if (o.i_end || o.j_start)
    throw std::runtime_error(std::string(pre) + "opts->i_end / opts->j_start must be 0: rows are the queries, cols the database");
  if (o.sweep_variant < 0 || o.sweep_variant > 2) throw std::runtime_error(std::string(pre) + "opts->sweep_variant must be 0, 1 or 2");
  if (nq >= (1ull << 31)) throw std::runtime_error(std::string(pre) + "nq: too many samples");
  db = db_lookup(h);
  tracs_db_info_t info;
  db_info(*db, info);
  L = info.L;
  check_pitch(pre, pitch, L, o.packed_input != 0, host_input, nq);
  o.shard_world = 1;
  o.shard_rank = 0;
  return o;
}

static void db_open_check(size_t n, size_t L, size_t pitch, const tracs_opts_t *opts, void **db, bool host_input) {
  const char *pre = "database open: ";
  if (!db) throw std::runtime_error(std::string(pre) + "db (the handle's address) is NULL");
  *db = nullptr;
  if (n == 0) throw std::runtime_error(std::string(pre) + "n must be at least 1");
  if (n >= (1ull << 31) - 1024) throw std::runtime_error(std::string(pre) + "n: too many samples");
  check_pitch(pre, pitch, L, opts && opts->packed_input, host_input, n);
}
}  // namespace tracs

extern "C" {

int tracs_db_open_host(const uint8_t *seqs, size_t n, size_t L, size_t pitch, const tracs_opts_t *opts, void **db) {
  memset(&g_stats, 0, sizeof g_stats);
  return guarded([&] {
    db_open_check(n, L, pitch, opts, db, true);
    require_device();
    InterruptScope sigint;
    DevBuf<uint8_t> nib;
    size_t pitch4 = 0;
    stream_host_to_packed(seqs, n, L, pitch, opts && opts->packed_input, nib, pitch4, 0);
    const uint8_t *rows = nib.p;
    ResidentDb *h = db_open(rows, n, L, pitch4, &nib, 0);
    db_register(h);
    *db = h;
  });
}

int tracs_db_open_device(const uint8_t *dev_seqs, size_t n, size_t L, size_t pitch, const tracs_opts_t *opts, void **db) {
  memset(&g_stats, 0, sizeof g_stats);
  return guarded([&] {
    db_open_check(n, L, pitch, opts, db, false);
    require_device();
    InterruptScope sigint;
    ResidentDb *h;
    if (opts && opts->packed_input) {
      h = db_open(dev_seqs, n, L, pitch, nullptr, 0);
    } else {  // ASCII rows are encoded once into 4-bit rows the handle owns (db.inl: one pack for both sides)
      DevBuf<uint8_t> nib;
      const size_t pitch4 = packed_pitch(L);
      nib.alloc(n * pitch4);
      encode_rows_device(dev_seqs, n, L, pitch, nib.p, pitch4, 0);
      const uint8_t *rows = nib.p;
      h = db_open(rows, n, L, pitch4, &nib, 0);
    }
    db_register(h);
    *db = h;
  });
}

int tracs_db_query_host(void *db, const uint8_t *seqs, size_t nq, size_t pitch, const tracs_opts_t *opts, tracs_edges_t *out) {
  if (out) memset(out, 0, sizeof *out);
  memset(&g_stats, 0, sizeof g_stats);
  return guarded([&] {
    ResidentDb *h = nullptr;
    uint64_t L = 0;
    tracs_opts_t o = db_query_check(db, nq, pitch, opts, out, true, h, L);
    require_device();
    InterruptScope sigint;
    HostEdges he;
    if (nq > 0) {
      DevBuf<uint8_t> nib;
      size_t pitch4 = 0;
      stream_host_to_packed(seqs, nq, L, pitch, o.packed_input != 0, nib, pitch4, 0);
      db_query(*h, nib.p, nq, pitch4, o, he, 0);
    }
    finish_edges(he, o, nq, L, out, 0);
  });
}

int tracs_db_query_device(void *db, const uint8_t *dev_seqs, size_t nq, size_t pitch, const tracs_opts_t *opts, tracs_edges_t *out) {
  if (out) memset(out, 0, sizeof *out);
  memset(&g_stats, 0, sizeof g_stats);
  return guarded([&] {
    ResidentDb *h = nullptr;
    uint64_t L = 0;
    tracs_opts_t o = db_query_check(db, nq, pitch, opts, out, false, h, L);
    require_device();
    InterruptScope sigint;
    HostEdges he;
    DevBuf<uint8_t> nib;
    size_t qpitch = pitch;
    if (!o.packed_input && nq > 0) {
      qpitch = packed_pitch(L);
      nib.alloc(nq * qpitch);
      encode_rows_device(dev_seqs, nq, L, pitch, nib.p, qpitch, 0);
    }
    db_query(*h, o.packed_input ? dev_seqs : nib.p, nq, qpitch, o, he, 0);
    finish_edges(he, o, nq, L, out, 0);
  });
}

int tracs_db_info(void *db, tracs_db_info_t *out) {
  return guarded([&] {
    if (!out) throw std::runtime_error("database info: out is NULL");
    db_info(*db_lookup(db), *out);
  });
}

int tracs_db_close(void *db) {
  return guarded([&] {
    ResidentDb *h = db_lookup(db);
    {
      std::lock_guard<std::mutex> g(g_db_mu);
      g_db_live.erase(h);
    }
    db_close(h);
  });
}

int tracs_write_distance_matrix(const char *path, const int32_t *m, size_t rows, size_t cols, size_t ld, const char *const *row_names,
                                const char *const *col_names, char sep) {
  return guarded([&] {
    if (sep != '\t' && sep != ',') throw std::runtime_error("write_distance_matrix: sep must be '\\t' or ','");
    if (ld < cols) throw std::runtime_error("write_distance_matrix: ld is smaller than the column count");
    if (!m && rows && cols) throw std::runtime_error("write_distance_matrix: m is NULL");
    if ((rows && !row_names) || (cols && !col_names)) throw std::runtime_error("write_distance_matrix: names are NULL");
    for (size_t r = 0; r < rows; ++r)
      if (!row_names[r]) throw std::runtime_error("write_distance_matrix: a row name is NULL");
    for (size_t c = 0; c < cols; ++c)
      if (!col_names[c]) throw std::runtime_error("write_distance_matrix: a column name is NULL");
    std::unique_ptr<FILE, int (*)(FILE *)> f(fopen(path, "wb"), fclose);
    if (!f) throw std::runtime_error(std::string("cannot open ") + path);
    std::string head;
    for (size_t c = 0; c < cols; ++c) {
      head += sep;
      head += col_names[c];
    }
    head += '\n';
    if (fwrite(head.data(), 1, head.size(), f.get()) != head.size()) throw std::runtime_error("write error");
    // rows are formatted by T threads, a batch of T consecutive row ranges at a time, and written in row order: the bytes
    // do not depend on T (TRACS_WRITE_THREADS, default: the hardware threads, at most 16)
    const char *env_t = getenv("TRACS_WRITE_THREADS");
    const unsigned hw = std::max(1u, std::thread::hardware_concurrency());
    const size_t T = env_t ? (size_t)std::max(1, atoi(env_t)) : (size_t)std::min(16u, hw);
    const size_t rows_per = std::max<size_t>(1, ((size_t)4 << 20) / (cols * 12 + 64));  // ~4 MB of text per range
    std::vector<std::string> bufs(T);
    for (size_t r0 = 0; r0 < rows; r0 += T * rows_per) {
      auto format = [&](size_t t) {
        std::string &b = bufs[t];
        b.clear();
        const size_t a = r0 + t * rows_per, e = std::min(rows, a + rows_per);
        char num[16];
        for (size_t r = a; r < e; ++r) {
          b += row_names[r];
          const int32_t *row = m + r * ld;
          for (size_t c = 0; c < cols; ++c) {
            b += sep;
            b.append(num, (size_t)(std::to_chars(num, num + sizeof num, row[c]).ptr - num));
          }
          b += '\n';
        }
      };
      const size_t used = std::min(T, (rows - r0 + rows_per - 1) / rows_per);
      std::vector<char> failed(used, 0);
      std::vector<std::thread> pool;
      for (size_t t = 1; t < used; ++t)
        pool.emplace_back([&, t] {
          try {
            format(t);
          } catch (...) {
            failed[t] = 1;
          }
        });
      format(0);
      for (auto &th : pool) th.join();
      for (char x : failed)
        if (x) throw std::bad_alloc();
      for (size_t t = 0; t < used; ++t)
        if (fwrite(bufs[t].data(), 1, bufs[t].size(), f.get()) != bufs[t].size()) throw std::runtime_error("write error");
    }
    if (fclose(f.release()) != 0) throw std::runtime_error("write error");
  });
}

int tracs_pairsnp(const char *const *paths, int n_paths, int n_threads, int32_t dist, int filter,
                  tracs_edges_t *out) {
  memset(out, 0, sizeof *out);
  memset(&g_stats, 0, sizeof g_stats);
  return guarded([&] {
    // src/pairsnp.hpp:340-343
    if (n_paths < 1 || n_paths > 2) throw std::runtime_error("Invalid number of fasta files!");
    require_device();
    InterruptScope sigint;
    // The reader hands completed rows to the device while it is still parsing (DeviceRowStreamer): host -> device
    // copies and the ASCII -> nibble encode overlap the parse; the pair sweep starts on the resident packed alignment
    // as soon as the last record is in. TRACS_FASTA_STREAM=0: parse everything first, then copy (tests compare).
    const char *env_stream = getenv("TRACS_FASTA_STREAM");
    const bool streaming = !(env_stream && !strcmp(env_stream, "0"));
    ByteBuf ascii;
    std::vector<std::string> names;
    uint64_t L = 0, L2 = 0;
    std::unique_ptr<DeviceRowStreamer> ds(streaming ? new DeviceRowStreamer(0) : nullptr);
    const uint64_t n1 = read_fasta(paths[0], n_threads, ascii, names, L, ds.get(), 0);
    uint64_t n = n1;
    tracs_opts_t o;
    memset(&o, 0, sizeof o);
    o.dist = dist; o.filter = filter; o.want_ncomp = 1; o.i_end = n1; o.j_start = 0;
    if (n_paths == 2) {
      L2 = L;
      // the reference does not cross-check the files (bitsets of unequal size: undefined); refuse (the streamer
      // raises the same error when the second file's rows have another length)
      const uint64_t n2 = read_fasta(paths[1], n_threads, ascii, names, L2, (n1 > 0 && L > 0) ? ds.get() : nullptr, n1);
      if (n2 > 0 && n1 > 0 && L2 != L) throw std::runtime_error("Error reading FASTA, variable sequence lengths!");
      if (n1 == 0) L = L2;
      n += n2;
      o.j_start = n1;
    }
    tracs_edges_t tmp;
    int rc = 0;
    if (n1 == 0 || o.j_start >= n) {
      memset(&tmp, 0, sizeof tmp);
      tmp.rows = (uint64_t *)calloc(1, 8); tmp.cols = (uint64_t *)calloc(1, 8); tmp.dist = (uint64_t *)calloc(1, 8);
      tmp.filt = nullptr; tmp.ncomp = (uint64_t *)calloc(1, 8);
      tmp.seq_length = L;
    } else if (ds && L > 0 && ds->n_rows == n) {
      ds->finish();
      memset(&tmp, 0, sizeof tmp);
      tracs_opts_t on = normalise(&o, n);
      on.packed_input = 1;
      HostEdges he;
      sweep_device(ds->nib.p, n, L, ds->pitch4, on, he, 0);
      finish_edges(he, on, n, L, &tmp, 0);
    } else {
      ds.reset();
      rc = tracs_pairsnp_host(ascii.data(), n, L, L, &o, &tmp);
    }
    if (rc) throw std::runtime_error(g_err);
    *out = tmp;
    out->n_names = names.size();
    out->names = (char **)malloc(std::max<size_t>(1, names.size()) * sizeof(char *));
    for (size_t i = 0; i < names.size(); ++i) out->names[i] = strdup(names[i].c_str());
  });
}

int tracs_read_fasta(const char *path, int n_threads, uint8_t **seqs, size_t *n, size_t *L, char ***names) {
  *seqs = nullptr; *names = nullptr; *n = 0; *L = 0;
  return guarded([&] {
    ByteBuf ascii;
    std::vector<std::string> nm;
    uint64_t len = 0;
    // TRACS_FASTA_SINK_CHECK=1 (tests): read with a collecting RowSink as well and insist that the rows it was fed while
    // the reader was parsing are exactly the rows of the finished matrix, in order
    struct CollectSink : RowSink {
      std::vector<uint8_t> buf;
      uint64_t L = 0, n = 0;
      bool bad = false;
      void expect(uint64_t, uint64_t) override {}
      void rows(const uint8_t *p, uint64_t first, uint64_t count, uint64_t Lr) override {
        if (L == 0) L = Lr;
        if (Lr != L || first != n) bad = true;
        buf.insert(buf.end(), p, p + count * Lr);
        n += count;
      }
      void reset() override { buf.clear(); n = 0; L = 0; }
    } sink;
    const char *chk = getenv("TRACS_FASTA_SINK_CHECK");
    const bool check = chk && !strcmp(chk, "1");
    const uint64_t cnt = read_fasta(path, n_threads, ascii, nm, len, check ? &sink : nullptr, 0);
    if (check && cnt > 0 && len > 0 &&
        (sink.bad || sink.n != cnt || sink.L != len || sink.buf.size() != ascii.size() || memcmp(sink.buf.data(), ascii.data(), ascii.size()) != 0))
      throw std::runtime_error("internal error: rows streamed by the reader differ from the parsed matrix");
    *seqs = ascii.release();
    *names = (char **)malloc(std::max<size_t>(1, nm.size()) * sizeof(char *));
    for (size_t i = 0; i < nm.size(); ++i) (*names)[i] = strdup(nm[i].c_str());
    *n = cnt;
    *L = len;
  });
}

void tracs_free_fasta(uint8_t *seqs, char **names, size_t n) {
  free(seqs);
  if (names) {
    for (size_t i = 0; i < n; ++i) free(names[i]);
    free(names);
  }
}

int tracs_shard_rowblocks(uint32_t n_rowblocks, int32_t world, int32_t rank, uint32_t *out, uint32_t *n_out) {
  return guarded([&] {
    if (world < 1 || rank < 0 || rank >= world) throw std::runtime_error("shard_rank >= shard_world");
    uint32_t k = 0;
    for (uint32_t rb = 0; rb < n_rowblocks; ++rb)
      if (shard_owner(rb, world) == rank) out[k++] = rb;
    *n_out = k;
  });
}

int tracs_trans_dist(const int32_t *snpdiff, const double *datediff, size_t n, double lamb, double beta,
                     double threshold_Ek, double *p0_log, double *eK) {
  return guarded([&] {
    require_device();
    trans_dist_device(snpdiff, datediff, n, lamb, beta, threshold_Ek, p0_log, eK, 0);
  });
}

// src/transcluster.hpp:62-75 (host copy for the scalar, test-only entry point)
static double lae_host(double x, double y) {
  const double t = x - y;
  if (x == y) return x + M_LN2;
  if (t > 0) return x + log1p(exp(-t));
  else if (t <= 0) return y + log1p(exp(t));
  return t;
}

int tracs_lprob_k_given_N(size_t N, size_t k, double delta, double lamb, double beta, const double *lg,
                          size_t n_lg, double out[2]) {
  return guarded([&] {
    if (n_lg < N + k + 2) throw std::out_of_range("lgamma table shorter than N + k + 2");
    // src/transcluster.hpp:90-129. The binomial-coefficient terms lg[i+1] cancel inside the
    // integral sum; they are kept out here and the remaining factor lg[N+k+1]-lg[N+1] hoisted.
    double lprob, lhs;
    const double M = (double)(N + k);
    if (delta > 0) {
      lprob = (double)(N + 1) * log(lamb) - delta * (lamb + beta) + (double)k * log(beta) - lg[k + 1];
      double pois = -INFINITY;
      const double lld = log(lamb * delta);
      for (size_t i = 0; i <= N; ++i) pois = lae_host((double)i * lld - lg[i + 1], pois);
      pois -= lamb * delta;
      lprob -= pois;
      double integ = -INFINITY;
      const double ld = log(delta), llb = log(lamb + beta);
      for (size_t i = 0; i <= N + k; ++i)
        integ = lae_host(lg[N + k + 1] - lg[N + k - i + 1] + (M - (double)i) * ld - (double)(i + 1) * llb, integ);
      integ -= lg[N + 1];
      lhs = lprob;
      lprob += integ;
    } else {
      lprob = (double)(N + 1) * log(lamb) + (double)k * log(beta) + lg[N + k + 1] - lg[N + 1] - lg[k + 1] -
              (M + 1.0) * log(lamb + beta);
      lhs = lprob;
    }
    out[0] = lprob;
    out[1] = lhs;
  });
}

// src/dmultinomial.hpp:8-86 -- align-stage helper kept for import compatibility (host arithmetic).
int tracs_calculate_posteriors(const double *counts, size_t rows, size_t cols, const double *alphas_in,
                               size_t n_alpha, int keep, double threshold, double *out) {
  return guarded([&] {
    if (n_alpha == 0) throw std::runtime_error("alphas must not be empty");
    if (n_alpha < cols) throw std::out_of_range("need at least one alpha per column");
    std::vector<double> alphas(alphas_in, alphas_in + n_alpha);
    std::sort(alphas.begin(), alphas.end(), std::greater<double>());
    const double a0 = std::accumulate(alphas.begin(), alphas.end(), 0.0);
    const double a_min = alphas[0] / a0;
    std::vector<size_t> order(cols);
    for (size_t r = 0; r < rows; ++r) {
      const double *row = counts + r * cols;
      double *res = out + r * cols;
      double total = 0;
      for (size_t c = 0; c < cols; ++c) total += row[c];
      std::iota(order.begin(), order.end(), 0);
      std::stable_sort(order.begin(), order.end(), [&](size_t x, size_t y) { return row[x] > row[y]; });
      if (total <= 0) {
        for (size_t c = 0; c < cols; ++c) res[c] = a_min;
      } else {
        // ties share one alpha: the rank only advances when the sorted count changes
        size_t rank = 0;
        for (size_t c = 0; c < cols; ++c) {
          const size_t id = order[c];
          res[id] = (row[id] + alphas[rank]) / (total + a0);
          if (c + 1 < cols && row[id] != row[order[c + 1]]) rank++;
        }
      }
      for (size_t c = 0; c < cols; ++c)
        if (res[c] <= threshold) res[c] = (keep && row[c] > 0) ? threshold : 0.0;
    }
  });
}

int tracs_min_over_refs(const uint64_t *a, const uint64_t *b, const double *val, size_t n, uint64_t *out_a,
                        uint64_t *out_b, double *out_val, size_t *n_out) {
  return guarded([&] {
    require_device();
    *n_out = 0;
    if (n == 0) return;
    std::vector<uint64_t> keys(n);
    for (size_t i = 0; i < n; ++i) {
      const uint64_t lo = std::min(a[i], b[i]), hi = std::max(a[i], b[i]);
      if (hi >= (1ull << 32)) throw std::runtime_error("sample id out of range");
      keys[i] = (lo << 32) | hi;
    }
    DevBuf<uint64_t> k1(n), k2(n), ku(n);
    DevBuf<double> v1(n), v2(n), vu(n);
    DevBuf<uint64_t> d_runs(1);
    TRACS_CK(cudaMemcpy(k1.p, keys.data(), n * 8, cudaMemcpyHostToDevice));
    TRACS_CK(cudaMemcpy(v1.p, val, n * 8, cudaMemcpyHostToDevice));
    size_t tb = 0, tb2 = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, tb, k1.p, k2.p, v1.p, v2.p, (int64_t)n);
    cub::DeviceReduce::ReduceByKey(nullptr, tb2, k2.p, ku.p, v2.p, vu.p, d_runs.p, cub::Min(), (int64_t)n);
    DevBuf<uint8_t> tmp(std::max(tb, tb2));
    cub::DeviceRadixSort::SortPairs(tmp.p, tb, k1.p, k2.p, v1.p, v2.p, (int64_t)n);
    cub::DeviceReduce::ReduceByKey(tmp.p, tb2, k2.p, ku.p, v2.p, vu.p, d_runs.p, cub::Min(), (int64_t)n);
    uint64_t runs = 0;
    TRACS_CK(cudaMemcpy(&runs, d_runs.p, 8, cudaMemcpyDeviceToHost));
    std::vector<uint64_t> hk(runs);
    TRACS_CK(cudaMemcpy(hk.data(), ku.p, runs * 8, cudaMemcpyDeviceToHost));
    TRACS_CK(cudaMemcpy(out_val, vu.p, runs * 8, cudaMemcpyDeviceToHost));
    for (size_t i = 0; i < runs; ++i) {
      out_a[i] = hk[i] >> 32;
      out_b[i] = hk[i] & 0xFFFFFFFFull;
    }
    *n_out = runs;
  });
}

// ---- single-linkage clusters = connected components (tracs/cluster.py:104-129) -------------------------
namespace tracs {
__device__ __forceinline__ uint32_t cc_find(uint32_t *parent, uint32_t v) {
  // path halving
  uint32_t p = parent[v];
  while (p != v) {
    const uint32_t gp = parent[p];
    if (gp != p) parent[v] = gp;
    v = p;
    p = gp;
  }
  return v;
}
__global__ void k_cc_init(uint32_t *parent, uint32_t n) {
  const uint32_t v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v < n) parent[v] = v;
}
// hook the larger root under the smaller one: the root of a finished component is its smallest node
__global__ void k_cc_hook(const uint64_t *__restrict__ a, const uint64_t *__restrict__ b, uint64_t E, uint32_t *parent) {
  const uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= E) return;
  uint32_t ru = cc_find(parent, (uint32_t)a[e]), rv = cc_find(parent, (uint32_t)b[e]);
  while (ru != rv) {
    const uint32_t hi = max(ru, rv), lo = min(ru, rv);
    const uint32_t old = atomicCAS(parent + hi, hi, lo);
    if (old == hi) break;          // hooked
    ru = cc_find(parent, old);     // somebody else hooked hi first: continue from its new root
    rv = lo;
    rv = cc_find(parent, rv);
  }
}
__global__ void k_cc_flatten(uint32_t *parent, uint32_t n, uint8_t *is_root) {
  const uint32_t v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= n) return;
  uint32_t r = v;
  while (parent[r] != r) r = parent[r];
  parent[v] = r;
  is_root[v] = (r == v);
}
__global__ void k_cc_label(const uint32_t *__restrict__ parent, const uint32_t *__restrict__ root_rank, uint32_t n,
                           uint32_t *__restrict__ labels) {
  const uint32_t v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v < n) labels[v] = root_rank[parent[v]];
}
}  // namespace tracs

int tracs_connected_components(const uint64_t *a, const uint64_t *b, size_t n_edges, size_t n_nodes, uint32_t *labels,
                               size_t *n_components) {
  return guarded([&] {
    require_device();
    *n_components = 0;
    if (n_nodes == 0) return;
    if (n_nodes >= (1ull << 32)) throw std::runtime_error("too many nodes");
    for (size_t e = 0; e < n_edges; ++e)
      if (a[e] >= n_nodes || b[e] >= n_nodes) throw std::out_of_range("edge endpoint out of range");
    const uint32_t n = (uint32_t)n_nodes;
    DevBuf<uint32_t> parent(n), rank(n), lab(n);
    DevBuf<uint8_t> is_root(n);
    DevBuf<uint64_t> da(std::max<size_t>(1, n_edges)), db(std::max<size_t>(1, n_edges));
    if (n_edges) {
      TRACS_CK(cudaMemcpy(da.p, a, n_edges * 8, cudaMemcpyHostToDevice));
      TRACS_CK(cudaMemcpy(db.p, b, n_edges * 8, cudaMemcpyHostToDevice));
    }
    k_cc_init<<<(n + 255) / 256, 256>>>(parent.p, n);
    if (n_edges) k_cc_hook<<<(unsigned)((n_edges + 255) / 256), 256>>>(da.p, db.p, n_edges, parent.p);
    k_cc_flatten<<<(n + 255) / 256, 256>>>(parent.p, n, is_root.p);
    // label of a component = rank of its root (= its smallest node) among all roots: the numbering
    // scipy.sparse.csgraph.connected_components produces (components discovered from node 0 upwards)
    size_t tb = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, tb, is_root.p, rank.p, (int64_t)n);
    DevBuf<uint8_t> tmp(tb);
    cub::DeviceScan::ExclusiveSum(tmp.p, tb, is_root.p, rank.p, (int64_t)n);
    k_cc_label<<<(n + 255) / 256, 256>>>(parent.p, rank.p, n, lab.p);
    TRACS_CK(cudaGetLastError());
    TRACS_CK(cudaMemcpy(labels, lab.p, (size_t)n * 4, cudaMemcpyDeviceToHost));
    uint32_t last_rank = 0;
    uint8_t last_root = 0;
    TRACS_CK(cudaMemcpy(&last_rank, rank.p + (n - 1), 4, cudaMemcpyDeviceToHost));
    TRACS_CK(cudaMemcpy(&last_root, is_root.p + (n - 1), 1, cudaMemcpyDeviceToHost));
    *n_components = (size_t)last_rank + last_root;
  });
}

// ---- native CSV writer for the distance stage (tracs/distance.py:206-258) --------------------------------
namespace tracs {
// Python's repr(float): shortest digits that round-trip; fixed notation while -4 < decpt <= 16, else d.ddde+XX
static size_t py_float_repr(double v, char *out) {
  if (std::isnan(v)) { memcpy(out, "nan", 3); return 3; }
  if (std::isinf(v)) { const char *t = v < 0 ? "-inf" : "inf"; size_t n = strlen(t); memcpy(out, t, n); return n; }
  char tmp[64];
  auto r = std::to_chars(tmp, tmp + sizeof tmp, v, std::chars_format::scientific);
  *r.ptr = 0;
  char *o = out;
  const char *p = tmp;
  if (*p == '-') *o++ = *p++;
  char digits[32];
  int nd = 0;
  for (; *p && *p != 'e'; ++p)
    if (*p != '.') digits[nd++] = *p;
  const int decpt = atoi(p + 1) + 1;
  while (nd > 1 && digits[nd - 1] == '0') --nd;  // to_chars is already shortest; be safe
  if (decpt > 16 || decpt < -3) {
    *o++ = digits[0];
    if (nd > 1) { *o++ = '.'; memcpy(o, digits + 1, nd - 1); o += nd - 1; }
    const int e = decpt - 1;
    o += sprintf(o, "e%c%02d", e < 0 ? '-' : '+', e < 0 ? -e : e);
  } else if (decpt <= 0) {
    *o++ = '0'; *o++ = '.';
    for (int k = 0; k < -decpt; ++k) *o++ = '0';
    memcpy(o, digits, nd); o += nd;
  } else if (decpt >= nd) {
    memcpy(o, digits, nd); o += nd;
    for (int k = nd; k < decpt; ++k) *o++ = '0';
    *o++ = '.'; *o++ = '0';
  } else {
    memcpy(o, digits, decpt); o += decpt;
    *o++ = '.';
    memcpy(o, digits + decpt, nd - decpt); o += nd - decpt;
  }
  return (size_t)(o - out);
}
}  // namespace tracs

size_t tracs_float_repr(double v, char *buf) {
  const size_t n = tracs::py_float_repr(v, buf);
  buf[n] = 0;
  return n;
}

int tracs_write_distance_csv(const char *path, int append, const tracs_edges_t *e, const char *const *names, size_t n_names,
                             const char *msa_label, int has_trans, int filter_on, int use_k_threshold, double k_threshold,
                             size_t *rows_written) {
  return guarded([&] {
    if (rows_written) *rows_written = 0;
    FILE *f = fopen(path, append ? "ab" : "wb");
    if (!f) throw std::runtime_error(std::string("cannot open ") + path);
    static const char HEADER[] =
        "sampleA,sampleB,date difference,SNP distance,transmission distance,expected K,filtered SNP distance,sites considered,MSA file\n";
    std::string buf;
    buf.reserve(1 << 22);
    if (!append) buf += HEADER;
    char num[96];
    size_t written = 0;
    const bool trans = has_trans && e->p0_log && e->eK && e->datediff;
    for (size_t k = 0; k < e->n_edges; ++k) {
      if (trans && use_k_threshold && !(k_threshold >= e->eK[k])) continue;  // tracs/distance.py:222
      if (e->rows[k] >= n_names || e->cols[k] >= n_names) throw std::out_of_range("edge index beyond the name list");
      buf += names[e->rows[k]]; buf += ',';
      buf += names[e->cols[k]]; buf += ',';
      if (trans) { buf.append(num, tracs::py_float_repr(e->datediff[k], num)); } else buf += "NA";
      buf += ',';
      buf.append(num, (size_t)sprintf(num, "%llu", (unsigned long long)e->dist[k])); buf += ',';
      if (trans) { buf.append(num, tracs::py_float_repr(exp(e->p0_log[k]), num)); } else buf += "NA";
      buf += ',';
      if (trans) { buf.append(num, tracs::py_float_repr(e->eK[k], num)); } else buf += "NA";
      buf += ',';
      // with metadata and no filter the reference writes NA, otherwise the number (zeros when the filter is off)
      if (trans && !filter_on) buf += "NA";
      else buf.append(num, (size_t)sprintf(num, "%llu", (unsigned long long)(e->filt ? e->filt[k] : 0ull)));
      buf += ',';
      buf.append(num, (size_t)sprintf(num, "%llu", (unsigned long long)e->ncomp[k])); buf += ',';
      buf += msa_label;
      buf += '\n';
      ++written;
      if (buf.size() > (1u << 22) - 4096) { fwrite(buf.data(), 1, buf.size(), f); buf.clear(); }
    }
    fwrite(buf.data(), 1, buf.size(), f);
    if (fclose(f) != 0) throw std::runtime_error("write error");
    if (rows_written) *rows_written = written;
  });
}

int tracs_synth_device(const tracs_synth_t *cfg, uint8_t *dev_seqs, int32_t *dev_days) {
  return guarded([&] {
    require_device();
    if (!cfg->packed && (cfg->pitch % 16 != 0 || cfg->pitch < cfg->L)) throw std::runtime_error("synth: pitch must be a multiple of 16 and >= L");
    if (cfg->packed && (cfg->pitch % 16 != 0 || cfg->pitch * 2 < cfg->L)) throw std::runtime_error("synth: packed pitch must be a multiple of 16 bytes and hold L sites");
    SynthDev c;
    c.packed = cfg->packed ? 1u : 0u;
    c.n = cfg->n; c.L = cfg->L; c.pitch = cfg->pitch; c.seed = cfg->seed;
    auto clamp01 = [](double x) { return x < 0 ? 0.0 : (x > 1 ? 1.0 : x); };
    c.thr_var24 = (uint32_t)(clamp01(cfg->p_var) * 16777216.0);
    c.thr_found16 = (uint32_t)(0.3 * 65536.0);
    c.thr_gc16 = (uint32_t)(clamp01(cfg->gc) * 65536.0);
    c.n_clusters = std::max(1u, cfg->n_clusters);
    c.site_offset = cfg->site_offset;
    c.L_total = cfg->L_total ? cfg->L_total : cfg->L;
    if (c.site_offset + c.L > c.L_total) throw std::runtime_error("synth: slab exceeds L_total");
    const double v = std::max(1.0, cfg->p_var * (double)c.L_total);
    c.thr_priv32 = (uint32_t)std::min(4294967295.0, clamp01(cfg->mu / v) * 4294967296.0);
    c.thr_N32 = (uint32_t)std::min(4294967295.0, clamp01(cfg->p_N) * 4294967296.0);
    c.thr_amb16 = (uint32_t)(clamp01(cfg->p_amb) * 65536.0);
    c.n_days = cfg->n_days; c.gaps = cfg->gaps;
    c.gap_len = c.L_total / 1000;
    const uint64_t total = c.n * ((c.packed ? c.pitch * 2 : c.pitch) / 16);
    if (total) {
      k_synth<<<(unsigned)((total + 255) / 256), 256>>>(c, dev_seqs);
      TRACS_CK(cudaGetLastError());
    }
    if (dev_days && c.n) k_synth_days<<<(unsigned)((c.n + 255) / 256), 256>>>(c.n, c.seed, c.n_days, dev_days);
    TRACS_CK(cudaDeviceSynchronize());
  });
}

int tracs_trim(void) {
  return guarded([&] {
    TRACS_CK(cudaDeviceSynchronize());
    {
      DevCache &dc = dev_cache();
      std::lock_guard<std::mutex> g(dc.mu);
      for (auto &kv : dc.idle) cudaFree(kv.second.first);
      dc.idle.clear();
    }
    HostPool &hp = host_pool();
    std::lock_guard<std::mutex> g(hp.mu);
    for (auto &kv : hp.idle)
      for (void *p : kv.second) cudaFreeHost(p);
    hp.idle.clear();
    hp.cached_bytes = 0;
  });
}

int tracs_dev_alloc(void **p, size_t bytes) {
  return guarded([&] { require_device(); TRACS_CK(cudaMalloc(p, bytes)); });
}
int tracs_dev_free(void *p) {
  return guarded([&] { TRACS_CK(cudaFree(p)); });
}
int tracs_host_alloc_pinned(void **p, size_t bytes) {
  return guarded([&] { require_device(); TRACS_CK(cudaMallocHost(p, bytes)); });
}
int tracs_host_free_pinned(void *p) {
  return guarded([&] { TRACS_CK(cudaFreeHost(p)); });
}
int tracs_host_register(void *p, size_t bytes) {
  return guarded([&] { require_device(); TRACS_CK(cudaHostRegister(p, bytes, cudaHostRegisterPortable)); });
}
int tracs_host_unregister(void *p) {
  return guarded([&] { TRACS_CK(cudaHostUnregister(p)); });
}
int tracs_memcpy_d2h(void *dst, const void *src, size_t bytes) {
  return guarded([&] { TRACS_CK(cudaMemcpy(dst, src, bytes, cudaMemcpyDeviceToHost)); });
}
int tracs_memcpy_h2d(void *dst, const void *src, size_t bytes) {
  return guarded([&] { TRACS_CK(cudaMemcpy(dst, src, bytes, cudaMemcpyHostToDevice)); });
}

int tracs_int_peak(double out[8]) {
  return guarded([&] {
    require_device();
    int dev = 0, n_sm = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev);
    const int blocks = n_sm * 4, threads = 256, iters = 4096;
    DevBuf<uint32_t> sink((size_t)blocks * threads);
    DevBuf<long long> cyc(1);
    Timer T(0);
    auto run = [&](int mode) -> double {
      float best = 1e30f;
      for (int rep = 0; rep < 4; ++rep) {
        T.start();
        switch (mode) {
          case 0: k_peak<0><<<blocks, threads>>>(sink.p, iters, cyc.p); break;
          case 1: k_peak<1><<<blocks, threads>>>(sink.p, iters, cyc.p); break;
          case 2: k_peak<2><<<blocks, threads>>>(sink.p, iters, cyc.p); break;
          case 3: k_peak<3><<<blocks, threads>>>(sink.p, iters, cyc.p); break;
          default: k_peak<4><<<blocks, threads>>>(sink.p, iters, cyc.p); break;
        }
        float ms = T.stop();
        TRACS_CK(cudaGetLastError());
        if (rep > 0 && ms < best) best = ms;
      }
      return (double)best * 1e-3;
    };
    const double lanes = (double)blocks * threads * iters;
    out[0] = lanes * 64 / run(0);  // LOP3 lane-ops / s
    out[1] = lanes * 64 / run(1);  // POPC
    out[2] = lanes * 64 / run(2);  // IADD
    out[3] = lanes * 32 / run(3);  // word-pairs / s, add on the ALU pipe
    out[4] = lanes * 32 / run(4);  // word-pairs / s, add as IMAD (FMA pipe)
    out[5] = (double)n_sm;
    out[6] = 0;
    out[7] = 0;
  });
}

}  // extern "C"
