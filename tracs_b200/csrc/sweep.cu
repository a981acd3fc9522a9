// Pair sweep for sm_100a: ASCII alignment (device) -> sparse edge list.
//
//   K0a k_pack      ASCII -> per-site AND of the 4-bit base masks over all samples (column mask),
//                   full-length N bit-plane + its block summary        [HBM-bound, reads n*L bytes]
//   K0b k_gather    variable sites only -> interleaved A/C/G/T bit-planes P[word][sample] (uint4)
//   K1  k_sweep     128x128 pair tiles, bulk-async (TMA engine, UBLKCP) staged panels, 8x8 register
//                   micro-tiles, LOP3 + POPC, fused threshold + edge append  [INT-pipe bound]
//                   (k_sweep<true>: every distance stored into a dense matrix instead, distance_matrix_device)
//   K2  k_ncomp     compared-site count for emitted edges via block-sparse N-plane intersection
//
// Semantics restated from the reference (paths relative to gtonkinhill/tracs):
//   base masks       src/pairsnp.hpp:107-199      d(i,j)   src/pairsnp.hpp:398-403
//   threshold/emit   src/pairsnp.hpp:405-410      nn(i,j)  src/pairsnp.hpp:417-419
//   pair range       src/pairsnp.hpp:352-360,395  order    src/pairsnp.hpp:450-457
// Dropping a site whose column AND is non-zero (some base shared by every sample) changes no
// d(i,j): such a site is a match for every pair (SURVEY A.4).
#include <cub/cub.cuh>

#include <algorithm>
#include <memory>
#include <stdexcept>
#include <type_traits>

#include "common.cuh"
#include "trans.cuh"

namespace tracs {

static inline uint64_t round_up(uint64_t x, uint64_t m) { return (x + m - 1) / m * m; }

// ------------------------------------------------------------------------------------------
// K0a: pack
//   thread <-> one 32-site word (32 ASCII bytes) ; loops over a chunk of samples.
//   No memory table: PRMT is used as an 8-entry byte table, four lookups per instruction. The index
//   is the low 3 bits of the base, which tell the plain alphabet apart:
//       A 001  C 011  G 111  T 100  N 110  - 101        (upper or lower case, bit 5 is ignored)
//   One table returns the 4-bit mask (+ an is-N flag), a second one the byte the index stands for;
//   a byte that differs from it (IUPAC 2-/3-base codes, anything else) is repaired from the exact
//   256-entry table on a rare branch, so the result is exact for every input byte.
//   Two adjacent words of one sample (8 sites) share one selector register: nibble 2k = word 0
//   byte k, nibble 2k+1 = word 1 byte k, so every lookup result holds sites (0, 4, 1, 5) or
//   (2, 6, 3, 7) of the 8-site group. The N-plane word is stored in that fixed site permutation:
//   its only consumers are population counts of ANDs (k_ncomp, k_block_n, k_pairs_sparse).
// ------------------------------------------------------------------------------------------
constexpr int PACK_THREADS = 256;
constexpr int PACK_SCHUNK = 256;
constexpr int PACK_BATCH = 4;

// bit-select: (a & m) | (b & ~m)  -> one LOP3
__device__ __forceinline__ uint32_t bsel(uint32_t a, uint32_t b, uint32_t m) { return (a & m) | (b & ~m); }

// bit i of result = nibble i of x is 0xF
__device__ __forceinline__ uint32_t nibbles_all_ones(uint32_t x) {
  uint32_t t = x & (x >> 1);
  t &= (t >> 2);
  t &= 0x11111111u;
  t = (t | (t >> 3)) & 0x03030303u;
  t = (t | (t >> 6)) & 0x000F000Fu;
  t = (t | (t >> 12)) & 0xFFu;
  return t;
}

// mask table indexed by (byte & 7); F = 1111 + the is-N flag in bit 4 + V
//   000 F   001 A=1   010 F   011 C=2   100 T=8   101 F   110 F   111 G=4
template <int V> struct PackTab {
  static constexpr uint32_t F = 0x0Fu | (0x10u << V);
  static constexpr uint32_t LO = F | (0x01u << 8) | (F << 16) | (0x02u << 24);
  static constexpr uint32_t HI = 0x08u | (F << 8) | (F << 16) | (0x04u << 24);
};
// the byte each index stands for; 000 and 010 stand for nothing (entry with other low bits)
constexpr uint32_t PACK_E_LO = 0x01u | (0x41u << 8) | (0x01u << 16) | (0x43u << 24);
constexpr uint32_t PACK_E_HI = 0x54u | (0x2Du << 8) | (0x4Eu << 16) | (0x47u << 24);

// rare path: bytes flagged in d (non-zero byte) get their exact mask from the 256-entry table
__device__ __noinline__ uint32_t pack_repair(uint32_t o, uint32_t d, uint32_t m, uint32_t flag, const uint8_t *slut) {
#pragma unroll 1
  for (int p = 0; p < 32; p += 8) {
    if ((d >> p) & 0xFFu) {
      const uint32_t bm = slut[(o >> p) & 0xFFu];
      const uint32_t nb = bm | (bm == 15u ? flag : 0u);
      m = (m & ~(0xFFu << p)) | (nb << p);
    }
  }
  return m;
}

// PRMT with a run-time selector (only selector bits 0-15 are read; bit 3 of every nibble must be 0)
__device__ __forceinline__ uint32_t tab8(uint32_t lo, uint32_t hi, uint32_t sel) {
  uint32_t r;
  asm("prmt.b32 %0, %1, %2, %3;" : "=r"(r) : "r"(lo), "r"(hi), "r"(sel));
  return r;
}

// eight sites (two words of one sample) -> two registers of per-site mask bytes
template <int V0, int V1>
__device__ __forceinline__ void pack_unit(uint32_t w1, uint32_t w2, const uint8_t *slut, uint32_t &m1, uint32_t &m2) {
  const uint32_t z = (w1 & 0x07070707u) | ((w2 << 4) & 0x70707070u);
  const uint32_t zh = z >> 16;
  m1 = tab8(PackTab<V0>::LO, PackTab<V0>::HI, z);
  m2 = tab8(PackTab<V1>::LO, PackTab<V1>::HI, zh);
  const uint32_t e1 = tab8(PACK_E_LO, PACK_E_HI, z), e2 = tab8(PACK_E_LO, PACK_E_HI, zh);
  const uint32_t o1 = __byte_perm(w1, w2, 0x5140), o2 = __byte_perm(w1, w2, 0x7362);
  const uint32_t d1 = (o1 ^ e1) & 0xDFDFDFDFu, d2 = (o2 ^ e2) & 0xDFDFDFDFu;
  if (__builtin_expect((d1 | d2) != 0u, 0)) {
    m1 = pack_repair(o1, d1, m1, 0x10u << V0, slut);
    m2 = pack_repair(o2, d2, m2, 0x10u << V1, slut);
  }
}

// N-plane bit of site t (0..31) of a word: see pack_unit / one_sample
__device__ __forceinline__ uint32_t pack_nbit(uint32_t t) {
  const uint32_t k = t >> 2, b = t & 3u, j = k >> 1;
  const uint32_t q = 2u * j + (b >> 1), pos = 2u * (b & 1u) + (k & 1u);
  return 8u * pos + 4u * (q >> 2) + (q & 3u);
}

// is-N word of one sample's 32 sites -> N-plane, per-sample N count (shared-memory counter) and block summary.
// The summary byte is only computed and stored when the warp saw an N at all (the buffer is pre-zeroed).
// SPARSE_N: the word is stored only when its 256-site group (8 lanes = one 32-byte sector of the row) holds an N. The
// plane is only ever read where the block summaries say so (k_block_n, k_pairs_sparse, k_ncomp), so the rest of the
// buffer may keep whatever it held: at p_N = 1e-3 three quarters of the plane's sectors are never written.
template <bool SPARSE_N = false>
__device__ __forceinline__ void pack_emit_n(uint32_t isn, uint32_t *np, uint8_t *sp, uint32_t *cnt, uint32_t lane) {
  const uint32_t nz = __ballot_sync(0xFFFFFFFFu, isn != 0);
  if (!SPARSE_N || ((nz >> (lane & 24u)) & 0xFFu)) __stcs(np, isn);
  if (nz) {
    // (two thirds of all (warp, sample) visits at p_N = 1e-3 come here, and this kernel is bound by instruction issue:
    // the few lanes that hold an N add their counts themselves -- no warp reduction --, and the summary byte (one bit
    // per 4 words = 128 sites, one byte per warp = 1024 sites) is a ballot over lanes 0..7 looking at one nibble of nz each)
    if (isn) atomicAdd(cnt, (uint32_t)__popc(isn));
    const uint32_t sbyte = __ballot_sync(0xFFFFFFFFu, lane < 8u && ((nz >> (4u * lane)) & 0xFu) != 0u);
    if (lane == 0) *sp = (uint8_t)sbyte;
  }
}

// One sample's 32 sites: lookups, column AND, is-N word, N count and block summary. Lanes past the
// end of the alignment carry 'N' bytes and validp == 0, so every lane of a warp runs the same code.
template <bool SPARSE_N = false>
__device__ __forceinline__ void pack_one_sample(const uint4 &a, const uint4 &b, uint32_t *np, uint8_t *sp, uint32_t *cnt,
                                                const uint8_t *slut, uint32_t (&acc)[8], uint32_t validp, uint32_t lane) {
  uint32_t m0, m1, m2, m3, m4, m5, m6, m7;
  pack_unit<0, 1>(a.x, a.y, slut, m0, m1);
  pack_unit<2, 3>(a.z, a.w, slut, m2, m3);
  pack_unit<0, 1>(b.x, b.y, slut, m4, m5);
  pack_unit<2, 3>(b.z, b.w, slut, m6, m7);
  acc[0] &= m0; acc[1] &= m1; acc[2] &= m2; acc[3] &= m3;
  acc[4] &= m4; acc[5] &= m5; acc[6] &= m6; acc[7] &= m7;
  // the four flag positions of a half are disjoint: OR them, then interleave the two halves
  const uint32_t f0 = m0 | m1 | m2 | m3, f1 = m4 | m5 | m6 | m7;
  const uint32_t isn = bsel(f1, f0 >> 4, 0xF0F0F0F0u) & validp;
  pack_emit_n<SPARSE_N>(isn, np, sp, cnt, lane);
}

// `rows` consecutive samples of one 32-site word. Running pointers (no 64-bit index arithmetic per sample);
// PACK_BATCH samples per trip: all global loads of the batch are issued before any lookup, so every thread
// keeps 2 * PACK_BATCH 16-byte loads in flight (evict-first: a single pass over the bytes).
__device__ __forceinline__ void pack_rows(const uint8_t *src, uint64_t pitch, uint32_t rows, bool has_sites, uint32_t *np,
                                          uint64_t npitch, uint8_t *sp, uint64_t spitch, uint32_t *cnt, const uint8_t *slut,
                                          uint32_t (&acc)[8], uint32_t validp, uint32_t lane) {
  auto load = [](const uint4 *p) { return __ldcs(p); };
  uint32_t r = 0;
  for (; r + PACK_BATCH <= rows; r += PACK_BATCH) {
    uint4 va[PACK_BATCH], vb[PACK_BATCH];
#pragma unroll
    for (int t = 0; t < PACK_BATCH; ++t) {
      // lanes past the end of the alignment read the start of the row instead: whatever they see is masked out
      // (validp == 0, no column word), so the loads need no per-lane predicate
      va[t] = load(reinterpret_cast<const uint4 *>(src + (size_t)t * pitch));
      vb[t] = load(reinterpret_cast<const uint4 *>(src + (size_t)t * pitch) + 1);
    }
    if (r + 2 * PACK_BATCH <= rows) {  // the next batch on its way into L2 while this one is handled
#pragma unroll
      for (int t = 0; t < PACK_BATCH; ++t) asm volatile("prefetch.global.L2 [%0];" ::"l"(src + (size_t)(PACK_BATCH + t) * pitch));
    }
#pragma unroll
    for (int t = 0; t < PACK_BATCH; ++t)
      pack_one_sample(va[t], vb[t], np + (size_t)t * npitch, sp + (size_t)t * spitch, cnt + t, slut, acc, validp, lane);
    src += (size_t)PACK_BATCH * pitch;
    np += (size_t)PACK_BATCH * npitch;
    sp += (size_t)PACK_BATCH * spitch;
    cnt += PACK_BATCH;
  }
  for (; r < rows; ++r) {  // tail
    const uint4 va = load(reinterpret_cast<const uint4 *>(src)), vb = load(reinterpret_cast<const uint4 *>(src) + 1);
    pack_one_sample(va, vb, np, sp, cnt, slut, acc, validp, lane);
    src += pitch; np += npitch; sp += spitch; ++cnt;
  }
}

// valid sites of a word, in N-plane bit order
__device__ __forceinline__ uint32_t pack_validp(uint32_t nvalid) {
  uint32_t validp = nvalid == 32u ? 0xFFFFFFFFu : 0u;
  if (nvalid > 0u && nvalid < 32u)
    for (uint32_t t = 0; t < nvalid; ++t) validp |= 1u << pack_nbit(t);
  return validp;
}

// column-AND word of sites 8j..8j+7 (site-ordered nibbles) from the byte-per-site accumulators
__device__ __forceinline__ uint32_t pack_colword(const uint32_t (&acc)[8], int j, uint32_t nvalid) {
  // acc[2j] holds sites (0, 4, 1, 5) of the group, acc[2j+1] sites (2, 6, 3, 7), one per byte
  const uint32_t A = acc[2 * j], B = acc[2 * j + 1];
  uint32_t cw = (A & 0xFu) | (((A >> 16) & 0xFu) << 4) | ((B & 0xFu) << 8) | (((B >> 16) & 0xFu) << 12) |
                (((A >> 8) & 0xFu) << 16) | (((A >> 24) & 0xFu) << 20) | (((B >> 8) & 0xFu) << 24) | (((B >> 24) & 0xFu) << 28);
  // sites >= L in the last word must not look variable: force their nibbles non-zero
  const uint32_t v = nvalid > (uint32_t)j * 8u ? min(8u, nvalid - (uint32_t)j * 8u) : 0u;
  if (v < 8u) cw |= (v == 0u ? 0xFFFFFFFFu : (0xFFFFFFFFu << (4u * v)));
  return cw;
}

__global__ void __launch_bounds__(PACK_THREADS)
k_pack(const uint8_t *__restrict__ seqs, uint64_t s_begin, uint64_t s_end, uint64_t L, uint64_t pitch, uint32_t *__restrict__ colmask,
       uint32_t *__restrict__ nplane, uint64_t npitch /*words*/, uint8_t *__restrict__ nsum, uint64_t spitch /*bytes*/,
       uint32_t *__restrict__ ncount) {
  __shared__ uint8_t slut[256];
  __shared__ uint32_t s_ncnt[PACK_SCHUNK];  // N count of this CTA's sites, per sample of the chunk
  for (int i = threadIdx.x; i < PACK_SCHUNK; i += PACK_THREADS) s_ncnt[i] = 0;
  for (int i = threadIdx.x; i < 256; i += PACK_THREADS) slut[i] = (uint8_t)base_mask(i);
  __syncthreads();
  const uint32_t lane = threadIdx.x & 31;
  const uint64_t w = (uint64_t)blockIdx.x * PACK_THREADS + threadIdx.x;  // word index
  const uint64_t s0 = s_begin + (uint64_t)blockIdx.y * PACK_SCHUNK;
  const uint64_t s1 = min(s_end, s0 + PACK_SCHUNK);
  const uint64_t site0 = w * 32;
  // npitch is a multiple of 32 words, so a whole warp is either inside or outside the N-plane row
  const bool in_row = w < npitch;
  const bool has_sites = site0 < L;
  uint32_t acc[8];
#pragma unroll
  for (int q = 0; q < 8; ++q) acc[q] = ~0u;
  const uint32_t nvalid = has_sites ? (uint32_t)min((uint64_t)32, L - site0) : 0u;
  const uint32_t validp = pack_validp(nvalid);
  if (in_row)  // warp-uniform
    pack_rows(seqs + s0 * pitch + (has_sites ? site0 : 0), pitch, (uint32_t)(s1 - s0), has_sites, nplane + s0 * npitch + w,
              npitch, nsum + s0 * spitch + (w >> 5), spitch, s_ncnt, slut, acc, validp, lane);
  __syncthreads();
  for (uint64_t i = threadIdx.x; i < s1 - s0; i += PACK_THREADS)
    if (s_ncnt[i]) atomicAdd(ncount + s0 + i, s_ncnt[i]);
  if (has_sites) {
    uint32_t *cm = colmask + w * 4;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const uint32_t cw = pack_colword(acc, j, nvalid);
      if (cw != ~0u) atomicAnd(cm + j, cw);
    }
  }
}

// Early extraction (second DRAM pass avoided). k_pack_x is k_pack for a launch that is given a list of sites
// already known to be variable (`elist`, sorted; found by packing a first chunk of samples): besides everything
// k_pack does, it stores the masks of the listed sites, one byte per (sample, listed site), in X. Every warp parks the
// PACK_BATCH x 1 KB it has just loaded in its own shared-memory slot (conflict-free STS.128, warp barriers only)
// and its lanes then pick the warp's listed bytes out of it -- no second read of global memory. k_gather, which
// pays one 64-byte DRAM atom per (sample, variable site), is then only needed for the sites found variable later
// (and for the first chunk).
constexpr int PACKX_AHEAD = 1;  // batches between the L2 prefetch and the loads

template <bool SPARSE_N>
__global__ void __launch_bounds__(PACK_THREADS, 3)
k_pack_x(const uint8_t *__restrict__ seqs, uint64_t s_begin, uint64_t s_end, uint64_t L, uint64_t pitch, uint32_t *__restrict__ colmask,
         uint32_t *__restrict__ nplane, uint64_t npitch /*words*/, uint8_t *__restrict__ nsum, uint64_t spitch /*bytes*/,
         uint32_t *__restrict__ ncount, const uint32_t *__restrict__ elist, uint32_t VE, uint8_t *__restrict__ X, uint64_t XP) {
  // per warp and sample of the batch: 512 B of first halves, 512 B of second halves
  __shared__ __align__(16) uint8_t wbuf[PACK_THREADS / 32][PACK_BATCH][1024];
  __shared__ uint8_t slut[256];
  __shared__ uint32_t s_ncnt[PACK_SCHUNK];
  for (int i = threadIdx.x; i < PACK_SCHUNK; i += PACK_THREADS) s_ncnt[i] = 0;
  for (int i = threadIdx.x; i < 256; i += PACK_THREADS) slut[i] = (uint8_t)base_mask(i);
  __syncthreads();
  const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const uint64_t w = (uint64_t)blockIdx.x * PACK_THREADS + threadIdx.x;  // word index
  const uint64_t s0 = s_begin + (uint64_t)blockIdx.y * PACK_SCHUNK;
  const uint64_t s1 = min(s_end, s0 + PACK_SCHUNK);
  const uint64_t site0 = w * 32;
  const bool in_row = w < npitch;
  const bool has_sites = site0 < L;
  uint32_t acc[8];
#pragma unroll
  for (int q = 0; q < 8; ++q) acc[q] = ~0u;
  const uint32_t nvalid = has_sites ? (uint32_t)min((uint64_t)32, L - site0) : 0u;
  const uint32_t validp = pack_validp(nvalid);
  // listed sites inside this warp's 1024 sites: elist[e_lo .. e_lo + nE)
  const uint64_t wsite0 = (w - lane) * 32;
  auto lower = [&](uint64_t key) {
    uint32_t a = 0, b = VE;
    while (a < b) {
      const uint32_t mid = (a + b) >> 1;
      if (__ldg(elist + mid) < key) a = mid + 1; else b = mid;
    }
    return a;
  };
  const uint32_t e_lo = lower(wsite0), nE = lower(wsite0 + 1024) - e_lo;
  // work item i of a batch = (sample t = i / nE, listed site e = i % nE): where its byte sits in the slot and in X
  auto slot = [&](uint32_t t, uint32_t e) {
    const uint32_t o = __ldg(elist + e_lo + e) - (uint32_t)wsite0, k = o & 31u;  // lane o/32, byte k
    return t * 1024 + (o >> 5) * 16 + (k & 15u) + (k >> 4) * 512;
  };
  const uint32_t items = nE * PACK_BATCH;
  // the first two rounds live in registers (a warp rarely lists more than 16 sites); further rounds recompute
  // (slot address; its bits 10+ are the sample t) and (offset in X relative to the batch's first row)
  uint32_t it_a[2], it_x[2];
#pragma unroll
  for (int r = 0; r < 2; ++r) {
    const uint32_t i = lane + 32u * r;
    it_a[r] = 0xFFFFFFFFu;  // t never below `rows`
    it_x[r] = 0;
    if (i < items) {
      const uint32_t t = i / nE, e = i - t * nE;
      it_a[r] = slot(t, e);
      it_x[r] = t * (uint32_t)XP + e;  // XP <= L / 16 < 2^27
    }
  }
  uint8_t *mine = &wbuf[warp][0][lane * 16];
  const uint8_t *wb = &wbuf[warp][0][0];
  if (in_row) {  // warp-uniform
    const uint4 kN = make_uint4(0x4E4E4E4Eu, 0x4E4E4E4Eu, 0x4E4E4E4Eu, 0x4E4E4E4Eu);
    const uint8_t *src = seqs + s0 * pitch + (has_sites ? site0 : 0);
    uint32_t *np = nplane + s0 * npitch + w;
    uint8_t *sp = nsum + s0 * spitch + (w >> 5);
    uint32_t *cnt = s_ncnt;
    uint8_t *xrow = X + s0 * XP + e_lo;
    const bool more_items = items > 64;  // warp-uniform
    // one batch of `rows` samples (FULL: rows == PACK_BATCH, nothing predicated on it)
    auto batch = [&](auto full_tag, uint32_t rows, bool prefetch_next) {
      constexpr bool FULL = decltype(full_tag)::value;
      uint4 va[PACK_BATCH], vb[PACK_BATCH];
#pragma unroll
      for (int t = 0; t < PACK_BATCH; ++t) {
        // lanes past the end of the alignment read the start of the row instead: whatever they see is masked out
        // (validp == 0, no column word, never listed), so the loads need no per-lane predicate
        if (FULL || (uint32_t)t < rows) {
          va[t] = __ldcs(reinterpret_cast<const uint4 *>(src + (size_t)t * pitch));
          vb[t] = __ldcs(reinterpret_cast<const uint4 *>(src + (size_t)t * pitch) + 1);
        } else {
          va[t] = vb[t] = kN;
        }
      }
      if (prefetch_next) {  // the next batch on its way into L2 while this one is handled
#pragma unroll
        for (int t = 0; t < PACK_BATCH; ++t)
          asm volatile("prefetch.global.L2 [%0];" ::"l"(src + (size_t)(PACKX_AHEAD * PACK_BATCH + t) * pitch));
      }
      // every sample is parked in the warp's slot right before it is packed (the later loads of the batch are still in
      // flight then); the listed bytes are picked out once the whole batch is in place
#pragma unroll
      for (int t = 0; t < PACK_BATCH; ++t) {
        if (nE) {  // warp-uniform
          *reinterpret_cast<uint4 *>(mine + t * 1024) = va[t];
          *reinterpret_cast<uint4 *>(mine + t * 1024 + 512) = vb[t];
        }
        if (FULL || (uint32_t)t < rows)
          pack_one_sample<SPARSE_N>(va[t], vb[t], np + (size_t)t * npitch, sp + (size_t)t * spitch, cnt + t, slut, acc, validp, lane);
      }
      if (nE) {  // warp-uniform
        __syncwarp();
#pragma unroll
        for (int r = 0; r < 2; ++r) {  // the lookups run unconditionally (slot 0 for idle lanes), only the store is predicated
          const uint8_t m = slut[wb[it_a[r] & 0xFFFu]];
          if (FULL ? it_a[r] != 0xFFFFFFFFu : (it_a[r] >> 10) < rows) xrow[it_x[r]] = m;
        }
        if (more_items)
          for (uint32_t i = lane + 64; i < items; i += 32) {
            const uint32_t t = i / nE, e = i - t * nE;
            if (t < rows) xrow[(size_t)t * XP + e] = slut[wb[slot(t, e)]];
          }
        __syncwarp();
      }
      src += (size_t)PACK_BATCH * pitch;
      np += (size_t)PACK_BATCH * npitch;
      sp += (size_t)PACK_BATCH * spitch;
      cnt += PACK_BATCH;
      xrow += (size_t)PACK_BATCH * XP;
    };
    uint64_t b0 = s0;
    for (; b0 + (PACKX_AHEAD + 1) * PACK_BATCH <= s1; b0 += PACK_BATCH) batch(std::true_type{}, PACK_BATCH, true);
    for (; b0 + PACK_BATCH <= s1; b0 += PACK_BATCH) batch(std::true_type{}, PACK_BATCH, false);
    if (b0 < s1) batch(std::false_type{}, (uint32_t)(s1 - b0), false);
  }
  __syncthreads();
  for (uint64_t i = threadIdx.x; i < s1 - s0; i += PACK_THREADS)
    if (s_ncnt[i]) atomicAdd(ncount + s0 + i, s_ncnt[i]);
  if (has_sites) {
    uint32_t *cm = colmask + w * 4;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const uint32_t cw = pack_colword(acc, j, nvalid);
      if (cw != ~0u) atomicAnd(cm + j, cw);
    }
  }
}

}  // namespace tracs
#include "pack4.inl"
namespace tracs {

void encode_rows_device(const uint8_t *dev_ascii, uint64_t rows, uint64_t L, uint64_t pitch, uint8_t *dev_nib, uint64_t pitch4,
                        cudaStream_t st) {
  if (pitch % 32 != 0 || pitch < round_up(L, 32)) throw std::runtime_error("encode: ASCII pitch must be a multiple of 32 and >= L rounded up to 32");
  if (pitch4 % 16 != 0 || pitch4 * 2 < std::max<uint64_t>(32, round_up(L, 32))) throw std::runtime_error("encode: packed pitch must be a multiple of 16 bytes and hold L rounded up to 32 sites");
  const uint64_t total = rows * (pitch4 / 16);
  if (!total) return;
  k_encode<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(dev_ascii, rows, L, pitch, dev_nib, pitch4);
  g_stats.kernel_launches++;
  TRACS_CK(cudaGetLastError());
}

// site s is variable iff its column-AND nibble is 0
__global__ void k_siteflags(const uint32_t *__restrict__ colmask, uint64_t L, uint8_t *__restrict__ flags) {
  uint64_t g = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;  // group of 8 sites
  if (g * 8 >= L) return;
  uint32_t m = colmask[g];
  uint64_t out = 0;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    bool var = ((m >> (4 * i)) & 0xFu) == 0 && (g * 8 + i) < L;
    out |= (uint64_t)(var ? 1 : 0) << (8 * i);
  }
  *reinterpret_cast<uint64_t *>(flags + g * 8) = out;
}

// mask of one site of one row: ASCII byte through the table, or the nibble of the packed format (pack4.inl)
template <bool PACKED>
__device__ __forceinline__ uint32_t site_mask(const uint8_t *__restrict__ row, uint64_t site, const uint8_t *lut) {
  if (PACKED) return ((uint32_t)__ldg(row + (site >> 1)) >> ((site & 1u) * 4u)) & 15u;
  return lut[__ldg(row + site)];
}

// K0b: bit-slice the variable sites. One warp per (word, sample-chunk); lane <-> site.
template <bool PACKED>
__global__ void __launch_bounds__(256)
k_gather(const uint8_t *__restrict__ seqs, uint64_t n, uint64_t pitch, const uint32_t *__restrict__ site_idx, uint64_t V,
         uint4 *__restrict__ planes, uint64_t Npad, uint4 *__restrict__ planesT, uint64_t Wp, uint32_t schunk,
         uint32_t *__restrict__ amb_flag) {
  __shared__ uint8_t lut[256];
  lut[threadIdx.x] = (uint8_t)base_mask(threadIdx.x);
  __syncthreads();
  const uint32_t lane = threadIdx.x & 31;
  const uint64_t w = (uint64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (w * 32 >= V) return;
  const uint64_t v = w * 32 + lane;
  const bool live = v < V;
  const uint64_t site = live ? site_idx[v] : 0;
  const uint64_t s0 = (uint64_t)blockIdx.y * schunk, s1 = min(n, s0 + schunk);
  constexpr int GB = 8;  // byte loads in flight per lane
  for (uint64_t sb = s0; sb < s1; sb += GB) {
    uint32_t mk[GB];
#pragma unroll
    for (int t = 0; t < GB; ++t) mk[t] = (live && sb + t < s1) ? site_mask<PACKED>(seqs + (sb + t) * pitch, site, lut) : 15u;
#pragma unroll
    for (int t = 0; t < GB; ++t) {
      const uint64_t s = sb + t;
      if (s >= s1) break;
      const uint32_t m = mk[t];
      // two- or three-base codes at a variable site rule out the tensor-core identity (sweep_tc3.inl)
      if (__any_sync(0xFFFFFFFFu, m != 15u && (m & (m - 1)) != 0u) && lane == 0) atomicOr(amb_flag, 1u);
      if (__any_sync(0xFFFFFFFFu, live && m == 15u) && lane == 0) atomicOr(amb_flag, 2u);  // an N at a variable site
      const uint32_t A = __ballot_sync(0xFFFFFFFFu, m & 1);
      const uint32_t C = __ballot_sync(0xFFFFFFFFu, m & 2);
      const uint32_t G = __ballot_sync(0xFFFFFFFFu, m & 4);
      const uint32_t T = __ballot_sync(0xFFFFFFFFu, m & 8);
      if (lane == 0) {
        const uint4 v = make_uint4(A, C, G, T);
        planes[w * Npad + s] = v;    // word-major: tile panels are contiguous 2 KB rows
        planesT[s * Wp + w] = v;     // sample-major: per-pair refinement streams rows
      }
    }
  }
}

// ---- early-extraction path: byte matrices X[s][e] (mask of listed site e in sample s) -> planes ----------------
// masks of the listed sites for a sample range (the scattered DRAM pass, used for the first sample chunk and for
// the sites found variable only later). One warp per 32 listed sites and sample chunk.
template <bool PACKED>
__global__ void __launch_bounds__(256)
k_gather_bytes(const uint8_t *__restrict__ seqs, uint64_t s_begin, uint64_t s_end, uint64_t pitch, const uint32_t *__restrict__ list,
               uint32_t n_list, uint8_t *__restrict__ X, uint64_t XP, uint32_t schunk) {
  __shared__ uint8_t lut[256];
  lut[threadIdx.x] = (uint8_t)base_mask(threadIdx.x);
  __syncthreads();
  const uint32_t lane = threadIdx.x & 31;
  const uint64_t e = ((uint64_t)blockIdx.x * 8 + (threadIdx.x >> 5)) * 32 + lane;
  if (e - lane >= n_list) return;
  const bool live = e < n_list;
  const uint64_t site = live ? list[e] : 0;
  const uint64_t s0 = s_begin + (uint64_t)blockIdx.y * schunk, s1 = min(s_end, s0 + schunk);
  constexpr int GB = 8;
  for (uint64_t sb = s0; sb < s1; sb += GB) {
    uint32_t mk[GB];
#pragma unroll
    for (int t = 0; t < GB; ++t) mk[t] = (live && sb + t < s1) ? site_mask<PACKED>(seqs + (sb + t) * pitch, site, lut) : 15u;
#pragma unroll
    for (int t = 0; t < GB; ++t)
      if (live && sb + t < s1) X[(sb + t) * XP + e] = (uint8_t)mk[t];
  }
}

// where variable site v (sorted list `vlist`) finds its masks: in X (listed early, index in `elist`) or in X2
// (late, index = v - #early sites before it; elist is a subset of vlist). Also writes the late site list.
__global__ void k_site_sources(const uint32_t *__restrict__ vlist, uint32_t V, const uint32_t *__restrict__ elist, uint32_t VE,
                               uint32_t *__restrict__ src, uint32_t *__restrict__ late) {
  const uint32_t v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= V) return;
  const uint32_t site = vlist[v];
  uint32_t a = 0, b = VE;
  while (a < b) {
    const uint32_t mid = (a + b) >> 1;
    if (elist[mid] < site) a = mid + 1; else b = mid;
  }
  if (a < VE && elist[a] == site) {
    src[v] = a;
  } else {
    src[v] = 0x80000000u | (v - a);
    late[v - a] = site;
  }
}

// bit-slice the mask bytes into planes; same outputs as k_gather. One warp per PAIR of plane words and sample chunk.
// Fast path (the 64 sites of the pair sit in 64 consecutive, 16-byte aligned columns of X): lane <-> sample, each lane
// loads its 64 mask bytes and gathers bit b of every byte with a multiply (SWAR), so that a warp finishes 32 samples x
// 2 words per pass with coalesced stores to both layouts. Otherwise (late sites mixed in, tail): lane <-> site, ballots.
__device__ __forceinline__ uint32_t slice_bits4(uint32_t r, int b) {  // bit j of the result = bit b of byte j of r
  return (((r >> b) & 0x01010101u) * 0x01020408u) >> 24;
}
__device__ __forceinline__ uint4 slice_word(const uint4 &q0, const uint4 &q1) {  // 32 mask bytes -> A, C, G, T words
  const uint32_t r[8] = {q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, q1.z, q1.w};
  uint32_t o[4];
#pragma unroll
  for (int b = 0; b < 4; ++b) {
    uint32_t v = 0;
#pragma unroll
    for (int k = 0; k < 8; ++k) v |= (slice_bits4(r[k], b) & 0xFu) << (4 * k);
    o[b] = v;
  }
  return make_uint4(o[0], o[1], o[2], o[3]);
}
__device__ __forceinline__ bool slice_ambiguous(const uint4 &p) {  // some site with 2 or 3 of the 4 bits
  const uint32_t two = (p.x & p.y) | (p.x & p.z) | (p.x & p.w) | (p.y & p.z) | (p.y & p.w) | (p.z & p.w);
  return (two & ~(p.x & p.y & p.z & p.w)) != 0u;
}

__global__ void __launch_bounds__(256)
k_slice(const uint8_t *__restrict__ X, uint64_t XP, const uint8_t *__restrict__ X2, uint64_t X2P, const uint32_t *__restrict__ src,
        uint64_t V, uint64_t n, uint4 *__restrict__ planes, uint64_t Npad, uint4 *__restrict__ planesT, uint64_t Wp, uint32_t schunk,
        uint32_t *__restrict__ amb_flag) {
  const uint32_t lane = threadIdx.x & 31;
  const uint64_t w0 = ((uint64_t)blockIdx.x * 8 + (threadIdx.x >> 5)) * 2;  // first word of the pair
  if (w0 * 32 >= V) return;
  const uint64_t s0 = (uint64_t)blockIdx.y * schunk, s1 = min(n, s0 + schunk);
  // fast path test: both words complete, sources = 64 consecutive columns of X starting at a multiple of 16
  bool fast = (w0 + 2) * 32 <= V;
  uint32_t base = 0;
  if (fast) {
    const uint32_t a = src[w0 * 32 + lane], b = src[w0 * 32 + 32 + lane];
    base = __shfl_sync(0xFFFFFFFFu, a, 0);
    fast = __all_sync(0xFFFFFFFFu, a == base + lane && b == base + 32 + lane) && !(base & 0x80000000u) && (base & 15u) == 0;
  }
  if (fast) {
    bool amb = false, hasn = false;
    for (uint64_t s = s0 + lane; s < s1; s += 32) {
      const uint4 *row = reinterpret_cast<const uint4 *>(X + s * XP + base);
      const uint4 q0 = __ldg(row), q1 = __ldg(row + 1), q2 = __ldg(row + 2), q3 = __ldg(row + 3);
      const uint4 pa = slice_word(q0, q1), pb = slice_word(q2, q3);
      amb |= slice_ambiguous(pa) | slice_ambiguous(pb);
      hasn |= ((pa.x & pa.y & pa.z & pa.w) | (pb.x & pb.y & pb.z & pb.w)) != 0u;
      planes[w0 * Npad + s] = pa;
      planes[(w0 + 1) * Npad + s] = pb;
      planesT[s * Wp + w0] = pa;
      planesT[s * Wp + w0 + 1] = pb;
    }
    if (__any_sync(0xFFFFFFFFu, amb) && lane == 0) atomicOr(amb_flag, 1u);
    if (__any_sync(0xFFFFFFFFu, hasn) && lane == 0) atomicOr(amb_flag, 2u);
    return;
  }
  for (uint64_t w = w0; w < w0 + 2 && w * 32 < V; ++w) {
    const uint64_t v = w * 32 + lane;
    const bool live = v < V;
    const uint32_t sv = live ? src[v] : 0u;
    const uint8_t *col = (sv & 0x80000000u) ? X2 + (sv & 0x7FFFFFFFu) : X + sv;
    const uint64_t cp = (sv & 0x80000000u) ? X2P : XP;
    constexpr int GB = 8;
    for (uint64_t sb = s0; sb < s1; sb += GB) {
      uint8_t mk[GB];
#pragma unroll
      for (int t = 0; t < GB; ++t) mk[t] = (live && sb + t < s1) ? __ldg(col + (sb + t) * cp) : (uint8_t)15;
#pragma unroll
      for (int t = 0; t < GB; ++t) {
        const uint64_t s = sb + t;
        if (s >= s1) break;
        const uint32_t m = mk[t];
        if (__any_sync(0xFFFFFFFFu, m != 15u && (m & (m - 1)) != 0u) && lane == 0) atomicOr(amb_flag, 1u);
        if (__any_sync(0xFFFFFFFFu, live && m == 15u) && lane == 0) atomicOr(amb_flag, 2u);
        const uint32_t A = __ballot_sync(0xFFFFFFFFu, m & 1);
        const uint32_t C = __ballot_sync(0xFFFFFFFFu, m & 2);
        const uint32_t G = __ballot_sync(0xFFFFFFFFu, m & 4);
        const uint32_t T = __ballot_sync(0xFFFFFFFFu, m & 8);
        if (lane == 0) {
          const uint4 o = make_uint4(A, C, G, T);
          planes[w * Npad + s] = o;
          planesT[s * Wp + w] = o;
        }
      }
    }
  }
}

// ------------------------------------------------------------------------------------------
// K1: the pair sweep
// ------------------------------------------------------------------------------------------
struct SweepArgs {
  const uint4 *planes;  // [Wp][Npad]
  uint32_t Wp;          // padded word count (multiple of KC)
  uint32_t Npad;
  uint32_t n, i_end, j_start;
  int32_t dist;
  // tile list: row-blocks of this launch and the prefix of their tile counts
  const uint32_t *rb_list;     // [n_rb]
  const uint32_t *tile_prefix; // [n_rb + 1]
  uint32_t n_rb;
  uint32_t n_tiles;
  uint32_t cb_min;  // first col-block allowed by j_start
  const uint2 *tile_table;  // [n_tiles] (row-block, col-block) of every tile of the launch (k_tile_table)
  const uint32_t *tc_ncnt;  // k_sweep_tc3<4>: per-sample N count over the swept words (k_tc_ncount), else null
  union {
    // thresholded sweeps: the edge list
    struct {
      unsigned long long *counter;
      uint64_t *keys;
      uint32_t *dvals;
      unsigned long long cap;
    };
    // dense sweeps (k_sweep<true>, k_sweep_tc3<NP, true>): d(i, j) of every pair of the range is stored at
    // dense[i * dense_ld + j - dense_col0], and with dense_mirror (square matrix) also at dense[j * dense_ld + i], plus an
    // explicit 0 on the diagonal. No threshold, no list, no atomics. (A union: the struct keeps its size, and a larger
    // parameter block changed the register allocation, and spills, of the existing tensor-core kernels.)
    struct {
      int32_t *dense;
      uint64_t dense_ld;
      uint32_t dense_col0;
      uint32_t dense_mirror;
    };
  };
  uint32_t one;  // == 1, opaque to the compiler: acc += popc * one issues as IMAD on the FMA pipe
};

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
  uint32_t done;
  do {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(done)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
  } while (!done);
}
// 1-D bulk async copy global -> shared, completion signalled on an mbarrier (SASS: UBLKCP)
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

// tile -> (row-block, col-block), once per launch list: the tile kernels then need one 8-byte load per tile instead of
// a binary search over the prefix array (ten dependent L2 round trips: 40 % of an 8-word prefilter tile)
__global__ void k_tile_table(const uint32_t *__restrict__ rb_list, const uint32_t *__restrict__ tile_prefix, uint32_t n_rb, uint32_t cb_min,
                             uint32_t n_tiles, uint2 *__restrict__ table) {
  const uint32_t tile = blockIdx.x * blockDim.x + threadIdx.x;
  if (tile >= n_tiles) return;
  uint32_t lo = 0, hi = n_rb;
  while (hi - lo > 1) {
    const uint32_t mid = (lo + hi) >> 1;
    if (tile_prefix[mid] <= tile) lo = mid; else hi = mid;
  }
  const uint32_t rb = rb_list[lo];
  table[tile] = make_uint2(rb, max(rb, cb_min) + (tile - tile_prefix[lo]));
}

constexpr int SWEEP_THREADS = 256;
constexpr int STAGE_U4 = KC * TILE;  // uint4 per stage per side
constexpr uint32_t PREFILTER_WORDS = 64;  // widest prefilter window: 2048 variable sites
// Prefilter window for a threshold: 32 * words sites must be many times the allowed distance for unrelated pairs to
// fall out of it; 8 sites per allowed SNP, in steps of 16 words (dist <= 63: 16 words = 512 sites).
static inline uint32_t prefilter_words(int64_t dist) {
  const uint64_t w = ((uint64_t)(dist + 1) * 8 + 31) / 32;
  return (uint32_t)std::min<uint64_t>(PREFILTER_WORDS, std::max<uint64_t>(16, round_up(w, 16)));
}
// Windows tried in turn by the filter-and-refine path: 4, 8, 16, 64 words (128 ... 2048 variable sites), starting where
// the window holds about six sites per allowed SNP (dist <= 20: 4 words). A failed attempt costs its own sweep only.
static inline uint32_t first_window(int64_t dist) {
  if (dist < 22) return 4;
  if (dist < 43) return 8;
  return prefilter_words(dist);
}
// narrowest prefilter window that goes to the tensor-core kernel when the masks allow it (DESIGN.md section 7)
constexpr uint32_t TC_MIN_WORDS = 17;
static inline uint32_t next_window(uint32_t pw) { return pw < 8 ? 8 : pw < 16 ? 16 : (pw < PREFILTER_WORDS ? PREFILTER_WORDS : 0); }
constexpr size_t SWEEP_SMEM = (size_t)STAGES * 2 * STAGE_U4 * sizeof(uint4);

// The dynamic shared-memory array of every tile kernel of this file: its first declaration fixes the alignment for all
// of them (128 B; the tensor-core kernels align their stages themselves). Declared here because k_sweep, a template,
// is only instantiated after the tensor-core kernels, whose own declarations ask for 1024 B.
extern __shared__ __align__(128) uint8_t smem_raw[];

// DENSE: the epilogue stores every distance of the range (SweepArgs.dense) instead of thresholding and appending; a
// template parameter, so that the thresholded instantiation compiles to the code it always had.
template <bool DENSE>
__global__ void __launch_bounds__(SWEEP_THREADS, 1) k_sweep(const SweepArgs a) {
  extern __shared__ __align__(128) uint8_t smem_raw[];
  uint4 *srow = reinterpret_cast<uint4 *>(smem_raw);       // [STAGES][KC][TILE]
  uint4 *scol = srow + (size_t)STAGES * STAGE_U4;          // [STAGES][KC][TILE]
  __shared__ __align__(8) uint64_t full[STAGES];
  __shared__ uint2 s_tile[4];  // coordinates of the tiles whose panels are in flight (written by the issuing thread)
  // Hits of a thresholded sweep are parked here and leave in batches: a lane with a hit used to reserve its place in the
  // global list with an atomic of its own, and its warp -- and through the chunk barrier the whole CTA -- sat out the
  // round trip to L2 (about 1 000 clk, on nearly every tile of a prefilter launch: a third of the kernel's samples).
  constexpr uint32_t HB_CAP = 1024, HB_FLUSH = 512, HB_LANE_MAX = 4;  // a tile parks at most 8 warps x 8 lanes x 4 entries
  __shared__ uint64_t hb_key[HB_CAP];
  __shared__ uint32_t hb_val[HB_CAP];
  __shared__ uint32_t hb_count;
  __shared__ unsigned long long hb_base;

  const uint32_t tid = threadIdx.x;
  const uint32_t tx = tid & 15, ty = tid >> 4;
  if (tid == 0) {
    for (int s = 0; s < STAGES; ++s) mbar_init(&full[s], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    hb_count = 0;
  }
  __syncthreads();
  // all threads, at a point where nobody appends (right after a chunk barrier / after the last tile)
  auto flush_hits = [&]() {
    const uint32_t cnt = hb_count;
    if (tid == 0) hb_base = cnt ? atomicAdd(a.counter, (unsigned long long)cnt) : 0ull;
    __syncthreads();
    const unsigned long long base = hb_base;
    for (uint32_t e = tid; e < cnt; e += SWEEP_THREADS)
      if (base + e < a.cap) {
        a.keys[base + e] = hb_key[e];
        a.dvals[base + e] = hb_val[e];
      }
    __syncthreads();
    if (tid == 0) hb_count = 0;
    __syncthreads();
  };

  // a window narrower than one stage (Wp = 4): one chunk per tile of which only the first Wp words are evaluated (the
  // copies still bring KC words; the planes always hold at least KC)
  const uint32_t nk = (a.Wp + KC - 1) / KC;
  const int kc_used = a.Wp < (uint32_t)KC ? (int)a.Wp : KC;
  const uint32_t one = a.one;
  // The panels of ALL tiles of this CTA form one stream of chunks g = tile_iter * nk + c (stage = g % STAGES, parity =
  // (g / STAGES) & 1): chunk g + STAGES is requested as soon as chunk g has been consumed, whichever tile it belongs to,
  // so the first panels of the next tile arrive during the epilogue of this one (short prefilter windows have 1-2
  // chunks per tile and would otherwise expose the full load latency on every tile).
  const uint32_t my_tiles = blockIdx.x < a.n_tiles ? (a.n_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
  const uint32_t total_chunks = my_tiles * nk;
  // Requests are made by the 32 lanes of warp 0 TOGETHER: lane 0 arms the barrier, lanes 0..15 each start one of the 16
  // bulk copies of a chunk, the position in the stream advances by counters (no division), and the coordinates of the
  // next tile are fetched one request ahead. (One thread doing all of this serially -- a table load, two integer
  // divisions, 16 address computations and copies, ~250 dependent instructions -- held warp 0, and through the chunk
  // barrier the whole CTA, for about 2 000 clk per chunk: a third of a 4-word prefilter tile, a fifth of an 8-word chunk.)
  const uint32_t warp_id = tid >> 5, lane_id = tid & 31;
  uint32_t iss_g = 0, iss_t = 0, iss_c = 0, iss_slot = 0;  // next chunk to request: stream index, tile iteration, chunk, stage
  uint2 rc_next = my_tiles ? __ldg(a.tile_table + blockIdx.x) : make_uint2(0u, 0u);  // coordinates of tile iteration iss_t
  auto issue = [&]() {
    const uint2 rc = rc_next;
    uint64_t *bar = &full[iss_slot];
    if (lane_id == 0) {
      if (iss_c == 0) s_tile[iss_t & 3] = rc;  // parked for everybody (read after a later barrier: at most 3 tiles in flight, 4 slots)
      mbar_expect_tx(bar, 2u * STAGE_U4 * (uint32_t)sizeof(uint4));
    }
    __syncwarp();
    if (lane_id < 2u * KC) {
      const uint32_t kk = lane_id >> 1;
      const bool is_col = (lane_id & 1u) != 0u;
      const uint4 *src = a.planes + (size_t)(is_col ? rc.y : rc.x) * TILE + (size_t)(iss_c * KC + kk) * a.Npad;
      uint4 *dst = (is_col ? scol : srow) + (size_t)iss_slot * STAGE_U4 + kk * TILE;
      bulk_g2s(dst, src, TILE * sizeof(uint4), bar);
    }
    ++iss_g;
    iss_slot = iss_slot + 1 == (uint32_t)STAGES ? 0u : iss_slot + 1;
    if (++iss_c == nk) {
      iss_c = 0;
      if (++iss_t < my_tiles) rc_next = __ldg(a.tile_table + blockIdx.x + (size_t)iss_t * gridDim.x);
    }
  };
  if (warp_id == 0)
    while (iss_g < (uint32_t)STAGES && iss_g < total_chunks) issue();
  __syncthreads();
  uint32_t it = 0;  // running chunk counter
  uint32_t t_iter = 0;

  for (uint32_t tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x, ++t_iter) {
    const uint2 rc = s_tile[t_iter & 3];
    const uint32_t rb = rc.x, cb = rc.y;

    uint32_t acc[8][8];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[i][j] = 0;

    for (uint32_t c = 0; c < nk; ++c, ++it) {
      const uint32_t slot = it % STAGES;
      mbar_wait(&full[slot], (it / STAGES) & 1u);
      const uint4 *pr = srow + (size_t)slot * STAGE_U4 + ty;
      const uint4 *pc = scol + (size_t)slot * STAGE_U4 + tx;
#pragma unroll 2
      for (int kk = 0; kk < kc_used; ++kk) {
        uint4 r[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) r[i] = pr[kk * TILE + i * 16];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const uint4 cv = pc[kk * TILE + j * 16];
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const uint32_t m = (r[i].x & cv.x) | (r[i].y & cv.y) | (r[i].z & cv.z) | (r[i].w & cv.w);
            // accumulate on the FMA pipe (IMAD) so the ALU pipe only carries the four LOP3
            acc[i][j] = __popc(m) * one + acc[i][j];
          }
        }
      }
      // The chunk barrier doubles as the vote on flushing the parked hits. Threads look at the counter BEFORE the
      // barrier, while slower warps may still be appending the previous tile's hits (at most 256), so they may see
      // different values: the OR makes the decision uniform, and a count above HB_FLUSH at one barrier is seen by
      // everybody at the next one at the latest: the buffer never holds more than HB_FLUSH + 2 x 256 = HB_CAP entries.
      const int want_flush = c + 1 == nk && *(volatile uint32_t *)&hb_count > HB_FLUSH;
      const int do_flush = __syncthreads_or(want_flush);
      if (warp_id == 0 && iss_g < total_chunks) issue();  // chunk it + STAGES
      if (do_flush) flush_hits();
    }

    // ---- epilogue: threshold + append -------------------------------------------------
    const uint32_t total_bits = a.Wp * 32u;
    if constexpr (DENSE) {
      // thread (tx, ty) holds rows rb*128 + i*16 + ty, cols cb*128 + j*16 + tx: the upper stores coalesce over tx, the
      // mirror stores (square matrix) are scattered
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const uint32_t gi = rb * TILE + i * 16 + ty;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const uint32_t gj = cb * TILE + j * 16 + tx;
          if (gi < a.i_end && gj < a.n && gj > gi && gj >= a.j_start) {
            const int32_t d = (int32_t)(total_bits - acc[i][j]);
            a.dense[(uint64_t)gi * a.dense_ld + (gj - a.dense_col0)] = d;
            if (a.dense_mirror) a.dense[(uint64_t)gj * a.dense_ld + gi] = d;
          }
        }
        if (a.dense_mirror && cb == rb && tx == ty && gi < a.n) a.dense[(uint64_t)gi * a.dense_ld + gi] = 0;
      }
      continue;
    }
    const uint32_t lane = tid & 31;
    // Most threads of a thresholded sweep hold no pair within the threshold (d = total_bits - matches): row maxima
    // of the 8 x 8 match counts decide that with ~70 instructions instead of ~15 per pair. A warp without any hit
    // skips the epilogue; a warp with a FEW hits lets just those lanes walk their qualifying rows and append with one
    // atomic per lane (the order of the list is restored by the sort); a warp with many hits (unthresholded or
    // dense output) takes the warp-aggregated path below.
    uint32_t rmax[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      uint32_t m = acc[i][0];
#pragma unroll
      for (int j = 1; j < 8; ++j) m = max(m, acc[i][j]);
      rmax[i] = m;
    }
    uint32_t mx = rmax[0];
#pragma unroll
    for (int i = 1; i < 8; ++i) mx = max(mx, rmax[i]);
    const bool hit = (int32_t)(total_bits - mx) <= a.dist;
    const uint32_t hits = __ballot_sync(0xFFFFFFFFu, hit);
    if (!hits) continue;
    if (__popc(hits) <= 8) {
      if (hit) {
        // Each of the few lanes with a hit walks ITS qualifying rows (usually one): the row is selected out of the 64
        // accumulators once (8 x 8 predicated moves), its eight pairs are tested, and a pair that passes is parked.
        // Different lanes work on different rows in the same trip. (Testing all 64 pairs into a bit mask and fetching
        // each hit with a 64-way select afterwards cost ~500 instructions per warp and tile; parking from inside fully
        // unrolled 8 x 8 loops was worse still: the compiler predicates the whole body 64 times.)
        uint32_t rowmask = 0;
#pragma unroll
        for (int i = 0; i < 8; ++i) rowmask |= ((int32_t)(total_bits - rmax[i]) <= a.dist ? 1u : 0u) << i;
        uint32_t parked = 0;
        while (rowmask) {
          const int i = __ffs(rowmask) - 1;
          rowmask &= rowmask - 1;
          uint32_t rv[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            uint32_t v = acc[0][j];
#pragma unroll
            for (int ii = 1; ii < 8; ++ii) v = i == ii ? acc[ii][j] : v;
            rv[j] = v;
          }
          const uint32_t gi = rb * TILE + (uint32_t)i * 16 + ty;
          uint32_t keepj = 0;
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const uint32_t gj = cb * TILE + j * 16 + tx;
            const bool ok = (int32_t)(total_bits - rv[j]) <= a.dist && gi < a.i_end && gj < a.n && gj > gi && gj >= a.j_start;
            keepj |= (ok ? 1u : 0u) << j;
          }
          while (keepj) {
            const int j = __ffs(keepj) - 1;
            keepj &= keepj - 1;
            uint32_t v = rv[0];
#pragma unroll
            for (int jj = 1; jj < 8; ++jj) v = j == jj ? rv[jj] : v;
            const uint64_t key = ((uint64_t)gi << 32) | (cb * TILE + (uint32_t)j * 16 + tx);
            if (parked < HB_LANE_MAX) {
              const uint32_t pos = atomicAdd(&hb_count, 1u);  // shared memory; < HB_CAP by construction
              hb_key[pos] = key;
              hb_val[pos] = total_bits - v;
              ++parked;
            } else {  // a lane with many hits: straight to the list
              const unsigned long long pos = atomicAdd(a.counter, 1ull);
              if (pos < a.cap) {
                a.keys[pos] = key;
                a.dvals[pos] = total_bits - v;
              }
            }
          }
        }
      }
      continue;
    }
    uint32_t cnt = 0;
    uint64_t keep = 0;  // bit (i*8+j)
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const uint32_t gi = rb * TILE + i * 16 + ty;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const uint32_t gj = cb * TILE + j * 16 + tx;
        const int32_t d = (int32_t)(total_bits - acc[i][j]);
        const bool ok = gi < a.i_end && gj < a.n && gj > gi && gj >= a.j_start && d <= a.dist;
        if (ok) {
          keep |= 1ull << (i * 8 + j);
          cnt++;
        }
      }
    }
    // warp-aggregated reservation
    uint32_t incl = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      uint32_t t = __shfl_up_sync(0xFFFFFFFFu, incl, o);
      if (lane >= (uint32_t)o) incl += t;
    }
    const uint32_t wtot = __shfl_sync(0xFFFFFFFFu, incl, 31);
    if (wtot) {
      unsigned long long base = 0;
      if (lane == 31) base = atomicAdd(a.counter, (unsigned long long)wtot);
      base = __shfl_sync(0xFFFFFFFFu, base, 31);
      unsigned long long pos = base + (incl - cnt);
#pragma unroll
      for (int i = 0; i < 8; ++i) {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          if ((keep >> (i * 8 + j)) & 1ull) {
            if (pos < a.cap) {
              const uint32_t gi = rb * TILE + i * 16 + ty;
              const uint32_t gj = cb * TILE + j * 16 + tx;
              a.keys[pos] = ((uint64_t)gi << 32) | gj;
              a.dvals[pos] = total_bits - acc[i][j];
            }
            pos++;
          }
        }
      }
    }
  }
  __syncthreads();
  flush_hits();
}

// expand sorted keys into the output columns
__global__ void k_expand(const uint64_t *__restrict__ keys, const uint32_t *__restrict__ dvals, uint64_t E,
                         uint64_t *__restrict__ rows, uint64_t *__restrict__ cols, uint64_t *__restrict__ dist) {
  uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= E) return;
  uint64_t k = keys[e];
  rows[e] = k >> 32;
  cols[e] = k & 0xFFFFFFFFull;
  dist[e] = dvals[e];
}

// ------------------------------------------------------------------------------------------
// K1b: refinement of prefilter candidates. The tile sweep over the first w0 words leaves only pairs
// whose PARTIAL distance is <= dist (d is monotone in the number of sites, so every other pair is
// already decided). One warp finishes one candidate over words [w0, Wp) of the sample-major planes.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
k_refine(const uint64_t *__restrict__ ckeys, const uint32_t *__restrict__ cdvals, uint64_t n_cand,
         const uint4 *__restrict__ planesT, uint32_t Wp, uint32_t w0, int32_t dist, unsigned long long *counter,
         uint64_t *__restrict__ keys, uint32_t *__restrict__ dvals) {
  const uint64_t e = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const uint32_t lane = threadIdx.x & 31;
  if (e >= n_cand) return;
  const uint64_t k = ckeys[e];
  const uint4 *ri = planesT + (k >> 32) * Wp;
  const uint4 *rj = planesT + (k & 0xFFFFFFFFull) * Wp;
  uint32_t mism = 0;
#pragma unroll 4
  for (uint32_t w = w0 + lane; w < Wp; w += 32) {
    const uint4 x = __ldg(ri + w), y = __ldg(rj + w);
    mism += __popc(~((x.x & y.x) | (x.y & y.y) | (x.z & y.z) | (x.w & y.w)));
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mism += __shfl_xor_sync(0xFFFFFFFFu, mism, o);
  if (lane == 0) {
    const uint32_t d = cdvals[e] + mism;
    if ((int32_t)d <= dist) {
      const unsigned long long pos = atomicAdd(counter, 1ull);
      keys[pos] = k;
      dvals[pos] = d;
    }
  }
}

// Second, per-candidate prefilter after a NARROW tile window (4 or 8 words): one thread continues each candidate over
// the next `extra` words of the sample-major planes and drops it once the partial distance passes `dist`. A narrow
// window lets a few unrelated pairs through; left in, they would bridge clusters into large, sparse components of
// the candidate graph (pairs.inl evaluates dense components as blocks). flags[e] = keep.
__global__ void __launch_bounds__(256)
k_cand_trim(const uint64_t *__restrict__ keys, const uint32_t *__restrict__ dvals, uint64_t n_cand, const uint4 *__restrict__ planesT,
            uint32_t Wp, uint32_t w0, uint32_t extra, int32_t dist, uint8_t *__restrict__ flags) {
  const uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n_cand) return;
  const uint64_t k = keys[e];
  const uint4 *ri = planesT + (k >> 32) * Wp + w0, *rj = planesT + (k & 0xFFFFFFFFull) * Wp + w0;
  uint32_t d = dvals[e];
  for (uint32_t w = 0; w < extra && (int32_t)d <= dist; w += 4) {
#pragma unroll
    for (uint32_t q = 0; q < 4; ++q) {
      if (w + q < extra) {
        const uint4 x = __ldg(ri + w + q), y = __ldg(rj + w + q);
        d += __popc(~((x.x & y.x) | (x.y & y.y) | (x.z & y.z) | (x.w & y.w)));
      }
    }
  }
  flags[e] = (int32_t)d <= dist ? 1 : 0;
}

// ------------------------------------------------------------------------------------------
// K4: recombination filter for emitted edges (filter=True). Restates src/pairsnp.hpp:251-318:
//   p = d / L; half-window h = clamp(int(1/p/2 + 1), 50, 5000); for every SNP of the pair, count the
//   pair's SNPs inside [pos-h, pos+h+1) (clipped to the alignment) and their span last-first+1
//   (range_count :223-248); the SNP is kept if it is alone in its window or
//   1 - BinomCDF(count; span, p) >= 0.05 / d.  filt = number of SNPs kept; d <= 1 -> d.
// SNPs only occur at variable sites, so positions come from the compacted planes + site index.
// The binomial CDF is summed term by term in fp64 (Boost uses the incomplete beta function: same
// value to rounding; see DESIGN.md "unpinned corner").
// Pass 1 (one warp per edge): ordered SNP positions into a scratch list. Pass 2: the window test.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
k_snp_positions(const uint64_t *__restrict__ keys, uint64_t e0, uint64_t e1, const uint4 *__restrict__ planesT, uint32_t Wp,
                const uint32_t *__restrict__ site_idx, uint64_t V, const uint64_t *__restrict__ offs, uint64_t base,
                uint32_t *__restrict__ pos) {
  const uint64_t e = e0 + (((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
  const uint32_t lane = threadIdx.x & 31;
  if (e >= e1) return;
  const uint64_t k = keys[e];
  const uint4 *ri = planesT + (k >> 32) * Wp;
  const uint4 *rj = planesT + (k & 0xFFFFFFFFull) * Wp;
  uint32_t *out = pos + (offs[e] - base);
  uint32_t written = 0;
  for (uint32_t w0 = 0; w0 < Wp; w0 += 32) {
    const uint32_t w = w0 + lane;
    uint32_t mis = 0;
    if (w < Wp) {
      const uint4 x = __ldg(ri + w), y = __ldg(rj + w);
      mis = ~((x.x & y.x) | (x.y & y.y) | (x.z & y.z) | (x.w & y.w));
    }
    const uint32_t c = __popc(mis);
    uint32_t incl = c;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, incl, o);
      if (lane >= (uint32_t)o) incl += t;
    }
    uint32_t at = written + incl - c;
    while (mis) {
      const uint32_t b = __ffs(mis) - 1;
      mis &= mis - 1;
      const uint64_t v = (uint64_t)w * 32 + b;
      out[at++] = v < V ? site_idx[v] : 0u;  // v >= V cannot happen: pad bits always match
    }
    written += __shfl_sync(0xFFFFFFFFu, incl, 31);
  }
}

__global__ void __launch_bounds__(256)
k_filter_recomb(const uint32_t *__restrict__ dvals, uint64_t e0, uint64_t e1, const uint64_t *__restrict__ offs, uint64_t base,
                const uint32_t *__restrict__ pos, uint64_t L, const double *__restrict__ lg, uint32_t *__restrict__ filt) {
  const uint64_t e = e0 + (((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
  const uint32_t lane = threadIdx.x & 31;
  if (e >= e1) return;
  const uint32_t d = dvals[e];
  if (d <= 1) {
    if (lane == 0) filt[e] = d;
    return;
  }
  const uint32_t *ps = pos + (offs[e] - base);
  const int aln = (int)L;
  const double dd = (double)d;
  const double p = dd / aln, thr = 0.05 / dd;
  int h = (int)(1.0 / p / 2.0 + 1);
  h = min(h, 5000);
  h = max(h, 50);
  const double lp = log(p), lq = log1p(-p);
  uint32_t kept = 0;
  for (uint32_t s = lane; s < d; s += 32) {
    const int i = (int)ps[s];
    const int left = max(0, i - h), right = min(aln, i + h + 1);
    // first SNP >= left, first SNP >= right
    uint32_t lo = 0, hi = s;
    while (lo < hi) { const uint32_t m = (lo + hi) >> 1; if ((int)ps[m] < left) lo = m + 1; else hi = m; }
    const uint32_t a = lo;
    lo = s; hi = d;
    while (lo < hi) { const uint32_t m = (lo + hi) >> 1; if ((int)ps[m] < right) lo = m + 1; else hi = m; }
    const uint32_t b = lo;
    const uint32_t cnt = b - a;
    if (cnt > 1) {
      const double n = (double)(int)(ps[b - 1] - ps[a] + 1), kk = (double)(int)cnt;
      double cdf;
      if (kk >= n) cdf = 1.0;
      else {
        cdf = 0.0;
        const int ni = (int)n;
        for (int t = 0; t <= (int)cnt; ++t)
          cdf += exp(lg[ni + 1] - lg[t + 1] - lg[ni - t + 1] + (double)t * lp + (double)(ni - t) * lq);
        if (cdf > 1.0) cdf = 1.0;
      }
      if (1.0 - cdf >= thr) kept++;
    } else {
      kept++;
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) kept += __shfl_xor_sync(0xFFFFFFFFu, kept, o);
  if (lane == 0) filt[e] = kept;
}
// compact device-resident copy of the edge columns (tracs_edges_t.dev_packed)
__global__ void k_pack_edges(const uint64_t *__restrict__ keys, const uint32_t *__restrict__ dvals, const uint64_t *__restrict__ ncomp,
                             const double *__restrict__ p0, const double *__restrict__ eK, uint64_t E, uint8_t *__restrict__ out) {
  const uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= E) return;
  uint32_t *u = reinterpret_cast<uint32_t *>(out);
  double *f = reinterpret_cast<double *>(out + 16 * E);
  const uint64_t k = keys[e];
  u[e] = (uint32_t)(k >> 32);
  u[E + e] = (uint32_t)k;
  u[2 * E + e] = dvals[e];
  u[3 * E + e] = ncomp ? (uint32_t)ncomp[e] : 0u;
  f[e] = p0 ? p0[e] : 0.0;
  f[E + e] = eK ? eK[e] : 0.0;
}
struct WidenU32 {
  __host__ __device__ __forceinline__ uint64_t operator()(const uint32_t &v) const { return (uint64_t)v; }
};
__global__ void k_widen(const uint32_t *__restrict__ in, uint64_t E, uint64_t *__restrict__ out) {
  const uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e < E) out[e] = in[e];
}

// Locality order for K2: rep[s] = smallest sample linked to s by an edge (the cluster's first member
// for clique-like clusters). Edges are processed grouped by rep[row], so the N-plane rows of one
// cluster stay in L2 while all of its edges are evaluated. Purely a schedule: results are written
// to each edge's own slot.
__global__ void k_rep_init(uint32_t *rep, uint32_t n) {
  uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s < n) rep[s] = s;
}
__global__ void k_rep_min(const uint64_t *__restrict__ keys, uint64_t E, uint32_t *rep) {
  const uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= E) return;
  const uint64_t k = keys[e];
  atomicMin(rep + (k & 0xFFFFFFFFull), (uint32_t)(k >> 32));
}
__global__ void k_rep_keys(const uint64_t *__restrict__ keys, uint64_t E, const uint32_t *__restrict__ rep,
                           uint32_t *__restrict__ okey, uint32_t *__restrict__ oval) {
  const uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= E) return;
  okey[e] = rep[keys[e] >> 32];
  oval[e] = (uint32_t)e;
}

// ------------------------------------------------------------------------------------------
// K2: compared sites. nn = L - |N_i u N_j| = L - (|N_i| + |N_j| - |N_i n N_j|).
// The intersection walks the block summaries (1 bit / 128 sites) and touches the N-plane only
// where BOTH samples have an N in the block. One warp per edge.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
k_ncomp(const uint64_t *__restrict__ keys, uint64_t E, const uint32_t *__restrict__ nplane, uint64_t npitch,
        const uint8_t *__restrict__ nsum, uint64_t spitch, const uint32_t *__restrict__ ncount, uint64_t L,
        const uint32_t *__restrict__ order, uint64_t *__restrict__ ncomp) {
  const uint64_t slot = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const uint32_t lane = threadIdx.x & 31;
  if (slot >= E) return;
  const uint64_t e = order ? order[slot] : slot;  // processing order groups edges of one cluster (L2 reuse)
  const uint64_t k = keys[e];
  const uint64_t i = k >> 32, j = k & 0xFFFFFFFFull;
  const uint32_t *si = reinterpret_cast<const uint32_t *>(nsum + i * spitch);
  const uint32_t *sj = reinterpret_cast<const uint32_t *>(nsum + j * spitch);
  const uint4 *ni = reinterpret_cast<const uint4 *>(nplane + i * npitch);
  const uint4 *nj = reinterpret_cast<const uint4 *>(nplane + j * npitch);
  uint32_t inter = 0;
  const uint64_t nq = spitch / 4;
  for (uint64_t q = lane; q < nq; q += 32) {
    uint32_t m = __ldg(si + q) & __ldg(sj + q);
    while (m) {
      uint32_t b = __ffs(m) - 1;
      m &= m - 1;
      uint64_t blk = q * 32 + b;
      uint4 x = __ldg(ni + blk), y = __ldg(nj + blk);
      inter += __popc(x.x & y.x) + __popc(x.y & y.y) + __popc(x.z & y.z) + __popc(x.w & y.w);
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) inter += __shfl_xor_sync(0xFFFFFFFFu, inter, o);
  if (lane == 0) ncomp[e] = L - ((uint64_t)ncount[i] + ncount[j] - inter);
}

// ------------------------------------------------------------------------------------------
// K3 (fused): transmission likelihood for the emitted edges, all on the device.
// Dates have day resolution (tracs/transcluster.py:26-33), so the memo key (N, delta) of
// src/transcluster.hpp:245-274 is (d, |day_i - day_j|): a dense table indexed d * DD + dd.
//   mark used keys -> compact -> one thread per used key runs the series -> per-edge gather
// ------------------------------------------------------------------------------------------
// (E_dev != nullptr: the edge count lives on the device, E is the launch's upper bound)
__global__ void k_trans_mark(const uint64_t *__restrict__ keys, const uint32_t *__restrict__ dvals, uint64_t E,
                             const uint64_t *__restrict__ E_dev, const int32_t *__restrict__ days, uint32_t DD,
                             uint8_t *__restrict__ used) {
  const uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= (E_dev ? *E_dev : E)) return;
  const uint64_t k = keys[e];
  const int32_t dd = abs(days[k >> 32] - days[k & 0xFFFFFFFFull]);
  uint8_t *u = used + (uint64_t)dvals[e] * DD + (uint32_t)dd;
  if (!*u) *u = 1;  // millions of edges share a few thousand keys: read first, the stores all hit the same lines
}
// key_idx == nullptr: the whole table (n_all entries), else the *n_keys listed entries
__global__ void k_trans_table(const uint32_t *__restrict__ key_idx, const uint64_t *__restrict__ n_keys, uint64_t n_all, uint32_t DD,
                              const double *__restrict__ lg, double lamb, double beta, double thr,
                              double *__restrict__ p0_lut, double *__restrict__ eK_lut) {
  const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (key_idx ? *n_keys : n_all)) return;
  const uint32_t id = key_idx ? key_idx[t] : (uint32_t)t;
  const double delta = ((double)(id % DD) * 86400.0) / 31556952.0;  // == |t_i - t_j| / SECONDS_IN_YEAR
  trans_eval((int64_t)(id / DD), delta, lg, lamb, beta, thr, &p0_lut[id], &eK_lut[id]);
}
__global__ void k_trans_gather(const uint64_t *__restrict__ keys, const uint32_t *__restrict__ dvals, uint64_t E,
                               const uint64_t *__restrict__ E_dev, const int32_t *__restrict__ days, uint32_t DD,
                               const double *__restrict__ p0_lut, const double *__restrict__ eK_lut, double *__restrict__ p0,
                               double *__restrict__ eK, double *__restrict__ dt) {
  const uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= (E_dev ? *E_dev : E)) return;
  const uint64_t k = keys[e];
  const int32_t dd = abs(days[k >> 32] - days[k & 0xFFFFFFFFull]);
  const uint64_t id = (uint64_t)dvals[e] * DD + (uint32_t)dd;
  p0[e] = p0_lut[id];
  eK[e] = eK_lut[id];
  dt[e] = ((double)dd * 86400.0) / 31556952.0;
}

}  // namespace tracs
#include "sweep_tc3.inl"
namespace tracs {

// One launch of the tile sweep over a.n_tiles tiles and a.Wp words: tensor-core kernel when the masks
// allow its identity (no 2-/3-base codes at variable sites), LOP3/POPC kernel otherwise.
// `has_n`: some variable site of some sample is N (ingest flag): the tensor-core kernel then needs its fourth plane.
// `dense`: the dense-output instantiations (k_sweep<true>, k_sweep_tc3<NP, true>) with a.dense set.
static void launch_tile_sweep(const SweepArgs &a_in, bool use_tc, cudaStream_t st, bool has_n, bool dense) {
  SweepArgs a = a_in;
  // the opt-in is per device (context): set on every call, it is a cheap driver call
  TRACS_CK(cudaFuncSetAttribute(k_sweep<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SWEEP_SMEM));
  TRACS_CK(cudaFuncSetAttribute(k_sweep<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SWEEP_SMEM));
  int dev = 0, n_sm = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev);
  if (a.n_tiles == 0) return;
  // which kernel ran: 0 = k_sweep, else 30 + operand planes executed (33/34 = k_sweep_tc3<3|4>)
  g_stats.tc_sweep = use_tc ? 30.0f + (has_n ? 4.0f : 3.0f) : 0.0f;
  if (use_tc) {
    DevBuf<uint32_t> ncnt;
    a.tc_ncnt = nullptr;
    if (has_n) {
      ncnt.alloc(a.Npad);
      k_tc_ncount<<<(a.Npad + 255) / 256, 256, 0, st>>>(a.planes, a.Npad, a.Wp, ncnt.p);
      g_stats.kernel_launches++;
      a.tc_ncnt = ncnt.p;
    }
    // 128 x 512 super-tiles: up to four consecutive tiles of a row-block share one expansion of the row panel
    TRACS_CK(cudaFuncSetAttribute(k_sweep_tc3<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Tc3Geom<3>::SMEM));
    TRACS_CK(cudaFuncSetAttribute(k_sweep_tc3<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Tc3Geom<4>::SMEM));
    TRACS_CK(cudaFuncSetAttribute((k_sweep_tc3<3, true>), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Tc3Geom<3>::SMEM));
    TRACS_CK(cudaFuncSetAttribute((k_sweep_tc3<4, true>), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Tc3Geom<4>::SMEM));
    std::vector<uint32_t> h_prefix(a.n_rb + 1), sprefix(a.n_rb + 1, 0);
    TRACS_CK(cudaMemcpyAsync(h_prefix.data(), a.tile_prefix, (a.n_rb + 1) * 4, cudaMemcpyDeviceToHost, st));
    TRACS_CK(cudaStreamSynchronize(st));
    for (uint32_t k = 0; k < a.n_rb; ++k) sprefix[k + 1] = sprefix[k] + (h_prefix[k + 1] - h_prefix[k] + 3) / 4;
    const uint32_t n_stiles = sprefix[a.n_rb];
    DevBuf<uint32_t> d_sprefix(a.n_rb + 1);
    DevBuf<uint2> d_stiles(std::max<uint32_t>(1, n_stiles));
    TRACS_CK(cudaMemcpyAsync(d_sprefix.p, sprefix.data(), (a.n_rb + 1) * 4, cudaMemcpyHostToDevice, st));
    k_stile_table<<<(n_stiles + 255) / 256, 256, 0, st>>>(a.rb_list, d_sprefix.p, a.n_rb, a.cb_min, a.Npad / TILE, n_stiles, d_stiles.p);
    g_stats.kernel_launches++;
    const unsigned grid = (unsigned)std::min<uint64_t>(n_stiles, (uint64_t)n_sm);
    const char *dbg_env = getenv("TRACS_TC3_DBG");  // timing experiments (profiles/r2_tc.md); never set in production
    const uint32_t dbg = dbg_env ? (uint32_t)atoi(dbg_env) : 0u;
    if (dense && has_n) k_sweep_tc3<4, true><<<grid, TC3_THREADS, Tc3Geom<4>::SMEM, st>>>(a, d_stiles.p, n_stiles, dbg);
    else if (dense) k_sweep_tc3<3, true><<<grid, TC3_THREADS, Tc3Geom<3>::SMEM, st>>>(a, d_stiles.p, n_stiles, dbg);
    else if (has_n) k_sweep_tc3<4><<<grid, TC3_THREADS, Tc3Geom<4>::SMEM, st>>>(a, d_stiles.p, n_stiles, dbg);
    else k_sweep_tc3<3><<<grid, TC3_THREADS, Tc3Geom<3>::SMEM, st>>>(a, d_stiles.p, n_stiles, dbg);
    TRACS_CK(cudaStreamSynchronize(st));  // sprefix (host) and the tables go out of scope
  } else {
    int occ = 1;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_sweep<false>, SWEEP_THREADS, SWEEP_SMEM);
    const unsigned grid = (unsigned)std::min<uint64_t>(a.n_tiles, (uint64_t)n_sm * std::max(1, occ));
    if (dense) k_sweep<true><<<grid, SWEEP_THREADS, SWEEP_SMEM, st>>>(a);
    else k_sweep<false><<<grid, SWEEP_THREADS, SWEEP_SMEM, st>>>(a);
  }
  g_stats.kernel_launches++;
  TRACS_CK(cudaGetLastError());
}

// ------------------------------------------------------------------------------------------
// host orchestration
// ------------------------------------------------------------------------------------------


// Everything the ingest stage leaves in device memory for one alignment (or one site slab of it).
struct Ingested {
  uint64_t n = 0, L = 0;
  uint64_t npitch = 0, spitch = 0;     // N-plane row pitch (words) / summary row pitch (bytes)
  uint64_t V = 0, W = 0;               // variable sites, 32-site words
  uint32_t Wp = KC, Npad = 0;          // padded words / samples
  DevBuf<uint32_t> nplane, ncount, site_idx;
  DevBuf<uint8_t> nsum;
  DevBuf<uint4> planes, planesT;
  bool partial_ambiguity = false;      // some variable site carries a 2- or 3-base IUPAC code
  uint64_t n_total = 0;                // N / gap / unknown sites over all samples (sum of ncount)
  bool has_n_var = true;               // some sample is N at some variable site (the tensor-core sweep needs its N plane)
  // Sparse N (decided on the first chunk of the early-extraction ingest): only the 256-site groups of the N bit-plane
  // that hold an N were stored; everything else in the buffer is undefined and never read (summary-guided consumers).
  bool nplane_sparse = false;
};

__global__ void k_sum_u32(const uint32_t *__restrict__ v, uint64_t n, unsigned long long *out) {
  unsigned long long s = 0;
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) s += v[i];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xFFFFFFFFu, s, o);
  if ((threadIdx.x & 31) == 0 && s) atomicAdd(out, s);
}

// ASCII matrix (device) -> N-plane + summaries + variable-site bit-planes (K0a + K0b)
// `packed`: dev_seqs holds 4-bit masks, two sites per byte (pack4.inl), pitch in bytes
// `rows_before`: the N-plane, its summary and the N counts get that many unused (zeroed-summary) rows before sample 0,
// which g.nplane.p etc. then point at (the resident database, db.inl, packs query rows there). `keep_colmask`: receives
// the column AND of the 4-bit masks (L / 8 words).
static void ingest_device(const uint8_t *dev_seqs, uint64_t n, uint64_t L, uint64_t pitch, bool packed, bool keep_site_idx,
                          Ingested &g, cudaStream_t st, uint64_t rows_before = 0, DevBuf<uint32_t> *keep_colmask = nullptr) {
  tracs_stats_t &S = g_stats;
  if (!packed && (pitch % 32 != 0 || pitch < round_up(L, 32)))
    throw std::runtime_error("device alignment pitch must be a multiple of 32 and >= L rounded up to 32");
  if (packed && (pitch % 16 != 0 || pitch * 2 < std::max<uint64_t>(32, round_up(L, 32))))
    throw std::runtime_error("packed alignment pitch must be a multiple of 16 bytes and hold L rounded up to 32 sites");
  Timer T(st);
  g.n = n;
  g.L = L;
  // ---- K0a ---------------------------------------------------------------------------
  const uint64_t Lw = (L + 31) / 32;                       // words with sites
  const uint64_t npitch = std::max<uint64_t>(32, round_up(Lw, 32));  // N-plane row pitch in words (whole warps)
  const uint64_t spitch = round_up(npitch / 32, 4);        // summary bytes per row (uint32 granules)
  g.npitch = npitch;
  g.spitch = spitch;
  DevBuf<uint32_t> colmask(std::max<uint64_t>(1, Lw * 4));
  DevBuf<uint32_t> &nplane = g.nplane, &ncount = g.ncount;
  DevBuf<uint8_t> &nsum = g.nsum;
  // Early extraction (see k_pack_x): pack a first chunk of samples, list the sites that already vary, and let the
  // pack of all other samples store those sites' masks on the way. TRACS_INGEST=split / =early overrides the rule.
  const char *mode_env = getenv("TRACS_INGEST");
  const uint64_t n_first = PACK_SCHUNK;
  bool early = L >= (1u << 16) && n >= 4 * n_first && L < (1ull << 31);
  if (mode_env && !strcmp(mode_env, "split")) early = false;
  if (mode_env && !strcmp(mode_env, "early")) early = L > 0 && n > n_first && L < (1ull << 31);
  // The N-plane comes out of the pack pass (same pass over the bytes). On the early-extraction path the first chunk's N
  // counts tell whether N is sparse; if so, the main launch stores only the sectors that hold an N (pack_emit_n<true>).
  // TRACS_NPLANE=always / sparse overrides the density rule; TRACS_NBLOCKS=dense (tests) wants whole rows.
  const char *np_env = getenv("TRACS_NPLANE");
  const char *nb_env = getenv("TRACS_NBLOCKS");
  const bool sparse_candidate = early && !(np_env && !strcmp(np_env, "always")) && !(nb_env && !strcmp(nb_env, "dense"));
  g.nplane_sparse = false;
  nplane.alloc((rows_before + n) * npitch);
  nsum.alloc((rows_before + n) * spitch);
  ncount.alloc(rows_before + n);
  uint32_t *const np0 = nplane.p + rows_before * npitch, *const nc0 = ncount.p + rows_before;
  uint8_t *const ns0 = nsum.p + rows_before * spitch;
  const uint32_t Npad = (uint32_t)round_up(n, TILE);
  DevBuf<uint32_t> &site_idx = g.site_idx;
  T.start();
  TRACS_CK(cudaMemsetAsync(colmask.p, 0xFF, colmask.n * sizeof(uint32_t), st));
  TRACS_CK(cudaMemsetAsync(nsum.p, 0, nsum.n, st));
  TRACS_CK(cudaMemsetAsync(ncount.p, 0, ncount.n * sizeof(uint32_t), st));

  // variable-site list from the column AND: flags -> select; returns the count (synchronises the stream)
  auto select_sites = [&](DevBuf<uint32_t> &list) -> uint64_t {
    DevBuf<uint8_t> flags(round_up(L, 8));
    k_siteflags<<<(unsigned)((Lw * 4 + 255) / 256), 256, 0, st>>>(colmask.p, L, flags.p);
    list.alloc(L);
    DevBuf<uint64_t> nsel(1);
    size_t tmp_bytes = 0;
    cub::CountingInputIterator<uint32_t> cnt_it(0);
    cub::DeviceSelect::Flagged(nullptr, tmp_bytes, cnt_it, flags.p, list.p, nsel.p, (int64_t)L, st);
    DevBuf<uint8_t> tmp(tmp_bytes);
    cub::DeviceSelect::Flagged(tmp.p, tmp_bytes, cnt_it, flags.p, list.p, nsel.p, (int64_t)L, st);
    S.kernel_launches += 3;
    uint64_t cnt = 0;
    TRACS_CK(cudaMemcpyAsync(&cnt, nsel.p, sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    TRACS_CK(cudaStreamSynchronize(st));
    return cnt;
  };
  auto launch_pack = [&](uint64_t sa, uint64_t sb, const uint32_t *elist, uint32_t VE, uint8_t *X, uint64_t XP) {
    if (sb <= sa) return;
    dim3 grid((unsigned)((npitch + PACK_THREADS - 1) / PACK_THREADS), (unsigned)((sb - sa + PACK_SCHUNK - 1) / PACK_SCHUNK));
    if (packed) {
      if (VE && g.nplane_sparse) {
        TRACS_CK(cudaFuncSetAttribute((k_pack4<true, true>), cudaFuncAttributePreferredSharedMemoryCarveout, 60));
        k_pack4<true, true><<<grid, PACK_THREADS, 0, st>>>(dev_seqs, sa, sb, L, pitch, colmask.p, np0, npitch, ns0, spitch,
                                                         nc0, elist, VE, X, XP);
      } else if (VE) {
        TRACS_CK(cudaFuncSetAttribute((k_pack4<true, false>), cudaFuncAttributePreferredSharedMemoryCarveout, 60));
        k_pack4<true><<<grid, PACK_THREADS, 0, st>>>(dev_seqs, sa, sb, L, pitch, colmask.p, np0, npitch, ns0, spitch, nc0,
                                                   elist, VE, X, XP);
      } else {
        k_pack4<false><<<grid, PACK_THREADS, 0, st>>>(dev_seqs, sa, sb, L, pitch, colmask.p, np0, npitch, ns0, spitch, nc0,
                                                    nullptr, 0, nullptr, 0);
      }
    } else if (VE) {
      TRACS_CK(cudaFuncSetAttribute(k_pack_x<false>, cudaFuncAttributePreferredSharedMemoryCarveout, 60));  // 3 x 34 KB per SM (per device)
      TRACS_CK(cudaFuncSetAttribute(k_pack_x<true>, cudaFuncAttributePreferredSharedMemoryCarveout, 60));
      if (g.nplane_sparse)
        k_pack_x<true><<<grid, PACK_THREADS, 0, st>>>(dev_seqs, sa, sb, L, pitch, colmask.p, np0, npitch, ns0, spitch, nc0,
                                                    elist, VE, X, XP);
      else
        k_pack_x<false><<<grid, PACK_THREADS, 0, st>>>(dev_seqs, sa, sb, L, pitch, colmask.p, np0, npitch, ns0, spitch, nc0,
                                                     elist, VE, X, XP);
    } else {
      k_pack<<<grid, PACK_THREADS, 0, st>>>(dev_seqs, sa, sb, L, pitch, colmask.p, np0, npitch, ns0, spitch, nc0);
    }
    S.kernel_launches++;
    TRACS_CK(cudaGetLastError());
  };
  DevBuf<uint32_t> elist;
  DevBuf<uint8_t> X;
  uint64_t VE = 0, XP = 0;
  if (L == 0) {
    TRACS_CK(cudaMemsetAsync(nplane.p, 0, nplane.n * sizeof(uint32_t), st));
  } else if (!early) {
    Timer Tm(st);
    Tm.start();
    launch_pack(0, n, nullptr, 0, nullptr, 0);
    S.ms_pack_main += Tm.stop();
  } else {
    launch_pack(0, n_first, nullptr, 0, nullptr, 0);
    std::vector<uint32_t> first_cnt(sparse_candidate ? n_first : 0);
    if (sparse_candidate)  // lands with the synchronisation inside select_sites
      TRACS_CK(cudaMemcpyAsync(first_cnt.data(), nc0, n_first * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    VE = select_sites(elist);
    if (VE > L / 16) VE = 0;  // very diverse alignment: the scattered pass reads dense lines anyway
    if (VE) {
      XP = round_up(VE, 32);
      X.alloc(n * XP);
    } else {
      early = false;
    }
    if (sparse_candidate && VE) {
      // same rule as the choice between the summary-guided and the dense compared-sites kernels (pairs.inl): sparse
      // while fewer than 35 % of the 128-site blocks hold an N
      double tot = 0;
      for (uint32_t c : first_cnt) tot += c;
      const double p_n = tot / ((double)n_first * (double)L);
      g.nplane_sparse = 1.0 - pow(1.0 - std::min(1.0, p_n), 128.0) <= 0.35;
      if (np_env && !strcmp(np_env, "sparse")) g.nplane_sparse = true;
      if (g.nplane_sparse) S.sparse_nplane = 1.0f;
    }
    Timer Tm(st);
    Tm.start();
    launch_pack(n_first, n, elist.p, (uint32_t)VE, X.p, XP);
    S.ms_pack_main += Tm.stop();
    S.n_early_sites += VE;
  }
  S.ms_pack += T.stop();

  // ---- K0b: variable sites -> planes -----------------------------------------------------
  T.start();
  uint64_t V = 0;
  if (L > 0) V = select_sites(site_idx);
  const uint64_t W = (V + 31) / 32;
  const uint32_t Wp = (uint32_t)std::max<uint64_t>(KC, round_up(W, KC));
  g.V = V; g.W = W; g.Wp = Wp; g.Npad = Npad;
  S.n_variable_sites += V;
  S.n_words += Wp;
  g.planes.alloc((size_t)Wp * Npad);
  g.planesT.alloc((size_t)Wp * n);
  TRACS_CK(cudaMemsetAsync(g.planes.p, 0xFF, g.planes.n * sizeof(uint4), st));
  TRACS_CK(cudaMemsetAsync(g.planesT.p, 0xFF, g.planesT.n * sizeof(uint4), st));
  g.partial_ambiguity = false;
  if (W > 0) {
    const uint32_t schunk = 512;
    DevBuf<uint32_t> amb(1);
    TRACS_CK(cudaMemsetAsync(amb.p, 0, 4, st));
    if (!early) {
      dim3 grid((unsigned)((W + 7) / 8), (unsigned)((n + schunk - 1) / schunk));
      if (packed) k_gather<true><<<grid, 256, 0, st>>>(dev_seqs, n, pitch, site_idx.p, V, g.planes.p, Npad, g.planesT.p, Wp, schunk, amb.p);
      else k_gather<false><<<grid, 256, 0, st>>>(dev_seqs, n, pitch, site_idx.p, V, g.planes.p, Npad, g.planesT.p, Wp, schunk, amb.p);
      S.kernel_launches++;
    } else {
      // listed sites of the first chunk, late sites of every sample: the scattered pass; then bit-slice
      const uint64_t VL = V - VE;  // elist is a subset of the final list
      DevBuf<uint32_t> src(V), late(std::max<uint64_t>(1, VL));
      DevBuf<uint8_t> X2;
      const uint64_t X2P = round_up(std::max<uint64_t>(1, VL), 32);
      k_site_sources<<<(unsigned)((V + 255) / 256), 256, 0, st>>>(site_idx.p, (uint32_t)V, elist.p, (uint32_t)VE, src.p, late.p);
      auto gather_bytes = [&](uint64_t sa, uint64_t sb, const uint32_t *list, uint64_t n_list, uint8_t *dst, uint64_t dpitch) {
        const dim3 gg((unsigned)((n_list + 255) / 256), (unsigned)((sb - sa + schunk - 1) / schunk));
        if (packed) k_gather_bytes<true><<<gg, 256, 0, st>>>(dev_seqs, sa, sb, pitch, list, (uint32_t)n_list, dst, dpitch, schunk);
        else k_gather_bytes<false><<<gg, 256, 0, st>>>(dev_seqs, sa, sb, pitch, list, (uint32_t)n_list, dst, dpitch, schunk);
      };
      gather_bytes(0, n_first, elist.p, VE, X.p, XP);
      S.kernel_launches += 2;
      if (VL) {
        X2.alloc(n * X2P);
        gather_bytes(0, n, late.p, VL, X2.p, X2P);
        S.kernel_launches++;
      }
      dim3 grid((unsigned)((W + 15) / 16), (unsigned)((n + schunk - 1) / schunk));
      k_slice<<<grid, 256, 0, st>>>(X.p, XP, X2.p, X2P, src.p, V, n, g.planes.p, Npad, g.planesT.p, Wp, schunk, amb.p);
      S.kernel_launches++;
    }
    TRACS_CK(cudaGetLastError());
    DevBuf<unsigned long long> ntot(1);
    TRACS_CK(cudaMemsetAsync(ntot.p, 0, 8, st));
    k_sum_u32<<<64, 256, 0, st>>>(nc0, n, ntot.p);
    S.kernel_launches++;
    uint32_t h_amb = 0;
    unsigned long long h_ntot = 0;
    TRACS_CK(cudaMemcpyAsync(&h_amb, amb.p, 4, cudaMemcpyDeviceToHost, st));
    TRACS_CK(cudaMemcpyAsync(&h_ntot, ntot.p, 8, cudaMemcpyDeviceToHost, st));
    TRACS_CK(cudaStreamSynchronize(st));
    g.partial_ambiguity = (h_amb & 1u) != 0;
    g.has_n_var = (h_amb & 2u) != 0;
    g.n_total = h_ntot;
  }
  S.ms_compact += T.stop();
  if (!keep_site_idx) site_idx.release();
  if (keep_colmask) {
    std::swap(keep_colmask->p, colmask.p);
    std::swap(keep_colmask->n, colmask.n);
  }
}

// Fused transmission likelihood (K3) for a sorted device edge list: dense table over (d, day difference).
struct TransLut {
  static constexpr uint64_t EAGER_MAX = 16384;
  bool on = false, eager = false;
  cudaEvent_t ready = nullptr;
  uint32_t DD = 0;
  uint64_t lut_size = 0;
  double lamb = 0, beta = 0, thr = 0;
  DevBuf<int32_t> d_days;
  DevBuf<double> d_lg, p0_lut, eK_lut;
  DevBuf<uint8_t> used, sel_tmp;
  DevBuf<uint32_t> key_idx;
  DevBuf<uint64_t> n_keys;
  size_t sel_tmp_bytes = 0;
  // d_top: distances are < d_top. Returns false (table too large / not requested): the caller falls back to the
  // unique-key path on the host side (trans_dist_device).
  bool setup(const tracs_opts_t &o, uint64_t n, uint64_t d_top, cudaStream_t st) {
    if (!(o.want_trans && o.days) || o.dist < 0) return false;
    int32_t dmin = o.days[0], dmaxday = o.days[0];
    for (uint64_t s = 0; s < n; ++s) {
      dmin = std::min(dmin, o.days[s]);
      dmaxday = std::max(dmaxday, o.days[s]);
    }
    const uint64_t dd_span = (uint64_t)((int64_t)dmaxday - (int64_t)dmin) + 1;
    if (dd_span * d_top > (1ull << 24)) return false;
    on = true;
    DD = (uint32_t)dd_span;
    lut_size = dd_span * d_top;
    lamb = o.lamb; beta = o.beta; thr = o.threshold_Ek;
    d_days.alloc(n);
    TRACS_CK(cudaMemcpyAsync(d_days.p, o.days, n * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    const size_t nlg = (size_t)d_top + 10000 + 8;
    const auto lg_keep = lgamma_table(nlg);
    d_lg.alloc(nlg);
    TRACS_CK(cudaMemcpyAsync(d_lg.p, lg_keep->data(), nlg * 8, cudaMemcpyHostToDevice, st));
    p0_lut.alloc(lut_size); eK_lut.alloc(lut_size);
    if (lut_size <= EAGER_MAX) {
      // small table (C2 / C3: 21 distances x 180 day differences): every entry is computed right away on the auxiliary
      // stream, under the ingest, instead of mark -> compact -> table behind the last kernel of the call
      eager = true;
      cudaStream_t aux = aux_stream();
      if (!ready) TRACS_CK(cudaEventCreateWithFlags(&ready, cudaEventDisableTiming));
      TRACS_CK(cudaEventRecord(ready, st));  // the two uploads above
      TRACS_CK(cudaStreamWaitEvent(aux, ready, 0));
      k_trans_table<<<(unsigned)((lut_size + 63) / 64), 64, 0, aux>>>(nullptr, nullptr, lut_size, DD, d_lg.p, lamb, beta, thr, p0_lut.p,
                                                                   eK_lut.p);
      g_stats.kernel_launches++;
      TRACS_CK(cudaGetLastError());
      TRACS_CK(cudaEventRecord(ready, aux));
      return true;
    }
    used.alloc(lut_size); key_idx.alloc(lut_size); n_keys.alloc(1);
    cub::CountingInputIterator<uint32_t> cnt_it(0);
    cub::DeviceSelect::Flagged(nullptr, sel_tmp_bytes, cnt_it, used.p, key_idx.p, n_keys.p, (int64_t)lut_size, st);
    sel_tmp.alloc(sel_tmp_bytes);
    return true;
  }
  // keys (i << 32 | j) and distances of E edges -> log p0, E[K], date difference (years), all device arrays.
  // E_dev != nullptr: the count is read on the device and E is only an upper bound (no host round trip before this).
  void apply(const uint64_t *keys, const uint32_t *dvals, uint64_t E, double *p0, double *eK, double *dt, cudaStream_t st,
             const uint64_t *E_dev = nullptr) {
    if (E == 0) return;
    if (eager) {
      TRACS_CK(cudaStreamWaitEvent(st, ready, 0));
    } else {
      TRACS_CK(cudaMemsetAsync(used.p, 0, lut_size, st));
      k_trans_mark<<<(unsigned)((E + 255) / 256), 256, 0, st>>>(keys, dvals, E, E_dev, d_days.p, DD, used.p);
      cub::CountingInputIterator<uint32_t> cnt_it(0);
      cub::DeviceSelect::Flagged(sel_tmp.p, sel_tmp_bytes, cnt_it, used.p, key_idx.p, n_keys.p, (int64_t)lut_size, st);
      k_trans_table<<<(unsigned)((lut_size + 63) / 64), 64, 0, st>>>(key_idx.p, n_keys.p, 0, DD, d_lg.p, lamb, beta, thr, p0_lut.p, eK_lut.p);
      g_stats.kernel_launches += 4;
    }
    k_trans_gather<<<(unsigned)((E + 255) / 256), 256, 0, st>>>(keys, dvals, E, E_dev, d_days.p, DD, p0_lut.p, eK_lut.p, p0, eK, dt);
    g_stats.kernel_launches += 1;
    TRACS_CK(cudaGetLastError());
  }
  ~TransLut() {
    if (eager) cudaStreamSynchronize(aux_stream());  // the table kernel must not outlive the buffers it writes
    if (ready) cudaEventDestroy(ready);
  }
};

// which row-blocks a shard sweeps, and how many pairs each holds
struct TilePlan {
  uint32_t n_cb = 0, cb_min = 0;
  std::vector<uint32_t> my_rb;
  std::vector<uint64_t> rb_pairs;
};
static TilePlan plan_tiles(uint64_t n, uint64_t i_end, uint64_t j_start, uint32_t Npad, int rank, int world) {
  TilePlan p;
  const uint32_t n_rb_all = (uint32_t)((i_end + TILE - 1) / TILE);
  p.n_cb = Npad / TILE;
  p.cb_min = (uint32_t)(j_start / TILE);
  if (rank >= world) throw std::runtime_error("shard_rank >= shard_world");
  // row-blocks dealt boustrophedon (0..w-1, w-1..0, ...) so every shard gets equal triangle area
  for (uint32_t rb = 0; rb < n_rb_all; ++rb) {
    if (shard_owner(rb, world) != rank || std::max(rb, p.cb_min) >= p.n_cb) continue;
    uint64_t tot = 0;
    const uint64_t r0 = (uint64_t)rb * TILE, r1 = std::min<uint64_t>(i_end, r0 + TILE);
    for (uint64_t i = r0; i < r1; ++i) {
      const uint64_t j0 = std::max<uint64_t>(j_start, i + 1);
      if (j0 < n) tot += n - j0;
    }
    p.my_rb.push_back(rb);
    p.rb_pairs.push_back(tot);
  }
  return p;
}

// Consecutive row-blocks of a plan cut into bands of at most `limit` pairs and `tile_limit` tiles (one launch each):
// my_rb[first, last).
struct Band { size_t first, last; uint64_t pairs; };
constexpr uint64_t BAND_PAIRS = 1ull << 28;  // pairs per band of a full-length sweep (the edge buffer holds every pair of one)
constexpr uint64_t BAND_TILES = 1ull << 31;  // tiles per launch (the kernels count tiles in 32 bits)
constexpr uint64_t CAND_CAP = 1ull << 26;    // prefilter candidates held at once (only a few per cent of the pairs may survive)
static std::vector<Band> make_bands(const TilePlan &plan, uint64_t limit, uint64_t tile_limit) {
  std::vector<Band> u;
  size_t b0 = 0;
  uint64_t acc = 0, tiles = 0;
  for (size_t k = 0; k < plan.my_rb.size(); ++k) {
    const uint64_t p = plan.rb_pairs[k], t = plan.n_cb - std::max(plan.my_rb[k], plan.cb_min);
    if (k > b0 && (acc + p > limit || tiles + t > tile_limit)) {
      u.push_back({b0, k, acc});
      b0 = k;
      acc = 0;
      tiles = 0;
    }
    acc += p;
    tiles += t;
  }
  if (b0 < plan.my_rb.size()) u.push_back({b0, plan.my_rb.size(), acc});
  return u;
}

// radix-sort end bit of the pair keys (i << 32 | j), i, j < n
static int key_end_bit(uint64_t n) {
  int end_bit = 32;
  while ((1ull << (end_bit - 32)) < n) end_bit++;
  return end_bit;
}

// Tensor cores unless forced off (sweep_variant 1) or inapplicable (2-/3-base codes at variable sites); sweep_variant 2
// insists on them.
static bool use_tensor_cores(const tracs_opts_t &o, const Ingested &g) {
  if (o.sweep_variant == 2 && g.partial_ambiguity)
    throw std::runtime_error("tensor-core sweep requested but the alignment has 2-/3-base IUPAC codes at variable sites");
  return o.sweep_variant != 1 && !g.partial_ambiguity;
}

// The fields every tile sweep of an ingested alignment shares; the caller adds the output (edge list or dense matrix),
// sweep_band() the tile list.
static SweepArgs sweep_args(const Ingested &g, uint64_t i_end, uint64_t j_start, int32_t dist) {
  SweepArgs a{};
  a.planes = g.planes.p; a.Wp = g.Wp; a.Npad = g.Npad; a.n = (uint32_t)g.n; a.i_end = (uint32_t)i_end;
  a.j_start = (uint32_t)j_start; a.dist = dist; a.one = 1;
  return a;
}

// One launch of the tile sweep over the row-blocks plan.my_rb[b.first, b.last): the tile list (prefix, copies,
// k_tile_table), the launch on `a` (planes, window, range and output already set) and its stats. Returns the tile count.
static uint32_t sweep_band(const TilePlan &plan, const Band &b, SweepArgs a, bool use_tc, bool has_n, bool dense, cudaStream_t st) {
  tracs_stats_t &S = g_stats;
  const std::vector<uint32_t> rbs(plan.my_rb.begin() + b.first, plan.my_rb.begin() + b.last);
  std::vector<uint32_t> prefix(rbs.size() + 1, 0);
  for (size_t k = 0; k < rbs.size(); ++k) prefix[k + 1] = prefix[k] + (plan.n_cb - std::max(rbs[k], plan.cb_min));
  const uint32_t n_tiles = prefix.back();
  DevBuf<uint32_t> d_rb(std::max<size_t>(1, rbs.size())), d_prefix(prefix.size());
  DevBuf<uint2> d_table(std::max<uint32_t>(1, n_tiles));
  TRACS_CK(cudaMemcpyAsync(d_rb.p, rbs.data(), rbs.size() * 4, cudaMemcpyHostToDevice, st));
  TRACS_CK(cudaMemcpyAsync(d_prefix.p, prefix.data(), prefix.size() * 4, cudaMemcpyHostToDevice, st));
  a.rb_list = d_rb.p; a.tile_prefix = d_prefix.p; a.n_rb = (uint32_t)rbs.size(); a.n_tiles = n_tiles; a.cb_min = plan.cb_min;
  a.tile_table = d_table.p;
  if (n_tiles) {
    k_tile_table<<<(n_tiles + 255) / 256, 256, 0, st>>>(d_rb.p, d_prefix.p, a.n_rb, plan.cb_min, n_tiles, d_table.p);
    S.kernel_launches++;
  }
  Timer T(st);
  T.start();
  launch_tile_sweep(a, use_tc, st, has_n, dense);
  S.ms_sweep += T.stop();
  S.n_tiles += n_tiles;
  return n_tiles;
}

// Edge (or candidate) list of a thresholded sweep: the tile kernels append (key, distance) pairs through `counter`; the
// second pair of buffers receives sorts and compactions.
struct EdgeList {
  uint64_t cap;
  DevBuf<uint64_t> keys, keys2;
  DevBuf<uint32_t> dv, dv2;
  DevBuf<unsigned long long> counter;
  explicit EdgeList(uint64_t c) : cap(c), keys(c), keys2(c), dv(c), dv2(c), counter(1) {}
  void output_to(SweepArgs &a) const { a.counter = counter.p; a.keys = keys.p; a.dvals = dv.p; a.cap = cap; }
  void reset(cudaStream_t st) { TRACS_CK(cudaMemsetAsync(counter.p, 0, sizeof(unsigned long long), st)); }
  uint64_t count(cudaStream_t st) const {
    unsigned long long c = 0;
    TRACS_CK(cudaMemcpyAsync(&c, counter.p, sizeof c, cudaMemcpyDeviceToHost, st));
    TRACS_CK(cudaStreamSynchronize(st));
    return c;
  }
  void swap() {  // (keys2, dv2) become the current list
    std::swap(keys.p, keys2.p);
    std::swap(dv.p, dv2.p);
  }
};

// Filter-and-refine, first step: tile-sweep only the first words of every pair of the plan into `c`; d is monotone in
// the number of sites, so a pair whose partial distance already exceeds a.dist is decided. Windows of 4, 8, 16 and 64
// words (at most the ingested words) are tried in turn until the candidates fit the list and are <= 4 % of `pairs` --
// per-pair refinement is then cheaper than tiles -- or the widest window has been swept. A narrow window (< 16 words)
// lets a few unrelated pairs through; left in, they would bridge clusters in the candidate graph, so its candidates are
// trimmed over the next words (k_cand_trim). Short windows run on the LOP3/POPC kernel (the tensor-core kernel pays its
// per-tile pipeline fill and its TMEM epilogue on every 128 x 128 tile: measured equal at 16 words, slower below), wider
// ones on the tensor cores when `tc_ok`. The candidates are left unsorted in (c.keys, c.dv).
struct Prefilter {
  uint64_t n_cand;
  uint32_t words;   // window that produced the candidates
  bool selective;   // they fit the list and are <= 4 % of the pairs
};
static Prefilter prefilter(const Ingested &g, const TilePlan &plan, uint64_t pairs, SweepArgs a, bool tc_ok, EdgeList &c,
                           cudaStream_t st) {
  tracs_stats_t &S = g_stats;
  const std::vector<Band> bands = make_bands(plan, UINT64_MAX, BAND_TILES);
  c.output_to(a);
  for (uint32_t pw = first_window(a.dist);; pw = next_window(pw)) {
    const uint32_t words = std::min(pw, g.Wp);
    a.Wp = words;
    c.reset(st);
    for (const Band &b : bands) sweep_band(plan, b, a, tc_ok && words >= TC_MIN_WORDS, g.has_n_var, false, st);
    S.swept_wordpairs += pairs * words;
    uint64_t n_cand = c.count(st);
    const bool selective = n_cand <= c.cap && n_cand * 25 <= pairs;
    if (selective && n_cand && words < 16 && g.Wp > words) {
      Timer T(st);
      T.start();
      const uint32_t extra = std::min<uint32_t>(g.Wp - words, 32 - words);
      DevBuf<uint8_t> flags(n_cand);
      DevBuf<uint64_t> n_sel(1);
      k_cand_trim<<<(unsigned)((n_cand + 255) / 256), 256, 0, st>>>(c.keys.p, c.dv.p, n_cand, g.planesT.p, g.Wp, words, extra, a.dist,
                                                                     flags.p);
      size_t tb = 0;
      cub::DeviceSelect::Flagged(nullptr, tb, c.keys.p, flags.p, c.keys2.p, n_sel.p, (int64_t)n_cand, st);
      DevBuf<uint8_t> tmp(tb);
      cub::DeviceSelect::Flagged(tmp.p, tb, c.keys.p, flags.p, c.keys2.p, n_sel.p, (int64_t)n_cand, st);
      cub::DeviceSelect::Flagged(tmp.p, tb, c.dv.p, flags.p, c.dv2.p, n_sel.p, (int64_t)n_cand, st);
      TRACS_CK(cudaMemcpyAsync(&n_cand, n_sel.p, 8, cudaMemcpyDeviceToHost, st));
      TRACS_CK(cudaStreamSynchronize(st));
      c.swap();
      S.kernel_launches += 5;
      S.ms_refine += T.stop();
    }
    if (selective || words >= std::min(PREFILTER_WORDS, g.Wp)) {
      S.n_candidates += n_cand;
      return {n_cand, words, selective};
    }
  }
}

// Where E new rows of an edge table start in each of its columns; null: the column is not filled.
struct HostColumns {
  uint64_t *rows, *cols, *dist, *ncomp, *filt;
  double *p0_log, *eK, *datediff;
};
// Appends E rows to the columns of `out` that the call fills (rows, cols, dist always; compared sites, filtered distance and
// the likelihood columns when asked for) and returns where they start.
static HostColumns append_rows(HostEdges &out, uint64_t E, bool ncomp, bool filt, bool trans) {
  const size_t old = out.rows.size();
  out.rows.resize(old + E); out.cols.resize(old + E); out.dist.resize(old + E);
  if (ncomp) out.ncomp.resize(old + E);
  if (filt) out.filt.resize(old + E);
  if (trans) { out.p0_log.resize(old + E); out.eK.resize(old + E); out.datediff.resize(old + E); }
  return {out.rows.data() + old, out.cols.data() + old, out.dist.data() + old, ncomp ? out.ncomp.data() + old : nullptr,
          filt ? out.filt.data() + old : nullptr, trans ? out.p0_log.data() + old : nullptr, trans ? out.eK.data() + old : nullptr,
          trans ? out.datediff.data() + old : nullptr};
}
// Enqueues the device -> host copies of E rows of every column that `src` (device) gives into the same column of `dst`.
static void copy_columns(const HostColumns &dst, const HostColumns &src, uint64_t E, cudaStream_t st) {
  auto copy = [&](void *d, const void *s) {
    if (!s) return;
    TRACS_CK(cudaMemcpyAsync(d, s, E * 8, cudaMemcpyDeviceToHost, st));
    g_stats.d2h_bytes += E * 8;
  };
  copy(dst.rows, src.rows); copy(dst.cols, src.cols); copy(dst.dist, src.dist); copy(dst.ncomp, src.ncomp); copy(dst.filt, src.filt);
  copy(dst.p0_log, src.p0_log); copy(dst.eK, src.eK); copy(dst.datediff, src.datediff);
}

// Two events that order the auxiliary stream against the main one, per host thread and device (an event belongs to the
// device it was created on, and a thread may drive several).
struct AuxEvents { cudaEvent_t a, b; };
static AuxEvents aux_events() {
  static thread_local AuxEvents ev[64] = {};
  int dev = 0;
  TRACS_CK(cudaGetDevice(&dev));
  AuxEvents &e = ev[dev & 63];
  if (!e.a) {
    TRACS_CK(cudaEventCreateWithFlags(&e.a, cudaEventDisableTiming));
    TRACS_CK(cudaEventCreateWithFlags(&e.b, cudaEventDisableTiming));
  }
  return e;
}

}  // namespace tracs
#include "pairs.inl"
namespace tracs {

static void eval_finish_overlapped(const Ingested &g, const uint64_t *keys, uint64_t n_keys, uint32_t *d, uint32_t *u, uint64_t n,
                                   uint64_t L_total, const tracs_opts_t &o, TransLut *lut, HostEdges &out, cudaStream_t st);

// Recombination filter (K4) of E sorted edges: filtered distances into filt32, and widened to the output type into filt64.
static void recomb_filter(const Ingested &g, const uint64_t *keys, const uint32_t *dvals, uint64_t E, DevBuf<uint32_t> &filt32,
                          DevBuf<uint64_t> &filt64, cudaStream_t st) {
  tracs_stats_t &S = g_stats;
  Timer T(st);
  T.start();
  filt32.alloc(E);
  filt64.alloc(E);
  DevBuf<uint64_t> offs(E + 1);
  DevBuf<uint8_t> stmp;
  size_t sb = 0;
  TRACS_CK(cudaMemsetAsync(offs.p, 0, sizeof(uint64_t), st));
  // the scan accumulates in the INPUT type: widen on the fly so offsets above 2^32 do not wrap
  cub::TransformInputIterator<uint64_t, WidenU32, const uint32_t *> d_in64(dvals, WidenU32());
  cub::DeviceScan::InclusiveSum(nullptr, sb, d_in64, offs.p + 1, (int64_t)E, st);
  stmp.alloc(sb);
  cub::DeviceScan::InclusiveSum(stmp.p, sb, d_in64, offs.p + 1, (int64_t)E, st);
  uint64_t total = 0;
  TRACS_CK(cudaMemcpyAsync(&total, offs.p + E, 8, cudaMemcpyDeviceToHost, st));
  TRACS_CK(cudaStreamSynchronize(st));
  const uint64_t LIMIT = 1ull << 29;  // SNP positions held at once (2 GB)
  std::vector<uint64_t> cuts{0};
  if (total > LIMIT) {
    std::vector<uint64_t> h(E + 1);
    TRACS_CK(cudaMemcpyAsync(h.data(), offs.p, (E + 1) * 8, cudaMemcpyDeviceToHost, st));
    TRACS_CK(cudaStreamSynchronize(st));
    uint64_t start = 0;
    for (uint64_t e = 0; e < E; ++e) {
      if (h[e + 1] - h[start] > LIMIT && e > start) {
        cuts.push_back(e);
        start = e;
      }
      if (h[e + 1] - h[e] > LIMIT) throw std::runtime_error("filter: a single pair has too many SNPs for the position scratch");
    }
    cuts.push_back(E);
    // per-cut sizes
    uint64_t mxn = 0;
    for (size_t c = 0; c + 1 < cuts.size(); ++c) mxn = std::max(mxn, h[cuts[c + 1]] - h[cuts[c]]);
    total = mxn;
  } else {
    cuts.push_back(E);
  }
  DevBuf<uint32_t> pos(std::max<uint64_t>(1, total));
  const size_t nlg = 10000 + 16;
  const auto lgh_keep = lgamma_table(nlg);
  const std::vector<double> &lgh = *lgh_keep;
  DevBuf<double> lg_f(nlg);
  TRACS_CK(cudaMemcpyAsync(lg_f.p, lgh.data(), nlg * 8, cudaMemcpyHostToDevice, st));
  for (size_t c = 0; c + 1 < cuts.size(); ++c) {
    const uint64_t e0 = cuts[c], e1 = cuts[c + 1];
    if (e1 == e0) continue;
    uint64_t base = 0;
    TRACS_CK(cudaMemcpyAsync(&base, offs.p + e0, 8, cudaMemcpyDeviceToHost, st));
    TRACS_CK(cudaStreamSynchronize(st));
    const unsigned grid = (unsigned)(((e1 - e0) * 32 + 255) / 256);
    k_snp_positions<<<grid, 256, 0, st>>>(keys, e0, e1, g.planesT.p, g.Wp, g.site_idx.p, g.V, offs.p, base, pos.p);
    k_filter_recomb<<<grid, 256, 0, st>>>(dvals, e0, e1, offs.p, base, pos.p, g.L, lg_f.p, filt32.p);
    S.kernel_launches += 2;
    TRACS_CK(cudaGetLastError());
  }
  k_widen<<<(unsigned)((E + 255) / 256), 256, 0, st>>>(filt32.p, E, filt64.p);
  S.kernel_launches += 3;
  S.ms_filter += T.stop();
}

// Sorted-edge tail of a thresholded sweep: the E edges in (c.keys, c.dv) are sorted and expanded into columns, given
// their filtered distance, likelihood and compared sites, and appended to `out`. The columns leave for the host on the
// auxiliary stream as soon as they exist, under the compared-sites kernel: (rows, cols, dist[, filt]) right away, the
// likelihood columns after the transmission kernels (which therefore run BEFORE k_ncomp), the compared-sites column last
// on the main stream. `keep_on_device`: also leave a packed copy of the columns on the device (tracs_edges_t.dev_packed).
static void emit_sorted_edges(const Ingested &g, EdgeList &c, uint64_t E, int end_bit, const tracs_opts_t &o, TransLut *lut,
                              bool keep_on_device, HostEdges &out, cudaStream_t st) {
  tracs_stats_t &S = g_stats;
  if (E == 0) return;
  const bool want_n = o.want_ncomp != 0;
  Timer T(st);
  T.start();
  size_t sort_bytes = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, sort_bytes, c.keys.p, c.keys2.p, c.dv.p, c.dv2.p, (int64_t)E, 0, end_bit, st);
  DevBuf<uint8_t> sort_tmp(sort_bytes);
  cub::DeviceRadixSort::SortPairs(sort_tmp.p, sort_bytes, c.keys.p, c.keys2.p, c.dv.p, c.dv2.p, (int64_t)E, 0, end_bit, st);
  S.kernel_launches += 2 + (end_bit + 7) / 8;  // histogram + scan + one onesweep pass per 8 key bits
  const uint64_t *keys = c.keys2.p;
  const uint32_t *dv = c.dv2.p;
  DevBuf<uint64_t> d_rows(E), d_cols(E), d_dist(E), d_nc;
  k_expand<<<(unsigned)((E + 255) / 256), 256, 0, st>>>(keys, dv, E, d_rows.p, d_cols.p, d_dist.p);
  S.kernel_launches++;
  S.ms_sort += T.stop();

  DevBuf<uint32_t> d_filt32;
  DevBuf<uint64_t> d_filt64;
  if (o.filter) recomb_filter(g, keys, dv, E, d_filt32, d_filt64, st);
  const cudaStream_t aux = aux_stream();
  const AuxEvents ev = aux_events();
  const HostColumns dst = append_rows(out, E, want_n, o.filter != 0, lut != nullptr);
  TRACS_CK(cudaEventRecord(ev.a, st));
  TRACS_CK(cudaStreamWaitEvent(aux, ev.a, 0));
  copy_columns(dst, {d_rows.p, d_cols.p, d_dist.p, nullptr, d_filt64.p, nullptr, nullptr, nullptr}, E, aux);
  DevBuf<double> d_p0, d_eK, d_dt;
  if (lut) {
    T.start();
    d_p0.alloc(E); d_eK.alloc(E); d_dt.alloc(E);
    // with the filter on, the likelihood is fed the filtered distance (tracs/distance.py:182-192)
    lut->apply(keys, o.filter ? d_filt32.p : dv, E, d_p0.p, d_eK.p, d_dt.p, st);
    S.ms_trans += T.stop();
    TRACS_CK(cudaEventRecord(ev.b, st));
    TRACS_CK(cudaStreamWaitEvent(aux, ev.b, 0));
    copy_columns(dst, {nullptr, nullptr, nullptr, nullptr, nullptr, d_p0.p, d_eK.p, d_dt.p}, E, aux);
  }
  if (want_n) {
    T.start();
    d_nc.alloc(E);
    const uint32_t *order = nullptr;
    DevBuf<uint32_t> rep, ok1, ok2, ov1, ov2;
    DevBuf<uint8_t> otmp;
    if (E >= 4096 && E < (1ull << 32)) {
      rep.alloc(g.n); ok1.alloc(E); ok2.alloc(E); ov1.alloc(E); ov2.alloc(E);
      k_rep_init<<<(unsigned)((g.n + 255) / 256), 256, 0, st>>>(rep.p, (uint32_t)g.n);
      k_rep_min<<<(unsigned)((E + 255) / 256), 256, 0, st>>>(keys, E, rep.p);
      k_rep_keys<<<(unsigned)((E + 255) / 256), 256, 0, st>>>(keys, E, rep.p, ok1.p, ov1.p);
      size_t ob = 0;
      cub::DeviceRadixSort::SortPairs(nullptr, ob, ok1.p, ok2.p, ov1.p, ov2.p, (int64_t)E, 0, end_bit - 32, st);
      otmp.alloc(ob);
      cub::DeviceRadixSort::SortPairs(otmp.p, ob, ok1.p, ok2.p, ov1.p, ov2.p, (int64_t)E, 0, end_bit - 32, st);
      S.kernel_launches += 5 + (end_bit - 32 + 7) / 8;
      order = ov2.p;
    }
    k_ncomp<<<(unsigned)((E * 32 + 255) / 256), 256, 0, st>>>(keys, E, g.nplane.p, g.npitch, g.nsum.p, g.spitch, g.ncount.p, g.L, order,
                                                            d_nc.p);
    S.kernel_launches++;
    TRACS_CK(cudaGetLastError());
    S.ms_ncomp += T.stop();
  }
  if (keep_on_device) {
    void *dp = nullptr;
    TRACS_CK(cudaMalloc(&dp, std::max<size_t>(32, 32 * E)));
    out.dev_packed = dp;
    out.dev_packed_bytes = 32 * E;
    k_pack_edges<<<(unsigned)((E + 255) / 256), 256, 0, st>>>(keys, dv, want_n ? d_nc.p : nullptr, lut ? d_p0.p : nullptr,
                                                             lut ? d_eK.p : nullptr, E, (uint8_t *)dp);
    S.kernel_launches++;
  }
  T.start();
  if (want_n) copy_columns(dst, {nullptr, nullptr, nullptr, d_nc.p, nullptr, nullptr, nullptr, nullptr}, E, st);
  TRACS_CK(cudaStreamSynchronize(st));
  TRACS_CK(cudaStreamSynchronize(aux));
  S.ms_d2h += T.stop();
  S.n_edges += E;
}

// Filter-and-refine over all of the plan's row-blocks (prefilter()), then every candidate is finished over the full
// length: per component block (pairs.inl) with threshold, compared sites, likelihood and the copies to the host in one
// go (eval_finish_overlapped), or -- filter=True, whose recombination filter needs the sorted edges -- per pair
// (k_refine) followed by the sorted-edge tail. Returns false, with nothing appended, when the prefilter is not selective.
static bool sweep_prefiltered(const Ingested &g, const TilePlan &plan, uint64_t pairs, const SweepArgs &a, bool tc_ok, int end_bit,
                              const tracs_opts_t &o, TransLut *lut, HostEdges &out, cudaStream_t st) {
  tracs_stats_t &S = g_stats;
  EdgeList c(std::min(std::max<uint64_t>(1, pairs), CAND_CAP));
  const Prefilter pf = prefilter(g, plan, pairs, a, tc_ok, c, st);
  if (!pf.selective) return false;
  const uint64_t n_cand = pf.n_cand;
  if (n_cand == 0) return true;
  Timer T(st);
  if (!o.filter) {
    // candidates in key order -> full-length d and |N u N| per candidate
    T.start();
    size_t kb = 0;
    cub::DeviceRadixSort::SortKeys(nullptr, kb, c.keys.p, c.keys2.p, (int64_t)n_cand, 0, end_bit, st);
    DevBuf<uint8_t> sort_tmp(kb);
    cub::DeviceRadixSort::SortKeys(sort_tmp.p, kb, c.keys.p, c.keys2.p, (int64_t)n_cand, 0, end_bit, st);
    S.kernel_launches += 2 + (end_bit + 7) / 8;
    const bool want_n = o.want_ncomp != 0;
    DevBuf<uint32_t> u_full(want_n ? n_cand : 1);
    S.ms_refine += T.stop();
    eval_finish_overlapped(g, c.keys2.p, n_cand, c.dv2.p, want_n ? u_full.p : nullptr, g.n, g.L, o, lut, out, st);
    return true;
  }
  T.start();
  c.reset(st);
  k_refine<<<(unsigned)((n_cand * 32 + 255) / 256), 256, 0, st>>>(c.keys.p, c.dv.p, n_cand, g.planesT.p, g.Wp, pf.words, o.dist,
                                                                 c.counter.p, c.keys2.p, c.dv2.p);
  S.kernel_launches++;
  TRACS_CK(cudaGetLastError());
  S.ms_refine += T.stop();
  const uint64_t E = c.count(st);
  c.swap();  // survivors now in (keys, dv) like the plain sweep leaves them
  emit_sorted_edges(g, c, E, end_bit, o, lut, o.keep_on_device != 0, out, st);
  return true;
}

// Full-length sweep in bands whose pair count fits the edge buffer (a full-length sweep may emit every pair); each band's
// edges go through the sorted-edge tail before the next band is swept. Ctrl-C is seen between bands.
static void sweep_banded(const Ingested &g, const TilePlan &plan, SweepArgs a, bool tc_ok, int end_bit, const tracs_opts_t &o,
                         TransLut *lut, HostEdges &out, cudaStream_t st) {
  tracs_stats_t &S = g_stats;
  const std::vector<Band> bands = make_bands(plan, BAND_PAIRS, BAND_TILES);
  uint64_t cap = 1;
  for (const Band &b : bands) cap = std::max(cap, b.pairs);
  EdgeList c(cap);
  c.output_to(a);
  for (const Band &b : bands) {
    check_interrupt();  // reference: PyErr_CheckSignals per row, src/pairsnp.hpp:385, 434-441
    c.reset(st);
    sweep_band(plan, b, a, tc_ok, g.has_n_var, false, st);
    S.swept_wordpairs += b.pairs * std::max<uint64_t>(g.W, 1);  // algorithmic words (padding not counted)
    const uint64_t E = c.count(st);
    if (E > cap) throw std::runtime_error("internal error: edge buffer overflow");
    emit_sorted_edges(g, c, E, end_bit, o, lut, o.keep_on_device && bands.size() == 1, out, st);
  }
}

// The pair sweep of an ingested alignment over the range of `o` (i_end already clipped to ing.n): tile plan, filter-and-refine
// or banded full-length sweep, sorted edges appended to `out`.
static void sweep_ingested(const Ingested &ing, const tracs_opts_t &o, uint64_t i_end, uint64_t j_start, HostEdges &out,
                           cudaStream_t st) {
  tracs_stats_t &S = g_stats;
  const uint64_t n = ing.n;
  const int world = std::max(1, (int)o.shard_world), rank = std::max(0, (int)o.shard_rank);
  const TilePlan plan = plan_tiles(n, i_end, j_start, ing.Npad, rank, world);
  uint64_t total_pairs = 0, total_tiles = 0;
  for (size_t k = 0; k < plan.my_rb.size(); ++k) {
    total_pairs += plan.rb_pairs[k];
    total_tiles += plan.n_cb - std::max(plan.my_rb[k], plan.cb_min);
  }
  S.n_pairs += total_pairs;
  if (plan.my_rb.empty()) return;
  const bool tc_ok = use_tensor_cores(o, ing);
  // A thresholded call first tries filter-and-refine over ALL owned row-blocks in one launch per window (the candidate
  // list is bounded: only a few per cent of the pairs may survive); otherwise, or when the prefilter is not selective,
  // the banded full-length sweep (cost of the failed attempts: 92 / Wp).
  const bool prefilter_mode = o.sweep_variant == 0 && o.dist >= 0 && (uint64_t)o.dist < (uint64_t)PREFILTER_WORDS * 32 &&
                              ing.Wp >= 4 * PREFILTER_WORDS && total_tiles < BAND_TILES;

  // ---- fused transmission likelihood set-up (device table over (d, day difference)) ----------
  TransLut lut;
  const bool fuse_trans = lut.setup(o, n, (uint64_t)std::min<int64_t>(std::max<int64_t>(o.dist, 0), (int64_t)ing.Wp * 32) + 1, st);
  if (fuse_trans) out.has_trans = true;

  const int end_bit = key_end_bit(n);
  const SweepArgs a = sweep_args(ing, i_end, j_start, o.dist);
  bool done = false;
  if (prefilter_mode) {
    check_interrupt();
    done = sweep_prefiltered(ing, plan, total_pairs, a, tc_ok, end_bit, o, fuse_trans ? &lut : nullptr, out, st);
  }
  if (!done) sweep_banded(ing, plan, a, tc_ok, end_bit, o, fuse_trans ? &lut : nullptr, out, st);
}

// Sweeps the device-resident ASCII matrix and appends edges (sorted) to `out`.
void sweep_device(const uint8_t *dev_seqs, uint64_t n, uint64_t L, uint64_t pitch, const tracs_opts_t &o,
                  HostEdges &out, cudaStream_t st) {
  tracs_stats_t &S = g_stats;
  S.n_samples = n;
  S.seq_length = L;
  const uint64_t i_end = std::min<uint64_t>(o.i_end, n);
  const uint64_t j_start = o.j_start;
  if (n == 0 || i_end == 0 || j_start >= n) return;
  if (n >= (1ull << 31)) throw std::runtime_error("too many samples");
  Timer Ttot(st);
  Ttot.start();
  Ingested ing;
  ingest_device(dev_seqs, n, L, pitch, o.packed_input != 0, o.filter != 0, ing, st);
  sweep_ingested(ing, o, i_end, j_start, out, st);
  S.ms_total = Ttot.stop();
}

// All-pairs distances of the device-resident alignment as a dense int32 matrix (tracs_distance_matrix_device): the
// ingest, the tile plan and the full-length tile sweep of sweep_device, with the dense epilogue instead of threshold,
// list, sort and compared sites. Square (o.i_end == n, o.j_start == 0): out[i][j] = out[j][i] = d(i, j), zero diagonal.
// Rectangle (o.j_start >= o.i_end): out[i][j - j_start] for i < i_end <= j_start <= j < n. Arguments validated by the caller.
void distance_matrix_device(const uint8_t *dev_seqs, uint64_t n, uint64_t L, uint64_t pitch, const tracs_opts_t &o, int32_t *out,
                            uint64_t ld, cudaStream_t st) {
  tracs_stats_t &S = g_stats;
  S.n_samples = n;
  S.seq_length = L;
  const uint64_t i_end = std::min<uint64_t>(o.i_end, n), j_start = o.j_start;
  if (n == 0 || i_end == 0 || j_start >= n) return;
  if (n >= (1ull << 31)) throw std::runtime_error("too many samples");
  const bool square = j_start == 0;
  Timer Ttot(st);
  Ttot.start();
  Ingested ing;
  ingest_device(dev_seqs, n, L, pitch, o.packed_input != 0, false, ing, st);
  const bool use_tc = use_tensor_cores(o, ing);
  const TilePlan plan = plan_tiles(n, i_end, j_start, ing.Npad, 0, 1);
  SweepArgs a = sweep_args(ing, i_end, j_start, INT32_MAX);
  a.dense = out; a.dense_ld = ld; a.dense_col0 = (uint32_t)j_start; a.dense_mirror = square ? 1u : 0u;
  // bands as on the sparse path: one launch each, Ctrl-C is seen between them
  for (const Band &b : make_bands(plan, BAND_PAIRS, BAND_TILES)) {
    check_interrupt();
    sweep_band(plan, b, a, use_tc, ing.has_n_var, true, st);
    S.n_pairs += b.pairs;
    S.swept_wordpairs += b.pairs * std::max<uint64_t>(ing.W, 1);
  }
  TRACS_CK(cudaStreamSynchronize(st));
  S.ms_total = Ttot.stop();
}

}  // namespace tracs

#include "shard.inl"
#include "db.inl"
#include "tc_peak.inl"
