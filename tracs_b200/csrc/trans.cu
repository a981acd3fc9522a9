// K3: TransCluster likelihood on the device (fp64).
//
// Restates reference src/transcluster.hpp (gtonkinhill/tracs):
//   logaddexpd :62-75   lprob_k_given_N_2 :131-170   upper_bound_E :173-188
//   expected_k :191-238 trans_dist :240-287 (memoised on (N, delta) -> here: unique-key table)
//
// One thread evaluates one unique (N, delta) key. The reference recomputes two O(N+k) log-sum-exp
// folds for every k; both are prefix sums of a series, so they are carried incrementally:
//   pois      = LSE_{i<=N}( i*ln(lamb*delta) - lg[i+1] )                      (fixed per key)
//   integral  = LSE_{i<=M}( (M-i)*ln(delta) - lg[M-i+1] - (i+1)*ln(lamb+beta) ),  M = N+k
//             = -(M+1)*ln(lamb+beta) + G_M,  G_M = LSE_{j<=M}( j*ln(delta*(lamb+beta)) - lg[j+1] )
// which is the same value up to fp64 rounding (tests hold 1e-6 relative; observed ~1e-13).
//
// delta <= 0 (same-day samples): the shipped -ffast-math reference never leaves the k loop and
// converges to the negative-binomial mean (N+1)*beta/lamb while over-reading its lgamma table
// (SURVEY F6). That closed form is returned here.
//
// Samples far apart (SURVEY F7): the reference stops the E[K] series once upper_bound_E - sum_k t_k <= thr. The bound grows
// like e^{delta lamb}; once 2^-32 of it exceeds thr the difference is rounding noise and the reference returns a partial
// sum that can be any fraction of E[K] (0.138 for 148.38 two years apart at the default rates). On those keys the loop
// stops on the geometric tail bound of the t_k instead (trans.cuh); the other keys keep the reference's rule and values.
// A series not converged by the reference's cap of k = 10000 returns E[K] = +inf instead of a truncated sum.
// A threshold <= 0 or NaN asks for E[K] to working precision: the tail bound is then compared with 2^-52 of the sum.
#include <math.h>

#include <memory>
#include <mutex>
#include <stdexcept>
#include <unordered_map>
#include <vector>

#include "common.cuh"
#include "trans.cuh"

namespace tracs {

__global__ void k_trans_keys(const int32_t *__restrict__ keyN, const double *__restrict__ keyD, uint32_t n_keys,
                             const double *__restrict__ lg, double lamb, double beta, double thr,
                             double *__restrict__ p0_log, double *__restrict__ eK) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_keys) return;
  trans_eval(keyN[t], keyD[t], lg, lamb, beta, thr, &p0_log[t], &eK[t]);
}

// lg[x] = lgamma(x) by the host libm, like the reference's table (transcluster.hpp:253-258) but long
// enough that k < 10000 never reads past it. Cached across calls.
// Returns a snapshot (shared, immutable): concurrent callers on other threads may grow the table meanwhile.
std::shared_ptr<const std::vector<double>> lgamma_table(size_t n) {
  static std::mutex mu;
  static std::shared_ptr<const std::vector<double>> cur;
  std::lock_guard<std::mutex> g(mu);
  if (!cur || cur->size() < n) {
    auto nx = std::make_shared<std::vector<double>>(cur ? *cur : std::vector<double>());
    const size_t old = nx->size();
    nx->resize(n);
    for (size_t i = old; i < n; ++i) (*nx)[i] = ::lgamma((double)i);
    cur = nx;
  }
  return cur;
}

namespace {
struct KeyHash {
  size_t operator()(const std::pair<int32_t, uint64_t> &k) const {
    uint64_t h = k.second * 0x9E3779B97F4A7C15ull ^ ((uint64_t)(uint32_t)k.first * 0xC2B2AE3D27D4EB4Full);
    return (size_t)(h ^ (h >> 29));
  }
};
}  // namespace

// host arrays in, host arrays out; the series runs on the device for the unique keys only
void trans_dist_device(const int32_t *snp, const double *dt, size_t n, double lamb, double beta, double thr,
                       double *p0_log, double *eK, cudaStream_t st) {
  if (n == 0) return;
  std::unordered_map<std::pair<int32_t, uint64_t>, uint32_t, KeyHash> idx;
  idx.reserve(1024);
  std::vector<int32_t> kN;
  std::vector<double> kD;
  std::vector<uint32_t> which(n);
  int32_t maxN = 0;
  for (size_t i = 0; i < n; ++i) {
    if (snp[i] < 0) throw std::runtime_error("negative SNP distance");
    uint64_t bits;
    memcpy(&bits, &dt[i], 8);
    auto key = std::make_pair(snp[i], bits);
    auto it = idx.find(key);
    if (it == idx.end()) {
      it = idx.emplace(key, (uint32_t)kN.size()).first;
      kN.push_back(snp[i]);
      kD.push_back(dt[i]);
      if (snp[i] > maxN) maxN = snp[i];
    }
    which[i] = it->second;
  }
  const uint32_t nk = (uint32_t)kN.size();
  // lg[x] = lgamma(x), host libm like the reference (transcluster.hpp:253-258), long enough for k < 10000
  const size_t nlg = (size_t)maxN + 10000 + 8;
  const auto lg_keep = lgamma_table(nlg);
  const std::vector<double> &lg = *lg_keep;
  DevBuf<double> d_lg(nlg), d_kD(nk), d_p0(nk), d_eK(nk);
  DevBuf<int32_t> d_kN(nk);
  Timer T(st);
  T.start();
  TRACS_CK(cudaMemcpyAsync(d_lg.p, lg.data(), nlg * 8, cudaMemcpyHostToDevice, st));
  TRACS_CK(cudaMemcpyAsync(d_kN.p, kN.data(), nk * 4, cudaMemcpyHostToDevice, st));
  TRACS_CK(cudaMemcpyAsync(d_kD.p, kD.data(), nk * 8, cudaMemcpyHostToDevice, st));
  k_trans_keys<<<(nk + 63) / 64, 64, 0, st>>>(d_kN.p, d_kD.p, nk, d_lg.p, lamb, beta, thr, d_p0.p, d_eK.p);
  g_stats.kernel_launches++;
  TRACS_CK(cudaGetLastError());
  std::vector<double> h_p0(nk), h_eK(nk);
  TRACS_CK(cudaMemcpyAsync(h_p0.data(), d_p0.p, nk * 8, cudaMemcpyDeviceToHost, st));
  TRACS_CK(cudaMemcpyAsync(h_eK.data(), d_eK.p, nk * 8, cudaMemcpyDeviceToHost, st));
  TRACS_CK(cudaStreamSynchronize(st));
  g_stats.ms_trans += T.stop();
  for (size_t i = 0; i < n; ++i) {
    p0_log[i] = h_p0[which[i]];
    eK[i] = h_eK[which[i]];
  }
}

}  // namespace tracs
