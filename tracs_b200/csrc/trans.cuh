// Device-side TransCluster series (shared by trans.cu and the fused path in sweep.cu).
// Restates reference src/transcluster.hpp:62-75,131-238 -- see trans.cu for the derivation.
#pragma once
#include <math.h>
#include <stdint.h>

namespace tracs {

__device__ __forceinline__ double lae(double x, double y) {
  // transcluster.hpp:62-75
  const double t = x - y;
  if (x == y) return x + 0.69314718055994530942;
  if (t > 0) return x + log1p(exp(-t));
  else if (t <= 0) return y + log1p(exp(t));
  return t;
}

// one (N, delta) key -> log P(k = 0 | N, delta) and E[K]
__device__ __forceinline__ void trans_eval(int64_t N, double delta, const double *__restrict__ lg, double lamb, double beta,
                                           double thr, double *p0_out, double *eK_out) {
  const double ln_l = log(lamb), ln_b = log(beta), ln_lb = log(lamb + beta);
  if (!(delta > 0)) {
    // transcluster.hpp:163-167 with k = 0 ; E[K]: negative-binomial mean (see trans.cu header)
    *p0_out = (double)(N + 1) * ln_l + lg[N + 1] - lg[N + 1] - lg[1] - (double)(N + 1) * ln_lb;
    *eK_out = (double)(N + 1) * beta / lamb;
    return;
  }
  const double ln_ld = log(lamb * delta);
  const double ln_d = log(delta);
  double pois = -INFINITY;
  for (int64_t i = 0; i <= N; ++i) pois = lae((double)i * ln_ld - lg[i + 1], pois);
  const double lx = ln_d + ln_lb;
  double G = -INFINITY;  // G_M = LSE_{j<=M}( j*ln(delta*(lamb+beta)) - lg[j+1] ), here M = N
  for (int64_t j = 0; j <= N; ++j) G = lae((double)j * lx - lg[j + 1], G);
  const double common = (double)(N + 1) * ln_l - lg[N + 1] - delta * beta - pois;
  {
    const double lhs = common + lg[N + 1] - lg[1];
    *p0_out = lhs + (G - (double)(N + 1) * ln_lb);
  }
  // ub = sum_k t_k, t_k = exp(lhs + ln k + delta (lamb + beta) - (M+1) ln(lamb+beta)) >= k P(k) (the integral's partial
  // sum replaced by its limit); the reference stops once ub - sum_{j<=k} t_j <= thr.
  const double lub = ln_b + delta * lamb + log((double)(N + 1)) - (ln_l + pois);
  const double ub = exp(lub);
  // That difference means something only while ub is small next to thr: the running sum gathers up to 10^4 terms whose
  // logarithms are each a few ulp off, so the difference is known to a few thousand ulp(ub) ~ 2^-40 ub, and
  // 2^-32 ub <= thr keeps that under thr / 256. Otherwise (ub ~ e^{delta lamb}: samples a year or more apart at the
  // default rates, or ub = inf) the difference is rounding noise, and the loop stops on a tail bound that cannot cancel.
  // Both rules sum the same terms; they differ only in the k at which they stop.
  // thr <= 0 or NaN (log NaN) is never resolvable: it asks for the series to working precision, below.
  const double ln_thr = log(thr);
  const bool resolvable = lub - 32.0 * 0.69314718055994530942 <= ln_thr;
  double lprob = -INFINITY;
  bool converged = false;
  if (resolvable) {
    // the reference's loop, as it was: same terms, same order, same values
    double elprob = -INFINITY, diff = thr + 1.0;
    int64_t k = 1;
    while (diff > thr && k < 10000) {  // a NaN bound ends the loop after one term, like the reference's `diff > threshold_Ek`
      const int64_t M = N + k;
      G = lae((double)M * lx - lg[M + 1], G);
      const double lhs = common + (double)k * ln_b + lg[M + 1] - lg[k + 1];
      const double lp = lhs + (G - (double)(M + 1) * ln_lb);
      const double lk = log((double)k);
      lprob = lae(lprob, lp + lk);
      elprob = lae(elprob, lhs + lk + delta * (lamb + beta) - (double)(M + 1) * ln_lb);
      diff = ub - exp(elprob);
      ++k;
    }
    converged = !(diff > thr);
  } else {
    for (int64_t k = 1; k < 10000 && !converged; ++k) {
      const int64_t M = N + k;
      G = lae((double)M * lx - lg[M + 1], G);
      const double lhs = common + (double)k * ln_b + lg[M + 1] - lg[k + 1];
      const double lp = lhs + (G - (double)(M + 1) * ln_lb);
      const double lk = log((double)k);
      lprob = lae(lprob, lp + lk);
      // t_(k+1) / t_k = rho_k = beta (N+k+1) / (k (lamb+beta)) falls monotonically towards beta / (lamb+beta) < 1, so
      // once rho_k < 1 the rest of the series, and with it E[K] - sum_{j<=k} j P(j), is at most t_k rho_k / (1 - rho_k)
      const double lt = lhs + lk + delta * (lamb + beta) - (double)(M + 1) * ln_lb;  // log t_k
      const double lrho = ln_b + log((double)(M + 1)) - lk - ln_lb;
      // a tail under 2^-52 of the sum changes nothing either: the stop for thr <= 0 (fmax ignores a NaN log thr). With
      // thr > 0 it never binds, as the sum of k P(k) over k < 10^4 is below 10^4 and 2^-52 * 10^4 < 2.3e-12.
      converged = lrho < 0 && lt + lrho - log1p(-exp(lrho)) <= fmax(ln_thr, lprob - 52.0 * 0.69314718055994530942);
    }
  }
  // not converged by the cap: the truncated sum can be any fraction of E[K], so none is returned (SURVEY F7, trans.cu)
  *eK_out = converged ? exp(lprob) : INFINITY;
}

}  // namespace tracs
