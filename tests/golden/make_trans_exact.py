"""Generates trans_exact.json: log P(k = 0 | N, delta) and E[K] = sum_k k P(k | N, delta) of the TransCluster
series, evaluated in arbitrary precision (mpmath) straight from the definition that lprob_k_given_N_2 restates
(reference src/transcluster.hpp:131-170, oracle/tracs_oracle.c:314-331):

    P(k | N, delta) = lamb^(N+1) beta^k (N+k)! / (N! k!)
                    * exp(-delta beta) / sum_{i<=N} (lamb delta)^i / i!
                    * sum_{i<=N+k} delta^(N+k-i) / (N+k-i)! / (lamb+beta)^(i+1)

delta = 0 (same-day samples) uses the closed forms of the negative-binomial limit: log p0 = (N+1) log(lamb / (lamb+beta)),
E[K] = (N+1) beta / lamb. Needs only mpmath (a SymPy dependency); nothing is read from outside this directory.

    python tests/golden/make_trans_exact.py [processes]
"""
import itertools
import json
import os
import sys

import mpmath

HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(HERE, "trans_exact.json")
DPS = 40
SECONDS_IN_YEAR = 31556952.0

# 2047: the largest SNP threshold the prefilter paths take
N_GRID = [0, 1, 2, 5, 10, 20, 40, 100, 200, 500, 1000, 2047]
DAYS_GRID = [0, 1, 7, 30, 90, 179, 365, 400, 548, 730, 1000, 1461, 2000, 2922, 3650, 7300, 10958, 36500]
RATES = [(29.903, 73.0), (5.3, 6.0), (0.5, 2.0), (1.0, 100.0)]


def delta_of(days):
    """The float64 date difference in years every device path computes for a day difference."""
    return (days * 86400.0) / SECONDS_IN_YEAR


def exact(N, delta, lamb, beta, dps=DPS):
    """(log p0, E[K], sum_k P(k)) of one key, each an mpf, or None when the sum is not proven converged.

    The factors are stepped k -> k+1 by their ratios: A_k = lamb^(N+1) beta^k (N+k)! / (N! k!) e^(-delta beta) / pois,
    A_(k+1) = A_k beta (N+k+1) / (k+1); S_M = sum_{i<=M} delta^(M-i) / (M-i)! / (lamb+beta)^(i+1),
    S_(M+1) = (S_M + delta^(M+1) / (M+1)!) / (lamb+beta). P(k) = A_k S_(N+k)."""
    with mpmath.workdps(dps):
        N = int(N)
        d, la, be = mpmath.mpf(delta), mpmath.mpf(lamb), mpmath.mpf(beta)
        lb = la + be
        if d == 0:
            return (N + 1) * mpmath.log(la / lb), (N + 1) * be / la, mpmath.mpf(1)
        pois, t = mpmath.mpf(0), mpmath.mpf(1)  # t = (lamb delta)^i / i!
        for i in range(N + 1):
            if i:
                t = t * la * d / i
            pois += t
        S, a = mpmath.mpf(0), mpmath.mpf(1)  # a = delta^j / j!
        for j in range(N + 1):  # S_N built up from S_0 = 1 / (lamb+beta)
            if j:
                a = a * d / j
            S = (S + a) / lb
        A = la ** (N + 1) * mpmath.exp(-d * be) / pois
        P = A * S
        p0 = P
        total, eK = P, mpmath.mpf(0)
        k, M = 0, N
        prev = P
        tiny = mpmath.mpf(10) ** (-(dps - 8))
        while True:
            A = A * be * (N + k + 1) / (k + 1)
            a = a * d / (M + 1)
            S = (S + a) / lb
            k, M = k + 1, M + 1
            P = A * S
            total += P
            eK += k * P
            # past the mode, and the remaining terms are negligible at this precision
            if P < prev and k * P < tiny * eK and P < tiny * total:
                break
            prev = P
        if abs(total - 1) > mpmath.mpf("1e-15"):
            return None
        return mpmath.log(p0), eK, total


def _one(key):
    N, days, lamb, beta = key
    r = exact(N, delta_of(days), lamb, beta)
    if r is None:
        return key, None
    lp0, eK, total = r
    return key, {"N": N, "days": days, "lamb": lamb, "beta": beta, "log_p0": float(lp0), "eK": float(eK)}


def main():
    procs = int(sys.argv[1]) if len(sys.argv) > 1 else (os.cpu_count() or 1)
    # the slowest keys (large N, small rates relative to the span) first, so the pool drains evenly
    keys = sorted(itertools.product(N_GRID, DAYS_GRID, RATES), key=lambda k: -(k[0] + 1) * k[2][1] / k[2][0] - k[1] * k[2][1] / 365.0)
    keys = [(N, days, lamb, beta) for N, days, (lamb, beta) in keys]
    if procs > 1:
        import multiprocessing
        with multiprocessing.Pool(procs) as pool:
            res = pool.map(_one, keys, chunksize=1)
    else:
        res = [_one(k) for k in keys]
    cases, skipped = [], []
    for key, c in res:
        (cases if c is not None else skipped).append(c if c is not None else key)
    if skipped:
        sys.exit("not converged, fixture not written: %r" % skipped)
    cases.sort(key=lambda c: (RATES.index((c["lamb"], c["beta"])), c["N"], c["days"]))
    out = {"dps": DPS, "seconds_in_year": SECONDS_IN_YEAR, "delta": "days * 86400 / seconds_in_year", "cases": cases}
    with open(OUT, "w") as f:
        json.dump(out, f, indent=0)
        f.write("\n")
    print("%d keys -> %s" % (len(cases), OUT))


if __name__ == "__main__":
    main()
