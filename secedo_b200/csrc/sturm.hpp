// Eigenvalues of a symmetric tridiagonal matrix by bisection on Sturm counts, after LAPACK DSTEBZ / DLAEBZ.
// Host and device code: eigenvalues.cu runs one eigenvalue index per thread, tests/sturm_host_check.cpp runs the same
// functions on the CPU against scipy.linalg.eigvalsh_tridiagonal.
//
// T has diagonal d[0..n) and off-diagonal e[0..n-1); only e2[i] = e[i]^2 enters the counts.
#pragma once

#include <cfloat>
#include <cmath>
#include <cstdint>

#ifdef __CUDACC__
#define STURM_HD __host__ __device__
#else
#define STURM_HD
#endif

namespace sturm {

// Guard against zero pivots (DSTEBZ: PIVMIN = SAFMIN * max(1, max e^2)): a pivot smaller than this in magnitude is
// replaced by -pivmin, so that the recurrence never divides by zero and the count stays monotone in x.
STURM_HD inline double pivmin(const double *e2, uint32_t n) {
    double m = 1.0;
    for (uint32_t i = 0; i + 1 < n; ++i) {
        m = fmax(m, e2[i]);
    }
    return DBL_MIN * m;
}

// Number of eigenvalues of T that are smaller than x (DLAEBZ's count: the non-positive pivots of LDL^T of T - x I).
STURM_HD inline uint32_t count_below(const double *d, const double *e2, uint32_t n, double x, double pmin) {
    double q = d[0] - x;
    if (fabs(q) <= pmin) {
        q = -pmin;
    }
    uint32_t c = q <= 0.0 ? 1u : 0u;
    for (uint32_t i = 1; i < n; ++i) {
        q = (d[i] - x) - e2[i - 1] / q;
        if (fabs(q) <= pmin) {
            q = -pmin;
        }
        c += q <= 0.0 ? 1u : 0u;
    }
    return c;
}

struct Interval {
    double lo, hi, atol; // Gershgorin interval (widened as DSTEBZ does), absolute tolerance of the bisection
};

// Gershgorin interval of T, widened by DSTEBZ's fudge so that no eigenvalue sits on an end, and the absolute tolerance
// 2 eps max_i (|d_i| + |e_i|) (e_i: both neighbours).
STURM_HD inline Interval gershgorin(const double *d, const double *e, uint32_t n, double pmin) {
    double lo = INFINITY, hi = -INFINITY, tnorm = 0.0;
    for (uint32_t i = 0; i < n; ++i) {
        const double r = (i > 0 ? fabs(e[i - 1]) : 0.0) + (i + 1 < n ? fabs(e[i]) : 0.0);
        lo = fmin(lo, d[i] - r);
        hi = fmax(hi, d[i] + r);
        tnorm = fmax(tnorm, fabs(d[i]) + r);
    }
    const double fudge = 2.1 * tnorm * DBL_EPSILON * n + 2.1 * 2.0 * pmin;
    return Interval{ lo - fudge, hi + fudge, 2.0 * DBL_EPSILON * tnorm };
}

// The k-th smallest eigenvalue (0-based) by bisection of iv: invariant count_below(lo) <= k < count_below(hi). Every
// index starts from the same interval and takes the same midpoints until its path separates from another index's, after
// which the two intervals no longer overlap: the results are non-decreasing in k by construction.
STURM_HD inline double bisect(const double *d, const double *e2, uint32_t n, uint32_t k, Interval iv, double pmin) {
    double lo = iv.lo, hi = iv.hi;
    // width / atol <= 2^54 (atol = 0 only for T = 0, whose interval is a few pmin wide): 128 steps always suffice
    for (int it = 0; it < 128 && hi - lo > iv.atol; ++it) {
        const double mid = 0.5 * (lo + hi);
        if (mid <= lo || mid >= hi) {
            break; // adjacent doubles
        }
        if (count_below(d, e2, n, mid, pmin) > k) {
            hi = mid;
        } else {
            lo = mid;
        }
    }
    return 0.5 * (lo + hi);
}

} // namespace sturm
