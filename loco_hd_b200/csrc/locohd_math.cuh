// locohd_math.cuh — FP64 leaf math of the LoCoHD scoring path as __device__ functions.
//
// Mirrors (freshly written, not translated):
//   weight-function CDFs      /root/reference/src/locohd/weight_function/cdfs.rs:5-63
//   integral_point semantics  /root/reference/src/locohd/weight_function.rs:95-120
//   statistical distances     /root/reference/src/locohd/pmf/statistical_distances.rs:4-142
// CUDA's pow/exp/log differ from glibc by <= 1-2 ulp; the scoring tolerance is 1e-9 absolute.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>
#include "../../include/locohd_b200.h"

namespace locohd {

// Device-side weight function: the ABI struct plus host-precomputed helpers.
struct WfDev {
    int kind;
    int n;
    int int_a;         // kumaraswamy: exponent a if it is a small non-negative integer, else -1
    int int_b;         // kumaraswamy: exponent b likewise
    int monotone;      // the device CDF is provably non-decreasing in floating point (uniform, integer kumaraswamy)
    int pad;
    double inv_range;  // uniform / kumaraswamy: 1 / (x_max - x_min)
    double inv_norm;   // hyper_exp: 1 / sum(a_i)
    double w_inf;      // CDF(+inf), evaluated on the host (1 except for degenerate dagum parameters)
    double p[LOCOHD_MAX_WF_PARAMS];
};

__device__ __forceinline__ double powi_small(double x, int e) {
    // e in [0, 64]: a handful of roundings (<= 1e-15 relative).  Straight-line code for the common small exponents
    // (the exponent is uniform over a launch), square-and-multiply otherwise.
    switch (e) {
        case 0: return 1.0;
        case 1: return x;
        case 2: return x * x;
        case 3: return x * x * x;
        case 4: { const double x2 = x * x; return x2 * x2; }
        case 5: { const double x2 = x * x; return x2 * x2 * x; }
        case 6: { const double x2 = x * x; return x2 * x2 * x2; }
        case 8: { const double x2 = x * x, x4 = x2 * x2; return x4 * x4; }
        default: break;
    }
    double r = 1.0;
    double b = x;
    while (e) {
        if (e & 1) r *= b;
        b *= b;
        e >>= 1;
    }
    return r;
}

// CDF(x) for x >= 0 (x may be +inf).  cdfs.rs:5-63.
__device__ __forceinline__ double wf_cdf(const WfDev& w, double x) {
    switch (w.kind) {
        case LOCOHD_WF_UNIFORM: {
            if (x < w.p[0]) return 0.0;
            if (x > w.p[1]) return 1.0;
            return (x - w.p[0]) * w.inv_range;
        }
        case LOCOHD_WF_KUMARASWAMY: {
            if (x < w.p[0]) return 0.0;
            if (x > w.p[1]) return 1.0;
            const double z = (x - w.p[0]) * w.inv_range;
            const double za = (w.int_a >= 0) ? powi_small(z, w.int_a) : pow(z, w.p[2]);
            const double u = 1.0 - za;
            const double ub = (w.int_b >= 0) ? powi_small(u, w.int_b) : pow(u, w.p[3]);
            return 1.0 - ub;
        }
        case LOCOHD_WF_DAGUM: {
            return pow(1.0 + pow(x / w.p[1], -w.p[0]), -w.p[2]);
        }
        default: {  // LOCOHD_WF_HYPER_EXP
            const int half = w.n >> 1;
            double sum = 0.0;
            for (int i = 0; i < half; ++i) sum += w.p[i] * exp(-w.p[half + i] * x);
            return 1.0 - sum * w.inv_norm;
        }
    }
}

// Density w(x) = W'(x) for x >= 0, branch by branch the derivative of wf_cdf (the same comparisons at the kinks of
// uniform and kumaraswamy: x < x_min -> 0, x > x_max -> 0).
__device__ __forceinline__ double wf_pdf(const WfDev& w, double x) {
    switch (w.kind) {
        case LOCOHD_WF_UNIFORM: {
            if (x < w.p[0] || x > w.p[1]) return 0.0;
            return w.inv_range;
        }
        case LOCOHD_WF_KUMARASWAMY: {
            if (x < w.p[0] || x > w.p[1]) return 0.0;
            const double a = w.p[2], b = w.p[3];
            const double z = (x - w.p[0]) * w.inv_range;
            const double za1 = (w.int_a >= 1) ? powi_small(z, w.int_a - 1) : pow(z, a - 1.0);   // z^(a-1)
            const double u = 1.0 - ((w.int_a >= 0) ? powi_small(z, w.int_a) : pow(z, a));
            const double ub1 = (w.int_b >= 1) ? powi_small(u, w.int_b - 1) : pow(u, b - 1.0);   // (1 - z^a)^(b-1)
            return a * b * za1 * ub1 * w.inv_range;
        }
        case LOCOHD_WF_DAGUM: {
            // W = (1 + u)^-p with u = (x/b)^-a:  w = (a p / x) u (1 + u)^-(p+1), all in one exponent so that neither
            // u, (1 + u) nor a p / x overflows for small x (inf * 0 would give NaN)
            const double a = w.p[0], b = w.p[1], p = w.p[2];
            if (!(x > 0.0)) {   // limit x -> 0 of (a p / x) (x/b)^(a p): 0, a p / b^(a p) or +inf
                const double ap = a * p;
                return ap > 1.0 ? 0.0 : (ap == 1.0 ? ap / b : INFINITY);
            }
            const double lx = log(x);
            const double lu = -a * (lx - log(b));   // log u (x / b would underflow for the smallest x)
            const double l = lu > 0.0 ? -p * lu - (p + 1.0) * log1p(exp(-lu)) : lu - (p + 1.0) * log1p(exp(lu));
            return exp(l + log(a * p) - lx);
        }
        default: {  // LOCOHD_WF_HYPER_EXP
            const int half = w.n >> 1;
            double sum = 0.0;
            for (int i = 0; i < half; ++i) sum += w.p[i] * w.p[half + i] * exp(-w.p[half + i] * x);
            return sum * w.inv_norm;
        }
    }
}

// ---- statistical distances on normalised compositions --------------------------------------------
// P1(i) / P2(i) are callables returning the i-th normalised probability.

template <class P1, class P2>
__device__ __forceinline__ double sd_hellinger(int C, double e, P1 p1, P2 p2) {
    // statistical_distances.rs:4-10
    const double inv_e = 1.0 / e;
    double dist = 0.0;
    for (int i = 0; i < C; ++i) dist += pow(fabs(pow(p1(i), inv_e) - pow(p2(i), inv_e)), e);
    return pow(dist / 2.0, inv_e);
}

template <class P1, class P2>
__device__ __forceinline__ double sd_ks(int C, P1 p1, P2 p2) {
    // statistical_distances.rs:12-21
    double best = 0.0;
    for (int i = 0; i < C; ++i) best = fmax(best, fabs(p1(i) - p2(i)));
    return best;
}

template <class P1, class P2>
__device__ __forceinline__ double sd_kl(int C, double eps, P1 p1, P2 p2) {
    // statistical_distances.rs:23-29
    double dist = 0.0;
    for (int i = 0; i < C; ++i) {
        const double x = p1(i);
        dist += x * log((x + eps) / (p2(i) + eps));
    }
    return dist;
}

template <class P1, class P2>
__device__ __forceinline__ double sd_renyi(int C, double alpha, double eps, P1 p1, P2 p2) {
    // statistical_distances.rs:31-78
    if (alpha == 1.0) return sd_kl(C, eps, p1, p2);
    if (isinf(alpha) && alpha > 0.0) {
        double best = (p1(0) + eps) / (p2(0) + eps);
        for (int i = 1; i < C; ++i) best = fmax(best, (p1(i) + eps) / (p2(i) + eps));
        return log(best);
    }
    if (alpha == 0.0) {
        double s = 0.0;
        for (int i = 0; i < C; ++i)
            if (p1(i) > 0.0) s += p2(i);
        return -log(s);
    }
    double s = 0.0;
    for (int i = 0; i < C; ++i) {
        const double x = p1(i);
        s += x * pow((x + eps) / (p2(i) + eps), alpha - 1.0);
    }
    return log(s) / (alpha - 1.0);
}

// x^y for the scoring walk (x >= 0): exp(y log x) for positive finite x (a few 1e-15 relative for the |y log x| < 50
// that occur here, against the 1e-9 bar; about a third of the instructions of pow()), pow() itself for 0, inf and NaN so
// that the special cases stay those of the reference's powf.
__device__ __forceinline__ double pow_walk(double x, double y) {
    if (x > 0.0 && x < 1.7e308) return exp(y * log(x));
    return pow(x, y);
}

// The statistical distances of the generic scoring kernel on pre-scaled inputs: pa(i) = val_a(i) * ia with ia = 1 / norm
// (one division per event instead of one per category and side).  Same formulas as sd_* above.
template <class VA, class VB>
__device__ __forceinline__ double sd_scaled(int kind, double q0, double q1, int C, VA va, VB vb, double ia, double ib) {
    switch (kind) {
        case LOCOHD_SD_KOLMOGOROV_SMIRNOV: {
            double best = 0.0;
            for (int i = 0; i < C; ++i) best = fmax(best, fabs(__dmul_rn(va(i), ia) - __dmul_rn(vb(i), ib)));   // both products rounded: identical compositions give exactly 0
            return best;
        }
        case LOCOHD_SD_KULLBACK_LEIBLER: {
            double dist = 0.0;
            for (int i = 0; i < C; ++i) {
                const double x = va(i) * ia;
                dist += x * log((x + q0) / (vb(i) * ib + q0));
            }
            return dist;
        }
        default: {   // Renyi (statistical_distances.rs:31-78)
            const double alpha = q0, eps = q1;
            if (alpha == 1.0) {
                double dist = 0.0;
                for (int i = 0; i < C; ++i) {
                    const double x = va(i) * ia;
                    dist += x * log((x + eps) / (vb(i) * ib + eps));
                }
                return dist;
            }
            if (isinf(alpha) && alpha > 0.0) {
                double best = (va(0) * ia + eps) / (vb(0) * ib + eps);
                for (int i = 1; i < C; ++i) best = fmax(best, (va(i) * ia + eps) / (vb(i) * ib + eps));
                return log(best);
            }
            if (alpha == 0.0) {
                double s = 0.0;
                for (int i = 0; i < C; ++i)
                    if (va(i) * ia > 0.0) s += vb(i) * ib;
                return -log(s);
            }
            double s = 0.0;
            for (int i = 0; i < C; ++i) {
                const double x = va(i) * ia;
                s += x * pow_walk((x + eps) / (vb(i) * ib + eps), alpha - 1.0);
            }
            return log(s) / (alpha - 1.0);
        }
    }
}

template <class P1, class P2>
__device__ __forceinline__ double sd_run(int kind, double q0, double q1, int C, P1 p1, P2 p2) {
    // statistical_distances.rs:123-142
    switch (kind) {
        case LOCOHD_SD_HELLINGER: return sd_hellinger(C, q0, p1, p2);
        case LOCOHD_SD_KOLMOGOROV_SMIRNOV: return sd_ks(C, p1, p2);
        case LOCOHD_SD_KULLBACK_LEIBLER: return sd_kl(C, q0, p1, p2);
        default: return sd_renyi(C, q0, q1, p1, p2);
    }
}

}  // namespace locohd
