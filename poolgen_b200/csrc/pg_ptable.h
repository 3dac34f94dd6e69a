// pg_ptable.h -- host-side construction of the per-scan Student-t tail table.
//
// The degrees of freedom are constant for a whole scan (n-1 for ols_iter, n-2 for pearson_corr), so the two-sided
// tail p(t) = I_{df/(df+t^2)}(df/2, 1/2) is a smooth function of ONE variable.  At pg_scan_open the host evaluates
// the statrs-compatible regularised incomplete beta (the same Lentz continued fraction the device keeps as its
// reference path, pg_device.cuh) on a grid given by the bits of w = 1 + |t| / sqrt(df) and stores one cubic per interval
// for ln p; the table is verified against the direct evaluation between the nodes and refined until the error in
// ln p is below 2e-9, i.e. 500x inside the 1e-6 relative tolerance on p.  The device then needs one FMA, integer
// operations on the high word of w, one 32-byte load, a Horner step and exp per p-value instead of up to 140
// continued-fraction iterations with four f64 divisions each.
#pragma once
#include <math.h>

#include <vector>

#include "pg_statrs_host.h"

namespace pg {

// Lentz continued fraction of statrs 0.16 checked_beta_reg, returning h (the fraction) for already swapped a, b, x
inline double host_beta_cf(double a, double b, double x) {
    const double eps = 1.1102230246251565e-16, fpmin = 2.2250738585072014e-308 / eps;
    const double qab = a + b, qap = a + 1.0, qam = a - 1.0;
    double c = 1.0, d = 1.0 - qab * x / qap;
    if (fabs(d) < fpmin) d = fpmin;
    d = 1.0 / d;
    double h = d;
    for (int mi = 1; mi < 5000; mi++) {
        const double m = mi, m2 = m * 2.0;
        double aa = m * (b - m) * x / ((qam + m2) * (a + m2));
        d = 1.0 + aa * d;
        if (fabs(d) < fpmin) d = fpmin;
        c = 1.0 + aa / c;
        if (fabs(c) < fpmin) c = fpmin;
        d = 1.0 / d;
        h = h * d * c;
        aa = -(a + m) * (qab + m) * x / ((a + m2) * (qap + m2));
        d = 1.0 + aa * d;
        if (fabs(d) < fpmin) d = fpmin;
        c = 1.0 + aa / c;
        if (fabs(c) < fpmin) c = fpmin;
        d = 1.0 / d;
        const double del = d * c;
        h *= del;
        if (fabs(del - 1.0) <= eps) break;
    }
    return h;
}

// ln of the two-sided tail p = I_x(df/2, 1/2), x = df/(df+t^2) = exp(-v^2), as a function of
// v = sqrt(log1p(t^2/df)); 1 - x = -expm1(-v^2) is formed without cancellation, so the value is accurate for every t
inline double host_ln_tail(double v, double df) {
    if (v <= 0.0) return 0.0;
    const double u = v * v;
    const double x = exp(-u);
    const double omx = -expm1(-u);
    const double a = df / 2.0, b = 0.5;
    // statrs' own ln_gamma (Lanczos): the constant the reference's beta_reg uses, not libm's lgamma (they differ by
    // up to 1e-12 at df ~ 1000, a systematic relative offset of every p-value of the scan)
    const double lnB = statrs::ln_gamma(a + b) - statrs::ln_gamma(a) - statrs::ln_gamma(b);
    const double lnbt = lnB + a * (-u) + b * log(omx);
    if (x >= (a + 1.0) / (a + b + 2.0)) {
        // symmetric branch: p = 1 - bt * h / a with (x, a, b) -> (1 - x, b, a)
        const double h = host_beta_cf(b, a, omx);
        return log1p(-exp(lnbt) * h / b);
    }
    const double h = host_beta_cf(a, b, x);
    return lnbt + log(h / a);
}

struct PTable {
    std::vector<double> coef;  // [M][4]: ln p = c0 + s (c1 + s (c2 + s c3)), s in [0,1) inside interval i
    int M = 0;
    // interval i = the top bits of the double w = 1 + |t| / sqrt(df): octave e = i >> bits, 2^bits intervals per octave
    double inv_sqrt_df = 0.0, bits = 0.0, max_err = 1.0;
    // statrs' cut-offs (student_t_cutoffs): the reference's p is exactly 1 for |t| <= t_one and exactly 0 for
    // |t| >= t_zero; the table, which holds the converged tail, must not be consulted there
    double t_one = 0.0, t_zero = 0.0;
};

// checked_beta_reg sets bt = 0 when x = df / (df + t^2) is below 1e-10 or within 4 ulps of 1, so the reference prints
// p = 0 resp. p = 1 exactly, whatever the tail is.  x is formed as the reference forms it (pg_statrs_host.h: no
// contraction); fl(t * t), fl(df + .) and fl(df / .) are monotone, so x is non-increasing in t and each set is an
// interval of t, found by bisection on the ordered bit patterns of the non-negative doubles.
//   t_one  = the largest t with ulps_eq_one(x)
//   t_zero = the smallest t with x < 1e-10
inline void student_t_cutoffs(double df, double &t_one, double &t_zero) {
    auto dbl = [](uint64_t u) {
        double d;
        memcpy(&d, &u, 8);
        return d;
    };
    auto x_of = [df](double t) { return df / (df + t * t); };
    const uint64_t inf_bits = 0x7ff0000000000000ull;
    uint64_t lo = 0, hi = inf_bits;  // ulps_eq_one(x(0)) holds, ulps_eq_one(x(inf)) = ulps_eq_one(0) does not
    while (hi - lo > 1) {
        const uint64_t mid = lo + (hi - lo) / 2;
        (statrs::ulps_eq_one(x_of(dbl(mid))) ? lo : hi) = mid;
    }
    t_one = dbl(lo);
    lo = 0, hi = inf_bits;  // x(0) = 1 is not below 1e-10, x(inf) = 0 is
    while (hi - lo > 1) {
        const uint64_t mid = lo + (hi - lo) / 2;
        (fabs(x_of(dbl(mid))) < 1e-10 ? hi : lo) = mid;
    }
    t_zero = dbl(hi);
}

// ln p as a function of x = |t| / sqrt(df) (t^2 / df = x^2)
inline double host_ln_tail_x(double x, double df) { return host_ln_tail(sqrt(log1p(x * x)), df); }

// The table is indexed by the BITS of w = 1 + x, x = |t| / sqrt(df): uniform in x below 1 (where ln p is smooth in
// x -- it is not in x^2, p ~ 1 - c x at 0), log-spaced above (where ln p ~ -df ln x).  The device then needs one FMA,
// a few integer operations on the high word, one 32-byte load, a Horner step and exp -- no log1p, no sqrt, no
// division on the dependent chain of a p-value (round 1 indexed by v = sqrt(log1p(t^2 / df))).
inline PTable build_ptable(double df) {
    PTable t;
    t.inv_sqrt_df = 1.0 / sqrt(df);
    student_t_cutoffs(df, t.t_one, t.t_zero);
    // x_max: beyond it ib = p/2 < 2^-62, so 1 - ib == 1 and the reference's p is exactly 0
    const double ln_floor = -43.0;
    double lo = 0.0, hi = 0.25;
    while (host_ln_tail_x(hi, df) > ln_floor && hi < 1e12) hi *= 2.0;
    for (int it = 0; it < 80; it++) {
        const double mid = 0.5 * (lo + hi);
        (host_ln_tail_x(mid, df) > ln_floor ? lo : hi) = mid;
    }
    const double x_max = hi;
    int n_oct = 1;
    while (ldexp(1.0, n_oct) < 1.0 + x_max) n_oct++;
    for (int B = 8; B <= 12; B++) {
        const int per = 1 << B;
        const int M = n_oct * per;
        t.M = M;
        t.bits = (double)B;
        t.coef.assign((size_t)M * 4, 0.0);
        auto w_of = [&](int i, double s) {
            const int e = i >> B, f = i & (per - 1);
            return ldexp(1.0 + ((double)f + s) / (double)per, e);
        };
        for (int i = 0; i < M; i++) {
            const double f0 = host_ln_tail_x(w_of(i, 0.0) - 1.0, df), f1 = host_ln_tail_x(w_of(i, 1.0 / 3.0) - 1.0, df),
                         f2 = host_ln_tail_x(w_of(i, 2.0 / 3.0) - 1.0, df), f3 = host_ln_tail_x(w_of(i, 1.0) - 1.0, df);
            // cubic through s = 0, 1/3, 2/3, 1
            t.coef[4 * (size_t)i + 0] = f0;
            t.coef[4 * (size_t)i + 1] = (-11.0 * f0 + 18.0 * f1 - 9.0 * f2 + 2.0 * f3) / 2.0;
            t.coef[4 * (size_t)i + 2] = (18.0 * f0 - 45.0 * f1 + 36.0 * f2 - 9.0 * f3) / 2.0;
            t.coef[4 * (size_t)i + 3] = (-9.0 * f0 + 27.0 * f1 - 27.0 * f2 + 9.0 * f3) / 2.0;
        }
        double err = 0.0;
        const int step = M > 4096 ? M / 4096 : 1;
        for (int i = 0; i < M; i += step)
            for (double s : {0.17, 0.5, 0.83}) {
                const double *c = &t.coef[4 * (size_t)i];
                const double approx = c[0] + s * (c[1] + s * (c[2] + s * c[3]));
                const double exact = host_ln_tail_x(w_of(i, s) - 1.0, df);
                if (exact < ln_floor - 1.0) continue;  // past the point where p is 0 anyway
                err = fmax(err, fabs(approx - exact));
            }
        t.max_err = err;
        if (err < 1e-9) break;
    }
    return t;
}

}  // namespace pg
