// pg_device.cuh -- device-side helpers: mbarrier / bulk-copy PTX (sm_90+ async proxy, SASS UBLKCP on
// sm_100a), warp multi-value reduction, and the statrs-compatible Student-t / chi-square tails.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace pg {

#define PG_FULL_MASK 0xffffffffu
constexpr double kEps = 2.220446049250313e-16;  // f64::EPSILON

__device__ __forceinline__ uint32_t smem_u32(const void *p) {
    return (uint32_t)__cvta_generic_to_shared(p);
}

// ---- mbarrier + 1-D bulk copy (TMA engine, no tensor map needed for contiguous blocks) --------
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void bulk_g2s(void *dst_smem, const void *src_gmem, uint32_t bytes, uint64_t *bar) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
            smem_u32(dst_smem)),
        "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
        : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "LAB_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
        "@P1 bra DONE;\n"
        "bra LAB_WAIT;\n"
        "DONE:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}

// ---- warp reduction of 32 accumulators at once (recursive halving): 31 shuffles of f64 instead
// of 160; on return v[0] of lane L holds the warp total of accumulator L. ------------------------
__device__ __forceinline__ void warp_reduce32(double (&v)[32], int lane) {
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) {
        const bool upper = (lane & off) != 0;
#pragma unroll
        for (int i = 0; i < off; i++) {
            const double a = v[i], b = v[i + off];
            const double send = upper ? a : b;
            const double keep = upper ? b : a;
            v[i] = keep + __shfl_xor_sync(PG_FULL_MASK, send, off);
        }
    }
}

// fixed-order butterfly sum: every lane ends up with the same bits
__device__ __forceinline__ double warp_sum_fixed(double v) {
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) v += __shfl_xor_sync(PG_FULL_MASK, v, off);
    return v;
}

// ---- statrs 0.16 compatible tails (SURVEY.md appendix B) -------------------------------------
// beta_reg(a, b, x) with ln_beta = lnG(a+b) - lnG(a) - lnG(b) supplied by the host (it only depends on
// the degrees of freedom, which are constant for a scan).
__device__ __forceinline__ double beta_reg_dev(double a, double b, double x, double ln_beta) {
    double bt;
    if (fabs(x) < 1e-10 || fabs(x - 1.0) <= 4.0 * 1.1102230246251565e-16) {
        bt = 0.0;
    } else {
        bt = exp(ln_beta + a * log(x) + b * log(1.0 - x));
    }
    const bool symm = x >= (a + 1.0) / (a + b + 2.0);
    const double eps = 1.1102230246251565e-16;
    const double fpmin = 2.2250738585072014e-308 / eps;
    if (symm) {
        const double sw = a;
        x = 1.0 - x;
        a = b;
        b = sw;
    }
    const double qab = a + b, qap = a + 1.0, qam = a - 1.0;
    double c = 1.0;
    double d = 1.0 - qab * x / qap;
    if (fabs(d) < fpmin) d = fpmin;
    d = 1.0 / d;
    double h = d;
    for (int mi = 1; mi < 141; mi++) {
        const double m = (double)mi;
        const double m2 = m * 2.0;
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
    return symm ? 1.0 - bt * h / a : bt * h / a;
}

// two-sided p-value exactly as the reference forms it: 2 * (1 - StudentsT(0,1,df).cdf(|t|))
// (src/gwas/ols.rs:153, src/gwas/correlation_test.rs:66) including the cancellation 1 - (1 - ib).
static __device__ __noinline__ double student_two_sided(double t_abs, double df, double ln_beta) {
    if (isinf(df)) return 2.0 * (1.0 - 0.5 * erfc(-t_abs / sqrt(2.0)));
    // x rounded as the reference rounds it (no FMA): near t_one one ulp of x moves p by up to 1e-8 relative, and it
    // decides statrs' cut-offs
    const double h = df / __dadd_rn(df, __dmul_rn(t_abs, t_abs));
    const double ib = 0.5 * beta_reg_dev(df / 2.0, 0.5, h, ln_beta);
    const double cdf = t_abs <= 0.0 ? ib : 1.0 - ib;
    return 2.0 * (1.0 - cdf);
}

// Same quantity through the per-scan table of ln p indexed by the bits of 1 + |t| / sqrt(df) (pg_ptable.h).  The final
// 2 * (1 - (1 - ib)) reproduces the reference's quantisation of small p-values.  |t| <= t_one and |t| >= t_zero are
// statrs' cut-offs, where the reference's p is exactly 1 resp. 0 (pg_ptable.h, student_t_cutoffs).
struct PTableDev {
    const double4 *coef;
    double inv_sqrt_df, bits;  // bits: intervals per octave of w = 1 + |t| / sqrt(df) as a power of two
    double t_one, t_zero;
    int M;
};
// interval and fraction of w = 1 + x from the bits of the double: idx = octave * 2^B + the top B mantissa bits
__device__ __forceinline__ int ptab_locate(double w, int B, double &s) {
    const int hi = __double2hiint(w);
    const int sh = 20 - B;
    const int idx = (hi >> sh) - (1023 << B);
    const double w0 = __hiloint2double(hi & ~((1 << sh) - 1), 0);
    const double scale = __hiloint2double((2046 + B - (hi >> 20)) << 20, 0);  // 2^(B - e), e = (hi >> 20) - 1023
    s = (w - w0) * scale;
    return idx;
}
__device__ __forceinline__ double student_two_sided_tab(double t_abs, double df, const PTableDev &tb) {
    const double w = fma(t_abs, tb.inv_sqrt_df, 1.0);
    double ptrue = 0.0;
    if (t_abs < tb.t_zero) {  // (NaN fails this test and the one below and gets p = 0 as before)
        double s;
        const int i = ptab_locate(w, (int)tb.bits, s);
        if (i < tb.M) {
            const double2 *cp = reinterpret_cast<const double2 *>(tb.coef + i);
            const double2 c01 = __ldg(cp), c23 = __ldg(cp + 1);
            ptrue = exp(fma(s, fma(s, fma(s, c23.y, c23.x), c01.y), c01.x));
        }
    }
    const double ib = 0.5 * ptrue;
    const double cdf = t_abs <= tb.t_one ? 0.5 : 1.0 - ib;  // p = 1 up to t_one (t = 0 included)
    return 2.0 * (1.0 - cdf);
}

// statrs ln_gamma (Lanczos g = 10.900511, 11 terms), needed on the device only for chi-square
__device__ inline double ln_gamma_dev(double x) {
    const double dk[11] = {2.48574089138753565546e-5,  1.05142378581721974210,     -3.45687097222016235469,
                           4.51227709466894823700,     -2.98285225323576655721,    1.05639711577126713077,
                           -1.95428773191645869583e-1, 1.70970543404441224307e-2,  -5.71926117404305781283e-4,
                           4.63399473359905636708e-6,  -2.71994908488607703910e-9};
    const double R = 10.900511, LN2SEP = 0.6207822376352452223455184457816472122518527279025978;
    const double LNPI = 1.1447298858494001741434273513530587116472948129153, E = 2.71828182845904523536028747135266250;
    if (x < 0.5) {
        double s = dk[0];
        for (int i = 1; i < 11; i++) s += dk[i] / ((double)i - x);
        return LNPI - log(sin(3.14159265358979323846264338327950288 * x)) - log(s) - LN2SEP -
               (0.5 - x) * log((0.5 - x + R) / E);
    }
    double s = dk[0];
    for (int i = 1; i < 11; i++) s += dk[i] / (x + (double)i - 1.0);
    return log(s) + LN2SEP + (x - 0.5) * log((x - 0.5 + R) / E);
}

// statrs checked_gamma_lr(a, x): regularised lower incomplete gamma
__device__ inline double gamma_lr_dev(double a, double x) {
    if (isnan(a) || isnan(x) || a <= 0.0 || isinf(a) || x <= 0.0 || isinf(x)) return nan("");
    const double eps = 0.000000000000001, big = 4503599627370496.0, big_inv = 2.22044604925031308085e-16;
    const double acc = 0.0000000000000011102230246251565;
    if (fabs(a) < acc) return 1.0;
    if (fabs(x) < acc) return 0.0;
    const double ax = a * log(x) - x - ln_gamma_dev(a);
    if (ax < -709.78271289338399) return a < x ? 1.0 : 0.0;
    if (x <= 1.0 || x <= a) {
        double r2 = a, c2 = 1.0, ans2 = 1.0;
        for (int it = 0; it < 100000; it++) {
            r2 += 1.0;
            c2 *= x / r2;
            ans2 += c2;
            if (c2 / ans2 <= eps) break;
        }
        return exp(ax) * ans2 / a;
    }
    double y = 1.0 - a, z = x + y + 1.0;
    int cnt = 0;
    double p3 = 1.0, q3 = x, p2 = x + 1.0, q2 = z * x, ans = p2 / q2;
    for (int it = 0; it < 100000; it++) {
        y += 1.0;
        z += 2.0;
        cnt += 1;
        const double yc = y * (double)cnt;
        const double p = p2 * z - p3 * yc;
        const double q = q2 * z - q3 * yc;
        p3 = p2;
        p2 = p;
        q3 = q2;
        q2 = q;
        if (fabs(p) > big) {
            p3 *= big_inv;
            p2 *= big_inv;
            q3 *= big_inv;
            q2 *= big_inv;
        }
        if (q != 0.0) {
            const double nextans = p / q;
            const double error = fabs((ans - nextans) / nextans);
            ans = nextans;
            if (error <= eps) break;
        }
    }
    return 1.0 - exp(ax) * ans;
}

}  // namespace pg
