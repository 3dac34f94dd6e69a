// pg_scan.cuh -- the per-locus OLS / Pearson scan kernel (ols_iterate: src/gwas/ols.rs:201-276,
// correlation: src/gwas/correlation_test.rs:73-129) for sm_100a.
//
// One persistent CTA per SM.  Every warp owns a private ring of shared-memory stage buffers fed by 1-D bulk copies
// (cp.async.bulk -> SASS UBLKCP, completion on an mbarrier), so there is no CTA-wide synchronisation in the steady
// state.  A warp works on blocks of G consecutive loci:
//   phase 1  stream the frequency matrix.  P lanes share one locus (P = 32: one locus per stage, row chunks of
//            Layout::rc pools; P = 8: four whole loci per stage, for pool counts that fit one chunk), each lane owns
//            row pairs (128-bit shared loads) and accumulates the column sums, the A(A+1)/2 products and the A*K
//            cross products with the centred phenotypes (resident in shared memory).  The partial sums are reduced
//            through a [accumulator][lane] transposition in the stage buffer that was just consumed and parked in
//            the warp's totals area.
//   phase 2  lane = locus, once per block: keep-mask (LocusCounts::filter, src/base/sync.rs:195-303) and allele
//            order (src/base/sync.rs:478-505) from the totals, centred normal equations, Cholesky, beta, residual
//            variance, t and the Student-t two-sided p-value, records written straight to global memory.
// Loci whose MAF-removed alleles carry reads need the frequencies renormalised over the kept alleles: when the ingest
// hint (pg_ingest.cu) vouches for the keep-mask they are rescaled in registers while they stream; decisions that land
// within a rounding bound of a threshold are re-evaluated in the reference's exact sequential order (bit-exact mask)
// and, with the pools without coverage and the cancellation-prone fits, are left to fixup_kernel, where a whole warp
// re-accumulates the locus from global memory.
#pragma once
#include "pg_device.cuh"
#include "pg_internal.h"

namespace pg {

constexpr int kScanWarps = 12;  // 384 threads -> up to 168 registers per thread
constexpr int kRedPitch = 33;   // row pitch (doubles) of the reduction scratch: conflict free both ways

template <int A, int K, bool W>
struct Acc {
    static constexpr int S0 = 0;                        // column sums
    static constexpr int P0 = S0 + A;                   // products f_j f_l, j <= l
    static constexpr int C0 = P0 + A * (A + 1) / 2;     // cross products f_j y_k
    static constexpr int Q0 = C0 + A * K;               // weighted column sums (unequal pool sizes only)
    static constexpr int N = Q0 + (W ? A : 0);
    static constexpr int NP = N | 1;                    // odd pitch of a totals row: lane = locus reads are conflict free
    __host__ __device__ static constexpr int tri(int j, int l) {  // j <= l
        return P0 + j * A - j * (j - 1) / 2 + (l - j);
    }
};

template <int A, int K, bool W, bool NANAWARE>
__device__ __forceinline__ void accum_row(double (&acc)[Acc<A, K, W>::N], const double (&f)[A], const double (&y)[K],
                                          double w) {
    using AC = Acc<A, K, W>;
#pragma unroll
    for (int j = 0; j < A; j++) {
        if (NANAWARE)
            acc[AC::S0 + j] += (f[j] != f[j]) ? 0.0 : f[j];  // column sums ignore NaN (sync.rs:483-489)
        else
            acc[AC::S0 + j] += f[j];
    }
#pragma unroll
    for (int j = 0; j < A; j++)
#pragma unroll
        for (int l = j; l < A; l++) acc[AC::tri(j, l)] = fma(f[j], f[l], acc[AC::tri(j, l)]);
#pragma unroll
    for (int j = 0; j < A; j++)
#pragma unroll
        for (int k = 0; k < K; k++) acc[AC::C0 + j * K + k] = fma(f[j], y[k], acc[AC::C0 + j * K + k]);
    if (W) {
#pragma unroll
        for (int j = 0; j < A; j++) acc[AC::Q0 + j] = fma(f[j], w, acc[AC::Q0 + j]);
    }
}

// two consecutive rows held as double2 per column
template <int A, int K, bool W>
__device__ __forceinline__ void accum_pair(double (&acc)[Acc<A, K, W>::N], const double2 (&f2)[A],
                                           const double2 (&y2)[K], double2 w2) {
    double fa[A], ya[K];
#pragma unroll
    for (int j = 0; j < A; j++) fa[j] = f2[j].x;
#pragma unroll
    for (int k = 0; k < K; k++) ya[k] = y2[k].x;
    accum_row<A, K, W, false>(acc, fa, ya, w2.x);
#pragma unroll
    for (int j = 0; j < A; j++) fa[j] = f2[j].y;
#pragma unroll
    for (int k = 0; k < K; k++) ya[k] = y2[k].y;
    accum_row<A, K, W, false>(acc, fa, ya, w2.y);
}

// Reduction of the per-lane partial sums: every lane stores its N accumulators into a [accumulator][lane] tile, then
// the totals of the 32/P loci of this step are formed by summing P consecutive entries of a row in a fixed order
// (so a locus gets the same bits wherever it lands) and written to tot[u * NP + a].  The scratch holds red_rows
// accumulators at a time.
template <int N, int NP, int P>
__device__ __forceinline__ void reduce_to_tot(const double (&acc)[N], double *red, int red_rows, double *tot,
                                              int lane) {
    constexpr int LPS = 32 / P;
    if (red_rows >= N) {
        // the whole accumulator set fits the scratch (small loci: this runs once per stage, so it is kept free of
        // run-time bounds -- constant store offsets, division by the constant N)
#pragma unroll
        for (int i = 0; i < N; i++) red[i * kRedPitch + lane] = acc[i];
        __syncwarp();
#pragma unroll
        for (int t0 = 0; t0 < N * LPS; t0 += 32) {
            const int t = t0 + lane;
            if (t < N * LPS) {
                const int u = (LPS == 1) ? 0 : t / N;
                const int a = t - u * N;
                const double *row = red + a * kRedPitch + u * P;
                double s0 = row[0], s1 = row[1], s2 = row[2], s3 = row[3];
#pragma unroll
                for (int i = 4; i < P; i += 4) {
                    s0 += row[i];
                    s1 += row[i + 1];
                    s2 += row[i + 2];
                    s3 += row[i + 3];
                }
                tot[u * NP + a] = (s0 + s1) + (s2 + s3);
            }
        }
        __syncwarp();
        return;
    }
    for (int b0 = 0; b0 < N; b0 += red_rows) {
        if (b0) __syncwarp();
#pragma unroll
        for (int i = 0; i < N; i++)
            if (i >= b0 && i < b0 + red_rows) red[(i - b0) * kRedPitch + lane] = acc[i];
        __syncwarp();
        const int nb = min(red_rows, N - b0);
        for (int t = lane; t < nb * LPS; t += 32) {
            const int u = (LPS == 1) ? 0 : t / nb;
            const int a = t - u * nb;
            const double *row = red + a * kRedPitch + u * P;
            double s0 = row[0], s1 = row[1], s2 = row[2], s3 = row[3];
#pragma unroll
            for (int i = 4; i < P; i += 4) {
                s0 += row[i];
                s1 += row[i + 1];
                s2 += row[i + 2];
                s3 += row[i + 3];
            }
            tot[u * NP + b0 + a] = (s0 + s1) + (s2 + s3);
        }
    }
    __syncwarp();
}

// q_j = sum_i f_ij * (s_i / S), accumulated in pool order with separately rounded multiply and add,
// NaN frequencies contribute 0 -- the exact arithmetic of src/base/sync.rs:258-271.  Called by the whole warp: 32 pools
// are loaded at once (one coalesced request instead of 32 dependent ones), every lane forms its own product, and the
// sum runs over the lanes in pool order through shuffles; every lane returns the same q.
static __device__ __noinline__ double exact_q(const ScanParams &p, int64_t locus, int j, const double *ws, int lane) {
    const Layout &lay = p.lay;
    const double *fl = p.freq + (size_t)locus * lay.freq_stride();
    double q = 0.0;
    int i0 = 0;
    for (int c = 0; c < lay.n_chunks; c++) {
        const int rcc = (c == lay.n_chunks - 1) ? lay.rc_last : lay.rc;
        const double *col = fl + (size_t)c * lay.A * lay.rc + (size_t)j * rcc;
        const int rows = min(rcc, lay.n - i0);
        for (int r0 = 0; r0 < rows; r0 += 32) {
            const int r = r0 + lane;
            double term = 0.0;
            if (r < rows) {
                const double f = col[r];
                const double w = ws ? ws[i0 + r] : p.w_uniform;
                term = (f != f) ? 0.0 : __dmul_rn(f, w);
            }
            const int m = min(32, rows - r0);
            for (int t = 0; t < m; t++) q = __dadd_rn(q, __shfl_sync(PG_FULL_MASK, term, t));
        }
        i0 += rcc;
    }
    return q;
}

// renormalised frequency of (pool i, column j) over the kept columns:
// c_ij / sum_{kept} c_i.  (LocusCounts::to_frequencies after the filter, src/base/sync.rs:166-192),
// with c_ij = rint(f_ij * depth_i) recovering the integer count exactly.
template <int A>
__device__ __forceinline__ void renorm_row(const double (&f)[A], uint32_t d, unsigned kept, double (&F)[A]) {
    double c[A];
    double dk = 0.0;
#pragma unroll
    for (int j = 0; j < A; j++) {
        c[j] = (d == 0u) ? 0.0 : rint(f[j] * (double)d);
        if ((kept >> j) & 1u) dk += c[j];
    }
#pragma unroll
    for (int j = 0; j < A; j++) {
        if ((kept >> j) & 1u)
            F[j] = (dk == 0.0) ? nan("") : c[j] / dk;
        else
            F[j] = 0.0;
    }
}

// the same with one division per row (c_ij * (1 / sum_kept c_i.)): within 1.5 ulp of the reference's quotient, used
// where only the regression sums are formed (every order- or threshold-sensitive decision has its own exact path)
template <int A>
__device__ __forceinline__ void renorm_row_fast(const double (&f)[A], uint32_t d, unsigned kept, double (&F)[A]) {
    double c[A];
    double dk = 0.0;
#pragma unroll
    for (int j = 0; j < A; j++) {
        c[j] = (d == 0u) ? 0.0 : rint(f[j] * (double)d);
        if ((kept >> j) & 1u) dk += c[j];
    }
    const double inv = (dk == 0.0) ? nan("") : 1.0 / dk;
#pragma unroll
    for (int j = 0; j < A; j++) F[j] = ((kept >> j) & 1u) ? c[j] * inv : 0.0;
}

// the streaming form for loci whose ingest hint names the kept alleles: two rows (row, row + 1) of first-stage
// frequencies f_ij = c_ij / depth_i become f_ij / sum_kept f_i. -- the depth cancels, so no depth load; within 4 ulp of
// the reference's c_ij / sum_kept c_i. (only the regression sums are formed from it; a tie of column sums or a lost
// digit still goes to the fix-up kernel).  A pool whose reads all sit on removed alleles gives NaN like the reference
// (0 / 0), padding rows stay 0.
// 1 / x for a sum of frequencies (0 < x <= 1 + a few ulp, or exactly 0): hardware seed + two Newton steps, within
// 1 ulp of the quotient -- a fifth of the instructions of the IEEE division; x = 0 gives NaN (inf seed), which is what
// the caller wants for 0 / 0
__device__ __forceinline__ double rcp_fast(double x) {
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
    double e = fma(-x, r, 1.0);
    r = fma(r, e, r);
    e = fma(-x, r, 1.0);
    return fma(r, e, r);
}

template <int A>
__device__ __forceinline__ void renorm_pair(double2 (&f2)[A], unsigned kept, int row, int n) {
    double sx = 0.0, sy = 0.0;
#pragma unroll
    for (int j = 0; j < A; j++)
        if ((kept >> j) & 1u) {
            sx += f2[j].x;
            sy += f2[j].y;
        }
    const double ix = (row < n) ? rcp_fast(sx) : 0.0, iy = (row + 1 < n) ? rcp_fast(sy) : 0.0;
#pragma unroll
    for (int j = 0; j < A; j++)
        f2[j] = ((kept >> j) & 1u) ? make_double2(f2[j].x * ix, f2[j].y * iy) : make_double2(0.0, 0.0);
}

// column sum of the renormalised frequencies in pool order, NaN ignored (src/base/sync.rs:483-489)
template <int A>
__device__ __noinline__ double exact_colsum(const ScanParams &p, int64_t locus, int jsel, unsigned kept) {
    const Layout &lay = p.lay;
    const double *fl = p.freq + (size_t)locus * lay.freq_stride();
    const uint32_t *dl = p.depth + (size_t)locus * lay.depth_stride();
    double s = 0.0;
    int i0 = 0;
    for (int c = 0; c < lay.n_chunks; c++) {
        const int rcc = (c == lay.n_chunks - 1) ? lay.rc_last : lay.rc;
        const double *blk = fl + (size_t)c * lay.A * lay.rc;
        const int rows = min(rcc, lay.n - i0);
        for (int r = 0; r < rows; r++) {
            double f[A], F[A];
#pragma unroll
            for (int j = 0; j < A; j++) f[j] = blk[(size_t)j * rcc + r];
            renorm_row<A>(f, dl[i0 + r], kept, F);
            double v = 0.0;
#pragma unroll
            for (int j = 0; j < A; j++)
                if (j == jsel) v = F[j];
            if (v == v) s = __dadd_rn(s, v);
        }
        i0 += rcc;
    }
    return s;
}

// Rows i = lane, lane + 32, ... of one locus straight from global memory, four rows per lane in flight:
// fn(i, f[A], depth_i).  The building block of the warp-cooperative slow paths.
template <int A, typename Fn>
__device__ __forceinline__ void for_rows_coop(const ScanParams &p, int64_t locus, int lane, Fn &&fn) {
    const Layout &lay = p.lay;
    const double *fl = p.freq + (size_t)locus * lay.freq_stride();
    const uint32_t *dl = p.depth + (size_t)locus * lay.depth_stride();
    int i0 = 0;
    for (int c = 0; c < lay.n_chunks; c++) {
        const int rcc = (c == lay.n_chunks - 1) ? lay.rc_last : lay.rc;
        const double *blk = fl + (size_t)c * lay.A * lay.rc;
        const int rows = min(rcc, lay.n - i0);
        for (int r0 = 0; r0 < rows; r0 += 128) {
            double f[4][A];
            uint32_t d[4];
#pragma unroll
            for (int i = 0; i < 4; i++) {
                const int r = r0 + lane + 32 * i;
                const bool ok = r < rows;
#pragma unroll
                for (int j = 0; j < A; j++) f[i][j] = ok ? blk[(size_t)j * rcc + r] : 0.0;
                d[i] = ok ? dl[i0 + r] : 1u;
            }
#pragma unroll
            for (int i = 0; i < 4; i++) {
                const int r = r0 + lane + 32 * i;
                if (r < rows) fn(i0 + r, f[i], d[i]);
            }
        }
        i0 += rcc;
    }
}

// Full reference pipeline for one locus straight from global memory, executed by the whole warp (lane = pool):
// exact q with NaN handling, missingness, renormalisation over the kept alleles.  Used when a pool has no coverage
// or when a removed allele carries reads (both rare).  Leaves the re-accumulated totals in tot[0..N).
template <int A, int K, bool W>
__device__ __noinline__ int slow_locus(const ScanParams &p, int64_t locus, const double *ys, const double *ws,
                                       double *tot, int lane, bool decide, unsigned &kept_out) {
    using AC = Acc<A, K, W>;
    const Layout &lay = p.lay;
    const uint32_t *dl = p.depth + (size_t)locus * lay.depth_stride();
    unsigned kept = kept_out;
    if (decide) {  // a pool without coverage poisoned the fast sums: redo the MAF decision exactly (lane j = column j)
        kept = 0;
        for (int j = 0; j < A; j++) {
            const double q = exact_q(p, locus, j, ws, lane);
            if (!((q < p.maf) | (q > p.one_minus_maf))) kept |= 1u << j;
        }
        kept_out = kept;
        if (__popc(kept) < 2) return PG_LOCUS_FILTERED;
        // missingness on the first kept column: NaN <=> the pool has no coverage (sync.rs:287-299)
        int miss = 0;
        for (int i = lane; i < lay.n; i += 32) miss += (dl[i] == 0u) ? 1 : 0;
        miss = __reduce_add_sync(PG_FULL_MASK, miss);
        if (miss == lay.n) return PG_LOCUS_FILTERED;
        if (((double)miss / (double)lay.n) > p.max_miss) return PG_LOCUS_FILTERED;
    }
    double acc[AC::N];
#pragma unroll
    for (int i = 0; i < AC::N; i++) acc[i] = 0.0;
    const int n_pad = lay.n_pad;
    for_rows_coop<A>(p, locus, lane, [&](int i, const double(&f)[A], uint32_t d) {
        double F[A], y[K];
        renorm_row_fast<A>(f, d, kept, F);
#pragma unroll
        for (int k = 0; k < K; k++) y[k] = ys[k * n_pad + i];
        accum_row<A, K, W, true>(acc, F, y, 0.0);
    });
#pragma unroll
    for (int i = 0; i < AC::N; i++) {
        const double v = warp_sum_fixed(acc[i]);
        if (lane == 0) tot[i] = v;
    }
    __syncwarp();
    return PG_LOCUS_OK;
}

// Cholesky of the m x m SPD matrix S (lower triangle filled) -> Li = L^-1 (lower), dg = diag(S^-1)
__device__ __forceinline__ bool chol_inv(int m, const double (&S)[PG_MAX_SLOTS][PG_MAX_SLOTS],
                                         double (&Li)[PG_MAX_SLOTS][PG_MAX_SLOTS], double (&dg)[PG_MAX_SLOTS]) {
    double Lm[PG_MAX_SLOTS][PG_MAX_SLOTS];
    bool ok = true;
    for (int a = 0; a < m; a++)
        for (int b = 0; b <= a; b++) {
            double s = S[a][b];
            for (int c = 0; c < b; c++) s -= Lm[a][c] * Lm[b][c];
            if (a == b) {
                if (!(s > 0.0)) {
                    ok = false;
                    s = 1.0;
                }
                Lm[a][a] = sqrt(s);
            } else {
                Lm[a][b] = s / Lm[b][b];
            }
        }
    for (int a = 0; a < m; a++) {
        Li[a][a] = 1.0 / Lm[a][a];
        for (int b = 0; b < a; b++) {
            double s = 0.0;
            for (int c = b; c < a; c++) s -= Lm[a][c] * Li[c][b];
            Li[a][b] = s / Lm[a][a];
        }
    }
    for (int b = 0; b < m; b++) {
        double s = 0.0;
        for (int a = b; a < m; a++) s += Li[a][b] * Li[a][b];
        dg[b] = s;
    }
    return ok;
}

// beta_k = S^-1 sxy_k through Li; returns z'z (= beta' sxy)
__device__ __forceinline__ double solve_rhs(int m, const double (&Li)[PG_MAX_SLOTS][PG_MAX_SLOTS],
                                            const double (&sxy)[PG_MAX_SLOTS], double (&beta)[PG_MAX_SLOTS]) {
    double z[PG_MAX_SLOTS];
    double zz = 0.0;
    for (int a = 0; a < m; a++) {
        double s = 0.0;
        for (int b = 0; b <= a; b++) s += Li[a][b] * sxy[b];
        z[a] = s;
        zz += s * s;
    }
    for (int b = 0; b < m; b++) {
        double s = 0.0;
        for (int a = b; a < m; a++) s += Li[a][b] * z[a];
        beta[b] = s;
    }
    return zz;
}

__device__ __forceinline__ int slot_col(unsigned cb, int s) { return (int)((cb >> (4 * s)) & 0xfu); }

enum { REDO_NONE = 0, REDO_OLS = 1, REDO_CORR = 2, REDO_CORR_NAN = 3, REDO_DEFER = 4, REDO_MINNORM = 5 };

// the analysis as a compile-time constant in the streaming kernel (KIND = PG_KIND_OLS / PG_KIND_CORR: the other
// analysis' phase-2 code is not even linked -- the small-locus kernels are sensitive to their instruction footprint),
// a run-time value in the fix-up kernel (KIND = -1)
template <int KIND>
__device__ __forceinline__ bool kind_is_ols(const ScanParams &p) {
    if constexpr (KIND >= 0) return KIND == PG_KIND_OLS;
    else return p.kind == PG_KIND_OLS;
}

// Reference-style two-pass evaluation of one locus straight from global memory by the whole warp (lane = pool):
// explicit centred moments and explicit residuals e = y - Xb as src/gwas/ols.rs:98-104.  Used when the single-pass
// Gram form would lose digits to cancellation (near-perfect fits, nearly constant or nearly collinear allele
// columns), and for pearsons_correlation with missing frequencies (src/gwas/correlation_test.rs:21-31: pools whose
// frequency is NaN are dropped pairwise, the means and centred sums run over the remaining pools).  Every lane ends
// up with the same numbers; lane 0 leaves (beta | r, var) per (slot, phenotype) in out[0 .. 2 (A-1) K).
template <int A, int K>
__device__ __noinline__ int redo_locus(const ScanParams &p, int64_t locus, unsigned kept, int m, unsigned cb, int mode,
                                       const double *ys, double *out, int lane) {
    constexpr int MS = A - 1;
    const Layout &lay = p.lay;
    const int n_pad = lay.n_pad;
    const double nn = (double)lay.n;
    double xbar[MS], ybar[K];
    double cntv = nn;
    // pass 0: means (the totals of the fast path are not trusted here)
    {
        double sx[MS], sy[K], cnt = 0.0;
#pragma unroll
        for (int a = 0; a < MS; a++) sx[a] = 0.0;
#pragma unroll
        for (int k = 0; k < K; k++) sy[k] = 0.0;
        for_rows_coop<A>(p, locus, lane, [&](int i, const double(&f)[A], uint32_t d) {
            double F[A], x[MS];
            renorm_row<A>(f, d, kept, F);
            bool valid = true;
#pragma unroll
            for (int a = 0; a < MS; a++) {
                double v = 0.0;
#pragma unroll
                for (int j = 0; j < A; j++)
                    if (a < m && j == slot_col(cb, a)) v = F[j];
                x[a] = v;
                valid &= (v == v);
            }
            if (mode == REDO_CORR_NAN && !valid) return;
            cnt += 1.0;
#pragma unroll
            for (int a = 0; a < MS; a++) sx[a] += x[a];
#pragma unroll
            for (int k = 0; k < K; k++) sy[k] += ys[k * n_pad + i];
        });
        cntv = warp_sum_fixed(cnt);
#pragma unroll
        for (int a = 0; a < MS; a++) xbar[a] = warp_sum_fixed(sx[a]) / cntv;
#pragma unroll
        for (int k = 0; k < K; k++) ybar[k] = warp_sum_fixed(sy[k]) / cntv;
    }
    // pass 1: centred moments
    double S[PG_MAX_SLOTS][PG_MAX_SLOTS], sxy[K][PG_MAX_SLOTS], syy[K];
    {
        double Sa[MS * (MS + 1) / 2], sxya[K][MS], syya[K];
#pragma unroll
        for (int i = 0; i < MS * (MS + 1) / 2; i++) Sa[i] = 0.0;
#pragma unroll
        for (int k = 0; k < K; k++) {
            syya[k] = 0.0;
#pragma unroll
            for (int a = 0; a < MS; a++) sxya[k][a] = 0.0;
        }
        for_rows_coop<A>(p, locus, lane, [&](int i, const double(&f)[A], uint32_t d) {
            double F[A], x[MS];
            renorm_row<A>(f, d, kept, F);
            bool valid = true;
#pragma unroll
            for (int a = 0; a < MS; a++) {
                double v = 0.0;
#pragma unroll
                for (int j = 0; j < A; j++)
                    if (a < m && j == slot_col(cb, a)) v = F[j];
                valid &= (v == v);
                x[a] = v - xbar[a];
            }
            if (mode == REDO_CORR_NAN && !valid) return;
#pragma unroll
            for (int a = 0; a < MS; a++)
#pragma unroll
                for (int b = 0; b <= a; b++) Sa[a * (a + 1) / 2 + b] = fma(x[a], x[b], Sa[a * (a + 1) / 2 + b]);
#pragma unroll
            for (int k = 0; k < K; k++) {
                const double dy = ys[k * n_pad + i] - ybar[k];
                syya[k] = fma(dy, dy, syya[k]);
#pragma unroll
                for (int a = 0; a < MS; a++) sxya[k][a] = fma(x[a], dy, sxya[k][a]);
            }
        });
#pragma unroll
        for (int a = 0; a < PG_MAX_SLOTS; a++)
#pragma unroll
            for (int b = 0; b < PG_MAX_SLOTS; b++) S[a][b] = 0.0;
#pragma unroll
        for (int a = 0; a < MS; a++)
#pragma unroll
            for (int b = 0; b <= a; b++) S[a][b] = warp_sum_fixed(Sa[a * (a + 1) / 2 + b]);
#pragma unroll
        for (int k = 0; k < K; k++) {
            syy[k] = warp_sum_fixed(syya[k]);
#pragma unroll
            for (int a = 0; a < PG_MAX_SLOTS; a++) sxy[k][a] = 0.0;
#pragma unroll
            for (int a = 0; a < MS; a++) sxy[k][a] = warp_sum_fixed(sxya[k][a]);
        }
    }
    if (mode != REDO_OLS) {
        if (lane == 0)
            for (int a = 0; a < m; a++)
                for (int k = 0; k < K; k++) {
                    const double den = (mode == REDO_CORR_NAN) ? sqrt(S[a][a]) * sqrt(syy[k])
                                                                : sqrt(S[a][a]) * sqrt(p.syy[k]);
                    out[(a * K + k) * 2 + 0] = sxy[k][a] / den;
                    out[(a * K + k) * 2 + 1] = 0.0;
                }
        __syncwarp();
        return PG_LOCUS_OK;
    }
    double Li[PG_MAX_SLOTS][PG_MAX_SLOTS], dg[PG_MAX_SLOTS], beta[K][PG_MAX_SLOTS];
    if (!chol_inv(m, S, Li, dg)) return PG_LOCUS_FAILED;
    for (int k = 0; k < K; k++) solve_rhs(m, Li, sxy[k], beta[k]);
    // pass 2: explicit residuals
    double rss[K];
    {
        double ra[K];
#pragma unroll
        for (int k = 0; k < K; k++) ra[k] = 0.0;
        for_rows_coop<A>(p, locus, lane, [&](int i, const double(&f)[A], uint32_t d) {
            double F[A], x[MS];
            renorm_row<A>(f, d, kept, F);
#pragma unroll
            for (int a = 0; a < MS; a++) {
                double v = 0.0;
#pragma unroll
                for (int j = 0; j < A; j++)
                    if (a < m && j == slot_col(cb, a)) v = F[j];
                x[a] = v - xbar[a];
            }
#pragma unroll
            for (int k = 0; k < K; k++) {
                double e = ys[k * n_pad + i] - ybar[k];
#pragma unroll
                for (int a = 0; a < MS; a++)
                    if (a < m) e -= beta[k][a] * x[a];
                ra[k] = fma(e, e, ra[k]);
            }
        });
#pragma unroll
        for (int k = 0; k < K; k++) rss[k] = warp_sum_fixed(ra[k]);
    }
    if (lane == 0) {
        const double dfe = nn - (double)(m + 1);
        for (int k = 0; k < K; k++) {
            const double ve = rss[k] / dfe;
            for (int b = 0; b < m; b++) {
                out[(b * K + k) * 2 + 0] = beta[k][b];
                out[(b * K + k) * 2 + 1] = ve * dg[b];
            }
        }
    }
    __syncwarp();
    return PG_LOCUS_OK;
}

// pearsons_correlation with missing values (src/gwas/correlation_test.rs:21-31) by the whole warp: for every
// phenotype the pools whose frequency OR phenotype is NaN are dropped pairwise, means and centred sums run over the
// remaining pools (so they differ per phenotype), n in the t statistic stays the full pool count.
template <int A, int K>
__device__ __noinline__ int corr_pairwise_locus(const ScanParams &p, int64_t locus, unsigned kept, int m, unsigned cb,
                                                const double *ys, double *out, int lane) {
    constexpr int MS = A - 1;
    const int n_pad = p.lay.n_pad;
    double xbar[K][MS], ybar[K];
    {
        double cnt[K], sx[K][MS], sy[K];
#pragma unroll
        for (int k = 0; k < K; k++) {
            cnt[k] = sy[k] = 0.0;
#pragma unroll
            for (int a = 0; a < MS; a++) sx[k][a] = 0.0;
        }
        for_rows_coop<A>(p, locus, lane, [&](int i, const double(&f)[A], uint32_t d) {
            double F[A], x[MS];
            renorm_row<A>(f, d, kept, F);
            bool xv = true;
#pragma unroll
            for (int a = 0; a < MS; a++) {
                double v = 0.0;
#pragma unroll
                for (int j = 0; j < A; j++)
                    if (a < m && j == slot_col(cb, a)) v = F[j];
                x[a] = v;
                xv &= (v == v);
            }
#pragma unroll
            for (int k = 0; k < K; k++) {
                const double y = ys[k * n_pad + i];
                if (xv && y == y) {
                    cnt[k] += 1.0;
                    sy[k] += y;
#pragma unroll
                    for (int a = 0; a < MS; a++) sx[k][a] += x[a];
                }
            }
        });
#pragma unroll
        for (int k = 0; k < K; k++) {
            const double c = warp_sum_fixed(cnt[k]);
            ybar[k] = warp_sum_fixed(sy[k]) / c;
#pragma unroll
            for (int a = 0; a < MS; a++) xbar[k][a] = warp_sum_fixed(sx[k][a]) / c;
        }
    }
    double sxx[K][MS], sxy[K][MS], syy[K];
#pragma unroll
    for (int k = 0; k < K; k++) {
        syy[k] = 0.0;
#pragma unroll
        for (int a = 0; a < MS; a++) sxx[k][a] = sxy[k][a] = 0.0;
    }
    for_rows_coop<A>(p, locus, lane, [&](int i, const double(&f)[A], uint32_t d) {
        double F[A], x[MS];
        renorm_row<A>(f, d, kept, F);
        bool xv = true;
#pragma unroll
        for (int a = 0; a < MS; a++) {
            double v = 0.0;
#pragma unroll
            for (int j = 0; j < A; j++)
                if (a < m && j == slot_col(cb, a)) v = F[j];
            x[a] = v;
            xv &= (v == v);
        }
#pragma unroll
        for (int k = 0; k < K; k++) {
            const double y = ys[k * n_pad + i];
            if (xv && y == y) {
                const double dy = y - ybar[k];
                syy[k] = fma(dy, dy, syy[k]);
#pragma unroll
                for (int a = 0; a < MS; a++) {
                    const double dx = x[a] - xbar[k][a];
                    sxx[k][a] = fma(dx, dx, sxx[k][a]);
                    sxy[k][a] = fma(dx, dy, sxy[k][a]);
                }
            }
        }
    });
#pragma unroll
    for (int k = 0; k < K; k++) {
        const double yy = warp_sum_fixed(syy[k]);
#pragma unroll
        for (int a = 0; a < MS; a++) {
            const double xx = warp_sum_fixed(sxx[k][a]), xy = warp_sum_fixed(sxy[k][a]);
            if (lane == 0 && a < m) {
                out[(a * K + k) * 2 + 0] = xy / (sqrt(xx) * sqrt(yy));
                out[(a * K + k) * 2 + 1] = 0.0;
            }
        }
    }
    __syncwarp();
    return PG_LOCUS_OK;
}

// Fewer pools than coefficients (n < p_x = 1 + m, i.e. at most 5 pools): the reference's other branch,
// b = X'(XX')^-1 y and var = ve diag(X'(XX')^-2 X) with ve = e'e / (n - p_x) (src/gwas/ols.rs:67-75, 106-111).  The fit
// interpolates, so e'e is rounding noise over a NEGATIVE n - p_x: var is a tiny negative number (t = NaN, p forced to 1,
// ols.rs:150-151) or -0 when every residual is exactly zero (t = +-inf, p = 0) -- both fall out of the same arithmetic
// in write_records.  LU with partial pivoting in dgetf2's order, so an exactly singular XX' (two pools with the same
// frequencies) fails like the reference's inv().  Whole warp, every lane computes the same numbers (n <= 5);
// lane 0 leaves (beta, var) per (slot, phenotype) in out.  ys holds the CENTRED phenotypes; the raw ones are ys + mean.
template <int A, int K>
__device__ __noinline__ int minnorm_locus(const ScanParams &p, int64_t locus, unsigned kept, int m, unsigned cb,
                                          const double *ys, double *out, int lane) {
    constexpr int MS = A - 1, PX = A, NR = 5;
    const int n = p.lay.n, n_pad = p.lay.n_pad, px = m + 1;
    double xrow[PX];
#pragma unroll
    for (int c = 0; c < PX; c++) xrow[c] = 0.0;
    for_rows_coop<A>(p, locus, lane, [&](int i, const double(&f)[A], uint32_t d) {
        double F[A];
        renorm_row<A>(f, d, kept, F);
        xrow[0] = 1.0;
#pragma unroll
        for (int a = 0; a < MS; a++) {
            double v = 0.0;
#pragma unroll
            for (int j = 0; j < A; j++)
                if (a < m && j == slot_col(cb, a)) v = F[j];
            xrow[1 + a] = v;
        }
    });
    double X[NR][PX], Y[NR][K];
#pragma unroll
    for (int i = 0; i < NR; i++) {
#pragma unroll
        for (int c = 0; c < PX; c++) X[i][c] = __shfl_sync(PG_FULL_MASK, xrow[c], i);
#pragma unroll
        for (int k = 0; k < K; k++) Y[i][k] = (i < n) ? ys[k * n_pad + i] + p.ymean[k] : 0.0;
    }
    // M = X X' (n x n); rows / columns >= n form an identity block
    double M[NR][NR];
#pragma unroll
    for (int i = 0; i < NR; i++)
#pragma unroll
        for (int j = 0; j < NR; j++) {
            double s = 0.0;
#pragma unroll
            for (int c = 0; c < PX; c++)
                if (c < px) s += X[i][c] * X[j][c];
            M[i][j] = (i < n && j < n) ? s : (i == j ? 1.0 : 0.0);
        }
    // right-hand sides: the K phenotypes, then the MS regressor columns of X (for diag(X'(XX')^-2 X))
    constexpr int NB = K + MS;
    double B[NR][NB];
#pragma unroll
    for (int i = 0; i < NR; i++) {
#pragma unroll
        for (int k = 0; k < K; k++) B[i][k] = Y[i][k];
#pragma unroll
        for (int a = 0; a < MS; a++) B[i][K + a] = (i < n) ? X[i][1 + a] : 0.0;
    }
    // Gaussian elimination with partial pivoting (first largest |a_ij| of the column, like idamax)
    bool singular = false;
#pragma unroll
    for (int j = 0; j < NR; j++) {
        int jp = j;
        double amax = fabs(M[j][j]);
#pragma unroll
        for (int i = j + 1; i < NR; i++) {
            const double v = fabs(M[i][j]);
            if (v > amax) {
                amax = v;
                jp = i;
            }
        }
#pragma unroll
        for (int i = j + 1; i < NR; i++)
            if (i == jp) {
#pragma unroll
                for (int c = 0; c < NR; c++) {
                    const double t = M[j][c];
                    M[j][c] = M[i][c];
                    M[i][c] = t;
                }
#pragma unroll
                for (int c = 0; c < NB; c++) {
                    const double t = B[j][c];
                    B[j][c] = B[i][c];
                    B[i][c] = t;
                }
            }
        if (!(fabs(M[j][j]) > 0.0)) {
            singular = true;
            M[j][j] = 1.0;
        }
        const double r = 1.0 / M[j][j];
#pragma unroll
        for (int i = j + 1; i < NR; i++) {
            const double l = M[i][j] * r;
#pragma unroll
            for (int c = j + 1; c < NR; c++) M[i][c] -= l * M[j][c];
#pragma unroll
            for (int c = 0; c < NB; c++) B[i][c] -= l * B[j][c];
        }
    }
    if (singular) return PG_LOCUS_FAILED;
#pragma unroll
    for (int j = NR - 1; j >= 0; j--) {
#pragma unroll
        for (int c = 0; c < NB; c++) {
            double s = B[j][c];
#pragma unroll
            for (int i = j + 1; i < NR; i++) s -= M[j][i] * B[i][c];
            B[j][c] = s / M[j][j];
        }
    }
    // B[:, k] = (XX')^-1 y_k, B[:, K + a] = (XX')^-1 x_a
    const double dfe = (double)n - (double)px;  // negative
    if (lane == 0) {
        for (int k = 0; k < K; k++) {
            double b[PX];
            for (int c = 0; c < PX; c++) {
                double s = 0.0;
                for (int i = 0; i < NR; i++)
                    if (i < n && c < px) s += X[i][c] * B[i][k];
                b[c] = s;
            }
            double ee = 0.0;
            for (int i = 0; i < NR; i++)
                if (i < n) {
                    double e = Y[i][k];
                    for (int c = 0; c < PX; c++)
                        if (c < px) e -= X[i][c] * b[c];
                    ee += e * e;
                }
            const double ve = ee / dfe;
            for (int a = 0; a < MS; a++)
                if (a < m) {
                    double dd = 0.0;
                    for (int i = 0; i < NR; i++)
                        if (i < n) dd += B[i][K + a] * B[i][K + a];
                    out[(a * K + k) * 2 + 0] = b[1 + a];
                    out[(a * K + k) * 2 + 1] = ve * dd;
                }
        }
    }
    __syncwarp();
    return PG_LOCUS_OK;
}

// Single-pass OLS from the reduced sums for M regressors, fully unrolled so that every matrix lives in registers.
// Returns false when the centred X'X is not positive definite; sets redo when the single-pass form loses digits.
// m <= M regressors are present; the slots m..M-1 are an identity block with zero right-hand sides.  They only append
// exact zeros to the END of every sum, so the m present coefficients come out bit for bit as from the variant with
// M = m -- a warp whose loci disagree on m runs this once with M = A - 1 instead of one specialised variant per value.
template <int M, int A, int K, bool W>
__device__ __forceinline__ bool ols_gram_m(const ScanParams &p, double *tg, unsigned cb, double nn, bool &redo, int m) {
    using AC = Acc<A, K, W>;
    double tbg[2 * M * K];
    double sx[M], S[M][M], Lm[M][M], Li[M][M], dg[M], rinv[M];
    int c[M];
#pragma unroll
    for (int a = 0; a < M; a++) {
        c[a] = slot_col(cb, a);
        sx[a] = (a < m) ? tg[AC::S0 + c[a]] : 0.0;
    }
    const double inv_n = p.inv_n;
    double amp = 1.0;
#pragma unroll
    for (int a = 0; a < M; a++)
#pragma unroll
        for (int b = 0; b <= a; b++) {
            const int lo = c[a] < c[b] ? c[a] : c[b], hi = c[a] < c[b] ? c[b] : c[a];
            const double raw = tg[AC::P0 + lo * A - lo * (lo - 1) / 2 + (hi - lo)];
            S[a][b] = (a < m) ? raw - sx[a] * sx[b] * inv_n : (a == b ? 1.0 : 0.0);
            if (a == b && a < m) amp = fmax(amp, raw / S[a][a]);
        }
    bool ok = true;
#pragma unroll
    for (int a = 0; a < M; a++)
#pragma unroll
        for (int b = 0; b <= a; b++) {
            double v = S[a][b];
#pragma unroll
            for (int q = 0; q < b; q++) v -= Lm[a][q] * Lm[b][q];
            if (a == b) {
                if (!(v > 0.0)) {
                    ok = false;
                    v = 1.0;
                }
                rinv[a] = rsqrt(v);  // 1 / L_aa in one step (1 ulp): the pivot's sqrt + division left the chain
            } else {
                Lm[a][b] = v * rinv[b];
            }
        }
#pragma unroll
    for (int a = 0; a < M; a++) {
        Li[a][a] = rinv[a];
#pragma unroll
        for (int b = 0; b < a; b++) {
            double v = 0.0;
#pragma unroll
            for (int q = b; q < a; q++) v -= Lm[a][q] * Li[q][b];
            Li[a][b] = v * rinv[a];
        }
    }
    double vif = 1.0;
#pragma unroll
    for (int b = 0; b < M; b++) {
        double v = 0.0;
#pragma unroll
        for (int a = b; a < M; a++) v += Li[a][b] * Li[a][b];
        dg[b] = v;
        vif = fmax(vif, S[b][b] * v);
    }
    redo = !ok || !(amp > 0.0);
    if (!ok) return false;
    const double inv_dfe = 1.0 / (nn - (double)(m + 1));
    const bool saturated = !(nn - (double)(m + 1) > 0.0);
#pragma unroll
    for (int k = 0; k < K; k++) {
        double z[M], zz = 0.0;
        const double ys_n = p.ysum[k] * inv_n;
#pragma unroll
        for (int a = 0; a < M; a++) {
            double v = 0.0;
#pragma unroll
            for (int b = 0; b <= a; b++) v += Li[a][b] * ((b < m) ? tg[AC::C0 + c[b] * K + k] - sx[b] * ys_n : 0.0);
            z[a] = v;
            zz += v * v;
        }
        double rss = p.syy[k] - zz;
        // digits lost by the single-pass form: centring (amp), collinearity (vif) and syy - zz
        if (!(64.0 * kEps * (amp * vif * zz + p.syy[k]) <= 1e-10 * rss)) redo = true;
        if (rss < 0.0) rss = 0.0;
        const double ve = saturated ? rss / (nn - (double)(m + 1)) : rss * inv_dfe;
#pragma unroll
        for (int b = 0; b < M; b++) {
            double v = 0.0;
#pragma unroll
            for (int a = b; a < M; a++) v += Li[a][b] * z[a];
            tbg[(b * K + k) * 2 + 0] = v;
            tbg[(b * K + k) * 2 + 1] = ve * dg[b];
        }
    }
#pragma unroll
    for (int i = 0; i < 2 * M * K; i++) tg[i] = tbg[i];  // every total has been read: the row now holds the results
    return true;
}

// ---- phase 2b (one lane per locus): allele order and the single-pass solve, everything in registers ------------
// in: the totals row tg of the locus.  out: m (rows), cb (allele column of each row, 4 bits per slot), redo (REDO_*)
// and, in place of the totals, tg[(s*K+k)*2 + {0,1}] = (beta | r, var) and tg[2(A-1)K + s] = mean frequency.
template <int A, int K, bool W, bool DEFER, int KIND>
__device__ __noinline__ void solve_locus(const ScanParams &p, int64_t locus, double *tg, int &status, unsigned kept,
                                         int &m, unsigned &cb, int &redo_mode) {
    using AC = Acc<A, K, W>;
    constexpr int T2 = 2 * (A - 1) * K;
    static_assert(T2 + A - 1 <= AC::NP, "the results of a locus must fit its totals row");
    double fmean[A - 1];
#pragma unroll
    for (int a = 0; a < A - 1; a++) fmean[a] = nan("");
    const Layout &lay = p.lay;
    const double nn = (double)lay.n;
    const double tol_rel = 2.0 * (nn + 8.0) * kEps;
    m = __popc(kept) - 1;
    cb = 0;
    if (kind_is_ols<KIND>(p)) {
        // stable sort by decreasing column sum, drop the first (major) allele (sync.rs:478-505, ols.rs:227-230)
        double cs[A];
        bool tie = false;
#pragma unroll
        for (int j = 0; j < A; j++) cs[j] = tg[AC::S0 + j];
#pragma unroll
        for (int j = 0; j < A; j++)
#pragma unroll
            for (int l = j + 1; l < A; l++)
                if (((kept >> j) & 1u) && ((kept >> l) & 1u) &&
                    fabs(cs[j] - cs[l]) <= tol_rel * fmax(fabs(cs[j]), fabs(cs[l])))
                    tie = true;
        if (tie) {
            if constexpr (DEFER) {  // the streaming kernel leaves exact evaluations to the fix-up kernel
                redo_mode = REDO_DEFER;
                return;
            } else {
#pragma unroll
                for (int j = 0; j < A; j++)
                    if ((kept >> j) & 1u) cs[j] = exact_colsum<A>(p, locus, j, kept);
            }
        }
#pragma unroll
        for (int j = 0; j < A; j++) {
            if (!((kept >> j) & 1u)) continue;
            int rank = 0;
#pragma unroll
            for (int l = 0; l < A; l++) {
                if (l == j || !((kept >> l) & 1u)) continue;
                if (cs[l] > cs[j] || (cs[l] == cs[j] && l < j)) rank++;
            }
            if (rank >= 1) cb |= (unsigned)j << (4 * (rank - 1));
            else cb |= (unsigned)j << 20;  // the major allele (dropped from the regressors; mle_iter / gwalpha need it)
        }
    } else {
        // kept columns in file order, the last one is dropped (correlation_test.rs:94-98)
        int sidx = 0;
#pragma unroll
        for (int j = 0; j < A; j++) {
            if (!((kept >> j) & 1u)) continue;
            if (sidx < m) cb |= (unsigned)j << (4 * sidx);
            sidx++;
        }
    }
    bool has_nan = false;
#pragma unroll
    for (int a = 0; a < A - 1; a++) {
        if (a < m) {
            const int c = slot_col(cb, a);
            const double pjj = tg[AC::P0 + c * A - c * (c - 1) / 2];
            has_nan |= (pjj != pjj);
            fmean[a] = (pjj != pjj) ? nan("") : tg[AC::S0 + c] / nn;
        }
    }
    if (kind_is_ols<KIND>(p)) {
        if (p.filter_only) {
            // mle_iter / gwalpha: only the keep-mask, the allele order and the mean frequencies are wanted here; the
            // statistics come from the Nelder-Mead kernels (pg_nm.cu)
        } else if (has_nan) {
            for (int i = 0; i < T2; i++) tg[i] = nan("");
        } else if (lay.n < m + 1) {
            // fewer pools than coefficients: the minimum-norm branch (src/gwas/ols.rs:67-75), left to the fix-up kernel
            redo_mode = REDO_MINNORM;
        } else {
            bool redo = false;
            // the lanes that got here agree on m (real data: nearly always biallelic) -> the variant of that size;
            // otherwise ONE pass of the full-size variant with masked slots instead of a pass per distinct m
            const unsigned here = __activemask();
            const bool uniform = __match_any_sync(here, m) == here;
            if (!uniform || m >= A - 1) {
                ols_gram_m<A - 1, A, K, W>(p, tg, cb, nn, redo, m);
            } else {
                switch (m) {  // m < A - 1, every variant is instantiated once
                    case 1:
                        if constexpr (A >= 3) ols_gram_m<1, A, K, W>(p, tg, cb, nn, redo, 1);
                        break;
                    case 2:
                        if constexpr (A >= 4) ols_gram_m<2, A, K, W>(p, tg, cb, nn, redo, 2);
                        break;
                    case 3:
                        if constexpr (A >= 5) ols_gram_m<3, A, K, W>(p, tg, cb, nn, redo, 3);
                        break;
                    default:
                        if constexpr (A >= 6) ols_gram_m<4, A, K, W>(p, tg, cb, nn, redo, 4);
                        break;
                }
            }
            if (redo) redo_mode = REDO_OLS;
        }
    } else {
        double tb[T2];
#pragma unroll
        for (int i = 0; i < T2; i++) tb[i] = nan("");
        bool redo = false;
#pragma unroll
        for (int a = 0; a < A - 1; a++) {
            if (a < m) {
                const int c = slot_col(cb, a);
                const double sxa = tg[AC::S0 + c];
                const double raw = tg[AC::P0 + c * A - c * (c - 1) / 2];
                const double sxx = raw - sxa * sxa * p.inv_n;
                if (!(raw <= 1e6 * sxx)) redo = true;  // up to 6 of 16 digits lost by the single-pass form: r keeps 1e-10
#pragma unroll
                for (int k = 0; k < K; k++) {
                    const double sxy = tg[AC::C0 + c * K + k] - sxa * (p.ysum[k] * p.inv_n);
                    const double r = sxy / (sqrt(sxx) * sqrt(p.syy[k]));
                    tb[(a * K + k) * 2 + 0] = r;
                    tb[(a * K + k) * 2 + 1] = 0.0;
                    // t = r / sqrt((1 - r^2) / (n - 2)) carries the error of r times r^2 / (1 - r^2): near a perfect
                    // correlation (a handful of pools) the digits the single-pass form loses reach the p-value
                    if (!(16.0 * kEps * raw <= 1e-8 * (1.0 - r * r) * sxx)) redo = true;
                }
            }
        }
        if (has_nan || p.y_has_nan)
            redo_mode = REDO_CORR_NAN;
        else if (redo)
            redo_mode = REDO_CORR;
#pragma unroll
        for (int i = 0; i < T2; i++) tg[i] = tb[i];
    }
#pragma unroll
    for (int a = 0; a < A - 1; a++) tg[T2 + a] = fmean[a];
}

// two-sided Student-t p-values of K statistics at once: the table loads of all K are in flight together
template <int K>
__device__ __forceinline__ void student_batch(const ScanParams &p, const PTableDev &tab, const double (&t_abs)[K],
                                              const bool (&need)[K], double (&pv)[K]) {
    if (!tab.coef) {
#pragma unroll
        for (int k = 0; k < K; k++)
            if (need[k]) pv[k] = student_two_sided(t_abs[k], p.df, p.ln_beta);
        return;
    }
    double s[K];
    const double2 *cp[K];
    bool in[K];
    const int B = (int)tab.bits;
#pragma unroll
    for (int k = 0; k < K; k++) {
        const double ta = need[k] ? t_abs[k] : 0.0;
        const double w = fma(ta, tab.inv_sqrt_df, 1.0);
        int i = ptab_locate(w, B, s[k]);
        // statrs' cut-offs (student_two_sided_tab): p = 0 from t_zero on (w is finite below it)
        in[k] = need[k] && (ta < tab.t_zero) && (i < tab.M);
        if (!in[k]) i = 0;
        cp[k] = reinterpret_cast<const double2 *>(tab.coef + i);
    }
    double2 c01[K], c23[K];
#pragma unroll
    for (int k = 0; k < K; k++) {
        c01[k] = __ldg(cp[k]);
        c23[k] = __ldg(cp[k] + 1);
    }
#pragma unroll
    for (int k = 0; k < K; k++) {
        const double ptrue = in[k] ? exp(fma(s[k], fma(s[k], fma(s[k], c23[k].y, c23[k].x), c01[k].y), c01[k].x)) : 0.0;
        const double ib = 0.5 * ptrue;
        // the reference's 2 * (1 - (1 - ib)) quantisation; p = 1 up to t_one (t = 0 included)
        const double cdf = t_abs[k] <= tab.t_one ? 0.5 : 1.0 - ib;
        if (need[k]) pv[k] = 2.0 * (1.0 - cdf);
    }
}

// ---- phase 2c (one lane per locus): t, p and the records ----------------------------------------------------------
template <int A, int K, int KIND>
__device__ __noinline__ void write_records(const ScanParams &p, const PTableDev &tab, int64_t locus, int status,
                                           int m, unsigned cb, const double *tb) {
    constexpr int T2 = 2 * (A - 1) * K;
    if (p.write_meta) {
        uint64_t mv = (uint64_t)status;
        if (status == PG_LOCUS_OK) {
            mv |= (uint64_t)m << 8;
#pragma unroll
            for (int s = 0; s < A - 1; s++)
                if (s < m) mv |= (uint64_t)p.codes[slot_col(cb, s)] << (16 + 8 * s);
            // the byte after the output rows' codes: the major allele (ols_iter; read by the Nelder-Mead kernels only)
            if (kind_is_ols<KIND>(p) && m < 6) mv |= (uint64_t)p.codes[(cb >> 20) & 0xfu] << (16 + 8 * m);
        }
        p.meta[locus] = mv;
#pragma unroll
        for (int s = 0; s < A - 1; s++)
            p.freq_mean[(size_t)locus * (A - 1) + s] = (status == PG_LOCUS_OK && s < m) ? tb[T2 + s] : nan("");
    }
#pragma unroll 1
    for (int s = 0; s < A - 1; s++) {
        const bool valid = status == PG_LOCUS_OK && s < m;
        double o0[K], o1[K], o2[K], o3[K], ta[K];
        bool need[K];
#pragma unroll
        for (int k = 0; k < K; k++) {
            const double v0 = valid ? tb[(s * K + k) * 2 + 0] : 0.0, v1 = valid ? tb[(s * K + k) * 2 + 1] : 0.0;
            o0[k] = o1[k] = o2[k] = o3[k] = nan("");
            need[k] = false;
            ta[k] = 0.0;
            if (valid) {
                if (kind_is_ols<KIND>(p)) {
                    // estimate_significance, src/gwas/ols.rs:139-154
                    const double se = sqrt(v1);
                    const double tt = (fabs(v0) <= kEps) ? 0.0 : v0 * rsqrt(v1);  // b / sqrt(var) off the sqrt's chain
                    o0[k] = v0;
                    o1[k] = se;
                    o2[k] = tt;
                    if (fabs(tt) <= kEps || tt != tt) {
                        o3[k] = 1.0;
                    } else {
                        need[k] = true;
                        ta[k] = fabs(tt);
                    }
                } else {
                    // pearsons_correlation, src/gwas/correlation_test.rs:52-70
                    const double r = v0;
                    if (r == r) {
                        const double s2 = (1.0 - r * r) * p.inv_nm2;  // the sign is that of 1 - r^2 either way
                        o1[k] = r;
                        if (s2 <= 0.0) {
                            o0[k] = r;
                            o3[k] = kEps;
                        } else {
                            const double tt = r * rsqrt(s2);
                            o2[k] = tt;
                            o0[k] = round(r * 1e7) / 1e7;
                            if (p.lay.n > 2) {
                                need[k] = true;
                                ta[k] = fabs(tt);
                            }
                        }
                    }
                }
            }
        }
        student_batch<K>(p, tab, ta, need, o3);
#pragma unroll
        for (int k = 0; k < K; k++) {
            double *o = p.stats + (((size_t)locus * (A - 1) + s) * p.k_total + p.phen_base + k) * 4;
            *reinterpret_cast<double2 *>(o) = make_double2(o0[k], o1[k]);
            *reinterpret_cast<double2 *>(o + 2) = make_double2(o2[k], o3[k]);
        }
    }
}

// ---- phase 2 (lane = locus of the block): keep-mask from the totals, solve, records -----------------------------
// DEFER = true (the streaming kernel): loci that need an exact re-evaluation (a threshold hit within rounding, tied
// column sums), the renormalised frequencies (a removed allele carries reads, a pool has no coverage) or the two-pass
// form are appended to the batch's fix-up list and left to fixup_kernel -- none of that code is linked into the
// streaming kernel, whose instruction footprint has to stay inside the instruction cache.
// DEFER = false (the fix-up kernel): the whole warp works on those paths.
// locus / act / dm are per lane; pre_kept != 0 (fix-up kernel only) says that the row already holds the totals of the
// renormalised frequencies over that kept set.
template <int A, int K, bool W, bool DEFER, int KIND>
__device__ __noinline__ void epilogue(const ScanParams &p, int64_t locus, bool act, double *tot, const double *ys,
                                      const double *ws, int lane, unsigned dm, unsigned pre_kept) {
    using AC = Acc<A, K, W>;
    const PTableDev ptab = {reinterpret_cast<const double4 *>(p.ptab), p.ptab_isd, p.ptab_bits, p.ptab_t1, p.ptab_t0, p.ptab_M};
    double *tg = tot + (size_t)lane * AC::NP;
    const double tol_rel = 2.0 * ((double)p.lay.n + 8.0) * kEps;
    int status = PG_LOCUS_FILTERED;
    unsigned kept = 0, exact_bits = 0;
    bool slow = false, slow_decide = false;
    double q[A];
#pragma unroll
    for (int j = 0; j < A; j++) q[j] = 0.0;
    bool deferred = false, kept_known = false;
    if (act && pre_kept) {
        status = PG_LOCUS_OK;
        kept = pre_kept;
        if (DEFER) {
            // streaming kernel under an ingest hint: the totals are those of the renormalised frequencies.  A pool
            // without reads on the kept alleles made them NaN -- the NaN-aware accumulation is the fix-up kernel's
            kept_known = true;
#pragma unroll
            for (int j = 0; j < A; j++)
                if (((kept >> j) & 1u) && tg[AC::S0 + j] != tg[AC::S0 + j]) deferred = true;
        }
    } else if (act) {
        if ((double)dm < p.min_depth_f) {
            status = PG_LOCUS_FILTERED;  // sync.rs:217-229
        } else if (dm == 0u) {
            status = PG_LOCUS_OK;  // a pool without coverage: NaN frequencies, decided on the slow path
            slow = slow_decide = true;
        } else {
            status = PG_LOCUS_OK;
#pragma unroll
            for (int j = 0; j < A; j++) {
                q[j] = W ? tg[AC::Q0 + j] : tg[AC::S0 + j] * p.w_uniform;
                const double tl = tol_rel * fmax(fabs(q[j]), 1.0);
                if (fabs(q[j] - p.maf) <= tl || fabs(q[j] - p.one_minus_maf) <= tl) exact_bits |= 1u << j;
            }
        }
    }
    if (DEFER) {
        if (exact_bits != 0u) deferred = true;
    } else {
        // thresholds hit within rounding: lane j re-evaluates q_j of that locus in the reference's order
        unsigned need = __ballot_sync(PG_FULL_MASK, exact_bits != 0u);
        while (need) {
            const int src = __ffs(need) - 1;
            need &= need - 1;
            const unsigned bits = __shfl_sync(PG_FULL_MASK, exact_bits, src);
            const int64_t lsrc = __shfl_sync(PG_FULL_MASK, locus, src);
#pragma unroll
            for (int j = 0; j < A; j++) {
                if (!((bits >> j) & 1u)) continue;  // warp-uniform: bits was broadcast
                const double v = exact_q(p, lsrc, j, ws, lane);
                if (lane == src) q[j] = v;
            }
        }
    }
    if (act && status == PG_LOCUS_OK && !slow && !deferred && !pre_kept) {
#pragma unroll
        for (int j = 0; j < A; j++)
            if (!((q[j] < p.maf) | (q[j] > p.one_minus_maf))) kept |= 1u << j;
        if (__popc(kept) < 2) {
            status = PG_LOCUS_FILTERED;  // sync.rs:284-286
        } else {
#pragma unroll
            for (int j = 0; j < A; j++)
                if (!((kept >> j) & 1u) && tg[AC::S0 + j] > 0.0) slow = true;  // a removed allele carries reads
        }
    }
    if (DEFER) {
        if (act && slow && status == PG_LOCUS_OK) {
            kept_known = !deferred && !slow_decide;  // the fix-up kernel can renormalise right away
            deferred = true;
        }
    } else {
        unsigned need = __ballot_sync(PG_FULL_MASK, act && slow && status == PG_LOCUS_OK);
        while (need) {
            const int src = __ffs(need) - 1;
            need &= need - 1;
            const bool dec = __shfl_sync(PG_FULL_MASK, (int)slow_decide, src) != 0;
            unsigned kk = __shfl_sync(PG_FULL_MASK, kept, src);
            const int64_t lsrc = __shfl_sync(PG_FULL_MASK, locus, src);
            const int st = slow_locus<A, K, W>(p, lsrc, ys, ws, tot + (size_t)src * AC::NP, lane, dec, kk);
            if (lane == src) {
                status = st;
                kept = kk;
            }
        }
        __syncwarp();
    }
    int m = 0, redo_mode = REDO_NONE;
    unsigned cb = 0;
    if (act && status == PG_LOCUS_OK && !deferred)
        solve_locus<A, K, W, DEFER, KIND>(p, locus, tg, status, kept, m, cb, redo_mode);
    if (DEFER) {
        // why (bits 56.., read only by the PG_REPORT_DEFER diagnostic): 1 threshold within rounding, 2 removed allele
        // with reads and no hint, 4 pool without coverage, 8 NaN under a hint, 16.. the redo mode
        uint64_t why = (exact_bits != 0u ? 1u : 0u) | ((slow && !slow_decide) ? 2u : 0u) | (slow_decide ? 4u : 0u) |
                       ((deferred && pre_kept) ? 8u : 0u);
        if (redo_mode != REDO_NONE) {
            deferred = true;
            why |= (uint64_t)redo_mode << 4;
        }
        if (deferred)
            p.defer_list[atomicAdd(p.defer_count, 1u)] =
                (uint64_t)locus | (kept_known ? ((uint64_t)kept << 40) : 0ull) | (why << 56);
    } else {
        // loci whose single-pass form is not trustworthy: explicit two-pass evaluation by the whole warp
        unsigned need = __ballot_sync(PG_FULL_MASK, redo_mode != REDO_NONE);
        while (need) {
            const int src = __ffs(need) - 1;
            need &= need - 1;
            const int md = __shfl_sync(PG_FULL_MASK, redo_mode, src);
            const unsigned kk = __shfl_sync(PG_FULL_MASK, kept, src);
            const int mm = __shfl_sync(PG_FULL_MASK, m, src);
            const unsigned cc = __shfl_sync(PG_FULL_MASK, cb, src);
            const int64_t lsrc = __shfl_sync(PG_FULL_MASK, locus, src);
            __syncwarp();
            const int st = (md == REDO_CORR_NAN)
                               ? corr_pairwise_locus<A, K>(p, lsrc, kk, mm, cc, ys, tot + (size_t)src * AC::NP, lane)
                           : (md == REDO_MINNORM)
                               ? minnorm_locus<A, K>(p, lsrc, kk, mm, cc, ys, tot + (size_t)src * AC::NP, lane)
                               : redo_locus<A, K>(p, lsrc, kk, mm, cc, md, ys, tot + (size_t)src * AC::NP, lane);
            if (lane == src) status = st;
        }
        __syncwarp();
    }
    if (act && !deferred) write_records<A, K, KIND>(p, ptab, locus, status, m, cb, tg);
    __syncwarp();
}

// ---- the fix-up kernel: a warp takes 32 deferred loci, accumulates each straight from global memory (lane = pool:
// the renormalised frequencies when the kept set is already known, else the first-stage frequencies like phase 1) and
// runs the full phase 2 with lane = locus -----------------------------------------------------------------------
constexpr int kFixWarps = 8;

template <int A, int K, bool W>
__global__ void __launch_bounds__(kFixWarps * 32) fixup_kernel(const __grid_constant__ ScanParams p) {
    using AC = Acc<A, K, W>;
    extern __shared__ __align__(16) unsigned char fsm[];  // totals [2][32][NP]: accumulate block i+1 during phase 2 of i
    __shared__ __align__(16) ScanParams sp_storage;
    for (int i = threadIdx.x; i < (int)(sizeof(ScanParams) / 4); i += blockDim.x)
        reinterpret_cast<uint32_t *>(&sp_storage)[i] = reinterpret_cast<const uint32_t *>(&p)[i];
    __syncthreads();
    const ScanParams &sp = sp_storage;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t count = *p.defer_count;
    const int n_pad = p.lay.n_pad;
    const double *ys = p.yc;  // the slow paths index [k * n_pad + pool]: global memory serves as well as shared
    const double *ws = W ? p.w : nullptr;
    // loci per block: 32 when the list is long; when it is short the loci are spread over the CTAs of the grid, because
    // the warp-cooperative exact paths of phase 2 handle the loci of a block one after the other (a handful of loci in
    // one block would cost their summed latency at the end of every step, with the rest of the GPU idle)
    const uint32_t per_blk = min(32u, max(1u, (count + gridDim.x - 1) / gridDim.x));
    const uint32_t n_blocks = (count + per_blk - 1) / per_blk;
    int it = 0;
    for (uint32_t blk = blockIdx.x; blk < n_blocks; blk += gridDim.x, it++) {
        double *tot = reinterpret_cast<double *>(fsm) + (size_t)(it & 1) * 32 * AC::NP;
        const uint32_t e0 = blk * per_blk;
        const int cnt = (int)min(per_blk, count - e0);
        for (int g = warp; g < cnt; g += kFixWarps) {  // the loci of the block are dealt over the warps
            const uint64_t e = p.defer_list[e0 + g];
            const int64_t locus = (int64_t)(e & 0xFFFFFFFFFFull);
            const unsigned kept = (unsigned)(e >> 40) & 0x3fu;
            double acc[AC::N];
#pragma unroll
            for (int a = 0; a < AC::N; a++) acc[a] = 0.0;
            if (kept) {
                for_rows_coop<A>(sp, locus, lane, [&](int r, const double(&f)[A], uint32_t d) {
                    double F[A], y[K];
                    renorm_row_fast<A>(f, d, kept, F);
#pragma unroll
                    for (int k = 0; k < K; k++) y[k] = ys[k * n_pad + r];
                    accum_row<A, K, W, true>(acc, F, y, 0.0);
                });
            } else {
                for_rows_coop<A>(sp, locus, lane, [&](int r, const double(&f)[A], uint32_t) {
                    double y[K];
#pragma unroll
                    for (int k = 0; k < K; k++) y[k] = ys[k * n_pad + r];
                    accum_row<A, K, W, false>(acc, f, y, W ? ws[r] : 0.0);
                });
            }
#pragma unroll
            for (int a = 0; a < AC::N; a++) {
                const double v = warp_sum_fixed(acc[a]);
                if (lane == 0) tot[(size_t)g * AC::NP + a] = v;
            }
        }
        __syncthreads();  // the block's rows are complete; phase 2 of the block two back (same buffer) has finished
        if (warp == (it % kFixWarps)) {
            const uint64_t mine = (lane < cnt) ? p.defer_list[e0 + lane] : 0ull;
            const int64_t locus = (int64_t)(mine & 0xFFFFFFFFFFull);
            const unsigned dm = (lane < cnt) ? __ldg(p.dmin + locus) : 0xFFFFFFFFu;
            epilogue<A, K, W, false, -1>(sp, locus, lane < cnt, tot, ys, ws, lane, dm, (unsigned)(mine >> 40) & 0x3fu);
        }
    }
}

// ---- the kernel ----------------------------------------------------------------------------------------------
template <int A, int K, bool W, int P, int KIND>
__global__ void __launch_bounds__(kScanWarps * 32, 1) scan_kernel(const __grid_constant__ ScanParams p) {
    using AC = Acc<A, K, W>;
    constexpr int LPS = 32 / P;  // loci per stage
    constexpr int RC = chunk_rows(A);
    extern __shared__ __align__(128) unsigned char smem[];
    // the out-of-line phase-2 functions take the parameter block by reference: give them a shared-memory copy
    // (a reference to the kernel parameter itself would be spilled to per-thread local memory)
    __shared__ __align__(16) ScanParams sp_storage;
    for (int i = threadIdx.x; i < (int)(sizeof(ScanParams) / 4); i += blockDim.x)
        reinterpret_cast<uint32_t *>(&sp_storage)[i] = reinterpret_cast<const uint32_t *>(&p)[i];
    const ScanParams &sp = sp_storage;
    const Layout lay = p.lay;
    const int n_pad = lay.n_pad;
    const int G = p.block_loci;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
    double *ys = reinterpret_cast<double *>(smem);
    double *ws = W ? ys + (size_t)K * n_pad : nullptr;
    unsigned char *wb = smem + p.common_bytes + (size_t)warp * p.warp_bytes;
    uint64_t *bars = reinterpret_cast<uint64_t *>(wb);
    unsigned char *stage0 = wb + 64;
    double *tot = reinterpret_cast<double *>(stage0 + (size_t)p.nbuf * p.stage_bytes);
    const int nbuf = p.nbuf;
    const int red_rows = max(1, min((int)(p.stage_bytes / (kRedPitch * 8)), AC::N));  // launch_scan_p keeps a stage >= one row

    for (int i = threadIdx.x; i < K * n_pad; i += blockDim.x) ys[i] = p.yc[i];
    if (W)
        for (int i = threadIdx.x; i < n_pad; i += blockDim.x) ws[i] = p.w[i];
    if (lane == 0) {
        for (int b = 0; b < nbuf; b++) mbar_init(&bars[b], 1);
        fence_mbar_init();
    }
    __syncthreads();

    const int64_t L = p.n_loci;
    const int64_t NB = (L + G - 1) / G;
    const int64_t gw = (int64_t)blockIdx.x * nwarps + warp;  // consecutive warps take consecutive blocks
    const int64_t TW = (int64_t)gridDim.x * nwarps;
    if (gw >= NB) return;
    const int n_chunks = lay.n_chunks;
    const size_t fstride = lay.freq_stride();
    const uint32_t full_bytes = (uint32_t)(A * lay.rc * 8), last_bytes = (uint32_t)(A * lay.rc_last * 8);
    const uint32_t locus_bytes = (uint32_t)(fstride * 8);

    // producer side of the ring: the stages of a block are one contiguous walk through the frequency matrix
    int64_t i_blk = gw;
    const unsigned char *i_src = reinterpret_cast<const unsigned char *>(p.freq + (size_t)(gw * G) * fstride);
    int i_left = (int)min((int64_t)G, L - gw * G);  // loci of the block not yet requested
    int i_chunk = 0;
    bool i_done = false;
    auto issue_next = [&](int b, bool scratch_used) {
        if (i_done) return;
        uint32_t bytes;
        int nl = 1;
        if (P == 32) {
            bytes = (i_chunk == n_chunks - 1) ? last_bytes : full_bytes;
        } else {
            nl = min(LPS, i_left);
            bytes = (uint32_t)nl * locus_bytes;
        }
        if (lane == 0) {
            if (scratch_used) fence_proxy_async();  // generic-proxy writes of the reduction before the async-proxy refill
            mbar_expect_tx(&bars[b], bytes);
            bulk_g2s(stage0 + (size_t)b * p.stage_bytes, i_src, bytes, &bars[b]);
        }
        i_src += bytes;
        if (P == 32) {
            if (++i_chunk == n_chunks) {
                i_chunk = 0;
                i_left--;
            }
        } else {
            i_left -= nl;
        }
        if (i_left == 0) {
            i_blk += TW;
            if (i_blk >= NB) {
                i_done = true;
            } else {
                i_src = reinterpret_cast<const unsigned char *>(p.freq + (size_t)(i_blk * G) * fstride);
                i_left = (int)min((int64_t)G, L - i_blk * G);
            }
        }
    };
    for (int b = 0; b < nbuf; b++) issue_next(b, false);

    int buf = 0;
    uint32_t parity = 0;
    // smallest depth (consumed by the epilogue) and ingest hint (pg_ingest.cu) of this lane's locus: the hint steers the
    // first stage of a block, so both are fetched one block ahead -- a block that starts by waiting for them exposes a
    // full global-memory latency per 32 loci (9 % of the stall samples at 100 pools)
    auto load_meta = [&](int64_t b, unsigned &dm_o, unsigned &hl_o) {
        const int64_t m0 = b * G;
        const bool in = b < NB && lane < (int)min((int64_t)G, L - m0);
        dm_o = in ? __ldg(p.dmin + m0 + lane) : 0xFFFFFFFFu;
        hl_o = in ? (unsigned)__ldg(p.hint + m0 + lane) : 0u;
    };
    unsigned dm_next, hl_next;
    load_meta(gw, dm_next, hl_next);
    for (int64_t blk = gw; blk < NB; blk += TW) {
        const int64_t l0 = blk * G;
        const int cnt = (int)min((int64_t)G, L - l0);
        const unsigned dm = dm_next, hl = hl_next;
        load_meta(blk + TW, dm_next, hl_next);
        if (P == 32) {
            for (int g = 0; g < cnt; g++) {
                const unsigned hk = __shfl_sync(PG_FULL_MASK, hl, g);
                const bool hinted = (hk & 0x80u) != 0u;
                const unsigned hkept = hk & 0x3fu;
                double acc[AC::N];
#pragma unroll
                for (int i = 0; i < AC::N; i++) acc[i] = 0.0;
                for (int chunk = 0; chunk < n_chunks; chunk++) {
                    const double *yrow = ys + chunk * RC + 2 * lane;
                    const double *wrow = W ? ws + chunk * RC + 2 * lane : nullptr;
                    mbar_wait(&bars[buf], parity);
                    double *fb = reinterpret_cast<double *>(stage0 + (size_t)buf * p.stage_bytes);
                    if (chunk < n_chunks - 1 || lay.rc_last == RC) {
                        const double *fl = fb + 2 * lane;
#pragma unroll
                        for (int it = 0; it < RC / 64; it++) {
                            double2 f2[A], y2[K];
#pragma unroll
                            for (int j = 0; j < A; j++) f2[j] = *reinterpret_cast<const double2 *>(fl + j * RC + it * 64);
#pragma unroll
                            for (int k = 0; k < K; k++)
                                y2[k] = *reinterpret_cast<const double2 *>(yrow + (size_t)k * n_pad + it * 64);
                            double2 w2 = make_double2(0.0, 0.0);
                            if (W) w2 = *reinterpret_cast<const double2 *>(wrow + it * 64);
                            if (hinted) renorm_pair<A>(f2, hkept, chunk * RC + it * 64 + 2 * lane, lay.n);
                            accum_pair<A, K, W>(acc, f2, y2, w2);
                        }
                    } else {
                        const int rcc = lay.rc_last;
                        for (int r = 2 * lane; r < rcc; r += 64) {
                            double2 f2[A], y2[K];
#pragma unroll
                            for (int j = 0; j < A; j++) f2[j] = *reinterpret_cast<const double2 *>(fb + (size_t)j * rcc + r);
#pragma unroll
                            for (int k = 0; k < K; k++)
                                y2[k] = *reinterpret_cast<const double2 *>(ys + chunk * RC + (size_t)k * n_pad + r);
                            double2 w2 = make_double2(0.0, 0.0);
                            if (W) w2 = *reinterpret_cast<const double2 *>(ws + chunk * RC + r);
                            if (hinted) renorm_pair<A>(f2, hkept, chunk * RC + r, lay.n);
                            accum_pair<A, K, W>(acc, f2, y2, w2);
                        }
                    }
                    __syncwarp();
                    if (chunk == n_chunks - 1)
                        reduce_to_tot<AC::N, AC::NP, 32>(acc, fb, red_rows, tot + (size_t)g * AC::NP, lane);
                    issue_next(buf, chunk == n_chunks - 1);  // refill this buffer with the stage nbuf ahead
                    if (++buf == nbuf) {
                        buf = 0;
                        parity ^= 1u;
                    }
                }
            }
        } else {
            const int u = lane / P, q0 = lane % P;
            const int nsteps = (cnt + LPS - 1) / LPS;
            for (int s = 0; s < nsteps; s++) {
                double acc[AC::N];
#pragma unroll
                for (int i = 0; i < AC::N; i++) acc[i] = 0.0;
                const unsigned hk = __shfl_sync(PG_FULL_MASK, hl, min(s * LPS + u, 31));
                const bool hinted = (hk & 0x80u) != 0u;
                const unsigned hkept = hk & 0x3fu;
                mbar_wait(&bars[buf], parity);
                double *fb = reinterpret_cast<double *>(stage0 + (size_t)buf * p.stage_bytes);
                const double *fl = fb + (size_t)u * fstride;
                if (__any_sync(PG_FULL_MASK, hinted)) {  // rare: kept out of the steady-state loop below
                    if (s * LPS + u < cnt) {
#pragma unroll 1
                        for (int r = 2 * q0; r < n_pad; r += 2 * P) {
                            double2 f2[A], y2[K];
#pragma unroll
                            for (int j = 0; j < A; j++)
                                f2[j] = *reinterpret_cast<const double2 *>(fl + (size_t)j * n_pad + r);
#pragma unroll
                            for (int k = 0; k < K; k++)
                                y2[k] = *reinterpret_cast<const double2 *>(ys + (size_t)k * n_pad + r);
                            double2 w2 = make_double2(0.0, 0.0);
                            if (W) w2 = *reinterpret_cast<const double2 *>(ws + r);
                            if (hinted) renorm_pair<A>(f2, hkept, r, lay.n);
                            accum_pair<A, K, W>(acc, f2, y2, w2);
                        }
                    }
                } else if (s * LPS + u < cnt) {  // the stage holds only the loci that exist
#pragma unroll 2
                    for (int r = 2 * q0; r < n_pad; r += 2 * P) {
                        double2 f2[A], y2[K];
#pragma unroll
                        for (int j = 0; j < A; j++) f2[j] = *reinterpret_cast<const double2 *>(fl + (size_t)j * n_pad + r);
#pragma unroll
                        for (int k = 0; k < K; k++) y2[k] = *reinterpret_cast<const double2 *>(ys + (size_t)k * n_pad + r);
                        double2 w2 = make_double2(0.0, 0.0);
                        if (W) w2 = *reinterpret_cast<const double2 *>(ws + r);
                        accum_pair<A, K, W>(acc, f2, y2, w2);
                    }
                }
                __syncwarp();
                reduce_to_tot<AC::N, AC::NP, P>(acc, fb, red_rows, tot + (size_t)(s * LPS) * AC::NP, lane);
                issue_next(buf, true);
                if (++buf == nbuf) {
                    buf = 0;
                    parity ^= 1u;
                }
            }
        }
        epilogue<A, K, W, true, KIND>(sp, l0 + lane, lane < cnt, tot, ys, ws, lane, dm, (hl & 0x80u) ? (hl & 0x3fu) : 0u);
    }
}

template <int A, int K, bool W, int P>
cudaError_t launch_scan_p(ScanParams p, int sm_count, cudaStream_t s) {
    using AC = Acc<A, K, W>;
    const Layout &lay = p.lay;
    const size_t avail = 227 * 1024 - 512;  // 512 B of static shared memory hold the parameter copy
    size_t common = (size_t)(K + (W ? 1 : 0)) * lay.n_pad * 8;
    common = (common + 127) / 128 * 128;
    size_t stage = (P == 32) ? (size_t)A * lay.rc * 8 : (size_t)(32 / P) * lay.freq_stride() * 8;
    stage = (stage + 127) / 128 * 128;
    // a stage doubles as the scratch of reduce_to_tot: at least one row of it (two alleles x four pools is a 256-byte stage)
    if (stage < (size_t)kRedPitch * 8) stage = ((size_t)kRedPitch * 8 + 127) / 128 * 128;
    // loci per epilogue block (= lanes busy in phase 2) and ring depth: prefer 32 loci and 3 stages, give way in
    // that order until the full set of warps fits (the scan is bound by the number of resident warps)
    int G = 32, nbuf = 3, nwarps = 0;
    size_t wbytes = 0;
    auto fit = [&](int g, int nb) {
        const size_t tot_bytes = ((size_t)g * AC::NP * 8 + 127) / 128 * 128;
        wbytes = 64 + (size_t)nb * stage + tot_bytes;
        nwarps = common + wbytes <= avail ? (int)((avail - common) / wbytes) : 0;
        if (nwarps > kScanWarps) nwarps = kScanWarps;
        return nwarps;
    };
    const int g_min = (P == 32) ? 16 : 32;
    if (p.nbuf_override >= 1 || p.g_override >= 1) {
        G = (p.g_override == 16 || p.g_override == 32) && P == 32 ? p.g_override : 32;
        nbuf = (p.nbuf_override >= 1 && p.nbuf_override <= 8) ? p.nbuf_override : 2;
        fit(G, nbuf);
    } else if (fit(32, 3) >= kScanWarps) {
        G = 32, nbuf = 3;
    } else if (fit(32, 2) >= kScanWarps) {
        G = 32, nbuf = 2;
    } else if (fit(g_min, 2) >= kScanWarps) {
        G = g_min, nbuf = 2;
    } else {
        G = 32, nbuf = 2;
        fit(G, nbuf);
    }
    if (p.warps_override >= 1 && p.warps_override < nwarps) nwarps = p.warps_override;
    if (nwarps < 1) return cudaErrorInvalidConfiguration;
    // block size: every warp of the grid should get the same number of blocks.  With r = ceil(L / (warps * 32)) rounds
    // the block shrinks from 32 loci to ceil(L / (warps * r)) -- a few idle lanes in phase 2 instead of a last round in
    // which most warps idle (L = 120,000: 2.1 blocks of 32 per warp -> 3 rounds at 70 %; 3 blocks of 23 -> 98 %).  Small
    // slabs of the streaming submit path fall out of the same rule (one short block per warp).
    if (p.g_override < 1 && p.n_loci > 0) {
        const int64_t gw = (int64_t)sm_count * nwarps;  // warps of the grid
        const int step = (P == 32) ? 1 : 32 / P;        // whole stages
        const int64_t r = (p.n_loci + gw * G - 1) / (gw * G);
        int64_t g = (p.n_loci + gw * r - 1) / (gw * r);
        g = (g + step - 1) / step * step;
        if (g < step) g = step;
        if (g < G) G = (int)g;
    }
    p.common_bytes = (uint32_t)common;
    p.warp_bytes = (uint32_t)wbytes;
    p.stage_bytes = (uint32_t)stage;
    p.nbuf = nbuf;
    p.block_loci = G;
    const size_t smem = common + (size_t)nwarps * wbytes;
    auto kern = (p.kind == PG_KIND_OLS) ? scan_kernel<A, K, W, P, PG_KIND_OLS> : scan_kernel<A, K, W, P, PG_KIND_CORR>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    const int64_t NB = (p.n_loci + G - 1) / G;
    int64_t ctas = (NB + nwarps - 1) / nwarps;
    if (ctas > sm_count) ctas = sm_count;
    if (ctas < 1) ctas = 1;
    e = cudaMemsetAsync(p.defer_count, 0, 4, s);
    if (e != cudaSuccess) return e;
    kern<<<(unsigned)ctas, nwarps * 32, smem, s>>>(p);
    e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    // deferred loci (count read on the device; an empty list costs one tiny launch)
    auto fix = fixup_kernel<A, K, W>;
    const size_t fsmem = (size_t)2 * 32 * AC::NP * 8;
    e = cudaFuncSetAttribute(fix, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fsmem);
    if (e != cudaSuccess) return e;
    fix<<<sm_count * 8, kFixWarps * 32, fsmem, s>>>(p);
    return cudaGetLastError();
}

template <int A, int K, bool W>
cudaError_t launch_scan_t(const ScanParams &p, int sm_count, cudaStream_t s) {
    if (p.lay.n_chunks == 1) {
        // 16 lanes per locus keep the stage at two loci (more resident warps); tiny pool counts use 8
        const int P = p.p_override ? p.p_override : (p.lay.n_pad > 64 ? 16 : 8);
        if (P == 16) return launch_scan_p<A, K, W, 16>(p, sm_count, s);
        return launch_scan_p<A, K, W, 8>(p, sm_count, s);
    }
    return launch_scan_p<A, K, W, 32>(p, sm_count, s);
}

template <int A>
cudaError_t launch_scan_a(const ScanParams &p, int sm_count, cudaStream_t s) {
    const bool w = p.weighted != 0;
    switch (p.K) {
        case 1: return w ? launch_scan_t<A, 1, true>(p, sm_count, s) : launch_scan_t<A, 1, false>(p, sm_count, s);
        case 2: return w ? launch_scan_t<A, 2, true>(p, sm_count, s) : launch_scan_t<A, 2, false>(p, sm_count, s);
        case 3:
            if constexpr (A <= 5) return w ? launch_scan_t<A, 3, true>(p, sm_count, s) : launch_scan_t<A, 3, false>(p, sm_count, s);
            else return cudaErrorInvalidValue;
        case 4:
            if constexpr (A <= 4) return w ? launch_scan_t<A, 4, true>(p, sm_count, s) : launch_scan_t<A, 4, false>(p, sm_count, s);
            else return cudaErrorInvalidValue;
        default: return cudaErrorInvalidValue;
    }
}

}  // namespace pg
