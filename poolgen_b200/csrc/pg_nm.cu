// pg_nm.cu -- the Nelder-Mead analyses of the per-locus scan (SURVEY.md 8f-3 / 8f-4):
//   mle_iter   gwas::mle_iterate  (src/gwas/mle.rs:232-305)    PG_KIND_MLE
//   gwalpha    gwas::gwalpha_ls / gwalpha_ml (src/gwas/gwalpha.rs:282-386)   PG_KIND_GWALPHA_LS / _ML
// Both start like ols_iter -- LocusCounts::filter, to_frequencies, sort_by_allele_freq, drop the major allele -- so the
// streaming scan kernel runs first in its filter-only mode and leaves status, allele order (plus the major allele's
// code) and mean frequencies; the kernels here read that, rebuild the renormalised frequency columns from the resident
// frequency matrix, and minimise the reference's cost functions with argmin 0.8.1's Nelder-Mead as
// `prepare_solver_neldermead` + `Executor::max_iters(1_000)` drive it (src/base/helpers.rs:132-146): the simplex steps
// (reflection, expansion, outside / inside contraction, shrink; stable sort by cost; standard-deviation stop) are
// those the CPU checker of this repository pins against the reference's own test_gwalpha lines, statement for statement.  A capped simplex search returns wherever its path ends, and the path turns on comparisons
// of nearly equal costs, so agreement with the reference is to the solver's own convergence (declared in the tests),
// not 1e-9 -- DESIGN.md 11.
//   mle_iter: a warp per locus forms the centred moments of [x | y] once (lane = pool); the cost
//       (n/2) ln(2 pi s2) + RSS(beta) / s2   (mle.rs:13-30, sic: no 1/2 on the second term)
//   is then a quadratic form in beta -- O(p^2) per evaluation instead of O(n p) -- and lane j minimises phenotype j.
//   gwalpha: a thread per (locus, allele); the cost sums squared differences (LS) or log10 differences (ML) of Beta
//   cdfs, statrs' continued fraction with the shapes of the current vertex.
//   mle_iter_with_kinship  gwas::mle_with_covariate (src/gwas/mle.rs:307-463): kin_mle_kernel over a pg_kin's columns.
#include "pg_device.cuh"
#include "pg_internal.h"

namespace pg {

constexpr int kNmMaxD = 8;  // parameters: sigma2 + intercept + up to 5 alleles (mle), 4 shapes (gwalpha)

__device__ __forceinline__ double bound_logit(double x, double lo, double hi) { return lo + ((hi - lo) / (1.00 + exp(-x))); }

// argmin 0.8.1 Nelder-Mead: alpha 1, gamma 2, rho = sigma =
// 0.5, sd_tolerance = f64::EPSILON, initial simplex h everywhere and h + 0.5 on the diagonal, stable sort by cost.
template <int MAXD, typename Cost>
__device__ void nelder_mead(const Cost &cost, int d, double h, int max_iters, double *best) {
    double v[MAXD + 1][MAXD], c[MAXD + 1];
    const int nv = d + 1;
    for (int i = 0; i < nv; i++)
        for (int j = 0; j < d; j++) v[i][j] = (i == j) ? h + 0.5 : h;
    for (int i = 0; i < nv; i++) c[i] = cost(v[i]);
    auto sort = [&]() {
        for (int a = 1; a < nv; a++) {
            const double ca = c[a];
            double va[MAXD];
            for (int j = 0; j < d; j++) va[j] = v[a][j];
            int b = a - 1;
            while (b >= 0 && ca < c[b]) {
                c[b + 1] = c[b];
                for (int j = 0; j < d; j++) v[b + 1][j] = v[b][j];
                b--;
            }
            c[b + 1] = ca;
            for (int j = 0; j < d; j++) v[b + 1][j] = va[j];
        }
    };
    auto shrink = [&]() {
        for (int i = 1; i < nv; i++) {
            for (int j = 0; j < d; j++) v[i][j] = v[0][j] + (v[i][j] - v[0][j]) * 0.5;
            c[i] = cost(v[i]);
        }
    };
    sort();
    for (int it = 0;; it++) {
        double c0 = 0.0;
        for (int i = 0; i < nv; i++) c0 = c0 + c[i];
        c0 = c0 / (double)nv;
        double ss = 0.0;
        for (int i = 0; i < nv; i++) ss = ss + (c[i] - c0) * (c[i] - c0);
        const double sd = sqrt(1.0 / ((double)nv - 1.0) * ss);
        if (sd < kEps) break;
        if (it >= max_iters) break;
        double x0[MAXD], xr[MAXD], xt[MAXD];
        for (int j = 0; j < d; j++) x0[j] = v[0][j];
        for (int i = 1; i < nv - 1; i++)
            for (int j = 0; j < d; j++) x0[j] = x0[j] + v[i][j];
        const double inv = 1.0 / (double)(nv - 1);
        for (int j = 0; j < d; j++) x0[j] = x0[j] * inv;
        for (int j = 0; j < d; j++) xr[j] = x0[j] + (x0[j] - v[nv - 1][j]) * 1.0;
        const double fr = cost(xr);
        if (fr < c[nv - 2] && fr >= c[0]) {
            for (int j = 0; j < d; j++) v[nv - 1][j] = xr[j];
            c[nv - 1] = fr;
        } else if (fr < c[0]) {
            for (int j = 0; j < d; j++) xt[j] = x0[j] + (xr[j] - x0[j]) * 2.0;
            const double fe = cost(xt);
            const bool take_e = fe < fr;
            for (int j = 0; j < d; j++) v[nv - 1][j] = take_e ? xt[j] : xr[j];
            c[nv - 1] = take_e ? fe : fr;
        } else if (fr >= c[nv - 2]) {
            if (fr < c[nv - 1]) {  // outside contraction
                for (int j = 0; j < d; j++) xt[j] = x0[j] + (xr[j] - x0[j]) * 0.5;
                const double fc = cost(xt);
                if (fc <= fr) {
                    for (int j = 0; j < d; j++) v[nv - 1][j] = xt[j];
                    c[nv - 1] = fc;
                } else {
                    shrink();
                }
            } else {  // inside contraction
                for (int j = 0; j < d; j++) xt[j] = x0[j] + (v[nv - 1][j] - x0[j]) * 0.5;
                const double fc = cost(xt);
                if (fc < c[nv - 1]) {
                    for (int j = 0; j < d; j++) v[nv - 1][j] = xt[j];
                    c[nv - 1] = fc;
                } else {
                    shrink();
                }
            }
        } else {
            shrink();  // only reachable with NaN costs
        }
        sort();
    }
    for (int j = 0; j < d; j++) best[j] = v[0][j];
}

// The same search as a state machine with ONE call site of the cost function, for costs that dwarf the bookkeeping
// (gwalpha: 4.7 x; mle_iter's quadratic form is so cheap that the indexed state costs 3 x -- it keeps the loop
// above): the lanes of a warp run independent searches
// and take different steps in the same iteration (one reflects, one expands, one shrinks); with a call per step the
// warp would walk through every call site in turn, each time with a few lanes active.  Here every lane names the
// point it needs next, all evaluate together, and each then advances its own state.  The sequence of points, costs
// and comparisons of a search is exactly the textbook loop's.
template <int MAXD, typename Cost>
__device__ void nelder_mead_one_site(const Cost &cost, int d, double h, int max_iters, double *best) {
    double v[MAXD + 1][MAXD], c[MAXD + 1];
    const int nv = d + 1;
    for (int i = 0; i < nv; i++)
        for (int j = 0; j < d; j++) v[i][j] = (i == j) ? h + 0.5 : h;
    auto sort = [&]() {
        for (int a = 1; a < nv; a++) {
            const double ca = c[a];
            double va[MAXD];
            for (int j = 0; j < d; j++) va[j] = v[a][j];
            int b = a - 1;
            while (b >= 0 && ca < c[b]) {
                c[b + 1] = c[b];
                for (int j = 0; j < d; j++) v[b + 1][j] = v[b][j];
                b--;
            }
            c[b + 1] = ca;
            for (int j = 0; j < d; j++) v[b + 1][j] = va[j];
        }
    };
    enum { kInit, kReflect, kExpand, kOutside, kInside, kShrink, kDone };
    int state = kInit, idx = 0, it = 0;
    double x0[MAXD], xr[MAXD], xt[MAXD], fr = 0.0;
    // the vertices are sorted: stop, or set up the next iteration (centroid of all but the worst, reflected point)
    auto next_iteration = [&]() {
        double c0 = 0.0;
        for (int i = 0; i < nv; i++) c0 = c0 + c[i];
        c0 = c0 / (double)nv;
        double ss = 0.0;
        for (int i = 0; i < nv; i++) ss = ss + (c[i] - c0) * (c[i] - c0);
        const double sd = sqrt(1.0 / ((double)nv - 1.0) * ss);
        if (sd < kEps || it >= max_iters) {
            state = kDone;
            return;
        }
        it++;
        for (int j = 0; j < d; j++) x0[j] = v[0][j];
        for (int i = 1; i < nv - 1; i++)
            for (int j = 0; j < d; j++) x0[j] = x0[j] + v[i][j];
        const double inv = 1.0 / (double)(nv - 1);
        for (int j = 0; j < d; j++) x0[j] = x0[j] * inv;
        for (int j = 0; j < d; j++) xr[j] = x0[j] + (x0[j] - v[nv - 1][j]) * 1.0;
        state = kReflect;
    };
    auto accept = [&](const double *x, double f) {  // replaces the worst vertex
        for (int j = 0; j < d; j++) v[nv - 1][j] = x[j];
        c[nv - 1] = f;
        sort();
        next_iteration();
    };
    auto begin_shrink = [&]() {  // every vertex half way towards the best one, then their costs one by one
        for (int i = 1; i < nv; i++)
            for (int j = 0; j < d; j++) v[i][j] = v[0][j] + (v[i][j] - v[0][j]) * 0.5;
        idx = 1;
        state = kShrink;
    };
    while (state != kDone) {
        const double *x = (state == kInit || state == kShrink) ? v[idx] : (state == kReflect ? xr : xt);
        const double f = cost(x);
        if (state == kInit || state == kShrink) {
            c[idx] = f;
            if (++idx == nv) {
                sort();
                next_iteration();
            }
        } else if (state == kReflect) {
            fr = f;
            if (fr < c[nv - 2] && fr >= c[0]) {
                accept(xr, fr);
            } else if (fr < c[0]) {
                for (int j = 0; j < d; j++) xt[j] = x0[j] + (xr[j] - x0[j]) * 2.0;
                state = kExpand;
            } else if (fr >= c[nv - 2]) {
                if (fr < c[nv - 1]) {  // outside contraction
                    for (int j = 0; j < d; j++) xt[j] = x0[j] + (xr[j] - x0[j]) * 0.5;
                    state = kOutside;
                } else {  // inside contraction
                    for (int j = 0; j < d; j++) xt[j] = x0[j] + (v[nv - 1][j] - x0[j]) * 0.5;
                    state = kInside;
                }
            } else {
                begin_shrink();  // only reachable with NaN costs
            }
        } else if (state == kExpand) {
            if (f < fr)
                accept(xt, f);
            else
                accept(xr, fr);
        } else if (state == kOutside) {
            if (f <= fr)
                accept(xt, f);
            else
                begin_shrink();
        } else {  // kInside
            if (f < c[nv - 1])
                accept(xt, f);
            else
                begin_shrink();
        }
    }
    for (int j = 0; j < d; j++) best[j] = v[0][j];
}

// the renormalised frequency of (pool i, device column j) over the kept columns, as the scan forms it
__device__ __forceinline__ void renorm_generic(const NmParams &p, const double *fl, const uint32_t *dl, int i, unsigned kept,
                                               double *F) {
    const int A = p.lay.A;
    const uint32_t d = dl[i];
    double c[PG_MAX_ALLELES], dk = 0.0;
    for (int j = 0; j < A; j++) {
        c[j] = (d == 0u) ? 0.0 : rint(fl[p.lay.freq_off(i, j)] * (double)d);
        if ((kept >> j) & 1u) dk += c[j];
    }
    for (int j = 0; j < A; j++) F[j] = ((kept >> j) & 1u) ? ((dk == 0.0) ? nan("") : c[j] / dk) : 0.0;
}

// device column of an allele code
__device__ __forceinline__ int col_of_code(const NmParams &p, unsigned code) {
    for (int j = 0; j < p.lay.A; j++)
        if (p.codes[j] == code) return j;
    return 0;
}

// ---- mle_iter: a warp takes 32 loci; moments by the whole warp (lane = pool), simplex searches with lane = locus ------
constexpr int kMlePhen = 4;                                   // phenotypes per pass over the loci of a block
// a locus' row of moments: xbar[5] | Sxx lower triangle [15] | per phenotype of the pass: ybar, syy, sxy[5]
// the per-locus row a launch actually uses: with fewer than kMlePhen phenotypes the rows shrink, and with them the
// shared memory per warp -- the searches are latency bound, so every resident warp counts (16 -> 20 per SM at k = 1)
__host__ __device__ inline int mle_mom_stride(int k) { return 20 + (k < kMlePhen ? k : kMlePhen) * 7; }
constexpr int kMleWarps = 4;

__global__ void __launch_bounds__(kMleWarps * 32) mle_kernel(const NmParams p) {
    extern __shared__ __align__(16) double mle_sm[];  // [warps][32][stride]
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int stride = mle_mom_stride(p.k);
    double *mom = mle_sm + (size_t)wib * 32 * stride;
    const int64_t warp = (int64_t)blockIdx.x * kMleWarps + wib;
    const int64_t nwarps = (int64_t)gridDim.x * kMleWarps;
    const int n = p.lay.n, n_pad = p.lay.n_pad, S = p.lay.A - 1, k = p.k;
    const PTableDev ptab = {reinterpret_cast<const double4 *>(p.ptab), p.ptab_isd, p.ptab_bits, p.ptab_t1, p.ptab_t0, p.ptab_M};
    const int64_t n_blocks = (p.n_loci + 31) / 32;
    for (int64_t blk = warp; blk < n_blocks; blk += nwarps) {
        const int64_t l0 = blk * 32;
        const int cnt = (int)min((int64_t)32, p.n_loci - l0);
        // this lane's locus: status, allele columns of X (the intercept comes on top), kept set
        const uint64_t mv = (lane < cnt) ? p.meta[l0 + lane] : 0ull;
        const bool act = (mv & 0xffu) == PG_LOCUS_OK;
        const int m = (int)((mv >> 8) & 0xffu);
        unsigned colw = 0, kept = 0;  // 4 bits per output slot: device column
        if (act) {
            for (int s = 0; s < m; s++) {
                const int c = col_of_code(p, (unsigned)((mv >> (16 + 8 * s)) & 0xffu));
                colw |= (unsigned)c << (4 * s);
                kept |= 1u << c;
            }
            kept |= 1u << col_of_code(p, (unsigned)((mv >> (16 + 8 * m)) & 0xffu));  // the major allele
        }
        // ---- moments of the allele columns, one locus after the other, lane = pool
        for (int g = 0; g < cnt; g++) {
            if (!__shfl_sync(PG_FULL_MASK, (int)act, g)) continue;  // warp-uniform
            const int mg = __shfl_sync(PG_FULL_MASK, m, g);
            const unsigned cg = __shfl_sync(PG_FULL_MASK, colw, g), kg = __shfl_sync(PG_FULL_MASK, kept, g);
            const double *fl = p.freq + (size_t)(l0 + g) * p.lay.freq_stride();
            const uint32_t *dl = p.depth + (size_t)(l0 + g) * p.lay.depth_stride();
            double sx[PG_MAX_SLOTS], lo[PG_MAX_SLOTS], hi[PG_MAX_SLOTS];
            for (int a = 0; a < PG_MAX_SLOTS; a++) sx[a] = 0.0, lo[a] = INFINITY, hi[a] = -INFINITY;
            for (int i = lane; i < n; i += 32) {
                double F[PG_MAX_ALLELES];
                renorm_generic(p, fl, dl, i, kg, F);
                for (int a = 0; a < mg; a++) {
                    const double f = F[(cg >> (4 * a)) & 0xfu];
                    sx[a] += f;
                    lo[a] = fmin(lo[a], f);
                    hi[a] = fmax(hi[a], f);
                }
            }
            // A column that is the same double in every pool is a multiple of the intercept.  Its mean is that double,
            // exactly: the sum / n form leaves an ulp-sized residue in every centred value for most n (1/3, 0.1), and
            // whether that residue is zero decides r = 0 / 0 (kept) or r = +-1 against another such column (removed),
            // and a zero or a 1e-31 pivot.  Centred to zero, the column is never removed, removes nothing, and its
            // zero row of Sxx makes the locus FAILED -- X'X is singular (DESIGN.md 11)
            double xb[PG_MAX_SLOTS];
            for (int a = 0; a < PG_MAX_SLOTS; a++) {
                if (a >= mg) {
                    xb[a] = 0.0;
                    continue;
                }
                double l = lo[a], h = hi[a];
#pragma unroll
                for (int off = 16; off >= 1; off >>= 1) {
                    l = fmin(l, __shfl_xor_sync(PG_FULL_MASK, l, off));
                    h = fmax(h, __shfl_xor_sync(PG_FULL_MASK, h, off));
                }
                const double mean = warp_sum_fixed(sx[a]) / (double)n;
                xb[a] = (l == h && mean == mean) ? l : mean;
            }
            double sxx[15];
            for (int e = 0; e < 15; e++) sxx[e] = 0.0;
            for (int i = lane; i < n; i += 32) {
                double F[PG_MAX_ALLELES];
                renorm_generic(p, fl, dl, i, kg, F);
                for (int a = 0; a < mg; a++)
                    for (int b = 0; b <= a; b++)
                        sxx[a * (a + 1) / 2 + b] = fma(F[(cg >> (4 * a)) & 0xfu] - xb[a], F[(cg >> (4 * b)) & 0xfu] - xb[b], sxx[a * (a + 1) / 2 + b]);
            }
            for (int e = 0; e < 15; e++) sxx[e] = (e < mg * (mg + 1) / 2) ? warp_sum_fixed(sxx[e]) : 0.0;
            if (lane == 0) {
                double *mo = mom + (size_t)g * stride;
                for (int a = 0; a < PG_MAX_SLOTS; a++) mo[a] = xb[a];
                for (int e = 0; e < 15; e++) mo[5 + e] = sxx[e];
            }
        }
        __syncwarp();
        // ---- lane = locus: collinear columns, (X'X)^-1
        double xbar[PG_MAX_SLOTS], Sxx[PG_MAX_SLOTS][PG_MAX_SLOTS];
        {
            const double *mo = mom + (size_t)lane * stride;
            for (int a = 0; a < PG_MAX_SLOTS; a++) xbar[a] = act ? mo[a] : 0.0;
            for (int a = 0; a < PG_MAX_SLOTS; a++)
                for (int b = 0; b <= a; b++) Sxx[a][b] = Sxx[b][a] = act ? mo[5 + a * (a + 1) / 2 + b] : 0.0;
        }
        // remove_collinearities_in_x (mle.rs:56-83), literally, on |r| rounded to 7 digits like pearsons_correlation.
        // X column c >= 1 is allele column c - 1; column 0 is the intercept (its correlation is NaN: never removed).
        int xc[PG_MAX_SLOTS + 1], pw = m + 1;
        for (int c = 0; c <= PG_MAX_SLOTS; c++) xc[c] = c;
        bool panic = false;
        if (act && pw != 2) {
            long i = 1;
            while (i < pw && !panic) {
                long j = i + 1;
                while (j < pw) {
                    if (i < 0) {
                        panic = true;  // the reference's `i -= 1` underflows and its next column() call panics
                        break;
                    }
                    double cor = nan("");
                    if (xc[i] >= 1 && xc[j] >= 1) {
                        const int a = xc[i] - 1, b = xc[j] - 1;
                        const double r = Sxx[a][b] / (sqrt(Sxx[a][a]) * sqrt(Sxx[b][b]));
                        cor = round(r * 1e7) / 1e7;
                    }
                    if (fabs(cor) >= 0.99) {
                        for (int c = (int)j; c + 1 < pw; c++) xc[c] = xc[c + 1];
                        pw -= 1;
                        i -= 1;
                        j -= 1;
                    }
                    j += 1;
                }
                i += 1;
            }
        }
        int status = !act ? (int)(mv & 0xffu) : (panic ? PG_LOCUS_PANIC : PG_LOCUS_OK);
        if (act && status == PG_LOCUS_OK && n < pw) status = PG_LOCUS_UNSUPPORTED;  // the X X' form of the variances (mle.rs:130-140)
        // (X'X)^-1 of the remaining columns through the centred moments: the allele block is Sxx^-1, the intercept's
        // diagonal entry 1/n + xbar' Sxx^-1 xbar
        const int q = pw - 1;  // allele columns left
        double dgi[PG_MAX_SLOTS + 1];
        for (int c = 0; c <= PG_MAX_SLOTS; c++) dgi[c] = 0.0;
        if (act && status == PG_LOCUS_OK) {
            double M[PG_MAX_SLOTS][2 * PG_MAX_SLOTS];
            for (int a = 0; a < q; a++)
                for (int b = 0; b < q; b++) {
                    M[a][b] = Sxx[xc[a + 1] - 1][xc[b + 1] - 1];
                    M[a][q + b] = a == b ? 1.0 : 0.0;
                }
            for (int c = 0; c < q && status == PG_LOCUS_OK; c++) {  // Gauss-Jordan with partial pivoting
                int pr = c;
                for (int r = c + 1; r < q; r++)
                    if (fabs(M[r][c]) > fabs(M[pr][c])) pr = r;
                if (!(fabs(M[pr][c]) > 0.0)) {
                    status = PG_LOCUS_FAILED;  // Non-invertible x_matrix (mle.rs:143-148)
                    break;
                }
                for (int e = 0; e < 2 * q; e++) {
                    const double tmp = M[c][e];
                    M[c][e] = M[pr][e];
                    M[pr][e] = tmp;
                }
                const double piv = 1.0 / M[c][c];
                for (int e = 0; e < 2 * q; e++) M[c][e] *= piv;
                for (int r = 0; r < q; r++) {
                    if (r == c) continue;
                    const double f = M[r][c];
                    for (int e = 0; e < 2 * q; e++) M[r][e] -= f * M[c][e];
                }
            }
            if (status == PG_LOCUS_OK) {
                double quad = 0.0;
                for (int a = 0; a < q; a++)
                    for (int b = 0; b < q; b++) quad += xbar[xc[a + 1] - 1] * M[a][q + b] * xbar[xc[b + 1] - 1];
                dgi[0] = 1.0 / (double)n + quad;
                for (int a = 0; a < q; a++) dgi[1 + a] = M[a][q + a];
            }
        }
        // ---- phenotypes, kMlePhen at a time: centred cross moments by the whole warp, then lane = locus again
        for (int j0 = 0; j0 < k; j0 += kMlePhen) {
            const int jn = min(kMlePhen, k - j0);
            __syncwarp();
            for (int g = 0; g < cnt; g++) {
                if (!__shfl_sync(PG_FULL_MASK, (int)act, g)) continue;
                const int mg = __shfl_sync(PG_FULL_MASK, m, g);
                const unsigned cg = __shfl_sync(PG_FULL_MASK, colw, g), kg = __shfl_sync(PG_FULL_MASK, kept, g);
                const double *fl = p.freq + (size_t)(l0 + g) * p.lay.freq_stride();
                const uint32_t *dl = p.depth + (size_t)(l0 + g) * p.lay.depth_stride();
                const double *mo = mom + (size_t)g * stride;
                double xb[PG_MAX_SLOTS];
                for (int a = 0; a < PG_MAX_SLOTS; a++) xb[a] = mo[a];
                for (int jj = 0; jj < jn; jj++) {
                    const double *y = p.yraw + (size_t)(j0 + jj) * n_pad;
                    double sy = 0.0;
                    for (int i = lane; i < n; i += 32) sy += y[i];
                    const double ybar = warp_sum_fixed(sy) / (double)n;
                    double syy = 0.0, sxy[PG_MAX_SLOTS];
                    for (int a = 0; a < PG_MAX_SLOTS; a++) sxy[a] = 0.0;
                    for (int i = lane; i < n; i += 32) {
                        double F[PG_MAX_ALLELES];
                        renorm_generic(p, fl, dl, i, kg, F);
                        const double dy = y[i] - ybar;
                        syy = fma(dy, dy, syy);
                        for (int a = 0; a < mg; a++) sxy[a] = fma(F[(cg >> (4 * a)) & 0xfu] - xb[a], dy, sxy[a]);
                    }
                    syy = warp_sum_fixed(syy);
                    for (int a = 0; a < PG_MAX_SLOTS; a++) sxy[a] = (a < mg) ? warp_sum_fixed(sxy[a]) : 0.0;
                    if (lane == 0) {
                        double *o = mom + (size_t)g * stride + 20 + jj * 7;
                        o[0] = ybar;
                        o[1] = syy;
                        for (int a = 0; a < PG_MAX_SLOTS; a++) o[2 + a] = sxy[a];
                    }
                }
            }
            __syncwarp();
            if (lane < cnt && (act || true)) {
                for (int jj = 0; jj < jn; jj++) {
                    const int j = j0 + jj;
                    const double *mo = mom + (size_t)lane * stride + 20 + jj * 7;
                    const double ybar_l = mo[0], syy_l = mo[1];
                    double sxy_l[PG_MAX_SLOTS];
                    for (int a = 0; a < PG_MAX_SLOTS; a++) sxy_l[a] = mo[2 + a];
                    double b[PG_MAX_SLOTS + 1], vb[PG_MAX_SLOTS + 1];
                    for (int c = 0; c <= PG_MAX_SLOTS; c++) b[c] = vb[c] = 0.0;  // Array2::zeros: rows of removed columns
                    if (act && status == PG_LOCUS_OK) {
                        const double nn = (double)n;
                        // cost(par): par[0] = logit of sigma2, par[1] = intercept, par[2..] = remaining allele columns
                        auto cost = [&](const double *par) {
                            const double s2 = bound_logit(par[0], kEps, 1e9);
                            double quad = 0.0, lin = 0.0, off = ybar_l - par[1];
                            for (int a = 0; a < q; a++) {
                                const int ia = xc[a + 1] - 1;
                                lin += par[2 + a] * sxy_l[ia];
                                off -= xbar[ia] * par[2 + a];
                                for (int c = 0; c < q; c++) quad += par[2 + a] * Sxx[ia][xc[c + 1] - 1] * par[2 + c];
                            }
                            const double rss = (syy_l - 2.0 * lin + quad) + nn * off * off;
                            return (nn / 2.00) * log(2.00 * 3.14159265358979323846264338327950288 * s2) + (1.00 / s2) * rss;
                        };
                        double par[kNmMaxD];
                        nelder_mead<kNmMaxD>(cost, pw + 1, 1.0, 1000, par);
                        const double ve = bound_logit(par[0], kEps, 1e9);
                        for (int c = 0; c < pw; c++) {
                            b[c] = par[1 + c];
                            vb[c] = ve * dgi[c];
                        }
                    }
                    // a locus the scan did not pass on keeps NaN records for every phenotype: its filter-only pass
                    // writes phenotype 0 only, and the rows of the others would be whatever the buffer held
                    for (int s = 0; s < S; s++) {
                        double o0 = nan(""), o1 = nan(""), o2 = nan(""), o3 = nan("");
                        if (status == PG_LOCUS_OK && s < m) {
                            // output row s is X column s + 1 of the UNREDUCED matrix: the reference fills rows 0..pw of a
                            // zero matrix and never maps them back (mle.rs:218-226: "does not account for the identities
                            // of the removed columns")
                            const int c = s + 1;
                            const bool filled = c < pw;
                            o0 = filled ? b[c] : 0.0;
                            o1 = filled ? vb[c] : 0.0;
                            if (filled) {
                                o2 = o0 / o1;  // mle.rs:176: the variance, not its square root
                                if (isinf(o2))
                                    o3 = 0.0;
                                else if (o2 != o2)
                                    o3 = 1.0;
                                else
                                    o3 = p.ptab ? student_two_sided_tab(fabs(o2), p.df, ptab) : student_two_sided(fabs(o2), p.df, p.ln_beta);
                            } else {
                                o3 = 0.0;
                            }
                        }
                        double *o = p.stats + (((size_t)(l0 + lane) * S + s) * k + j) * 4;
                        o[0] = o0, o[1] = o1, o[2] = o2, o[3] = o3;
                    }
                }
            }
        }
        if (act && status != PG_LOCUS_OK) p.meta[l0 + lane] = (mv & ~0xffull) | (uint64_t)status;
        __syncwarp();
    }
}

// ---- gwalpha: one thread per (locus, allele) ------------------------------------------------------------------------
constexpr int kGwMaxPools = 64;

__device__ double nd_sum(const double *xs, int len) {  // ndarray 0.15 unrolled_fold (what `.sum()` does on a slice)
    double acc = 0.0, p0 = 0, p1 = 0, p2 = 0, p3 = 0, p4 = 0, p5 = 0, p6 = 0, p7 = 0;
    while (len >= 8) {
        p0 = p0 + xs[0], p1 = p1 + xs[1], p2 = p2 + xs[2], p3 = p3 + xs[3];
        p4 = p4 + xs[4], p5 = p5 + xs[5], p6 = p6 + xs[6], p7 = p7 + xs[7];
        xs += 8;
        len -= 8;
    }
    acc = acc + (p0 + p4);
    acc = acc + (p1 + p5);
    acc = acc + (p2 + p6);
    acc = acc + (p3 + p7);
    for (int i = 0; i < len && i < 7; i++) acc = acc + xs[i];
    return acc;
}

// statrs Beta::cdf with the shapes' ln B precomputed
__device__ __forceinline__ double beta_cdf_dev(double a, double b, double lnb, double x) {
    if (x < 0.0) return 0.0;
    if (x >= 1.0) return 1.0;
    if (fabs(a - 1.0) <= 4.0 * 1.1102230246251565e-16 && fabs(b - 1.0) <= 4.0 * 1.1102230246251565e-16) return x;
    return beta_reg_dev(a, b, x, lnb);
}

__global__ void __launch_bounds__(128) gwalpha_kernel(const NmParams p) {
    const int S = p.lay.A - 1, n = p.lay.n, n_pad = p.lay.n_pad;
    const int64_t total = p.n_loci * S;
    const double *bins = p.yraw, *q = p.yraw + n_pad;
    for (int64_t item = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; item < total;
         item += (int64_t)gridDim.x * blockDim.x) {
        const int64_t locus = item / S;
        const int s = (int)(item - locus * S);
        const uint64_t mv = p.meta[locus];
        double *o = p.stats + ((size_t)locus * S + s) * 4;
        const int m = (int)((mv >> 8) & 0xffu);
        if ((mv & 0xffu) != PG_LOCUS_OK || s >= m) {
            o[0] = o[1] = o[2] = o[3] = nan("");
            continue;
        }
        unsigned kept = 0;
        for (int a = 0; a <= m; a++) kept |= 1u << col_of_code(p, (unsigned)((mv >> (16 + 8 * a)) & 0xffu));
        const int cj = col_of_code(p, (unsigned)((mv >> (16 + 8 * s)) & 0xffu));
        const double *fl = p.freq + (size_t)locus * p.lay.freq_stride();
        const uint32_t *dl = p.depth + (size_t)locus * p.lay.depth_stride();
        // prepare_freqs_and_qprime (gwalpha.rs:225-280)
        double fa[kGwMaxPools], qp[kGwMaxPools], pa[kGwMaxPools], pb[kGwMaxPools], pa0[kGwMaxPools], pb0[kGwMaxPools];
        double p_a = 0.0;
        for (int i = 0; i < n; i++) {
            double F[PG_MAX_ALLELES];
            renorm_generic(p, fl, dl, i, kept, F);
            fa[i] = F[cj];
        }
        if (m == 1) {  // a one-column matrix: the column view is contiguous and ndarray takes its unrolled dot
            double prod[kGwMaxPools];
            double s0 = 0.0, ps[8] = {0, 0, 0, 0, 0, 0, 0, 0};
            int len = n, at = 0;
            while (len >= 8) {
                for (int e = 0; e < 8; e++) ps[e] = ps[e] + fa[at + e] * bins[at + e];
                at += 8;
                len -= 8;
            }
            s0 = s0 + (ps[0] + ps[4]);
            s0 = s0 + (ps[1] + ps[5]);
            s0 = s0 + (ps[2] + ps[6]);
            s0 = s0 + (ps[3] + ps[7]);
            for (int i = 0; i < len && i < 7; i++) s0 = s0 + fa[at + i] * bins[at + i];
            p_a = s0;
            (void)prod;
        } else {
            for (int i = 0; i < n; i++) p_a += fa[i] * bins[i];
        }
        qp[0] = 0.0;
        for (int i = 1; i < n; i++) qp[i] = (q[i] - p.gw_min) / (p.gw_max - p.gw_min);
        {
            double ba[kGwMaxPools], bb[kGwMaxPools];
            for (int i = 0; i < n; i++) {
                ba[i] = (fa[i]) * bins[i] / (p_a);
                bb[i] = (1.0 - fa[i]) * bins[i] / (1.0 - p_a);
            }
            pa[0] = ba[0];
            pb[0] = bb[0];
            for (int i = 1; i < n; i++) {
                pa[i] = nd_sum(ba, i + 1);
                pb[i] = nd_sum(bb, i + 1);
            }
        }
        pa0[0] = pb0[0] = 0.0;
        for (int i = 0; i < n - 1; i++) {
            pa0[i + 1] = pa[i];
            pb0[i + 1] = pb[i];
        }
        const bool ml = p.kind == PG_KIND_GWALPHA_ML;
        auto cost = [&](const double *par) {
            double sh[4];
            for (int e = 0; e < 4; e++) sh[e] = bound_logit(par[e], kEps, 10.00);
            const double lna = ln_gamma_dev(sh[0] + sh[1]) - ln_gamma_dev(sh[0]) - ln_gamma_dev(sh[1]);
            const double lnb = ln_gamma_dev(sh[2] + sh[3]) - ln_gamma_dev(sh[2]) - ln_gamma_dev(sh[3]);
            double ra = 0.0, rb = 0.0;
            if (!ml) {  // least_squares_beta (gwalpha.rs:11-41)
                for (int i = 0; i < n; i++) {
                    const double da = pa[i] - beta_cdf_dev(sh[0], sh[1], lna, qp[i]);
                    const double db = pb[i] - beta_cdf_dev(sh[2], sh[3], lnb, qp[i]);
                    ra += da * da;
                    rb += db * db;
                }
                return ra + rb;
            }
            // maximum_likelihood_beta (gwalpha.rs:43-82).  The lower percentile of bin i is the upper one of bin i - 1
            // (pa0[i] = pa[i - 1], bit for bit), so its cdf is the value the previous turn computed: the same
            // numbers as the reference's two evaluations per bin at half the continued fractions
            double lo_a = beta_cdf_dev(sh[0], sh[1], lna, pa0[0]), lo_b = beta_cdf_dev(sh[2], sh[3], lnb, pb0[0]);
            for (int i = 0; i < n; i++) {
                const double hi_a = beta_cdf_dev(sh[0], sh[1], lna, pa[i]), hi_b = beta_cdf_dev(sh[2], sh[3], lnb, pb[i]);
                double da = hi_a - lo_a;
                double db = hi_b - lo_b;
                lo_a = hi_a;
                lo_b = hi_b;
                if (da < kEps) da = kEps;
                if (db < kEps) db = kEps;
                ra += log10(da);
                rb += log10(db);
            }
            return -ra - rb;
        };
        double par[kNmMaxD];
        nelder_mead_one_site<kNmMaxD>(cost, 4, 1.0, 1000, par);
        double sol[4];
        for (int e = 0; e < 4; e++) sol[e] = bound_logit(par[e], kEps, 10.00);
        const double a_mu = p.gw_min + (p.gw_max - p.gw_min) * (sol[0] / (sol[0] + sol[1]));
        const double b_mu = p.gw_min + (p.gw_max - p.gw_min) * (sol[2] / (sol[2] + sol[3]));
        const double alpha = (2.00 * sqrt(p_a * (1.0 - p_a))) * (a_mu - b_mu) / p.gw_sig;
        o[0] = alpha;
        o[1] = p_a;
        o[2] = nan("");
        o[3] = nan("");
    }
}

// ---- mle_iter_with_kinship: mle_with_covariate (mle.rs:307-463) over the resident allele columns --------------------
// One regression per (column, phenotype) with X = [1 | PCs | g] (mle.rs:370-392) and mle(x, y, false): Nelder-Mead over
// [logit sigma2, b_0, b_PC.., b_g] from the all-ones simplex, v_b = sigma2 [(X'X)^-1]_gg, t = b / v_b (sic, mle.rs:176),
// p from Student-t(n - 1).  A warp takes 32 columns: the whole warp forms the centred moments of a column against the
// covariates and phenotypes (lane = pool; everything that does not involve g is formed once on the host), then lane =
// column runs the searches on the quadratic form
//   RSS(b) = Syy - 2 (b_z'Szy + b_g Sgy) + b_z'Szz b_z + 2 b_g b_z'Szg + b_g^2 Sgg + n (ybar - b_0 - b_z'zbar - b_g gbar)^2
constexpr int kKmWarps = 4;
constexpr int kKmMaxD = kKinMleMaxM + 3;

__global__ void __launch_bounds__(kKmWarps * 32) kin_mle_kernel(const KinMleParams p, int fix_pad) {
    extern __shared__ __align__(16) double km_sm[];  // fix | [warps][32][2 + m + k]
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int m = p.m, k = p.k, n = p.n;
    const int nfix = m + 2 * m * m + k * (2 + m);
    for (int i = threadIdx.x; i < nfix; i += blockDim.x) km_sm[i] = p.fix[i];
    __syncthreads();
    const double *zbar = km_sm, *Szz = zbar + m, *Wzz = Szz + m * m, *phf = Wzz + m * m;
    const int mw = 2 + m + k;  // gbar, Sgg, Szg[m], Sgy[k]
    double *mom = km_sm + fix_pad + (size_t)wib * 32 * mw;
    const PTableDev ptab = {reinterpret_cast<const double4 *>(p.ptab), p.ptab_isd, p.ptab_bits, p.ptab_t1, p.ptab_t0, p.ptab_M};
    const double nn = (double)n;
    const int64_t n_blocks = (p.P + 31) / 32;
    for (int64_t blk = (int64_t)blockIdx.x * kKmWarps + wib; blk < n_blocks; blk += (int64_t)gridDim.x * kKmWarps) {
        const int64_t c0 = blk * 32;
        const int cnt = (int)min((int64_t)32, p.P - c0);
        for (int g = 0; g < cnt; g++) {
            const double *col = p.G + (size_t)(c0 + g) * p.ldg;
            double *mo = mom + (size_t)g * mw;
            double s = 0.0;
            for (int i = lane; i < n; i += 32) s += col[i];
            const double gbar = warp_sum_fixed(s) / nn;
            double sgg = 0.0;
            for (int i = lane; i < n; i += 32) {
                const double d = col[i] - gbar;
                sgg = fma(d, d, sgg);
            }
            sgg = warp_sum_fixed(sgg);
            if (lane == 0) mo[0] = gbar, mo[1] = sgg;
            for (int v0 = 0; v0 < m + k; v0 += 4) {
                const int nv = min(4, m + k - v0);
                double a[4] = {0.0, 0.0, 0.0, 0.0};
                for (int i = lane; i < n; i += 32) {
                    const double d = col[i] - gbar;
#pragma unroll
                    for (int e = 0; e < 4; e++)
                        if (e < nv) a[e] = fma(p.Z[(size_t)(v0 + e) * p.ldg + i], d, a[e]);
                }
#pragma unroll
                for (int e = 0; e < 4; e++) {
                    const double t = warp_sum_fixed(a[e]);
                    if (lane == 0 && e < nv) mo[2 + v0 + e] = t;
                }
            }
        }
        __syncwarp();
        if (lane < cnt) {
            const double *mo = mom + (size_t)lane * mw;
            const double gbar = mo[0], Sgg = mo[1];
            double Szg[kKinMleMaxM];
            for (int l = 0; l < kKinMleMaxM; l++) Szg[l] = l < m ? mo[2 + l] : 0.0;
            // [(X'X)^-1]_gg = 1 / (Sgg - Szg' Szz^-1 Szg); a column inside span[1 | PCs] has no inverse (mle.rs:143-148: Err -> NaN)
            double proj = 0.0;
            for (int a = 0; a < m; a++)
                for (int b = 0; b < m; b++) proj += Szg[a] * Wzz[a * m + b] * Szg[b];
            const double den = Sgg - proj;
            const bool singular = !(den > fmax(64.0, nn * nn) * kEps * kEps * (Sgg + nn * gbar * gbar));
            const double dgi = 1.0 / den;
            for (int j = 0; j < k; j++) {
                const double *pf = phf + (size_t)j * (2 + m);
                const double ybar = pf[0], Syy = pf[1], Sgy = mo[2 + m + j];
                const double *Szy = pf + 2;
                double o0 = nan(""), o1 = nan(""), o3 = nan("");
                if (!singular) {
                    auto cost = [&](const double *par) {
                        const double s2 = bound_logit(par[0], kEps, 1e9);
                        const double *bz = par + 2, bg = par[2 + m];
                        double lin = bg * Sgy, quad = bg * bg * Sgg, off = ybar - par[1] - bg * gbar, cross = 0.0;
                        for (int a = 0; a < m; a++) {
                            lin += bz[a] * Szy[a];
                            off -= bz[a] * zbar[a];
                            cross += bz[a] * Szg[a];
                            double r = 0.0;
                            for (int b = 0; b < m; b++) r += Szz[a * m + b] * bz[b];
                            quad += bz[a] * r;
                        }
                        const double rss = (Syy - 2.0 * lin + (quad + 2.0 * bg * cross)) + nn * off * off;
                        return (nn / 2.00) * log(2.00 * 3.14159265358979323846264338327950288 * s2) + (1.00 / s2) * rss;
                    };
                    double par[kKmMaxD];
                    nelder_mead<kKmMaxD>(cost, m + 3, 1.0, 1000, par);
                    const double ve = bound_logit(par[0], kEps, 1e9);
                    o0 = par[2 + m];
                    o1 = ve * dgi;
                    const double t = o0 / o1;
                    if (isinf(t))
                        o3 = 0.0;
                    else if (t != t)
                        o3 = 1.0;
                    else
                        o3 = p.ptab ? student_two_sided_tab(fabs(t), p.df, ptab) : student_two_sided(fabs(t), p.df, p.ln_beta);
                }
                const size_t at = (size_t)j * p.P + (size_t)(c0 + lane);
                p.beta[at] = o0;
                p.var[at] = o1;
                p.pval[at] = o3;
            }
        }
        __syncwarp();
    }
}

cudaError_t launch_kin_mle(const KinMleParams &p, int sm_count, cudaStream_t s) {
    if (p.P == 0) return cudaSuccess;
    const int nfix = p.m + 2 * p.m * p.m + p.k * (2 + p.m);
    const int fix_pad = (nfix + 1) & ~1;
    const size_t smem = ((size_t)fix_pad + (size_t)kKmWarps * 32 * (2 + p.m + p.k)) * 8;
    cudaError_t e = cudaFuncSetAttribute(kin_mle_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    int64_t grid = ((p.P + 31) / 32 + kKmWarps - 1) / kKmWarps;
    if (grid > (int64_t)sm_count * 4) grid = (int64_t)sm_count * 4;
    kin_mle_kernel<<<(unsigned)grid, kKmWarps * 32, smem, s>>>(p, fix_pad);
    return cudaGetLastError();
}

cudaError_t launch_nm(const NmParams &p, int sm_count, cudaStream_t s) {
    if (p.n_loci == 0) return cudaSuccess;
    if (p.kind == PG_KIND_MLE) {
        const size_t smem = (size_t)kMleWarps * 32 * mle_mom_stride(p.k) * 8;
        cudaError_t e = cudaFuncSetAttribute(mle_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        int per_sm = 0;  // resident CTAs per SM as registers and shared memory allow: whole waves of them
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, mle_kernel, kMleWarps * 32, smem);
        if (e != cudaSuccess) return e;
        if (per_sm < 1) per_sm = 1;
        int64_t grid = ((p.n_loci + 31) / 32 + kMleWarps - 1) / kMleWarps;
        if (grid > (int64_t)sm_count * per_sm) grid = (int64_t)sm_count * per_sm;
        mle_kernel<<<(unsigned)grid, kMleWarps * 32, smem, s>>>(p);
    } else {
        int64_t grid = (p.n_loci * (p.lay.A - 1) + 127) / 128;
        if (grid > (int64_t)sm_count * 8) grid = (int64_t)sm_count * 8;
        gwalpha_kernel<<<(unsigned)grid, 128, 0, s>>>(p);
    }
    return cudaGetLastError();
}

}  // namespace pg
