// pg_kinship.cu -- ols_iter_with_kinship (ols_with_covariate, src/gwas/ols.rs:278-436) on sm_100a:
//   load_*        LoadAll::load + into_genotypes_and_phenotypes (src/base/sync.rs:973-1179): a slab of parsed loci ->
//                 filter -> renormalised frequencies of the kept alleles -> allele columns G[:, c] (column-major,
//                 one column contiguous), i.e. intercept_and_allele_frequencies[:, 1..]
//   gram_kernel   K_partial = G G' (src/gwas/ols.rs:295), FP64 tensor cores (mma.sync m8n8k4 f64 -> SASS DMMA),
//                 operands staged through shared memory by bulk copies, split over column slices and the upper
//                 triangle of 128 x 128 tiles; the slices are summed in a fixed order (bit-reproducible)
//   eig_select    kinship.eig() + PC selection (ols.rs:296-315): cuSOLVER syevd, eigenvalues taken from high to low
//                 as the reference assumes, covariates = the first m eigenvectors
//   covar_kernel  the per-column regression with X = [1 | PCs | g] (ols.rs:340-370) in its Frisch-Waugh form: with Q
//                 an orthonormal basis of [1 | PCs] and y~ = y - QQ'y,  b = g'y~ / (g'g - |Q'g|^2),
//                 RSS = y~'y~ - b g'y~, var = RSS / (n - (2+m)) / (g'g - |Q'g|^2), p from Student-t(n-1) -- identical to
//                 the last coefficient of the reference's normal equations up to rounding
#include <cub/device/device_scan.cuh>
#include <cusolverDn.h>
#include <dlfcn.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <chrono>
#include <new>
#include <vector>

#include "pg_device.cuh"
#include "pg_internal.h"
#include "pg_ptable.h"
#include "pg_kin.h"

namespace pg {

// ================================================================================================================
// 1. column loader
// ================================================================================================================
struct LoadParams {
    const uint32_t *counts;  // [locus][A_in][n]
    int64_t n_loci;
    int n, A_in, drop_col, ldg;
    int keep_p_minus_1;
    double maf, one_minus_maf, max_miss, min_depth_f;
    const double *w;  // [n] s_i / sum(s)
    uint8_t codes[8];
    uint32_t *sel;      // [locus] number of columns (bits 0-3) | 3-bit input column index of emitted column s << (4 + 3 s),
                        // s < 6 (bits 4-21) | kept set << 24 (bits 24-29)
    int64_t *offsets;   // [locus] exclusive scan of the column counts
    double *G;          // [column][ldg]
    int64_t col_base;
    int64_t *col_locus;  // [column] locus ordinal inside the slab
    uint8_t *col_allele; // [column] allele code
};

// pass 1: one warp per locus, lane = pool (stride 32): the reference's keep-mask and, with keep_p_minus_1, its order
__global__ void __launch_bounds__(256) load_decide_kernel(const LoadParams p) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int A = p.A_in - (p.drop_col >= 0 ? 1 : 0);
    for (int64_t locus = warp; locus < p.n_loci; locus += nwarps) {
        const uint32_t *cl = p.counts + (size_t)locus * p.A_in * p.n;
        int col_of[PG_MAX_ALLELES];
        {
            int jj = 0;
            for (int j = 0; j < p.A_in; j++)
                if (j != p.drop_col) col_of[jj++] = j;
        }
        // depth filter and first-stage pooled frequencies q_j (parallel sums, exact re-evaluation near a threshold)
        double qs[PG_MAX_ALLELES];
        for (int j = 0; j < PG_MAX_ALLELES; j++) qs[j] = 0.0;
        uint32_t dmin = 0xFFFFFFFFu;
        int miss = 0;
        for (int i = lane; i < p.n; i += 32) {
            uint64_t d = 0;
            uint32_t c[PG_MAX_ALLELES];
            for (int j = 0; j < A; j++) {
                c[j] = cl[(size_t)col_of[j] * p.n + i];
                d += c[j];
            }
            if (d > 0xFFFFFFFEull) d = 0xFFFFFFFEull;
            dmin = min(dmin, (uint32_t)d);
            if (d == 0) {
                miss++;
            } else {
                const double dd = (double)d, wi = p.w[i];
                for (int j = 0; j < A; j++) qs[j] = fma((double)c[j] / dd, wi, qs[j]);
            }
        }
        dmin = __reduce_min_sync(PG_FULL_MASK, dmin);
        miss = __reduce_add_sync(PG_FULL_MASK, miss);
        uint32_t sel = 0;
        bool keep = !((double)dmin < p.min_depth_f);
        unsigned kept = 0;
        if (keep) {
            const double tol = 2.0 * ((double)p.n + 8.0) * kEps;
            for (int j = 0; j < A; j++) {
                double q = qs[j];
                for (int off = 16; off >= 1; off >>= 1) q += __shfl_xor_sync(PG_FULL_MASK, q, off);
                const double tl = tol * fmax(fabs(q), 1.0);
                if (fabs(q - p.maf) <= tl || fabs(q - p.one_minus_maf) <= tl) {
                    // the reference's order: sequential over the pools, separately rounded multiply and add
                    double qe = 0.0;
                    if (lane == 0) {
                        for (int i = 0; i < p.n; i++) {
                            uint64_t d = 0;
                            for (int l = 0; l < A; l++) d += cl[(size_t)col_of[l] * p.n + i];
                            if (d == 0) continue;
                            const double f = (double)cl[(size_t)col_of[j] * p.n + i] / (double)d;
                            qe = __dadd_rn(qe, __dmul_rn(f, p.w[i]));
                        }
                    }
                    q = __shfl_sync(PG_FULL_MASK, qe, 0);
                }
                if (!((q < p.maf) | (q > p.one_minus_maf))) kept |= 1u << j;
            }
            if (__popc(kept) < 2) keep = false;
            // missingness on the first kept column (sync.rs:287-299)
            if (keep && (miss == p.n || ((double)miss / (double)p.n) > p.max_miss)) keep = false;
        }
        if (keep) {
            int order[PG_MAX_ALLELES], no = 0;
            for (int j = 0; j < A; j++)
                if ((kept >> j) & 1u) order[no++] = j;
            if (p.keep_p_minus_1) {
                // sort_by_allele_freq(true) then drop the first column (sync.rs:1017-1027, 478-505): column sums of the
                // renormalised frequencies, sequential over the pools (lane j sums column j)
                double cs = 0.0;
                if (lane < A && ((kept >> lane) & 1u)) {
                    for (int i = 0; i < p.n; i++) {
                        uint64_t dk = 0;
                        for (int l = 0; l < A; l++)
                            if ((kept >> l) & 1u) dk += cl[(size_t)col_of[l] * p.n + i];
                        if (dk == 0) continue;
                        cs = __dadd_rn(cs, (double)cl[(size_t)col_of[lane] * p.n + i] / (double)dk);
                    }
                }
                double csj[PG_MAX_ALLELES];
                for (int j = 0; j < A; j++) csj[j] = __shfl_sync(PG_FULL_MASK, cs, j);
                int sorted[PG_MAX_ALLELES];
                for (int a = 0; a < no; a++) {
                    const int j = order[a];
                    int rank = 0;
                    for (int b = 0; b < no; b++) {
                        const int l = order[b];
                        if (l != j && (csj[l] > csj[j] || (csj[l] == csj[j] && l < j))) rank++;
                    }
                    sorted[rank] = j;
                }
                no -= 1;
                for (int a = 0; a < no; a++) order[a] = sorted[a + 1];
            }
            sel = (uint32_t)no;
            for (int a = 0; a < no; a++) sel |= (uint32_t)order[a] << (4 + 3 * a);
            sel |= kept << 24;
        }
        if (lane == 0) {
            p.sel[locus] = sel;
            p.offsets[locus] = (int64_t)(sel & 0xf);
        }
    }
}

// pass 2: renormalised frequencies of the emitted columns (to_frequencies after the filter, sync.rs:166-192)
__global__ void __launch_bounds__(256) load_emit_kernel(const LoadParams p) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int A = p.A_in - (p.drop_col >= 0 ? 1 : 0);
    for (int64_t locus = warp; locus < p.n_loci; locus += nwarps) {
        const uint32_t sel = p.sel[locus];
        const int no = (int)(sel & 0xf);
        if (no == 0) continue;
        const unsigned kept = (sel >> 24) & 0x3fu;
        const int64_t c0 = p.col_base + p.offsets[locus];
        const uint32_t *cl = p.counts + (size_t)locus * p.A_in * p.n;
        int col_of[PG_MAX_ALLELES];
        {
            int jj = 0;
            for (int j = 0; j < p.A_in; j++)
                if (j != p.drop_col) col_of[jj++] = j;
        }
        for (int i = lane; i < p.ldg; i += 32) {
            uint64_t dk = 0;
            if (i < p.n)
                for (int l = 0; l < A; l++)
                    if ((kept >> l) & 1u) dk += cl[(size_t)col_of[l] * p.n + i];
            for (int a = 0; a < no; a++) {
                const int j = (int)((sel >> (4 + 3 * a)) & 0x7);
                double v = 0.0;
                if (i < p.n) v = dk ? (double)cl[(size_t)col_of[j] * p.n + i] / (double)dk : nan("");
                p.G[(size_t)(c0 + a) * p.ldg + i] = v;
            }
        }
        if (lane < no) {
            const int j = (int)((sel >> (4 + 3 * lane)) & 0x7);
            p.col_locus[c0 + lane - p.col_base] = locus;
            p.col_allele[c0 + lane - p.col_base] = p.codes[col_of[j]];
        }
    }
}

// synthetic biallelic columns for the C4 workload: locus l contributes two columns f and 1 - f over the pools, built
// from the same integer-hash counts as the scan workload (alleles A and T only)
__global__ void __launch_bounds__(256) kin_synth_kernel(uint64_t seed, int64_t first_locus, int64_t n_loci, int n,
                                                        int ldg, double *G) {
    const int64_t total = n_loci * ldg;
    for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
         idx += (int64_t)gridDim.x * blockDim.x) {
        const int64_t l = idx / ldg;
        const int i = (int)(idx - l * ldg);
        double f0 = 0.0, f1 = 0.0;
        if (i < n) {
            uint32_t c[PG_MAX_ALLELES];
            synth_counts(seed, first_locus + l, i, 4, c);
            const uint32_t a = c[0] + c[2], b = c[1] + c[3];  // fold to two alleles, depth 20..100 (or 0)
            const uint32_t d = a + b;
            f0 = d ? (double)a / (double)d : 0.5;
            f1 = d ? (double)b / (double)d : 0.5;
        }
        G[(size_t)(2 * l) * ldg + i] = f0;
        G[(size_t)(2 * l + 1) * ldg + i] = f1;
    }
}

// ================================================================================================================
// 2. kinship Gram matrix: FP64 DMMA SYRK
// ================================================================================================================
constexpr int kTile = 128;           // C tile edge
constexpr int kKC = 16;              // columns of G (the contraction index) per stage
constexpr int kPitch = kTile + 4;    // shared row pitch: 132 = 4 (mod 16) doubles -> conflict-free fragment loads
constexpr int kStages = 4;
constexpr int kGramWarps = 8;        // consumer warps: 2 (rows) x 4 (columns), warp tile 64 x 32

__device__ __forceinline__ void dmma884(double &d0, double &d1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(d0), "+d"(d1)
                 : "d"(a), "d"(b));
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

struct GramParams {
    const double *G;   // [P_pad][ldg]
    int64_t P_pad;     // multiple of kKC, the pad columns are zero
    int ldg, n;
    int nt;            // tiles per edge
    int n_slices;
    int64_t slice_cols;  // multiple of kKC
    double *ws;        // [slice][tile][kTile*kTile]
};

__global__ void __launch_bounds__((kGramWarps + 1) * 32, 1) gram_kernel(const GramParams p) {
    extern __shared__ __align__(128) unsigned char smem[];
    uint64_t *full = reinterpret_cast<uint64_t *>(smem);
    uint64_t *empty = full + kStages;
    double *tiles = reinterpret_cast<double *>(smem + 128);  // [stage][2][kKC][kPitch]
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        for (int s = 0; s < kStages; s++) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], kGramWarps);
        }
        fence_mbar_init();
    }
    __syncthreads();
    const int ntiles = p.nt * (p.nt + 1) / 2;
    const int64_t n_items = (int64_t)ntiles * p.n_slices;
    uint32_t it_stage = 0;  // running stage counter (same sequence on the producer and the consumers)
    for (int64_t item = blockIdx.x; item < n_items; item += gridDim.x) {
        const int slice = (int)(item / ntiles);
        int tile = (int)(item - (int64_t)slice * ntiles);
        int ti = 0;
        while (tile >= p.nt - ti) {  // row ti of the upper triangle holds nt - ti tiles
            tile -= p.nt - ti;
            ti++;
        }
        const int tj = ti + tile;
        const bool diag = ti == tj;
        const int64_t k_begin = (int64_t)slice * p.slice_cols;
        const int64_t k_end = min(p.P_pad, k_begin + p.slice_cols);
        const int n_steps = (int)((k_end - k_begin + kKC - 1) / kKC);
        if (warp == kGramWarps) {
            // ---- producer warp: lane r < 16 copies row r of the A tile, lane 16 + r row r of the B tile
            for (int st = 0; st < n_steps; st++) {
                const uint32_t s = (it_stage + st) % kStages, use = (it_stage + st) / kStages;
                if (use > 0) mbar_wait(&empty[s], (use - 1) & 1u);
                if (lane == 0) mbar_expect_tx(&full[s], (uint32_t)(kKC * kTile * 8 * (diag ? 1 : 2)));
                __syncwarp();
                const int r = lane & 15, which = lane >> 4;
                if (which == 0 || !diag) {
                    const int64_t k = k_begin + (int64_t)st * kKC + r;
                    const double *src = p.G + (size_t)k * p.ldg + (size_t)(which ? tj : ti) * kTile;
                    double *dst = tiles + ((size_t)(s * 2 + which) * kKC + r) * kPitch;
                    bulk_g2s(dst, src, kTile * 8, &full[s]);
                }
            }
        } else {
            // ---- consumer warps
            const int wm = warp >> 2, wn = warp & 3, g = lane >> 2, t = lane & 3;
            double acc[8][4][2];
#pragma unroll
            for (int mi = 0; mi < 8; mi++)
#pragma unroll
                for (int ni = 0; ni < 4; ni++) acc[mi][ni][0] = acc[mi][ni][1] = 0.0;
            for (int st = 0; st < n_steps; st++) {
                const uint32_t s = (it_stage + st) % kStages, use = (it_stage + st) / kStages;
                mbar_wait(&full[s], use & 1u);
                const double *As = tiles + (size_t)(s * 2) * kKC * kPitch + wm * 64 + g;
                const double *Bs = tiles + (size_t)(s * 2 + (diag ? 0 : 1)) * kKC * kPitch + wn * 32 + g;
#pragma unroll
                for (int kk = 0; kk < kKC / 4; kk++) {
                    double a[8], b[4];
#pragma unroll
                    for (int mi = 0; mi < 8; mi++) a[mi] = As[(kk * 4 + t) * kPitch + mi * 8];
#pragma unroll
                    for (int ni = 0; ni < 4; ni++) b[ni] = Bs[(kk * 4 + t) * kPitch + ni * 8];
#pragma unroll
                    for (int mi = 0; mi < 8; mi++)
#pragma unroll
                        for (int ni = 0; ni < 4; ni++) dmma884(acc[mi][ni][0], acc[mi][ni][1], a[mi], b[ni]);
                }
                __syncwarp();
                if (lane == 0) mbar_arrive(&empty[s]);
            }
            // partial tile of this (slice, tile) -> workspace
            double *out = p.ws + ((size_t)slice * ntiles + (item - (int64_t)slice * ntiles)) * (kTile * kTile);
#pragma unroll
            for (int mi = 0; mi < 8; mi++)
#pragma unroll
                for (int ni = 0; ni < 4; ni++) {
                    const int row = wm * 64 + mi * 8 + g, col = wn * 32 + ni * 8 + 2 * t;
                    *reinterpret_cast<double2 *>(out + (size_t)row * kTile + col) =
                        make_double2(acc[mi][ni][0], acc[mi][ni][1]);
                }
        }
        it_stage += (uint32_t)n_steps;
    }
}

// K[i][j] = K[j][i] = sum over the slices (fixed order) of the partial tiles; with `accumulate` that sum is added to the
// K a previous block left (read from the upper triangle, both triangles written from the one value: K stays exactly
// symmetric and a given split into blocks is bit-repeatable)
__global__ void __launch_bounds__(256) gram_reduce_kernel(const double *ws, int nt, int n_slices, int n, int accumulate,
                                                          double *K) {
    const int ntiles = nt * (nt + 1) / 2;
    const int64_t total = (int64_t)ntiles * kTile * kTile;
    for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
         idx += (int64_t)gridDim.x * blockDim.x) {
        int tile = (int)(idx / (kTile * kTile));
        const int e = (int)(idx - (int64_t)tile * kTile * kTile);
        const int tile_id = tile;
        int ti = 0;
        while (tile >= nt - ti) {
            tile -= nt - ti;
            ti++;
        }
        const int tj = ti + tile;
        const int i = ti * kTile + e / kTile, j = tj * kTile + e % kTile;
        if (i >= n || j >= n || j < i) continue;
        double s = 0.0;
        for (int sl = 0; sl < n_slices; sl++) s += ws[((size_t)sl * ntiles + tile_id) * (kTile * kTile) + e];
        if (accumulate) s = K[(size_t)i * n + j] + s;
        K[(size_t)i * n + j] = s;
        K[(size_t)j * n + i] = s;
    }
}

// ================================================================================================================
// 3. covariate scan
// ================================================================================================================
struct CovarParams {
    const double *G;
    int64_t P;
    int ldg, n;
    int nq;            // columns of Q = 1 + m
    int k;             // phenotypes
    const double *V;   // [nq + k][ldg]: Q columns then y~ columns (device)
    double yy[kMaxPhenPerPass * 4];  // y~'y~ per phenotype (k <= 16)
    double dfe;        // n - (2 + m)
    double df;         // n - 1
    // n < p branch (src/gwas/ols.rs:67-75): the threshold was never reached, so ALL n eigenvectors are covariates
    // (ols.rs:300-311) and X = [1 | V | g] has n + 2 columns.  With V orthogonal XX' = I + 11' + gg', and the last
    // coefficient of X'(XX')^-1 y follows from the same sums the kernel forms with Q = [1/sqrt(n)] and the RAW
    // phenotypes (Woodbury on the rank-2 update); var = (e'e / -2) (...) is rounding noise over a negative number, so
    // t is NaN and p is forced to 1 (ols.rs:150-151)
    int minnorm;
    int y0;            // covar_mma_kernel: first phenotype of this pass (p.k counts the phenotypes of the pass)
    // covar_mma_kernel over a pool range [pr0, pr0 + pn): with V of all pools in shared memory little L1 is left for the
    // loads in flight, so wide V is taken in pool passes -- a pass that is not the last leaves its partial U and g'g per
    // column block in `part` (part_mode bit 0), a pass that is not the first adds them to its own (bit 1) and the last
    // one finishes; 0 = all pools at once
    int pr0, pn, part_mode;
    double *part;      // [column block][(8 MT + 1) * 8]
    int64_t *defer_list;     // covar_mma_kernel: columns whose centred g'g is lost to cancellation, finished by
    unsigned *defer_count;   //   covar_generic_kernel (two-pass form); covar_generic_kernel: the columns to process
    double nf, sqrt_n;
    double sy[kMaxPhenPerPass * 4];  // sum of the raw phenotype
    const void *ptab;
    double ptab_isd, ptab_bits, ptab_t1, ptab_t0;  // t1 / t0: PTable::t_one / t_zero
    int ptab_M;
    double ln_beta;
    double *beta, *var, *pval;  // [k][P]
};

// last coefficient of the minimum-norm solution with X = [1 | V | g], V orthogonal: b = g'(I + UU')^-1 y, U = [1 g];
// (I + UU')^-1 = I - U (I_2 + U'U)^-1 U'.  u0 = g'1 / sqrt(n), gy = g'y (raw phenotype j)
__device__ __forceinline__ void covar_minnorm(const CovarParams &p, double gg, double u0, double gy, int j, double &b,
                                              double &pv) {
    const double s = u0 * p.sqrt_n;
    const double w11 = 1.0 + p.nf, w22 = 1.0 + gg;
    const double det = w11 * w22 - s * s;  // >= 1 + n + gg > 0 (Cauchy-Schwarz: s^2 <= n gg)
    const double z0 = (w22 * p.sy[j] - s * gy) / det, z1 = (w11 * gy - s * p.sy[j]) / det;
    b = gy - (s * z0 + gg * z1);
    pv = (b == b) ? 1.0 : nan("");
}

// the residual sum of squares y~'y~ - b g~'y~ carries the digits the centred g'g lost times y~'y~ / rss: beyond this
// product it is re-formed from explicit residuals (4 eps x 1e5 keeps 1e-10)
constexpr double kCovarRssRedo = 1e-5;  // (g'g / g~'g~) (y~'y~ / rss) above 1e5

// NV = (1 + m) + k vectors in shared memory; a warp streams C allele columns at once so that every shared-memory load
// of a Q / y~ element feeds C pairs of FMAs (with m = 10 covariates the one-column form spends its time on 12 LDS per
// element of g: 0.30 of the HBM roofline; C = 4 columns share them)
template <int NV, int C, bool LIST>
__global__ void __launch_bounds__(512) covar_kernel(const CovarParams p) {
    static_assert(!LIST || C == 1, "the column list is walked one column at a time");
    extern __shared__ __align__(16) double vs[];  // [NV][ldg]
    const int ldg = p.ldg;
    for (int i = threadIdx.x; i < NV * ldg; i += blockDim.x) vs[i] = p.V[i];
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const PTableDev ptab = {reinterpret_cast<const double4 *>(p.ptab), p.ptab_isd, p.ptab_bits, p.ptab_t1, p.ptab_t0, p.ptab_M};
    const int nq = p.nq, k = p.k;
    // LIST: the columns a streaming kernel (this one with LIST = false, or the DMMA form) left to the explicit-residual
    // forms; the streaming instantiations carry none of that code
    const int64_t n_items = LIST ? (int64_t)*p.defer_count : p.P;
    for (int64_t i0 = warp * C; i0 < n_items; i0 += nwarps * C) {
        const int64_t c0 = LIST ? p.defer_list[i0] : i0;
        double accs[C][NV], ggs[C];
#pragma unroll
        for (int cc = 0; cc < C; cc++) {
            ggs[cc] = 0.0;
#pragma unroll
            for (int v = 0; v < NV; v++) accs[cc][v] = 0.0;
        }
        const double *g0 = p.G + (size_t)c0 * ldg;
#pragma unroll(C == 1 ? 4 : 2)
        for (int r = 2 * lane; r < ldg; r += 64) {
            double2 g2[C];
#pragma unroll
            for (int cc = 0; cc < C; cc++)
                g2[cc] = (c0 + cc < p.P) ? __ldcs(reinterpret_cast<const double2 *>(g0 + (size_t)cc * ldg + r))
                                         : make_double2(0.0, 0.0);
#pragma unroll
            for (int cc = 0; cc < C; cc++) {
                ggs[cc] = fma(g2[cc].x, g2[cc].x, ggs[cc]);
                ggs[cc] = fma(g2[cc].y, g2[cc].y, ggs[cc]);
            }
#pragma unroll
            for (int v = 0; v < NV; v++) {
                const double2 q2 = *reinterpret_cast<const double2 *>(vs + (size_t)v * ldg + r);
#pragma unroll
                for (int cc = 0; cc < C; cc++) {
                    accs[cc][v] = fma(g2[cc].x, q2.x, accs[cc][v]);
                    accs[cc][v] = fma(g2[cc].y, q2.y, accs[cc][v]);
                }
            }
        }
#pragma unroll
        for (int cc = 0; cc < C; cc++) {
            const int64_t c = c0 + cc;
            if (c >= p.P) continue;  // warp-uniform (no break: the loop must unroll so that accs stays in registers)
            const double *g = g0 + (size_t)cc * ldg;
            double acc[NV];
            double gg = warp_sum_fixed(ggs[cc]);
#pragma unroll
            for (int v = 0; v < NV; v++) acc[v] = warp_sum_fixed(accs[cc][v]);
            double uu = 0.0;
#pragma unroll
            for (int v = 0; v < NV; v++)
                if (v < nq) uu = fma(acc[v], acc[v], uu);
            double ggc = gg - uu;
            double gy[NV];
#pragma unroll
            for (int v = 0; v < NV; v++) gy[v] = acc[v];
            const bool redone = !p.minnorm && gg == gg && !(gg <= 1e4 * ggc);  // NaN frequencies: nothing to redo
            if (redone) {
                // cancellation: second pass with explicit residuals g - Q u (the column is still in L2)
                double s2 = 0.0, sy[NV];
#pragma unroll
                for (int v = 0; v < NV; v++) sy[v] = 0.0;
                // (pool pairs, two of them in flight per lane: the chain over the Q columns is latency bound; rows
                // n..ldg hold zeros in G and in V)
                double s2b = 0.0;
#pragma unroll 2
                for (int r = 2 * lane; r < ldg; r += 64) {
                    double2 e = *reinterpret_cast<const double2 *>(g + r);
#pragma unroll
                    for (int v = 0; v < NV; v++)
                        if (v < nq) {
                            const double2 q2 = *reinterpret_cast<const double2 *>(vs + (size_t)v * ldg + r);
                            e.x = fma(-acc[v], q2.x, e.x);
                            e.y = fma(-acc[v], q2.y, e.y);
                        }
                    s2 = fma(e.x, e.x, s2);
                    s2b = fma(e.y, e.y, s2b);
#pragma unroll
                    for (int v = 0; v < NV; v++)
                        if (v >= nq) {
                            const double2 q2 = *reinterpret_cast<const double2 *>(vs + (size_t)v * ldg + r);
                            sy[v] = fma(e.x, q2.x, sy[v]);
                            sy[v] = fma(e.y, q2.y, sy[v]);
                        }
                }
                ggc = warp_sum_fixed(s2 + s2b);
#pragma unroll
                for (int v = 0; v < NV; v++)
                    if (v >= nq) gy[v] = warp_sum_fixed(sy[v]);
                // the column lies in span([1 | PCs]) to working precision (a monomorphic locus gives g = 1 or g = 0):
                // the reference's X'X is singular (exactly so for those two) and inv() fails -> NaN (ols.rs:359-364)
                if (ggc <= fmax(64.0, p.nf * p.nf) * kEps * kEps * gg) ggc = 0.0;  // below (n eps)^2 the reference's pivot is noise
            }
            // lane j < k finishes phenotype j
            double b = nan(""), vb = nan(""), pv = nan("");
            double gyj = 0.0, yyj = 0.0;
#pragma unroll
            for (int v = 0; v < NV; v++)
                if (v - nq == lane) gyj = gy[v];
#pragma unroll
            for (int j = 0; j < kMaxPhenPerPass * 4; j++)
                if (j == lane) yyj = p.yy[j];
            const bool solve = lane < k && !p.minnorm && ggc > 0.0 && p.dfe > 0.0;
            double rss = 0.0;
            if (solve) {
                b = gyj / ggc;
                rss = yyj - b * gyj;
            }
            // a near-perfect fit (everyday with a handful of pools: 1 - r^2 of three points piles up at 0) leaves
            // y~'y~ - b g~'y~ to cancellation, on top of what the centred g'g lost: explicit residuals
            // y~ - b (g - Q u) like the reference (ols.rs:102).  The streaming form only names the column.
            unsigned small = __ballot_sync(PG_FULL_MASK, solve && !(kCovarRssRedo * (redone ? ggc : gg) * yyj <= rss * ggc));
            if (!LIST) {
                if (small && lane == 0) p.defer_list[atomicAdd(p.defer_count, 1u)] = c;
            } else {
                while (small) {
                    const int j = __ffs(small) - 1;
                    small &= small - 1;
                    const double bj = __shfl_sync(PG_FULL_MASK, b, j);
                    double s2 = 0.0, s2b = 0.0;
#pragma unroll 2
                    for (int r = 2 * lane; r < ldg; r += 64) {
                        double2 e = *reinterpret_cast<const double2 *>(g + r);
#pragma unroll
                        for (int v = 0; v < NV; v++)
                            if (v < nq) {
                                const double2 q2 = *reinterpret_cast<const double2 *>(vs + (size_t)v * ldg + r);
                                e.x = fma(-acc[v], q2.x, e.x);
                                e.y = fma(-acc[v], q2.y, e.y);
                            }
                        const double2 y2 = *reinterpret_cast<const double2 *>(vs + (size_t)(nq + j) * ldg + r);
                        e.x = fma(-bj, e.x, y2.x);
                        e.y = fma(-bj, e.y, y2.y);
                        s2 = fma(e.x, e.x, s2);
                        s2b = fma(e.y, e.y, s2b);
                    }
                    s2 = warp_sum_fixed(s2 + s2b);
                    if (lane == j) rss = s2;
                }
            }
            if (lane < k) {
                if (p.minnorm) {
                    covar_minnorm(p, gg, acc[0], gyj, lane, b, pv);
                } else if (solve) {
                    if (rss < 0.0) rss = 0.0;
                    vb = rss / p.dfe / ggc;
                    // estimate_significance, src/gwas/ols.rs:139-154
                    const double tt = (fabs(b) <= kEps) ? 0.0 : b / sqrt(vb);
                    if (fabs(tt) <= kEps || tt != tt)
                        pv = 1.0;
                    else
                        pv = p.ptab ? student_two_sided_tab(fabs(tt), p.df, ptab) : student_two_sided(fabs(tt), p.df, p.ln_beta);
                } else if (gg != gg) {
                    pv = 1.0;  // NaN frequencies: the reference's t is NaN and its p is forced to 1 (ols.rs:150-151)
                }
                p.beta[(size_t)lane * p.P + c] = b;
                p.var[(size_t)lane * p.P + c] = vb;
                p.pval[(size_t)lane * p.P + c] = pv;
            }
        }
    }
}

// ---- covariate scan with selected PCs as a blocked FP64 contraction -----------------------------------------------
// With m covariates the per-column work is U = V'g for the NV = 1 + m + k vectors (Q columns, then y~): a NV x n by
// n x P contraction.  As per-warp dot products every element of g costs NV shared-memory operand loads (m = 10: 0.35 of
// the HBM roofline, shared-memory bandwidth and issue bound).  Here a warp owns 8 allele columns and forms
// U[v][c] with mma.sync.m8n8k4.f64 (SASS DMMA): M = vectors (MT tiles of 8), N = the 8 columns, K = pools.
// The sum over pools may take the pools in any order as long as both operands agree: of a 16-pool block lane (g, t)
// holds pools {2t, 2t+1, 8+2t, 8+2t+1} of its column g -- two 128-bit loads straight from global memory (G is streamed
// once, no staging: the shared memory belongs to V; the four lanes of a column cover 64 contiguous bytes per request,
// i.e. whole sectors) -- and the matching elements of vector row g from shared memory (pitch = 8 mod 16 doubles:
// conflict-free LDS.128); DMMA number s of a block contracts the s-th of those pools.  HBM wants ~110 KB in flight per
// SM and the shared memory is taken, so the in-flight data lives in REGISTERS: a lane holds a ring of eight blocks and
// reloads a slot the moment its block has been consumed (across the boundary to the warp's next column block), which
// keeps 224 bytes per lane = 115 KB per SM in flight with 16 warps.  Two accumulator sets per M tile keep four
// independent DMMA chains per warp; g'g accumulates beside it.  Every U[v][c] ends up in exactly one lane (no
// cross-lane reduction); a per-warp scratch hands the 8 columns' sums to the lanes that finish (column, phenotype)
// pairs.  Columns whose centred g'g is lost to cancellation (nearly constant columns) go to a list that
// covar_kernel<NV, 1> finishes in its two-pass form -- the streaming kernel carries no slow path.
// Measured alternatives (DESIGN.md 5): loads and DMMAs in alternating trips (24 warps), a two-trip register double
// buffer, L2 bulk prefetches ahead of the loads, 16 columns per warp, and a CTA-cooperative form in which the warps
// split the pools of one column block and hand partial tiles over named barriers.
constexpr int kCmMaxWarps = 16;
constexpr int kCmRing = 8;  // 16-pool blocks a lane holds in registers (256 bytes)

template <int MT>
__global__ void __launch_bounds__(kCmMaxWarps * 32, 1) covar_mma_kernel(const CovarParams p, int ldq, int n_warps) {
    extern __shared__ __align__(16) double cm_sm[];  // V [NV][ldq] | scratch [n_warps][(8 MT + 1) * 8]
    const int ldg = p.ldg, n = p.pn, nq = p.nq, k = p.k, NV = nq + k;  // n: the pools of this pass
    double *Vs = cm_sm;
    for (int i = threadIdx.x; i < NV * ldq; i += blockDim.x) {
        const int v = i / ldq, r = i - v * ldq;
        // the Q columns, then the y~ columns of this phenotype pass (p.k of them, starting at p.V's column nq + p.y0)
        Vs[i] = (r < n) ? p.V[(size_t)(v < nq ? v : v + p.y0) * ldg + p.pr0 + r] : 0.0;
    }
    __syncthreads();
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5, g = lane >> 2, t = lane & 3;
    constexpr int SCR = (8 * MT + 1) * 8;
    double *scr = cm_sm + (size_t)NV * ldq + (size_t)wib * SCR;  // U [8 MT][8] | g'g [8]
    const PTableDev ptab = {reinterpret_cast<const double4 *>(p.ptab), p.ptab_isd, p.ptab_bits, p.ptab_t1, p.ptab_t0, p.ptab_M};
    const int64_t n_blocks = (p.P + 7) / 8;
    const int64_t wg = (int64_t)blockIdx.x * n_warps + wib, nwg = (int64_t)gridDim.x * n_warps;
    // vector rows of this lane in each M tile.  A row of D depends on its own row of A only and a column on its own
    // column of B, so rows >= NV (address clamped to row 0) and columns past the end (clamped to the block's first
    // column) simply produce sums nobody reads -- no masking multiplies on the FP64 pipe the DMMAs need
    const double *arow[MT];
#pragma unroll
    for (int mt = 0; mt < MT; mt++) {
        const int v = 8 * mt + g;
        arow[mt] = Vs + (size_t)(v < NV ? v : 0) * ldq + 2 * t;
    }
    const int nbf = n / 16;                       // whole 16-pool blocks: all of them go through the register ring
    const int nbm = nbf / kCmRing * kCmRing;      // blocks of the full ring rounds; a last partial round takes the rest
    auto col_ptr = [&](int64_t blk) {
        const int64_t c0 = blk * 8;
        return p.G + (size_t)(c0 + g < p.P ? c0 + g : c0) * ldg + p.pr0 + 2 * t;
    };
    double2 ring[kCmRing][2];
    if (wg < n_blocks) {
        const double *g0 = col_ptr(wg);
#pragma unroll
        for (int u = 0; u < kCmRing; u++) {
            if (u < nbf) {
                ring[u][0] = __ldcs(reinterpret_cast<const double2 *>(g0 + u * 16));
                ring[u][1] = __ldcs(reinterpret_cast<const double2 *>(g0 + u * 16 + 8));
            }
        }
    }
    for (int64_t blk = wg; blk < n_blocks; blk += nwg) {
        const int64_t c0 = blk * 8;
        const bool cval = c0 + g < p.P;
        const double *gb = col_ptr(blk);
        const bool has_next = blk + nwg < n_blocks;
        const double *gb_next = has_next ? col_ptr(blk + nwg) : gb;
        double acc[MT][2][2], gg = 0.0;
#pragma unroll
        for (int mt = 0; mt < MT; mt++) acc[mt][0][0] = acc[mt][0][1] = acc[mt][1][0] = acc[mt][1][1] = 0.0;
        // one 16-pool block: b0 = pools {2t, 2t+1}, b1 = pools {8+2t, 8+2t+1} of this lane's column
        auto block16 = [&](const double2 b0, const double2 b1, int i0) {
#pragma unroll
            for (int mt = 0; mt < MT; mt++) {
                const double2 a0 = *reinterpret_cast<const double2 *>(arow[mt] + i0);
                const double2 a1 = *reinterpret_cast<const double2 *>(arow[mt] + i0 + 8);
                dmma884(acc[mt][0][0], acc[mt][0][1], a0.x, b0.x);
                dmma884(acc[mt][1][0], acc[mt][1][1], a0.y, b0.y);
                dmma884(acc[mt][0][0], acc[mt][0][1], a1.x, b1.x);
                dmma884(acc[mt][1][0], acc[mt][1][1], a1.y, b1.y);
            }
            gg = fma(b0.x, b0.x, gg);
            gg = fma(b0.y, b0.y, gg);
            gg = fma(b1.x, b1.x, gg);
            gg = fma(b1.y, b1.y, gg);
        };
        // the ring: slot u holds 16-pool block rb (rb % kCmRing == u) of this column block; as soon as a block has been
        // consumed its registers take the block kCmRing further on -- of this column block or, near its end, of the
        // warp's next one -- so kCmRing - 1 blocks (224 bytes per lane) are in flight at any time
        for (int rb0 = 0; rb0 < nbm; rb0 += kCmRing) {
#pragma unroll
            for (int u = 0; u < kCmRing; u++) {
                const int rb = rb0 + u;
                block16(ring[u][0], ring[u][1], rb * 16);
                // the slot's next block: kCmRing further on in this column block, else block u of the warp's next one
                const bool here = rb + kCmRing < nbf;
                const double *src = here ? gb + (rb + kCmRing) * 16 : gb_next + u * 16;
                if (here || has_next) {
                    ring[u][0] = __ldcs(reinterpret_cast<const double2 *>(src));
                    ring[u][1] = __ldcs(reinterpret_cast<const double2 *>(src + 8));
                }
            }
        }
        if (nbm < nbf) {  // the last, partial round (slots past it already hold the next column block's data)
#pragma unroll
            for (int u = 0; u < kCmRing; u++) {
                if (nbm + u < nbf) {
                    block16(ring[u][0], ring[u][1], (nbm + u) * 16);
                    if (has_next) {
                        ring[u][0] = __ldcs(reinterpret_cast<const double2 *>(gb_next + u * 16));
                        ring[u][1] = __ldcs(reinterpret_cast<const double2 *>(gb_next + u * 16 + 8));
                    }
                }
            }
        }
        for (int i0 = nbf * 16; i0 < n; i0 += 16) {  // the partial block, if any: pools >= n read as zero
            double2 b[2];
#pragma unroll
            for (int h = 0; h < 2; h++) {
                const int r = i0 + 8 * h + 2 * t;
                b[h].x = (cval && r < n) ? __ldcs(gb + i0 + 8 * h) : 0.0;
                b[h].y = (cval && r + 1 < n) ? __ldcs(gb + i0 + 8 * h + 1) : 0.0;
            }
            block16(b[0], b[1], i0);
        }
        // g'g of column g: sum over the four lanes that share it
        gg += __shfl_xor_sync(PG_FULL_MASK, gg, 1);
        gg += __shfl_xor_sync(PG_FULL_MASK, gg, 2);
        __syncwarp();
#pragma unroll
        for (int mt = 0; mt < MT; mt++)
            *reinterpret_cast<double2 *>(scr + (8 * mt + g) * 8 + 2 * t) =
                make_double2(acc[mt][0][0] + acc[mt][1][0], acc[mt][0][1] + acc[mt][1][1]);
        if (t == 0) scr[8 * MT * 8 + g] = gg;
        __syncwarp();
        if (p.part_mode & 2) {  // not the first pool pass: add what the earlier ones parked
            const double *src = p.part + (size_t)blk * SCR;
            for (int i = lane; i < SCR; i += 32) scr[i] += src[i];
            __syncwarp();
        }
        if (p.part_mode & 1) {  // not the last pool pass: park the partial sums of this column block
            double *dst = p.part + (size_t)blk * SCR;
            for (int i = lane; i < SCR; i += 32) dst[i] = scr[i];
            __syncwarp();
            continue;
        }
        // lane = (column cc, phenotype group): centred g'g, cancellation check, records
        const int cc = lane & 7;
        const int64_t c = c0 + cc;
        const double ggv = scr[8 * MT * 8 + cc];
        double uu = 0.0;
        for (int v = 0; v < nq; v++) uu = fma(scr[v * 8 + cc], scr[v * 8 + cc], uu);
        const double ggc = ggv - uu;
        // cancellation: the column goes to the two-pass kernel (explicit residuals g - Q u), which rewrites its records
        // (a column with a NaN frequency -- a pool without coverage -- is finished below: NaN, NaN, p = 1; nothing to redo)
        bool flag = c < p.P && ggv == ggv && !(ggv <= 1e4 * ggc);
        // most flagged columns of real data are CONSTANT over the pools (a monomorphic locus gives g = 1): X'X is singular
        // like the reference's (NaN records) and the explicit-residual kernel has nothing to find out.  The warp looks at
        // such a column once more -- bit for bit against its first pool, from L2 -- here, outside the streaming loop
        bool constant = false;
        {
            unsigned todo = __ballot_sync(PG_FULL_MASK, flag && lane < 8);
            while (todo) {
                const int cf = __ffs(todo) - 1;
                todo &= todo - 1;
                const double *gc = p.G + (size_t)(c0 + cf) * ldg;
                const unsigned long long first = __double_as_longlong(__ldg(gc));
                unsigned long long differs = 0ull;
#pragma unroll 4
                for (int r = lane; r < p.n; r += 32) differs |= __double_as_longlong(__ldg(gc + r)) ^ first;
                const bool same = !__any_sync(PG_FULL_MASK, differs != 0ull);
                if (cc == cf && same) constant = true;
            }
            if (constant) flag = false;
        }
        bool small = false;  // a near-perfect fit of some phenotype: the residual sum of squares wants explicit residuals
        for (int j = lane >> 3; j < k; j += 4) {
            if (c >= p.P) break;
            const double gyj = scr[(nq + j) * 8 + cc], yyj = p.yy[p.y0 + j];
            double b = nan(""), vb = nan(""), pv = nan("");
            if (!flag && !constant && ggc > 0.0 && p.dfe > 0.0) {
                b = gyj / ggc;
                double rss = yyj - b * gyj;
                if (!(kCovarRssRedo * ggv * yyj <= rss * ggc)) small = true;
                if (rss < 0.0) rss = 0.0;
                vb = rss / p.dfe / ggc;
                // estimate_significance, src/gwas/ols.rs:139-154
                const double tt = (fabs(b) <= kEps) ? 0.0 : b / sqrt(vb);
                if (fabs(tt) <= kEps || tt != tt)
                    pv = 1.0;
                else
                    pv = p.ptab ? student_two_sided_tab(fabs(tt), p.df, ptab) : student_two_sided(fabs(tt), p.df, p.ln_beta);
            } else if (ggv != ggv) {
                pv = 1.0;  // NaN frequencies: the reference's t is NaN and its p is forced to 1 (ols.rs:150-151)
            }
            p.beta[(size_t)(p.y0 + j) * p.P + c] = b;
            p.var[(size_t)(p.y0 + j) * p.P + c] = vb;
            p.pval[(size_t)(p.y0 + j) * p.P + c] = pv;
        }
        // the four lanes of a column agree; one entry per column and pass (the list kernel redoes every phenotype)
        small |= __shfl_xor_sync(PG_FULL_MASK, (int)small, 8) != 0;
        small |= __shfl_xor_sync(PG_FULL_MASK, (int)small, 16) != 0;
        if (lane < 8 && ((flag && p.y0 == 0) || (!flag && small))) p.defer_list[atomicAdd(p.defer_count, 1u)] = c;
        __syncwarp();
    }
}

// Any number of covariates: the column is staged in shared memory (one slot per warp), the 1 + m + k vectors stream
// from global memory (L2 resident), u = Q'g goes to the warp's shared slot.  O(n (m + k)) per column like the fast
// kernel, without its register / shared-memory limits.
__global__ void __launch_bounds__(256) covar_generic_kernel(const CovarParams p) {
    extern __shared__ __align__(16) double gs[];  // [warps][ldg + nv]
    const int ldg = p.ldg, nq = p.nq, k = p.k, nv = nq + k;
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    double *gcol = gs + (size_t)wib * (ldg + nv);
    double *u = gcol + ldg;
    const int64_t warp = (int64_t)blockIdx.x * (blockDim.x >> 5) + wib;
    const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
    const PTableDev ptab = {reinterpret_cast<const double4 *>(p.ptab), p.ptab_isd, p.ptab_bits, p.ptab_t1, p.ptab_t0, p.ptab_M};
    const int64_t n_items = p.defer_list ? (int64_t)*p.defer_count : p.P;
    for (int64_t item = warp; item < n_items; item += nwarps) {
        const int64_t c = p.defer_list ? p.defer_list[item] : item;
        const double *g = p.G + (size_t)c * ldg;
        double gg = 0.0;
        for (int r = lane; r < ldg; r += 32) {
            const double v = g[r];
            gcol[r] = v;
            gg = fma(v, v, gg);
        }
        gg = warp_sum_fixed(gg);
        __syncwarp();
        double uu = 0.0;
        for (int v = 0; v < nv; v++) {
            const double *q = p.V + (size_t)v * ldg;
            double a = 0.0;
            for (int r = lane; r < ldg; r += 32) a = fma(gcol[r], q[r], a);
            a = warp_sum_fixed(a);
            if (lane == 0) u[v] = a;
            if (v < nq) uu = fma(a, a, uu);
        }
        __syncwarp();
        double ggc = gg - uu;
        const bool redo = !p.minnorm && gg == gg && !(gg <= 1e4 * ggc);
        if (redo) {  // explicit residual e = g - Q u, then e'e and e'y~
            for (int r = lane; r < ldg; r += 32) {
                double e = gcol[r];
                for (int v = 0; v < nq; v++) e = fma(-u[v], p.V[(size_t)v * ldg + r], e);
                gcol[r] = e;
            }
            __syncwarp();
            double s2 = 0.0;
            for (int r = lane; r < p.n; r += 32) s2 = fma(gcol[r], gcol[r], s2);
            ggc = warp_sum_fixed(s2);
            if (ggc <= fmax(64.0, p.nf * p.nf) * kEps * kEps * gg) ggc = 0.0;  // g in span([1 | PCs]): singular X'X, NaN like the reference
            for (int j = 0; j < k; j++) {
                const double *yt = p.V + (size_t)(nq + j) * ldg;
                double a = 0.0;
                for (int r = lane; r < p.n; r += 32) a = fma(gcol[r], yt[r], a);
                a = warp_sum_fixed(a);
                if (lane == 0) u[nq + j] = a;
            }
            __syncwarp();
        }
        const bool solve = lane < k && !p.minnorm && ggc > 0.0 && p.dfe > 0.0;
        double b = nan(""), rss = 0.0;
        const double gyj = lane < k ? u[nq + lane] : 0.0, yyj = lane < k ? p.yy[lane] : 0.0;
        if (solve) {
            b = gyj / ggc;
            rss = yyj - b * gyj;
        }
        unsigned small = __ballot_sync(PG_FULL_MASK, solve && !(kCovarRssRedo * (redo ? ggc : gg) * yyj <= rss * ggc));  // see covar_kernel
        while (small) {
            const int j = __ffs(small) - 1;
            small &= small - 1;
            const double bj = __shfl_sync(PG_FULL_MASK, b, j);
            const double *yt = p.V + (size_t)(nq + j) * ldg;
            double s2 = 0.0;
            for (int r = lane; r < p.n; r += 32) {
                double e = gcol[r];  // already g - Q u after the cancellation branch above
                if (!redo)
                    for (int v = 0; v < nq; v++) e = fma(-u[v], p.V[(size_t)v * ldg + r], e);
                e = fma(-bj, e, yt[r]);
                s2 = fma(e, e, s2);
            }
            s2 = warp_sum_fixed(s2);
            if (lane == j) rss = s2;
        }
        if (lane < k) {
            double vb = nan(""), pv = nan("");
            if (p.minnorm) {
                covar_minnorm(p, gg, u[0], gyj, lane, b, pv);
            } else if (solve) {
                if (rss < 0.0) rss = 0.0;
                vb = rss / p.dfe / ggc;
                const double tt = (fabs(b) <= kEps) ? 0.0 : b / sqrt(vb);
                if (fabs(tt) <= kEps || tt != tt)
                    pv = 1.0;
                else
                    pv = p.ptab ? student_two_sided_tab(fabs(tt), p.df, ptab) : student_two_sided(fabs(tt), p.df, p.ln_beta);
            } else if (gg != gg) {
                pv = 1.0;
            }
            p.beta[(size_t)lane * p.P + c] = b;
            p.var[(size_t)lane * p.P + c] = vb;
            p.pval[(size_t)lane * p.P + c] = pv;
        }
        __syncwarp();
    }
}

}  // namespace pg

// ================================================================================================================
// C ABI
// ================================================================================================================
// cuSOLVER is loaded on first use: linking it would make every process that opens this library map cuSOLVER, cuSPARSE,
// cuBLAS, cuBLASLt and nvJitLink (1.5 GB of shared objects, minutes on a cold file system) although only the eigen
// step of ols_iter_with_kinship calls into it
namespace {
struct CusolverApi {
    cusolverStatus_t (*create)(cusolverDnHandle_t *) = nullptr;
    cusolverStatus_t (*destroy)(cusolverDnHandle_t) = nullptr;
    cusolverStatus_t (*set_stream)(cusolverDnHandle_t, cudaStream_t) = nullptr;
    cusolverStatus_t (*syevd_buffer)(cusolverDnHandle_t, cusolverEigMode_t, cublasFillMode_t, int, const double *, int,
                                     const double *, int *) = nullptr;
    cusolverStatus_t (*syevd)(cusolverDnHandle_t, cusolverEigMode_t, cublasFillMode_t, int, double *, int, double *,
                              double *, int, int *) = nullptr;
    bool ok = false;
};
const CusolverApi &cusolver_api() {
    static const CusolverApi api = [] {
        CusolverApi a;
        void *lib = nullptr;
        for (const char *name : {"libcusolver.so.11", "libcusolver.so.12", "libcusolver.so",
                                 "/usr/local/cuda/lib64/libcusolver.so.11", "/usr/local/cuda/lib64/libcusolver.so"}) {
            lib = dlopen(name, RTLD_NOW | RTLD_LOCAL);
            if (lib) break;
        }
        if (!lib) return a;
        a.create = reinterpret_cast<decltype(a.create)>(dlsym(lib, "cusolverDnCreate"));
        a.destroy = reinterpret_cast<decltype(a.destroy)>(dlsym(lib, "cusolverDnDestroy"));
        a.set_stream = reinterpret_cast<decltype(a.set_stream)>(dlsym(lib, "cusolverDnSetStream"));
        a.syevd_buffer = reinterpret_cast<decltype(a.syevd_buffer)>(dlsym(lib, "cusolverDnDsyevd_bufferSize"));
        a.syevd = reinterpret_cast<decltype(a.syevd)>(dlsym(lib, "cusolverDnDsyevd"));
        a.ok = a.create && a.destroy && a.set_stream && a.syevd_buffer && a.syevd;
        return a;
    }();
    return api;
}
}  // namespace

using pg::fail;

static int64_t round_up(int64_t v, int64_t m) { return (v + m - 1) / m * m; }

extern "C" {

// The eigen step's one-off costs -- mapping cuSOLVER and its dependencies (1.5 GB of shared objects) and creating the
// handle, 0.3-3 s on a cold box, more when eight ranks do it at once -- start in a background thread when the kinship
// handle is opened, so they overlap the column loading, the Gram kernel and the exchange step instead of sitting in
// front of the first pg_kin_eig_select.  The thread is joined by pg_kin_eig_select and by pg_kin_close (a detached
// thread that is still inside dlopen when the process runs its exit handlers corrupts the heap -- measured): a caller
// that only loads columns (sync2csv) waits for the mapping once per process, at its first close.
static void kin_warm_solver(pg_kin *h) {
    const CusolverApi &sol = cusolver_api();
    if (!sol.ok) return;
    if (cudaSetDevice(h->ctx->device) != cudaSuccess) return;
    cusolverDnHandle_t cs = nullptr;
    if (sol.create(&cs) == CUSOLVER_STATUS_SUCCESS) h->solver = cs;
}

// the warm-up thread is joined, and the cuSOLVER handle bound to the stream destroyed, before anything else
pg_kin::~pg_kin() {
    if (warm.joinable()) warm.join();
    if (solver) cusolver_api().destroy(static_cast<cusolverDnHandle_t>(solver));
    if (stream) cudaStreamSynchronize(stream);
    if (ev0) cudaEventDestroy(ev0);
    if (ev1) cudaEventDestroy(ev1);
    if (stream) cudaStreamDestroy(stream);
}

int pg_kin_open(pg_ctx *ctx, int n_pools, int64_t max_columns, pg_kin **out) {
    if (!ctx || !out || n_pools < 2 || max_columns < 1) return fail(ctx, PG_ERR_ARG, "pg_kin_open: bad argument");
    *out = nullptr;
    PG_CUDA(ctx, cudaSetDevice(ctx->device));
    pg_kin *h = new (std::nothrow) pg_kin();
    if (!h) return fail(ctx, PG_ERR_ARG, "out of host memory");
    h->ctx = ctx;
    h->n = n_pools;
    h->ldg = (n_pools + 3) & ~3;
    h->cap = round_up(max_columns, pg::kKC);
    h->nt = (h->ldg + pg::kTile - 1) / pg::kTile;
    cudaError_t e = cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaEventCreate(&h->ev0);
    if (e == cudaSuccess) e = cudaEventCreate(&h->ev1);
    // + one tile of slack: the last tile of a row reads past ldg into the next column
    const size_t g_elems = (size_t)h->cap * h->ldg + pg::kTile;
    if (e == cudaSuccess) e = h->d_G.reserve(g_elems, h->stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(h->d_G.get(), 0, g_elems * 8, h->stream);
    if (e == cudaSuccess) e = h->d_K.reserve((size_t)n_pools * n_pools, h->stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(h->d_K.get(), 0, (size_t)n_pools * n_pools * 8, h->stream);
    if (e != cudaSuccess) {
        delete h;
        return fail(ctx, PG_ERR_CUDA, "pg_kin_open(%d pools, %lld columns): %s", n_pools, (long long)max_columns,
                     cudaGetErrorString(e));
    }
    h->warm = std::thread(kin_warm_solver, h);
    *out = h;
    return PG_OK;
}

int pg_kin_close(pg_kin *h) {
    delete h;
    return PG_OK;
}

int pg_kin_reset(pg_kin *h) {
    if (!h) return PG_ERR_ARG;
    PG_CUDA(h->ctx, cudaSetDevice(h->ctx->device));
    PG_CUDA(h->ctx, cudaMemsetAsync(h->d_G.get(), 0, h->d_G.capacity() * 8, h->stream));
    h->P = 0;
    h->P_total = 0;
    h->text_cols = -1;
    return PG_OK;
}

int64_t pg_kin_columns(pg_kin *h) { return h ? h->P : -1; }

int pg_kin_append_columns(pg_kin *h, const double *cols, int64_t P_add) {
    if (!h || (!cols && P_add > 0) || P_add < 0) return PG_ERR_ARG;
    pg_ctx *ctx = h->ctx;
    if (h->P + P_add > h->cap) return fail(ctx, PG_ERR_ARG, "pg_kin_append_columns: %lld + %lld columns > capacity %lld",
                                            (long long)h->P, (long long)P_add, (long long)h->cap);
    PG_CUDA(ctx, cudaSetDevice(ctx->device));
    h->text_cols = -1;
    if (P_add == 0) return PG_OK;
    PG_CUDA(ctx, cudaMemcpy2DAsync(h->d_G.get() + (size_t)h->P * h->ldg, (size_t)h->ldg * 8, cols, (size_t)h->n * 8,
                                 (size_t)h->n * 8, (size_t)P_add, cudaMemcpyHostToDevice, h->stream));
    h->P += P_add;
    return PG_OK;
}

// loader scratch for n_loci loci of n_alleles stored columns
static int kin_reserve(pg_kin *h, int64_t n_loci, int n_alleles) {
    pg_ctx *ctx = h->ctx;
    PG_CUDA(ctx, h->d_sel.reserve((size_t)n_loci, h->stream));
    PG_CUDA(ctx, h->d_off.reserve((size_t)n_loci + 1, h->stream));
    PG_CUDA(ctx, h->d_col_locus.reserve((size_t)n_loci * PG_MAX_ALLELES, h->stream));
    PG_CUDA(ctx, h->d_col_allele.reserve((size_t)n_loci * PG_MAX_ALLELES, h->stream));
    size_t tmp = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, tmp, h->d_off.get(), h->d_off.get(), (int)(n_loci + 1), h->stream);
    PG_CUDA(ctx, h->d_scan_tmp.reserve(tmp, h->stream));
    PG_CUDA(ctx, h->d_counts.reserve((size_t)n_loci * n_alleles * h->n, h->stream));
    return PG_OK;
}

// LoadAll over the n_loci loci whose counts are in h->d_counts ([locus][allele][pool])
static int kin_load_resident(pg_kin *h, const pg_filter *filter, int n_alleles, const uint8_t *codes, int64_t n_loci,
                             int keep_p_minus_1, int64_t *n_cols_added, const char *who) {
    pg_ctx *ctx = h->ctx;
    PG_CUDA(ctx, h->d_w.reserve((size_t)h->n, h->stream));
    {
        std::vector<double> w(h->n);
        double S = 0.0;
        for (int i = 0; i < h->n; i++) S = S + filter->pool_sizes[i];
        for (int i = 0; i < h->n; i++) w[i] = filter->pool_sizes[i] / S;  // sync.rs:262-270
        PG_CUDA(ctx, cudaMemcpyAsync(h->d_w.get(), w.data(), (size_t)h->n * 8, cudaMemcpyHostToDevice, h->stream));
        PG_CUDA(ctx, cudaStreamSynchronize(h->stream));
    }
    pg::LoadParams lp;
    memset(&lp, 0, sizeof lp);
    lp.counts = h->d_counts.get();
    lp.n_loci = n_loci;
    lp.n = h->n;
    lp.A_in = n_alleles;
    lp.drop_col = -1;
    for (int j = 0; j < n_alleles; j++) {
        lp.codes[j] = codes[j];
        if (filter->remove_ns && codes[j] == 4) lp.drop_col = j;
    }
    lp.ldg = h->ldg;
    lp.keep_p_minus_1 = keep_p_minus_1 != 0;
    lp.maf = filter->min_allele_frequency;
    lp.one_minus_maf = 1.00 - filter->min_allele_frequency;
    lp.max_miss = filter->max_missingness_rate;
    lp.min_depth_f = (double)filter->min_coverage_depth;
    lp.w = h->d_w.get();
    lp.sel = h->d_sel.get();
    lp.offsets = h->d_off.get();
    lp.G = h->d_G.get();
    lp.col_base = h->P;
    lp.col_locus = h->d_col_locus.get();
    lp.col_allele = h->d_col_allele.get();
    const int grid = (int)std::min<int64_t>((n_loci * 32 + 255) / 256, (int64_t)ctx->sm_count * 8);
    pg::load_decide_kernel<<<grid, 256, 0, h->stream>>>(lp);
    PG_CUDA(ctx, cudaGetLastError());
    PG_CUDA(ctx, cudaMemsetAsync(h->d_off.get() + n_loci, 0, 8, h->stream));
    size_t tmp = h->d_scan_tmp.capacity();
    PG_CUDA(ctx, cub::DeviceScan::ExclusiveSum(h->d_scan_tmp.get(), tmp, h->d_off.get(), h->d_off.get(), (int)(n_loci + 1),
                                               h->stream));
    int64_t added = 0;
    PG_CUDA(ctx, cudaMemcpyAsync(&added, h->d_off.get() + n_loci, 8, cudaMemcpyDeviceToHost, h->stream));
    PG_CUDA(ctx, cudaStreamSynchronize(h->stream));
    if (h->P + added > h->cap)
        return fail(ctx, PG_ERR_ARG, "%s: %lld + %lld columns > capacity %lld", who, (long long)h->P,
                     (long long)added, (long long)h->cap);
    pg::load_emit_kernel<<<grid, 256, 0, h->stream>>>(lp);
    PG_CUDA(ctx, cudaGetLastError());
    h->P += added;
    if (n_cols_added) *n_cols_added = added;
    return PG_OK;
}

int pg_kin_append_counts(pg_kin *h, const pg_filter *filter, int n_alleles, const uint8_t *codes,
                         const uint32_t *counts, int64_t n_loci, int keep_p_minus_1, int64_t *n_cols_added) {
    if (!h || !filter || !codes || (!counts && n_loci > 0) || n_loci < 0 || n_alleles < 1 || n_alleles > PG_MAX_ALLELES)
        return PG_ERR_ARG;
    pg_ctx *ctx = h->ctx;
    if (filter->n_pool_sizes != h->n || !filter->pool_sizes)
        return fail(ctx, PG_ERR_ARG, "pg_kin_append_counts: %d pool sizes for %d pools", filter->n_pool_sizes, h->n);
    PG_CUDA(ctx, cudaSetDevice(ctx->device));
    h->text_cols = -1;
    if (n_cols_added) *n_cols_added = 0;
    if (n_loci == 0) return PG_OK;
    int rc = kin_reserve(h, n_loci, n_alleles);
    if (rc) return rc;
    PG_CUDA(ctx, cudaMemcpyAsync(h->d_counts.get(), counts, (size_t)n_loci * n_alleles * h->n * 4, cudaMemcpyHostToDevice,
                               h->stream));
    return kin_load_resident(h, filter, n_alleles, codes, n_loci, keep_p_minus_1, n_cols_added, "pg_kin_append_counts");
}

// the same from a line-aligned chunk of sync TEXT: parsed on the device (pg_text.cu) straight into the loader's count
// slab; pg_kin_text_labels hands out line offsets and positions of the parsed loci for the output rows
int pg_kin_append_sync_text(pg_kin *h, const pg_filter *filter, const char *text, size_t n_bytes, int64_t max_loci,
                            int keep_p_minus_1, int64_t *n_loci_out, int64_t *n_cols_added) {
    if (!h || !filter || (!text && n_bytes > 0) || max_loci < 1) return PG_ERR_ARG;
    pg_ctx *ctx = h->ctx;
    if (filter->n_pool_sizes != h->n || !filter->pool_sizes)
        return fail(ctx, PG_ERR_ARG, "pg_kin_append_sync_text: %d pool sizes for %d pools", filter->n_pool_sizes, h->n);
    PG_CUDA(ctx, cudaSetDevice(ctx->device));
    h->text_cols = -1;
    if (n_cols_added) *n_cols_added = 0;
    if (n_loci_out) *n_loci_out = 0;
    int rc = kin_reserve(h, max_loci, 6);
    if (rc) return rc;
    cudaError_t ce = cudaSuccess;
    uint64_t at = 0;
    int64_t L = 0;
    size_t line_cap = 0;
    for (int attempt = 0; attempt < 2; attempt++) {
        PG_CUDA(ctx, pg::text_parse_async(&h->text, text, n_bytes, h->n, h->d_counts.get(), max_loci, line_cap,
                                          ctx->sm_count, h->stream));
        L = pg::text_parse_finish(&h->text, h->stream, &ce, &at);
        if (L != -5) break;
        line_cap = (size_t)at + 1;  // more comment / blank lines than the default bound: repeat with the exact number
    }
    if (L < 0) return pg::text_parse_fail(ctx, "pg_kin_append_sync_text", L, ce, at, h->n, max_loci);
    if (n_loci_out) *n_loci_out = L;
    int64_t added = 0;
    if (L > 0) {
        static const uint8_t sync_codes[6] = {0, 1, 2, 3, 4, 5};
        rc = kin_load_resident(h, filter, 6, sync_codes, L, keep_p_minus_1, &added, "pg_kin_append_sync_text");
        if (rc) return rc;
    }
    if (n_cols_added) *n_cols_added = added;
    h->text_first = h->P - added;  // pg_kin_format_frequency_rows formats these columns
    h->text_cols = added;
    return PG_OK;
}

int pg_kin_text_labels(pg_kin *h, const uint64_t **line_offsets, const uint64_t **positions) {
    if (!h) return PG_ERR_ARG;
    if (!h->text.parsed) return fail(h->ctx, PG_ERR_STATE, "pg_kin_text_labels before pg_kin_append_sync_text");
    PG_CUDA(h->ctx, cudaStreamSynchronize(h->stream));  // the label copy was enqueued by the parse
    if (line_offsets) *line_offsets = h->text.h_out_offset.get();
    if (positions) *positions = h->text.h_out_pos.get();
    return PG_OK;
}

int pg_kin_last_labels(pg_kin *h, int64_t n_cols, int64_t *col_locus, uint8_t *col_allele) {
    if (!h || n_cols < 0) return PG_ERR_ARG;
    if (n_cols == 0) return PG_OK;
    PG_CUDA(h->ctx, cudaMemcpyAsync(col_locus, h->d_col_locus.get(), (size_t)n_cols * 8, cudaMemcpyDeviceToHost, h->stream));
    PG_CUDA(h->ctx, cudaMemcpyAsync(col_allele, h->d_col_allele.get(), (size_t)n_cols, cudaMemcpyDeviceToHost, h->stream));
    PG_CUDA(h->ctx, cudaStreamSynchronize(h->stream));
    return PG_OK;
}

int pg_kin_synth(pg_kin *h, uint64_t seed, int64_t first_locus, int64_t n_loci) {
    if (!h || n_loci < 0) return PG_ERR_ARG;
    pg_ctx *ctx = h->ctx;
    if (h->P + 2 * n_loci > h->cap) return fail(ctx, PG_ERR_ARG, "pg_kin_synth: capacity");
    PG_CUDA(ctx, cudaSetDevice(ctx->device));
    h->text_cols = -1;
    if (n_loci == 0) return PG_OK;
    const int grid = (int)std::min<int64_t>((n_loci * h->ldg + 255) / 256, (int64_t)ctx->sm_count * 16);
    pg::kin_synth_kernel<<<grid, 256, 0, h->stream>>>(seed, first_locus, n_loci, h->n, h->ldg,
                                                      h->d_G.get() + (size_t)h->P * h->ldg);
    PG_CUDA(ctx, cudaGetLastError());
    h->P += 2 * n_loci;
    return PG_OK;
}

int pg_kin_get_columns(pg_kin *h, int64_t first, int64_t count, double *out) {
    if (!h || first < 0 || count < 0 || first + count > h->P || (!out && count)) return PG_ERR_ARG;
    if (!count) return PG_OK;
    PG_CUDA(h->ctx, cudaMemcpy2DAsync(out, (size_t)h->n * 8, h->d_G.get() + (size_t)first * h->ldg, (size_t)h->ldg * 8,
                                    (size_t)h->n * 8, (size_t)count, cudaMemcpyDeviceToHost, h->stream));
    PG_CUDA(h->ctx, cudaStreamSynchronize(h->stream));
    return PG_OK;
}

static int gram_launch(pg_kin *h, bool accumulate) {
    pg_ctx *ctx = h->ctx;
    const int ntiles = h->nt * (h->nt + 1) / 2;
    const int64_t P_pad = round_up(std::max<int64_t>(h->P, 1), pg::kKC);
    // column slices: enough (slice, tile) items for ~8 waves over the SMs, each slice a multiple of kKC columns
    int n_slices = (int)std::max<int64_t>(1, std::min<int64_t>((8LL * ctx->sm_count + ntiles - 1) / ntiles, P_pad / pg::kKC));
    int64_t slice_cols = round_up((P_pad + n_slices - 1) / n_slices, pg::kKC);
    n_slices = (int)((P_pad + slice_cols - 1) / slice_cols);
    PG_CUDA(ctx, h->d_ws.reserve((size_t)n_slices * ntiles * pg::kTile * pg::kTile, h->stream));
    h->n_slices = n_slices;
    pg::GramParams gp;
    gp.G = h->d_G.get();
    gp.P_pad = P_pad;
    gp.ldg = h->ldg;
    gp.n = h->n;
    gp.nt = h->nt;
    gp.n_slices = n_slices;
    gp.slice_cols = slice_cols;
    gp.ws = h->d_ws.get();
    const size_t smem = 128 + (size_t)pg::kStages * 2 * pg::kKC * pg::kPitch * 8;
    PG_CUDA(ctx, cudaFuncSetAttribute(pg::gram_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int64_t items = (int64_t)ntiles * n_slices;
    const int grid = (int)std::min<int64_t>(items, ctx->sm_count);
    pg::gram_kernel<<<grid, (pg::kGramWarps + 1) * 32, smem, h->stream>>>(gp);
    PG_CUDA(ctx, cudaGetLastError());
    pg::gram_reduce_kernel<<<ctx->sm_count * 4, 256, 0, h->stream>>>(h->d_ws.get(), h->nt, n_slices, h->n,
                                                                     accumulate ? 1 : 0, h->d_K.get());
    PG_CUDA(ctx, cudaGetLastError());
    return PG_OK;
}

int pg_kin_gram(pg_kin *h) {
    if (!h) return PG_ERR_ARG;
    PG_CUDA(h->ctx, cudaSetDevice(h->ctx->device));
    return gram_launch(h, false);
}

// K += G G' of the resident columns: a file larger than the device is taken in blocks (pg_kin_gram on the first,
// pg_kin_gram_accumulate on the others, pg_kin_reset in between), and K ends up the Gram matrix of all of them
int pg_kin_gram_accumulate(pg_kin *h) {
    if (!h) return PG_ERR_ARG;
    PG_CUDA(h->ctx, cudaSetDevice(h->ctx->device));
    return gram_launch(h, true);
}

int pg_kin_gram_time(pg_kin *h, int iters, float *ms_total) {
    if (!h || iters < 1 || !ms_total) return PG_ERR_ARG;
    pg_ctx *ctx = h->ctx;
    PG_CUDA(ctx, cudaSetDevice(ctx->device));
    PG_CUDA(ctx, cudaStreamSynchronize(h->stream));
    PG_CUDA(ctx, cudaEventRecord(h->ev0, h->stream));
    for (int i = 0; i < iters; i++) {
        int rc = gram_launch(h, false);
        if (rc) return rc;
    }
    PG_CUDA(ctx, cudaEventRecord(h->ev1, h->stream));
    PG_CUDA(ctx, cudaEventSynchronize(h->ev1));
    PG_CUDA(ctx, cudaEventElapsedTime(ms_total, h->ev0, h->ev1));
    return PG_OK;
}

int pg_kin_partial(pg_kin *h, double **dev_ptr, size_t *n_elems) {
    if (!h || !dev_ptr) return PG_ERR_ARG;
    PG_CUDA(h->ctx, cudaStreamSynchronize(h->stream));
    *dev_ptr = h->d_K.get();
    if (n_elems) *n_elems = (size_t)h->n * h->n;
    return PG_OK;
}

int pg_kin_partial_get(pg_kin *h, double *out) {
    if (!h || !out) return PG_ERR_ARG;
    PG_CUDA(h->ctx, cudaMemcpyAsync(out, h->d_K.get(), (size_t)h->n * h->n * 8, cudaMemcpyDeviceToHost, h->stream));
    PG_CUDA(h->ctx, cudaStreamSynchronize(h->stream));
    return PG_OK;
}

int pg_kin_partial_set(pg_kin *h, const double *in) {
    if (!h || !in) return PG_ERR_ARG;
    PG_CUDA(h->ctx, cudaMemcpyAsync(h->d_K.get(), in, (size_t)h->n * h->n * 8, cudaMemcpyHostToDevice, h->stream));
    PG_CUDA(h->ctx, cudaStreamSynchronize(h->stream));
    return PG_OK;
}

// h->C = the m covariates, covariate l at pool i being cov[i * pool_stride + l * cov_stride]; h->Q = an orthonormal
// basis of [1 | C] (modified Gram-Schmidt, twice).  Returns the first column of [1 | C] found collinear with the
// columns before it, -1 when there is none.
static int kin_set_basis(pg_kin *h, int m, const double *cov, ptrdiff_t pool_stride, ptrdiff_t cov_stride) {
    const int n = h->n, ldg = h->ldg, nq = 1 + m;
    h->Q.assign((size_t)nq * ldg, 0.0);
    for (int i = 0; i < n; i++) h->Q[i] = 1.0;
    for (int l = 0; l < m; l++)
        for (int i = 0; i < n; i++) h->Q[(size_t)(1 + l) * ldg + i] = cov[i * pool_stride + l * cov_stride];
    h->C.assign(h->Q.begin() + ldg, h->Q.end());
    for (int c = 0; c < nq; c++) {
        double *qc = &h->Q[(size_t)c * ldg];
        for (int pass = 0; pass < 2; pass++)
            for (int b = 0; b < c; b++) {
                const double *qb = &h->Q[(size_t)b * ldg];
                double d = 0.0;
                for (int i = 0; i < n; i++) d += qb[i] * qc[i];
                for (int i = 0; i < n; i++) qc[i] -= d * qb[i];
            }
        double nn = 0.0;
        for (int i = 0; i < n; i++) nn += qc[i] * qc[i];
        nn = sqrt(nn);
        if (!(nn > 1e-12)) return c;
        for (int i = 0; i < n; i++) qc[i] /= nn;
    }
    return -1;
}

// K = (sum of the partial Gram matrices) / P_total; eigen-decomposition; number of PCs by the reference's rule
int pg_kin_eig_select(pg_kin *h, int64_t P_total, double threshold, int *m_out) {
    if (!h || P_total < 0) return PG_ERR_ARG;
    if (P_total == 0) P_total = h->P_total > 0 ? h->P_total : h->P;  // the count pg_kin_allreduce summed, else the resident columns
    if (P_total < 1) return fail(h->ctx, PG_ERR_STATE, "pg_kin_eig_select: no columns");
    pg_ctx *ctx = h->ctx;
    const int n = h->n;
    PG_CUDA(ctx, cudaSetDevice(ctx->device));
    PG_CUDA(ctx, cudaStreamSynchronize(h->stream));
    std::vector<double> A((size_t)n * n), W(n);
    if (h->warm.joinable()) h->warm.join();  // the handle the background thread of pg_kin_open creates
    const CusolverApi &sol = cusolver_api();
    if (!sol.ok) return fail(ctx, PG_ERR_CUDA, "pg_kin_eig_select: libcusolver could not be loaded (%s)", dlerror() ? dlerror() : "missing symbols");
    if (!h->solver) {
        cusolverDnHandle_t made = nullptr;
        if (sol.create(&made) != CUSOLVER_STATUS_SUCCESS) return fail(ctx, PG_ERR_CUDA, "cusolverDnCreate failed");
        h->solver = made;
    }
    cusolverDnHandle_t cs = static_cast<cusolverDnHandle_t>(h->solver);
    sol.set_stream(cs, h->stream);
    pg::DeviceBuffer<double> dA, dW, dwork;
    pg::DeviceBuffer<int> dinfo;
    if (dA.reserve((size_t)n * n, h->stream) != cudaSuccess || dW.reserve((size_t)n, h->stream) != cudaSuccess ||
        dinfo.reserve(1, h->stream) != cudaSuccess)
        return fail(ctx, PG_ERR_CUDA, "pg_kin_eig_select: out of device memory");
    // scale on the host path is avoided: eigenvectors do not depend on the scale, eigenvalue SHARES neither
    cudaMemcpyAsync(dA.get(), h->d_K.get(), (size_t)n * n * 8, cudaMemcpyDeviceToDevice, h->stream);
    int lwork = 0;
    if (sol.syevd_buffer(cs, CUSOLVER_EIG_MODE_VECTOR, CUBLAS_FILL_MODE_LOWER, n, dA.get(), n, dW.get(), &lwork) !=
        CUSOLVER_STATUS_SUCCESS)
        return fail(ctx, PG_ERR_CUDA, "Dsyevd_bufferSize failed");
    if (dwork.reserve((size_t)lwork, h->stream) != cudaSuccess) return fail(ctx, PG_ERR_CUDA, "syevd workspace");
    if (sol.syevd(cs, CUSOLVER_EIG_MODE_VECTOR, CUBLAS_FILL_MODE_LOWER, n, dA.get(), n, dW.get(), dwork.get(), lwork,
                  dinfo.get()) != CUSOLVER_STATUS_SUCCESS)
        return fail(ctx, PG_ERR_CUDA, "Dsyevd failed");
    int info = 0;
    cudaMemcpyAsync(&info, dinfo.get(), 4, cudaMemcpyDeviceToHost, h->stream);
    cudaMemcpyAsync(A.data(), dA.get(), (size_t)n * n * 8, cudaMemcpyDeviceToHost, h->stream);
    cudaMemcpyAsync(W.data(), dW.get(), (size_t)n * 8, cudaMemcpyDeviceToHost, h->stream);
    if (cudaStreamSynchronize(h->stream) != cudaSuccess || info != 0) return fail(ctx, PG_ERR_CUDA, "Dsyevd info %d", info);
    // syevd returns ascending eigenvalues, column j of A (column-major) = eigenvector j; the reference walks them
    // "sorted from high to low" (ols.rs:296)
    h->eigvals.resize(n);
    for (int i = 0; i < n; i++) h->eigvals[i] = W[n - 1 - i] / (double)P_total;
    double sum = 0.0;
    for (int i = 0; i < n; i++) sum = sum + h->eigvals[i];
    std::vector<double> cum(n);
    for (int i = 0; i < n; i++) cum[i] = h->eigvals[i] / sum;
    int m = n;
    for (int i = 1; i < n; i++) {  // ols.rs:303-311
        cum[i] = cum[i - 1] + cum[i];
        if (cum[i - 1] >= threshold && (i - 1) < m) m = i - 1;
    }
    h->m = m;
    h->minnorm = false;
    if (m_out) *m_out = m;
    if (m == n) {
        // the threshold is never reached (ols.rs:300-311 leaves n_eigenvecs = n): all eigenvectors are covariates and
        // X = [1 | V | g] has more columns than rows -- the reference's n < p branch (ols.rs:67-75).  span(V) is the
        // whole space, so only the intercept direction is kept here; covar_kernel forms the minimum-norm coefficient
        h->minnorm = true;
        h->C.clear();
        h->Q.assign((size_t)h->ldg, 0.0);
        for (int i = 0; i < n; i++) h->Q[i] = 1.0 / sqrt((double)n);
        return PG_OK;
    }
    // the covariates are v_1 .. v_m: column n - 1 - l of A (column-major)
    const int c = kin_set_basis(h, m, A.data() + (size_t)(n - 1) * n, 1, -(ptrdiff_t)n);
    if (c >= 0) return fail(ctx, PG_ERR_UNSUPPORTED, "pg_kin_eig_select: covariate %d is collinear with the intercept", c);
    return PG_OK;
}

// one process driving several GPUs: the eigen step runs once (it is replicated work) and the other handles take its
// outcome -- number of PCs, the orthonormal basis of [1 | PCs], the eigenvalues
int pg_kin_copy_covariates(pg_kin *dst, const pg_kin *src) {
    if (!dst || !src) return PG_ERR_ARG;
    if (src->m < 0) return fail(dst->ctx, PG_ERR_STATE, "pg_kin_copy_covariates: the source has no covariates yet");
    if (dst->n != src->n) return fail(dst->ctx, PG_ERR_ARG, "pg_kin_copy_covariates: %d vs %d pools", dst->n, src->n);
    dst->m = src->m;
    dst->minnorm = src->minnorm;
    dst->Q = src->Q;
    dst->C = src->C;
    dst->eigvals = src->eigvals;
    dst->P_total = src->P_total;
    return PG_OK;
}

int pg_kin_eigvals(pg_kin *h, double *out, int count) {
    if (!h || !out || count < 0 || (size_t)count > h->eigvals.size()) return PG_ERR_ARG;
    for (int i = 0; i < count; i++) out[i] = h->eigvals[i];
    return PG_OK;
}

// explicit covariates instead of the eigen step (tests; a caller that already holds the PCs): cov is n x m row-major
int pg_kin_set_covariates(pg_kin *h, const double *cov, int m) {
    if (!h || m < 0 || (m > 0 && !cov)) return PG_ERR_ARG;
    pg_ctx *ctx = h->ctx;
    const int n = h->n;
    if (m + 2 > n) return fail(ctx, PG_ERR_UNSUPPORTED, "pg_kin_set_covariates: %d covariates for %d pools", m, n);
    h->m = m;
    h->minnorm = false;
    const int c = kin_set_basis(h, m, cov, m, 1);
    if (c >= 0) return fail(ctx, PG_ERR_UNSUPPORTED, "pg_kin_set_covariates: covariate %d is collinear", c);
    return PG_OK;
}

}  // extern "C"

// covar_kernel<NV, 1, true> over a column list (cp.defer_list / cp.defer_count)
template <int NV>
static cudaError_t covar_launch_list(const pg::CovarParams &cp, int sm_count, cudaStream_t s) {
    const size_t smem = (size_t)NV * cp.ldg * 8;
    auto kern = pg::covar_kernel<NV, 1, true>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    kern<<<sm_count, 512, smem, s>>>(cp);
    return cudaGetLastError();
}

template <int NV>
static cudaError_t covar_launch_nv(const pg::CovarParams &cp, int sm_count, cudaStream_t s) {
    const size_t smem = (size_t)NV * cp.ldg * 8;
    auto kern = pg::covar_kernel<NV, (NV >= 9 ? 3 : (NV >= 5 ? 4 : (NV >= 3 ? 2 : 1))), false>;  // C * NV accumulators fit the registers
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    int ctas_per_sm = (int)std::min<size_t>(4, (227 * 1024) / std::max<size_t>(smem, 1));
    if (ctas_per_sm < 1) ctas_per_sm = 1;
    kern<<<sm_count * ctas_per_sm, 512, smem, s>>>(cp);
    return cudaGetLastError();
}

// the DMMA form: nv <= 16 vectors whose shared-memory copy leaves room for the warps' scratch
static bool covar_mma_fits(const pg::CovarParams &cp, int nv, int *ldq_out, int *warps_out, size_t *smem_out,
                           int pools = 0) {
    if (cp.minnorm || nv > 16) return false;
    if (pools <= 0) pools = cp.n;
    int ldq = (pools + 15) & ~15;  // whole 16-pool blocks, zero padded
    ldq += 8;                     // pitch = 8 (mod 16) doubles: conflict-free 128-bit fragment loads
    const int mt = nv <= 8 ? 1 : 2;
    const size_t vbytes = (size_t)nv * ldq * 8, per_warp = (size_t)(8 * mt + 1) * 8 * 8;
    const size_t budget = 227 * 1024;
    if (vbytes + 8 * per_warp > budget) return false;  // V and the warps' partial tiles
    int warps = (int)std::min<size_t>(pg::kCmMaxWarps, (budget - vbytes) / per_warp);
    static const int warps_env = getenv("PG_CM_WARPS") ? atoi(getenv("PG_CM_WARPS")) : 0;
    if (warps_env >= 4 && warps_env < warps) warps = warps_env;
    *ldq_out = ldq;
    *warps_out = warps;
    *smem_out = vbytes + (size_t)warps * per_warp;
    return true;
}

// covar_generic_kernel over all columns (list = false) or over the deferred list
static int covar_launch_generic(pg_kin *h, const pg::CovarParams &cp) {
    pg_ctx *ctx = h->ctx;
    const int nv = cp.nq + cp.k;
    const size_t per_warp = (size_t)(cp.ldg + nv) * 8;
    const int warps = (int)std::min<size_t>(8, (200 * 1024) / per_warp);
    if (warps < 1) return fail(ctx, PG_ERR_UNSUPPORTED, "covariate scan: %d pools x %d vectors exceed shared memory", cp.n, nv);
    const size_t smem = per_warp * warps;
    cudaError_t e = cudaFuncSetAttribute(pg::covar_generic_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e == cudaSuccess) {
        pg::covar_generic_kernel<<<ctx->sm_count, warps * 32, smem, h->stream>>>(cp);
        e = cudaGetLastError();
    }
    if (e != cudaSuccess) return fail(ctx, PG_ERR_CUDA, "covar_generic_kernel: %s", cudaGetErrorString(e));
    return PG_OK;
}

static int covar_launch(pg_kin *h, const pg::CovarParams &cp_in) {
    pg_ctx *ctx = h->ctx;
    const int nv = cp_in.nq + cp_in.k;
    cudaError_t e = cudaSuccess;
    int ldq = 0, warps = 0;
    size_t smem_mma = 0;
    static const bool no_mma = getenv("PG_COVAR_NO_MMA") != nullptr;  // tests: the per-warp dot-product kernels
    // with covariates (nv >= 5): as many phenotypes per pass as fit beside the Q columns in shared memory, G is
    // streamed once per pass
    // pool passes of the DMMA form: shared memory beyond the 196 KB carve-out leaves 28 KB of L1 for the loads in flight
    // (n = 2,000 with 12 vectors: V = 193 KB, 0.58 of the roofline; the same kernel runs each half of the pools at 0.90)
    // -- then the pools are taken in the fewest passes that stay within that carve-out, the partial sums parked in
    // global memory in between (1.7 % of the column traffic per extra pass)
    static const int passes_env = getenv("PG_CM_POOL_PASSES") ? atoi(getenv("PG_CM_POOL_PASSES")) : 0;
    auto pool_plan = [&](int nvp, int *per_out) {
        const size_t scratch = (size_t)pg::kCmMaxWarps * (size_t)(8 * (nvp <= 8 ? 1 : 2) + 1) * 8 * 8;
        int np = 1, per = cp_in.n;
        for (; np <= 16; np++) {
            per = (((cp_in.n + np - 1) / np) + 15) & ~15;  // pools per pass, whole 16-pool blocks
            if ((size_t)nvp * (per + 8) * 8 + scratch <= 196 * 1024) break;
        }
        if (passes_env >= 1) {
            np = passes_env;
            per = (((cp_in.n + np - 1) / np) + 15) & ~15;
        }
        *per_out = per;
        return (cp_in.n + per - 1) / per;
    };
    auto fits_nv = [&](int nvp) {
        int per = 0;
        pool_plan(nvp, &per);
        return covar_mma_fits(cp_in, nvp, &ldq, &warps, &smem_mma, per);
    };
    int kk = cp_in.k;
    while (kk > 1 && !fits_nv(cp_in.nq + kk)) kk--;
    const bool mma = !no_mma && nv >= 5 && fits_nv(cp_in.nq + kk);
    // the list of columns the streaming kernels leave to the explicit-residual forms: [count | columns], at most one
    // entry per column and pass
    PG_CUDA(ctx, h->d_defer.reserve((size_t)cp_in.P * (size_t)(mma ? (cp_in.k + kk - 1) / kk : 1) + 2, h->stream));
    PG_CUDA(ctx, cudaMemsetAsync(h->d_defer.get(), 0, 8, h->stream));
    pg::CovarParams cp = cp_in;
    cp.defer_count = reinterpret_cast<unsigned *>(h->d_defer.get());
    cp.defer_list = h->d_defer.get() + 1;
    const bool fits = (size_t)nv * cp.ldg * 8 <= 227 * 1024;  // the vectors in shared memory (covar_kernel)
    if (mma) {
        for (int y0 = 0; y0 < cp.k; y0 += kk) {
            pg::CovarParams pp = cp;
            pp.y0 = y0;
            pp.k = std::min(kk, cp.k - y0);
            const int nvp = pp.nq + pp.k, mt = nvp <= 8 ? 1 : 2;
            int per = 0;
            const int np = pool_plan(nvp, &per);
            if (np > 1) PG_CUDA(ctx, h->d_part.reserve((size_t)((cp.P + 7) / 8) * (size_t)(8 * mt + 1) * 8, h->stream));
            auto kern = mt == 1 ? pg::covar_mma_kernel<1> : pg::covar_mma_kernel<2>;
            for (int ip = 0; ip < np; ip++) {
                pp.pr0 = ip * per;
                pp.pn = std::min(per, cp.n - pp.pr0);
                pp.part_mode = (ip + 1 < np ? 1 : 0) | (ip > 0 ? 2 : 0);
                pp.part = h->d_part.get();
                if (!covar_mma_fits(pp, nvp, &ldq, &warps, &smem_mma, pp.pn))
                    return fail(ctx, PG_ERR_UNSUPPORTED, "covariate scan: %d vectors x %d pools do not fit a pool pass", nvp, pp.pn);
                e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_mma);
                if (e == cudaSuccess) {
                    kern<<<ctx->sm_count, warps * 32, smem_mma, h->stream>>>(pp, ldq, warps);
                    e = cudaGetLastError();
                }
                if (e != cudaSuccess) return fail(ctx, PG_ERR_CUDA, "covar_mma_kernel: %s", cudaGetErrorString(e));
            }
        }
    } else {
        switch (fits ? nv : 0) {
            case 2: e = covar_launch_nv<2>(cp, ctx->sm_count, h->stream); break;
            case 3: e = covar_launch_nv<3>(cp, ctx->sm_count, h->stream); break;
            case 4: e = covar_launch_nv<4>(cp, ctx->sm_count, h->stream); break;
            case 5: e = covar_launch_nv<5>(cp, ctx->sm_count, h->stream); break;
            case 6: e = covar_launch_nv<6>(cp, ctx->sm_count, h->stream); break;
            case 7: e = covar_launch_nv<7>(cp, ctx->sm_count, h->stream); break;
            case 8: e = covar_launch_nv<8>(cp, ctx->sm_count, h->stream); break;
            case 9: e = covar_launch_nv<9>(cp, ctx->sm_count, h->stream); break;
            case 10: e = covar_launch_nv<10>(cp, ctx->sm_count, h->stream); break;
            case 11: e = covar_launch_nv<11>(cp, ctx->sm_count, h->stream); break;
            case 12: e = covar_launch_nv<12>(cp, ctx->sm_count, h->stream); break;
            case 13: e = covar_launch_nv<13>(cp, ctx->sm_count, h->stream); break;
            case 14: e = covar_launch_nv<14>(cp, ctx->sm_count, h->stream); break;
            case 15: e = covar_launch_nv<15>(cp, ctx->sm_count, h->stream); break;
            case 16: e = covar_launch_nv<16>(cp, ctx->sm_count, h->stream); break;
            default: {
                // every column through the generic kernel, which carries the explicit-residual forms itself
                pg::CovarParams pp = cp;
                pp.defer_list = nullptr;
                pp.defer_count = nullptr;
                return covar_launch_generic(h, pp);
            }
        }
        if (e != cudaSuccess) return fail(ctx, PG_ERR_CUDA, "covar_kernel: %s", cudaGetErrorString(e));
    }
    // the deferred columns (a centred g'g or a residual sum of squares lost to cancellation): explicit residuals, every
    // phenotype; an empty list costs one tiny launch
    switch (fits ? nv : 0) {
        case 2: e = covar_launch_list<2>(cp, ctx->sm_count, h->stream); break;
        case 3: e = covar_launch_list<3>(cp, ctx->sm_count, h->stream); break;
        case 4: e = covar_launch_list<4>(cp, ctx->sm_count, h->stream); break;
        case 5: e = covar_launch_list<5>(cp, ctx->sm_count, h->stream); break;
        case 6: e = covar_launch_list<6>(cp, ctx->sm_count, h->stream); break;
        case 7: e = covar_launch_list<7>(cp, ctx->sm_count, h->stream); break;
        case 8: e = covar_launch_list<8>(cp, ctx->sm_count, h->stream); break;
        case 9: e = covar_launch_list<9>(cp, ctx->sm_count, h->stream); break;
        case 10: e = covar_launch_list<10>(cp, ctx->sm_count, h->stream); break;
        case 11: e = covar_launch_list<11>(cp, ctx->sm_count, h->stream); break;
        case 12: e = covar_launch_list<12>(cp, ctx->sm_count, h->stream); break;
        case 13: e = covar_launch_list<13>(cp, ctx->sm_count, h->stream); break;
        case 14: e = covar_launch_list<14>(cp, ctx->sm_count, h->stream); break;
        case 15: e = covar_launch_list<15>(cp, ctx->sm_count, h->stream); break;
        case 16: e = covar_launch_list<16>(cp, ctx->sm_count, h->stream); break;
        default: return covar_launch_generic(h, cp);
    }
    if (e != cudaSuccess) return fail(ctx, PG_ERR_CUDA, "covariate scan (deferred columns): %s", cudaGetErrorString(e));
    return PG_OK;
}

// the Student-t(n - 1) table and the [3][k][P] record buffers shared by pg_kin_covar_scan and pg_kin_mle_scan
static int kin_prepare_records(pg_kin *h, int k) {
    pg_ctx *ctx = h->ctx;
    const double df = (double)h->n - 1.0;
    if (!h->d_ptab.get()) {
        pg::PTable tab = pg::build_ptable(df);
        if (tab.max_err < 2e-9) {
            PG_CUDA(ctx, h->d_ptab.reserve(tab.coef.size(), h->stream));
            PG_CUDA(ctx, cudaMemcpyAsync(h->d_ptab.get(), tab.coef.data(), tab.coef.size() * 8, cudaMemcpyHostToDevice, h->stream));
            PG_CUDA(ctx, cudaStreamSynchronize(h->stream));
            h->ptab_M = tab.M;
            h->ptab_isd = tab.inv_sqrt_df;
            h->ptab_bits = tab.bits;
            h->ptab_t1 = tab.t_one;
            h->ptab_t0 = tab.t_zero;
        }
    }
    const size_t elems = (size_t)3 * k * std::max<int64_t>(h->P, 1);
    PG_CUDA(ctx, h->d_res.reserve(elems, h->stream));
    PG_CUDA(ctx, h->h_res.reserve(elems, h->stream));
    h->k = k;
    return PG_OK;
}

extern "C" {

// per-column regression; phen n x k row-major.  Results (host, pinned, valid until the next call / close):
// beta, var, pval each [k][P].  iters > 0: time `iters` launches (ms_total), results from the last one.
int pg_kin_covar_scan(pg_kin *h, const double *phen, int k, int iters, float *ms_total, const double **beta,
                      const double **var, const double **pval) {
    if (!h || !phen || k < 1) return PG_ERR_ARG;
    pg_ctx *ctx = h->ctx;
    if (h->m < 0) return fail(ctx, PG_ERR_STATE, "pg_kin_covar_scan before pg_kin_eig_select / pg_kin_set_covariates");
    const int n = h->n, ldg = h->ldg, nq = h->minnorm ? 1 : 1 + h->m;
    if (k > pg::kMaxPhenPerPass * 4)
        return fail(ctx, PG_ERR_UNSUPPORTED, "pg_kin_covar_scan: %d phenotypes > %d per call", k, pg::kMaxPhenPerPass * 4);
    PG_CUDA(ctx, cudaSetDevice(ctx->device));
    // y~ = y - Q Q'y on the host (n x k, tiny)
    std::vector<double> V((size_t)(nq + k) * ldg, 0.0);
    std::copy(h->Q.begin(), h->Q.end(), V.begin());
    pg::CovarParams cp;
    memset(&cp, 0, sizeof cp);
    for (int j = 0; j < k; j++) {
        double *yt = &V[(size_t)(nq + j) * ldg];
        for (int i = 0; i < n; i++) yt[i] = phen[(size_t)i * k + j];
        if (h->minnorm) {  // the n < p branch works on the raw phenotype
            double sy = 0.0;
            for (int i = 0; i < n; i++) sy += yt[i];
            cp.sy[j] = sy;
            continue;
        }
        for (int pass = 0; pass < 2; pass++)
            for (int b = 0; b < nq; b++) {
                const double *qb = &h->Q[(size_t)b * ldg];
                double d = 0.0;
                for (int i = 0; i < n; i++) d += qb[i] * yt[i];
                for (int i = 0; i < n; i++) yt[i] -= d * qb[i];
            }
        double yy = 0.0;
        for (int i = 0; i < n; i++) yy += yt[i] * yt[i];
        cp.yy[j] = yy;
    }
    PG_CUDA(ctx, h->d_V.reserve(V.size(), h->stream));
    PG_CUDA(ctx, cudaMemcpyAsync(h->d_V.get(), V.data(), V.size() * 8, cudaMemcpyHostToDevice, h->stream));
    PG_CUDA(ctx, cudaStreamSynchronize(h->stream));
    const double df = (double)n - 1.0;
    if (int rc = kin_prepare_records(h, k)) return rc;
    cp.G = h->d_G.get();
    cp.P = h->P;
    cp.ldg = ldg;
    cp.n = n;
    cp.nq = nq;
    cp.k = k;
    cp.V = h->d_V.get();
    cp.dfe = (double)n - (double)(2 + h->m);
    cp.minnorm = h->minnorm ? 1 : 0;
    cp.nf = (double)n;
    cp.sqrt_n = sqrt((double)n);
    cp.df = df;
    cp.ptab = h->d_ptab.get();
    cp.ptab_isd = h->ptab_isd;
    cp.ptab_bits = h->ptab_bits;
    cp.ptab_t1 = h->ptab_t1;
    cp.ptab_t0 = h->ptab_t0;
    cp.ptab_M = h->ptab_M;
    cp.ln_beta = pg::statrs::ln_gamma(df / 2.0 + 0.5) - pg::statrs::ln_gamma(df / 2.0) - pg::statrs::ln_gamma(0.5);
    cp.beta = h->d_res.get();
    cp.var = h->d_res.get() + (size_t)k * h->P;
    cp.pval = h->d_res.get() + (size_t)2 * k * h->P;
    const int reps = iters > 0 ? iters : 1;
    if (iters > 0) PG_CUDA(ctx, cudaEventRecord(h->ev0, h->stream));
    for (int i = 0; i < reps; i++) {
        int rc = covar_launch(h, cp);
        if (rc) return rc;
    }
    if (iters > 0) PG_CUDA(ctx, cudaEventRecord(h->ev1, h->stream));
    PG_CUDA(ctx, cudaMemcpyAsync(h->h_res.get(), h->d_res.get(), (size_t)3 * k * h->P * 8, cudaMemcpyDeviceToHost, h->stream));
    PG_CUDA(ctx, cudaStreamSynchronize(h->stream));
    if (iters > 0 && ms_total) PG_CUDA(ctx, cudaEventElapsedTime(ms_total, h->ev0, h->ev1));
    static const bool debug = getenv("PG_COVAR_DEBUG") != nullptr;  // how many columns took the explicit-residual forms
    if (debug && h->d_defer.get()) {
        unsigned cnt = 0;
        cudaMemcpy(&cnt, h->d_defer.get(), 4, cudaMemcpyDeviceToHost);
        fprintf(stderr, "pg_kin_covar_scan: %u of %lld columns deferred to the explicit-residual kernel\n", cnt, (long long)h->P);
    }
    if (beta) *beta = h->h_res.get();
    if (var) *var = h->h_res.get() + (size_t)k * h->P;
    if (pval) *pval = h->h_res.get() + (size_t)2 * k * h->P;
    return PG_OK;
}

// mle_iter_with_kinship: mle_with_covariate (src/gwas/mle.rs:307-463) over the resident columns, with the covariates
// pg_kin_eig_select / pg_kin_set_covariates left.  Everything that does not involve the allele column -- the centred
// covariates and phenotypes and their moments, Szz^-1 -- is formed here on the host (n x (m + k), tiny)
int pg_kin_mle_scan(pg_kin *h, const double *phen, int k, float *ms, const double **beta, const double **var,
                    const double **pval) {
    if (!h || !phen || k < 1) return PG_ERR_ARG;
    pg_ctx *ctx = h->ctx;
    if (h->m < 0) return fail(ctx, PG_ERR_STATE, "pg_kin_mle_scan before pg_kin_eig_select / pg_kin_set_covariates");
    const int n = h->n, ldg = h->ldg, m = h->m;
    if (h->minnorm || m + 2 > n)
        return fail(ctx, PG_ERR_UNSUPPORTED, "pg_kin_mle_scan: %d covariates for %d pools (the n < p form of mle.rs:130-140)", m, n);
    if (m > pg::kKinMleMaxM)
        return fail(ctx, PG_ERR_UNSUPPORTED, "pg_kin_mle_scan: %d covariates > %d (simplex of at most 16 parameters)", m, pg::kKinMleMaxM);
    if (k > 16) return fail(ctx, PG_ERR_UNSUPPORTED, "pg_kin_mle_scan: %d phenotypes > 16 per call", k);
    if ((int)h->C.size() != m * ldg) return fail(ctx, PG_ERR_STATE, "pg_kin_mle_scan: covariates missing");
    PG_CUDA(ctx, cudaSetDevice(ctx->device));
    const int nfix = m + 2 * m * m + k * (2 + m);
    std::vector<double> Z((size_t)(m + k) * ldg + nfix, 0.0);
    double *fix = Z.data() + (size_t)(m + k) * ldg;
    double *zbar = fix, *Szz = fix + m, *Wzz = Szz + m * m, *phf = Wzz + m * m;
    for (int l = 0; l < m; l++) {
        const double *c = &h->C[(size_t)l * ldg];
        double s = 0.0;
        for (int i = 0; i < n; i++) s += c[i];
        zbar[l] = s / (double)n;
        for (int i = 0; i < n; i++) Z[(size_t)l * ldg + i] = c[i] - zbar[l];
    }
    for (int a = 0; a < m; a++)
        for (int b = 0; b <= a; b++) {
            double s = 0.0;
            for (int i = 0; i < n; i++) s += Z[(size_t)a * ldg + i] * Z[(size_t)b * ldg + i];
            Szz[a * m + b] = Szz[b * m + a] = s;
        }
    if (m > 0) {  // Szz^-1 by Gauss-Jordan with partial pivoting
        std::vector<double> M((size_t)m * 2 * m, 0.0);
        for (int a = 0; a < m; a++) {
            for (int b = 0; b < m; b++) M[(size_t)a * 2 * m + b] = Szz[a * m + b];
            M[(size_t)a * 2 * m + m + a] = 1.0;
        }
        for (int c = 0; c < m; c++) {
            int pr = c;
            for (int r = c + 1; r < m; r++)
                if (fabs(M[(size_t)r * 2 * m + c]) > fabs(M[(size_t)pr * 2 * m + c])) pr = r;
            if (!(fabs(M[(size_t)pr * 2 * m + c]) > 1e-12 * fabs(Szz[c * m + c])))
                return fail(ctx, PG_ERR_UNSUPPORTED, "pg_kin_mle_scan: covariate %d is collinear with the others", c);
            for (int e = 0; e < 2 * m; e++) std::swap(M[(size_t)c * 2 * m + e], M[(size_t)pr * 2 * m + e]);
            const double piv = 1.0 / M[(size_t)c * 2 * m + c];
            for (int e = 0; e < 2 * m; e++) M[(size_t)c * 2 * m + e] *= piv;
            for (int r = 0; r < m; r++) {
                if (r == c) continue;
                const double f = M[(size_t)r * 2 * m + c];
                for (int e = 0; e < 2 * m; e++) M[(size_t)r * 2 * m + e] -= f * M[(size_t)c * 2 * m + e];
            }
        }
        for (int a = 0; a < m; a++)
            for (int b = 0; b < m; b++) Wzz[a * m + b] = M[(size_t)a * 2 * m + m + b];
    }
    for (int j = 0; j < k; j++) {
        double *yt = &Z[(size_t)(m + j) * ldg], *pf = phf + (size_t)j * (2 + m);
        double s = 0.0;
        for (int i = 0; i < n; i++) s += phen[(size_t)i * k + j];
        const double ybar = s / (double)n;
        double syy = 0.0;
        for (int i = 0; i < n; i++) {
            yt[i] = phen[(size_t)i * k + j] - ybar;
            syy += yt[i] * yt[i];
        }
        pf[0] = ybar;
        pf[1] = syy;
        for (int l = 0; l < m; l++) {
            double c = 0.0;
            for (int i = 0; i < n; i++) c += Z[(size_t)l * ldg + i] * yt[i];
            pf[2 + l] = c;
        }
    }
    PG_CUDA(ctx, h->d_mle.reserve(Z.size(), h->stream));
    PG_CUDA(ctx, cudaMemcpyAsync(h->d_mle.get(), Z.data(), Z.size() * 8, cudaMemcpyHostToDevice, h->stream));
    PG_CUDA(ctx, cudaStreamSynchronize(h->stream));
    if (int rc = kin_prepare_records(h, k)) return rc;
    const double df = (double)n - 1.0;
    pg::KinMleParams mp;
    memset(&mp, 0, sizeof mp);
    mp.G = h->d_G.get();
    mp.P = h->P;
    mp.n = n;
    mp.ldg = ldg;
    mp.m = m;
    mp.k = k;
    mp.Z = h->d_mle.get();
    mp.fix = h->d_mle.get() + (size_t)(m + k) * ldg;
    mp.df = df;
    mp.ln_beta = pg::statrs::ln_gamma(df / 2.0 + 0.5) - pg::statrs::ln_gamma(df / 2.0) - pg::statrs::ln_gamma(0.5);
    mp.ptab = h->d_ptab.get();
    mp.ptab_isd = h->ptab_isd;
    mp.ptab_bits = h->ptab_bits;
    mp.ptab_t1 = h->ptab_t1;
    mp.ptab_t0 = h->ptab_t0;
    mp.ptab_M = h->ptab_M;
    mp.beta = h->d_res.get();
    mp.var = h->d_res.get() + (size_t)k * h->P;
    mp.pval = h->d_res.get() + (size_t)2 * k * h->P;
    PG_CUDA(ctx, cudaEventRecord(h->ev0, h->stream));
    PG_CUDA(ctx, pg::launch_kin_mle(mp, ctx->sm_count, h->stream));
    PG_CUDA(ctx, cudaEventRecord(h->ev1, h->stream));
    PG_CUDA(ctx, cudaMemcpyAsync(h->h_res.get(), h->d_res.get(), (size_t)3 * k * h->P * 8, cudaMemcpyDeviceToHost, h->stream));
    PG_CUDA(ctx, cudaStreamSynchronize(h->stream));
    if (ms) PG_CUDA(ctx, cudaEventElapsedTime(ms, h->ev0, h->ev1));
    if (beta) *beta = h->h_res.get();
    if (var) *var = h->h_res.get() + (size_t)k * h->P;
    if (pval) *pval = h->h_res.get() + (size_t)2 * k * h->P;
    return PG_OK;
}

}  // extern "C"
