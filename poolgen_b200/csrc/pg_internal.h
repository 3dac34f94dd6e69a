// pg_internal.h -- shared declarations of libpoolgen_cuda (not part of the ABI).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>
#include <string>
#include <utility>
#include <vector>

#include "poolgen_cuda.h"
#include "pg_synth.h"

namespace pg {

// ---- device data layout of one batch --------------------------------------------------------
// Per locus the first-stage frequency matrix (n_pools x A, reference LocusFrequencies.matrix of
// src/base/sync.rs:166-192 before the MAF filter) is stored allele-major ("column-major n x A"),
// split into row chunks of RC pools so that a chunk [A][rc] is one contiguous block a single
// cp.async.bulk can fetch:
//   freq  : [locus][chunk][A][rc_chunk] f64     locus stride = A * n_pad doubles
//   depth : [locus][chunk][rc_chunk]    u32     locus stride = n_pad
//   dmin  : [locus]                    u32     min over the pools of depth (the min-depth filter and the
//                                               "a pool has no coverage" test need nothing else on the fast path;
//                                               the per-pool depths are only read by the rare renormalisation paths)
// n_pad = n rounded up to a multiple of 4 (16-byte granules for bulk copies); padding rows hold
// freq = 0, depth = 0xFFFFFFFF.  When n_pad <= chunk_rows(A) there is one chunk and consecutive loci
// are contiguous, so several loci travel in one bulk copy.  A full chunk is 4..6 KB for every A.
__host__ __device__ constexpr int chunk_rows(int A) { return A <= 2 ? 256 : (A == 3 ? 192 : 128); }

struct Layout {
    int n;         // pools
    int n_pad;     // rounded up to 4
    int A;         // allele columns on the device (N already dropped when remove_ns)
    int rc;        // rows of a full chunk
    int n_chunks;  // chunks per locus
    int rc_last;   // rows of the last chunk (multiple of 4)
    __host__ __device__ size_t freq_stride() const { return (size_t)A * n_pad; }
    __host__ __device__ size_t depth_stride() const { return (size_t)n_pad; }
    // element offset of (row i, allele j) inside one locus
    __host__ __device__ size_t freq_off(int i, int j) const {
        int c = i / rc, r = i - c * rc;
        int rcc = (c == n_chunks - 1) ? rc_last : rc;
        return (size_t)c * A * rc + (size_t)j * rcc + r;
    }
};

inline Layout make_layout(int n, int A) {
    Layout l;
    l.n = n;
    l.n_pad = (n + 3) & ~3;
    l.A = A;
    const int cr = chunk_rows(A);
    if (l.n_pad <= cr) {
        l.rc = l.n_pad;
        l.n_chunks = 1;
        l.rc_last = l.n_pad;
    } else {
        l.rc = cr;
        l.n_chunks = (l.n_pad + cr - 1) / cr;
        l.rc_last = l.n_pad - (l.n_chunks - 1) * cr;
    }
    return l;
}

constexpr int kMaxPhenPerPass = 4;
// phenotypes per kernel pass: bounded by the accumulator registers (A + A(A+1)/2 + A*K doubles per lane)
inline int max_phen_per_pass(int A) { return A <= 4 ? 4 : (A == 5 ? 3 : 2); }

// The OLS / Pearson scan keeps a pass's phenotype vectors and the pool weights resident in shared memory, in at most
// 96 KB: one phenotype and the weights fit up to 6,144 pools.  Above that scan_kernel_wide (pg_scan.cuh) reads them
// from L2 and takes as many phenotypes per pass as the registers allow.  PG_SCAN_WIDE (tests, read once per process)
// takes the wide kernel wherever the scan runs 32 lanes per locus (more than one row chunk).
constexpr int kResidentPhenPools = 6144;
inline bool scan_wide(const Layout &lay) {
    static const bool force = getenv("PG_SCAN_WIDE") != nullptr;
    return lay.n_chunks > 1 && (lay.n_pad > kResidentPhenPools || force);
}

// parameters of one ols/corr scan launch (passed by value)
struct ScanParams {
    Layout lay;
    const double *freq;
    const uint32_t *depth;
    const uint32_t *dmin;
    const uint8_t *hint;
    int64_t n_loci;
    int kind;
    int weighted;         // pool weights differ
    double maf, one_minus_maf, max_miss;
    double min_depth_f;   // (min_coverage_depth as f64)
    double w_uniform;     // s_0 / sum(s) when all weights are equal
    double df;            // Student-t degrees of freedom (n-1 ols, n-2 corr)
    double inv_df;        // 1 / df
    double inv_n, inv_nm2; // 1 / n, 1 / (n - 2)
    double ln_beta;       // lnG(df/2 + 1/2) - lnG(df/2) - lnG(1/2)
    const void *ptab;     // per-scan table of ln p(v) (double4 per interval), NULL = continued fraction on the device
    double ptab_isd, ptab_bits, ptab_t1, ptab_t0;  // t1 / t0: PTable::t_one / t_zero
    int ptab_M;
    const double *yc;     // [K][n_pad] centred phenotypes of this pass (device)
    const double *w;      // [n_pad] s_i / sum(s) (device)
    double ysum[kMaxPhenPerPass];  // sum of the centred phenotype (rounding residue)
    double syy[kMaxPhenPerPass];   // centred sum of squares
    double ymean[kMaxPhenPerPass]; // mean of the phenotype (the n < p branch needs the uncentred values)
    int y_has_nan;
    int filter_only;      // mle_iter / gwalpha: phase 2 stops after the keep-mask, the allele order and the means
    uint8_t codes[8];     // allele code of device column j
    uint64_t *meta;
    double *freq_mean;
    double *stats;
    uint64_t *defer_list;   // [n_loci] loci left to the fix-up kernel: locus | kept set << 40 (0 = undecided)
    uint32_t *defer_count;  // [1]
    int k_total, phen_base, K;  // output indexing when k > kMaxPhenPerPass
    int write_meta;             // only the first phenotype pass writes meta / freq_mean
    // launch geometry, filled in by the launcher
    uint32_t common_bytes, warp_bytes, stage_bytes;
    int nbuf, block_loci;
    int nbuf_override, warps_override, g_override, p_override;  // tuning knobs (PG_NBUF / PG_WARPS / PG_G), 0 = automatic
};

struct TableParams {
    const uint32_t *counts;  // [locus][A_in][n]
    int64_t n_loci;
    int n, A_in;
    int kind;
    int drop_col;  // column index coded N to drop (-1 none)
    double maf, one_minus_maf, max_miss, min_depth_f;
    const double *w;
    uint8_t codes[8];
    uint64_t *meta;
    double *stats;
};

// parameters of the Nelder-Mead analyses (pg_nm.cu): mle_iter and gwalpha run after the scan kernel's filter-only pass
struct NmParams {
    Layout lay;
    const double *freq;
    const uint32_t *depth;
    int64_t n_loci;
    int kind;
    int k;                 // phenotypes (mle) | 1 (gwalpha)
    const double *yraw;    // mle: [k][n_pad] raw phenotypes; gwalpha: bins [n_pad] then q [n_pad]
    double gw_sig, gw_min, gw_max;
    double df, ln_beta;    // Student-t(n - 1)
    const void *ptab;
    double ptab_isd, ptab_bits, ptab_t1, ptab_t0;  // t1 / t0: PTable::t_one / t_zero
    int ptab_M;
    uint8_t codes[8];      // allele code of device column j
    uint64_t *meta;
    double *stats;         // [locus][A-1][k][4]
};
cudaError_t launch_nm(const NmParams &p, int sm_count, cudaStream_t s);

// mle_with_covariate (src/gwas/mle.rs:307-463) over the resident allele columns of a pg_kin (pg_nm.cu): X = [1 | PCs | g]
constexpr int kKinMleMaxM = 13;  // covariates: the simplex search runs over sigma2 + (2 + m) coefficients <= 16 parameters
struct KinMleParams {
    const double *G;     // [P][ldg] allele columns
    int64_t P;
    int n, ldg, m, k;
    const double *Z;     // [m + k][ldg]: centred covariates, then centred phenotypes
    const double *fix;   // zbar[m] | Szz[m][m] | Szz^-1 [m][m] | per phenotype: ybar, Syy, Szy[m]
    double df, ln_beta;  // Student-t(n - 1)
    const void *ptab;
    double ptab_isd, ptab_bits, ptab_t1, ptab_t0;  // t1 / t0: PTable::t_one / t_zero
    int ptab_M;
    double *beta, *var, *pval;  // [k][P]
};
cudaError_t launch_kin_mle(const KinMleParams &p, int sm_count, cudaStream_t s);

// launchers implemented in the kernel translation units
cudaError_t launch_scan(const ScanParams &p, int sm_count, cudaStream_t s);
cudaError_t launch_tables(const TableParams &p, int sm_count, cudaStream_t s);
// what an ingest kernel produces for a slab of loci (device pointers already offset to the first locus of the slab)
struct IngestOut {
    double *freq;
    uint32_t *depth;
    uint32_t *dmin;
    uint8_t *hint;   // [locus] renormalisation hint of the scan (pg_ingest.cu:locus_hint)
    const double *w; // [n_pad] pool weights s_i / sum(s)
    double maf, one_minus_maf, min_depth_f;
};
cudaError_t launch_ingest_u32(const uint32_t *counts, int64_t n_loci, int n, int A_in, int drop_col, const Layout &lay,
                              const IngestOut &o, cudaStream_t s);
cudaError_t launch_ingest_u16(const uint16_t *counts, int64_t n_loci, int n, int A_in, int drop_col, const Layout &lay,
                              const IngestOut &o, cudaStream_t s);
cudaError_t launch_ingest_u8(const uint8_t *counts, int64_t n_loci, int n, int A_in, int drop_col, const Layout &lay,
                             const IngestOut &o, cudaStream_t s);
cudaError_t launch_ingest_freq(const double *freq_in, const uint32_t *depth_in, int64_t n_loci, int n, const Layout &lay,
                               const IngestOut &o, cudaStream_t s);
cudaError_t launch_synth(uint64_t seed, int64_t first_locus, int64_t n_loci, int n, int A_in,
                         uint32_t *counts, cudaStream_t s);
// u8 / u16 counts -> u32 (the count tests read u32)
cudaError_t launch_widen(const void *src, int elem_bytes, uint32_t *dst, size_t count, cudaStream_t s);

// ---- host-side ownership ---------------------------------------------------------------------
// One allocation of device memory (Pinned = false) or pinned host memory (Pinned = true), freed by the destructor.
// The handles below own every buffer through this type.  A handle's destructor synchronises its stream before the
// buffers (members) are freed, so no queued work still reads or writes one; its events and stream are destroyed after
// that synchronisation.
template <typename T, bool Pinned>
class Buffer {
  public:
    Buffer() = default;
    Buffer(const Buffer &) = delete;
    Buffer &operator=(const Buffer &) = delete;
    Buffer(Buffer &&o) noexcept : p_(o.p_), cap_(o.cap_) { o.p_ = nullptr, o.cap_ = 0; }
    Buffer &operator=(Buffer &&o) noexcept {
        std::swap(p_, o.p_);
        std::swap(cap_, o.cap_);
        return *this;
    }
    ~Buffer() { release(); }

    // Nothing when `count` elements fit.  Otherwise waits for `stream` (queued work may still use the old allocation),
    // frees it and allocates exactly `count` elements.  After a failed reserve the buffer is empty: get() is null and
    // capacity() is 0, so the next reserve allocates again.
    cudaError_t reserve(size_t count, cudaStream_t stream) {
        if (cap_ >= count) return cudaSuccess;
        cudaError_t e = p_ ? cudaStreamSynchronize(stream) : cudaSuccess;
        release();
        if (e != cudaSuccess) return e;
        void *q = nullptr;
        if constexpr (Pinned)
            e = cudaHostAlloc(&q, count * sizeof(T), cudaHostAllocDefault);
        else
            e = cudaMalloc(&q, count * sizeof(T));
        if (e != cudaSuccess) {
            (void)cudaGetLastError();  // the error is returned here: a later launch check must not report it again
            return e;
        }
        p_ = static_cast<T *>(q);
        cap_ = count;
        return cudaSuccess;
    }
    T *get() const { return p_; }
    size_t capacity() const { return cap_; }

  private:
    void release() {
        if constexpr (Pinned) {
            if (p_) cudaFreeHost(p_);
        } else {
            cudaFree(p_);
        }
        p_ = nullptr;
        cap_ = 0;
    }
    T *p_ = nullptr;
    size_t cap_ = 0;
};
template <typename T>
using DeviceBuffer = Buffer<T, false>;
template <typename T>
using PinnedBuffer = Buffer<T, true>;

// sync text -> counts[locus][6][n_pools] on the device (pg_text.cu)
struct TextScratch {
    DeviceBuffer<char> d_text;
    DeviceBuffer<uint32_t> d_sep;
    DeviceBuffer<uint64_t> d_tok_blk;
    DeviceBuffer<uint32_t> d_nl, d_first, d_grp;
    DeviceBuffer<uint8_t> d_keep;
    DeviceBuffer<uint64_t> d_line_pos;
    DeviceBuffer<uint32_t> d_info;  // [4]: n_loci, error code, error offset, n_lines
    PinnedBuffer<uint32_t> h_info;  // its copy
    DeviceBuffer<uint8_t> d_tmp;
    DeviceBuffer<uint64_t> d_out_offset, d_out_pos;
    PinnedBuffer<uint64_t> h_out_offset, h_out_pos;  // the labels of the parsed loci: line offsets, positions
    cudaEvent_t parsed = nullptr;  // created by the first text_parse_async
    bool pending = false;          // text_parse_async issued, text_parse_finish not yet called
    int64_t max_loci = 0;
    ~TextScratch();  // the owner has synchronised the stream the parse ran on
};
cudaError_t text_parse_async(TextScratch *t, const char *text, size_t n_bytes, int n_pools, uint32_t *d_counts,
                             int64_t max_loci, size_t line_cap, int sm_count, cudaStream_t s);
int64_t text_parse_finish(TextScratch *t, cudaStream_t s, cudaError_t *cuda_err, uint64_t *err_offset);

}  // namespace pg

// opaque ABI types
struct pg_ctx {
    int device = 0;
    int sm_count = 0;
    int cc_major = 0, cc_minor = 0;
    size_t total_mem = 0;
};

namespace pg {
// sets the message pg_last_error() returns to the calling thread (printf format) and returns `code` (pg_api.cu)
int fail(pg_ctx *ctx, int code, const char *fmt, ...);
// the return code and message of a negative text_parse_finish result: `who` names the caller, `cap` is the number of
// loci the chunk may hold (pg_text.cu)
int text_parse_fail(pg_ctx *ctx, const char *who, int64_t status, cudaError_t cuda_err, uint64_t err_offset,
                    int n_pools, int64_t cap);
}  // namespace pg

#define PG_CUDA(ctx, call)                                                                              \
    do {                                                                                                \
        cudaError_t e_ = (call);                                                                        \
        if (e_ != cudaSuccess)                                                                          \
            return pg::fail((ctx), PG_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), \
                            __FILE__, __LINE__);                                                        \
    } while (0)

struct pg_scan {
    pg_ctx *ctx = nullptr;
    int kind = 0;
    int n = 0, A_in = 0, A_dev = 0, k = 0;
    int drop_col = -1;
    uint8_t codes_in[8] = {0};
    uint8_t codes_dev[8] = {0};
    pg::Layout lay;
    // filter
    int remove_ns = 1;
    uint64_t min_depth = 1;
    double maf = 0, max_miss = 0;
    int weighted = 0;
    double w_uniform = 0;
    std::vector<double> w_host;
    // phenotypes
    std::vector<double> yc_host;  // [k][n_pad]
    std::vector<double> ysum, syy, ymean;
    int y_has_nan = 0;
    double df = 0, ln_beta = 0;
    pg::DeviceBuffer<double> d_yc;
    pg::DeviceBuffer<double> d_w;
    pg::DeviceBuffer<double> d_yraw;  // mle_iter: raw phenotypes [k][n_pad]; gwalpha: bins [n_pad], q [n_pad]
    double gw_sig = 0, gw_min = 0, gw_max = 0;  // gwalpha_fmt: sig, MIN, MAX
    pg::DeviceBuffer<double> d_ptab;
    double ptab_isd = 0, ptab_bits = 0, ptab_err = 0, ptab_t1 = 0, ptab_t0 = 0;
    int ptab_M = 0;
    int n_slots = 0;
    // streaming
    pg_batch *slabs[PG_STREAM_DEPTH] = {nullptr, nullptr, nullptr};
    int next_slab = 0;
    int64_t slab_cap = 0;
    ~pg_scan();  // destroys the slabs
};

struct pg_batch {
    pg_scan *scan = nullptr;
    int64_t cap = 0, n_loci = 0;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    // device
    pg::DeviceBuffer<double> d_freq;
    pg::DeviceBuffer<uint32_t> d_depth;
    pg::DeviceBuffer<uint32_t> d_dmin;
    pg::DeviceBuffer<uint64_t> d_defer;  // [cap + 1]: list then its counter
    pg::DeviceBuffer<uint8_t> d_hint;    // [cap]
    pg::DeviceBuffer<uint8_t> d_stage;   // raw uploaded slab (counts u32/u16 or unpadded freq+depth)
    pg::DeviceBuffer<uint64_t> d_meta;
    pg::DeviceBuffer<double> d_fmean;
    pg::DeviceBuffer<double> d_stats;
    // pinned host results
    pg::PinnedBuffer<uint64_t> h_meta;
    pg::PinnedBuffer<double> h_fmean;
    pg::PinnedBuffer<double> h_stats;
    int have_input = 0;
    int input_is_counts = 0;
    pg::TextScratch text;
    const char *text_src = nullptr;  // the caller's chunk of the last text upload (valid until its slab is collected)
    size_t text_bytes = 0;
    ~pg_batch();
};

