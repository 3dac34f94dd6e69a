// pg_api.cu -- the C ABI of include/poolgen_cuda.h: context, scan configuration, batches, streaming.
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <new>

#include "pg_internal.h"
#include "pg_ptable.h"

namespace pg {
cudaError_t launch_scan_a2(const ScanParams &, int, cudaStream_t);
cudaError_t launch_scan_a3(const ScanParams &, int, cudaStream_t);
cudaError_t launch_scan_a4(const ScanParams &, int, cudaStream_t);
cudaError_t launch_scan_a5(const ScanParams &, int, cudaStream_t);
cudaError_t launch_scan_a6(const ScanParams &, int, cudaStream_t);

cudaError_t launch_scan(const ScanParams &p, int sm_count, cudaStream_t s) {
    switch (p.lay.A) {
        case 2: return launch_scan_a2(p, sm_count, s);
        case 3: return launch_scan_a3(p, sm_count, s);
        case 4: return launch_scan_a4(p, sm_count, s);
        case 5: return launch_scan_a5(p, sm_count, s);
        case 6: return launch_scan_a6(p, sm_count, s);
        default: return cudaErrorInvalidValue;
    }
}
}  // namespace pg

// The last error message is per THREAD: reader threads share one pg_ctx (src/base/sync.rs:917-939 runs one reader per
// file chunk), and the thread that made the failing call is the one that asks for the message.
static thread_local std::string g_last_err;

int pg::fail(pg_ctx *, int code, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_last_err = buf;
    return code;
}

using pg::fail;

pg_scan::~pg_scan() {
    for (pg_batch *b : slabs) delete b;
}

pg_batch::~pg_batch() {
    if (stream) cudaStreamSynchronize(stream);
    if (ev0) cudaEventDestroy(ev0);
    if (ev1) cudaEventDestroy(ev1);
    if (stream) cudaStreamDestroy(stream);
}

extern "C" {

int pg_abi_version(void) { return PG_ABI_VERSION; }

int pg_init(int device, pg_ctx **out) {
    if (!out) return fail(nullptr, PG_ERR_ARG, "pg_init: out is NULL");
    *out = nullptr;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(nullptr, PG_ERR_CUDA, "pg_init: no CUDA device (%s); this library has no CPU fallback",
                    e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
    if (device < 0 || device >= ndev) return fail(nullptr, PG_ERR_ARG, "pg_init: device %d of %d", device, ndev);
    cudaDeviceProp prop;
    PG_CUDA(nullptr, cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10)
        return fail(nullptr, PG_ERR_CUDA, "pg_init: device %d is sm_%d%d; the kernels are built for sm_100a only",
                    device, prop.major, prop.minor);
    PG_CUDA(nullptr, cudaSetDevice(device));
    pg_ctx *c = new (std::nothrow) pg_ctx();
    if (!c) return fail(nullptr, PG_ERR_ARG, "pg_init: out of host memory");
    c->device = device;
    c->sm_count = prop.multiProcessorCount;
    c->cc_major = prop.major;
    c->cc_minor = prop.minor;
    c->total_mem = prop.totalGlobalMem;
    *out = c;
    return PG_OK;
}

void pg_destroy(pg_ctx *ctx) { delete ctx; }

const char *pg_last_error(const pg_ctx *) { return g_last_err.c_str(); }

int pg_device_info(pg_ctx *ctx, int *sm_count, int *cc_major, int *cc_minor, size_t *total_mem) {
    if (!ctx) return PG_ERR_ARG;
    if (sm_count) *sm_count = ctx->sm_count;
    if (cc_major) *cc_major = ctx->cc_major;
    if (cc_minor) *cc_minor = ctx->cc_minor;
    if (total_mem) *total_mem = ctx->total_mem;
    return PG_OK;
}

// free and total device memory now (cudaMemGetInfo): other processes share the GPU, so a caller that sizes its blocks
// from the device takes them from what is free
int pg_device_mem_info(pg_ctx *ctx, size_t *free_bytes, size_t *total_bytes) {
    if (!ctx) return PG_ERR_ARG;
    PG_CUDA(ctx, cudaSetDevice(ctx->device));
    size_t f = 0, t = 0;
    PG_CUDA(ctx, cudaMemGetInfo(&f, &t));
    if (free_bytes) *free_bytes = f;
    if (total_bytes) *total_bytes = t;
    return PG_OK;
}

int pg_pinned_alloc(pg_ctx *ctx, size_t bytes, void **out) {
    if (!ctx || !out) return PG_ERR_ARG;
    PG_CUDA(ctx, cudaSetDevice(ctx->device));
    PG_CUDA(ctx, cudaHostAlloc(out, bytes ? bytes : 1, cudaHostAllocDefault));
    return PG_OK;
}

int pg_pinned_free(pg_ctx *ctx, void *p) {
    if (!ctx) return PG_ERR_ARG;
    if (p) PG_CUDA(ctx, cudaFreeHost(p));
    return PG_OK;
}

// ---------------------------------------------------------------------------------------------
int pg_scan_open(pg_ctx *ctx, int kind, const pg_filter *filter, int n_pools, int n_alleles,
                 const uint8_t *allele_codes, const double *phen, int k, pg_scan **out) {
    if (!ctx || !out || !filter || !allele_codes) return fail(ctx, PG_ERR_ARG, "pg_scan_open: NULL argument");
    *out = nullptr;
    const bool gwalpha = (kind == PG_KIND_GWALPHA_LS || kind == PG_KIND_GWALPHA_ML);
    if (!((kind >= PG_KIND_OLS && kind <= PG_KIND_FISHER) || kind == PG_KIND_MLE || gwalpha))
        return fail(ctx, PG_ERR_ARG, "pg_scan_open: kind %d", kind);
    if (n_pools < 1) return fail(ctx, PG_ERR_ARG, "pg_scan_open: n_pools %d", n_pools);
    if (n_alleles < 1 || n_alleles > PG_MAX_ALLELES)
        return fail(ctx, PG_ERR_ARG, "pg_scan_open: n_alleles %d not in 1..6", n_alleles);
    for (int j = 0; j < n_alleles; j++) {
        if (allele_codes[j] > 5) return fail(ctx, PG_ERR_ARG, "pg_scan_open: allele code %d", allele_codes[j]);
        if (j && allele_codes[j] <= allele_codes[j - 1])
            return fail(ctx, PG_ERR_ARG, "pg_scan_open: allele codes must be strictly increasing (sync column order)");
    }
    // assert!(n == filter_stats.pool_sizes.len()) src/base/sync.rs:254-257
    if (filter->n_pool_sizes != n_pools || !filter->pool_sizes)
        return fail(ctx, PG_ERR_ARG, "pg_scan_open: %d pool sizes for %d pools (the reference asserts equality)",
                    filter->n_pool_sizes, n_pools);
    const bool regression = (kind == PG_KIND_OLS || kind == PG_KIND_CORR || kind == PG_KIND_MLE || gwalpha);
    if (regression && (!phen || k < 1)) return fail(ctx, PG_ERR_ARG, "pg_scan_open: phenotypes required");
    // gwalpha: `phen` is the gwalpha_fmt matrix, k rows x 3 (column 0 bins, column 1 q, column 2 = sig, MIN, MAX, then
    // -inf fillers, src/gwas/gwalpha.rs:197-216); the scan's own "phenotype" is only a stand-in for the filter-only pass
    std::vector<double> gw_bins, gw_q, gw_stand_in;
    const int gw_rows = k;
    if (gwalpha) {
        if (k < 3) return fail(ctx, PG_ERR_ARG, "pg_scan_open: the gwalpha_fmt matrix needs at least 3 rows (sig, MIN, MAX)");
        for (int i = 0; i < k; i++) {
            if (phen[(size_t)i * 3 + 0] != -INFINITY) gw_bins.push_back(phen[(size_t)i * 3 + 0]);
            if (phen[(size_t)i * 3 + 1] != -INFINITY) gw_q.push_back(phen[(size_t)i * 3 + 1]);
        }
        if ((int)gw_bins.size() != n_pools || (int)gw_q.size() < n_pools)
            return fail(ctx, PG_ERR_ARG, "pg_scan_open: %d bins for %d pools (the reference returns None for every locus, "
                                         "src/gwas/gwalpha.rs:218-223)", (int)gw_bins.size(), n_pools);
        if (n_pools > 64) return fail(ctx, PG_ERR_UNSUPPORTED, "pg_scan_open: gwalpha is built for up to 64 pools (got %d)", n_pools);
        gw_stand_in.assign(n_pools, 0.0);
        for (int i = 0; i < n_pools; i++) gw_stand_in[i] = (double)(i % 7) - 3.0;
        k = 1;
    }
    const double *gw_fmt = phen;
    if (gwalpha) phen = gw_stand_in.data();
    PG_CUDA(ctx, cudaSetDevice(ctx->device));

    pg_scan *s = new (std::nothrow) pg_scan();
    if (!s) return fail(ctx, PG_ERR_ARG, "out of host memory");
    s->ctx = ctx;
    s->kind = kind;
    s->n = n_pools;
    s->A_in = n_alleles;
    s->k = regression ? k : 1;
    s->remove_ns = filter->remove_ns != 0;
    s->min_depth = filter->min_coverage_depth;
    s->maf = filter->min_allele_frequency;
    s->max_miss = filter->max_missingness_rate;
    s->drop_col = -1;
    int jj = 0;
    for (int j = 0; j < n_alleles; j++) {
        s->codes_in[j] = allele_codes[j];
        if (s->remove_ns && allele_codes[j] == 4) {
            s->drop_col = j;  // src/base/sync.rs:200-213
            continue;
        }
        s->codes_dev[jj++] = allele_codes[j];
    }
    s->A_dev = jj;
    if (regression && (s->A_dev < 2 || s->A_dev > 6)) {
        delete s;
        return fail(ctx, PG_ERR_ARG, "pg_scan_open: %d usable allele columns, need 2..6", jj);
    }
    s->lay = pg::make_layout(n_pools, s->A_dev);
    s->n_slots = regression ? s->A_dev - 1 : 1;
    // pool weights exactly as src/base/sync.rs:262-270: s_i / (sequential sum of s)
    double S = 0.0;
    for (int i = 0; i < n_pools; i++) S = S + filter->pool_sizes[i];
    s->w_host.assign(s->lay.n_pad, 0.0);
    for (int i = 0; i < n_pools; i++) s->w_host[i] = filter->pool_sizes[i] / S;
    s->weighted = 0;
    for (int i = 1; i < n_pools; i++)
        if (s->w_host[i] != s->w_host[0]) s->weighted = 1;
    s->w_uniform = s->w_host[0];

    if (regression) {
        const int n = n_pools, np = s->lay.n_pad;
        s->yc_host.assign((size_t)k * np, 0.0);
        s->ysum.assign(k, 0.0);
        s->syy.assign(k, 0.0);
        s->ymean.assign(k, 0.0);
        for (int j = 0; j < k; j++) {
            double sum = 0.0;
            int n_valid = 0;
            for (int i = 0; i < n; i++) {
                const double v = phen[(size_t)i * k + j];
                if (v != v) {
                    s->y_has_nan = 1;  // NA phenotype (src/base/phen.rs:68-75)
                    continue;
                }
                sum += v;
                n_valid++;
            }
            const double mean = n_valid ? sum / n_valid : 0.0;  // = sum / n without missing values
            double s1 = 0.0, s2 = 0.0;
            for (int i = 0; i < n; i++) {
                const double c = phen[(size_t)i * k + j] - mean;
                s->yc_host[(size_t)j * np + i] = c;
                s1 += c;
                s2 += c * c;
            }
            s->ysum[j] = s1;
            s->ymean[j] = mean;
            s->syy[j] = s2 - s1 * s1 / n;
        }
        if (s->y_has_nan && (kind == PG_KIND_OLS || kind == PG_KIND_MLE)) {
            // ols_iterate: remove_missing() shrinks the pools but not FilterStats.pool_sizes, so the reference
            // panics at src/base/sync.rs:254-257.  pearson_corr drops NaN pairs per phenotype
            // (correlation_test.rs:21-31): every locus of such a scan takes the pairwise path of the fix-up kernel.
            delete s;
            return fail(ctx, PG_ERR_UNSUPPORTED,
                        "pg_scan_open: missing phenotype values (the reference's ols_iter panics on them, "
                        "src/base/sync.rs:254-257)");
        }
        s->df = (kind != PG_KIND_CORR) ? (double)n - 1.0 : (double)n - 2.0;
        if (kind != PG_KIND_CORR && !(s->df > 0.0)) {
            delete s;  // StudentsT::new(0,1,0).unwrap() panics (src/gwas/ols.rs:139)
            return fail(ctx, PG_ERR_UNSUPPORTED, "pg_scan_open: ols_iter needs at least 2 pools");
        }
        s->ln_beta = s->df > 0.0 ? pg::statrs::ln_gamma(s->df / 2.0 + 0.5) - pg::statrs::ln_gamma(s->df / 2.0) - pg::statrs::ln_gamma(0.5) : 0.0;
        const char *pv_mode = getenv("PG_PVALUE");
        if (s->df > 0.0 && !(pv_mode && strcmp(pv_mode, "cf") == 0)) {
            pg::PTable tab = pg::build_ptable(s->df);
            if (tab.max_err < 2e-9) {  // otherwise keep the continued fraction
                cudaError_t et = s->d_ptab.reserve(tab.coef.size(), nullptr);
                if (et == cudaSuccess)
                    et = cudaMemcpy(s->d_ptab.get(), tab.coef.data(), tab.coef.size() * 8, cudaMemcpyHostToDevice);
                if (et != cudaSuccess) {
                    delete s;
                    return fail(ctx, PG_ERR_CUDA, "pg_scan_open: p-value table upload: %s", cudaGetErrorString(et));
                }
                s->ptab_M = tab.M;
                s->ptab_isd = tab.inv_sqrt_df;
                s->ptab_bits = tab.bits;
                s->ptab_t1 = tab.t_one;
                s->ptab_t0 = tab.t_zero;
                s->ptab_err = tab.max_err;
            }
        }
        cudaError_t e = s->d_yc.reserve(s->yc_host.size(), nullptr);
        if (e == cudaSuccess) e = cudaMemcpy(s->d_yc.get(), s->yc_host.data(), s->yc_host.size() * 8, cudaMemcpyHostToDevice);
        if (e != cudaSuccess) {
            delete s;
            return fail(ctx, PG_ERR_CUDA, "pg_scan_open: phenotype upload: %s", cudaGetErrorString(e));
        }
    }
    {
        cudaError_t e = s->d_w.reserve(s->w_host.size(), nullptr);
        if (e == cudaSuccess) e = cudaMemcpy(s->d_w.get(), s->w_host.data(), s->w_host.size() * 8, cudaMemcpyHostToDevice);
        if (e != cudaSuccess) {
            delete s;
            return fail(ctx, PG_ERR_CUDA, "pg_scan_open: weight upload: %s", cudaGetErrorString(e));
        }
    }
    if (kind == PG_KIND_MLE || gwalpha) {
        // what the Nelder-Mead kernels read: raw phenotypes [k][n_pad] (mle_iter) | bins [n_pad], q [n_pad] (gwalpha)
        const int np = s->lay.n_pad;
        std::vector<double> raw((size_t)(gwalpha ? 2 : k) * np, 0.0);
        if (gwalpha) {
            for (int i = 0; i < n_pools; i++) {
                raw[i] = gw_bins[i];
                raw[(size_t)np + i] = gw_q[i];
            }
            s->gw_sig = gw_fmt[0 * 3 + 2];
            s->gw_min = gw_fmt[1 * 3 + 2];
            s->gw_max = gw_fmt[2 * 3 + 2];
            (void)gw_rows;
        } else {
            for (int j = 0; j < k; j++)
                for (int i = 0; i < n_pools; i++) raw[(size_t)j * np + i] = phen[(size_t)i * k + j];
        }
        cudaError_t e = s->d_yraw.reserve(raw.size(), nullptr);
        if (e == cudaSuccess) e = cudaMemcpy(s->d_yraw.get(), raw.data(), raw.size() * 8, cudaMemcpyHostToDevice);
        if (e != cudaSuccess) {
            delete s;
            return fail(ctx, PG_ERR_CUDA, "pg_scan_open: phenotype upload: %s", cudaGetErrorString(e));
        }
    }
    // pageable-memory copies may return before the DMA has landed and the batches' streams are non-blocking (not
    // ordered against the legacy stream): the phenotype, weight and p-table uploads are complete when this returns
    {
        cudaError_t e = cudaDeviceSynchronize();
        if (e != cudaSuccess) {
            delete s;
            return fail(ctx, PG_ERR_CUDA, "pg_scan_open: %s", cudaGetErrorString(e));
        }
    }
    *out = s;
    return PG_OK;
}

int pg_scan_close(pg_scan *s) {
    delete s;
    return PG_OK;
}

// ---------------------------------------------------------------------------------------------
static bool is_nm(const pg_scan *s) { return s->kind == PG_KIND_MLE || s->kind == PG_KIND_GWALPHA_LS || s->kind == PG_KIND_GWALPHA_ML; }
static bool is_regression(const pg_scan *s) { return s->kind == PG_KIND_OLS || s->kind == PG_KIND_CORR || is_nm(s); }

int pg_batch_create(pg_scan *s, int64_t cap, pg_batch **out) {
    if (!s || !out || cap < 1 || cap > 0x7FFFFFFFLL) return fail(s ? s->ctx : nullptr, PG_ERR_ARG, "pg_batch_create: bad argument (1 <= capacity < 2^31 loci)");
    pg_ctx *ctx = s->ctx;
    *out = nullptr;
    PG_CUDA(ctx, cudaSetDevice(ctx->device));
    pg_batch *b = new (std::nothrow) pg_batch();
    if (!b) return fail(ctx, PG_ERR_ARG, "out of host memory");
    b->scan = s;
    b->cap = cap;
    cudaError_t e = cudaStreamCreateWithFlags(&b->stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaEventCreate(&b->ev0);
    if (e == cudaSuccess) e = cudaEventCreate(&b->ev1);
    if (e == cudaSuccess && is_regression(s)) {
        e = b->d_freq.reserve((size_t)cap * s->lay.freq_stride(), b->stream);
        if (e == cudaSuccess) e = b->d_depth.reserve((size_t)cap * s->lay.depth_stride(), b->stream);
        if (e == cudaSuccess) e = b->d_dmin.reserve((size_t)cap, b->stream);
        if (e == cudaSuccess) e = b->d_defer.reserve((size_t)cap + 1, b->stream);
        if (e == cudaSuccess) e = b->d_hint.reserve((size_t)cap, b->stream);
    }
    const size_t S = s->n_slots, K = s->k;
    if (e == cudaSuccess) e = b->d_meta.reserve((size_t)cap, b->stream);
    if (e == cudaSuccess) e = b->d_fmean.reserve((size_t)cap * S, b->stream);
    if (e == cudaSuccess) e = b->d_stats.reserve((size_t)cap * S * K * 4, b->stream);
    if (e != cudaSuccess) {
        delete b;
        return fail(ctx, PG_ERR_CUDA, "pg_batch_create(%lld loci): %s", (long long)cap, cudaGetErrorString(e));
    }
    *out = b;
    return PG_OK;
}

int pg_batch_destroy(pg_batch *b) {
    delete b;
    return PG_OK;
}

static pg::IngestOut ingest_out(pg_batch *b, int64_t first_locus) {
    pg_scan *s = b->scan;
    pg::IngestOut o;
    o.freq = b->d_freq.get() + (size_t)first_locus * s->lay.freq_stride();
    o.depth = b->d_depth.get() + (size_t)first_locus * s->lay.depth_stride();
    o.dmin = b->d_dmin.get() + first_locus;
    o.hint = b->d_hint.get() + first_locus;
    o.w = s->d_w.get();
    o.maf = s->maf;
    o.one_minus_maf = 1.00 - s->maf;
    o.min_depth_f = (double)s->min_depth;
    return o;
}

}  // extern "C"

// the staging area of the uploads: at least `bytes` bytes
static int ensure_stage(pg_batch *b, size_t bytes) {
    PG_CUDA(b->scan->ctx, b->d_stage.reserve(bytes, b->stream));
    return PG_OK;
}

template <typename CT>
static int upload_counts_t(pg_batch *b, const CT *counts, int64_t n_loci) {
    if (!b || (!counts && n_loci > 0)) return PG_ERR_ARG;
    pg_scan *s = b->scan;
    pg_ctx *ctx = s->ctx;
    if (n_loci < 0 || n_loci > b->cap) return fail(ctx, PG_ERR_ARG, "upload: %lld loci > capacity %lld", (long long)n_loci, (long long)b->cap);
    PG_CUDA(ctx, cudaSetDevice(ctx->device));
    b->n_loci = n_loci;
    b->have_input = 1;
    if (n_loci == 0) return PG_OK;
    const size_t bytes = (size_t)n_loci * s->A_in * s->n * sizeof(CT);
    const bool reg = is_regression(s);
    const size_t wide_bytes = (size_t)b->cap * s->A_in * s->n * 4;
    // the count tests read u32 counts: narrow slabs land behind the u32 area and are widened on the device
    int rc = ensure_stage(b, reg ? (size_t)b->cap * s->A_in * s->n * sizeof(CT) : wide_bytes + (sizeof(CT) == 4 ? 0 : bytes));
    if (rc) return rc;
    if (reg) {
        PG_CUDA(ctx, cudaMemcpyAsync(b->d_stage.get(), counts, bytes, cudaMemcpyHostToDevice, b->stream));
        if constexpr (sizeof(CT) == 4)
            PG_CUDA(ctx, pg::launch_ingest_u32((const uint32_t *)b->d_stage.get(), n_loci, s->n, s->A_in, s->drop_col, s->lay,
                                               ingest_out(b, 0), b->stream));
        else if constexpr (sizeof(CT) == 1)
            PG_CUDA(ctx, pg::launch_ingest_u8((const uint8_t *)b->d_stage.get(), n_loci, s->n, s->A_in, s->drop_col, s->lay,
                                              ingest_out(b, 0), b->stream));
        else
            PG_CUDA(ctx, pg::launch_ingest_u16((const uint16_t *)b->d_stage.get(), n_loci, s->n, s->A_in, s->drop_col, s->lay,
                                               ingest_out(b, 0), b->stream));
    } else if constexpr (sizeof(CT) == 4) {
        PG_CUDA(ctx, cudaMemcpyAsync(b->d_stage.get(), counts, bytes, cudaMemcpyHostToDevice, b->stream));
    } else {
        void *narrow = (char *)b->d_stage.get() + wide_bytes;
        PG_CUDA(ctx, cudaMemcpyAsync(narrow, counts, bytes, cudaMemcpyHostToDevice, b->stream));
        PG_CUDA(ctx, pg::launch_widen(narrow, (int)sizeof(CT), (uint32_t *)b->d_stage.get(), (size_t)n_loci * s->A_in * s->n,
                                      b->stream));
    }
    b->input_is_counts = 1;
    return PG_OK;
}

extern "C" {

int pg_batch_upload_counts(pg_batch *b, const uint32_t *counts, int64_t n_loci) {
    return upload_counts_t<uint32_t>(b, counts, n_loci);
}
int pg_batch_upload_counts_u16(pg_batch *b, const uint16_t *counts, int64_t n_loci) {
    return upload_counts_t<uint16_t>(b, counts, n_loci);
}
int pg_batch_upload_counts_u8(pg_batch *b, const uint8_t *counts, int64_t n_loci) {
    return upload_counts_t<uint8_t>(b, counts, n_loci);
}

int pg_batch_upload_freq(pg_batch *b, const double *freq, const uint32_t *depth, int64_t n_loci) {
    if (!b || ((!freq || !depth) && n_loci > 0)) return PG_ERR_ARG;
    pg_scan *s = b->scan;
    pg_ctx *ctx = s->ctx;
    if (!is_regression(s)) return fail(ctx, PG_ERR_UNSUPPORTED, "upload_freq: the table tests need counts");
    if (s->drop_col >= 0)
        return fail(ctx, PG_ERR_ARG, "upload_freq: the frequency matrix must not contain the N column when remove_ns is set");
    if (n_loci < 0 || n_loci > b->cap) return fail(ctx, PG_ERR_ARG, "upload: %lld loci > capacity %lld", (long long)n_loci, (long long)b->cap);
    PG_CUDA(ctx, cudaSetDevice(ctx->device));
    b->n_loci = n_loci;
    b->have_input = 1;
    if (n_loci == 0) return PG_OK;
    const size_t fbytes_cap = (size_t)b->cap * s->A_dev * s->n * 8, dbytes_cap = (size_t)b->cap * s->n * 4;
    int rc = ensure_stage(b, fbytes_cap + dbytes_cap);
    if (rc) return rc;
    double *sf = (double *)b->d_stage.get();
    uint32_t *sd = (uint32_t *)((char *)b->d_stage.get() + fbytes_cap);
    PG_CUDA(ctx, cudaMemcpyAsync(sf, freq, (size_t)n_loci * s->A_dev * s->n * 8, cudaMemcpyHostToDevice, b->stream));
    PG_CUDA(ctx, cudaMemcpyAsync(sd, depth, (size_t)n_loci * s->n * 4, cudaMemcpyHostToDevice, b->stream));
    PG_CUDA(ctx, pg::launch_ingest_freq(sf, sd, n_loci, s->n, s->lay, ingest_out(b, 0), b->stream));
    b->input_is_counts = 0;
    return PG_OK;
}

// stage A of a text upload: copy + device parse, asynchronous (pg_text.cu)
static int text_stage_a(pg_batch *b, const char *text, size_t n_bytes, size_t line_cap) {
    if (!b || (!text && n_bytes > 0)) return PG_ERR_ARG;
    pg_scan *s = b->scan;
    pg_ctx *ctx = s->ctx;
    if (s->A_in != 6) return fail(ctx, PG_ERR_ARG, "upload_sync_text: the scan must be opened with the six sync columns A:T:C:G:N:D");
    for (int j = 0; j < 6; j++)
        if (s->codes_in[j] != j) return fail(ctx, PG_ERR_ARG, "upload_sync_text: allele codes must be 0..5 in sync order");
    PG_CUDA(ctx, cudaSetDevice(ctx->device));
    b->n_loci = 0;
    b->have_input = 1;
    b->input_is_counts = 1;
    b->text_src = text;
    b->text_bytes = n_bytes;
    int rc = ensure_stage(b, (size_t)b->cap * 6 * s->n * 4);
    if (rc) return rc;
    const cudaError_t pe = pg::text_parse_async(&b->text, text, n_bytes, s->n, (uint32_t *)b->d_stage.get(), b->cap, line_cap,
                                                ctx->sm_count, b->stream);
    if (pe != cudaSuccess) {
        b->have_input = 0;  // nothing usable is resident: a later run / collect must not scan the previous chunk
        b->n_loci = 0;
        return fail(ctx, PG_ERR_CUDA, "upload_sync_text: %s", cudaGetErrorString(pe));
    }
    return PG_OK;
}

// stage B: wait for the parse, learn the number of loci, enqueue the label copy and the ingest
static int text_stage_b(pg_batch *b, int64_t *n_loci_out) {
    pg_scan *s = b->scan;
    pg_ctx *ctx = s->ctx;
    if (n_loci_out) *n_loci_out = 0;
    cudaError_t ce = cudaSuccess;
    uint64_t at = 0;
    int64_t L = pg::text_parse_finish(&b->text, b->stream, &ce, &at);
    if (L == -5) {  // more (comment / blank) lines than the default bound: repeat with the exact number
        int rc = text_stage_a(b, b->text_src, b->text_bytes, (size_t)at + 1);
        if (rc) return rc;
        L = pg::text_parse_finish(&b->text, b->stream, &ce, &at);
    }
    if (L < 0) return pg::text_parse_fail(ctx, "upload_sync_text", L, ce, at, s->n, b->cap);
    b->n_loci = L;
    if (n_loci_out) *n_loci_out = L;
    if (L > 0 && is_regression(s))
        PG_CUDA(ctx, pg::launch_ingest_u32((const uint32_t *)b->d_stage.get(), L, s->n, s->A_in, s->drop_col, s->lay,
                                           ingest_out(b, 0), b->stream));
    return PG_OK;
}

int pg_batch_upload_sync_text(pg_batch *b, const char *text, size_t n_bytes, int64_t *n_loci_out) {
    if (n_loci_out) *n_loci_out = 0;
    int rc = text_stage_a(b, text, n_bytes, 0);
    if (rc) return rc;
    rc = text_stage_b(b, n_loci_out);
    if (rc) return rc;
    PG_CUDA(b->scan->ctx, cudaStreamSynchronize(b->stream));  // the labels are on the host when this returns
    return PG_OK;
}

int pg_batch_text_labels(pg_batch *b, const uint64_t **line_offsets, const uint64_t **positions) {
    if (!b) return PG_ERR_ARG;
    if (!b->text.parsed) return fail(b->scan->ctx, PG_ERR_STATE, "pg_batch_text_labels before pg_batch_upload_sync_text");
    if (line_offsets) *line_offsets = b->text.h_out_offset.get();
    if (positions) *positions = b->text.h_out_pos.get();
    return PG_OK;
}

int pg_batch_synth(pg_batch *b, uint64_t seed, int64_t first_locus, int64_t n_loci) {
    if (!b) return PG_ERR_ARG;
    pg_scan *s = b->scan;
    pg_ctx *ctx = s->ctx;
    if (n_loci < 0 || n_loci > b->cap) return fail(ctx, PG_ERR_ARG, "synth: %lld loci > capacity %lld", (long long)n_loci, (long long)b->cap);
    PG_CUDA(ctx, cudaSetDevice(ctx->device));
    b->n_loci = n_loci;
    b->have_input = 1;
    if (n_loci == 0) return PG_OK;
    const size_t per_locus = (size_t)s->A_in * s->n * 4;
    if (!is_regression(s)) {
        int rc = ensure_stage(b, (size_t)b->cap * per_locus);
        if (rc) return rc;
        PG_CUDA(ctx, pg::launch_synth(seed, first_locus, n_loci, s->n, s->A_in, (uint32_t *)b->d_stage.get(), b->stream));
        b->input_is_counts = 1;
        return PG_OK;
    }
    // generate in slices so that the staging buffer stays small next to the resident frequency matrix
    int64_t slice = (int64_t)((size_t)256 << 20) / (int64_t)per_locus;
    if (slice < 1) slice = 1;
    if (slice > n_loci) slice = n_loci;
    if (b->d_stage.capacity() < (size_t)slice * per_locus) {
        int rc = ensure_stage(b, (size_t)slice * per_locus);
        if (rc) return rc;
    } else {
        slice = (int64_t)(b->d_stage.capacity() / per_locus);
        if (slice > n_loci) slice = n_loci;
    }
    for (int64_t l0 = 0; l0 < n_loci; l0 += slice) {
        const int64_t m = (n_loci - l0 < slice) ? n_loci - l0 : slice;
        PG_CUDA(ctx, pg::launch_synth(seed, first_locus + l0, m, s->n, s->A_in, (uint32_t *)b->d_stage.get(), b->stream));
        PG_CUDA(ctx, pg::launch_ingest_u32((const uint32_t *)b->d_stage.get(), m, s->n, s->A_in, s->drop_col, s->lay,
                                           ingest_out(b, l0), b->stream));
    }
    b->input_is_counts = 1;
    return PG_OK;
}

static int run_once(pg_batch *b, int *launches) {
    pg_scan *s = b->scan;
    pg_ctx *ctx = s->ctx;
    if (!b->have_input) return fail(ctx, PG_ERR_STATE, "pg_batch_run: no input uploaded");
    if (b->n_loci == 0) return PG_OK;
    if (is_regression(s)) {
        // phenotypes per pass: bounded by the accumulator registers and, unless the scan reads them from L2
        // (pg::scan_wide), by the shared memory the resident phenotype vectors may take (96 KB of the 227 KB, the
        // rest belongs to the warps' rings)
        int kpass = pg::max_phen_per_pass(s->A_dev);
        if (!pg::scan_wide(s->lay)) {
            const int fit = (int)((size_t)(96 * 1024) / ((size_t)s->lay.n_pad * 8)) - (s->weighted ? 1 : 0);
            if (kpass > fit) kpass = fit < 1 ? 1 : fit;
        }
        static const int nbuf_env = getenv("PG_NBUF") ? atoi(getenv("PG_NBUF")) : 0;
        static const int warps_env = getenv("PG_WARPS") ? atoi(getenv("PG_WARPS")) : 0;
        static const int g_env = getenv("PG_G") ? atoi(getenv("PG_G")) : 0;
        static const int p_env = getenv("PG_P") ? atoi(getenv("PG_P")) : 0;
        if (is_nm(s)) kpass = 1;  // one filter-only pass: keep-mask, allele order, mean frequencies
        for (int base = 0; base < (is_nm(s) ? 1 : s->k); base += kpass) {
            pg::ScanParams p;
            memset(&p, 0, sizeof p);
            p.lay = s->lay;
            p.freq = b->d_freq.get();
            p.depth = b->d_depth.get();
            p.dmin = b->d_dmin.get();
            p.hint = b->d_hint.get();
            p.n_loci = b->n_loci;
            p.kind = is_nm(s) ? PG_KIND_OLS : s->kind;
            p.filter_only = is_nm(s) ? 1 : 0;
            p.weighted = s->weighted;
            p.maf = s->maf;
            p.one_minus_maf = 1.00 - s->maf;
            p.max_miss = s->max_miss;
            p.min_depth_f = (double)s->min_depth;
            p.w_uniform = s->w_uniform;
            p.df = s->df;
            p.inv_df = 1.0 / s->df;
            p.inv_n = 1.0 / (double)s->n;
            p.inv_nm2 = 1.0 / ((double)s->n - 2.0);
            p.ln_beta = s->ln_beta;
            p.ptab = s->d_ptab.get();
            p.ptab_isd = s->ptab_isd;
            p.ptab_bits = s->ptab_bits;
            p.ptab_t1 = s->ptab_t1;
            p.ptab_t0 = s->ptab_t0;
            p.ptab_M = s->ptab_M;
            p.K = std::min(kpass, s->k - base);
            p.y_has_nan = s->y_has_nan;
            p.yc = s->d_yc.get() + (size_t)base * s->lay.n_pad;
            p.w = s->d_w.get();
            for (int j = 0; j < p.K; j++) {
                p.ysum[j] = s->ysum[base + j];
                p.syy[j] = s->syy[base + j];
                p.ymean[j] = s->ymean[base + j];
            }
            for (int j = 0; j < s->A_dev; j++) p.codes[j] = s->codes_dev[j];
            p.meta = b->d_meta.get();
            p.freq_mean = b->d_fmean.get();
            p.stats = b->d_stats.get();
            p.defer_list = b->d_defer.get();
            p.defer_count = reinterpret_cast<uint32_t *>(b->d_defer.get() + b->cap);
            p.k_total = s->k;
            p.phen_base = base;
            p.write_meta = base == 0;
            p.nbuf_override = nbuf_env;
            p.warps_override = warps_env;
            p.g_override = g_env;
            p.p_override = p_env;
            PG_CUDA(ctx, pg::launch_scan(p, ctx->sm_count, b->stream));
            if (launches) (*launches) += 2;  // streaming kernel + fix-up kernel
        }
        if (is_nm(s)) {
            pg::NmParams q;
            memset(&q, 0, sizeof q);
            q.lay = s->lay;
            q.freq = b->d_freq.get();
            q.depth = b->d_depth.get();
            q.n_loci = b->n_loci;
            q.kind = s->kind;
            q.k = s->k;
            q.yraw = s->d_yraw.get();
            q.gw_sig = s->gw_sig;
            q.gw_min = s->gw_min;
            q.gw_max = s->gw_max;
            q.df = s->df;
            q.ln_beta = s->ln_beta;
            q.ptab = s->d_ptab.get();
            q.ptab_isd = s->ptab_isd;
            q.ptab_bits = s->ptab_bits;
            q.ptab_t1 = s->ptab_t1;
            q.ptab_t0 = s->ptab_t0;
            q.ptab_M = s->ptab_M;
            for (int j = 0; j < s->A_dev; j++) q.codes[j] = s->codes_dev[j];
            q.meta = b->d_meta.get();
            q.stats = b->d_stats.get();
            PG_CUDA(ctx, pg::launch_nm(q, ctx->sm_count, b->stream));
            if (launches) (*launches)++;
        }
    } else {
        pg::TableParams p;
        memset(&p, 0, sizeof p);
        p.counts = (const uint32_t *)b->d_stage.get();
        p.n_loci = b->n_loci;
        p.n = s->n;
        p.A_in = s->A_in;
        p.kind = s->kind;
        p.drop_col = s->drop_col;
        p.maf = s->maf;
        p.one_minus_maf = 1.00 - s->maf;
        p.max_miss = s->max_miss;
        p.min_depth_f = (double)s->min_depth;
        p.w = s->d_w.get();
        for (int j = 0; j < s->A_in; j++) p.codes[j] = s->codes_in[j];
        p.meta = b->d_meta.get();
        p.stats = b->d_stats.get();
        PG_CUDA(ctx, pg::launch_tables(p, ctx->sm_count, b->stream));
        if (launches) (*launches)++;
    }
    return PG_OK;
}

int pg_batch_run(pg_batch *b) {
    if (!b) return PG_ERR_ARG;
    PG_CUDA(b->scan->ctx, cudaSetDevice(b->scan->ctx->device));
    return run_once(b, nullptr);
}

int pg_batch_time_runs(pg_batch *b, int iters, float *ms_total, int *n_launches) {
    if (!b || iters < 1 || !ms_total) return PG_ERR_ARG;
    pg_ctx *ctx = b->scan->ctx;
    PG_CUDA(ctx, cudaSetDevice(ctx->device));
    int launches = 0;
    PG_CUDA(ctx, cudaStreamSynchronize(b->stream));
    PG_CUDA(ctx, cudaEventRecord(b->ev0, b->stream));
    for (int i = 0; i < iters; i++) {
        int rc = run_once(b, &launches);
        if (rc) return rc;
    }
    PG_CUDA(ctx, cudaEventRecord(b->ev1, b->stream));
    PG_CUDA(ctx, cudaEventSynchronize(b->ev1));
    PG_CUDA(ctx, cudaEventElapsedTime(ms_total, b->ev0, b->ev1));
    if (n_launches) *n_launches = launches;
    static const bool report = getenv("PG_REPORT_DEFER") != nullptr;  // diagnostic: why loci went to the fix-up kernel
    if (report && b->d_defer.get() && is_regression(b->scan)) {
        uint32_t count = 0;
        PG_CUDA(ctx, cudaMemcpy(&count, b->d_defer.get() + b->cap, 4, cudaMemcpyDeviceToHost));
        std::vector<uint64_t> list(count);
        if (count) PG_CUDA(ctx, cudaMemcpy(list.data(), b->d_defer.get(), (size_t)count * 8, cudaMemcpyDeviceToHost));
        uint32_t h[8] = {0, 0, 0, 0, 0, 0, 0, 0};
        for (uint64_t e : list) {
            const unsigned why = (unsigned)(e >> 56);
            if (why & 1u) h[0]++;
            if (why & 2u) h[1]++;
            if (why & 4u) h[2]++;
            if (why & 8u) h[3]++;
            if ((why >> 4) >= 1 && (why >> 4) <= 4) h[3 + (why >> 4)]++;
        }
        fprintf(stderr, "[pg] deferred %u of %lld loci (last phenotype pass): threshold %u, removed-with-reads %u, no coverage %u, "
                        "NaN under hint %u, redo ols %u, redo corr %u, corr NaN %u, tie %u\n",
                count, (long long)b->n_loci, h[0], h[1], h[2], h[3], h[4], h[5], h[6], h[7]);
    }
    return PG_OK;
}

int pg_batch_bytes(pg_batch *b, size_t *input_bytes, size_t *result_bytes) {
    if (!b) return PG_ERR_ARG;
    pg_scan *s = b->scan;
    const size_t L = (size_t)b->n_loci;
    if (input_bytes)
        *input_bytes = is_regression(s) ? L * (s->lay.freq_stride() * 8 + 4)  // frequency matrix + dmin
                                        : L * (size_t)s->A_in * s->n * 4;
    if (result_bytes) *result_bytes = L * (8 + (size_t)s->n_slots * 8 + (size_t)s->n_slots * s->k * 32);
    return PG_OK;
}

int pg_batch_download(pg_batch *b) {
    if (!b) return PG_ERR_ARG;
    pg_scan *s = b->scan;
    pg_ctx *ctx = s->ctx;
    PG_CUDA(ctx, cudaSetDevice(ctx->device));
    const size_t S = s->n_slots, K = s->k;
    PG_CUDA(ctx, b->h_meta.reserve((size_t)b->cap, b->stream));
    PG_CUDA(ctx, b->h_fmean.reserve((size_t)b->cap * S, b->stream));
    PG_CUDA(ctx, b->h_stats.reserve((size_t)b->cap * S * K * 4, b->stream));
    const size_t L = (size_t)b->n_loci;
    if (L == 0) return PG_OK;
    PG_CUDA(ctx, cudaMemcpyAsync(b->h_meta.get(), b->d_meta.get(), L * 8, cudaMemcpyDeviceToHost, b->stream));
    PG_CUDA(ctx, cudaMemcpyAsync(b->h_fmean.get(), b->d_fmean.get(), L * S * 8, cudaMemcpyDeviceToHost, b->stream));
    PG_CUDA(ctx, cudaMemcpyAsync(b->h_stats.get(), b->d_stats.get(), L * S * K * 32, cudaMemcpyDeviceToHost, b->stream));
    return PG_OK;
}

int pg_batch_sync(pg_batch *b) {
    if (!b) return PG_ERR_ARG;
    PG_CUDA(b->scan->ctx, cudaStreamSynchronize(b->stream));
    return PG_OK;
}

int pg_batch_results(pg_batch *b, pg_results *out) {
    if (!b || !out) return PG_ERR_ARG;
    if (b->n_loci > 0 && !(b->h_meta.get() && b->h_fmean.get() && b->h_stats.get())) return fail(b->scan->ctx, PG_ERR_STATE, "pg_batch_results before pg_batch_download");
    out->n_loci = b->n_loci;
    out->n_slots = b->scan->n_slots;
    out->n_phen = b->scan->k;
    out->meta = b->h_meta.get();
    out->freq_mean = b->h_fmean.get();
    out->stats = b->h_stats.get();
    return PG_OK;
}

// ---- streaming ------------------------------------------------------------------------------
int pg_scan_stream_begin(pg_scan *s, int64_t max_loci) {
    if (!s || max_loci < 1) return PG_ERR_ARG;
    for (int i = 0; i < PG_STREAM_DEPTH; i++) {
        delete s->slabs[i];
        s->slabs[i] = nullptr;
        int rc = pg_batch_create(s, max_loci, &s->slabs[i]);
        if (rc) return rc;
    }
    s->slab_cap = max_loci;
    s->next_slab = 0;
    return PG_OK;
}

static int submit_common(pg_scan *s, int *ticket, pg_batch **b) {
    if (!s || !ticket) return PG_ERR_ARG;
    if (!s->slabs[0]) return fail(s->ctx, PG_ERR_STATE, "pg_scan_submit before pg_scan_stream_begin");
    *ticket = s->next_slab;
    *b = s->slabs[s->next_slab];
    s->next_slab = (s->next_slab + 1) % PG_STREAM_DEPTH;
    return pg_batch_sync(*b);  // the slab's previous results must have been collected by now
}

int pg_scan_submit_counts(pg_scan *s, const uint32_t *counts, int64_t n_loci, int *ticket) {
    pg_batch *b = nullptr;
    int rc = submit_common(s, ticket, &b);
    if (rc) return rc;
    if ((rc = pg_batch_upload_counts(b, counts, n_loci))) return rc;
    if ((rc = pg_batch_run(b))) return rc;
    return pg_batch_download(b);
}
int pg_scan_submit_counts_u16(pg_scan *s, const uint16_t *counts, int64_t n_loci, int *ticket) {
    pg_batch *b = nullptr;
    int rc = submit_common(s, ticket, &b);
    if (rc) return rc;
    if ((rc = pg_batch_upload_counts_u16(b, counts, n_loci))) return rc;
    if ((rc = pg_batch_run(b))) return rc;
    return pg_batch_download(b);
}
int pg_scan_submit_counts_u8(pg_scan *s, const uint8_t *counts, int64_t n_loci, int *ticket) {
    pg_batch *b = nullptr;
    int rc = submit_common(s, ticket, &b);
    if (rc) return rc;
    if ((rc = pg_batch_upload_counts_u8(b, counts, n_loci))) return rc;
    if ((rc = pg_batch_run(b))) return rc;
    return pg_batch_download(b);
}
int pg_scan_submit_freq(pg_scan *s, const double *freq, const uint32_t *depth, int64_t n_loci, int *ticket) {
    pg_batch *b = nullptr;
    int rc = submit_common(s, ticket, &b);
    if (rc) return rc;
    if ((rc = pg_batch_upload_freq(b, freq, depth, n_loci))) return rc;
    if ((rc = pg_batch_run(b))) return rc;
    return pg_batch_download(b);
}
// a slab submitted as text whose parse has been enqueued but whose scan has not: finish it (stage B, scan, download)
static int finish_text_slab(pg_scan *s, int slab, int64_t *n_loci) {
    pg_batch *b = s->slabs[slab];
    if (!b || !b->text.pending) return PG_OK;
    int rc = text_stage_b(b, n_loci);
    if (rc) return rc;
    if ((rc = pg_batch_run(b))) return rc;
    return pg_batch_download(b);
}
int pg_scan_submit_sync_text(pg_scan *s, const char *text, size_t n_bytes, int *ticket, int64_t *n_loci) {
    pg_batch *b = nullptr;
    int rc = submit_common(s, ticket, &b);
    if (rc) return rc;
    // the copy + parse of this slab is enqueued BEFORE the host waits for the previous slab's parse, so the copy
    // engine never idles; the previous slab's scan is launched as soon as its locus count is known
    if ((rc = text_stage_a(b, text, n_bytes, 0))) return rc;
    for (int i = 1; i < PG_STREAM_DEPTH; i++) {
        const int prev = (*ticket + i) % PG_STREAM_DEPTH;  // oldest first
        if ((rc = finish_text_slab(s, prev, nullptr))) return rc;
    }
    if (n_loci) return finish_text_slab(s, *ticket, n_loci);  // the caller wants the count now: no deferral
    return PG_OK;
}
int pg_scan_text_labels(pg_scan *s, int ticket, const uint64_t **line_offsets, const uint64_t **positions) {
    if (!s || ticket < 0 || ticket >= PG_STREAM_DEPTH || !s->slabs[ticket]) return PG_ERR_ARG;
    return pg_batch_text_labels(s->slabs[ticket], line_offsets, positions);
}
int pg_scan_collect(pg_scan *s, int ticket, pg_results *out) {
    if (!s || ticket < 0 || ticket >= PG_STREAM_DEPTH || !s->slabs[ticket]) return PG_ERR_ARG;
    int rc = finish_text_slab(s, ticket, nullptr);
    if (rc) return rc;
    rc = pg_batch_sync(s->slabs[ticket]);
    if (rc) return rc;
    return pg_batch_results(s->slabs[ticket], out);
}

}  // extern "C"
