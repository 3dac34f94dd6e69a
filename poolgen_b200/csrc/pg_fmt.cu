// pg_fmt.cu -- sync2csv rows formatted on the device (SaveCsv::write_csv, src/base/sync.rs:1243-1260): the allele
// columns a pg_kin took from its last sync text append become `chr,pos,allele,f_1,...,f_n\n` rows, byte for byte
// those of pg_format_frequency_rows (pg_writer.cpp) with locus_order = NULL.
//   fmt_length_kernel  one warp per column, lanes over the pools: the byte count of its row (and whether a value falls
//                      outside what the device prints)
//   cub exclusive scan the row offsets; fmt_fit_kernel finds the last whole row that fits the caller's capacity
//   fmt_write_kernel   one warp per row: each lane forms its numbers' text, a warp scan of their lengths places them in
//                      a shared-memory staging area, which leaves in 16-byte stores (bytewise at the row's two ends,
//                      whose 16-byte granules a neighbouring row shares)
// A frequency goes through parse_f64_roundup_and_own(x, 6) (src/base/helpers.rs:111-117) as Rounder(6).put prints
// it: k = round(x * 1e6), one IEEE multiply (no FMA) and round-half-away; NaN prints "NaN", k = 0 prints "0" or "-0",
// any other k the decimal k / 10^6 with its trailing zeros trimmed.  |x * 1e6| >= 9e14 and infinities need the
// shortest-digit printer of the host; the loader's frequencies never get there, and such a column is refused.
#include <cub/device/device_scan.cuh>
#include <math.h>

#include "pg_device.cuh"
#include "pg_internal.h"
#include "pg_kin.h"

namespace pg {

constexpr int kFmtThreads = 256;
constexpr int kFmtWarps = kFmtThreads / 32;
constexpr int kFmtStage = 2048;   // staging bytes per warp
constexpr int kFmtRound = 32 * 19; // the most bytes one round of 32 numbers adds: ",-" + 9 + "." + 6 digits each
constexpr int kFmtPiece = 512;     // chromosome bytes staged at a time

struct FmtParams {
    const double *G;              // first column of the range, [column][ldg]
    int ldg, n;
    const int64_t *col_locus;     // first column of the range
    const uint8_t *col_allele;
    const char *text;             // the parsed sync text (device)
    const uint64_t *line_offset;  // [locus]
    const uint64_t *pos;          // [locus]
    int64_t rows;
    uint64_t *off;                // [rows + 1] row lengths, then their exclusive scan
    uint32_t *chr_len;            // [rows]
    unsigned long long *info;     // [0] rows that fit, [1] their bytes, [2] unsupported value seen, [3] bytes of row 0
    char *out;
};

// one frequency: kind 0 NaN, 1 zero, 2 number ip.fp (fp trimmed to fd digits), 3 outside the device's range
struct FmtNum {
    int kind, neg, fd;
    uint32_t ip, fp;
};

__device__ __forceinline__ FmtNum fmt_num(double x) {
    FmtNum r;
    r.neg = 0;
    r.fd = 0;
    r.ip = r.fp = 0;
    const double y = __dmul_rn(x, 1.0e6);
    if (!(fabs(y) < 9.0e14)) {
        r.kind = (y != y) ? 0 : 3;
        return r;
    }
    const double kd = round(y);  // half away from zero, like std::round
    if (kd == 0.0) {
        r.kind = 1;
        r.neg = signbit(kd) ? 1 : 0;
        return r;
    }
    r.kind = 2;
    r.neg = kd < 0.0;
    const uint64_t k = (uint64_t)fabs(kd);
    r.ip = (uint32_t)(k / 1000000u);  // < 9e8
    uint32_t fp = (uint32_t)(k % 1000000u);
    int fd = 6;
    if (fp)
        while (fp % 10u == 0u) {
            fp /= 10u;
            fd--;
        }
    r.fp = fp;
    r.fd = fp ? fd : 0;
    return r;
}

__device__ __forceinline__ int dec_digits(uint64_t v) {
    int d = 1;
    while (v >= 10u) {
        v /= 10u;
        d++;
    }
    return d;
}

// bytes of ",<number>"
__device__ __forceinline__ int fmt_len(const FmtNum &v) {
    if (v.kind == 0) return 4;
    if (v.kind == 1) return 2 + v.neg;
    return 1 + v.neg + dec_digits(v.ip) + (v.fp ? 1 + v.fd : 0);
}

// ",<number>" ending just before e
__device__ __forceinline__ void fmt_put(const FmtNum &v, char *e) {
    char *p = e;
    if (v.kind == 0) {
        *--p = 'N';
        *--p = 'a';
        *--p = 'N';
    } else if (v.kind == 1) {
        *--p = '0';
        if (v.neg) *--p = '-';
    } else {
        uint32_t fp = v.fp, ip = v.ip;
        if (fp) {
            for (int j = 0; j < v.fd; j++) {
                *--p = (char)('0' + fp % 10u);
                fp /= 10u;
            }
            *--p = '.';
        }
        do {
            *--p = (char)('0' + ip % 10u);
            ip /= 10u;
        } while (ip);
        if (v.neg) *--p = '-';
    }
    *--p = ',';
}

// bytes of the chromosome name: the line up to its first tab (a locus line has one), 32 bytes per step
__device__ __forceinline__ uint32_t chr_bytes(const char *s, int lane) {
    for (uint32_t at = 0;; at += 32) {
        const unsigned m = __ballot_sync(PG_FULL_MASK, s[at + lane] == '\t');
        if (m) return at + (uint32_t)(__ffs(m) - 1);
    }
}

__global__ void __launch_bounds__(kFmtThreads) fmt_length_kernel(const FmtParams p) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t r = warp; r < p.rows; r += nwarps) {
        const double *g = p.G + (size_t)r * p.ldg;
        uint32_t len = 0;
        bool bad = false;
        for (int i = lane; i < p.n; i += 32) {
            const FmtNum v = fmt_num(g[i]);
            bad |= v.kind == 3;
            len += (uint32_t)fmt_len(v);
        }
        len = __reduce_add_sync(PG_FULL_MASK, len);
        if (__any_sync(PG_FULL_MASK, bad) && lane == 0) atomicOr(p.info + 2, 1ull);
        const int64_t l = p.col_locus[r];
        const uint32_t cn = chr_bytes(p.text + p.line_offset[l], lane);
        if (lane == 0) {
            p.chr_len[r] = cn;
            // chr "," pos "," allele <numbers> "\n"
            p.off[r] = (uint64_t)cn + 1 + (uint64_t)dec_digits(p.pos[l]) + 2 + len + 1;
        }
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) p.off[p.rows] = 0;
}

// the largest r with off[r] <= capacity (rows have at least one byte: off is strictly increasing)
__global__ void fmt_fit_kernel(const FmtParams p, uint64_t capacity) {
    int64_t lo = 0, hi = p.rows;
    while (lo < hi) {
        const int64_t mid = (lo + hi + 1) >> 1;
        if (p.off[mid] <= capacity) lo = mid;
        else hi = mid - 1;
    }
    p.info[0] = (unsigned long long)lo;
    p.info[1] = p.off[lo];
    p.info[3] = p.off[1];
}

// writes stage[lead, upto) to out[gbase + ...]: whole 16-byte granules of the staging area with one store, the rest
// bytewise; `upto` is a multiple of 16 except for the last flush of a row
__device__ __forceinline__ void fmt_flush(const char *stage, int lead, int upto, char *out, uint64_t gbase, int lane) {
    for (int j = lane; j * 16 < upto; j += 32) {
        const int b0 = j * 16, b1 = min(b0 + 16, upto);
        if (b0 >= lead && b1 - b0 == 16) {
            *reinterpret_cast<uint4 *>(out + gbase + b0) = *reinterpret_cast<const uint4 *>(stage + b0);
        } else {
            for (int b = max(b0, lead); b < b1; b++) out[gbase + b] = stage[b];
        }
    }
    __syncwarp();
}

__global__ void __launch_bounds__(kFmtThreads) fmt_write_kernel(const FmtParams p, int64_t rows) {
    __shared__ __align__(16) char stage_all[kFmtWarps][kFmtStage];
    const int lane = threadIdx.x & 31;
    char *stage = stage_all[threadIdx.x >> 5];
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t r = warp; r < rows; r += nwarps) {
        // stage[s] is out[gbase + s]; gbase is 16-byte aligned, the row starts at stage[lead]
        const uint64_t row = p.off[r];
        uint64_t gbase = row & ~(uint64_t)15;
        int lead = (int)(row & 15), fill = lead;
        // keeps at least `need` bytes free: the whole granules leave, the partial one moves to the front
        auto make_room = [&](int need) {
            if (fill + need <= kFmtStage) return;
            const int upto = fill & ~15, rem = fill - upto;
            fmt_flush(stage, lead, upto, p.out, gbase, lane);
            const char c = lane < rem ? stage[upto + lane] : 0;
            __syncwarp();
            if (lane < rem) stage[lane] = c;
            __syncwarp();
            gbase += (uint64_t)upto;
            lead = upto ? 0 : lead;
            fill = rem;
        };
        const int64_t l = p.col_locus[r];
        const char *chr = p.text + p.line_offset[l];
        const uint32_t cn = p.chr_len[r];
        for (uint32_t s = 0; s < cn; s += kFmtPiece) {
            const int m = (int)min((uint32_t)kFmtPiece, cn - s);
            make_room(m);
            for (int b = lane; b < m; b += 32) stage[fill + b] = chr[s + b];
            __syncwarp();
            fill += m;
        }
        // ",pos,allele"
        make_room(24);
        {
            const uint64_t v = p.pos[l];
            const int d = dec_digits(v);
            if (lane == 0) {
                char *o = stage + fill;
                o[0] = ',';
                uint64_t x = v;
                for (int j = d; j >= 1; j--) {
                    o[j] = (char)('0' + x % 10u);
                    x /= 10u;
                }
                o[d + 1] = ',';
                const uint8_t a = p.col_allele[r];
                o[d + 2] = "ATCGND"[a < 6 ? a : 4];
            }
            __syncwarp();
            fill += d + 3;
        }
        const double *g = p.G + (size_t)r * p.ldg;
        for (int base = 0; base < p.n; base += 32) {
            const int i = base + lane;
            FmtNum v;
            int len = 0;
            if (i < p.n) {
                v = fmt_num(g[i]);
                len = fmt_len(v);
            }
            int incl = len;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int t = __shfl_up_sync(PG_FULL_MASK, incl, o);
                if (lane >= o) incl += t;
            }
            const int total = __shfl_sync(PG_FULL_MASK, incl, 31);
            make_room(kFmtRound);
            if (i < p.n) fmt_put(v, stage + fill + incl);
            __syncwarp();
            fill += total;
        }
        make_room(1);
        if (lane == 0) stage[fill] = '\n';
        __syncwarp();
        fill += 1;
        fmt_flush(stage, lead, fill, p.out, gbase, lane);
    }
}

}  // namespace pg

using pg::fail;

extern "C" {

int pg_kin_format_frequency_rows(pg_kin *h, int64_t first, int64_t count, char *out, size_t capacity, size_t *n_bytes,
                                 int64_t *n_rows) {
    if (!h) return PG_ERR_ARG;
    pg_ctx *ctx = h->ctx;
    if (n_bytes) *n_bytes = 0;
    if (n_rows) *n_rows = 0;
    if (h->text_cols < 0)
        return fail(ctx, PG_ERR_STATE, "pg_kin_format_frequency_rows: the last append was not pg_kin_append_sync_text");
    if (first < 0 || count < 0 || first + count > h->text_cols || (!out && capacity))
        return fail(ctx, PG_ERR_ARG, "pg_kin_format_frequency_rows: columns [%lld, %lld) of %lld", (long long)first,
                    (long long)(first + count), (long long)h->text_cols);
    if (count == 0) return PG_OK;
    PG_CUDA(ctx, cudaSetDevice(ctx->device));
    PG_CUDA(ctx, h->d_fmt_off.reserve((size_t)count + 1, h->stream));
    PG_CUDA(ctx, h->d_fmt_chr.reserve((size_t)count, h->stream));
    PG_CUDA(ctx, h->d_fmt_info.reserve(4, h->stream));
    PG_CUDA(ctx, h->h_fmt_info.reserve(4, h->stream));
    size_t tmp = 0;
    PG_CUDA(ctx, cub::DeviceScan::ExclusiveSum(nullptr, tmp, h->d_fmt_off.get(), h->d_fmt_off.get(), (int)(count + 1),
                                               h->stream));
    PG_CUDA(ctx, h->d_fmt_tmp.reserve(tmp, h->stream));
    PG_CUDA(ctx, cudaMemsetAsync(h->d_fmt_info.get(), 0, 4 * sizeof(unsigned long long), h->stream));
    pg::FmtParams fp;
    fp.G = h->d_G.get() + (size_t)(h->text_first + first) * h->ldg;
    fp.ldg = h->ldg;
    fp.n = h->n;
    fp.col_locus = h->d_col_locus.get() + first;
    fp.col_allele = h->d_col_allele.get() + first;
    fp.text = h->text.d_text.get();
    fp.line_offset = h->text.d_out_offset.get();
    fp.pos = h->text.d_out_pos.get();
    fp.rows = count;
    fp.off = h->d_fmt_off.get();
    fp.chr_len = h->d_fmt_chr.get();
    fp.info = h->d_fmt_info.get();
    fp.out = nullptr;
    const int grid = (int)std::min<int64_t>((count * 32 + pg::kFmtThreads - 1) / pg::kFmtThreads, (int64_t)ctx->sm_count * 8);
    pg::fmt_length_kernel<<<grid, pg::kFmtThreads, 0, h->stream>>>(fp);
    PG_CUDA(ctx, cudaGetLastError());
    tmp = h->d_fmt_tmp.capacity();
    PG_CUDA(ctx, cub::DeviceScan::ExclusiveSum(h->d_fmt_tmp.get(), tmp, h->d_fmt_off.get(), h->d_fmt_off.get(),
                                               (int)(count + 1), h->stream));
    pg::fmt_fit_kernel<<<1, 1, 0, h->stream>>>(fp, (uint64_t)capacity);
    PG_CUDA(ctx, cudaGetLastError());
    PG_CUDA(ctx, cudaMemcpyAsync(h->h_fmt_info.get(), h->d_fmt_info.get(), 4 * 8, cudaMemcpyDeviceToHost, h->stream));
    PG_CUDA(ctx, cudaStreamSynchronize(h->stream));
    const unsigned long long *info = h->h_fmt_info.get();
    if (info[2])
        return fail(ctx, PG_ERR_UNSUPPORTED, "pg_kin_format_frequency_rows: a value with |x * 1e6| >= 9e14 or infinite "
                                             "in columns [%lld, %lld) (the loader emits none; pg_format_frequency_rows "
                                             "prints it)", (long long)first, (long long)(first + count));
    const int64_t rows = (int64_t)info[0];
    const size_t bytes = (size_t)info[1];
    if (rows == 0)
        return fail(ctx, PG_ERR_ARG, "pg_kin_format_frequency_rows: capacity %zu below the %llu bytes of one row",
                    capacity, (unsigned long long)info[3]);
    PG_CUDA(ctx, h->d_fmt_text.reserve(bytes, h->stream));
    fp.out = h->d_fmt_text.get();
    const int wgrid = (int)std::min<int64_t>((rows * 32 + pg::kFmtThreads - 1) / pg::kFmtThreads, (int64_t)ctx->sm_count * 8);
    pg::fmt_write_kernel<<<wgrid, pg::kFmtThreads, 0, h->stream>>>(fp, rows);
    PG_CUDA(ctx, cudaGetLastError());
    PG_CUDA(ctx, cudaMemcpyAsync(out, h->d_fmt_text.get(), bytes, cudaMemcpyDeviceToHost, h->stream));
    PG_CUDA(ctx, cudaStreamSynchronize(h->stream));
    if (n_bytes) *n_bytes = bytes;
    if (n_rows) *n_rows = rows;
    return PG_OK;
}

}  // extern "C"
