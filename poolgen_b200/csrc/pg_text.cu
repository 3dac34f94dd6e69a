// pg_text.cu -- sync text on the fast path (SURVEY.md 8f rank 1): a line-aligned chunk of a sync file
// (chr \t pos \t ref \t A:T:C:G:N:D per pool ...) is copied to the device as it is and parsed there into the count slab
// the scan and the count tests consume.  Parse semantics are those of `impl Parse<LocusCounts> for String`
// (src/base/sync.rs:100-156) as driven by the chunk readers (src/base/sync.rs:827-868):
//   - a line that starts with '#' is skipped (ErrorKind::Other -> continue);
//   - a line whose second field is not an unsigned integer is skipped (same error kind);
//   - the number of pools is (tab-separated fields - 3) and must equal the scan's pool count (the reference would
//     trip the pool-size assert of the filter, src/base/sync.rs:254-257): reported as an error;
//   - every pool field holds at least six ':'-separated unsigned integers, the first six are A:T:C:G:N:D
//     (src/base/sync.rs:134-137, 144-150); anything else makes the reference panic (`expect`): reported as an error;
//   - a trailing '\r' before the newline is dropped (src/base/sync.rs:104-109);
//   - an empty line or a line with fewer than three fields makes the reference panic (index out of bounds,
//     src/base/sync.rs:112,121); such lines are skipped here.
// Pipeline, every step asynchronous on the batch's stream (all counts stay on the device, so the host never waits
// between the copy of the text and the parsed slab -- text_parse_async; text_parse_finish reads the outcome):
//   tokenizer   16 bytes per thread: tok_count_kernel counts tabs + newlines and newlines per 4 KB block, an exclusive
//               scan of the block counts, tok_scatter_kernel writes their positions in order;
//   lines       one thread per line classifies it (comment / position / pool count) and counts the locus lines of its
//               group of 256 lines; an exclusive scan over the groups numbers them;
//   fields      one warp per locus line parses the pool fields (lane = pool, stride 32) straight into
//               counts[locus][allele][pool].
#include <cub/device/device_scan.cuh>

#include "pg_device.cuh"
#include "pg_internal.h"

namespace pg {

enum { TEXT_OK = 0, TEXT_ERR_POOLS = 1, TEXT_ERR_FIELD = 2, TEXT_ERR_LINES = 3, TEXT_ERR_LOCI = 4 };

constexpr int kTokThreads = 256;
constexpr int kTokBytes = 16;                           // per thread: one 128-bit load
constexpr int kTokBlock = kTokThreads * kTokBytes;      // 4 KB of text per block
constexpr int kLineGroup = 256;                         // lines per numbering group

struct TextParams {
    const char *text;
    uint32_t n_bytes;
    uint32_t *sep;         // positions of '\t' and '\n', ascending
    uint32_t *nl;          // positions of '\n', ascending (line_cap entries)
    uint64_t *tok_blk;     // [n_tok_blocks + 1] per-block (n_sep << 32 | n_nl), then its exclusive scan
    uint32_t n_tok_blocks;
    uint32_t line_cap;     // lines the per-line arrays hold
    uint32_t max_loci;
    int n_pools;
    uint8_t *keep;         // [line_cap] 1 = a locus line
    uint32_t *first_sep;   // [line_cap] index into sep of the first separator of the line
    uint64_t *line_pos;    // [line_cap] parsed position
    uint32_t *grp;         // [line_cap / 256 + 2] locus lines per group of 256 lines, then its exclusive scan
    uint32_t n_groups_max;
    uint32_t *counts;      // [locus][6][n_pools]
    uint64_t *out_offset;  // [locus] byte offset of the line in the chunk
    uint64_t *out_pos;     // [locus]
    uint32_t *info;        // [0] n_loci, [1] error code, [2] byte offset of the error, [3] n_lines
};

__device__ __forceinline__ void text_error(const TextParams &p, uint32_t code, uint32_t at) {
    if (atomicCAS(p.info + 1, 0u, code) == 0u) p.info[2] = at;
}

// 16 bytes of text -> bit masks of (tab | newline) and of newline
__device__ __forceinline__ void tok_masks(const TextParams &p, uint32_t base, uint32_t &m_sep, uint32_t &m_nl) {
    m_sep = m_nl = 0;
    if (base >= p.n_bytes) return;
    const uint4 v = *reinterpret_cast<const uint4 *>(p.text + base);  // the buffer is padded to 16 bytes
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int i = 0; i < 16; i++) {
        const uint32_t c = (w[i >> 2] >> (8 * (i & 3))) & 0xffu;
        if (base + i < p.n_bytes) {
            m_nl |= (uint32_t)(c == '\n') << i;
            m_sep |= (uint32_t)((c == '\n') | (c == '\t')) << i;
        }
    }
}

__global__ void __launch_bounds__(kTokThreads) tok_count_kernel(const TextParams p) {
    __shared__ uint32_t ws[kTokThreads / 32];
    for (uint32_t blk = blockIdx.x; blk < p.n_tok_blocks; blk += gridDim.x) {
        uint32_t ms, mn;
        tok_masks(p, blk * kTokBlock + threadIdx.x * kTokBytes, ms, mn);
        uint32_t c = ((uint32_t)__popc(ms) << 16) | (uint32_t)__popc(mn);  // <= 4096 each per block: no carry
        c = __reduce_add_sync(PG_FULL_MASK, c);
        if ((threadIdx.x & 31) == 0) ws[threadIdx.x >> 5] = c;
        __syncthreads();
        if (threadIdx.x == 0) {
            uint32_t t = 0;
#pragma unroll
            for (int i = 0; i < kTokThreads / 32; i++) t += ws[i];
            p.tok_blk[blk] = ((uint64_t)(t >> 16) << 32) | (uint64_t)(t & 0xffffu);
        }
        __syncthreads();
    }
}

__global__ void __launch_bounds__(kTokThreads) tok_scatter_kernel(const TextParams p) {
    __shared__ uint32_t ws[kTokThreads / 32];
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        const uint64_t tot = p.tok_blk[p.n_tok_blocks];
        const uint32_t n_lines = (uint32_t)(tot & 0xffffffffu);
        p.info[3] = n_lines;
        if (n_lines > p.line_cap) text_error(p, TEXT_ERR_LINES, n_lines);
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (uint32_t blk = blockIdx.x; blk < p.n_tok_blocks; blk += gridDim.x) {
        const uint32_t base = blk * kTokBlock + threadIdx.x * kTokBytes;
        uint32_t ms, mn;
        tok_masks(p, base, ms, mn);
        const uint32_t c = ((uint32_t)__popc(ms) << 16) | (uint32_t)__popc(mn);
        uint32_t incl = c;  // inclusive scan within the warp, both halves at once
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            const uint32_t v = __shfl_up_sync(PG_FULL_MASK, incl, off);
            if (lane >= off) incl += v;
        }
        if (lane == 31) ws[warp] = incl;
        __syncthreads();
        uint32_t before = 0;
#pragma unroll
        for (int i = 0; i < kTokThreads / 32; i++)
            if (i < warp) before += ws[i];
        __syncthreads();
        const uint32_t excl = before + incl - c;
        const uint64_t off = p.tok_blk[blk];
        uint32_t o_sep = (uint32_t)(off >> 32) + (excl >> 16), o_nl = (uint32_t)(off & 0xffffffffu) + (excl & 0xffffu);
        while (ms) {
            const int b = __ffs(ms) - 1;
            ms &= ms - 1;
            p.sep[o_sep++] = base + b;
        }
        while (mn) {
            const int b = __ffs(mn) - 1;
            mn &= mn - 1;
            if (o_nl < p.line_cap) p.nl[o_nl] = base + b;
            o_nl++;
        }
    }
}

// one thread per line: comment / position / field count; a group of 256 lines leaves its number of locus lines
__global__ void __launch_bounds__(kLineGroup) text_lines_kernel(const TextParams p) {
    const uint32_t n_lines = min(p.info[3], p.line_cap);
    const uint32_t n_sep = (uint32_t)(p.tok_blk[p.n_tok_blocks] >> 32);
    const uint32_t n_groups = (n_lines + kLineGroup - 1) / kLineGroup;
    for (uint32_t g = blockIdx.x; g < n_groups; g += gridDim.x) {
        const uint32_t l = g * kLineGroup + threadIdx.x;
        uint32_t keep = 0;
        if (l < n_lines) {
            const uint32_t start = l ? p.nl[l - 1] + 1 : 0u, end = p.nl[l];  // [start, end) without the newline
            // rank of this line's newline among the separators (binary search); the line's tabs are the ones before
            uint32_t lo = 0, hi = n_sep;
            while (lo < hi) {
                const uint32_t mid = (lo + hi) >> 1;
                if (p.sep[mid] < end) lo = mid + 1; else hi = mid;
            }
            const uint32_t nl_rank = lo;
            uint32_t lo2 = 0, hi2 = nl_rank;
            while (lo2 < hi2) {
                const uint32_t mid = (lo2 + hi2) >> 1;
                if (p.sep[mid] < start) lo2 = mid + 1; else hi2 = mid;
            }
            const uint32_t first = lo2;            // first tab of the line
            const uint32_t n_tabs = nl_rank - first;
            p.first_sep[l] = first;
            if (end > start && p.text[start] != '#' && n_tabs >= 2) {
                // position = second field, `parse::<u64>()`: optional '+', then digits only
                uint32_t a = p.sep[first] + 1, b = p.sep[first + 1];
                if (a < b && p.text[a] == '+') a++;
                bool ok = a < b;
                uint64_t v = 0;
                for (uint32_t i = a; i < b && ok; i++) {
                    const unsigned d = (unsigned)(p.text[i] - '0');
                    if (d > 9u || v > (0xFFFFFFFFFFFFFFFFull - d) / 10ull) ok = false;
                    v = v * 10ull + d;
                }
                if (ok) {
                    keep = 1;
                    p.line_pos[l] = v;
                    if ((int)n_tabs != p.n_pools + 2) text_error(p, TEXT_ERR_POOLS, start);
                }
            }
            p.keep[l] = (uint8_t)keep;
        }
        const int c = __syncthreads_count((int)keep);
        if (threadIdx.x == 0) p.grp[g] = (uint32_t)c;
    }
}

// one warp per locus line: lane = pool (stride 32), six ':'-separated unsigned integers per pool field
__global__ void __launch_bounds__(256) text_parse_kernel(const TextParams p) {
    const int lane = threadIdx.x & 31;
    const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = (gridDim.x * blockDim.x) >> 5;
    const int n = p.n_pools;
    const uint32_t n_lines = min(p.info[3], p.line_cap);
    const uint32_t n_loci = p.grp[p.n_groups_max];
    if (warp == 0 && lane == 0) {
        p.info[0] = n_loci;
        if (n_loci > p.max_loci) text_error(p, TEXT_ERR_LOCI, n_loci);
    }
    for (uint32_t l = warp; l < n_lines; l += nwarps) {
        if (!p.keep[l]) continue;
        // ordinal = locus lines of the earlier groups + locus lines before this one in its group
        const uint32_t g0 = l & ~(uint32_t)(kLineGroup - 1);
        uint32_t before = 0;
        for (uint32_t j = g0 + lane; j < l; j += 32) before += p.keep[j];
        const uint32_t ord = p.grp[l / kLineGroup] + __reduce_add_sync(PG_FULL_MASK, before);
        if (ord >= p.max_loci) continue;
        const uint32_t start = l ? p.nl[l - 1] + 1 : 0u;
        const uint32_t first = p.first_sep[l];
        if (lane == 0) {
            p.out_offset[ord] = start;
            p.out_pos[ord] = p.line_pos[l];
        }
        // a line with the wrong number of fields was reported by text_lines_kernel: parse only what exists
        const uint32_t end_rank = (l + 1 < n_lines) ? p.first_sep[l + 1] : (uint32_t)(p.tok_blk[p.n_tok_blocks] >> 32);
        uint32_t *out = p.counts + (size_t)ord * 6 * n;
        for (int i = lane; i < n; i += 32) {
            if (first + 3 + i >= end_rank) break;
            uint32_t a = p.sep[first + 2 + i] + 1, b = p.sep[first + 3 + i];
            if (b > a && p.text[b - 1] == '\r') b--;  // Windows line end on the last pool field
            int j = 0;
            uint64_t v = 0;
            bool digits = false, bad = false, plus = false;
            for (uint32_t q = a; q <= b; q++) {
                const char c = (q < b) ? p.text[q] : ':';
                if (c == ':') {
                    if (!digits) bad = true;
                    if (j < 6) out[(size_t)j * n + i] = v > 0xFFFFFFFFull ? 0xFFFFFFFFu : (uint32_t)v;
                    j++;
                    v = 0;
                    digits = false;
                    plus = false;
                } else if (c == '+' && !digits && !plus) {
                    plus = true;  // `parse::<u64>()` accepts one leading '+'
                } else {
                    const unsigned d = (unsigned)(c - '0');
                    if (d > 9u) bad = true;
                    v = v * 10ull + d;
                    if (v > 0xFFFFFFFFFFFFull) v = 0xFFFFFFFFFFFFull;
                    digits = true;
                }
            }
            if (bad || j < 6) text_error(p, TEXT_ERR_FIELD, a);
        }
    }
}

TextScratch::~TextScratch() {
    if (parsed) cudaEventDestroy(parsed);
}

// capacity with headroom: consecutive chunks of a file differ by a few lines, and a reallocation (cudaFree
// synchronises the device) in the middle of the stream costs more than the memory
static size_t with_headroom(size_t need) { return need + need / 8 + 65536; }

#define TCK(call)                      \
    do {                               \
        cudaError_t e_ = (call);       \
        if (e_ != cudaSuccess) return e_; \
    } while (0)

// Enqueues copy + parse of `text` (host; pinned for a truly asynchronous copy; n_bytes, ends with '\n' or at a line
// end) into counts[locus][6][n_pools] (device, capacity max_loci) on stream s and records the `parsed` event.  The
// per-line arrays hold line_cap lines (0 = a default bound from max_loci); text_parse_finish reports when a chunk has
// more (comment / blank lines) so that the caller can repeat with the exact bound.
static cudaError_t text_parse_enqueue(TextScratch *t, const char *text, size_t n_bytes, int n_pools, uint32_t *d_counts,
                                      int64_t max_loci, size_t line_cap, int sm_count, cudaStream_t s) {
    t->max_loci = max_loci;
    if (!t->parsed) TCK(cudaEventCreateWithFlags(&t->parsed, cudaEventDisableTiming));
    TCK(t->d_info.reserve(4, s));
    TCK(t->h_info.reserve(4, s));
    TCK(cudaMemsetAsync(t->d_info.get(), 0, 16, s));
    if (n_bytes >= 0xFFFFFFF0ull) return cudaErrorInvalidValue;
    if (n_bytes == 0) {
        TCK(cudaMemcpyAsync(t->h_info.get(), t->d_info.get(), 16, cudaMemcpyDeviceToHost, s));
        return cudaEventRecord(t->parsed, s);
    }
    const bool add_nl = text[n_bytes - 1] != '\n';  // a last line without its newline
    const size_t nb = n_bytes + (add_nl ? 1 : 0);
    if (line_cap == 0) line_cap = (size_t)max_loci + (size_t)max_loci / 4 + 4096;
    if (line_cap > nb) line_cap = nb;
    if (t->d_text.capacity() < nb + 32) TCK(t->d_text.reserve(with_headroom(nb + 32), s));
    TCK(cudaMemcpyAsync(t->d_text.get(), text, n_bytes, cudaMemcpyHostToDevice, s));
    if (add_nl) TCK(cudaMemsetAsync(t->d_text.get() + n_bytes, '\n', 1, s));
    const size_t n_tok = (nb + kTokBlock - 1) / kTokBlock;
    const size_t n_grp = (line_cap + kLineGroup - 1) / kLineGroup;
    if (t->d_sep.capacity() < nb) TCK(t->d_sep.reserve(with_headroom(nb), s));  // worst case: every byte is a separator
    if (t->d_tok_blk.capacity() < n_tok + 1) TCK(t->d_tok_blk.reserve(with_headroom(n_tok + 1), s));
    // the per-line arrays are sized for exactly line_cap lines
    TCK(t->d_nl.reserve(line_cap, s));
    TCK(t->d_keep.reserve(line_cap, s));
    TCK(t->d_first.reserve(line_cap, s));
    TCK(t->d_line_pos.reserve(line_cap, s));
    TCK(t->d_grp.reserve(n_grp + 2, s));
    TCK(t->d_out_offset.reserve((size_t)max_loci, s));
    TCK(t->d_out_pos.reserve((size_t)max_loci, s));
    TCK(t->h_out_offset.reserve((size_t)max_loci, s));
    TCK(t->h_out_pos.reserve((size_t)max_loci, s));
    size_t tmp1 = 0, tmp2 = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, tmp1, (uint64_t *)nullptr, (uint64_t *)nullptr, (int)(n_tok + 1), s);
    cub::DeviceScan::ExclusiveSum(nullptr, tmp2, (uint32_t *)nullptr, (uint32_t *)nullptr, (int)(n_grp + 1), s);
    TCK(t->d_tmp.reserve(std::max(tmp1, tmp2), s));
    TextParams tp;
    tp.text = t->d_text.get();
    tp.n_bytes = (uint32_t)nb;
    tp.sep = t->d_sep.get();
    tp.nl = t->d_nl.get();
    tp.tok_blk = t->d_tok_blk.get();
    tp.n_tok_blocks = (uint32_t)n_tok;
    tp.line_cap = (uint32_t)line_cap;
    tp.max_loci = (uint32_t)std::min<int64_t>(max_loci, 0xFFFFFFFFll);
    tp.n_pools = n_pools;
    tp.keep = t->d_keep.get();
    tp.first_sep = t->d_first.get();
    tp.line_pos = t->d_line_pos.get();
    tp.grp = t->d_grp.get();
    tp.n_groups_max = (uint32_t)n_grp;
    tp.counts = d_counts;
    tp.out_offset = t->d_out_offset.get();
    tp.out_pos = t->d_out_pos.get();
    tp.info = t->d_info.get();
    const int grid_tok = (int)std::min<size_t>(n_tok, (size_t)sm_count * 16);
    TCK(cudaMemsetAsync(t->d_tok_blk.get() + n_tok, 0, 8, s));
    tok_count_kernel<<<grid_tok, kTokThreads, 0, s>>>(tp);
    TCK(cudaGetLastError());
    size_t tb = t->d_tmp.capacity();
    TCK(cub::DeviceScan::ExclusiveSum(t->d_tmp.get(), tb, t->d_tok_blk.get(), t->d_tok_blk.get(), (int)(n_tok + 1), s));
    tok_scatter_kernel<<<grid_tok, kTokThreads, 0, s>>>(tp);
    TCK(cudaGetLastError());
    TCK(cudaMemsetAsync(t->d_grp.get(), 0, (n_grp + 2) * 4, s));
    const int grid_lines = (int)std::min<size_t>(n_grp, (size_t)sm_count * 8);
    text_lines_kernel<<<grid_lines, kLineGroup, 0, s>>>(tp);
    TCK(cudaGetLastError());
    tb = t->d_tmp.capacity();
    TCK(cub::DeviceScan::ExclusiveSum(t->d_tmp.get(), tb, t->d_grp.get(), t->d_grp.get(), (int)(n_grp + 1), s));
    const int grid_parse = (int)std::min<uint64_t>(((uint64_t)line_cap * 32 + 255) / 256, (uint64_t)sm_count * 8);
    text_parse_kernel<<<grid_parse, 256, 0, s>>>(tp);
    TCK(cudaGetLastError());
    TCK(cudaMemcpyAsync(t->h_info.get(), t->d_info.get(), 16, cudaMemcpyDeviceToHost, s));
    return cudaEventRecord(t->parsed, s);
}
#undef TCK

// a slab is 'pending' only once everything up to the `parsed` event has been enqueued: a failed allocation or launch
// must not leave text_parse_finish waiting on a stale event and trusting the previous chunk's h_info
cudaError_t text_parse_async(TextScratch *t, const char *text, size_t n_bytes, int n_pools, uint32_t *d_counts,
                             int64_t max_loci, size_t line_cap, int sm_count, cudaStream_t s) {
    t->pending = false;
    const cudaError_t e = text_parse_enqueue(t, text, n_bytes, n_pools, d_counts, max_loci, line_cap, sm_count, s);
    t->pending = (e == cudaSuccess);
    return e;
}

// Waits for the parse and returns the number of loci, or a negative code: -1 CUDA error (*cuda_err), -2 more loci than
// capacity, -3 pool count mismatch, -4 malformed pool field (*err_offset = byte offset in the chunk), -5 more lines
// than the per-line arrays hold (*err_offset = the number of lines: repeat with that line_cap).  On success the copy
// of the labels (line offsets, positions) to pinned host memory is enqueued on s.
int64_t text_parse_finish(TextScratch *t, cudaStream_t s, cudaError_t *cuda_err, uint64_t *err_offset) {
    if (!t->pending) return 0;
    t->pending = false;
    cudaError_t e = cudaEventSynchronize(t->parsed);
    if (e != cudaSuccess) {
        *cuda_err = e;
        return -1;
    }
    const uint32_t *info = t->h_info.get();
    const uint32_t n_loci = info[0], code = info[1];
    *err_offset = info[2];
    if (code == TEXT_ERR_LINES) return -5;
    if (code == TEXT_ERR_POOLS) return -3;
    if (code == TEXT_ERR_FIELD) return -4;
    if (code == TEXT_ERR_LOCI || (int64_t)n_loci > t->max_loci) return -2;
    if (n_loci == 0) return 0;
    e = cudaMemcpyAsync(t->h_out_offset.get(), t->d_out_offset.get(), (size_t)n_loci * 8, cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess)
        e = cudaMemcpyAsync(t->h_out_pos.get(), t->d_out_pos.get(), (size_t)n_loci * 8, cudaMemcpyDeviceToHost, s);
    if (e != cudaSuccess) {
        *cuda_err = e;
        return -1;
    }
    return (int64_t)n_loci;
}

int text_parse_fail(pg_ctx *ctx, const char *who, int64_t status, cudaError_t cuda_err, uint64_t err_offset,
                    int n_pools, int64_t cap) {
    const unsigned long long at = err_offset;
    if (status == -1) return fail(ctx, PG_ERR_CUDA, "%s: %s", who, cudaGetErrorString(cuda_err));
    if (status == -2) return fail(ctx, PG_ERR_ARG, "%s: more loci in the chunk than the capacity %lld", who, (long long)cap);
    if (status == -3)
        return fail(ctx, PG_ERR_ARG, "%s: the line at byte %llu does not hold %d pools (the reference asserts the pool count, "
                                     "src/base/sync.rs:254-257)", who, at, n_pools);
    if (status == -4)
        return fail(ctx, PG_ERR_ARG, "%s: malformed pool field at byte %llu (the reference panics: allele counts are not "
                                     "valid integers, src/base/sync.rs:146)", who, at);
    return fail(ctx, PG_ERR_ARG, "%s: the chunk could not be parsed (%lld)", who, (long long)status);
}

}  // namespace pg
