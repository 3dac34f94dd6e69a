// pg_comm.cu -- the multi-GPU side of the C ABI (SURVEY.md 8b / 8e).
//
// The reference runs `ols_with_covariate` in ONE process (src/main.rs:280-298): the kinship matrix is
// `g.dot(&g.t())` over all allele columns (src/gwas/ols.rs:295).  With the columns sharded over the GPUs of a box
// that product is a sum over the shards, i.e. the path's one exchange step: an all-reduce of the n x n partial Gram
// matrices.  This file puts that step behind the C ABI: the NCCL communicator is created by the library
// (ncclCommInitAll for one process driving n GPUs, ncclCommInitRank for one process per GPU), the all-reduce runs on
// the kinship handles' own streams straight on their device buffers, and the column counts are summed in the same
// NCCL group.  The scans themselves need no collective: pg_shard_range gives the contiguous ranges (rank order = file
// order, like the reference's contiguous byte ranges, src/base/helpers.rs:74-91).
//
// NCCL is loaded on first use (dlopen, like cuSOLVER in pg_kinship.cu): a process that only scans never maps it, and a
// process that already holds a libnccl.so.2 (e.g. one that imported torch) shares that copy.
#include <dlfcn.h>
#include <nccl.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <new>
#include <vector>

#include "pg_kin.h"

namespace {

struct NcclApi {
    ncclResult_t (*get_version)(int *) = nullptr;
    ncclResult_t (*get_unique_id)(ncclUniqueId *) = nullptr;
    ncclResult_t (*comm_init_rank)(ncclComm_t *, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*comm_init_all)(ncclComm_t *, int, const int *) = nullptr;
    ncclResult_t (*comm_destroy)(ncclComm_t) = nullptr;
    ncclResult_t (*all_reduce)(const void *, void *, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*group_start)() = nullptr;
    ncclResult_t (*group_end)() = nullptr;
    const char *(*error_string)(ncclResult_t) = nullptr;
    bool ok = false;
    const char *why = "";
};

const NcclApi &nccl_api() {
    static const NcclApi api = [] {
        NcclApi a;
        // PG_NCCL_LIB names the library file explicitly.  A process that will ALSO load another component linked against
        // a newer libnccl.so.2 (e.g. a Python process importing torch with its bundled NCCL) must point it at that same
        // file: the dynamic loader keeps one object per SONAME, and whichever copy is mapped first serves both.
        void *lib = nullptr;
        if (const char *forced = getenv("PG_NCCL_LIB")) lib = dlopen(forced, RTLD_NOW | RTLD_LOCAL);
        if (!lib)
            for (const char *name : {"libnccl.so.2", "libnccl.so", "/usr/lib/x86_64-linux-gnu/libnccl.so.2"}) {
                lib = dlopen(name, RTLD_NOW | RTLD_LOCAL);
                if (lib) break;
            }
        if (!lib) {
            a.why = "libnccl.so.2 could not be loaded";
            return a;
        }
#define PG_SYM(field, name) a.field = reinterpret_cast<decltype(a.field)>(dlsym(lib, name))
        PG_SYM(get_version, "ncclGetVersion");
        PG_SYM(get_unique_id, "ncclGetUniqueId");
        PG_SYM(comm_init_rank, "ncclCommInitRank");
        PG_SYM(comm_init_all, "ncclCommInitAll");
        PG_SYM(comm_destroy, "ncclCommDestroy");
        PG_SYM(all_reduce, "ncclAllReduce");
        PG_SYM(group_start, "ncclGroupStart");
        PG_SYM(group_end, "ncclGroupEnd");
        PG_SYM(error_string, "ncclGetErrorString");
#undef PG_SYM
        a.ok = a.get_version && a.get_unique_id && a.comm_init_rank && a.comm_init_all && a.comm_destroy &&
               a.all_reduce && a.group_start && a.group_end && a.error_string;
        if (!a.ok) a.why = "libnccl.so.2 lacks a required symbol";
        return a;
    }();
    return api;
}
}  // namespace

using pg::fail;

static_assert(sizeof(ncclUniqueId) == PG_COMM_ID_BYTES, "PG_COMM_ID_BYTES must equal sizeof(ncclUniqueId)");

struct pg_comm {
    int world = 0;       // ranks of the communicator
    int n_local = 0;     // ranks this process drives
    int first_rank = 0;  // rank of local index 0 (local ranks are consecutive)
    std::vector<ncclComm_t> comms;
    std::vector<pg_ctx *> ctxs;
    // one int64 per local rank on its device and pinned on the host: the column counts summed with the matrices
    std::vector<pg::DeviceBuffer<int64_t>> d_count;
    std::vector<pg::PinnedBuffer<int64_t>> h_count;
    ~pg_comm();
};

// each local rank's counter is freed, and its communicator destroyed, with that rank's device current
pg_comm::~pg_comm() {
    const NcclApi &nccl = nccl_api();
    for (int i = 0; i < n_local; i++) {
        if (i < (int)ctxs.size() && ctxs[i]) cudaSetDevice(ctxs[i]->device);
        if (i < (int)d_count.size()) d_count[i] = {};
        if (i < (int)h_count.size()) h_count[i] = {};
        if (nccl.ok && i < (int)comms.size() && comms[i]) nccl.comm_destroy(comms[i]);
    }
}

#define CNCCL(ctx, call)                                                                                     \
    do {                                                                                                     \
        ncclResult_t r_ = (call);                                                                            \
        if (r_ != ncclSuccess)                                                                               \
            return fail((ctx), PG_ERR_NCCL, "%s failed: %s (%s:%d)", #call, nccl.error_string(r_), __FILE__, __LINE__); \
    } while (0)

static int comm_alloc_counters(pg_comm *c) {
    c->d_count.resize(c->n_local);
    c->h_count.resize(c->n_local);
    for (int i = 0; i < c->n_local; i++) {
        PG_CUDA(c->ctxs[i], cudaSetDevice(c->ctxs[i]->device));
        PG_CUDA(c->ctxs[i], c->d_count[i].reserve(1, nullptr));
        PG_CUDA(c->ctxs[i], c->h_count[i].reserve(1, nullptr));
    }
    return PG_OK;
}

extern "C" {

int pg_shard_range(int64_t total, int rank, int world, int64_t *begin, int64_t *end) {
    if (world < 1 || rank < 0 || rank >= world || total < 0 || !begin || !end)
        return fail(nullptr, PG_ERR_ARG, "pg_shard_range(total=%lld, rank=%d, world=%d)", (long long)total, rank, world);
    const int64_t base = total / world, rem = total % world;
    *begin = rank * base + (rank < rem ? rank : rem);
    *end = *begin + base + (rank < rem ? 1 : 0);
    return PG_OK;
}

int pg_nccl_version(int *version) {
    const NcclApi &nccl = nccl_api();
    if (!version) return PG_ERR_ARG;
    if (!nccl.ok) return fail(nullptr, PG_ERR_NCCL, "pg_nccl_version: %s", nccl.why);
    CNCCL(nullptr, nccl.get_version(version));
    return PG_OK;
}

int pg_init_multi(const int *devices, int n, pg_ctx **ctxs_out, pg_comm **comm_out) {
    if (!devices || n < 1 || !ctxs_out || !comm_out) return fail(nullptr, PG_ERR_ARG, "pg_init_multi: bad argument");
    *comm_out = nullptr;
    for (int i = 0; i < n; i++) ctxs_out[i] = nullptr;
    for (int i = 0; i < n; i++)
        for (int j = 0; j < i; j++)
            if (devices[i] == devices[j]) return fail(nullptr, PG_ERR_ARG, "pg_init_multi: device %d listed twice", devices[i]);
    const NcclApi &nccl = nccl_api();
    if (!nccl.ok) return fail(nullptr, PG_ERR_NCCL, "pg_init_multi: %s", nccl.why);
    auto undo = [&] {
        for (int i = 0; i < n; i++) {
            pg_destroy(ctxs_out[i]);
            ctxs_out[i] = nullptr;
        }
    };
    for (int i = 0; i < n; i++) {
        int rc = pg_init(devices[i], &ctxs_out[i]);
        if (rc) {
            undo();
            return rc;
        }
    }
    pg_comm *c = new (std::nothrow) pg_comm();
    if (!c) {
        undo();
        return fail(nullptr, PG_ERR_ARG, "out of host memory");
    }
    c->world = n;
    c->n_local = n;
    c->first_rank = 0;
    c->ctxs.assign(ctxs_out, ctxs_out + n);
    c->comms.assign(n, nullptr);
    ncclResult_t r = nccl.comm_init_all(c->comms.data(), n, devices);
    if (r != ncclSuccess) {
        delete c;
        undo();
        return fail(nullptr, PG_ERR_NCCL, "ncclCommInitAll(%d devices) failed: %s", n, nccl.error_string(r));
    }
    int rc = comm_alloc_counters(c);
    if (rc) {
        delete c;
        undo();
        return rc;
    }
    *comm_out = c;
    return PG_OK;
}

int pg_comm_unique_id(uint8_t *id) {
    if (!id) return PG_ERR_ARG;
    const NcclApi &nccl = nccl_api();
    if (!nccl.ok) return fail(nullptr, PG_ERR_NCCL, "pg_comm_unique_id: %s", nccl.why);
    ncclUniqueId u;
    CNCCL(nullptr, nccl.get_unique_id(&u));
    memcpy(id, &u, sizeof u);
    return PG_OK;
}

int pg_comm_init_rank(pg_ctx *ctx, const uint8_t *id, int rank, int world, pg_comm **out) {
    if (!ctx || !id || !out || world < 1 || rank < 0 || rank >= world)
        return fail(ctx, PG_ERR_ARG, "pg_comm_init_rank: bad argument (rank %d of %d)", rank, world);
    *out = nullptr;
    const NcclApi &nccl = nccl_api();
    if (!nccl.ok) return fail(ctx, PG_ERR_NCCL, "pg_comm_init_rank: %s", nccl.why);
    PG_CUDA(ctx, cudaSetDevice(ctx->device));
    pg_comm *c = new (std::nothrow) pg_comm();
    if (!c) return fail(ctx, PG_ERR_ARG, "out of host memory");
    c->world = world;
    c->n_local = 1;
    c->first_rank = rank;
    c->ctxs.assign(1, ctx);
    c->comms.assign(1, nullptr);
    ncclUniqueId u;
    memcpy(&u, id, sizeof u);
    ncclResult_t r = nccl.comm_init_rank(&c->comms[0], world, u, rank);
    if (r != ncclSuccess) {
        delete c;
        return fail(ctx, PG_ERR_NCCL, "ncclCommInitRank(rank %d of %d) failed: %s", rank, world, nccl.error_string(r));
    }
    int rc = comm_alloc_counters(c);
    if (rc) {
        delete c;
        return rc;
    }
    *out = c;
    return PG_OK;
}

int pg_comm_info(const pg_comm *c, int *world, int *n_local, int *first_rank) {
    if (!c) return PG_ERR_ARG;
    if (world) *world = c->world;
    if (n_local) *n_local = c->n_local;
    if (first_rank) *first_rank = c->first_rank;
    return PG_OK;
}

int pg_comm_destroy(pg_comm *c) {
    delete c;
    return PG_OK;
}

// K_total = sum over the ranks of the partial Gram matrices, in place on every rank's device buffer; the column counts
// are summed in the same group.  kins[i] belongs to local rank i of the communicator (its context's device).
int pg_kin_allreduce(pg_comm *c, pg_kin *const *kins, int n_local, int64_t *P_total, float *ms) {
    if (!c || !kins || n_local != c->n_local) return fail(nullptr, PG_ERR_ARG, "pg_kin_allreduce: %d handles for %d local ranks", n_local, c ? c->n_local : -1);
    const NcclApi &nccl = nccl_api();
    if (!nccl.ok) return fail(nullptr, PG_ERR_NCCL, "pg_kin_allreduce: %s", nccl.why);
    for (int i = 0; i < n_local; i++) {
        if (!kins[i]) return fail(nullptr, PG_ERR_ARG, "pg_kin_allreduce: handle %d is NULL", i);
        if (kins[i]->ctx->device != c->ctxs[i]->device)
            return fail(kins[i]->ctx, PG_ERR_ARG, "pg_kin_allreduce: handle %d lives on device %d, local rank %d on device %d", i,
                         kins[i]->ctx->device, i, c->ctxs[i]->device);
        if (kins[i]->n != kins[0]->n) return fail(kins[i]->ctx, PG_ERR_ARG, "pg_kin_allreduce: pool counts differ");
    }
    const size_t elems = (size_t)kins[0]->n * kins[0]->n;
    for (int i = 0; i < n_local; i++) {
        pg_kin *h = kins[i];
        PG_CUDA(h->ctx, cudaSetDevice(h->ctx->device));
        *c->h_count[i].get() = h->P;
        PG_CUDA(h->ctx, cudaMemcpyAsync(c->d_count[i].get(), c->h_count[i].get(), 8, cudaMemcpyHostToDevice, h->stream));
        if (ms && i == 0) PG_CUDA(h->ctx, cudaEventRecord(h->ev0, h->stream));
    }
    CNCCL(kins[0]->ctx, nccl.group_start());
    for (int i = 0; i < n_local; i++) {
        pg_kin *h = kins[i];
        ncclResult_t r = nccl.all_reduce(h->d_K.get(), h->d_K.get(), elems, ncclDouble, ncclSum, c->comms[i], h->stream);
        if (r == ncclSuccess)
            r = nccl.all_reduce(c->d_count[i].get(), c->d_count[i].get(), 1, ncclInt64, ncclSum, c->comms[i], h->stream);
        if (r != ncclSuccess) {
            nccl.group_end();
            return fail(h->ctx, PG_ERR_NCCL, "ncclAllReduce (local rank %d) failed: %s", i, nccl.error_string(r));
        }
    }
    CNCCL(kins[0]->ctx, nccl.group_end());
    for (int i = 0; i < n_local; i++) {
        pg_kin *h = kins[i];
        PG_CUDA(h->ctx, cudaSetDevice(h->ctx->device));
        if (ms && i == 0) PG_CUDA(h->ctx, cudaEventRecord(h->ev1, h->stream));
        PG_CUDA(h->ctx, cudaMemcpyAsync(c->h_count[i].get(), c->d_count[i].get(), 8, cudaMemcpyDeviceToHost, h->stream));
    }
    for (int i = 0; i < n_local; i++) {
        pg_kin *h = kins[i];
        PG_CUDA(h->ctx, cudaSetDevice(h->ctx->device));
        PG_CUDA(h->ctx, cudaStreamSynchronize(h->stream));
        h->P_total = *c->h_count[i].get();
    }
    if (ms) PG_CUDA(kins[0]->ctx, cudaEventElapsedTime(ms, kins[0]->ev0, kins[0]->ev1));
    if (P_total) *P_total = kins[0]->P_total;
    return PG_OK;
}

}  // extern "C"
