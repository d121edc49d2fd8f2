// batch_driver.cuh -- NDJSON / multi-document batch driver behind the C ABI (include/simdjson_b200.h, sjb200_batch_*).
// Included at the end of capi.cu (it uses the context internals).
//
// A batch is cut at '\n' into shards (one per GPU) and every shard into segments by the rule of sjb200_batch_split_host
// (segments of up to 2 * seg_bytes - 1 bytes, each cut after the last newline of its seg_bytes window); a segment is
// exactly one reference stage-1 call (segment-relative indexes, own trailer, own verdict: what
// DomParserImplementation.stage1, include/generic/dom_parser_implementation.mojo:65-69, would return for that byte
// range).  Bulk data never leaves its GPU.  The only inter-GPU traffic is ONE NCCL all-gather per pass of the
// {error, n} rows of every segment (the worst error is the maximum over the gathered rows: no separate all-reduce).
//
// Two ways to own the GPUs:
//   sjb200_batch_create       one process drives `ngpus` devices (ncclCommInitAll) -- what a Mojo host would call
//   sjb200_batch_create_rank  one process per GPU (torchrun, MPI): rank r of `world`, communicator from a unique id
//                             made by sjb200_batch_unique_id on rank 0 and carried to the others by the caller
// NCCL is loaded at run time (dlopen "libnccl.so.2", or the path in SJB200_NCCL_LIB) and only when more than one GPU
// takes part, so the library has no link-time dependency on it.
#pragma once
#include <dlfcn.h>

#include <vector>

namespace {

// the few NCCL declarations this file needs (stable ABI since NCCL 2.0)
typedef struct ncclComm *ncclComm_t;
typedef struct {
    char internal[128];
} ncclUniqueId;
enum { NCCL_SUCCESS = 0, NCCL_INT32 = 2 };

struct NcclApi {
    void *handle = nullptr;
    int (*GetUniqueId)(ncclUniqueId *) = nullptr;
    int (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int) = nullptr;
    int (*CommInitAll)(ncclComm_t *, int, const int *) = nullptr;
    int (*AllGather)(const void *, void *, size_t, int, ncclComm_t, cudaStream_t) = nullptr;
    int (*GroupStart)() = nullptr;
    int (*GroupEnd)() = nullptr;
    int (*CommDestroy)(ncclComm_t) = nullptr;
    const char *(*GetErrorString)(int) = nullptr;
    bool ok = false;
};

const NcclApi &nccl() {
    static const NcclApi api = [] {
        NcclApi a;
        const char *path = getenv("SJB200_NCCL_LIB");
        a.handle = dlopen(path && *path ? path : "libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
        if (!a.handle) a.handle = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
        if (!a.handle) {
            fprintf(stderr, "[simdjson_b200] cannot load NCCL (%s); set SJB200_NCCL_LIB\n", dlerror());
            return a;
        }
#define SJ_NCCL_SYM(field, name) a.field = reinterpret_cast<decltype(a.field)>(dlsym(a.handle, name))
        SJ_NCCL_SYM(GetUniqueId, "ncclGetUniqueId");
        SJ_NCCL_SYM(CommInitRank, "ncclCommInitRank");
        SJ_NCCL_SYM(CommInitAll, "ncclCommInitAll");
        SJ_NCCL_SYM(AllGather, "ncclAllGather");
        SJ_NCCL_SYM(GroupStart, "ncclGroupStart");
        SJ_NCCL_SYM(GroupEnd, "ncclGroupEnd");
        SJ_NCCL_SYM(CommDestroy, "ncclCommDestroy");
        SJ_NCCL_SYM(GetErrorString, "ncclGetErrorString");
#undef SJ_NCCL_SYM
        a.ok = a.GetUniqueId && a.CommInitRank && a.CommInitAll && a.AllGather && a.GroupStart && a.GroupEnd && a.CommDestroy;
        return a;
    }();
    return api;
}

int32_t nccl_err(int r) {
    if (r == NCCL_SUCCESS) return SJB200_SUCCESS;
    fprintf(stderr, "[simdjson_b200] NCCL error: %s\n", nccl().GetErrorString ? nccl().GetErrorString(r) : "?");
    return SJB200_UNEXPECTED_ERROR;
}

}  // namespace

struct BatchGpu {                       // one GPU this process drives
    sjb200_ctx *ctx = nullptr;
    ncclComm_t comm = nullptr;
    cudaStream_t xstream = nullptr;     // the verdict exchange runs here, beside the kernels of the next pass
    cudaEvent_t pass_done[2] = {nullptr, nullptr};   // kernels of the pass that used buffer set k are done
    cudaEvent_t xchg_done[2] = {nullptr, nullptr};   // the exchange that read buffer set k is done
    int32_t *d_rows[2] = {nullptr, nullptr};         // this GPU's {error, n} rows, max_segments of them
    int32_t *d_all[2] = {nullptr, nullptr};          // gathered rows of every rank: [world][max_segments][2]
    int32_t *h_all = nullptr;                        // pinned copy of the most recent gathered rows
    std::vector<uint64_t> seg_offsets;               // planned segments of the resident shard (byte offsets, nseg + 1)
    std::vector<uint64_t> idx_offsets;               // where each segment's indexes start in this GPU's index array
    const uint8_t *d_shard = nullptr;
};

struct sjb200_batch {
    int world = 1;                       // ranks taking part in the exchange (GPUs over all processes)
    int first_rank = 0;                  // rank of local GPU 0
    std::vector<BatchGpu> gpus;          // local GPUs
    uint64_t max_shard_bytes = 0, seg_bytes = 0;
    uint32_t max_segments = 0;
    uint64_t passes = 0;
    int last_set = -1;
};

namespace {

void batch_free(sjb200_batch *b) {
    if (!b) return;
    for (BatchGpu &g : b->gpus) {
        if (g.ctx) cudaSetDevice(g.ctx->device);
        if (g.ctx) cudaStreamSynchronize(g.ctx->stream);
        if (g.xstream) cudaStreamSynchronize(g.xstream);
        if (g.comm && nccl().ok) nccl().CommDestroy(g.comm);
        for (int k = 0; k < 2; k++) {
            cudaFree(g.d_rows[k]);
            cudaFree(g.d_all[k]);
            if (g.pass_done[k]) cudaEventDestroy(g.pass_done[k]);
            if (g.xchg_done[k]) cudaEventDestroy(g.xchg_done[k]);
        }
        if (g.h_all) cudaFreeHost(g.h_all);
        if (g.xstream) cudaStreamDestroy(g.xstream);
        if (g.ctx) sjb200_ctx_destroy(g.ctx);
    }
    delete b;
}

int32_t batch_init_gpu(sjb200_batch *b, BatchGpu &g, int device, uint64_t max_host_bytes) {
    int32_t rc = sjb200_ctx_create(device, b->seg_bytes * 2 < 0xFFFFFFFFull ? b->seg_bytes * 2 : 0xFFFFFFFFull, 0, 0, &g.ctx);
    if (rc != SJB200_SUCCESS) return rc;
    CK(cudaSetDevice(device));
    if (max_host_bytes) {   // host-batch entry point: staging for one shard and its indexes
        CK(cudaMalloc(&g.ctx->d_in, (size_t)max_host_bytes + 256));
        g.ctx->d_out_cap = max_host_bytes + 3ull * b->max_segments;
        CK(cudaMalloc(&g.ctx->d_out, (size_t)(g.ctx->d_out_cap + 4) * 4));
        g.ctx->max_len_host = max_host_bytes;
    }
    CK(cudaStreamCreateWithFlags(&g.xstream, cudaStreamNonBlocking));
    const size_t row_bytes = (size_t)b->max_segments * 8;
    for (int k = 0; k < 2; k++) {
        CK(cudaEventCreateWithFlags(&g.pass_done[k], cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&g.xchg_done[k], cudaEventDisableTiming));
        CK(cudaMalloc(&g.d_rows[k], row_bytes));
        CK(cudaMalloc(&g.d_all[k], row_bytes * b->world));
        CK(cudaMemset(g.d_rows[k], 0xFF, row_bytes));
        CK(cudaMemset(g.d_all[k], 0xFF, row_bytes * b->world));
    }
    CK(cudaHostAlloc(&g.h_all, row_bytes * b->world, cudaHostAllocDefault));
    memset(g.h_all, 0xFF, row_bytes * b->world);
    CK(cudaDeviceSynchronize());
    return SJB200_SUCCESS;
}

int32_t batch_check_params(uint64_t seg_bytes, uint32_t max_segments) {
    if (seg_bytes == 0 || seg_bytes > 0x7FFFFFFFull) return SJB200_CAPACITY;
    if (max_segments == 0 || max_segments > RESULT_SLOTS) return SJB200_CAPACITY;
    return SJB200_SUCCESS;
}

// one pass over the planned segments of local GPU `gi` into d_idx, rows into buffer set `set`; the exchange follows on xstream
int32_t batch_enqueue_gpu(sjb200_batch *b, int gi, uint32_t *d_idx, uint64_t idx_capacity, int set, uint32_t flags) {
    BatchGpu &g = b->gpus[gi];
    sjb200_ctx *c = g.ctx;
    CK(cudaSetDevice(c->device));
    const uint32_t nseg = (uint32_t)(g.seg_offsets.size() - 1);
    // this buffer set was last read by the exchange of two passes ago
    CK(cudaStreamWaitEvent(c->stream, g.xchg_done[set], 0));
    // (rows of segments that do not exist read {-1, -1}: batch_reset_rows, whenever the plan changes -- not once per pass,
    // a memset between two passes costs the GPU ~2 us)
    const int32_t rc = sjb200_batch_run_device_async(c, g.d_shard, g.seg_offsets.data(), 0, nseg, d_idx, g.idx_offsets.data(), idx_capacity,
                                                     g.d_rows[set], flags);
    CK(cudaEventRecord(g.pass_done[set], c->stream));
    return rc == SJB200_UNINITIALIZED ? rc : SJB200_SUCCESS;   // per-segment launch errors travel in the rows
}

int32_t batch_exchange(sjb200_batch *b, int set) {
    const size_t count = (size_t)b->max_segments * 2;
    if (b->world == 1) {
        BatchGpu &g = b->gpus[0];
        CK(cudaSetDevice(g.ctx->device));
        CK(cudaStreamWaitEvent(g.xstream, g.pass_done[set], 0));
        CK(cudaMemcpyAsync(g.d_all[set], g.d_rows[set], count * 4, cudaMemcpyDeviceToDevice, g.xstream));
        CK(cudaEventRecord(g.xchg_done[set], g.xstream));
        return SJB200_SUCCESS;
    }
    const NcclApi &n = nccl();
    for (BatchGpu &g : b->gpus) {
        CK(cudaSetDevice(g.ctx->device));
        CK(cudaStreamWaitEvent(g.xstream, g.pass_done[set], 0));
    }
    int r = b->gpus.size() > 1 ? n.GroupStart() : NCCL_SUCCESS;
    for (BatchGpu &g : b->gpus)
        if (r == NCCL_SUCCESS) r = n.AllGather(g.d_rows[set], g.d_all[set], count, NCCL_INT32, g.comm, g.xstream);
    if (b->gpus.size() > 1) {
        const int r2 = n.GroupEnd();
        if (r == NCCL_SUCCESS) r = r2;
    }
    if (r != NCCL_SUCCESS) return nccl_err(r);
    for (BatchGpu &g : b->gpus) {
        CK(cudaSetDevice(g.ctx->device));
        CK(cudaEventRecord(g.xchg_done[set], g.xstream));
    }
    return SJB200_SUCCESS;
}

// a new plan: both row-buffer sets of a GPU read "no such segment" everywhere; the kernels then fill the rows that exist.
// Stream ordered behind every exchange that still reads them.
int32_t batch_reset_rows(sjb200_batch *b, BatchGpu &g) {
    CK(cudaSetDevice(g.ctx->device));
    for (int k = 0; k < 2; k++) {
        CK(cudaStreamWaitEvent(g.ctx->stream, g.xchg_done[k], 0));
        CK(cudaMemsetAsync(g.d_rows[k], 0xFF, (size_t)b->max_segments * 8, g.ctx->stream));
    }
    return SJB200_SUCCESS;
}

// cut [lo, hi) of a host batch forward to line starts, the rule every shard applies to both of its ends
uint64_t next_line_start(const uint8_t *buf, uint64_t p, uint64_t total) {
    if (p == 0) return 0;
    while (p < total && buf[p - 1] != '\n') p++;
    return p;
}

}  // namespace

#pragma GCC visibility push(default)
extern "C" {

int32_t sjb200_batch_unique_id(void *id128) {
    if (!id128) return SJB200_UNINITIALIZED;
    if (!nccl().ok) return SJB200_UNEXPECTED_ERROR;
    ncclUniqueId id;
    const int r = nccl().GetUniqueId(&id);
    if (r != NCCL_SUCCESS) return nccl_err(r);
    memcpy(id128, &id, sizeof id);
    return SJB200_SUCCESS;
}

int32_t sjb200_batch_create(int32_t ngpus, const int32_t *devices, uint64_t max_shard_bytes, uint64_t seg_bytes, uint32_t max_segments,
                            uint32_t flags, sjb200_batch **out) {
    (void)flags;
    if (!out) return SJB200_UNINITIALIZED;
    *out = nullptr;
    if (ngpus < 1 || ngpus > sjb200_device_count()) return SJB200_CAPACITY;
    int32_t rc = batch_check_params(seg_bytes, max_segments);
    if (rc != SJB200_SUCCESS) return rc;
    if (ngpus > 1 && !nccl().ok) return SJB200_UNEXPECTED_ERROR;
    sjb200_batch *b = new (std::nothrow) sjb200_batch();
    if (!b) return SJB200_MEMALLOC;
    b->world = ngpus;
    b->max_shard_bytes = max_shard_bytes;
    b->seg_bytes = seg_bytes;
    b->max_segments = max_segments;
    b->gpus.resize(ngpus);
    std::vector<int> devs(ngpus);
    for (int g = 0; g < ngpus; g++) devs[g] = devices ? devices[g] : g;
    for (int g = 0; g < ngpus && rc == SJB200_SUCCESS; g++) rc = batch_init_gpu(b, b->gpus[g], devs[g], max_shard_bytes);
    if (rc == SJB200_SUCCESS && ngpus > 1) {
        std::vector<ncclComm_t> comms(ngpus);
        rc = nccl_err(nccl().CommInitAll(comms.data(), ngpus, devs.data()));
        if (rc == SJB200_SUCCESS)
            for (int g = 0; g < ngpus; g++) b->gpus[g].comm = comms[g];
    }
    if (rc != SJB200_SUCCESS) {
        batch_free(b);
        return rc;
    }
    *out = b;
    return SJB200_SUCCESS;
}

int32_t sjb200_batch_create_rank(int32_t device, int32_t rank, int32_t world, const void *nccl_id, uint64_t max_shard_bytes, uint64_t seg_bytes,
                                 uint32_t max_segments, uint32_t flags, sjb200_batch **out) {
    (void)flags;
    if (!out) return SJB200_UNINITIALIZED;
    *out = nullptr;
    if (world < 1 || rank < 0 || rank >= world || (world > 1 && !nccl_id)) return SJB200_CAPACITY;
    int32_t rc = batch_check_params(seg_bytes, max_segments);
    if (rc != SJB200_SUCCESS) return rc;
    if (world > 1 && !nccl().ok) return SJB200_UNEXPECTED_ERROR;
    sjb200_batch *b = new (std::nothrow) sjb200_batch();
    if (!b) return SJB200_MEMALLOC;
    b->world = world;
    b->first_rank = rank;
    b->max_shard_bytes = max_shard_bytes;
    b->seg_bytes = seg_bytes;
    b->max_segments = max_segments;
    b->gpus.resize(1);
    rc = batch_init_gpu(b, b->gpus[0], device, 0);
    if (rc == SJB200_SUCCESS && world > 1) {
        ncclUniqueId id;
        memcpy(&id, nccl_id, sizeof id);
        rc = nccl_err(nccl().CommInitRank(&b->gpus[0].comm, world, id, rank));
    }
    if (rc != SJB200_SUCCESS) {
        batch_free(b);
        return rc;
    }
    *out = b;
    return SJB200_SUCCESS;
}

int32_t sjb200_batch_destroy(sjb200_batch *b) {
    batch_free(b);
    return SJB200_SUCCESS;
}

int32_t sjb200_batch_local_gpus(sjb200_batch *b) { return b ? (int32_t)b->gpus.size() : 0; }

int32_t sjb200_batch_ctx(sjb200_batch *b, int32_t local_gpu, sjb200_ctx **ctx) {
    if (!b || !ctx || local_gpu < 0 || local_gpu >= (int32_t)b->gpus.size()) return SJB200_UNINITIALIZED;
    *ctx = b->gpus[local_gpu].ctx;
    return SJB200_SUCCESS;
}

int32_t sjb200_batch_plan_resident(sjb200_batch *b, int32_t local_gpu, const uint8_t *d_shard, uint64_t shard_len, uint64_t *seg_offsets,
                                   uint64_t *idx_offsets, uint32_t *n_segments) {
    if (!b || local_gpu < 0 || local_gpu >= (int32_t)b->gpus.size()) return SJB200_UNINITIALIZED;
    BatchGpu &g = b->gpus[local_gpu];
    std::vector<uint64_t> offs(b->max_segments + 1);
    uint32_t nseg = 0;
    const int32_t rc = sjb200_batch_split_device(g.ctx, d_shard, shard_len, b->seg_bytes, offs.data(), b->max_segments, &nseg);
    if (rc != SJB200_SUCCESS) return rc;
    const int32_t rr = batch_reset_rows(b, g);
    if (rr != SJB200_SUCCESS) return rr;
    g.d_shard = d_shard;
    g.seg_offsets.assign(offs.begin(), offs.begin() + nseg + 1);
    g.idx_offsets.assign(nseg + 1, 0);
    for (uint32_t s = 0; s < nseg; s++) g.idx_offsets[s + 1] = g.idx_offsets[s] + (g.seg_offsets[s + 1] - g.seg_offsets[s]) + 3;
    for (uint32_t s = 0; s <= nseg; s++) {
        if (seg_offsets) seg_offsets[s] = g.seg_offsets[s];
        if (idx_offsets) idx_offsets[s] = g.idx_offsets[s];
    }
    if (n_segments) *n_segments = nseg;
    return SJB200_SUCCESS;
}

int32_t sjb200_batch_run_resident_async(sjb200_batch *b, uint32_t *const *d_idx, const uint64_t *idx_capacities, uint32_t flags) {
    if (!b || !d_idx || !idx_capacities) return SJB200_UNINITIALIZED;
    const int set = (int)(b->passes & 1);
    for (size_t gi = 0; gi < b->gpus.size(); gi++) {
        if (b->gpus[gi].seg_offsets.size() < 2) return SJB200_UNINITIALIZED;   // not planned
        const int32_t rc = batch_enqueue_gpu(b, (int)gi, d_idx[gi], idx_capacities[gi], set, flags);
        if (rc != SJB200_SUCCESS) return rc;
    }
    const int32_t rc = batch_exchange(b, set);
    if (rc != SJB200_SUCCESS) return rc;
    b->last_set = set;
    b->passes++;
    return SJB200_SUCCESS;
}

int32_t sjb200_batch_finish(sjb200_batch *b, int32_t *all_rows, int32_t *global_error) {
    if (!b) return SJB200_UNINITIALIZED;
    if (b->last_set < 0) return SJB200_UNINITIALIZED;
    const size_t bytes = (size_t)b->max_segments * 8 * b->world;
    // every exchange still in flight, on every local GPU; then the gathered rows of the most recent pass (identical on all of them)
    for (BatchGpu &g : b->gpus) {
        CK(cudaSetDevice(g.ctx->device));
        CK(cudaStreamSynchronize(g.ctx->stream));
        CK(cudaStreamSynchronize(g.xstream));
    }
    BatchGpu &g0 = b->gpus[0];
    CK(cudaSetDevice(g0.ctx->device));
    CK(cudaMemcpy(g0.h_all, g0.d_all[b->last_set], bytes, cudaMemcpyDeviceToHost));
    int32_t worst = SJB200_SUCCESS;
    for (size_t k = 0; k < (size_t)b->max_segments * b->world; k++)
        if (g0.h_all[2 * k] > worst) worst = g0.h_all[2 * k];
    if (all_rows) memcpy(all_rows, g0.h_all, bytes);
    if (global_error) *global_error = worst;
    return SJB200_SUCCESS;
}

int32_t sjb200_batch_run(sjb200_batch *b, const uint8_t *buf, uint64_t len, uint32_t *idx_out, uint64_t idx_capacity, uint64_t *seg_offsets,
                         uint64_t *seg_idx_offsets, uint32_t *seg_counts, int32_t *seg_errors, uint32_t max_total_segments, uint32_t *n_segments,
                         int32_t *global_error, uint32_t flags) {
    if (!b || !buf || !idx_out || !seg_offsets || !seg_idx_offsets || !n_segments) return SJB200_UNINITIALIZED;
    if (b->first_rank != 0 || (int)b->gpus.size() != b->world) return SJB200_UNINITIALIZED;   // single-process mode only
    if (len == 0) return SJB200_EMPTY;
    const int G = b->world;
    // shards: equal contiguous slices, both ends moved forward to a line start; segments inside every shard
    std::vector<uint64_t> shard(G + 1);
    const uint64_t per = (len + G - 1) / G;
    for (int g = 0; g < G; g++) shard[g] = next_line_start(buf, (uint64_t)g * per < len ? (uint64_t)g * per : len, len);
    shard[G] = len;
    uint32_t total = 0;
    seg_offsets[0] = 0;
    std::vector<uint32_t> first_seg(G + 1, 0);
    for (int g = 0; g < G; g++) {
        BatchGpu &gp = b->gpus[g];
        const uint64_t lo = shard[g], hi = shard[g + 1];
        first_seg[g] = total;
        gp.seg_offsets.assign(1, 0);
        if (hi > lo) {
            if (hi - lo > b->max_shard_bytes) return SJB200_CAPACITY;
            std::vector<uint64_t> offs(b->max_segments + 1);
            uint32_t nseg = 0;
            const int32_t rc = sjb200_batch_split_host(buf + lo, hi - lo, b->seg_bytes, offs.data(), b->max_segments, &nseg);
            if (rc != SJB200_SUCCESS) return rc;
            if (total + nseg > max_total_segments) return SJB200_CAPACITY;
            gp.seg_offsets.assign(offs.begin(), offs.begin() + nseg + 1);
            for (uint32_t s = 0; s < nseg; s++) seg_offsets[total + s + 1] = lo + offs[s + 1];
            total += nseg;
        }
        const uint32_t nseg = (uint32_t)gp.seg_offsets.size() - 1;
        gp.idx_offsets.assign(nseg + 1, 0);
        for (uint32_t s = 0; s < nseg; s++) gp.idx_offsets[s + 1] = gp.idx_offsets[s] + (gp.seg_offsets[s + 1] - gp.seg_offsets[s]) + 3;
    }
    first_seg[G] = total;
    *n_segments = total;
    for (uint32_t s = 0; s <= total; s++) seg_idx_offsets[s] = seg_offsets[s] + 3ull * s;   // entries; segment s owns [s, s+1)
    if (seg_idx_offsets[total] > idx_capacity) return SJB200_CAPACITY;
    // copy in, index: every GPU on its own stream
    const int set = (int)(b->passes & 1);
    for (int g = 0; g < G; g++) {
        BatchGpu &gp = b->gpus[g];
        sjb200_ctx *c = gp.ctx;
        CK(cudaSetDevice(c->device));
        const uint64_t lo = shard[g], hi = shard[g + 1];
        if (hi > lo) CK(cudaMemcpyAsync(c->d_in, buf + lo, (size_t)(hi - lo), cudaMemcpyHostToDevice, c->stream));
        gp.d_shard = c->d_in;
        {
            const int32_t rr = batch_reset_rows(b, gp);   // the host entry point plans anew on every call
            if (rr != SJB200_SUCCESS) return rr;
        }
        if (gp.seg_offsets.size() >= 2) {
            const int32_t rc = batch_enqueue_gpu(b, g, c->d_out, c->d_out_cap, set, flags);
            if (rc != SJB200_SUCCESS) return rc;
        } else {
            CK(cudaEventRecord(gp.pass_done[set], c->stream));
        }
    }
    int32_t rc = batch_exchange(b, set);
    if (rc != SJB200_SUCCESS) return rc;
    b->last_set = set;
    b->passes++;
    std::vector<int32_t> rows((size_t)b->max_segments * 2 * G);
    int32_t worst = 0;
    rc = sjb200_batch_finish(b, rows.data(), &worst);
    if (rc != SJB200_SUCCESS) return rc;
    // copy every segment's n + 3 entries back
    for (int g = 0; g < G; g++) {
        BatchGpu &gp = b->gpus[g];
        sjb200_ctx *c = gp.ctx;
        CK(cudaSetDevice(c->device));
        const uint32_t nseg = (uint32_t)gp.seg_offsets.size() - 1;
        for (uint32_t s = 0; s < nseg; s++) {
            const int32_t err = rows[((size_t)g * b->max_segments + s) * 2], n = rows[((size_t)g * b->max_segments + s) * 2 + 1];
            const uint32_t gs = first_seg[g] + s;
            if (seg_errors) seg_errors[gs] = err;
            if (seg_counts) seg_counts[gs] = n > 0 ? (uint32_t)n : 0u;
            const Stage1Result r = c->h_results[s];
            const uint64_t have = c->launch_rc[s] != SJB200_SUCCESS ? 0 : (r.n_valid ? (uint64_t)r.n + 3 : r.n_written);
            const uint64_t room = gp.idx_offsets[s + 1] - gp.idx_offsets[s];
            const uint64_t take = have < room ? have : room;
            if (take) CK(cudaMemcpyAsync(idx_out + seg_idx_offsets[gs], c->d_out + gp.idx_offsets[s], (size_t)take * 4, cudaMemcpyDeviceToHost, c->stream));
        }
    }
    for (int g = 0; g < G; g++) {
        CK(cudaSetDevice(b->gpus[g].ctx->device));
        CK(cudaStreamSynchronize(b->gpus[g].ctx->stream));
    }
    if (global_error) *global_error = worst;
    return SJB200_SUCCESS;
}

}  // extern "C"
#pragma GCC visibility pop
