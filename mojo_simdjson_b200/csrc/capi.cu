// capi.cu -- C ABI (include/simdjson_b200.h) over the sm_100a stage-1 kernels: context, buffers, launches.
// There is no CPU fallback anywhere in this file: without a CUDA device every entry point fails.
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <new>

#include "../../include/simdjson_b200.h"
#include "stage1_kernel.cuh"
#include "stage1_persistent.cuh"
#include "stage1_split.cuh"
#include "stage1_stream.cuh"

using namespace sjb200;

namespace {

constexpr uint32_t RESULT_SLOTS = 256;
constexpr uint64_t MIN_TILE = 2 * 2048;
// Kernel organisation by document size (device-resident documents; tools/sizesweep.py, measured): the persistent tile kernel
// for small documents (all 148 SMs get a tile even at a few hundred KiB), the split pair from SPLIT_MIN_BYTES, the stream
// pipeline from STREAM_MIN_BYTES.  (A fused single-launch organisation and a windowed two-stream pipeline were measured in
// round 2 and removed again: profiles/r2_overlap_experiments.txt.)
constexpr uint64_t SPLIT_MIN_BYTES = 24ull << 20;
constexpr uint64_t STREAM_MIN_BYTES = 80ull << 20;
constexpr int FLATTEN_FW = 4;   // warps (= units of two chunks) per CTA of the flatten kernel (2 and 4 measure alike, 8: -4 %)
constexpr int STREAM_NW = 8;    // compute warps per CTA of the stream classify kernel

inline int32_t cuda_err(cudaError_t e) {
    if (e == cudaSuccess) return SJB200_SUCCESS;
    if (e == cudaErrorMemoryAllocation) return SJB200_MEMALLOC;
    fprintf(stderr, "[simdjson_b200] CUDA error: %s\n", cudaGetErrorString(e));
    return SJB200_UNEXPECTED_ERROR;
}
#define CK(call)                                  \
    do {                                          \
        cudaError_t e__ = (call);                 \
        if (e__ != cudaSuccess) return cuda_err(e__); \
    } while (0)

bool valid_warps(int w) { return w == 2 || w == 4 || w == 8 || w == 16 || w == 24; }

}  // namespace

struct sjb200_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    uint64_t max_len = 0, max_len_host = 0;
    uint8_t *d_in = nullptr;        // host-path input staging on the device
    uint32_t *d_out = nullptr;      // host-path output on the device
    uint64_t d_out_cap = 0;
    uint64_t *desc = nullptr;           // look-back descriptors, one 8-byte word per tile / block
    uint32_t max_tiles = 0;
    uint32_t *ticket = nullptr;
    Stage1Result *h_results = nullptr;  // mapped pinned, RESULT_SLOTS entries
    Stage1Result *d_results = nullptr;  // device alias of h_results
    int32_t launch_rc[RESULT_SLOTS] = {};   // host-side launch status per result slot (never written by the device)
    uint32_t slot = 0;                  // slot used by the most recent launch
    uint32_t gen = 0;
    int forced_warps = 0;
    int kernel_kind = SJB200_KERNEL_AUTO;  // sjb200_ctx_set_kernel
    int sm_count = 0;
    int persist_occ[5] = {0, 0, 0, 0, 0};  // resident CTAs per SM of the persistent kernel for NW = 2, 4, 8, 16, 24
    int split_occ[2] = {0, 0};             // same for the classify kernel of the split pair, NW = 8, 16
    int stream_occ = 0;                    // same for the stream classify kernel
    // scratch of the split / stream organisations, sized for `scratch_chunks` 2 KiB chunks (sjb200_ctx_reserve, or
    // grown on demand with the stream-ordered allocator: no call ever synchronises for it)
    uint64_t *d_masks = nullptr;           // the two structural mask planes of every chunk (512 B per chunk)
    uint64_t *d_carry = nullptr;           // one carry word per chunk
    uint32_t *d_chunk_sum = nullptr;       // 16-byte chunk summaries
    uint32_t *d_block_sum = nullptr;       // stream pipeline: the same per 4096 chunks
    uint64_t scratch_chunks = 0;
    bool scratch_failed = false;           // an allocation failed once: automatic choice stays with the persistent kernel
    uint32_t *d_spec_flag = nullptr;       // [0] speculation failed, [1] deferred UTF-8 violation (generation valued)
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    bool timed = false;
    uint64_t launches = 0;
    uint32_t last_flags = 0;
    bool pending = false;
    uint64_t *d_split = nullptr;        // scratch for batch_split_device
    uint64_t *d_trace = nullptr;        // debug builds only
    uint32_t launch_seq = 0;            // alternates the persistent kernel's ticket counters
    cudaMemPool_t pool = nullptr;       // stream-ordered pool of the stage-2 temporaries; keeps its memory between calls
    uint64_t resident_len = 0;          // host path: the document of the last successful sjb200_stage1 is still in d_in / d_out
    uint32_t resident_n = 0;
    // streaming host path: second stream for the device-to-host copies, one event + one mapped progress word per chunk
    cudaStream_t copy_stream = nullptr;
    static constexpr int MAX_CHUNKS = 256;
    cudaEvent_t chunk_ev[MAX_CHUNKS] = {};
    uint32_t *h_progress = nullptr, *d_progress = nullptr;
    uint64_t chunk_bytes = 32ull << 20;
};

namespace {

template <typename K>
cudaError_t prepare_kernel(K kernel_utf8, K kernel_plain, int threads, int smem, int *occ) {
    cudaError_t e = cudaFuncSetAttribute(kernel_utf8, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(kernel_plain, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    cudaFuncSetAttribute(kernel_utf8, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
    cudaFuncSetAttribute(kernel_plain, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
    int a = 0, b = 0;
    if (e == cudaSuccess) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&a, kernel_utf8, threads, smem);
    if (e == cudaSuccess) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&b, kernel_plain, threads, smem);
    *occ = a < b ? a : b;
    if (*occ < 1) *occ = 1;
    return e;
}
template <int NW>
cudaError_t prepare_persist(int *occ) {
    using Cfg = PersistCfg<NW>;
    return prepare_kernel(stage1_persistent_kernel<NW, true>, stage1_persistent_kernel<NW, false>, Cfg::THREADS, Cfg::SMEM_BYTES, occ);
}
template <int NW>
cudaError_t prepare_split(int *occ) {
    using Cfg = SplitCfg<NW>;
    cudaFuncSetAttribute(stage1_flatten2_kernel<FLATTEN_FW>, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
    return prepare_kernel(stage1_classify_kernel<NW, true>, stage1_classify_kernel<NW, false>, Cfg::THREADS, Cfg::SMEM_BYTES, occ);
}
cudaError_t prepare_stream(int *occ) {
    using Cfg = StreamCfg<STREAM_NW>;
    // every kernel of the pipeline asks for the same shared-memory carve-out: kernels with different L1 / shared splits
    // cannot share an SM, and scan + flatten of one window must run beside the classify CTAs of the next
    cudaFuncSetAttribute(stage1_span_scan_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
    cudaFuncSetAttribute(stage1_flatten2_kernel<FLATTEN_FW>, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
    return prepare_kernel(stage1_stream_classify_kernel<STREAM_NW, true>, stage1_stream_classify_kernel<STREAM_NW, false>, Cfg::THREADS, Cfg::SMEM_BYTES, occ);
}
// Launch `kernel` so that it may be scheduled while the previous kernel of the stream drains (programmatic dependent
// launch); the kernel itself waits for its predecessor (griddepcontrol.wait) before it reads anything.
template <typename... KArgs, typename... Args>
cudaError_t launch_dependent(void (*kernel)(KArgs...), unsigned grid, unsigned block, size_t smem, cudaStream_t s, bool pdl, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(block);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}
template <int NW, bool UTF8>
cudaError_t launch_persist(const Stage1Params &p, cudaStream_t s, int max_ctas) {
    using Cfg = PersistCfg<NW>;
    const unsigned span = p.tile_end - p.tile_begin;
    const unsigned grid = span < (unsigned)max_ctas ? span : (unsigned)max_ctas;
    // as the fallback of the stream pipeline (spec_flag set) it follows the flatten kernel as a dependent launch
    return launch_dependent(stage1_persistent_kernel<NW, UTF8>, grid, Cfg::THREADS, Cfg::SMEM_BYTES, s, p.spec_flag != nullptr, p);
}
// flatten chunks [c0, c1) (c0 even): units of two chunks per warp
cudaError_t launch_flatten(const Stage1Params &p, uint32_t c0, uint32_t c1, cudaStream_t s) {
    constexpr int FW = FLATTEN_FW;
    return launch_dependent(stage1_flatten2_kernel<FW>, (c1 - c0 + FW * 2 - 1) / (FW * 2), Flatten2Cfg<FW>::THREADS, Flatten2Cfg<FW>::SMEM_BYTES, s, true, p, c0, c1);
}

template <int NW, bool UTF8>
cudaError_t launch_split(const Stage1Params &p, cudaStream_t s, int max_ctas) {
    using Cfg = SplitCfg<NW>;
    const unsigned span = p.tile_end - p.tile_begin;
    const unsigned grid = span < (unsigned)max_ctas ? span : (unsigned)max_ctas;
    stage1_classify_kernel<NW, UTF8><<<grid, Cfg::THREADS, Cfg::SMEM_BYTES, s>>>(p);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    const uint32_t c0 = p.tile_begin * NW, c1 = p.tile_end * NW;
    return launch_flatten(p, c0, c1, s);
}
// The stream pipeline (stage1_stream.cuh): classify -> span_scan -> flatten, stream ordered; the dependent
// launches overlap their launch latency with their predecessor (programmatic dependent launch).
template <bool UTF8>
cudaError_t launch_stream(sjb200_ctx *c, const Stage1Params &p, cudaStream_t s, int max_ctas) {
    using Cfg = StreamCfg<STREAM_NW>;
    const uint32_t nchunks = (uint32_t)((p.alen + 2047) / 2048);
    const unsigned want = (nchunks + STREAM_NW - 1) / STREAM_NW;
    const unsigned grid = want < (unsigned)max_ctas ? want : (unsigned)max_ctas;
    // (the first launch of a document is a dependent launch too: back-to-back documents overlap their launch latencies)
    cudaError_t e = launch_dependent(stage1_stream_classify_kernel<STREAM_NW, UTF8>, grid, Cfg::THREADS, Cfg::SMEM_BYTES, s, true, p, nchunks, 0u, nchunks, p.abase - Cfg::HALO);
    const unsigned nblocks = (nchunks + SPAN_BLOCK - 1) / SPAN_BLOCK;
    if (e == cudaSuccess) e = launch_dependent(stage1_span_scan_kernel, nblocks, SPAN_SCAN_THREADS, 0, s, true, p, nchunks);
    if (e == cudaSuccess) e = launch_flatten(p, 0u, nchunks, s);
    c->launches += 3;
    return e;
}

int pick_warps(const sjb200_ctx *c, uint64_t alen) {
    if (c->forced_warps) return c->forced_warps;
    // small documents: smaller tiles so that the work spreads over all 148 SMs (measured, tools/quickbench.py: 16-warp tiles
    // win from 8 MiB on -- 8 MiB: 480 vs 411 GB/s, 16 MiB: 761 vs 718, 48 MiB: 1060 vs 996)
    if (alen >= (uint64_t)8 << 20) return 16;
    if (alen >= (uint64_t)148 * 4 * 16384) return 8;
    if (alen >= (uint64_t)148 * 4 * 8192) return 4;
    return 2;
}

// Describes one document: geometry, tile shape and generation.  A document is indexed by one launch (tile range =
// everything) or, on the streaming host path, by several launches over consecutive tile ranges sharing the generation.
struct DocPlan {
    Stage1Params p;
    int warps;       // tile shape of the persistent kernel (also the exact fallback of the speculating organisations)
    int kind;        // SJB200_KERNEL_PERSISTENT / SPLIT / STREAM
    bool utf8;
};

void free_scratch(sjb200_ctx *c, cudaStream_t s) {
    // stream ordered: kernels already enqueued on `s` keep their buffers until they have run
    if (c->d_masks) cudaFreeAsync(c->d_masks, s);
    if (c->d_carry) cudaFreeAsync(c->d_carry, s);
    if (c->d_chunk_sum) cudaFreeAsync(c->d_chunk_sum, s);
    if (c->d_block_sum) cudaFreeAsync(c->d_block_sum, s);
    c->d_masks = c->d_carry = nullptr;
    c->d_chunk_sum = c->d_block_sum = nullptr;
    c->scratch_chunks = 0;
}

// Scratch for documents of up to `chunks` 2 KiB chunks (0.26 bytes per input byte: mask planes len/4, summaries and carry
// words; the stream pipeline's parked UTF-8 lanes add 0.31 bytes per input byte and are allocated only when it is used).
// Grows geometrically; allocation and release are stream ordered (cudaMallocAsync), so an enqueue never synchronises.
cudaError_t ensure_scratch(sjb200_ctx *c, uint64_t chunks, cudaStream_t s) {
    if (chunks <= c->scratch_chunks) return cudaSuccess;
    uint64_t n = chunks + 64;
    if (n < c->scratch_chunks) n = c->scratch_chunks;
    if (chunks > c->scratch_chunks && n < c->scratch_chunks * 3 / 2) n = c->scratch_chunks * 3 / 2;
    const uint64_t max_chunks = (c->max_len + 16) / 2048 + 64;
    if (n > max_chunks) n = max_chunks > chunks + 64 ? max_chunks : chunks + 64;
    free_scratch(c, s);
    cudaError_t e = cudaMallocAsync(&c->d_masks, n * 512, s);
    if (e == cudaSuccess) e = cudaMallocAsync(&c->d_carry, n * 8, s);
    if (e == cudaSuccess) e = cudaMallocAsync(&c->d_chunk_sum, n * 16, s);
    if (e == cudaSuccess) e = cudaMallocAsync(&c->d_block_sum, (n / SPAN_BLOCK + 2) * 32, s);
    if (e == cudaSuccess) e = cudaMemsetAsync(c->d_block_sum, 0, (n / SPAN_BLOCK + 2) * 32, s);   // generation-tagged: no stale tag may match
    if (e != cudaSuccess) {
        free_scratch(c, s);
        cudaGetLastError();
        return e;
    }
    c->scratch_chunks = n;
    return cudaSuccess;
}

int32_t plan_document(sjb200_ctx *c, DocPlan &d, const uint8_t *d_buf, uint64_t len, uint32_t *d_idx, uint64_t cap,
                      uint32_t flags, uint32_t slot, int32_t *d_status, bool whole_document = true) {
    Stage1Params &p = d.p;
    memset(&p, 0, sizeof p);
    const uintptr_t addr = reinterpret_cast<uintptr_t>(d_buf);
    p.mis = (uint32_t)(addr & 15u);
    p.abase = d_buf - p.mis;
    p.alen = (uint64_t)p.mis + len;
    p.len = (uint32_t)len;
    p.out = d_idx;
    p.cap = cap;
    p.desc = c->desc;
    p.result = c->d_results + slot;
    p.dev_status = d_status;
    p.trace = c->d_trace;
    c->gen = (c->gen + 1) & GEN_MASK;
    if (c->gen == 0) {  // the 20-bit generation wrapped: clear everything generation tagged once (stream ordered), restart at 1
        cudaMemsetAsync(c->desc, 0, (size_t)c->max_tiles * 8, c->stream);
        cudaMemsetAsync(c->ticket, 0, 256, c->stream);
        cudaMemsetAsync(c->d_spec_flag, 0, 256, c->stream);
        if (c->d_block_sum) cudaMemsetAsync(c->d_block_sum, 0, (c->scratch_chunks / SPAN_BLOCK + 2) * 32, c->stream);
        c->gen = 1;
    }
    p.gen = c->gen;
    p.flags = flags;
    d.utf8 = !(flags & SJB200_FLAG_NO_UTF8);
    int kind = c->kernel_kind;
    const bool auto_kind = kind == SJB200_KERNEL_AUTO;
    if (auto_kind) {
        kind = SJB200_KERNEL_PERSISTENT;
        if (whole_document && !c->scratch_failed && p.alen >= SPLIT_MIN_BYTES) kind = p.alen >= STREAM_MIN_BYTES ? SJB200_KERNEL_STREAM : SJB200_KERNEL_SPLIT;
    }
    if (!whole_document) kind = SJB200_KERNEL_PERSISTENT;   // ranges of a document (streaming host path): look-back across launches
    d.warps = pick_warps(c, p.alen);
    if (kind == SJB200_KERNEL_SPLIT && d.warps != 8 && d.warps != 16) {
        // the split pair exists for 8- and 16-warp tiles only: an explicit shape it does not have is an error, never a silent
        // substitution of another kernel shape
        if (c->forced_warps) {
            if (!auto_kind) return SJB200_UNEXPECTED_ERROR;
            kind = SJB200_KERNEL_PERSISTENT;   // chosen automatically: the persistent kernel has every shape
        } else {
            d.warps = 16;
        }
    }
    if (!valid_warps(d.warps)) return SJB200_UNEXPECTED_ERROR;
    const uint64_t chunks = (p.alen + 2047) / 2048;
    if (kind != SJB200_KERNEL_PERSISTENT) {
        const cudaError_t e = ensure_scratch(c, chunks + 32, c->stream);
        if (e != cudaSuccess) {
            if (!auto_kind) return SJB200_MEMALLOC;   // the caller asked for this organisation explicitly
            c->scratch_failed = true;                 // chosen automatically: the persistent kernel needs no scratch
            kind = SJB200_KERNEL_PERSISTENT;
        }
    }
    d.kind = kind;
    const uint64_t tile = (uint64_t)d.warps * 2048;
    const uint64_t ntiles = (p.alen + tile - 1) / tile;
    if (ntiles > c->max_tiles) return SJB200_CAPACITY;
    p.ntiles = (uint32_t)ntiles;
    p.tile_begin = 0;
    p.tile_end = p.ntiles;
    p.ticket = c->ticket;   // [0],[1] alternate between persistent launches, [3] and [5] serve the stream pipeline
    if (kind != SJB200_KERNEL_PERSISTENT) {
        p.masks = c->d_masks;
        p.carry = c->d_carry;
        p.chunk_sum = c->d_chunk_sum;
        p.block_sum = c->d_block_sum;
    }
    if (kind == SJB200_KERNEL_STREAM) p.spec_flag = c->d_spec_flag;
    return SJB200_SUCCESS;
}

cudaError_t launch_persistent_range(sjb200_ctx *c, const Stage1Params &p, int warps, bool utf8, cudaStream_t stream) {
    const int idx = warps == 24 ? 4 : (warps == 16 ? 3 : (warps == 8 ? 2 : (warps == 4 ? 1 : 0)));
    const int max_ctas = c->sm_count * c->persist_occ[idx];
    switch (warps) {
    case 24: return utf8 ? launch_persist<24, true>(p, stream, max_ctas) : launch_persist<24, false>(p, stream, max_ctas);
    case 16: return utf8 ? launch_persist<16, true>(p, stream, max_ctas) : launch_persist<16, false>(p, stream, max_ctas);
    case 8: return utf8 ? launch_persist<8, true>(p, stream, max_ctas) : launch_persist<8, false>(p, stream, max_ctas);
    case 4: return utf8 ? launch_persist<4, true>(p, stream, max_ctas) : launch_persist<4, false>(p, stream, max_ctas);
    case 2: return utf8 ? launch_persist<2, true>(p, stream, max_ctas) : launch_persist<2, false>(p, stream, max_ctas);
    default: return cudaErrorInvalidValue;   // a shape that is not instantiated is an error, never another shape
    }
}

// launch the tiles [tile_begin, tile_end) of a planned document on `stream`
int32_t launch_range(sjb200_ctx *c, DocPlan &d, uint32_t tile_begin, uint32_t tile_end, uint32_t *progress, cudaStream_t stream) {
    Stage1Params p = d.p;
    p.tile_begin = tile_begin;
    p.tile_end = tile_end;
    p.progress = progress;
    const bool utf8 = d.utf8;
    const bool whole = tile_begin == 0 && tile_end == d.p.ntiles;
    cudaError_t e = cudaSuccess;
    const bool speculating = d.kind == SJB200_KERNEL_STREAM && whole;
    if (speculating) {
        e = utf8 ? launch_stream<true>(c, p, stream, c->sm_count * c->stream_occ) : launch_stream<false>(c, p, stream, c->sm_count * c->stream_occ);
        // ... then the persistent kernel as the exact fallback: returns at once unless a chunk raised the speculation flag
    } else {
        p.spec_flag = nullptr;   // the persistent kernel alone indexes this range
    }
    if (e == cudaSuccess) {
        p.ticket_sel = c->launch_seq & 1u;   // persistent launches alternate two ticket counters
        if (d.kind == SJB200_KERNEL_SPLIT && whole) {
            const int max_ctas = c->sm_count * c->split_occ[d.warps == 16 ? 1 : 0];
            if (d.warps == 16) e = utf8 ? launch_split<16, true>(p, stream, max_ctas) : launch_split<16, false>(p, stream, max_ctas);
            else e = utf8 ? launch_split<8, true>(p, stream, max_ctas) : launch_split<8, false>(p, stream, max_ctas);
            c->launches += 2;
        } else {
            e = launch_persistent_range(c, p, d.warps, utf8, stream);
            c->launches += 1;
        }
    }
    if (e != cudaSuccess) {
        // a half-issued document may leave a ticket counter non-zero or skip the reset of the other one
        cudaMemsetAsync(c->ticket, 0, 256, stream);
        cudaGetLastError();
        return cuda_err(e);
    }
    c->launch_seq++;   // only a launch that really went out flips the ticket counters
    return SJB200_SUCCESS;
}

// enqueue one stage-1 kernel over a whole document; the result lands in result slot `slot`
int32_t enqueue(sjb200_ctx *c, const uint8_t *d_buf, uint64_t len, uint32_t *d_idx, uint64_t cap, uint32_t flags,
                uint32_t slot, int32_t *d_status = nullptr) {
    DocPlan d;
    int32_t rc = plan_document(c, d, d_buf, len, d_idx, cap, flags, slot, d_status);
    if (rc != SJB200_SUCCESS) return rc;
    if (c->timed) cudaEventRecord(c->ev0, c->stream);
    rc = launch_range(c, d, 0, d.p.ntiles, nullptr, c->stream);
    if (c->timed) cudaEventRecord(c->ev1, c->stream);
    return rc;
}

int32_t check_args(sjb200_ctx *c, uint64_t len, uint32_t flags) {
    if (!c) return SJB200_UNINITIALIZED;
    if (len == 0) return SJB200_EMPTY;                 // json_structural_indexer.mojo:91-92
    if (len > 0xFFFFFFFFull || len > c->max_len) return SJB200_CAPACITY;  // :87-89, base.mojo:2
    c->timed = (flags & SJB200_FLAG_TIMING) != 0;
    return SJB200_SUCCESS;
}

// SURVEY.md section 8(f) rank 2 (first half): the byte every structural index points at.  Stage 2 reads
// buffer[next_structural[k]] once per step (reference generic/stage2/json_iterator.mojo:256-262), a dependent random read
// on the CPU; here it is one streaming pass: a thread takes four consecutive indexes (one 16-byte load), fetches the
// four bytes (consecutive structurals are a few bytes apart, so a warp's 128 reads fall into a handful of lines) and
// stores them as one 32-bit word.
__global__ void __launch_bounds__(256) structural_bytes_kernel(const uint8_t *__restrict__ buf, uint32_t len, const uint32_t *__restrict__ idx,
                                                             uint64_t n, uint8_t *__restrict__ out, uint32_t head) {
    // [0, head): scalar until idx and out are 16- / 4-byte aligned together; then groups of four; then a scalar tail
    const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    auto byte_at = [&](uint32_t i) -> uint32_t { return i < len ? (uint32_t)__ldg(buf + i) : 0u; };
    const uint64_t groups = (n - head) / 4;
    if (t < groups) {
        const uint64_t k = head + 4 * t;
        const uint4 i4 = __ldcs(reinterpret_cast<const uint4 *>(idx + k));
        const uint32_t w = byte_at(i4.x) | (byte_at(i4.y) << 8) | (byte_at(i4.z) << 16) | (byte_at(i4.w) << 24);
        __stcs(reinterpret_cast<uint32_t *>(out + k), w);
    } else {
        // the ragged ends: at most `head` + 3 entries, one thread each
        const uint64_t r = t - groups;
        const uint64_t tail0 = head + 4 * groups;
        uint64_t k = n;
        if (r < head) k = r;
        else if (r - head < n - tail0) k = tail0 + (r - head);
        if (k < n) out[k] = (uint8_t)byte_at(idx[k]);
    }
}

// SURVEY.md section 8(f) rank 2 (second half): where top-level documents start in a stream of structurals (NDJSON, or
// any concatenation of documents).  depth(k) = number of '{' '[' minus number of '}' ']' among structurals [0, k); a
// structural with depth(k) == 0 is the first one of a document.  Three launches: per 4096 structurals the sum of the
// +1 / -1 steps; an exclusive scan of those sums by one CTA; then every thread re-walks its 16 structurals from the
// block's depth.  All of it on bytes produced by structural_bytes_kernel.
constexpr int DEPTH_PER_THREAD = 16, DEPTH_THREADS = 256, DEPTH_BLOCK = DEPTH_PER_THREAD * DEPTH_THREADS;

__device__ __forceinline__ int depth_step(uint32_t b) {      // '{' 7B '[' 5B -> +1, '}' 7D ']' 5D -> -1
    const uint32_t low = b | 0x20u;                            // fold [ ] onto { }
    return low == 0x7Bu ? 1 : (low == 0x7Du ? -1 : 0);
}
// loads thread t's 16 bytes of the block (zero beyond n: zero is not a bracket)
__device__ __forceinline__ void depth_load(const uint8_t *bytes, uint64_t n, uint64_t k0, uint32_t w[4]) {
    if ((reinterpret_cast<uintptr_t>(bytes + k0) & 15) == 0 && k0 + 16 <= n) {
        const uint4 v = __ldg(reinterpret_cast<const uint4 *>(bytes + k0));
        w[0] = v.x; w[1] = v.y; w[2] = v.z; w[3] = v.w;
    } else {
#pragma unroll
        for (int q = 0; q < 4; q++) {
            uint32_t x = 0;
#pragma unroll
            for (int j = 0; j < 4; j++) {
                const uint64_t k = k0 + 4 * q + j;
                if (k < n) x |= (uint32_t)__ldg(bytes + k) << (8 * j);
            }
            w[q] = x;
        }
    }
}
__device__ __forceinline__ int block_sum_i32(int v, int *s_w) {   // sum over the CTA's 256 threads, result in every thread
    v = __reduce_add_sync(0xFFFFFFFFu, v);
    if ((threadIdx.x & 31) == 0) s_w[threadIdx.x >> 5] = v;
    __syncthreads();
    int t = 0;
#pragma unroll
    for (int q = 0; q < DEPTH_THREADS / 32; q++) t += s_w[q];
    __syncthreads();
    return t;
}
__global__ void __launch_bounds__(DEPTH_THREADS) depth_block_sums_kernel(const uint8_t *__restrict__ bytes, uint64_t n, int *__restrict__ block_sum) {
    __shared__ int s_w[DEPTH_THREADS / 32];
    const uint64_t k0 = (uint64_t)blockIdx.x * DEPTH_BLOCK + (uint64_t)threadIdx.x * DEPTH_PER_THREAD;
    uint32_t w[4];
    depth_load(bytes, n, k0, w);
    int d = 0;
#pragma unroll
    for (int j = 0; j < 16; j++) d += depth_step((w[j >> 2] >> (8 * (j & 3))) & 0xFFu);
    const int total = block_sum_i32(d, s_w);
    if (threadIdx.x == 0) block_sum[blockIdx.x] = total;
}
// one CTA: block_sum[b] <- depth before block b (exclusive scan, in place)
__global__ void __launch_bounds__(1024) depth_scan_blocks_kernel(int *block_sum, uint32_t nblocks) {
    __shared__ int s_w[32];
    __shared__ int s_carry;
    if (threadIdx.x == 0) s_carry = 0;
    __syncthreads();
    for (uint32_t b0 = 0; b0 < nblocks; b0 += 1024u) {
        const uint32_t b = b0 + threadIdx.x;
        const int v = b < nblocks ? block_sum[b] : 0;
        int incl = v;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int o = __shfl_up_sync(0xFFFFFFFFu, incl, d);
            if ((int)(threadIdx.x & 31) >= d) incl += o;
        }
        if ((threadIdx.x & 31) == 31) s_w[threadIdx.x >> 5] = incl;
        __syncthreads();
        int before_warp = 0;
        for (int q = 0; q < (int)(threadIdx.x >> 5); q++) before_warp += s_w[q];
        const int carry = s_carry;
        if (b < nblocks) block_sum[b] = carry + before_warp + incl - v;
        __syncthreads();
        if (threadIdx.x == 1023) s_carry = carry + before_warp + incl;
        __syncthreads();
    }
}
__global__ void __launch_bounds__(DEPTH_THREADS) depth_starts_kernel(const uint8_t *__restrict__ bytes, uint64_t n, const int *__restrict__ block_depth,
                                                                   uint8_t *__restrict__ starts) {
    __shared__ int s_w[DEPTH_THREADS / 32];
    const uint64_t k0 = (uint64_t)blockIdx.x * DEPTH_BLOCK + (uint64_t)threadIdx.x * DEPTH_PER_THREAD;
    uint32_t w[4];
    depth_load(bytes, n, k0, w);
    int d = 0;
#pragma unroll
    for (int j = 0; j < 16; j++) d += depth_step((w[j >> 2] >> (8 * (j & 3))) & 0xFFu);
    // exclusive prefix of the per-thread sums inside the CTA
    int incl = d;
#pragma unroll
    for (int s = 1; s < 32; s <<= 1) {
        const int o = __shfl_up_sync(0xFFFFFFFFu, incl, s);
        if ((int)(threadIdx.x & 31) >= s) incl += o;
    }
    if ((threadIdx.x & 31) == 31) s_w[threadIdx.x >> 5] = incl;
    __syncthreads();
    int depth = block_depth[blockIdx.x] + incl - d;
    for (int q = 0; q < (int)(threadIdx.x >> 5); q++) depth += s_w[q];
    uint32_t o[4] = {0, 0, 0, 0};
#pragma unroll
    for (int j = 0; j < 16; j++) {
        if (depth == 0) o[j >> 2] |= 1u << (8 * (j & 3));
        depth += depth_step((w[j >> 2] >> (8 * (j & 3))) & 0xFFu);
    }
    if ((reinterpret_cast<uintptr_t>(starts + k0) & 15) == 0 && k0 + 16 <= n) {
        *reinterpret_cast<uint4 *>(starts + k0) = make_uint4(o[0], o[1], o[2], o[3]);
    } else {
        for (int j = 0; j < 16; j++)
            if (k0 + j < n) starts[k0 + j] = (uint8_t)((o[j >> 2] >> (8 * (j & 3))) & 0xFFu);
    }
}

__global__ void split_kernel(const uint8_t *buf, uint64_t len, uint64_t seg_bytes, uint64_t *cuts, uint32_t ncuts) {
    // one warp per cut k: the position after the last '\n' inside (k*seg_bytes, min((k+1)*seg_bytes, len)],
    // or len itself for the final cut; ~0 if that window holds no newline.
    const uint32_t k = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (k >= ncuts) return;
    const uint64_t hi = (uint64_t)(k + 1) * seg_bytes;
    if (hi >= len) {
        if (lane == 0) cuts[k] = len;
        return;
    }
    const uint64_t lo = (uint64_t)k * seg_bytes;
    uint64_t found = ~0ull;
    for (uint64_t end = hi; end > lo;) {
        const uint64_t span = end - lo < 32 ? end - lo : 32;
        const bool hit = (uint64_t)lane < span && buf[end - 1 - lane] == '\n';
        const uint32_t b = __ballot_sync(0xFFFFFFFFu, hit);
        if (b) {
            found = end - (uint64_t)(__ffs((int)b) - 1);  // the byte after the newline
            break;
        }
        end -= span;
    }
    if (lane == 0) cuts[k] = found;
}

}  // namespace

#pragma GCC visibility push(default)
extern "C" {

int32_t sjb200_version(void) { return SJB200_ABI_VERSION; }

int32_t sjb200_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
    return n;
}

int32_t sjb200_ctx_create(int32_t device, uint64_t max_len, uint64_t max_len_host, uint32_t flags, sjb200_ctx **out) {
    (void)flags;
    if (!out) return SJB200_UNINITIALIZED;
    *out = nullptr;
    if (max_len > 0xFFFFFFFFull || max_len_host > max_len) return SJB200_CAPACITY;
    CK(cudaSetDevice(device));
    sjb200_ctx *c = new (std::nothrow) sjb200_ctx();
    if (!c) return SJB200_MEMALLOC;
    c->device = device;
    c->max_len = max_len;
    c->max_len_host = max_len_host;
    cudaError_t e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking);
    c->own_stream = (e == cudaSuccess);
    c->max_tiles = (uint32_t)((max_len + 16 + MIN_TILE - 1) / MIN_TILE + 1);
    if (e == cudaSuccess) e = cudaMalloc(&c->desc, (size_t)c->max_tiles * 8);
    if (e == cudaSuccess) e = cudaMalloc(&c->ticket, 256);
    if (e == cudaSuccess) e = cudaMalloc(&c->d_split, 8 * 4096);
    if (e == cudaSuccess) e = cudaMemset(c->desc, 0, (size_t)c->max_tiles * 8);
    if (e == cudaSuccess) e = cudaMemset(c->ticket, 0, 256);
    if (e == cudaSuccess) e = cudaHostAlloc(&c->h_results, sizeof(Stage1Result) * RESULT_SLOTS, cudaHostAllocMapped);
    if (e == cudaSuccess) e = cudaHostGetDevicePointer(&c->d_results, c->h_results, 0);
    if (e == cudaSuccess && max_len_host) {
        e = cudaMalloc(&c->d_in, (size_t)max_len_host + 256);
        c->d_out_cap = max_len_host + 3;
        if (e == cudaSuccess) e = cudaMalloc(&c->d_out, (size_t)(c->d_out_cap + 4) * 4);
    }
#if SJ_TRACE
    if (e == cudaSuccess) e = cudaMalloc(&c->d_trace, (size_t)c->max_tiles * 16 * 8);
    if (e == cudaSuccess) e = cudaMemset(c->d_trace, 0, (size_t)c->max_tiles * 16 * 8);
#endif
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking);
    for (int k = 0; k < sjb200_ctx::MAX_CHUNKS && e == cudaSuccess; k++) e = cudaEventCreateWithFlags(&c->chunk_ev[k], cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaHostAlloc(&c->h_progress, 4 * sjb200_ctx::MAX_CHUNKS, cudaHostAllocMapped);
    if (e == cudaSuccess) e = cudaHostGetDevicePointer(&c->d_progress, c->h_progress, 0);
    if (e == cudaSuccess) e = cudaEventCreate(&c->ev0);
    if (e == cudaSuccess) e = cudaEventCreate(&c->ev1);
    if (e == cudaSuccess) e = prepare_persist<2>(&c->persist_occ[0]);
    if (e == cudaSuccess) e = prepare_persist<4>(&c->persist_occ[1]);
    if (e == cudaSuccess) e = prepare_persist<8>(&c->persist_occ[2]);
    if (e == cudaSuccess) e = prepare_persist<16>(&c->persist_occ[3]);
    if (e == cudaSuccess) e = prepare_persist<24>(&c->persist_occ[4]);
    if (e == cudaSuccess) e = prepare_split<8>(&c->split_occ[0]);
    if (e == cudaSuccess) e = prepare_split<16>(&c->split_occ[1]);
    if (e == cudaSuccess) e = prepare_stream(&c->stream_occ);
    if (e == cudaSuccess) {
        cudaMemPoolProps props = {};
        props.allocType = cudaMemAllocationTypePinned;
        props.handleTypes = cudaMemHandleTypeNone;
        props.location.type = cudaMemLocationTypeDevice;
        props.location.id = device;
        e = cudaMemPoolCreate(&c->pool, &props);
        if (e == cudaSuccess) {
            uint64_t keep = ~0ull;   // freed blocks stay in the pool: a second call of the same size allocates nothing
            e = cudaMemPoolSetAttribute(c->pool, cudaMemPoolAttrReleaseThreshold, &keep);
        }
    }
    if (e == cudaSuccess) e = cudaMalloc(&c->d_spec_flag, 256);
    if (e == cudaSuccess) e = cudaMemset(c->d_spec_flag, 0, 256);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&c->sm_count, cudaDevAttrMultiProcessorCount, device);
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    if (e != cudaSuccess) {
        const int32_t code = cuda_err(e);
        sjb200_ctx_destroy(c);
        return code;
    }
    memset(c->h_results, 0, sizeof(Stage1Result) * RESULT_SLOTS);
    *out = c;
    return SJB200_SUCCESS;
}

int32_t sjb200_ctx_destroy(sjb200_ctx *c) {
    if (!c) return SJB200_SUCCESS;
    cudaSetDevice(c->device);
    if (c->stream) cudaStreamSynchronize(c->stream);
    cudaFree(c->d_in);
    cudaFree(c->d_out);
    cudaFree(c->desc);
    cudaFree(c->ticket);
    cudaFree(c->d_split);
    cudaFree(c->d_trace);
    cudaFree(c->d_spec_flag);
    if (c->stream) {
        free_scratch(c, c->stream);
        cudaStreamSynchronize(c->stream);
    }
    if (c->h_results) cudaFreeHost(c->h_results);
    if (c->h_progress) cudaFreeHost(c->h_progress);
    for (int k = 0; k < sjb200_ctx::MAX_CHUNKS; k++)
        if (c->chunk_ev[k]) cudaEventDestroy(c->chunk_ev[k]);
    if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
    if (c->ev0) cudaEventDestroy(c->ev0);
    if (c->ev1) cudaEventDestroy(c->ev1);
    if (c->own_stream && c->stream) cudaStreamDestroy(c->stream);
    delete c;
    return SJB200_SUCCESS;
}

int32_t sjb200_ctx_set_stream(sjb200_ctx *c, void *cuda_stream) {
    if (!c) return SJB200_UNINITIALIZED;
    cudaStreamSynchronize(c->stream);
    if (c->own_stream && c->stream) cudaStreamDestroy(c->stream);
    c->stream = reinterpret_cast<cudaStream_t>(cuda_stream);
    c->own_stream = false;
    return SJB200_SUCCESS;
}

int32_t sjb200_ctx_set_kernel(sjb200_ctx *c, int32_t kind) {
    if (!c) return SJB200_UNINITIALIZED;
    if (kind != SJB200_KERNEL_AUTO && kind != SJB200_KERNEL_PERSISTENT && kind != SJB200_KERNEL_SPLIT && kind != SJB200_KERNEL_STREAM)
        return SJB200_UNEXPECTED_ERROR;
    c->kernel_kind = kind;
    return SJB200_SUCCESS;
}

int32_t sjb200_ctx_set_warps(sjb200_ctx *c, int32_t warps) {
    if (!c) return SJB200_UNINITIALIZED;
    if (warps != 0 && !valid_warps(warps)) return SJB200_UNEXPECTED_ERROR;
    c->forced_warps = warps;
    return SJB200_SUCCESS;
}

int32_t sjb200_ctx_reserve(sjb200_ctx *c, uint64_t len, uint32_t flags) {
    if (!c) return SJB200_UNINITIALIZED;
    if (len > 0xFFFFFFFFull || len > c->max_len) return SJB200_CAPACITY;
    CK(cudaSetDevice(c->device));
    (void)flags;                         // (bit 0 once asked for the global UTF-8 parking area; the lanes are parked in shared memory now)
    const cudaError_t e = ensure_scratch(c, (len + 15 + 2047) / 2048 + 32, c->stream);
    if (e != cudaSuccess) return SJB200_MEMALLOC;
    c->scratch_failed = false;
    return SJB200_SUCCESS;
}

int32_t sjb200_ctx_set_chunk_bytes(sjb200_ctx *c, uint64_t bytes) {
    if (!c) return SJB200_UNINITIALIZED;
    if (bytes < 4096) return SJB200_UNEXPECTED_ERROR;
    c->chunk_bytes = bytes;
    return SJB200_SUCCESS;
}

int32_t sjb200_stage1_device_async(sjb200_ctx *c, const uint8_t *d_buf, uint64_t len, uint32_t *d_idx,
                                   uint64_t idx_capacity, uint32_t flags) {
    int32_t rc = check_args(c, len, flags);
    if (rc != SJB200_SUCCESS) {
        if (c) c->pending = false;
        return rc;
    }
    CK(cudaSetDevice(c->device));
    c->slot = (c->slot + 1) % RESULT_SLOTS;
    c->last_flags = flags;
    rc = enqueue(c, d_buf, len, d_idx, idx_capacity, flags, c->slot);
    c->pending = (rc == SJB200_SUCCESS);
    return rc;
}

int32_t sjb200_stage1_finish(sjb200_ctx *c, uint32_t *n_out, uint32_t *n_written_out, int32_t *utf8_err_out) {
    if (!c) return SJB200_UNINITIALIZED;
    if (!c->pending) return SJB200_UNINITIALIZED;
    CK(cudaStreamSynchronize(c->stream));
    c->pending = false;
    const Stage1Result r = c->h_results[c->slot];
    if (r.n_valid && n_out) *n_out = r.n;  // untouched on the reference's early-return paths
    if (n_written_out) *n_written_out = r.n_written;
    if (utf8_err_out) *utf8_err_out = (c->last_flags & SJB200_FLAG_NO_UTF8) ? -1 : r.utf8_error;
    return r.error;
}

int32_t sjb200_stage1_device(sjb200_ctx *c, const uint8_t *d_buf, uint64_t len, uint32_t *d_idx, uint64_t idx_capacity,
                             uint32_t *n_out, int32_t *utf8_err_out, uint32_t flags) {
    const int32_t rc = sjb200_stage1_device_async(c, d_buf, len, d_idx, idx_capacity, flags);
    if (rc != SJB200_SUCCESS) return rc;
    return sjb200_stage1_finish(c, n_out, nullptr, utf8_err_out);
}

int32_t sjb200_stage1(sjb200_ctx *c, const uint8_t *buf, uint64_t len, uint32_t *idx_out, uint64_t idx_capacity,
                      uint32_t *n_out, int32_t *utf8_err_out, uint32_t flags) {
    int32_t rc = check_args(c, len, flags);
    if (rc != SJB200_SUCCESS) return rc;
    if (len > c->max_len_host || !c->d_in) return SJB200_CAPACITY;
    CK(cudaSetDevice(c->device));
    const uint64_t cap = idx_capacity < c->d_out_cap ? idx_capacity : c->d_out_cap;
    c->slot = (c->slot + 1) % RESULT_SLOTS;
    c->last_flags = flags;
    DocPlan d;
    rc = plan_document(c, d, c->d_in, len, c->d_out, cap, flags, c->slot, nullptr, /*whole_document=*/false);  // indexed chunk by chunk
    if (rc != SJB200_SUCCESS) return rc;
    // Streaming: the document goes to the device in chunks of whole tiles; chunk k is indexed by its own launch as soon
    // as it has arrived (same generation: the look-back carries parity and cursor across launches), and its indexes
    // travel back on a second stream while chunk k+1 is still being copied in -- both PCIe directions stay busy.
    const uint64_t tile = (uint64_t)d.warps * 2048;
    uint64_t tiles_per_chunk = c->chunk_bytes / tile;
    if (tiles_per_chunk == 0) tiles_per_chunk = 1;
    uint64_t nchunks = (d.p.ntiles + tiles_per_chunk - 1) / tiles_per_chunk;
    if (nchunks > (uint64_t)sjb200_ctx::MAX_CHUNKS) {
        tiles_per_chunk = (d.p.ntiles + sjb200_ctx::MAX_CHUNKS - 1) / sjb200_ctx::MAX_CHUNKS;
        nchunks = (d.p.ntiles + tiles_per_chunk - 1) / tiles_per_chunk;
    }
    for (uint64_t k = 0; k < nchunks; k++) {
        const uint64_t t0 = k * tiles_per_chunk, t1 = (t0 + tiles_per_chunk < d.p.ntiles) ? t0 + tiles_per_chunk : d.p.ntiles;
        const uint64_t b0 = t0 * tile, b1 = t1 * tile < len ? t1 * tile : len;
        CK(cudaMemcpyAsync(c->d_in + b0, buf + b0, (size_t)(b1 - b0), cudaMemcpyHostToDevice, c->stream));
        c->h_progress[k] = 0;
        rc = launch_range(c, d, (uint32_t)t0, (uint32_t)t1, c->d_progress + k, c->stream);
        if (rc != SJB200_SUCCESS) return rc;
        CK(cudaEventRecord(c->chunk_ev[k], c->stream));
    }
    uint64_t copied = 0;
    for (uint64_t k = 0; k < nchunks; k++) {
        CK(cudaEventSynchronize(c->chunk_ev[k]));
        uint64_t have = *reinterpret_cast<volatile uint32_t *>(&c->h_progress[k]);  // indexes produced so far
        if (k + 1 == nchunks) {
            const Stage1Result r = c->h_results[c->slot];
            have = r.n_valid ? (uint64_t)r.n + 3 : r.n_written;                      // the trailer travels with the last chunk
        }
        if (have > cap) have = cap;
        if (have > copied) {
            CK(cudaMemcpyAsync(idx_out + copied, c->d_out + copied, (size_t)(have - copied) * 4, cudaMemcpyDeviceToHost,
                               c->copy_stream));
            copied = have;
        }
    }
    CK(cudaStreamSynchronize(c->copy_stream));
    const Stage1Result r = c->h_results[c->slot];
    if (r.n_valid && n_out) *n_out = r.n;
    if (utf8_err_out) *utf8_err_out = (flags & SJB200_FLAG_NO_UTF8) ? -1 : r.utf8_error;
    // the document and its index array stay resident: sjb200_stage2 walks them without another copy
    c->resident_len = (r.error == SJB200_SUCCESS || r.error == SJB200_UTF8_ERROR) && r.n_valid ? len : 0;
    c->resident_n = c->resident_len ? r.n : 0;
    return r.error;
}

int32_t sjb200_sync(sjb200_ctx *c) {
    if (!c) return SJB200_UNINITIALIZED;
    CK(cudaStreamSynchronize(c->stream));
    return SJB200_SUCCESS;
}

float sjb200_last_elapsed_ms(sjb200_ctx *c) {
    if (!c || !c->timed) return -1.0f;
    float ms = -1.0f;
    if (cudaEventSynchronize(c->ev1) != cudaSuccess) return -1.0f;
    if (cudaEventElapsedTime(&ms, c->ev0, c->ev1) != cudaSuccess) return -1.0f;
    return ms;
}

uint64_t sjb200_launch_count(sjb200_ctx *c) { return c ? c->launches : 0; }

// debug builds (-DSJ_TRACE=1) only: copies the per-tile timestamp trace (16 x u64 per tile) of the last launch
int32_t sjb200_debug_trace(sjb200_ctx *c, uint64_t *host_out, uint64_t n_words) {
    if (!c || !c->d_trace) return SJB200_UNINITIALIZED;
    CK(cudaStreamSynchronize(c->stream));
    CK(cudaMemcpy(host_out, c->d_trace, (size_t)n_words * 8, cudaMemcpyDeviceToHost));
    return SJB200_SUCCESS;
}

int32_t sjb200_pinned_alloc(uint64_t bytes, void **p) {
    if (!p) return SJB200_UNINITIALIZED;
    CK(cudaHostAlloc(p, (size_t)bytes, cudaHostAllocDefault));
    return SJB200_SUCCESS;
}
int32_t sjb200_pinned_free(void *p) {
    CK(cudaFreeHost(p));
    return SJB200_SUCCESS;
}
int32_t sjb200_device_alloc(sjb200_ctx *c, uint64_t bytes, void **p) {
    if (!c || !p) return SJB200_UNINITIALIZED;
    CK(cudaSetDevice(c->device));
    CK(cudaMalloc(p, (size_t)bytes));
    return SJB200_SUCCESS;
}
int32_t sjb200_device_free(sjb200_ctx *c, void *p) {
    if (!c) return SJB200_UNINITIALIZED;
    CK(cudaSetDevice(c->device));
    CK(cudaFree(p));
    return SJB200_SUCCESS;
}
int32_t sjb200_copy_to_device(sjb200_ctx *c, void *d_dst, const void *h_src, uint64_t bytes) {
    if (!c) return SJB200_UNINITIALIZED;
    CK(cudaMemcpyAsync(d_dst, h_src, (size_t)bytes, cudaMemcpyHostToDevice, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    return SJB200_SUCCESS;
}
int32_t sjb200_copy_to_host(sjb200_ctx *c, void *h_dst, const void *d_src, uint64_t bytes) {
    if (!c) return SJB200_UNINITIALIZED;
    CK(cudaMemcpyAsync(h_dst, d_src, (size_t)bytes, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    return SJB200_SUCCESS;
}

int32_t sjb200_batch_split_host(const uint8_t *buf, uint64_t len, uint64_t seg_bytes, uint64_t *seg_offsets,
                                uint32_t max_segments, uint32_t *n_segments) {
    // same rule as split_kernel: nominal cuts at multiples of seg_bytes, each moved left to a line start
    if (!seg_offsets || !n_segments || seg_bytes == 0 || seg_bytes > 0x7FFFFFFFull) return SJB200_CAPACITY;
    const uint64_t ncuts = (len + seg_bytes - 1) / seg_bytes;
    if (ncuts > max_segments) return SJB200_CAPACITY;
    uint32_t n = 0;
    seg_offsets[0] = 0;
    for (uint64_t k = 0; k < ncuts; k++) {
        const uint64_t hi = (k + 1) * seg_bytes, lo = k * seg_bytes;
        uint64_t cut;
        if (hi >= len) {
            cut = len;
        } else {
            uint64_t p = hi;
            while (p > lo && buf[p - 1] != '\n') p--;
            if (p == lo) return SJB200_CAPACITY;  // no newline inside a whole nominal segment
            cut = p;
        }
        if (cut > seg_offsets[n]) seg_offsets[++n] = cut;
    }
    *n_segments = n;
    return SJB200_SUCCESS;
}

int32_t sjb200_structural_bytes_device_async(sjb200_ctx *c, const uint8_t *d_buf, uint64_t len, const uint32_t *d_idx, uint64_t n,
                                             uint8_t *d_bytes) {
    if (!c || (n && (!d_buf || !d_idx || !d_bytes))) return SJB200_UNINITIALIZED;
    if (len > 0xFFFFFFFFull) return SJB200_CAPACITY;
    if (n == 0) return SJB200_SUCCESS;
    CK(cudaSetDevice(c->device));
    // entries before the first position where idx is 16-byte aligned; the vector path also needs out + head 4-byte aligned
    uint32_t head = (uint32_t)(((16 - (reinterpret_cast<uintptr_t>(d_idx) & 15)) & 15) / 4);
    if (head > n) head = (uint32_t)n;
    const bool vec_ok = ((reinterpret_cast<uintptr_t>(d_bytes) + head) & 3) == 0;
    if (!vec_ok) head = (uint32_t)(n < 0xFFFFFFFFull ? n : 0);   // misaligned pair of buffers: everything on the scalar path
    if (!vec_ok && n >= 0xFFFFFFFFull) return SJB200_CAPACITY;
    const uint64_t groups = (n - head) / 4;
    const uint64_t threads = groups + head + ((n - head) - 4 * groups);
    structural_bytes_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, c->stream>>>(d_buf, (uint32_t)len, d_idx, n, d_bytes, head);
    c->launches++;
    return cuda_err(cudaGetLastError());
}

int32_t sjb200_document_starts_device_async(sjb200_ctx *c, const uint8_t *d_bytes, uint64_t n, uint8_t *d_starts, int32_t *d_scratch,
                                            uint64_t scratch_entries) {
    if (!c || (n && (!d_bytes || !d_starts || !d_scratch))) return SJB200_UNINITIALIZED;
    if (n == 0) return SJB200_SUCCESS;
    const uint64_t nblocks = (n + DEPTH_BLOCK - 1) / DEPTH_BLOCK;
    if (nblocks > scratch_entries || nblocks > 0x7FFFFFFFull) return SJB200_CAPACITY;
    CK(cudaSetDevice(c->device));
    depth_block_sums_kernel<<<(unsigned)nblocks, DEPTH_THREADS, 0, c->stream>>>(d_bytes, n, d_scratch);
    depth_scan_blocks_kernel<<<1, 1024, 0, c->stream>>>(d_scratch, (uint32_t)nblocks);
    depth_starts_kernel<<<(unsigned)nblocks, DEPTH_THREADS, 0, c->stream>>>(d_bytes, n, d_scratch, d_starts);
    c->launches += 3;
    return cuda_err(cudaGetLastError());
}

int32_t sjb200_batch_split_device(sjb200_ctx *c, const uint8_t *d_buf, uint64_t len, uint64_t seg_bytes,
                                  uint64_t *seg_offsets, uint32_t max_segments, uint32_t *n_segments) {
    if (!c) return SJB200_UNINITIALIZED;
    if (!seg_offsets || !n_segments || seg_bytes == 0 || seg_bytes > 0x7FFFFFFFull) return SJB200_CAPACITY;
    CK(cudaSetDevice(c->device));
    // nominal boundaries at multiples of seg_bytes, each moved left to the nearest line start
    const uint64_t ncuts64 = (len + seg_bytes - 1) / seg_bytes;
    if (ncuts64 > max_segments || ncuts64 > 4096) return SJB200_CAPACITY;
    const uint32_t ncuts = (uint32_t)ncuts64;
    if (ncuts == 0) {
        seg_offsets[0] = 0;
        *n_segments = 0;
        return SJB200_SUCCESS;
    }
    split_kernel<<<(ncuts + 3) / 4, 128, 0, c->stream>>>(d_buf, len, seg_bytes, c->d_split, ncuts);
    c->launches++;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(seg_offsets + 1, c->d_split, (size_t)ncuts * 8, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    seg_offsets[0] = 0;
    uint32_t n = 0;
    for (uint32_t k = 1; k <= ncuts; k++) {
        if (seg_offsets[k] == ~0ull) return SJB200_CAPACITY;  // no newline inside a whole nominal segment
        if (seg_offsets[k] > seg_offsets[n]) seg_offsets[++n] = seg_offsets[k];
    }
    *n_segments = n;
    return SJB200_SUCCESS;
}

int32_t sjb200_batch_run_device_async(sjb200_ctx *c, const uint8_t *d_buf, const uint64_t *seg_offsets, uint32_t first,
                                      uint32_t count, uint32_t *d_idx, const uint64_t *idx_offsets, uint64_t idx_capacity,
                                      int32_t *d_status, uint32_t flags) {
    if (!c) return SJB200_UNINITIALIZED;
    if (count > RESULT_SLOTS) return SJB200_CAPACITY;
    CK(cudaSetDevice(c->device));
    c->timed = false;
    int32_t worst = SJB200_SUCCESS;
    for (uint32_t i = 0; i < count; i++) {
        const uint32_t s = first + i;
        const uint64_t beg = seg_offsets[s], end = seg_offsets[s + 1], len = end - beg;
        int32_t rc;
        const uint64_t next = (i + 1 < count) ? idx_offsets[s + 1] : idx_capacity;
        if (len == 0) rc = SJB200_EMPTY;
        else if (len > 0xFFFFFFFFull || len > c->max_len || next <= idx_offsets[s] || next > idx_capacity) rc = SJB200_CAPACITY;
        else rc = enqueue(c, d_buf + beg, len, d_idx + idx_offsets[s], next - idx_offsets[s], flags, i,
                          d_status ? d_status + 2 * i : nullptr);
        c->launch_rc[i] = rc;   // host-side launch status of this slot; the device-written slot itself is never touched here
        if (rc != SJB200_SUCCESS) {
            if (d_status) {
                const int32_t pair[2] = {rc, 0};
                cudaMemcpyAsync(d_status + 2 * i, pair, sizeof pair, cudaMemcpyHostToDevice, c->stream);
            }
            if (rc > worst) worst = rc;
        }
    }
    return worst;
}

int32_t sjb200_batch_run_device(sjb200_ctx *c, const uint8_t *d_buf, const uint64_t *seg_offsets, uint32_t first,
                                uint32_t count, uint32_t *d_idx, const uint64_t *idx_offsets, uint64_t idx_capacity,
                                uint32_t *seg_counts, int32_t *seg_errors, int32_t *seg_utf8, uint32_t flags) {
    if (!c) return SJB200_UNINITIALIZED;
    int32_t worst = sjb200_batch_run_device_async(c, d_buf, seg_offsets, first, count, d_idx, idx_offsets, idx_capacity,
                                                  nullptr, flags);
    if (worst == SJB200_UNINITIALIZED) return worst;
    if (count > RESULT_SLOTS) return SJB200_CAPACITY;
    CK(cudaStreamSynchronize(c->stream));
    worst = SJB200_SUCCESS;
    for (uint32_t i = 0; i < count; i++) {
        const uint32_t s = first + i;
        Stage1Result r = c->h_results[i];
        const bool launched = c->launch_rc[i] == SJB200_SUCCESS;
        if (!launched) {   // nothing ran for this segment: the slot holds an older result
            r.error = c->launch_rc[i];
            r.n_valid = 0;
        }
        if (seg_errors) seg_errors[s] = r.error;
        if (seg_counts) seg_counts[s] = r.n_valid ? r.n : 0;
        if (seg_utf8) seg_utf8[s] = (!launched || (flags & SJB200_FLAG_NO_UTF8)) ? -1 : r.utf8_error;
        if (r.error > worst) worst = r.error;
    }
    return worst;
}

}  // extern "C"
#pragma GCC visibility pop

#include "batch_driver.cuh"
#include "stage2_primitives.cuh"
#include "stage2_tape.cuh"
#include "stage2_pointer.cuh"
#include "stage2_columns.cuh"
