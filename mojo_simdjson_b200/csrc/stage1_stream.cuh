// stage1_stream.cuh -- stage 1 of a large, device-resident document as a pipeline of three stream-ordered launches with no
// waiting between warps, CTAs or launches other than stream order (and programmatic dependent launch between them):
//
//   stream_classify : every warp is its own pipeline.  A warp draws runs of 4 consecutive 2 KiB chunks from an atomic
//                     counter, each chunk fetched with its own bulk copy (cp.async.bulk, DEPTH chunks in flight per warp, one
//                     mbarrier each) together with the 32 bytes before it, which decide the escape / scalar carries
//                     entering the chunk.  Output per chunk: the two structural mask planes (string state entering the
//                     chunk unknown -> one plane per parity) and a 16-byte summary {count0, count1, flags}.  At most 8
//                     lanes per chunk with bytes >= 0x80 park their bit planes in the warp's shared-memory slots and are
//                     validated 32 at a time at the end of the run (instead of one warp per lane).
//   span_scan       : one CTA per 4096 chunk summaries: ordered (non-commutative span_concat) local reduction -> block
//                     aggregate, published; the aggregates of the earlier blocks -> one carry word per chunk (bit 63 =
//                     starts inside a string, bits 0..39 = rank of its first index) and the verdict.
//   flatten         : stage1_flatten2_kernel (stage1_split.cuh), one warp per unit of two chunks.
//
// The carries a 32-byte look-behind cannot decide are the escape state after a backslash run that covers all of it and the
// scalar state after a quote preceded by 31 backslashes.  A chunk that sees either walks back through global memory
// until the run ends (backslash_run_global, up to WALK_MAX = 64 KiB).  Only a run longer than that raises `spec_flag`
// (stores the document generation); the later launches then do nothing and the persistent kernel, enqueued behind them
// with Stage1Params::spec_flag set, redoes the document exactly.  Otherwise that kernel returns at once.  Results are
// identical either way.
//
// Overlapping classify (ALU pipe) with flatten (shared memory / XU) was measured in round 2 -- windows on two streams, and
// the two kernels side by side with no dependency at all as an upper bound -- and is worth 2 % at best: the pass as a
// whole is bound by instruction issue (profiles/r2_overlap_experiments.txt).
// Reference: json_structural_indexer.mojo:83-186 (step / next / finish), restated in oracle/stage1_oracle.c.
#pragma once
#include "stage1_split.cuh"

namespace sjb200 {

#if defined(__CUDACC__)

// streaming stores: the planes of a large document do not fit the L2 anyway
__device__ __forceinline__ void st_mask(uint64_t *p, uint64_t v) { __stcs(reinterpret_cast<unsigned long long *>(p), (unsigned long long)v); }

// One thread draws from the chunk counter.  Plain PTX: atomicAdd() makes the compiler aggregate over the active lanes (vote,
// elect, shuffle), and that shuffle waits for the atomic at once -- here its result is not needed before the next run.
__device__ __forceinline__ uint32_t ticket_draw(uint32_t *counter, uint32_t n) {
    uint32_t old;
    asm volatile("atom.global.add.u32 %0, [%1], %2;" : "=r"(old) : "l"(counter), "r"(n) : "memory");
    return old;
}

template <int NW>
struct StreamCfg {
    static constexpr int THREADS = NW * 32;
    static constexpr int DEPTH = 2;                         // chunks in flight per warp
    static constexpr int HALO = 32;
    static constexpr int BUF = 2048 + HALO;                 // 16-byte multiple
    static constexpr int PARK = 32 * 80;                    // 32 parked UTF-8 lanes of 80 B per warp; validated when fewer than U8_DEFER_MAX slots are left
    static constexpr int WARP_BYTES = DEPTH * BUF + PARK;
    static constexpr int SMEM_BYTES = NW * WARP_BYTES;
    static constexpr int MAXREG = 64;
};

// phase 1 input of one lane from the warp's private buffer; `chunk` is the shared-space address of the chunk's first byte, HALO
// bytes before it are the preceding input (chunk > 0).  `edge`: first chunk, or a last chunk that is not full.
// `follows`: this warp has just processed chunk c - 1, whose carries out (`prev_tail`: bit 0 escaped, bit 1 scalar) are exact:
// no look-behind needed (three of the four chunks of a run).
__device__ __forceinline__ uint4 lds_u4(uint32_t a) {
    uint4 v;
    asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a) : "memory");
    return v;
}
__device__ __forceinline__ uint32_t lds_u32(uint32_t a) {
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a) : "memory");
    return v;
}
__device__ __forceinline__ uint32_t lds_u8(uint32_t a) {
    uint32_t v;
    asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(a) : "memory");
    return v;
}
template <bool UTF8>
__device__ __forceinline__ void chunk_load(LaneInput &in, uint32_t chunk /* shared-space address of the chunk's first byte */, int lane, uint32_t c, bool edge,
                                           bool is_last, uint32_t last_bytes, const Stage1Params &P, bool follows, uint32_t prev_tail, uint32_t &unresolved) {
    in.g0 = (int64_t)c * 2048 + lane * 64;
    const uint32_t src = chunk + (uint32_t)lane * 64u;
#pragma unroll
    for (int q = 0; q < 4; q++) {
        const uint4 v = lds_u4(src + 16u * q);
        in.w[4 * q + 0] = v.x;
        in.w[4 * q + 1] = v.y;
        in.w[4 * q + 2] = v.z;
        in.w[4 * q + 3] = v.w;
    }
    in.prev = UTF8 ? lds_u32(src - 4u) : 0u;
    // the document may end exactly with this lane's last byte (also when the last chunk is full: not an "edge" chunk then)
    in.ends = is_last && ((uint32_t)lane * 64u + 64u == last_bytes);
    if (edge) {  // bytes outside [mis, alen) read as 0x20 (reference tail padding)
        const int64_t alen = (int64_t)P.alen;
#pragma unroll
        for (int k = 0; k < 16; k++) in.w[k] = mask_word(in.w[k], in.g0 + 4 * k, (int64_t)P.mis, alen);
        if (UTF8) in.prev = (in.g0 == 0) ? 0x20202020u : mask_word(in.prev, in.g0 - 4, (int64_t)P.mis, alen);
    }
    PrevState st = {0, 0, 0};
    if (follows) {
        st.e = prev_tail & 1u;
        st.p = (prev_tail >> 1) & 1u;
    } else if (c > 0) {  // 32 bytes of look-behind, all inside the document (c >= 1, mis < 16)
        const uint32_t b = lds_u8(chunk - 1u - (uint32_t)lane);
        const uint32_t bsm = __ballot_sync(0xFFFFFFFFu, b == 0x5Cu);
        const uint32_t c1 = __shfl_sync(0xFFFFFFFFu, b, 0);
        st = prev_state(bsm, 32, c1);
    }
    unresolved = st.unresolved;
    in.wst = st;
}

// ---------------------------------------------------------------------------------------------
// Long backslash runs.  The escape state entering a chunk (and the "previous byte is a non-quote scalar" state after a
// quote) follows from the parity of the backslash run that ends at the chunk boundary.  32 bytes of look-behind decide
// it unless the run fills them; then the warp walks back through global memory, 512 bytes per step (the bytes were
// just read by a neighbouring warp: L2 hits), up to WALK_MAX bytes.  Only a longer run -- kilobytes of nothing but
// backslashes -- raises spec_flag and costs the document a second, exact pass (stage1_persistent.cuh).
// Reference: the carry `next_is_escaped` of json_escape_scanner.mojo:13,31, resolved without a serial dependency.
// ---------------------------------------------------------------------------------------------
constexpr uint32_t WALK_MAX = 64u << 10;
__device__ __forceinline__ uint32_t ld_acquire_u32(const uint32_t *p) {
    uint32_t v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_u32(uint32_t *p, uint32_t v) {
    asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint4 ld_cg_u4(const void *p) {
    uint4 v;
    asm volatile("ld.global.cg.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p) : "memory");
    return v;
}
// Length of the backslash run that ends just before aligned coordinate `end` (a multiple of 16), walking back through
// global memory 512 bytes per step; bytes before the document start (coordinate < mis) end the run.  `skip` = 1: the byte
// at end-1 is not part of the question (it is the quote whose escapedness is asked) and the run ends at end-2.
// Returns false if the run is longer than max_bytes.
__device__ __forceinline__ bool backslash_run_global(const uint8_t *abase, uint64_t end, uint32_t mis, uint32_t skip, int lane,
                                                     uint32_t max_bytes, uint32_t &run_out) {
    uint32_t run = 0;
    for (uint32_t step = 0; step * 512u < max_bytes + 512u; step++) {
        const int64_t pos = (int64_t)end - 512ll * step - 16ll * (lane + 1);   // lane 0 holds the 16 bytes nearest to `end`
        uint32_t w[4] = {0u, 0u, 0u, 0u};
        if (pos >= 0) {
            const uint4 v = ld_cg_u4(abase + pos);
            w[0] = v.x; w[1] = v.y; w[2] = v.z; w[3] = v.w;
        }
        // t = number of consecutive backslashes counted from byte 15 downwards
        uint32_t t = 0;
        bool open = true;
#pragma unroll
        for (int k = 15; k >= 0; k--) {
            uint32_t b = (w[k >> 2] >> (8 * (k & 3))) & 0xFFu;
            if (skip && step == 0 && lane == 0 && k == 15) b = 0x5Cu;
            if (pos + k < (int64_t)mis) b = 0u;
            open = open && (b == 0x5Cu);
            t += open ? 1u : 0u;
        }
        const uint32_t brk = __ballot_sync(0xFFFFFFFFu, t != 16u);
        if (brk) {
            const int first = __ffs((int)brk) - 1;
            run += 16u * (uint32_t)first + __shfl_sync(0xFFFFFFFFu, t, first);
            run_out = run - skip;
            return true;
        }
        run += 512u;
    }
    run_out = 0;
    return false;
}


// Resolves the carries chunk_load left open (`unresolved`, warp-uniform).  Returns false if a run exceeds WALK_MAX: the
// caller raises spec_flag.  Once the flag is up the document is going to be redone anyway: no further walks.
__device__ __forceinline__ bool resolve_long_runs(const Stage1Params &P, uint32_t c, uint32_t unresolved, int lane, PrevState &wst) {
    if (*reinterpret_cast<volatile uint32_t *>(P.spec_flag) == P.gen) return true;
    uint32_t run;
    if (unresolved & 1u) {
        if (!backslash_run_global(P.abase, (uint64_t)c * 2048u, P.mis, 0u, lane, WALK_MAX, run)) return false;
        wst.e = run & 1u;
    }
    if (unresolved & 2u) {
        if (!backslash_run_global(P.abase, (uint64_t)c * 2048u, P.mis, 1u, lane, WALK_MAX, run)) return false;
        wst.p = run & 1u;
    }
    return true;
}

// Chunks are handed out dynamically, TICKET_CHUNKS consecutive chunks per draw from P.ticket[3] (zero at launch; the scan
// kernel that follows resets it).  A static partition would be slightly cheaper but assumes that every CTA of the grid is
// resident from the start: with another kernel on the device (the NCCL verdict exchange of the previous pass, a second
// context) a displaced CTA would start only when some other CTA has finished its whole share, doubling the kernel time.
constexpr uint32_t TICKET_CHUNKS = 4;
constexpr uint32_t NO_CHUNK = 0xFFFFFFFFu;

// validates the `parked` lanes a warp left in its shared-memory slots (80 B each: 16 bit-plane words, the 4 bytes before the
// lane, its end-of-document bit), one thread per lane: the same lead / continuation / range algebra as the inline path,
// now with every lane of the warp doing useful work
__device__ __forceinline__ bool validate_parked_lanes(const uint8_t *park, uint32_t parked, int lane) {
    bool bad = false;
    if ((uint32_t)lane < parked) {
        const uint4 *s = reinterpret_cast<const uint4 *>(park) + 5 * lane;
        const uint4 a = s[0], bb = s[1], d = s[2], e = s[3], f = s[4];
        const uint32_t pl[8] = {a.x, a.y, a.z, a.w, bb.x, bb.y, bb.z, bb.w};
        const uint32_t ph[8] = {d.x, d.y, d.z, d.w, e.x, e.y, e.z, e.w};
        Utf8Pre32 ul, uh;
        utf8_pre32(pl, ul);
        utf8_pre32(ph, uh);
        const Utf8Carry uc = utf8_carry_from_prev_word(f.x);
        uint32_t tail_must;
        const uint64_t ue = utf8_errors64(ul, uh, uc, &tail_must);
        bad = (ue != 0) || (f.y != 0 && tail_must != 0);
    }
    return __any_sync(0xFFFFFFFFu, bad);
}

// chunks [chunk_begin, chunk_end) of the document (chunk_begin a multiple of TICKET_CHUNKS; the pipeline passes the whole document)
//
// Ring of DEPTH private buffers per warp.  The bookkeeping (which chunk sits in which buffer, the run being worked on, the
// next run) is kept in registers by ALL lanes -- straight-line, warp-uniform code; only the bulk copy itself and the atomic
// draw are issued by lane 0.  A chunk number >= chunk_end means "nothing more": tickets only grow, so once a buffer holds
// such a number every later one does too, and no copy is outstanding when the warp leaves.
template <int NW, bool UTF8>
__global__ void __launch_bounds__(NW * 32) __maxnreg__(StreamCfg<NW>::MAXREG) stage1_stream_classify_kernel(const Stage1Params P, uint32_t nchunks,
                                                                                                            uint32_t chunk_begin, uint32_t chunk_end,
                                                                                                            const uint8_t *src0 /* P.abase - HALO */) {
    using Cfg = StreamCfg<NW>;
    constexpr int DEPTH = Cfg::DEPTH;
    static_assert(U8_DEFER_MAX <= 32, "a chunk must not park more lanes than the warp's slots hold");
    extern __shared__ __align__(128) uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t s_bar[NW * DEPTH];
    // the lane number is read once (volatile: the compiler would otherwise re-derive it from %tid inside the loop, a
    // long-latency special-register read in front of dependent instructions each time)
    int lane;
    asm volatile("mov.u32 %0, %%laneid;" : "=r"(lane));
    const uint32_t lt = lanemask_lt();
    const int warp = threadIdx.x >> 5;
    uint8_t *wbase = smem_raw + warp * Cfg::WARP_BYTES;
    const uint32_t buf0 = smem_u32(wbase);                    // shared-space addresses: 32-bit arithmetic only
    uint8_t *park = wbase + DEPTH * Cfg::BUF;                 // parked UTF-8 lanes of the current run
    const uint32_t bar0 = smem_u32(&s_bar[warp * DEPTH]);
    uint32_t *ticket = P.ticket + 3, *exits = P.ticket + 5;
    // every chunk is 2048 bytes except possibly the last one; every chunk but chunk 0 has HALO bytes of look-behind
    const uint32_t last = nchunks - 1u;
    const uint32_t last_bytes = (uint32_t)(P.alen - (uint64_t)last * 2048u);   // 1 .. 2048
    const uint32_t last_tx = (last_bytes + 15u) & ~15u;                        // stays inside the last 16-byte line of the data
    const bool last_partial = last_bytes < 2048u;

    // The first run of every warp is fixed (warp g: chunks 4g .. 4g+3 of the window), so that a launch does not begin with
    // thousands of atomics on one address; the counter hands out the runs after those.  The draw for the run after the
    // current one is always in flight (lane 0 holds its result), so the atomic's latency is never waited for.
    grid_dependency_wait();   // launched while the previous kernel of the stream drains: nothing global is touched before this
    // (Runs that shrink to single chunks towards the end of the range were measured: no gain, 1 GiB and 64 MiB alike.)
    const uint32_t t_base = chunk_begin + gridDim.x * NW * TICKET_CHUNKS;
    uint32_t t_cur = chunk_begin + (blockIdx.x * NW + warp) * TICKET_CHUNKS, t_left = TICKET_CHUNKS;
    uint32_t drawn = lane == 0 ? ticket_draw(ticket, TICKET_CHUNKS) : 0u;      // lane 0: the run after this one (relative to t_base)
    auto next_chunk = [&]() -> uint32_t {   // warp-uniform
        if (t_left == 0u) {
            t_cur = t_base + __shfl_sync(0xFFFFFFFFu, drawn, 0);
            t_left = TICKET_CHUNKS;
            if (lane == 0) drawn = ticket_draw(ticket, TICKET_CHUNKS);
        }
        t_left--;
        return t_cur++;
    };
    // lane 0: start the bulk copy of chunk c (< chunk_end) and its look-behind into buffer b
    auto issue = [&](int b, uint32_t c) {
        const uint32_t bar = bar0 + 8u * b, dst = buf0 + b * Cfg::BUF;
        if (c - 1u < last - 1u) {   // 0 < c < last: the common case, constant size
            mbar_expect_tx(bar, 2048u + Cfg::HALO);
            bulk_load(dst, src0 + (size_t)c * 2048u, 2048u + Cfg::HALO, bar);   // src0 = P.abase - HALO
        } else {
            const uint32_t halo = c > 0u ? (uint32_t)Cfg::HALO : 0u;
            const uint32_t tx = (c == last ? last_tx : 2048u) + halo;
            mbar_expect_tx(bar, tx);
            bulk_load(dst + Cfg::HALO - halo, P.abase + (size_t)c * 2048u - halo, tx, bar);
        }
    };
    uint32_t held[DEPTH];          // the chunk each buffer holds (all lanes)
    if (lane == 0) {
        for (int b = 0; b < DEPTH; b++) mbar_init(bar0 + 8 * b, 1);
        fence_mbar_init();
    }
    __syncwarp();
#pragma unroll
    for (int b = 0; b < DEPTH; b++) {
        held[b] = next_chunk();
        const bool more = held[b] < chunk_end;
        if (more && lane == 0) issue(b, held[b]);
    }
    uint32_t phase = 0;
    uint32_t parked = 0;           // lanes parked in `park` during the current run
    bool u8_bad = false;
    uint32_t prev_c = NO_CHUNK - 1u, prev_tail = 0;   // the chunk this warp processed last and its carries out
    bool done = false;
    while (!done) {
#pragma unroll
        for (int b = 0; b < DEPTH; b++) {   // static buffer index: no address arithmetic on it
            const uint32_t c = held[b];
            if (c >= chunk_end) {
                done = true;
                break;
            }
            mbar_wait(bar0 + 8 * b, phase);
            LanePhase1 ph;
            {
                LaneInput in;
                uint32_t unresolved;
                const bool edge = (c == 0u) || (c == last && last_partial);
                chunk_load<UTF8>(in, buf0 + b * Cfg::BUF + Cfg::HALO, lane, c, edge, c == last, last_bytes, P, c == prev_c + 1u, prev_tail, unresolved);
                __syncwarp();  // every lane has its bytes in registers: the buffer can be refilled
                held[b] = next_chunk();
                const bool more = held[b] < chunk_end;   // (decided by all lanes: chunk_end sits in a uniform register)
                if (more && lane == 0) issue(b, held[b]);
                if (unresolved && !resolve_long_runs(P, c, unresolved, lane, in.wst) && lane == 0)
                    *P.spec_flag = P.gen;   // someone else has to do this document (see the header)
                warp_compute<UTF8, 1>(ph, in, lane, P, reinterpret_cast<uint4 *>(park) + 5 * parked, lt);
                parked += (uint32_t)__popc(ph.u8_lanes);
                prev_c = c;
                prev_tail = ph.tail;
            }
            uint64_t *mp = P.masks + (size_t)c * 64 + lane;
            st_mask(mp, ph.m0);
            st_mask(mp + 32, ph.m1);
            if (lane == 0) reinterpret_cast<uint4 *>(P.chunk_sum)[c] = make_uint4(ph.wc0, ph.wc1, ph.wflags, 0u);
            if (UTF8 && parked > 32u - U8_DEFER_MAX) {
                // the next chunk might not find room: the lanes whose validation was deferred, up to 32 at a time
                __syncwarp();
                u8_bad |= validate_parked_lanes(park, parked, lane);
                parked = 0;
                __syncwarp();
            }
        }
        phase ^= 1u;
    }
    if (UTF8 && parked) {   // the lanes still parked when the warp runs out of chunks
        __syncwarp();
        u8_bad |= validate_parked_lanes(park, parked, lane);
    }
    // a violation among the deferred lanes: the document's last launch folds it into the verdict (stage1_persistent.cuh)
    if (UTF8 && u8_bad && lane == 0) P.spec_flag[1] = P.gen;
    // the last CTA to leave frees the chunk counter for the next launch
    __syncthreads();
    if (threadIdx.x == 0 && atomicAdd(exits, 1u) == gridDim.x - 1u) {
        *ticket = 0;
        *exits = 0;
    }
}

// ---------------------------------------------------------------------------------------------
// ordered scan of chunk summaries (SPAN_BLOCK = 4096 per CTA, four consecutive ones per thread)
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ SpanAcc span_from_summary(const uint4 s) {
    SpanAcc a;
    a.par = s.z & 1u;
    a.c[0] = s.x;
    a.c[1] = s.y;
    a.un[0] = (s.z >> 1) & 1u;
    a.un[1] = (s.z >> 2) & 1u;
    a.u8 = (s.z >> 3) & 1u;
    return a;
}
__device__ __forceinline__ uint32_t span_flags(const SpanAcc &a) { return (a.par & 1u) | (a.un[0] << 1) | (a.un[1] << 2) | (a.u8 << 3); }
__device__ __forceinline__ SpanAcc span_shfl_up(const SpanAcc &a, int d) {
    SpanAcc r;
    r.c[0] = __shfl_up_sync(0xFFFFFFFFu, a.c[0], d);
    r.c[1] = __shfl_up_sync(0xFFFFFFFFu, a.c[1], d);
    const uint32_t f = __shfl_up_sync(0xFFFFFFFFu, span_flags(a), d);
    r.par = f & 1u;
    r.un[0] = (f >> 1) & 1u;
    r.un[1] = (f >> 2) & 1u;
    r.u8 = (f >> 3) & 1u;
    return r;
}
__device__ __forceinline__ SpanAcc warp_span_inclusive(SpanAcc a, int lane) {
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const SpanAcc o = span_shfl_up(a, d);
        if (lane >= d) a = span_concat(o, a);
    }
    return a;
}
constexpr uint32_t SPAN_SCAN_THREADS = 1024;
// inclusive scan over the CTA's threads in thread order; returns this thread's inclusive span, `total` = the CTA's
__device__ __forceinline__ SpanAcc block_span_inclusive(const SpanAcc mine, uint4 *s_w /* [32] */, SpanAcc &total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    constexpr int NWARPS = SPAN_SCAN_THREADS / 32;
    SpanAcc a = warp_span_inclusive(mine, lane);
    if (lane == 31) s_w[warp] = make_uint4(a.c[0], a.c[1], span_flags(a), 0u);
    __syncthreads();
    if (warp == 0) {
        SpanAcc w = warp_span_inclusive(lane < NWARPS ? span_from_summary(s_w[lane]) : span_empty(), lane);
        __syncwarp();
        if (lane < NWARPS) s_w[lane] = make_uint4(w.c[0], w.c[1], span_flags(w), 0u);   // inclusive over warps
    }
    __syncthreads();
    total = span_from_summary(s_w[NWARPS - 1]);
    if (warp > 0) a = span_concat(span_from_summary(s_w[warp - 1]), a);
    __syncthreads();   // s_w may be reused by the caller
    return a;
}

constexpr int SPAN_PER_THREAD = 4;        // consecutive chunk summaries per thread
constexpr uint32_t SPAN_BLOCK = SPAN_SCAN_THREADS * SPAN_PER_THREAD;   // chunk summaries per CTA (8 MiB of input)

// One launch, one CTA per SPAN_BLOCK chunk summaries (8 MiB of input): local ordered reduction -> the block aggregate,
// published with a generation tag -> the aggregates of all earlier blocks (a CTA only ever waits for CTAs with a lower
// block index, which are resident or finished: CTAs are dispatched in index order) -> one carry word per chunk; the
// thread that owns the document's last chunk writes the verdict (finish(), reference json_structural_indexer.mojo:147-186).
// block_sum: 32 bytes per block, {count0, count1, flags, 0} then {generation, 0, 0, 0}.
__global__ void __launch_bounds__(SPAN_SCAN_THREADS) stage1_span_scan_kernel(const Stage1Params P, uint32_t nchunks) {
    __shared__ uint4 s_w[32];
    grid_dependency_wait();
    if (*reinterpret_cast<volatile uint32_t *>(P.spec_flag) == P.gen) return;
    const uint32_t blk = blockIdx.x;
    const uint32_t c0 = blk * SPAN_BLOCK + threadIdx.x * SPAN_PER_THREAD;
    uint4 sum[SPAN_PER_THREAD];
    SpanAcc mine = span_empty();
#pragma unroll
    for (int k = 0; k < SPAN_PER_THREAD; k++) {
        sum[k] = c0 + k < nchunks ? reinterpret_cast<const uint4 *>(P.chunk_sum)[c0 + k] : make_uint4(0u, 0u, 0u, 0u);
        mine = span_concat(mine, span_from_summary(sum[k]));
    }
    SpanAcc total;
    const SpanAcc local = block_span_inclusive(mine, s_w, total);
    uint4 *agg = reinterpret_cast<uint4 *>(P.block_sum);
    if (threadIdx.x == 0 && blk + 1u < gridDim.x) {
        agg[2 * blk] = make_uint4(total.c[0], total.c[1], span_flags(total), 0u);
        __threadfence();
        st_release_u32(P.block_sum + 8 * blk + 4, P.gen);
    }
    // everything before this block: ordered reduction of the block aggregates 0 .. blk-1 (1024 per round)
    SpanAcc before = span_empty();
    for (uint32_t b0 = 0; b0 < blk; b0 += SPAN_SCAN_THREADS) {
        const uint32_t j = b0 + threadIdx.x;
        SpanAcc bj = span_empty();
        if (j < blk) {
            while (ld_acquire_u32(P.block_sum + 8 * j + 4) != P.gen) __nanosleep(100);
            bj = span_from_summary(ld_cg_u4(agg + 2 * j));
        }
        SpanAcc round;
        block_span_inclusive(bj, s_w, round);
        before = span_concat(before, round);
    }
    const SpanAcc incl = span_concat(before, local);
    // the document starts outside a string: the state entering a chunk is the span before it evaluated at s = 0.
    // Walk this thread's chunks backwards from its inclusive span: before(k) = inclusive(k) "minus" chunk k.
    uint32_t par = incl.par & 1u, cnt = incl.c[0], un = incl.un[0], u8 = incl.u8;
    if (c0 < nchunks && c0 + SPAN_PER_THREAD >= nchunks) {   // this thread owns the last chunk: the verdict
        TilePrefix pre;
        pre.s_out = par;
        pre.e_out = 0;
        pre.p_out = 0;
        // (a violation among the deferred UTF-8 lanes is folded in later, by the document's last launch)
        pre.err = (un ? EF_UNESCAPED : 0u) | (u8 ? EF_UTF8 : 0u);
        pre.count = cnt;
        write_verdict(P, pre);
    }
#pragma unroll
    for (int k = SPAN_PER_THREAD - 1; k >= 0; k--) {
        const uint32_t s_in = (par ^ sum[k].z) & 1u;               // parity before chunk k
        cnt -= s_in ? sum[k].y : sum[k].x;                          // rank of its first index
        par = s_in;
        if (c0 + k < nchunks) P.carry[c0 + k] = (uint64_t)cnt | (s_in ? CARRY_INSIDE : 0ull);
    }
}

#endif  // __CUDACC__

}  // namespace sjb200
