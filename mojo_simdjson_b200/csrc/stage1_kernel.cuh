// stage1_kernel.cuh -- device code shared by every organisation of the sm_100a stage-1 indexer: PTX helpers
// (mbarrier, cp.async.bulk, relaxed descriptor loads / stores), the decoupled look-back over generation-tagged tile
// descriptors, phase 1 of a warp (2 KiB of input -> dual structural masks + warp summary), the verdict (finish()),
// and the bitmask -> index flattening pieces.  Replaces JsonStructuralIndexer.index/step/next/finish and BitIndexer
// (reference generic/stage1/json_structural_indexer.mojo:33-58,81-186) and the scanners they call.
//
// Work decomposition
//   lane  : 64 consecutive bytes (one 64-bit word of every mask)
//   warp  : 2 KiB chunk; carries between lanes resolved with ballots
// Carries (stage1_core.cuh): "escaped" and "previous scalar" are resolved locally from the bytes just before a
// warp / tile.  The in-string parity is the only global carry: every lane produces its structural bits for BOTH
// values of it, every tile / chunk publishes {quote parity, count if it starts outside a string, count if inside,
// error flags for both}, and ONE ordered scan yields both the parity entering it and the output cursor.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "stage1_core.cuh"

// -DSJ_TRACE=1: per-tile timeline of the persistent kernel (sjb200_debug_trace).  The split pair's classify kernel shares
// its tile fetch and aggregate steps (stage1_persistent.cuh), so in such builds it fills slots 0 and 2 of its tiles too.
#ifndef SJ_TRACE
#define SJ_TRACE 0
#endif

namespace sjb200 {

// simdjson error codes that stage 1 can produce (reference errors.mojo:2-34)
enum : int32_t {
    ERR_SUCCESS = 0,
    ERR_CAPACITY = 1,
    ERR_MEMALLOC = 2,
    ERR_UTF8_ERROR = 11,
    ERR_UNINITIALIZED = 12,
    ERR_EMPTY = 13,
    ERR_UNESCAPED_CHARS = 14,
    ERR_UNCLOSED_STRING = 15,
    ERR_UNEXPECTED_ERROR = 24,
};

struct Stage1Result {       // written by the last tile (mapped pinned host memory or device memory)
    int32_t error;          // verdict, reference priority order
    uint32_t n;             // n_structural_indexes (valid iff n_valid)
    uint32_t n_valid;       // 0 on UNCLOSED_STRING / UNESCAPED_CHARS / CAPACITY: the reference leaves n untouched
    uint32_t n_written;     // entries produced by the indexer (clipped to capacity in memory)
    int32_t utf8_error;     // 1 iff the input is not valid UTF-8 (always reported when validation is compiled in)
    uint32_t final_state;   // bit1 = still inside a string after the last byte
    uint32_t reserved[2];
};

struct Stage1Params {
    const uint8_t *abase;   // input pointer rounded down to 16 bytes
    uint64_t alen;          // mis + len: end of the data in aligned coordinates
    uint32_t mis;           // bytes between abase and the first input byte (0..15)
    uint32_t len;           // input length (< 2^32, reference base.mojo:2)
    uint32_t *out;          // device index array
    uint64_t cap;           // its capacity in entries
    uint64_t *desc;         // per-tile look-back descriptors
    uint32_t *ticket;       // tile ticket counter, 0 at launch, reset by the last tile
    Stage1Result *result;
    int32_t *dev_status;    // optional device copy of {error, n} for on-device consumers (NCCL), may be null
    uint32_t gen;           // generation of this document (1 .. 2^20-1); all launches over one document share it
    uint32_t ntiles;        // tiles of the whole document
    uint32_t tile_begin;    // this launch covers tiles [tile_begin, tile_end): a document may be indexed in several
    uint32_t tile_end;      //   launches (streaming host path); the look-back simply continues across them
    uint32_t ticket_sel;    // which of the two alternating ticket counters this launch uses (persistent kernel)
    uint32_t *progress;     // optional: indexes produced up to and including tile_end-1 (mapped host memory), may be null
    uint32_t flags;         // bit0: fold the UTF-8 verdict into the error code
    uint64_t *masks;        // split pair only: [chunk][parity][lane] structural masks, 512 bytes per 2 KiB chunk
    uint64_t *carry;        // split pair only: per chunk, bit 63 = starts inside a string, bits 0..39 = rank of its first index
    uint32_t *chunk_sum;    // stream pipeline only: 16 bytes per chunk {count0, count1, flags, 0}
    uint32_t *block_sum;    // stream pipeline only: the same per 1024 chunks
    uint32_t *spec_flag;    // stream pipeline: == gen once a chunk could not resolve its escape carry locally.  Persistent
                            // kernel: if non-null, run only when *spec_flag == gen (it is the exact fallback)
    uint64_t *trace;        // debug builds (-DSJ_TRACE=1): 16 x u64 of timestamps per tile, else unused
};

#if defined(__CUDACC__)

// ---------------------------------------------------------------------------------------------
// PTX helpers
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint64_t gtime() {
    uint64_t t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
#if SJ_TRACE
#define TRACE(P, tile, slot, val) do { if ((P).trace) (P).trace[(size_t)(tile) * 16 + (slot)] = (val); } while (0)
#else
#define TRACE(P, tile, slot, val) do { } while (0)
#endif
// Programmatic dependent launch: blocks until the kernel this one depends on has completed and its writes are visible.
// A no-op when the kernel was launched without the attribute.
__device__ __forceinline__ void grid_dependency_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ uint32_t lanemask_lt() {   // bits of the lanes below this one
    uint32_t m;
    asm("mov.u32 %0, %%lanemask_lt;" : "=r"(m));
    return m;
}

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_load(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
                 "l"(src), "r"(bytes), "r"(bar)
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    // try_wait suspends the thread in hardware until the phase completes or a system-dependent time limit expires (no busy spin)
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "SJ_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra SJ_DONE;\n"
        "bra SJ_WAIT;\n"
        "SJ_DONE:\n"
        "}\n" ::"r"(bar),
        "r"(parity)
        : "memory");
}
__device__ __forceinline__ uint64_t ld_desc(const uint64_t *p) {
    uint64_t v;
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_desc(uint64_t *p, uint64_t v) {
    asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
// back-off between two polls of a look-back descriptor (ns)
constexpr unsigned DESC_POLL_NS = 20;
// spin until tile j has published something for this generation
__device__ __forceinline__ uint64_t wait_desc(const uint64_t *desc, int j, uint32_t gen) {
    uint64_t d = ld_desc(desc + j);
    while (desc_gen(d) != (gen & GEN_MASK)) {
        __nanosleep(DESC_POLL_NS);
        d = ld_desc(desc + j);
    }
    return d;
}

__device__ __forceinline__ uint32_t mask_word(uint32_t w, int64_t g, int64_t vbeg, int64_t vend) {
    int64_t lo = vbeg - g, hi = vend - g;
    lo = lo < 0 ? 0 : (lo > 4 ? 4 : lo);
    hi = hi < 0 ? 0 : (hi > 4 ? 4 : hi);
    const uint32_t mh = hi >= 4 ? 0xFFFFFFFFu : ((1u << (8 * (int)hi)) - 1u);
    const uint32_t ml = lo >= 4 ? 0xFFFFFFFFu : ((1u << (8 * (int)lo)) - 1u);
    const uint32_t m = hi > lo ? (mh & ~ml) : 0u;
    return (w & m) | (0x20202020u & ~m);
}

// ---------------------------------------------------------------------------------------------
// local carry resolution: (e, p) entering the tile / a warp, from the bytes before it
// ---------------------------------------------------------------------------------------------
// tile level: 16 halo bytes at smem_tile[-16..-1]; if they do not decide, the predecessor's descriptor does
__device__ __forceinline__ PrevState tile_prev_state(const uint8_t *smem_tile, int tile, int lane, const uint64_t *desc,
                                                     uint32_t gen) {
    PrevState st = {0, 0, 0};
    if (tile == 0) return st;  // nothing before the document
    const uint32_t c = lane < 16 ? (uint32_t)smem_tile[-1 - lane] : 0x20u;
    const uint32_t bsm = __ballot_sync(0xFFFFFFFFu, c == 0x5Cu);
    const uint32_t c1 = __shfl_sync(0xFFFFFFFFu, c, 0);
    st = prev_state(bsm, 16, c1);
    if (st.unresolved) {  // a backslash run fills the halo: the previous tile knows (it resolved its own carries first)
        const uint64_t d = wait_desc(desc, tile - 1, gen);
        const uint32_t f = (uint32_t)(d >> 36);  // e_out / p_out sit at the same bits in both descriptor kinds
        if (st.unresolved & 1u) st.e = (f >> 4) & 1u;
        if (st.unresolved & 2u) st.p = (f >> 3) & 1u;
        st.unresolved = 0;
    }
    return st;
}

// warp level (warp > 0): 32 bytes before the warp's first byte, all inside this tile
__device__ __forceinline__ PrevState warp_prev_state(const uint8_t *smem_tile, int woff, int lane, int64_t tb, int64_t vbeg,
                                                     int64_t vend, bool edge, int tile, const uint64_t *desc, uint32_t gen) {
    uint32_t c = (uint32_t)smem_tile[woff - 1 - lane];
    if (edge) {
        const int64_t g = tb + woff - 1 - lane;
        if (g < vbeg || g >= vend) c = 0x20u;  // outside the document: reads as the reference's 0x20 padding
    }
    const uint32_t bsm = __ballot_sync(0xFFFFFFFFu, c == 0x5Cu);
    const uint32_t c1 = __shfl_sync(0xFFFFFFFFu, c, 0);
    PrevState st = prev_state(bsm, 32, c1);
    if (st.unresolved) {  // rare: a backslash run of 31+ bytes ends at the warp boundary; walk it inside the tile
        const PrevState t = tile_prev_state(smem_tile, tile, lane, desc, gen);
        // bytes of this tile that may be read before the warp (tile 0: not before the document start)
        const uint32_t room = (uint32_t)woff - (tile == 0 ? (uint32_t)vbeg : 0u);
        if (st.unresolved & 1u) {
            const uint32_t r = backslash_run_before(smem_tile + woff, room);
            st.e = r < room ? (r & 1u) : escaped_after_run(room, t.e);
        }
        if (st.unresolved & 2u) {  // byte -1 is a quote: is it escaped?
            const uint32_t r = backslash_run_before(smem_tile + woff - 1, room - 1);
            st.p = r < room - 1 ? (r & 1u) : escaped_after_run(room - 1, t.e);
        }
        st.unresolved = 0;
    }
    return st;
}

// ---------------------------------------------------------------------------------------------
// look-back (executed by warp 0 of a tile > 0): parity entering the tile, indexes before it, errors so far
// ---------------------------------------------------------------------------------------------
struct LookbackResult {
    uint32_t s_in, base, err;
};
__device__ __forceinline__ LookbackResult lookback(const uint64_t *desc, uint32_t gen, int tile, int lane) {
    SpanAcc acc = span_empty();  // the already visited (newer) tiles as a function of the parity entering them
    const uint32_t want = gen & GEN_MASK;
    int base = tile - 1;
    uint64_t dnext = base - lane >= 0 ? ld_desc(desc + (base - lane)) : 0;
    while (true) {
        const int j = base - lane;
        uint64_t d = dnext;
        // have the following window in flight before we start waiting on this one
        dnext = j - 32 >= 0 ? ld_desc(desc + (j - 32)) : 0;
        uint32_t st = DESC_PREFIX;  // before the first tile: outside a string, nothing produced
        if (j >= 0) {
            while (desc_gen(d) != want) {
                __nanosleep(DESC_POLL_NS);
                d = ld_desc(desc + j);
            }
            st = desc_status(d);
        }
        const uint32_t pm = __ballot_sync(0xFFFFFFFFu, st == DESC_PREFIX);
        const int k = pm ? (__ffs((int)pm) - 1) : 32;  // nearest tile whose inclusive state is known
        const bool isagg = lane < k;
        const TileAgg a = desc_unpack_agg(d);
        // parity of the AGG tiles older than this lane's tile inside the window (higher lanes are older)
        const uint32_t pbm = __ballot_sync(0xFFFFFFFFu, isagg && a.par);
        const uint32_t rel = (uint32_t)__popc(pbm & ~((2u << lane) - 1u)) & 1u;
        SpanAcc win;
        win.par = (uint32_t)__popc(pbm) & 1u;
        win.c[0] = __reduce_add_sync(0xFFFFFFFFu, isagg ? (rel ? a.c[1] : a.c[0]) : 0u);
        win.c[1] = __reduce_add_sync(0xFFFFFFFFu, isagg ? (rel ? a.c[0] : a.c[1]) : 0u);
        const uint32_t unx = rel ? a.un[1] : a.un[0], uny = rel ? a.un[0] : a.un[1];
        const uint32_t eall = __reduce_or_sync(0xFFFFFFFFu, isagg ? (unx | (uny << 1) | (a.u8 << 2)) : 0u);
        win.un[0] = eall & 1u;
        win.un[1] = (eall >> 1) & 1u;
        win.u8 = (eall >> 2) & 1u;
        acc = span_concat(win, acc);
        if (pm) {
            const uint64_t dk = __shfl_sync(0xFFFFFFFFu, d, k);
            TilePrefix p = {0, 0, 0, 0, 0};              // state before the first tile
            if (base - k >= 0) p = desc_unpack_prefix(dk);
            LookbackResult r;
            r.s_in = p.s_out ^ acc.par;
            r.base = p.count + (p.s_out ? acc.c[1] : acc.c[0]);
            r.err = p.err | ((p.s_out ? acc.un[1] : acc.un[0]) ? EF_UNESCAPED : 0u) | (acc.u8 ? EF_UTF8 : 0u);
            return r;
        }
        base -= 32;
    }
}

// ---------------------------------------------------------------------------------------------
// phase 1 of a warp: 2 KiB of shared-memory input -> per-lane dual structural masks + warp summary
// ---------------------------------------------------------------------------------------------
struct LaneInput {
    uint32_t w[16];   // this lane's 64 bytes
    uint32_t prev;    // the 4 bytes before them (UTF-8 look-behind)
    PrevState wst;    // carries entering the warp
    int64_t g0;       // aligned coordinate of the lane's first byte
    uint32_t ends;    // the document ends exactly at this lane's last byte (only ever set in the last tile / chunk)
};
struct LanePhase1 {
    uint64_t m0, m1;  // structural bits if the warp starts outside / inside a string
    uint32_t c0, c1;  // their popcounts
    uint32_t v0;      // index value of bit 0
    // warp-uniform
    uint32_t wc0, wc1;
    uint32_t wflags;  // bit0 quote parity, bit1/2 unescaped control (outside/inside), bit3 UTF-8 violation
    uint32_t tail;    // bit0 e_out, bit1 p_out after the warp's last byte
    uint32_t u8_lanes;  // stream pipeline: lanes parked for deferred UTF-8 validation (else 0)
};

// every shared-memory read of the input happens here (the persistent kernel frees the buffer right after)
template <bool UTF8>
__device__ __forceinline__ void warp_load(LaneInput &in, const uint8_t *smem_tile, int warp, int lane, int tile, int64_t tb,
                                          int tile_bytes, const Stage1Params &P) {
    const int64_t alen = (int64_t)P.alen;
    const int woff = warp * 2048;
    const int off = woff + lane * 64;
    in.g0 = tb + off;
    const bool edge = (tile == 0) || (tb + tile_bytes > alen);
    const uint4 *src = reinterpret_cast<const uint4 *>(smem_tile + off);
#pragma unroll
    for (int q = 0; q < 4; q++) {
        const uint4 v = src[q];
        in.w[4 * q + 0] = v.x;
        in.w[4 * q + 1] = v.y;
        in.w[4 * q + 2] = v.z;
        in.w[4 * q + 3] = v.w;
    }
    in.prev = UTF8 ? *reinterpret_cast<const uint32_t *>(smem_tile + off - 4) : 0u;
    // the document may end exactly with this lane's last byte (also when the last tile is full: not an "edge" tile then)
    in.ends = (tile == (int)P.ntiles - 1) && (in.g0 + 64 == alen);
    if (edge) {  // only the first and last tile: bytes outside [mis, alen) read as 0x20 (reference tail padding)
#pragma unroll
        for (int k = 0; k < 16; k++) in.w[k] = mask_word(in.w[k], in.g0 + 4 * k, (int64_t)P.mis, alen);
        if (UTF8) in.prev = (in.g0 == 0) ? 0x20202020u : mask_word(in.prev, in.g0 - 4, (int64_t)P.mis, alen);
    }
    // carries entering the warp, from the bytes before it (warp 0: the halo / the previous tile)
    in.wst = warp == 0 ? tile_prev_state(smem_tile, tile, lane, P.desc, P.gen)
                       : warp_prev_state(smem_tile, woff, lane, tb, (int64_t)P.mis, alen, edge, tile, P.desc, P.gen);
}

// DEFER_U8: when only a few lanes of the warp hold (or directly follow) bytes >= 0x80, do not validate UTF-8 here -- the
// whole warp would pay ~75 ALU instructions for them -- but park those lanes (16 bit-plane words, the 4 bytes before the
// lane, its end-of-document bit: 80 B) in the warp's own shared-memory slots and report them; the same warp validates them
// 32 at a time at the end of its run of chunks (stage1_stream.cuh: validate_parked_lanes).  `u8_slots` points at the
// first free slot.  DEFER_U8 == 0: always validate inline.
constexpr int U8_DEFER_MAX = 8;   // most lanes of a chunk that DEFER_U8 parks
template <bool UTF8, int DEFER_U8 = 0>
__device__ __forceinline__ void warp_compute(LanePhase1 &r, const LaneInput &in, int lane, const Stage1Params &P,
                                             uint4 *u8_slots = nullptr /* DEFER_U8: the warp's free shared-memory slots, 5 uint4 each */,
                                             uint32_t lt = lanemask_lt() /* bits of the lanes below this one */) {
    LaneMasks m;
    uint32_t u8err = 0;
    r.u8_lanes = 0;
    {
        uint32_t pl[8], ph[8];
        bitplanes32(in.w, pl);
        bitplanes32(in.w + 8, ph);
        Classes32 cl, ch;
        classify_json32(pl, cl);
        classify_json32(ph, ch);
        m.bs = join64(cl.bs, ch.bs);
        m.rq = join64(cl.rq, ch.rq);
        m.op = join64(cl.op, ch.op);
        m.ws = join64(cl.ws, ch.ws);
        m.ctl = join64(cl.ctl, ch.ctl);
        if (UTF8) {
            // whole-warp fast path: nothing >= 0x80 in these 2 KiB nor in the 4 bytes before each lane's 64 (the lead /
            // continuation classes are not even computed then)
            const bool any_hi = ((pl[7] | ph[7]) != 0) || ((in.prev & 0x80808080u) != 0);
            const uint32_t hi_lanes = __ballot_sync(0xFFFFFFFFu, any_hi);
            r.u8_lanes = 0;
            if (DEFER_U8 && __popc(hi_lanes) <= U8_DEFER_MAX) {
                // the k-th flagged lane parks its bit planes, the 4 bytes before it and its end-of-document bit in slot k
                r.u8_lanes = hi_lanes;
                if (any_hi) {
                    uint4 *s = u8_slots + 5 * __popc(hi_lanes & lt);   // 80 contiguous bytes per slot
                    s[0] = make_uint4(pl[0], pl[1], pl[2], pl[3]);
                    s[1] = make_uint4(pl[4], pl[5], pl[6], pl[7]);
                    s[2] = make_uint4(ph[0], ph[1], ph[2], ph[3]);
                    s[3] = make_uint4(ph[4], ph[5], ph[6], ph[7]);
                    s[4] = make_uint4(in.prev, in.ends, 0u, 0u);
                }
            } else if (hi_lanes) {
                Utf8Pre32 ul, uh;
                utf8_pre32(pl, ul);
                utf8_pre32(ph, uh);
                // what the three bytes before this lane's 64 demand of its first bytes: nothing unless one of them is a lead
                // byte (>= 0xC0), i.e. a multi-byte character straddles a lane boundary somewhere in the warp
                Utf8Carry uc = {0, 0, 0, 0};
                const bool straddle = (in.prev & (in.prev << 1) & 0x80808000u) != 0;
                if (__any_sync(0xFFFFFFFFu, straddle)) uc = utf8_carry_from_prev_word(in.prev);
                uint32_t tail_must;
                const uint64_t ue = utf8_errors64(ul, uh, uc, &tail_must);
                u8err = (ue != 0) || (in.ends && tail_must != 0);
            }
        }
    }
    // escapes and quotes, exact; structural bits for both in-string parities
    // A = lanes that are one long backslash run, O = parity of the backslash run each lane ends with; both are zero unless
    // some lane ends in a backslash, which one ballot on the top bit decides
    // Without such a lane no escape crosses a lane boundary: lane 0 inherits the warp's carry, every other lane starts clean.
    uint32_t e_in = lane ? 0u : in.wst.e, e_out = 0u;
    if (__ballot_sync(0xFFFFFFFFu, (uint32_t)(m.bs >> 32) >> 31)) {
        const uint32_t bA = __ballot_sync(0xFFFFFFFFu, lane_all_backslash(m.bs));
        const uint32_t bO = __ballot_sync(0xFFFFFFFFu, lane_trailing_run_parity(m.bs));
        e_in = warp_lane_e_in(bA, bO, lane, in.wst.e);
        e_out = warp_lane_e_in(bA, bO, 32, in.wst.e);
    }
    const LaneQuotes q = lane_quotes(m, e_in);
    const uint32_t bPB = __ballot_sync(0xFFFFFFFFu, (q.ps >> 63) != 0);
    const uint32_t bNQ = __ballot_sync(0xFFFFFFFFu, (q.nqs >> 63) != 0);
    const uint32_t rel = (uint32_t)__popc(bPB & lt) & 1u;
    const uint32_t p_in = lane ? ((bNQ >> (lane - 1)) & 1u) : in.wst.p;
    const LaneDual dual = lane_structurals_dual(m, q, rel, p_in);
    r.m0 = dual.m0;
    r.m1 = dual.m1;
    r.c0 = (uint32_t)__popcll(dual.m0);
    r.c1 = (uint32_t)__popcll(dual.m1);
    r.v0 = (uint32_t)(in.g0 - (int64_t)P.mis);
    r.wc0 = __reduce_add_sync(0xFFFFFFFFu, r.c0);
    r.wc1 = __reduce_add_sync(0xFFFFFFFFu, r.c1);
    r.wflags = __reduce_or_sync(0xFFFFFFFFu, (dual.u0 << 1) | (dual.u1 << 2) | (u8err << 3)) | ((uint32_t)__popc(bPB) & 1u);
    r.tail = e_out | ((bNQ >> 31) << 1);
}

// combine the warp summaries of a tile (called by one full warp): the tile aggregate, and for every warp (lane < nwarps)
// the parity of the warps before it and its rank offsets for both tile parities
__device__ __forceinline__ TileAgg tile_aggregate(uint32_t fl, uint32_t a0, uint32_t a1, uint32_t tail, int nwarps, int lane,
                                                  uint32_t &R, uint32_t &off0, uint32_t &off1) {
    const uint32_t lt = (1u << lane) - 1u;
    const uint32_t parb = __ballot_sync(0xFFFFFFFFu, fl & 1u);
    R = (uint32_t)__popc(parb & lt) & 1u;                  // parity of the warps before this one
    const uint32_t t0 = R ? a1 : a0, t1 = R ? a0 : a1;     // this warp's count if the TILE starts outside / inside
    uint32_t i0 = t0, i1 = t1;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t x0 = __shfl_up_sync(0xFFFFFFFFu, i0, d);
        const uint32_t x1 = __shfl_up_sync(0xFFFFFFFFu, i1, d);
        if (lane >= d) {
            i0 += x0;
            i1 += x1;
        }
    }
    off0 = i0 - t0;
    off1 = i1 - t1;
    TileAgg agg;
    agg.par = (uint32_t)__popc(parb) & 1u;
    agg.c[0] = __shfl_sync(0xFFFFFFFFu, i0, nwarps - 1);
    agg.c[1] = __shfl_sync(0xFFFFFFFFu, i1, nwarps - 1);
    const uint32_t un0 = (fl >> (R ? 2 : 1)) & 1u, un1 = (fl >> (R ? 1 : 2)) & 1u;
    const uint32_t eall = __reduce_or_sync(0xFFFFFFFFu, un0 | (un1 << 1) | (((fl >> 3) & 1u) << 2));
    agg.un[0] = eall & 1u;
    agg.un[1] = (eall >> 1) & 1u;
    agg.u8 = (eall >> 2) & 1u;
    agg.e_out = tail & 1u;
    agg.p_out = (tail >> 1) & 1u;
    return agg;
}

// finish(): reference json_structural_indexer.mojo:147-186, same priority order.  One thread of the last tile.
__device__ __forceinline__ void write_verdict(const Stage1Params &P, const TilePrefix &pre) {
    const uint64_t n = pre.count;
    Stage1Result r;
    r.n = (uint32_t)n;
    r.n_written = (uint32_t)n;
    r.n_valid = 0;
    r.utf8_error = (pre.err & EF_UTF8) ? 1 : 0;
    r.final_state = pre.s_out << 1;
    r.reserved[0] = r.reserved[1] = 0;
    if (pre.s_out) {
        r.error = ERR_UNCLOSED_STRING;
    } else if (pre.err & EF_UNESCAPED) {
        r.error = ERR_UNESCAPED_CHARS;
    } else if (n + 3 > P.cap) {
        r.error = ERR_CAPACITY;
    } else {
        r.n_valid = 1;
        P.out[n] = P.len;      // trailer: len, len, 0 (:167-173)
        P.out[n + 1] = P.len;
        P.out[n + 2] = 0;
        if (n == 0) r.error = ERR_EMPTY;
        else if ((P.flags & 1u) && (pre.err & EF_UTF8)) r.error = ERR_UTF8_ERROR;
        else r.error = ERR_SUCCESS;
    }
    *P.result = r;
    if (P.dev_status) {
        P.dev_status[0] = r.error;
        P.dev_status[1] = (int32_t)(r.n_valid ? r.n : 0u);
    }
}

// flatten one lane's structural bits (BitIndexer.write, reference json_structural_indexer.mojo:46-58) into a staging area in
// shared memory.
// Flattening is bound by instruction issue, so its two inner pieces are written out by hand.
//
// flatten_word_pair: the structurals of one 32-bit word into shared memory at byte address `sptr`, two per trip.  The
// word is bit-reversed, so bfind (FLO) returns 31 - position; xor clears the bit and its result predicates the second
// half and the loop (LOP3 with predicate output): FLO, SHF, LOP3, IADD, STS twice, one pointer bump, one branch.
__device__ __forceinline__ void flatten_word_pair(uint32_t sptr, uint32_t bits, uint32_t v31) {
    uint32_t r = __brev(bits);
    asm volatile(
        "{\n"
        ".reg .pred p, q;\n"
        ".reg .u32 h, m, x, ptr;\n"
        "mov.u32 ptr, %1;\n"
        "setp.ne.u32 p, %0, 0;\n"
        "@!p bra FW_DONE;\n"
        "FW_LOOP:\n"
        "bfind.u32 h, %0;\n"
        "shl.b32 m, 1, h;\n"
        "xor.b32 %0, %0, m;\n"
        "sub.u32 x, %2, h;\n"
        "st.shared.u32 [ptr], x;\n"
        "setp.ne.u32 q, %0, 0;\n"
        "bfind.u32 h, %0;\n"
        "@q shl.b32 m, 1, h;\n"
        "@q xor.b32 %0, %0, m;\n"
        "@q sub.u32 x, %2, h;\n"
        "@q st.shared.u32 [ptr+4], x;\n"
        "add.u32 ptr, ptr, 8;\n"
        "setp.ne.u32 p, %0, 0;\n"
        "@p bra FW_LOOP;\n"
        "FW_DONE:\n"
        "}\n"
        : "+r"(r)
        : "r"(sptr), "r"(v31)
        : "memory");
}

// stage[a .. a+total) -> out[first .. first+total) by one warp, a + total < 4 * NV + 4: up to NV 16-byte copies, the lanes'
// predicated ones unrolled, plus the ragged head / tail entries (a = phase of `first` in its 16-byte line, so stage and out
// are congruent)
template <int NV>
__device__ __forceinline__ void copy_out_warp_n(const uint32_t *stage, uint32_t a, uint32_t total, uint32_t *out, uint64_t first,
                                                uint64_t cap, uint32_t lane) {
    const uint32_t end = a + total;
    uint32_t *g0 = out + ((int64_t)first - (int64_t)a);   // 16-byte aligned, may point below `out` by up to 3 entries
    if (first + total <= cap) {
        const uint32_t v_lo = (a + 3u) >> 2, v_hi = end >> 2;
        const uint32_t nvec = v_hi > v_lo ? v_hi - v_lo : 0u;      // whole vectors; none when the run is shorter than a line
        const uint4 *sv = reinterpret_cast<const uint4 *>(stage) + lane;
        uint4 *gv = reinterpret_cast<uint4 *>(g0) + lane;
#pragma unroll
        for (int k = 0; k < (NV + 31) / 32; k++) {
            const uint32_t v = lane + 32u * k;
            if (v - v_lo < nvec) gv[32 * k] = sv[32 * k];          // v_lo <= v < v_hi in one unsigned compare
        }
        if (lane < 8u) {
            const uint32_t j = lane < 4u ? lane : 4u * v_hi + (lane - 4u);
            const bool head = lane < 4u && j >= a && j < end && j < 4u * v_lo;
            const bool tail = lane >= 4u && j < end && j >= a && v_hi >= v_lo;
            if (head || tail) g0[j] = stage[j];
        }
    } else {
        for (uint32_t j = a + lane; j < end; j += 32u)
            if (first + (j - a) < cap) g0[j] = stage[j];
    }
}

__device__ __forceinline__ void flatten_to(uint32_t *dst, uint64_t structural, uint32_t v0) {
    const uint32_t lo = (uint32_t)structural, sp = smem_u32(dst);   // dst is always a shared-memory staging area
    flatten_word_pair(sp, lo, v0 + 31u);
    flatten_word_pair(sp + 4u * (uint32_t)__popc(lo), (uint32_t)(structural >> 32), v0 + 63u);
}
__device__ __forceinline__ void flatten_direct(uint32_t *out, uint64_t cap, uint64_t o, uint64_t structural, uint32_t v0) {
    uint32_t rlo = __brev((uint32_t)structural), rhi = __brev((uint32_t)(structural >> 32));
    while (rlo) {
        const int b = __clz((int)rlo);
        if (o < cap) out[o] = v0 + (uint32_t)b;
        o++;
        rlo &= ~(0x80000000u >> b);
    }
    while (rhi) {
        const int b = __clz((int)rhi);
        if (o < cap) out[o] = v0 + 32u + (uint32_t)b;
        o++;
        rhi &= ~(0x80000000u >> b);
    }
}
// inclusive warp scan; the shuffle's in-range predicate guards the add (no compare / select per step)
__device__ __forceinline__ uint32_t warp_inclusive_sum(uint32_t x) {
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        asm volatile(
            "{\n"
            ".reg .u32 t;\n"
            ".reg .pred p;\n"
            "shfl.sync.up.b32 t|p, %0, %1, 0, 0xffffffff;\n"
            "@p add.u32 %0, %0, t;\n"
            "}\n"
            : "+r"(x)
            : "r"(d));
    }
    return x;
}
__device__ __forceinline__ uint32_t out_phase(const uint32_t *out) { return (uint32_t)((reinterpret_cast<uintptr_t>(out) >> 2) & 3u); }

#endif  // __CUDACC__

}  // namespace sjb200
