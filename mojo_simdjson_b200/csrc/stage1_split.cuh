// stage1_split.cuh -- stage 1 as two launches for large documents: classify, then flatten.
//
// The persistent kernel (stage1_persistent.cuh) is bound by latency, not by a pipe: a warp that
// classifies 2 KiB and then extracts its indexes spends long stretches waiting (bulk copy, look-back, the serial
// clear-lowest-bit chain of the extraction loop), and registers cap the SM at ~34 such warps.  Measured standalone
// (tools/ubench_stages.cu) both halves only reach their issue-bound rate with >= 32 warps per SM *each*.  So for
// documents large enough to amortise a second launch the two halves run as separate grids, each at the occupancy its own
// register budget allows, and neither ever waits for a carry:
//
//   stage1_classify_kernel : persistent CTAs of NW compute warps + 1 scan warp, tiles drawn from the ticket counter
//                            exactly as in the persistent kernel.  A compute warp turns 2 KiB into the two structural masks
//                            (string state entering the chunk unknown -> one mask per parity), stores both (16 bytes per
//                            64 input bytes) and moves on.  The scan warp runs the decoupled look-back for every tile
//                            and leaves, per 2 KiB chunk, one 8-byte carry word: bit 63 = chunk starts inside a string,
//                            bits 0..39 = rank of its first structural in the output.  It also writes the verdict.
//                            (Fetch, aggregate and prefix steps are shared with the persistent kernel; in -DSJ_TRACE=1
//                            builds they fill trace slots 0 and 2 of this kernel's tiles.)
//   stage1_flatten2_kernel : one warp per unit of two chunks, no shared state between warps: carry word -> pick the mask
//                            plane -> every lane extracts the same number of consecutive indexes (balanced, see below)
//                            into the warp's staging area, 16-byte stores.
//
// Extra HBM traffic: the mask planes, 16 B written + 8 B read per 64 input bytes (+23 % over the algorithmic bytes at the
// bench document's density of 0.161 structurals per byte).
// Same arithmetic, same descriptors, same results as the persistent kernel (reference json_structural_indexer.mojo:83-186).
#pragma once
#include "stage1_persistent.cuh"

namespace sjb200 {

#if defined(__CUDACC__)

constexpr uint64_t CARRY_INSIDE = 1ull << 63;
constexpr uint64_t CARRY_RANK_MASK = (1ull << 40) - 1;

template <int NW>
struct SplitCfg {
    static constexpr int THREADS = (NW + 1) * 32;
    static constexpr int TILE = NW * 2048;
    static constexpr int NIN = 2;                                         // input buffers (bulk copy of tile i+2 overlaps tile i+1)
    static constexpr int IN_STRIDE = ((16 + TILE) + 127) & ~127;          // halo + tile
    static constexpr int SMEM_BYTES = NIN * IN_STRIDE;
    static constexpr int MAXREG = 56;                                    // registers per thread of the classify kernel
};

template <int NW, bool UTF8>
__global__ void __launch_bounds__((NW + 1) * 32) __maxnreg__(SplitCfg<NW>::MAXREG) stage1_classify_kernel(const Stage1Params P) {
    using Cfg = SplitCfg<NW>;
    constexpr int TILE = Cfg::TILE;
    constexpr int NIN = Cfg::NIN;
    constexpr int NS = 4;
    extern __shared__ __align__(128) uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t s_bar[NIN + 2 * NS];   // in_full[NIN], sum_full[NS], slot_free[NS]
    __shared__ TileSlot s_slot[NS];
    __shared__ int32_t s_tile_of[NIN];
    __shared__ uint32_t s_loaded[NIN];

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t bar_in = smem_u32(&s_bar[0]), bar_sum = smem_u32(&s_bar[NIN]), bar_free = smem_u32(&s_bar[NIN + NS]);

    if (tid == 0) {
        for (int k = 0; k < NIN; k++) {
            mbar_init(bar_in + 8 * k, 1);
            s_loaded[k] = 0;
        }
        for (int k = 0; k < NS; k++) {
            mbar_init(bar_sum + 8 * k, 1);
            mbar_init(bar_free + 8 * k, 1);
            s_slot[k].arrived = 0;
        }
        fence_mbar_init();
        if (blockIdx.x == 0) P.ticket[(P.ticket_sel + 1) & 1u] = 0;   // the counter the NEXT launch will use
    }
    __syncthreads();
    uint32_t *ticket = P.ticket + (P.ticket_sel & 1u);

    // draw the ticket of iteration `it` and start its bulk copy into input buffer it % NIN (free by construction)
    auto produce = [&](int it) {
        const int b = it % NIN;
        if (!fetch_tile<TILE>(P, ticket, s_tile_of[b], smem_u32(smem_raw) + b * Cfg::IN_STRIDE, bar_in + 8 * b))
            mbar_arrive(bar_in + 8 * b);   // no more work
    };
    if (tid == 0) {
        for (int k = 0; k < NIN; k++) produce(k);
    }

    if (warp == NW) {
        // =============================== scan warp ===============================
        for (int i = 0;; i++) {
            const int slot = i & (NS - 1);
            mbar_wait(bar_sum + 8 * slot, (uint32_t)(i / NS) & 1u);
            TileSlot &S = s_slot[slot];
            const int cur = *reinterpret_cast<volatile int32_t *>(&S.tile);
            if (cur < 0) break;
            const TileAgg agg = desc_unpack_agg(S.agg);
            const bool have = lane < NW;
            const uint32_t R = have ? S.R[lane] : 0u, off0 = have ? S.off0[lane] : 0u, off1 = have ? S.off1[lane] : 0u;
            __syncwarp();
            if (lane == 0) mbar_arrive(bar_free + 8 * slot);   // everything we need is in registers: the slot may be reused
            const TileStart st = publish_tile_prefix(P, agg, cur, lane);
            if (have) {
                const uint64_t first = (uint64_t)st.base + (st.s_in ? off1 : off0);
                P.carry[(size_t)cur * NW + lane] = first | (((st.s_in ^ R) & 1u) ? CARRY_INSIDE : 0ull);
            }
        }
    } else {
        // =============================== compute warps ===============================
        int i = 0;
        while (true) {
            const int b = i % NIN;
            mbar_wait(bar_in + 8 * b, (uint32_t)(i / NIN) & 1u);
            const int tile = *reinterpret_cast<volatile int32_t *>(&s_tile_of[b]);
            if (tile < 0) break;
            const int slot = i & (NS - 1);
            const int64_t tb = (int64_t)tile * TILE;
            LanePhase1 ph;
            {
                LaneInput in;
                warp_load<UTF8>(in, smem_raw + b * Cfg::IN_STRIDE + 16, warp, lane, tile, tb, TILE, P);
                __syncwarp();
                if (lane == 0) {                            // this warp no longer needs the input buffer
                    __threadfence_block();
                    if (atomicAdd(&s_loaded[b], 1u) == NW - 1) {
                        s_loaded[b] = 0;                    // everyone has it in registers: refill the buffer
                        __threadfence_block();
                        produce(i + NIN);
                    }
                }
                warp_compute<UTF8>(ph, in, lane, P);
            }
            {   // both mask planes of the chunk: [chunk][parity][lane], 256 contiguous bytes per plane
                uint64_t *mp = P.masks + ((size_t)tile * NW + warp) * 64 + lane;
                __stcs(reinterpret_cast<unsigned long long *>(mp), (unsigned long long)ph.m0);
                __stcs(reinterpret_cast<unsigned long long *>(mp + 32), (unsigned long long)ph.m1);
            }
            if (i >= NS) mbar_wait(bar_free + 8 * slot, (uint32_t)(i / NS - 1) & 1u);   // the scan warp is done with iteration i - NS
            publish_tile_aggregate<NW>(s_slot[slot], ph, warp, lane, tile, P, bar_sum + 8 * slot);
            i++;
        }
        if (warp == 0 && lane == 0) {   // tell the scan warp that iteration i does not exist
            const int slot = i & (NS - 1);
            if (i >= NS) mbar_wait(bar_free + 8 * slot, (uint32_t)(i / NS - 1) & 1u);
            s_slot[slot].tile = -1;
            mbar_arrive(bar_sum + 8 * slot);
        }
    }
}

// one warp flattens chunk c, every lane its own 64-bit mask word (the balanced kernel's path for units denser than its staging
// area): carry word -> plane -> popcount, warp scan, extraction into `stage` (the warp's staging area of WCAP + 4 entries in
// shared memory), 16-byte stores.  BitIndexer.write, reference json_structural_indexer.mojo:46-58.
template <int WCAP>
__device__ __forceinline__ void flatten_chunk(const Stage1Params &P, uint32_t c, uint64_t carry, uint64_t structural, uint32_t *stage, int lane) {
    const uint64_t first = carry & CARRY_RANK_MASK;
    const uint32_t lo = (uint32_t)structural, hi = (uint32_t)(structural >> 32);
    const uint32_t cnt_lo = (uint32_t)__popc(lo), cnt = cnt_lo + (uint32_t)__popc(hi);
    const uint32_t incl = warp_inclusive_sum(cnt);
    const uint32_t wtotal = __shfl_sync(0xFFFFFFFFu, incl, 31);
    const uint32_t v0 = c * 2048u + (uint32_t)lane * 64u - P.mis;
    if (wtotal <= (uint32_t)WCAP) {
        const uint32_t a = ((uint32_t)first + out_phase(P.out)) & 3u;
        const uint32_t sp = smem_u32(stage) + 4u * (a + (incl - cnt));
        flatten_word_pair(sp, lo, v0 + 31u);
        flatten_word_pair(sp + 4u * cnt_lo, hi, v0 + 63u);   // (the popcount of the low word is needed for the scan anyway)
        __syncwarp();
        copy_out_warp_n<128>(stage, a, wtotal, P.out, first, P.cap, (uint32_t)lane);
    } else {
        flatten_direct(P.out, P.cap, first + (incl - cnt), structural, v0);
    }
}

// ---------------------------------------------------------------------------------------------
// Balanced flatten.  Giving every lane the 64 bits of its own mask word (flatten_chunk above; the whole kernel until the
// second half of round 2) makes the extraction loop run max-over-lanes trips (27.5 per chunk on the bench document for 10.3 indexes per lane on average -- 39 % of the
// lanes do useful work).  Here a warp takes a UNIT of two consecutive chunks (4 KiB of input, ~660 indexes; lane t holds the
// four 32-bit mask words of bytes [128 t, 128 t + 128)), and every lane extracts the SAME number q = ceil(K / 32) of
// consecutive indexes of the unit's output:
//   1. the unit's non-empty mask words are compacted into shared memory in stream order as 16-byte entries {word bit-reversed,
//      index value of its bit 31, exclusive prefix count} (index = value - bfind(word)); the k-th empty word fills the k-th
//      slot behind them with a sentinel, so all 128 slots are written;
//   2. lane t binary-searches the prefix counts for the word that holds output t * q, drops the bits before it (a binary
//      select, no loop), and then runs exactly q trips of {next word if this one is used up; find, clear, subtract, store}
//      -- uniform trip count, no divergence, and with q forced odd the staging stores of the 32 lanes (stride q) never
//      share a bank;
//   3. the staged indexes go out as 16-byte vectors exactly as before.
// Units with more than CAP indexes (denser than 0.19 structurals per byte) take the per-chunk path (flatten_chunk).
// BitIndexer.write, reference json_structural_indexer.mojo:46-58.
// ---------------------------------------------------------------------------------------------
template <int FW>
struct Flatten2Cfg {
    static constexpr int THREADS = FW * 32;
    static constexpr int MIN_CTAS = 11;                           // resident CTAs per SM the register budget must allow
    static constexpr int CAP = 768;                               // indexes of a unit flattened through the balanced path
    static constexpr int QMAX = ((CAP + 31) / 32) | 1;            // trips per lane (odd)
    static constexpr int STAGE = 32 * QMAX + 4;                   // every lane writes q slots (the last ones past K) + output phase
    static constexpr int NVEC = (CAP + 3 + 3) / 4;                // 16-byte vectors the copy-out may have to move
    // per warp: 128 entries {word bit-reversed, address of the next non-empty entry} in stream order (word j of lane t at
    // 32 t + 8 j), the sentinel entry at 1024; the staging area; the prefix counts (four 16-bit values per lane); the lane
    // that holds the first output of every lane's share
    static constexpr int ENT_OFF = 0;
    static constexpr int STAGE_OFF = 1024 + 16;
    static constexpr int PX_OFF = STAGE_OFF + STAGE * 4;
    static constexpr int TAB_OFF = PX_OFF + 256;
    static constexpr int WARP_BYTES = ((TAB_OFF + 32) + 15) & ~15;
    static constexpr int SMEM_BYTES = FW * WARP_BYTES;
    static_assert(QMAX < 64 && CAP + QMAX < 4200, "range of the division table");
    static_assert(STAGE >= 512 + 4, "the per-chunk fallback stages up to 512 indexes");
    static_assert(STAGE_OFF % 16 == 0 && PX_OFF % 16 == 0, "16-byte vectors");
};
__constant__ uint32_t FL2_MAGIC[64] = {SJ_FL2_MAGIC_VALUES};   // floor(x / q) = fl2_div(x, FL2_MAGIC[q]), stage1_core.cuh

// q trips of the balanced extraction loop (q >= 1, warp-uniform).  w: current word (bit-reversed; may be 0 = used up), vb: the
// index value of its bit 31, na: shared-memory address of the next non-empty entry {word, address of the one after it} (the
// sentinel entry points at itself), sp: shared-memory address of this lane's first slot.  The value base of an entry follows
// from its address: vb = 4 * address + vc (entries are 8 bytes and cover 32 input bytes each).
__device__ __forceinline__ void flatten_balanced_loop(uint32_t w, uint32_t vb, uint32_t na, uint32_t sp, uint32_t q, uint32_t vc) {
    asm volatile(
        "{\n"
        ".reg .pred p, c;\n"
        ".reg .u32 h, m, x, n;\n"
        "mov.u32 n, %4;\n"
        "FB_LOOP:\n"
        "setp.eq.u32 p, %0, 0;\n"
        "@p mad.lo.u32 %1, %2, 4, %5;\n"
        "@p ld.shared.v2.u32 {%0, %2}, [%2];\n"
        "bfind.u32 h, %0;\n"
        "shl.b32 m, 1, h;\n"
        "xor.b32 %0, %0, m;\n"
        "sub.u32 x, %1, h;\n"
        "st.shared.u32 [%3], x;\n"
        "add.u32 %3, %3, 4;\n"
        "sub.u32 n, n, 1;\n"
        "setp.ne.u32 c, n, 0;\n"
        "@c bra FB_LOOP;\n"
        "}\n"
        : "+r"(w), "+r"(vb), "+r"(na), "+r"(sp)
        : "r"(q), "r"(vc)
        : "memory");
}

__device__ __forceinline__ void sts_u2(uint32_t a, uint32_t x, uint32_t y) {
    asm volatile("st.shared.v2.u32 [%0], {%1,%2};" ::"r"(a), "r"(x), "r"(y) : "memory");
}

// units of two chunks in [chunk_begin, chunk_end): unit u = chunks chunk_begin + 2u and + 1 (the last one may be missing)
template <int FW>
__global__ void __launch_bounds__(FW * 32, Flatten2Cfg<FW>::MIN_CTAS) stage1_flatten2_kernel(const Stage1Params P, uint32_t chunk_begin, uint32_t chunk_end) {
    using Cfg = Flatten2Cfg<FW>;
    extern __shared__ __align__(128) uint8_t smem_raw[];
    const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    uint8_t *wbase = smem_raw + warp * Cfg::WARP_BYTES;
    uint32_t *stage = reinterpret_cast<uint32_t *>(wbase + Cfg::STAGE_OFF);
    const uint32_t ent0 = smem_u32(wbase), px0 = smem_u32(wbase + Cfg::PX_OFF), tab0 = smem_u32(wbase + Cfg::TAB_OFF);
    const uint32_t c0 = chunk_begin + (blockIdx.x * FW + warp) * 2u;
    grid_dependency_wait();
    if (c0 >= chunk_end) return;
    const bool two = c0 + 1u < chunk_end;
    const uint32_t half = lane >> 4;                       // lanes 16..31 hold chunk c0 + 1
    const bool have = half == 0u || two;
    const uint32_t gave_up = P.spec_flag ? __ldcg(P.spec_flag) : 0u;   // stream pipeline only; loaded together with the carries
    const uint64_t carry = have ? __ldcg(reinterpret_cast<const unsigned long long *>(P.carry + c0 + half)) : 0ull;
    if (P.spec_flag && gave_up == P.gen) return;
    // this lane's 128 input bytes = two consecutive 64-bit words of its chunk's plane
    uint4 mw = make_uint4(0u, 0u, 0u, 0u);
    if (have) {
        const uint8_t *mp = reinterpret_cast<const uint8_t *>(P.masks) + (size_t)(c0 + half) * 512u + ((uint32_t)(carry >> 63) * 256u + (lane & 15u) * 16u);
        asm volatile("ld.global.cs.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(mw.x), "=r"(mw.y), "=r"(mw.z), "=r"(mw.w) : "l"(mp) : "memory");
    }
    const uint32_t na = (uint32_t)__popc(mw.x), nb = na + (uint32_t)__popc(mw.y), nc = nb + (uint32_t)__popc(mw.z), n = nc + (uint32_t)__popc(mw.w);
    const uint32_t incl = warp_inclusive_sum(n);
    const uint32_t Kt = __shfl_sync(0xFFFFFFFFu, incl, 31);
    const uint64_t first = __shfl_sync(0xFFFFFFFFu, (unsigned long long)carry, 0) & CARRY_RANK_MASK;   // the unit's indexes are out[first .. first + Kt)
    if (Kt > (uint32_t)Cfg::CAP) {   // a dense unit: chunk by chunk, one 64-bit word per lane
        for (uint32_t j = 0; j < (two ? 2u : 1u); j++) {
            const uint64_t cj = __ldcg(reinterpret_cast<const unsigned long long *>(P.carry + c0 + j));
            const uint64_t sj = __ldcs(reinterpret_cast<const unsigned long long *>(P.masks + (size_t)(c0 + j) * 64 + (uint32_t)(cj >> 63) * 32 + lane));
            flatten_chunk<512>(P, c0 + j, cj, sj, stage, (int)lane);
            __syncwarp();
        }
        return;
    }
    if (Kt == 0u) return;
    const uint32_t sentinel = ent0 + 1024u;
    const uint32_t q = fl2_share(Kt);                       // every lane's share: q consecutive outputs (odd: conflict-free staging stores)
    {   // this lane's four entries, their prefix counts, and the lanes whose share starts inside its 128 bytes
        const uint32_t e = incl - n;
        const uint32_t mine = ent0 + lane * 32u;
        // the next non-empty word after this lane's: the first one of the next lane that has any
        const uint32_t any = __ballot_sync(0xFFFFFFFFu, n != 0u);
        const uint32_t above = any & (0xFFFFFFFEu << lane);
        const uint32_t f = mw.x ? 0u : mw.y ? 8u : mw.z ? 16u : 24u;          // offset of this lane's first non-empty entry
        const uint32_t src = (uint32_t)__ffs((int)above) - 1u;                 // (none: the value is not used)
        const uint32_t fs = __shfl_sync(0xFFFFFFFFu, f, src & 31u);
        const uint32_t a3 = above ? ent0 + src * 32u + fs : sentinel;
        const uint32_t a2 = mw.w ? mine + 24u : a3;
        const uint32_t a1 = mw.z ? mine + 16u : a2;
        const uint32_t a0 = mw.y ? mine + 8u : a1;
        asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(mine), "r"(__brev(mw.x)), "r"(a0), "r"(__brev(mw.y)), "r"(a1) : "memory");
        asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(mine + 16u), "r"(__brev(mw.z)), "r"(a2), "r"(__brev(mw.w)), "r"(a3) : "memory");
        sts_u2(px0 + lane * 8u, e | ((e + na) << 16), (e + nb) | ((e + nc) << 16));
        if (lane == 0u) sts_u2(sentinel, 0xFFFFFFFFu, sentinel);
        // shares u with e <= u q < e + n start here
        const uint32_t M = FL2_MAGIC[q];
        const uint32_t u_hi = fl2_div(e + n + q - 1u, M);
        for (uint32_t u = fl2_div(e + q - 1u, M); u < u_hi; u++)
            asm volatile("st.shared.u8 [%0], %1;" ::"r"(tab0 + u), "r"(lane) : "memory");
    }
    __syncwarp();
    const uint32_t j0 = lane * q;                           // this lane's share: outputs [j0, j0 + q)
    const bool live = j0 < Kt;                              // (a lane past the end starts used up and only reads the sentinel)
    uint32_t w = 0u, vb = 0u, nxt = sentinel;
    if (live) {
        uint32_t t, rx, ry;
        asm volatile("ld.shared.u8 %0, [%1];" : "=r"(t) : "r"(tab0 + lane) : "memory");
        asm volatile("ld.shared.v2.u32 {%0,%1}, [%2];" : "=r"(rx), "=r"(ry) : "r"(px0 + t * 8u) : "memory");
        // the last of that lane's words whose prefix count is <= j0 (an empty word repeats the count of the word after it)
        const uint32_t p1 = rx >> 16, p2 = ry & 0xFFFFu, p3 = ry >> 16;
        uint32_t j = 0u, pj = rx & 0xFFFFu;
        if (p1 <= j0) { j = 1u; pj = p1; }
        if (p2 <= j0) { j = 2u; pj = p2; }
        if (p3 <= j0) { j = 3u; pj = p3; }
        uint32_t ex, ey;
        asm volatile("ld.shared.v2.u32 {%0,%1}, [%2];" : "=r"(ex), "=r"(ey) : "r"(ent0 + t * 32u + j * 8u) : "memory");
        w = drop_high_bits(ex, j0 - pj);                    // the bits that belong to the lanes before this one
        nxt = ey;
        vb = c0 * 2048u - P.mis + 31u + t * 128u + j * 32u;
    }
    const uint32_t vc = c0 * 2048u - P.mis + 31u - 4u * ent0;   // value base of the entry at address A: 4 A + vc
    const uint32_t a = ((uint32_t)first + out_phase(P.out)) & 3u;
    flatten_balanced_loop(w, vb, nxt, smem_u32(stage + a + j0), q, vc);
    __syncwarp();
    copy_out_warp_n<Cfg::NVEC>(stage, a, Kt, P.out, first, P.cap, lane);
}

#endif  // __CUDACC__

}  // namespace sjb200
