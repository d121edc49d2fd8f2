// stage1_persistent.cuh -- persistent, warp-specialised stage-1 kernel, and the tile steps it shares with the split pair's
// classify kernel (stage1_split.cuh).
//
// Arithmetic and look-back descriptors are those of stage1_kernel.cuh; what this organisation decides is who waits for whom.
// Rather than have every warp of a tile sit at a barrier while one warp walks the look-back chain, a CTA is NW compute
// warps + 1 scan warp and loops over tiles drawn from the ticket counter:
//   scan warp    : for every tile of the CTA, runs the look-back, publishes the inclusive prefix and hands
//                  (parity, output cursor) to the compute warps.  It does nothing else, so a slow look-back never
//                  delays a load or an aggregate.
//   compute warp : phase 1 of tile i (bytes -> dual structural masks), then flattens tile i-1, whose look-back
//                  ran concurrently with phase 1 of tile i.  Indexes are staged per warp, so compute warps never
//                  barrier with each other; the last warp to finish phase 1 publishes the tile aggregate itself, and
//                  the last warp to pull a tile into registers draws the next ticket and starts its bulk copy
//                  (cp.async.bulk), so the copy overlaps the whole of phase 1.
// All hand-offs are mbarriers in shared memory (SYNCS in SASS); there is no __syncthreads in the loop.
#pragma once
#include "stage1_kernel.cuh"

namespace sjb200 {

#if defined(__CUDACC__)

__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}

template <int NW>
struct PersistCfg {
    static constexpr int THREADS = (NW + 1) * 32;
    static constexpr int TILE = NW * 2048;
    static constexpr int WCAP = 512;                           // staged indexes per warp (density <= 0.25 per 2 KiB)
    static constexpr int IN_BYTES = 16 + TILE;                 // halo + tile, single buffer
    static constexpr int STAGE_BYTES = NW * (WCAP + 4) * 4;
    static constexpr int SMEM_BYTES = ((IN_BYTES + 127) & ~127) + STAGE_BYTES;
    // registers per thread: chosen so that enough CTAs of this shape are resident per SM (64 K registers / SM)
    static constexpr int MAXREG = NW >= 24 ? 72 : (NW == 16 ? 56 : (NW == 8 ? 56 : (NW == 4 ? 64 : 80)));
};

struct TileSlot {                 // hand-off of one tile between the compute warps and the scan warp
    uint32_t wc0[32], wc1[32], wflags[32];
    uint32_t R[32], off0[32], off1[32];
    uint64_t agg;                 // packed aggregate of the tile (what was published)
    uint32_t tail;
    uint32_t arrived;             // compute warps done with phase 1 of this tile
    uint32_t s_in, base;          // from the look-back (persistent kernel only)
    int32_t tile;
};

// Draws the next ticket into `tile_of`: -1 when the tickets are used up, else the tile, whose bulk copy into `dst` (16-byte
// halo at [0, 16), the tile from 16 on) is started on barrier `bar`.  Returns whether there was a tile.
template <int TILE>
__device__ __forceinline__ bool fetch_tile(const Stage1Params &P, uint32_t *ticket, int32_t &tile_of, uint32_t dst, uint32_t bar) {
    const uint32_t k = P.tile_begin + atomicAdd(ticket, 1u);
    if (k >= P.tile_end) {
        tile_of = -1;
        return false;
    }
    const int t = (int)k;
    tile_of = t;
    TRACE(P, t, 0, gtime());  // ticket drawn / copy issued
    const int64_t tb = (int64_t)t * TILE;
    int64_t nbytes = (int64_t)P.alen - tb;
    nbytes = nbytes > TILE ? TILE : nbytes;
    nbytes = (nbytes + 15) & ~15ll;
    const uint32_t halo = t > 0 ? 16u : 0u;
    mbar_expect_tx(bar, (uint32_t)nbytes + halo);
    bulk_load(dst + 16u - halo, P.abase + tb - halo, (uint32_t)nbytes + halo, bar);
    return true;
}

// Compute warp `warp` leaves its phase-1 summary in the slot; the last of the NW warps to do so builds the tile aggregate
// and the per-warp offsets, publishes the AGG descriptor (tile 0 goes straight to its prefix) and arrives on `bar_sum`.
template <int NW>
__device__ __forceinline__ void publish_tile_aggregate(TileSlot &S, const LanePhase1 &ph, int warp, int lane, int tile, const Stage1Params &P,
                                                       uint32_t bar_sum) {
    uint32_t order = 0;
    if (lane == 0) {
        S.wc0[warp] = ph.wc0;
        S.wc1[warp] = ph.wc1;
        S.wflags[warp] = ph.wflags;
        if (warp == NW - 1) S.tail = ph.tail;
        __threadfence_block();
        order = atomicAdd(&S.arrived, 1u);
    }
    order = __shfl_sync(0xFFFFFFFFu, order, 0);
    if (order != NW - 1) return;
    __threadfence_block();
    const bool have = lane < NW;
    uint32_t R, off0, off1;
    const TileAgg agg = tile_aggregate(have ? S.wflags[lane] : 0u, have ? S.wc0[lane] : 0u, have ? S.wc1[lane] : 0u,
                                       S.tail, NW, lane, R, off0, off1);
    if (have) {
        S.R[lane] = R;
        S.off0[lane] = off0;
        S.off1[lane] = off1;
    }
    const uint64_t packed = desc_pack_agg(P.gen, agg);
    if (lane == 0) {
        if (tile > 0) st_desc(P.desc + tile, packed);
        TRACE(P, tile, 2, gtime());  // aggregate published
        S.agg = packed;
        S.tile = tile;
        S.arrived = 0;
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(bar_sum);     // release: slot contents visible to the scan warp
}

struct TileStart {
    uint32_t s_in;   // in-string parity entering the tile
    uint32_t base;   // rank of the tile's first index in the output
};
// Scan warp: the look-back for tile `cur` with aggregate `agg`, then its PREFIX descriptor, the progress word (last tile of
// the launch) and the verdict (last tile of the document).
__device__ __forceinline__ TileStart publish_tile_prefix(const Stage1Params &P, const TileAgg &agg, int cur, int lane) {
    LookbackResult lb = {0, 0, 0};
    if (cur > 0) lb = lookback(P.desc, P.gen, cur, lane);
    const uint32_t s_in = lb.s_in & 1u;
    const uint32_t total = s_in ? agg.c[1] : agg.c[0];
    TilePrefix pre;
    pre.s_out = s_in ^ agg.par;
    pre.e_out = agg.e_out;
    pre.p_out = agg.p_out;
    pre.err = lb.err | ((s_in ? agg.un[1] : agg.un[0]) ? EF_UNESCAPED : 0u) | (agg.u8 ? EF_UTF8 : 0u);
    pre.count = lb.base + total;
    if (lane == 0) {
        st_desc(P.desc + cur, desc_pack_prefix(P.gen, pre));
        if (cur == (int)P.tile_end - 1 && P.progress) *P.progress = pre.count;
        if (cur == (int)P.ntiles - 1) write_verdict(P, pre);
    }
    return {s_in, lb.base};
}

template <int NW, bool UTF8>
__global__ void __launch_bounds__((NW + 1) * 32) __maxnreg__(PersistCfg<NW>::MAXREG) stage1_persistent_kernel(const Stage1Params P) {
    using Cfg = PersistCfg<NW>;
    constexpr int TILE = Cfg::TILE;
    extern __shared__ __align__(128) uint8_t smem_raw[];
    uint8_t *smem_in = smem_raw;                                           // [0,16) halo, [16, 16+TILE) tile
    uint32_t *smem_stage = reinterpret_cast<uint32_t *>(smem_raw + ((Cfg::IN_BYTES + 127) & ~127));
    constexpr int NS = 4;                        // hand-off slots (a tile is flushed one iteration after its phase 1)
    __shared__ __align__(8) uint64_t s_bar[2 + 2 * NS];  // 0 in_full, 1 in_empty, 2.. sum_full[NS], 2+NS.. carry_full[NS]
    __shared__ TileSlot s_slot[NS];
    __shared__ int32_t s_tile_of;               // tile held by the input buffer, -1 = no more work
    __shared__ uint32_t s_loaded;               // compute warps that have pulled the current tile into registers

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    grid_dependency_wait();   // as the pipeline's fallback it is launched while the flatten kernel drains (a no-op otherwise)
    if (P.spec_flag && __ldcg(P.spec_flag) != P.gen) {
        // launched as the exact fallback of the stream pipeline (stage1_stream.cuh) and not needed: only keep the
        // ticket-counter alternation intact
        if (blockIdx.x == 0 && tid == 0) {
            P.ticket[(P.ticket_sel + 1) & 1u] = 0;
            if (__ldcg(P.spec_flag + 1) == P.gen) {
                // the stream classify kernel found a violation among the lanes whose validation it had deferred: same
                // place in the verdict as in write_verdict (after EMPTY, before SUCCESS; reference :185-186 slot)
                Stage1Result *r = P.result;
                r->utf8_error = 1;
                if ((P.flags & 1u) && r->error == ERR_SUCCESS) {
                    r->error = ERR_UTF8_ERROR;
                    if (P.dev_status) P.dev_status[0] = ERR_UTF8_ERROR;
                }
            }
        }
        return;
    }
    const uint32_t bar_in_full = smem_u32(&s_bar[0]), bar_in_empty = smem_u32(&s_bar[1]);
    const uint32_t bar_sum = smem_u32(&s_bar[2]), bar_carry = smem_u32(&s_bar[2 + NS]);  // + 8 * slot

    if (tid == 0) {
        mbar_init(bar_in_full, 1);
        mbar_init(bar_in_empty, NW);
        s_loaded = 0;
        for (int k = 0; k < NS; k++) {
            mbar_init(bar_sum + 8 * k, 1);
            mbar_init(bar_carry + 8 * k, 1);
            s_slot[k].arrived = 0;
        }
        fence_mbar_init();
        // two ticket counters used alternately by successive launches: clear the one the NEXT launch will use
        if (blockIdx.x == 0) P.ticket[(P.ticket_sel + 1) & 1u] = 0;
    }
    __syncthreads();
    uint32_t *ticket = P.ticket + (P.ticket_sel & 1u);

    // produce(it): one thread draws the ticket of iteration `it` and starts its bulk copy into the (free) input buffer;
    // when the tickets are exhausted it wakes the compute warps and the scan warp with "no more work"
    auto produce = [&](int it) {
        if (!fetch_tile<TILE>(P, ticket, s_tile_of, smem_u32(smem_in), bar_in_full)) {
            s_slot[it & (NS - 1)].tile = -1;
            mbar_arrive(bar_in_full);
            mbar_arrive(bar_sum + 8 * (it & (NS - 1)));
        }
    };
    if (tid == 0) produce(0);

    if (warp == NW) {
        // =============================== scan warp ===============================
        for (int i = 0;; i++) {
            const int slot = i & (NS - 1);
            mbar_wait(bar_sum + 8 * slot, (uint32_t)(i / NS) & 1u);
            TileSlot &S = s_slot[slot];
            const int cur = *reinterpret_cast<volatile int32_t *>(&S.tile);
            if (cur < 0) break;
            TRACE(P, cur, 3, gtime());  // look-back starts
            const TileStart st = publish_tile_prefix(P, desc_unpack_agg(S.agg), cur, lane);
            if (lane == 0) {
                S.s_in = st.s_in;
                S.base = st.base;
                TRACE(P, cur, 4, gtime());  // look-back done
                mbar_arrive(bar_carry + 8 * slot);  // release: S.s_in / S.base visible to the waiters
            }
            __syncwarp();
        }
    } else {
        // =============================== compute warps ===============================
        uint32_t *stage = smem_stage + warp * (Cfg::WCAP + 4);
        // the previous tile of this warp, waiting for its look-back (registers).  Holding two tiles was measured: worse.
        struct Held {
            uint64_t m0, m1;
            uint32_t c0, c1, v0;
        };
        Held old1 = {0, 0, 0, 0, 0};
        bool held = false;
        int i = 0;

        // flatten a held tile (iteration `it`) once its look-back has delivered parity and cursor
        auto flush_old = [&](const Held &old, int it) {
            const int slot = it & (NS - 1);
#if SJ_TRACE
            const uint64_t tc0 = gtime();
#endif
            mbar_wait(bar_carry + 8 * slot, (uint32_t)(it / NS) & 1u);
            const TileSlot &S = s_slot[slot];
#if SJ_TRACE
            if (lane == 0 && (warp == 0 || warp == NW - 1)) { TRACE(P, S.tile, warp == 0 ? 8 : 9, gtime() - tc0); TRACE(P, S.tile, warp == 0 ? 10 : 11, gtime()); }  // carry wait, flush start
#endif
            const uint32_t s_in = S.s_in & 1u;
            const uint32_t s_w = (s_in ^ S.R[warp]) & 1u;
            const uint64_t structural = s_w ? old.m1 : old.m0;
            const uint32_t cnt = s_w ? old.c1 : old.c0;
            const uint32_t incl = warp_inclusive_sum(cnt);
            const uint32_t wtotal = __shfl_sync(0xFFFFFFFFu, incl, 31);
            const uint64_t first = (uint64_t)S.base + (s_in ? S.off1[warp] : S.off0[warp]);  // the warp's first index
            if (wtotal <= (uint32_t)Cfg::WCAP) {
                const uint32_t a = ((uint32_t)first + out_phase(P.out)) & 3u;
                flatten_to(stage + a + (incl - cnt), structural, old.v0);
                __syncwarp();
                copy_out_warp_n<128>(stage, a, wtotal, P.out, first, P.cap, (uint32_t)lane);
                __syncwarp();  // the staging area is reused by the next tile
#if SJ_TRACE
                if (lane == 0 && (warp == 0 || warp == NW - 1)) TRACE(P, S.tile, warp == 0 ? 12 : 13, gtime());  // flush done
#endif
            } else {
                flatten_direct(P.out, P.cap, first + (incl - cnt), structural, old.v0);
            }
        };

        while (true) {
#if SJ_TRACE
            const uint64_t tw0 = gtime();
#endif
            mbar_wait(bar_in_full, (uint32_t)i & 1u);
            const int tile = *reinterpret_cast<volatile int32_t *>(&s_tile_of);
            if (tile < 0) break;
#if SJ_TRACE
            if (lane == 0 && (warp == 0 || warp == NW - 1)) { TRACE(P, tile, warp == 0 ? 5 : 6, gtime() - tw0); TRACE(P, tile, warp == 0 ? 1 : 7, gtime()); }  // input wait, phase-1 start
#endif
            const int slot = i & (NS - 1);
            const int64_t tb = (int64_t)tile * TILE;
            LanePhase1 ph;
            {
                LaneInput in;
                warp_load<UTF8>(in, smem_in + 16, warp, lane, tile, tb, TILE, P);
                __syncwarp();
                if (lane == 0) {                            // this warp no longer needs the input buffer
                    __threadfence_block();
                    if (atomicAdd(&s_loaded, 1u) == NW - 1) {
                        s_loaded = 0;                       // everyone has it in registers: refill the buffer now
                        __threadfence_block();
                        produce(i + 1);
                    }
                }
                warp_compute<UTF8>(ph, in, lane, P);
            }
            publish_tile_aggregate<NW>(s_slot[slot], ph, warp, lane, tile, P, bar_sum + 8 * slot);
            // flatten tile i-1: its look-back ran on the scan warp during phase 1 of tile i
            if (held) flush_old(old1, i - 1);
            old1.m0 = ph.m0;
            old1.m1 = ph.m1;
            old1.c0 = ph.c0;
            old1.c1 = ph.c1;
            old1.v0 = ph.v0;
            held = true;
            i++;
        }
        if (held) flush_old(old1, i - 1);
    }
}

#endif  // __CUDACC__

}  // namespace sjb200
