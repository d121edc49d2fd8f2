// tests/emu/emulate_stage1.cpp -- TEST INFRASTRUCTURE.
//
// Host-side lane-by-lane emulation of the CUDA stage-1 kernel's phase structure, built from the very
// same header (mojo_simdjson_b200/csrc/stage1_core.cuh) the kernel compiles.  It lets the CPU test suite
// check every bit trick (byte transpose, bit-plane butterfly, plane classifier, bit-sliced UTF-8, local
// carry resolution, dual-parity structural masks, descriptor packing, look-back window algebra, edge
// masking, index arithmetic) against the oracle with no GPU.  Warp collectives are emulated by looping over
// the 32 lanes between phases; the decoupled look-back is emulated over the packed descriptors with a small
// window and an arbitrary pattern of "which earlier tiles already published their inclusive prefix".
// It is NOT a CPU fallback: the product library never links it.
#include <stdint.h>
#include <string.h>
#include <vector>

#include "../../mojo_simdjson_b200/csrc/stage1_core.cuh"

using namespace sjb200;

namespace {

uint32_t mask_word(uint32_t w, int64_t g, int64_t vbeg, int64_t vend) {
    // keep the bytes of w whose aligned coordinate g+k lies in [vbeg, vend); others become 0x20
    int64_t lo = vbeg - g, hi = vend - g;
    if (lo < 0) lo = 0;
    if (lo > 4) lo = 4;
    if (hi < 0) hi = 0;
    if (hi > 4) hi = 4;
    uint32_t mh = hi >= 4 ? 0xFFFFFFFFu : ((1u << (8 * hi)) - 1u);
    uint32_t ml = lo >= 4 ? 0xFFFFFFFFu : ((1u << (8 * lo)) - 1u);
    uint32_t m = hi > lo ? (mh & ~ml) : 0u;
    return (w & m) | (0x20202020u & ~m);
}

struct Lane {
    LaneMasks m;
    LaneQuotes q;
    LaneDual d;
    uint32_t u8err, rel, c0, c1;
};

// mirrors tile_prev_state() of the kernel
PrevState tile_prev_state(const uint8_t *smem_tile, int64_t tile, const std::vector<uint64_t> &desc) {
    PrevState st = {0, 0, 0};
    if (tile == 0) return st;
    uint32_t bsm = 0;
    for (int l = 0; l < 16; l++) bsm |= (uint32_t)(smem_tile[-1 - l] == 0x5C) << l;
    st = prev_state(bsm, 16, smem_tile[-1]);
    if (st.unresolved) {
        const uint64_t d = desc[(size_t)tile - 1];
        const uint32_t f = (uint32_t)(d >> 36);
        if (st.unresolved & 1u) st.e = (f >> 4) & 1u;
        if (st.unresolved & 2u) st.p = (f >> 3) & 1u;
        st.unresolved = 0;
    }
    return st;
}

// mirrors warp_prev_state()
PrevState warp_prev_state(const uint8_t *smem_tile, int woff, int64_t tb, int64_t vbeg, int64_t vend, bool edge, int64_t tile,
                          const std::vector<uint64_t> &desc) {
    uint32_t bsm = 0, c1 = 0;
    for (int l = 0; l < 32; l++) {
        uint32_t c = smem_tile[woff - 1 - l];
        if (edge) {
            const int64_t g = tb + woff - 1 - l;
            if (g < vbeg || g >= vend) c = 0x20;
        }
        if (l == 0) c1 = c;
        bsm |= (uint32_t)(c == 0x5C) << l;
    }
    PrevState st = prev_state(bsm, 32, c1);
    if (st.unresolved) {
        const PrevState t = tile_prev_state(smem_tile, tile, desc);
        const uint32_t room = (uint32_t)woff - (tile == 0 ? (uint32_t)vbeg : 0u);
        if (st.unresolved & 1u) {
            const uint32_t r = backslash_run_before(smem_tile + woff, room);
            st.e = r < room ? (r & 1u) : escaped_after_run(room, t.e);
        }
        if (st.unresolved & 2u) {
            const uint32_t r = backslash_run_before(smem_tile + woff - 1, room - 1);
            st.p = r < room - 1 ? (r & 1u) : escaped_after_run(room - 1, t.e);
        }
        st.unresolved = 0;
    }
    return st;
}

struct LookbackResult {
    uint32_t s_in, base, err;
};
// mirrors lookback(): `window` lanes instead of 32; visible[j] says which descriptor kind tile j shows
LookbackResult lookback(const std::vector<uint64_t> &agg, const std::vector<uint64_t> &prefix, const std::vector<char> &shows_prefix,
                        int64_t tile, int window) {
    SpanAcc acc = span_empty();
    int64_t base = tile - 1;
    for (;;) {
        // lane l looks at tile base - l
        int k = window;
        std::vector<uint64_t> d((size_t)window, 0);
        for (int l = window - 1; l >= 0; l--) {
            const int64_t j = base - l;
            bool is_prefix = true;
            if (j >= 0) {
                is_prefix = shows_prefix[(size_t)j] != 0;
                d[(size_t)l] = is_prefix ? prefix[(size_t)j] : agg[(size_t)j];
            }
            if (is_prefix) k = l;  // ends with the lowest such lane = nearest tile
        }
        uint32_t pbm = 0;
        for (int l = 0; l < k; l++) pbm |= (desc_unpack_agg(d[(size_t)l]).par & 1u) << l;
        SpanAcc win = span_empty();
        win.par = (uint32_t)popc32(pbm) & 1u;
        for (int l = 0; l < k; l++) {
            const TileAgg a = desc_unpack_agg(d[(size_t)l]);
            const uint32_t rel = (uint32_t)popc32(pbm & ~((2u << l) - 1u)) & 1u;
            win.c[0] += a.c[rel];
            win.c[1] += a.c[rel ^ 1u];
            win.un[0] |= a.un[rel];
            win.un[1] |= a.un[rel ^ 1u];
            win.u8 |= a.u8;
        }
        acc = span_concat(win, acc);
        if (k < window) {
            TilePrefix p = {0, 0, 0, 0, 0};
            if (base - k >= 0) p = desc_unpack_prefix(d[(size_t)k]);
            LookbackResult r;
            r.s_in = p.s_out ^ acc.par;
            r.base = p.count + acc.c[p.s_out];
            r.err = p.err | (acc.un[p.s_out] ? EF_UNESCAPED : 0u) | (acc.u8 ? EF_UTF8 : 0u);
            return r;
        }
        base -= window;
    }
}

}  // namespace

extern "C" int32_t emu_stage1(const uint8_t *buf, uint64_t len, uint32_t mis, int warps, uint32_t *out, uint64_t cap,
                              uint32_t *n_out, uint64_t *n_written_out, int32_t *utf8_err_out, uint32_t flags) {
    if (n_written_out) *n_written_out = 0;
    if (utf8_err_out) *utf8_err_out = 0;
    if (len > 0xFFFFFFFFull) return 1;
    if (len == 0) return 13;
    const uint32_t gen = 0x5A5A5u;
    const int64_t TILE = (int64_t)warps * 2048;
    const int64_t alen = (int64_t)mis + (int64_t)len;
    const int64_t ntiles = (alen + TILE - 1) / TILE;
    // aligned image of memory: hostile bytes wherever the kernel must not look
    std::vector<uint8_t> mem((size_t)(ntiles * TILE + 64), 0);
    for (size_t i = 0; i < mem.size(); i++) mem[i] = (i & 1) ? 0x5C : 0xF4;
    memcpy(mem.data() + mis, buf, (size_t)len);

    std::vector<uint64_t> d_agg((size_t)ntiles), d_prefix((size_t)ntiles), d_either((size_t)ntiles);
    std::vector<char> shows_prefix((size_t)ntiles);
    uint64_t total_written = 0;
    TilePrefix last = {0, 0, 0, 0, 0};
    std::vector<uint8_t> smem((size_t)TILE + 16);

    for (int64_t tile = 0; tile < ntiles; tile++) {
        const int64_t tb = tile * TILE;
        for (size_t i = 0; i < smem.size(); i++) smem[i] = 0x5C;  // stale shared memory
        int64_t nbytes = alen - tb;
        if (nbytes > TILE) nbytes = TILE;
        nbytes = (nbytes + 15) & ~15ll;
        memcpy(smem.data() + 16, mem.data() + tb, (size_t)nbytes);
        if (tile > 0) memcpy(smem.data(), mem.data() + tb - 16, 16);
        const uint8_t *smem_tile = smem.data() + 16;
        const bool edge = (tile == 0) || (tb + TILE > alen);

        std::vector<Lane> L((size_t)warps * 32);
        std::vector<uint32_t> wc0(warps), wc1(warps), wflags(warps);
        uint32_t tail = 0;
        for (int w = 0; w < warps; w++) {
            const int woff = w * 2048;
            const PrevState wst = w == 0 ? tile_prev_state(smem_tile, tile, d_either)
                                         : warp_prev_state(smem_tile, woff, tb, mis, alen, edge, tile, d_either);
            uint32_t A = 0, O = 0;
            for (int l = 0; l < 32; l++) {
                Lane &ln = L[(size_t)w * 32 + l];
                const int64_t off = woff + (int64_t)l * 64;
                const int64_t g0 = tb + off;
                uint32_t words[16], prev;
                memcpy(words, smem_tile + off, 64);
                memcpy(&prev, smem_tile + off - 4, 4);
                if (edge) {
                    for (int k = 0; k < 16; k++) words[k] = mask_word(words[k], g0 + 4 * k, mis, alen);
                    prev = (g0 == 0) ? 0x20202020u : mask_word(prev, g0 - 4, mis, alen);
                }
                uint32_t pl[8], ph[8];
                bitplanes32(words, pl);
                bitplanes32(words + 8, ph);
                Classes32 cl, ch;
                Utf8Pre32 ul, uh;
                classify32<true>(pl, cl, ul);
                classify32<true>(ph, ch, uh);
                ln.m.bs = join64(cl.bs, ch.bs);
                ln.m.rq = join64(cl.rq, ch.rq);
                ln.m.op = join64(cl.op, ch.op);
                ln.m.ws = join64(cl.ws, ch.ws);
                ln.m.ctl = join64(cl.ctl, ch.ctl);
                Utf8Carry uc = utf8_carry_from_prev_word(prev);
                uint32_t tail_must;
                uint64_t ue = utf8_errors64(ul, uh, uc, &tail_must);
                ln.u8err = (ue != 0) || (g0 + 64 == alen && tail_must != 0);
                A |= (uint32_t)lane_all_backslash(ln.m.bs) << l;
                O |= lane_trailing_run_parity(ln.m.bs) << l;
            }
            uint32_t PB = 0, NQ = 0;
            for (int l = 0; l < 32; l++) {
                Lane &ln = L[(size_t)w * 32 + l];
                ln.q = lane_quotes(ln.m, warp_lane_e_in(A, O, l, wst.e));
                PB |= (uint32_t)(ln.q.ps >> 63) << l;
                NQ |= (uint32_t)(ln.q.nqs >> 63) << l;
            }
            uint32_t fl = 0;
            wc0[w] = wc1[w] = 0;
            for (int l = 0; l < 32; l++) {
                Lane &ln = L[(size_t)w * 32 + l];
                ln.rel = (uint32_t)popc32(PB & ((1u << l) - 1u)) & 1u;
                const uint32_t p_in = l ? ((NQ >> (l - 1)) & 1u) : wst.p;
                ln.d = lane_structurals_dual(ln.m, ln.q, ln.rel, p_in);
                ln.c0 = (uint32_t)popc64(ln.d.m0);
                ln.c1 = (uint32_t)popc64(ln.d.m1);
                wc0[w] += ln.c0;
                wc1[w] += ln.c1;
                fl |= (ln.d.u0 << 1) | (ln.d.u1 << 2) | (ln.u8err << 3);
            }
            wflags[w] = fl | ((uint32_t)popc32(PB) & 1u);
            if (w == warps - 1) tail = warp_lane_e_in(A, O, 32, wst.e) | ((NQ >> 31) << 1);
        }
        // ---- "warp 0": tile aggregate, look-back, prefix ----
        TileAgg agg;
        memset(&agg, 0, sizeof agg);
        std::vector<uint32_t> R(warps), off0(warps), off1(warps);
        uint32_t par = 0, run0 = 0, run1 = 0;
        for (int w = 0; w < warps; w++) {
            R[w] = par;
            const uint32_t t0 = R[w] ? wc1[w] : wc0[w], t1 = R[w] ? wc0[w] : wc1[w];
            off0[w] = run0;
            off1[w] = run1;
            run0 += t0;
            run1 += t1;
            agg.un[0] |= (wflags[w] >> (R[w] ? 2 : 1)) & 1u;
            agg.un[1] |= (wflags[w] >> (R[w] ? 1 : 2)) & 1u;
            agg.u8 |= (wflags[w] >> 3) & 1u;
            par ^= wflags[w] & 1u;
        }
        agg.par = par;
        agg.c[0] = run0;
        agg.c[1] = run1;
        agg.e_out = tail & 1u;
        agg.p_out = (tail >> 1) & 1u;
        d_agg[(size_t)tile] = desc_pack_agg(gen, agg);
        if (desc_gen(d_agg[(size_t)tile]) != gen || desc_status(d_agg[(size_t)tile]) != DESC_AGG) return -100;
        LookbackResult lb = {0, 0, 0};
        if (tile > 0) lb = lookback(d_agg, d_prefix, shows_prefix, tile, 4);
        const uint32_t s_in = lb.s_in & 1u;
        const uint32_t total = agg.c[s_in];
        TilePrefix pre;
        pre.s_out = s_in ^ agg.par;
        pre.e_out = agg.e_out;
        pre.p_out = agg.p_out;
        pre.err = lb.err | (agg.un[s_in] ? EF_UNESCAPED : 0u) | (agg.u8 ? EF_UTF8 : 0u);
        pre.count = lb.base + total;
        d_prefix[(size_t)tile] = desc_pack_prefix(gen, pre);
        if (desc_gen(d_prefix[(size_t)tile]) != gen || desc_status(d_prefix[(size_t)tile]) != DESC_PREFIX) return -101;
        // which kind later tiles will see for this tile: an irregular pattern, tile 0 always inclusive
        shows_prefix[(size_t)tile] = (tile == 0) || ((tile * 7 + tile / 3) % 5 == 0);
        d_either[(size_t)tile] = shows_prefix[(size_t)tile] ? d_prefix[(size_t)tile] : d_agg[(size_t)tile];
        last = pre;
        if (lb.base != total_written) return -102;  // the look-back must reproduce the running count
        // ---- flatten ----
        for (int w = 0; w < warps; w++) {
            const uint32_t sw = s_in ^ R[w];
            uint32_t rank = s_in ? off1[w] : off0[w];
            for (int l = 0; l < 32; l++) {
                Lane &ln = L[(size_t)w * 32 + l];
                const uint32_t s_lane = sw & 1u;  // ln.rel is already folded into m0 / m1
                uint64_t st = s_lane ? ln.d.m1 : ln.d.m0;
                const int64_t g0 = tb + (int64_t)w * 2048 + (int64_t)l * 64;
                while (st) {
                    int bit = __builtin_ctzll(st);
                    st &= st - 1;
                    const uint64_t o = (uint64_t)lb.base + rank++;
                    if (o < cap) out[o] = (uint32_t)(g0 + bit - (int64_t)mis);
                }
            }
            if (w == warps - 1 && rank != total) return -103;
        }
        total_written += total;
    }
    const uint64_t n = last.count;
    if (n_written_out) *n_written_out = n;
    if (utf8_err_out) *utf8_err_out = (last.err & EF_UTF8) ? 1 : 0;
    if (last.s_out) return 15;
    if (last.err & EF_UNESCAPED) return 14;
    if (n + 3 > cap) return 1;
    if (n_out) *n_out = (uint32_t)n;
    out[n] = (uint32_t)len;
    out[n + 1] = (uint32_t)len;
    out[n + 2] = 0;
    if (n == 0) return 13;
    if ((flags & 1u) && (last.err & EF_UTF8)) return 11;
    return 0;
}

// direct checks of the transposition on arbitrary 32 bytes
extern "C" void emu_bitplanes32(const uint8_t *bytes32, uint32_t *planes8) {
    uint32_t w[8];
    memcpy(w, bytes32, 32);
    bitplanes32(w, planes8);
}

// ---------------------------------------------------------------------------------------------------------------
// Stream pipeline (csrc/stage1_stream.cuh) on the host: per 2 KiB chunk the classify step with a 32-byte look-behind and
// no other knowledge of what precedes it, the two mask planes and the chunk summary; then the ordered scan in the same
// two levels as the kernels (blocks of 4096 summaries, block prefix, per-thread groups of 4 walked backwards); then the
// flatten step driven only by the carry words.  *spec_out = 1 iff a chunk could not resolve its escape carry locally
// (the GPU then hands the document to the persistent kernel); the output is unspecified in that case.
// ---------------------------------------------------------------------------------------------------------------
namespace {
struct Summary {
    uint32_t c0, c1, flags;
};
SpanAcc span_of(const Summary &s) {
    SpanAcc a;
    a.par = s.flags & 1u;
    a.c[0] = s.c0;
    a.c[1] = s.c1;
    a.un[0] = (s.flags >> 1) & 1u;
    a.un[1] = (s.flags >> 2) & 1u;
    a.u8 = (s.flags >> 3) & 1u;
    return a;
}
}  // namespace

extern "C" int32_t emu_stage1_stream(const uint8_t *buf, uint64_t len, uint32_t mis, uint32_t *out, uint64_t cap, uint32_t *n_out,
                                     uint64_t *n_written_out, int32_t *utf8_err_out, int32_t *spec_out, uint32_t flags) {
    if (spec_out) *spec_out = 0;
    if (len == 0) return 13;
    const int64_t alen = (int64_t)mis + (int64_t)len;
    const int64_t nchunks = (alen + 2047) / 2048;
    std::vector<uint8_t> mem((size_t)(nchunks * 2048 + 64));
    for (size_t i = 0; i < mem.size(); i++) mem[i] = (i & 1) ? 0x5C : 0xF4;  // hostile bytes around the document
    memcpy(mem.data() + mis, buf, (size_t)len);
    const int64_t last = nchunks - 1;
    const int64_t last_bytes = alen - last * 2048;

    std::vector<uint64_t> plane0((size_t)nchunks * 32), plane1((size_t)nchunks * 32);
    std::vector<Summary> sum((size_t)nchunks);
    std::vector<uint32_t> deferred((size_t)nchunks, 0u);
    std::vector<uint32_t> slots((size_t)nchunks * 8 * 18, 0xA5A5A5A5u);  // parked {planes[16], prev, ends} of deferred lanes
    std::vector<uint8_t> stage(32 + 2048);
    bool gave_up = false;
    for (int64_t c = 0; c < nchunks; c++) {
        // what the bulk copy brings: the chunk (the last one rounded up to 16 bytes) and 32 bytes before it; the rest of the
        // buffer is stale
        for (size_t i = 0; i < stage.size(); i++) stage[i] = 0x5C;
        const int64_t nb = c == last ? ((last_bytes + 15) & ~15ll) : 2048;
        memcpy(stage.data() + 32, mem.data() + c * 2048, (size_t)nb);
        if (c > 0) memcpy(stage.data(), mem.data() + c * 2048 - 32, 32);
        const uint8_t *chunk = stage.data() + 32;
        const bool edge = (c == 0) || (c == last && last_bytes < 2048);
        PrevState wst = {0, 0, 0};
        if (c > 0) {
            uint32_t bsm = 0;
            for (int l = 0; l < 32; l++) bsm |= (uint32_t)(chunk[-1 - l] == 0x5C) << l;
            wst = prev_state(bsm, 32, chunk[-1]);
        }
        if (wst.unresolved) gave_up = true;
        Lane L[32];
        uint32_t A = 0, O = 0;
        for (int l = 0; l < 32; l++) {
            Lane &ln = L[l];
            const int64_t g0 = c * 2048 + (int64_t)l * 64;
            uint32_t words[16], prev;
            memcpy(words, chunk + l * 64, 64);
            memcpy(&prev, chunk + l * 64 - 4, 4);
            const bool ends = (c == last) && ((int64_t)l * 64 + 64 == last_bytes);  // also when the last chunk is full
            if (edge) {
                for (int k = 0; k < 16; k++) words[k] = mask_word(words[k], g0 + 4 * k, mis, alen);
                prev = (g0 == 0) ? 0x20202020u : mask_word(prev, g0 - 4, mis, alen);
            }
            uint32_t pl[8], ph[8];
            bitplanes32(words, pl);
            bitplanes32(words + 8, ph);
            Classes32 cl, ch;
            classify_json32(pl, cl);
            classify_json32(ph, ch);
            ln.m.bs = join64(cl.bs, ch.bs);
            ln.m.rq = join64(cl.rq, ch.rq);
            ln.m.op = join64(cl.op, ch.op);
            ln.m.ws = join64(cl.ws, ch.ws);
            ln.m.ctl = join64(cl.ctl, ch.ctl);
            ln.u8err = 0;
            ln.c0 = ((pl[7] | ph[7]) != 0) || ((prev & 0x80808080u) != 0);  // any_hi (kept in c0 until the ballot below)
            ln.c1 = prev;
            ln.rel = ends;
            memcpy(&ln.d, pl, 0);  // (planes are recomputed below when needed)
            A |= (uint32_t)lane_all_backslash(ln.m.bs) << l;
            O |= lane_trailing_run_parity(ln.m.bs) << l;
        }
        uint32_t hi_lanes = 0;
        for (int l = 0; l < 32; l++) hi_lanes |= (uint32_t)(L[l].c0 != 0) << l;
        if (popc32(hi_lanes) <= 8) {
            deferred[(size_t)c] = hi_lanes;  // few lanes: parked for the second pass below (stage1_utf8_lanes_kernel)
            int rank = 0;
            for (int l = 0; l < 32; l++) {
                if (!((hi_lanes >> l) & 1u)) continue;
                const int64_t g0 = c * 2048 + (int64_t)l * 64;
                uint32_t words[16];
                memcpy(words, chunk + l * 64, 64);
                if (edge)
                    for (int k = 0; k < 16; k++) words[k] = mask_word(words[k], g0 + 4 * k, mis, alen);
                uint32_t *sl = slots.data() + ((size_t)c * 8 + rank++) * 18;
                bitplanes32(words, sl);
                bitplanes32(words + 8, sl + 8);
                sl[16] = L[l].c1;   // prev (already masked)
                sl[17] = L[l].rel;  // the document ends with this lane
            }
        } else {  // the whole warp takes the UTF-8 path
            for (int l = 0; l < 32; l++) {
                const int64_t g0 = c * 2048 + (int64_t)l * 64;
                uint32_t words[16];
                memcpy(words, chunk + l * 64, 64);
                if (edge)
                    for (int k = 0; k < 16; k++) words[k] = mask_word(words[k], g0 + 4 * k, mis, alen);
                uint32_t pl[8], ph[8];
                bitplanes32(words, pl);
                bitplanes32(words + 8, ph);
                Utf8Pre32 ul, uh;
                utf8_pre32(pl, ul);
                utf8_pre32(ph, uh);
                const Utf8Carry uc = utf8_carry_from_prev_word(L[l].c1);
                uint32_t tail_must;
                const uint64_t ue = utf8_errors64(ul, uh, uc, &tail_must);
                L[l].u8err = (ue != 0) || (L[l].rel && tail_must != 0);
            }
        }
        uint32_t PB = 0, NQ = 0;
        for (int l = 0; l < 32; l++) {
            L[l].q = lane_quotes(L[l].m, warp_lane_e_in(A, O, l, wst.e));
            PB |= (uint32_t)(L[l].q.ps >> 63) << l;
            NQ |= (uint32_t)(L[l].q.nqs >> 63) << l;
        }
        uint32_t fl = 0, wc0 = 0, wc1 = 0;
        for (int l = 0; l < 32; l++) {
            const uint32_t rel = (uint32_t)popc32(PB & ((1u << l) - 1u)) & 1u;
            const uint32_t p_in = l ? ((NQ >> (l - 1)) & 1u) : wst.p;
            const LaneDual d = lane_structurals_dual(L[l].m, L[l].q, rel, p_in);
            plane0[(size_t)c * 32 + l] = d.m0;
            plane1[(size_t)c * 32 + l] = d.m1;
            wc0 += (uint32_t)popc64(d.m0);
            wc1 += (uint32_t)popc64(d.m1);
            fl |= (d.u0 << 1) | (d.u1 << 2) | (L[l].u8err << 3);
        }
        sum[(size_t)c] = {wc0, wc1, fl | ((uint32_t)popc32(PB) & 1u)};
    }
    if (gave_up) {
        if (spec_out) *spec_out = 1;
        return 0;
    }
    // ---- stage1_utf8_lanes_kernel: one "thread" per parked slot ----
    bool u8_deferred_bad = false;
    for (int64_t c = 0; c < nchunks; c++) {
        const int cnt = popc32(deferred[(size_t)c]);
        for (int slot = 0; slot < cnt; slot++) {
            const uint32_t *sl = slots.data() + ((size_t)c * 8 + slot) * 18;
            Utf8Pre32 ul, uh;
            utf8_pre32(sl, ul);
            utf8_pre32(sl + 8, uh);
            const Utf8Carry uc = utf8_carry_from_prev_word(sl[16]);
            uint32_t tail_must;
            const uint64_t ue = utf8_errors64(ul, uh, uc, &tail_must);
            if (ue != 0 || (sl[17] != 0 && tail_must != 0)) u8_deferred_bad = true;
        }
    }
    // ---- span_reduce: one aggregate per block of 4096 summaries ----
    const int64_t BLOCK = 4096, PER_THREAD = 4;
    const int64_t nblocks = (nchunks + BLOCK - 1) / BLOCK;
    std::vector<SpanAcc> block((size_t)nblocks);
    for (int64_t b = 0; b < nblocks; b++) {
        SpanAcc acc = span_empty();
        for (int64_t c = b * BLOCK; c < nchunks && c < (b + 1) * BLOCK; c++) acc = span_concat(acc, span_of(sum[(size_t)c]));
        block[(size_t)b] = acc;
    }
    // ---- span_carries: block prefix, inclusive span per thread group, backwards walk ----
    std::vector<uint64_t> carry((size_t)nchunks);
    TilePrefix fin = {0, 0, 0, 0, 0};
    for (int64_t b = 0; b < nblocks; b++) {
        SpanAcc before = span_empty();
        for (int64_t j = 0; j < b; j++) before = span_concat(before, block[(size_t)j]);
        SpanAcc run = before;
        for (int64_t c0 = b * BLOCK; c0 < nchunks && c0 < (b + 1) * BLOCK; c0 += PER_THREAD) {
            Summary s4[4] = {{0, 0, 0}, {0, 0, 0}, {0, 0, 0}, {0, 0, 0}};
            for (int k = 0; k < PER_THREAD; k++)
                if (c0 + k < nchunks) s4[k] = sum[(size_t)(c0 + k)];
            for (int k = 0; k < PER_THREAD; k++) run = span_concat(run, span_of(s4[k]));  // inclusive span of this "thread"
            uint32_t par = run.par & 1u, cnt = run.c[0];
            if (c0 < nchunks && c0 + PER_THREAD >= nchunks) {
                fin.s_out = par;
                fin.err = (run.un[0] ? EF_UNESCAPED : 0u) | ((run.u8 || u8_deferred_bad) ? EF_UTF8 : 0u);
                fin.count = cnt;
            }
            for (int k = PER_THREAD - 1; k >= 0; k--) {
                const uint32_t s_in = (par ^ s4[k].flags) & 1u;
                cnt -= s_in ? s4[k].c1 : s4[k].c0;
                par = s_in;
                if (c0 + k < nchunks) carry[(size_t)(c0 + k)] = (uint64_t)cnt | (s_in ? (1ull << 63) : 0ull);
            }
        }
    }
    // ---- flatten: only the carry word and the chosen plane ----
    for (int64_t c = 0; c < nchunks; c++) {
        const uint64_t cw = carry[(size_t)c];
        const bool inside = (cw >> 63) != 0;
        uint64_t o = cw & ((1ull << 40) - 1);
        for (int l = 0; l < 32; l++) {
            uint64_t st = inside ? plane1[(size_t)c * 32 + l] : plane0[(size_t)c * 32 + l];
            const uint32_t v0 = (uint32_t)c * 2048u + (uint32_t)l * 64u - mis;
            while (st) {
                const int bit = __builtin_ctzll(st);
                st &= st - 1;
                if (o < cap) out[o] = v0 + (uint32_t)bit;
                o++;
            }
        }
    }
    const uint64_t n = fin.count;
    if (n_written_out) *n_written_out = n;
    if (utf8_err_out) *utf8_err_out = (fin.err & EF_UTF8) ? 1 : 0;
    if (fin.s_out) return 15;
    if (fin.err & EF_UNESCAPED) return 14;
    if (n + 3 > cap) return 1;
    if (n_out) *n_out = (uint32_t)n;
    out[n] = (uint32_t)len;
    out[n + 1] = (uint32_t)len;
    out[n + 2] = 0;
    if (n == 0) return 13;
    if ((flags & 1u) && (fin.err & EF_UTF8)) return 11;
    return 0;
}

// ---------------------------------------------------------------------------------------------------------------
// The stream pipeline with its UTF-8 deferral as the classify kernel does it (csrc/stage1_stream.cuh,
// stage1_stream_classify_kernel, and warp_compute<UTF8, 1> in csrc/stage1_kernel.cuh):
//   - per chunk, the flagged lanes (any_hi: a byte >= 0x80 in the lane or in the 4 bytes before it).  More than
//     U8_DEFER_MAX = 8: the chunk validates inline, the carry from the previous lane computed only if some lane of the
//     chunk passes the straddle gate; 1 to 8: the k-th flagged lane parks {bit planes, prev, end bit} in slot k of the
//     warp's ring.
//   - the schedule: `warps` warps in the grid; warp g first takes chunks 4g .. 4g+3, the runs after the first 4 * warps
//     chunks go to warps in the order a seeded generator picks them (any order the ticket counter can produce); a warp
//     works through its runs in the order it drew them.
//   - one 32-slot ring per warp, kept across its runs, validated when a chunk leaves more than 32 - 8 slots in use
//     (mid-run flush) and when the warp runs out of chunks (end-of-warp flush).
//   - the fold of a violation among parked lanes (stage1_persistent.cuh): utf8_error = 1, and UTF8_ERROR only if the
//     verdict is SUCCESS and flag 1 is set.
// Besides the results of emu_stage1_stream it reports the flushes (stats[0] mid-run, stats[1] end-of-warp, stats[2]
// the largest fill of a ring at a flush, stats[3] the mask of the slots any lane was parked in, stats[4] the chunks
// validated inline) and, for each document byte position probe_pos[i], how the lane holding it was validated:
// probe_out[4 i ..] = {kind (0 no byte >= 0x80 anywhere near: skipped, 1 inline, 2 parked), warp, slot, flush kind
// (1 mid-run, 2 end-of-warp)}, -1 where not applicable.
// ---------------------------------------------------------------------------------------------------------------
namespace {
constexpr int DEFER_MAX = 8, RING = 32, RUN = 4;

struct Parked {
    uint32_t pl[8], ph[8], prev, ends;
    int64_t chunk;
    int lane;
};

bool parked_lane_bad(const Parked &s) {   // validate_parked_lanes, one lane
    Utf8Pre32 ul, uh;
    utf8_pre32(s.pl, ul);
    utf8_pre32(s.ph, uh);
    const Utf8Carry uc = utf8_carry_from_prev_word(s.prev);
    uint32_t tail_must;
    const uint64_t ue = utf8_errors64(ul, uh, uc, &tail_must);
    return (ue != 0) || (s.ends != 0 && tail_must != 0);
}

bool straddle_gate(uint32_t prev) { return (prev & (prev << 1) & 0x80808000u) != 0; }   // stage1_kernel.cuh, inline path

uint64_t splitmix(uint64_t &s) {
    uint64_t z = (s += 0x9E3779B97F4A7C15ull);
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}
}  // namespace

extern "C" int32_t emu_stage1_stream_sched(const uint8_t *buf, uint64_t len, uint32_t mis, uint32_t *out, uint64_t cap, uint32_t *n_out,
                                           uint64_t *n_written_out, int32_t *utf8_err_out, int32_t *spec_out, uint32_t flags,
                                           uint32_t warps, uint64_t seed, int64_t *stats, const uint64_t *probe_pos, uint32_t nprobe,
                                           int32_t *probe_out) {
    for (int k = 0; k < 5; k++) stats[k] = 0;
    for (uint32_t i = 0; i < 4 * nprobe; i++) probe_out[i] = -1;
    if (spec_out) *spec_out = 0;
    if (len == 0 || warps == 0) return 13;
    const int64_t alen = (int64_t)mis + (int64_t)len;
    const int64_t nchunks = (alen + 2047) / 2048;
    std::vector<uint8_t> mem((size_t)(nchunks * 2048 + 64));
    for (size_t i = 0; i < mem.size(); i++) mem[i] = (i & 1) ? 0x5C : 0xF4;  // hostile bytes around the document
    memcpy(mem.data() + mis, buf, (size_t)len);
    const int64_t last = nchunks - 1;
    const int64_t last_bytes = alen - last * 2048;

    // ---- classify: everything but the parked lanes' validation, per chunk in any order ----
    std::vector<uint64_t> plane0((size_t)nchunks * 32), plane1((size_t)nchunks * 32);
    std::vector<Summary> sum((size_t)nchunks);
    std::vector<std::vector<Parked>> parks((size_t)nchunks);   // the chunk's parked lanes in slot order
    std::vector<uint8_t> kind((size_t)nchunks * 32, 0);        // per lane: 0 skipped, 1 inline, 2 parked
    std::vector<uint8_t> stage(32 + 2048);
    bool gave_up = false;
    for (int64_t c = 0; c < nchunks; c++) {
        for (size_t i = 0; i < stage.size(); i++) stage[i] = 0x5C;
        const int64_t nb = c == last ? ((last_bytes + 15) & ~15ll) : 2048;
        memcpy(stage.data() + 32, mem.data() + c * 2048, (size_t)nb);
        if (c > 0) memcpy(stage.data(), mem.data() + c * 2048 - 32, 32);
        const uint8_t *chunk = stage.data() + 32;
        const bool edge = (c == 0) || (c == last && last_bytes < 2048);
        PrevState wst = {0, 0, 0};
        if (c > 0) {
            uint32_t bsm = 0;
            for (int l = 0; l < 32; l++) bsm |= (uint32_t)(chunk[-1 - l] == 0x5C) << l;
            wst = prev_state(bsm, 32, chunk[-1]);
        }
        if (wst.unresolved) gave_up = true;
        LaneMasks m[32];
        uint32_t pl[32][8], ph[32][8], prev[32], ends[32], hi_lanes = 0, gate = 0, A = 0, O = 0;
        for (int l = 0; l < 32; l++) {
            const int64_t g0 = c * 2048 + (int64_t)l * 64;
            uint32_t words[16];
            memcpy(words, chunk + l * 64, 64);
            memcpy(&prev[l], chunk + l * 64 - 4, 4);
            ends[l] = (c == last) && ((int64_t)l * 64 + 64 == last_bytes);
            if (edge) {
                for (int k = 0; k < 16; k++) words[k] = mask_word(words[k], g0 + 4 * k, mis, alen);
                prev[l] = (g0 == 0) ? 0x20202020u : mask_word(prev[l], g0 - 4, mis, alen);
            }
            bitplanes32(words, pl[l]);
            bitplanes32(words + 8, ph[l]);
            Classes32 cl, ch;
            classify_json32(pl[l], cl);
            classify_json32(ph[l], ch);
            m[l].bs = join64(cl.bs, ch.bs);
            m[l].rq = join64(cl.rq, ch.rq);
            m[l].op = join64(cl.op, ch.op);
            m[l].ws = join64(cl.ws, ch.ws);
            m[l].ctl = join64(cl.ctl, ch.ctl);
            hi_lanes |= (uint32_t)(((pl[l][7] | ph[l][7]) != 0) || ((prev[l] & 0x80808080u) != 0)) << l;
            gate |= (uint32_t)straddle_gate(prev[l]) << l;
            A |= (uint32_t)lane_all_backslash(m[l].bs) << l;
            O |= lane_trailing_run_parity(m[l].bs) << l;
        }
        uint32_t u8err = 0;
        if (popc32(hi_lanes) <= DEFER_MAX) {
            for (int l = 0; l < 32; l++) {
                if (!((hi_lanes >> l) & 1u)) continue;
                Parked s;
                memcpy(s.pl, pl[l], sizeof s.pl);
                memcpy(s.ph, ph[l], sizeof s.ph);
                s.prev = prev[l];
                s.ends = ends[l];
                s.chunk = c;
                s.lane = l;
                parks[(size_t)c].push_back(s);
                kind[(size_t)c * 32 + l] = 2;
            }
        } else {
            stats[4]++;
            for (int l = 0; l < 32; l++) {
                kind[(size_t)c * 32 + l] = 1;
                Utf8Pre32 ul, uh;
                utf8_pre32(pl[l], ul);
                utf8_pre32(ph[l], uh);
                Utf8Carry uc = {0, 0, 0, 0};
                if (gate) uc = utf8_carry_from_prev_word(prev[l]);
                uint32_t tail_must;
                const uint64_t ue = utf8_errors64(ul, uh, uc, &tail_must);
                u8err |= (ue != 0) || (ends[l] && tail_must != 0);
            }
        }
        uint32_t PB = 0, NQ = 0;
        LaneQuotes q[32];
        for (int l = 0; l < 32; l++) {
            q[l] = lane_quotes(m[l], warp_lane_e_in(A, O, l, wst.e));
            PB |= (uint32_t)(q[l].ps >> 63) << l;
            NQ |= (uint32_t)(q[l].nqs >> 63) << l;
        }
        uint32_t fl = 0, wc0 = 0, wc1 = 0;
        for (int l = 0; l < 32; l++) {
            const uint32_t rel = (uint32_t)popc32(PB & ((1u << l) - 1u)) & 1u;
            const uint32_t p_in = l ? ((NQ >> (l - 1)) & 1u) : wst.p;
            const LaneDual d = lane_structurals_dual(m[l], q[l], rel, p_in);
            plane0[(size_t)c * 32 + l] = d.m0;
            plane1[(size_t)c * 32 + l] = d.m1;
            wc0 += (uint32_t)popc64(d.m0);
            wc1 += (uint32_t)popc64(d.m1);
            fl |= (d.u0 << 1) | (d.u1 << 2);
        }
        sum[(size_t)c] = {wc0, wc1, fl | (u8err << 3) | ((uint32_t)popc32(PB) & 1u)};
    }

    // ---- the schedule: which warp takes which run, in which order ----
    const int64_t nruns = (nchunks + RUN - 1) / RUN;
    std::vector<std::vector<int64_t>> runs_of((size_t)warps);
    for (int64_t r = 0; r < nruns && r < (int64_t)warps; r++) runs_of[(size_t)r].push_back(r);
    uint64_t rng = seed;
    for (int64_t r = warps; r < nruns; r++) runs_of[(size_t)(splitmix(rng) % warps)].push_back(r);

    // ---- each warp's ring ----
    std::vector<int32_t> slot_of((size_t)nchunks * 32, -1), warp_of((size_t)nchunks * 32, -1), flush_of((size_t)nchunks * 32, -1);
    bool u8_bad = false;
    std::vector<const Parked *> ring;
    auto flush = [&](int how) {
        stats[how == 1 ? 0 : 1]++;
        if ((int64_t)ring.size() > stats[2]) stats[2] = (int64_t)ring.size();
        for (const Parked *s : ring) {
            flush_of[(size_t)s->chunk * 32 + s->lane] = how;
            u8_bad |= parked_lane_bad(*s);
        }
        ring.clear();
    };
    for (uint32_t w = 0; w < warps; w++) {
        ring.clear();
        for (int64_t r : runs_of[w]) {
            for (int64_t c = r * RUN; c < (r + 1) * RUN && c < nchunks; c++) {
                for (const Parked &s : parks[(size_t)c]) {
                    if (ring.size() >= (size_t)RING) return -110;   // cannot happen: a flush leaves room for 8
                    slot_of[(size_t)c * 32 + s.lane] = (int32_t)ring.size();
                    warp_of[(size_t)c * 32 + s.lane] = (int32_t)w;
                    stats[3] |= 1ll << ring.size();
                    ring.push_back(&s);
                }
                if (ring.size() > (size_t)(RING - DEFER_MAX)) flush(1);
            }
        }
        if (!ring.empty()) flush(2);
    }
    for (uint32_t i = 0; i < nprobe; i++) {
        const int64_t g = (int64_t)probe_pos[i] + mis;
        if (probe_pos[i] >= len) continue;
        const size_t j = (size_t)(g / 64);
        probe_out[4 * i] = kind[j];
        if (kind[j] == 2) {
            probe_out[4 * i + 1] = warp_of[j];
            probe_out[4 * i + 2] = slot_of[j];
            probe_out[4 * i + 3] = flush_of[j];
        }
    }
    if (gave_up) {
        if (spec_out) *spec_out = 1;
        return 0;
    }

    // ---- span scan and flatten, as emu_stage1_stream (the deferred lanes are not in the summaries) ----
    const int64_t BLOCK = 4096, PER_THREAD = 4;
    const int64_t nblocks = (nchunks + BLOCK - 1) / BLOCK;
    std::vector<SpanAcc> block((size_t)nblocks);
    for (int64_t b = 0; b < nblocks; b++) {
        SpanAcc acc = span_empty();
        for (int64_t c = b * BLOCK; c < nchunks && c < (b + 1) * BLOCK; c++) acc = span_concat(acc, span_of(sum[(size_t)c]));
        block[(size_t)b] = acc;
    }
    std::vector<uint64_t> carry((size_t)nchunks);
    TilePrefix fin = {0, 0, 0, 0, 0};
    SpanAcc before = span_empty();
    for (int64_t b = 0; b < nblocks; b++) {
        SpanAcc run = before;
        for (int64_t c0 = b * BLOCK; c0 < nchunks && c0 < (b + 1) * BLOCK; c0 += PER_THREAD) {
            Summary s4[4] = {{0, 0, 0}, {0, 0, 0}, {0, 0, 0}, {0, 0, 0}};
            for (int k = 0; k < PER_THREAD; k++)
                if (c0 + k < nchunks) s4[k] = sum[(size_t)(c0 + k)];
            for (int k = 0; k < PER_THREAD; k++) run = span_concat(run, span_of(s4[k]));
            uint32_t par = run.par & 1u, cnt = run.c[0];
            if (c0 < nchunks && c0 + PER_THREAD >= nchunks) {
                fin.s_out = par;
                fin.err = (run.un[0] ? EF_UNESCAPED : 0u) | (run.u8 ? EF_UTF8 : 0u);
                fin.count = cnt;
            }
            for (int k = PER_THREAD - 1; k >= 0; k--) {
                const uint32_t s_in = (par ^ s4[k].flags) & 1u;
                cnt -= s_in ? s4[k].c1 : s4[k].c0;
                par = s_in;
                if (c0 + k < nchunks) carry[(size_t)(c0 + k)] = (uint64_t)cnt | (s_in ? (1ull << 63) : 0ull);
            }
        }
        before = span_concat(before, block[(size_t)b]);
    }
    for (int64_t c = 0; c < nchunks; c++) {
        const uint64_t cw = carry[(size_t)c];
        const bool inside = (cw >> 63) != 0;
        uint64_t o = cw & ((1ull << 40) - 1);
        for (int l = 0; l < 32; l++) {
            uint64_t st = inside ? plane1[(size_t)c * 32 + l] : plane0[(size_t)c * 32 + l];
            const uint32_t v0 = (uint32_t)c * 2048u + (uint32_t)l * 64u - mis;
            while (st) {
                const int bit = __builtin_ctzll(st);
                st &= st - 1;
                if (o < cap) out[o] = v0 + (uint32_t)bit;
                o++;
            }
        }
    }
    // ---- write_verdict (stage1_kernel.cuh) ----
    const uint64_t n = fin.count;
    int32_t err, utf8 = (fin.err & EF_UTF8) ? 1 : 0;
    if (n_written_out) *n_written_out = n;
    if (fin.s_out) err = 15;
    else if (fin.err & EF_UNESCAPED) err = 14;
    else if (n + 3 > cap) err = 1;
    else {
        if (n_out) *n_out = (uint32_t)n;
        out[n] = (uint32_t)len;
        out[n + 1] = (uint32_t)len;
        out[n + 2] = 0;
        err = n == 0 ? 13 : ((flags & 1u) && utf8) ? 11 : 0;
    }
    // ---- the fold by the persistent kernel launched behind the pipeline (stage1_persistent.cuh) ----
    if (u8_bad) {
        utf8 = 1;
        if ((flags & 1u) && err == 0) err = 11;
    }
    if (utf8_err_out) *utf8_err_out = utf8;
    return err;
}

// the straddle gate against the carry it guards: over every value of the three bytes before a lane (the fourth, the
// lowest, does not enter either), the number of values for which the gate is closed but the carry is not {0, 0, 0, 0}
extern "C" uint64_t emu_straddle_gate_misses(uint64_t *closed_out) {
    uint64_t miss = 0, closed = 0;
    for (uint32_t v = 0; v < (1u << 24); v++) {
        const uint32_t prev = (v << 8) | 0x41u;
        if (straddle_gate(prev)) continue;
        closed++;
        const Utf8Carry c = utf8_carry_from_prev_word(prev);
        miss += (c.must | c.u | c.v | c.w) != 0;
    }
    *closed_out = closed;
    return miss;
}

// ---------------------------------------------------------------------------------------------------------------
// Balanced flatten of one unit (csrc/stage1_split.cuh: stage1_flatten2_kernel) on the host: 128 mask words in stream order
// (lane t owns words 4t .. 4t+3), every lane extracts the same number q of consecutive indexes.  Same steps as the kernel:
// entries {word bit-reversed, next non-empty entry}, prefix counts, the table "share u starts in lane t" filled by the word
// owners with the division-by-multiplication, the start word from the owner's four prefix counts, drop_high_bits, q trips of
// {next entry if the word is used up; find, clear, subtract, store}.  Returns 1 if the unit is denser than the staging
// capacity (the kernel then flattens it chunk by chunk), else 0 with the unit's indexes in out[0 .. *count).
// ---------------------------------------------------------------------------------------------------------------
namespace {
uint32_t brev32(uint32_t x) {
    x = ((x >> 1) & 0x55555555u) | ((x & 0x55555555u) << 1);
    x = ((x >> 2) & 0x33333333u) | ((x & 0x33333333u) << 2);
    x = ((x >> 4) & 0x0F0F0F0Fu) | ((x & 0x0F0F0F0Fu) << 4);
    x = ((x >> 8) & 0x00FF00FFu) | ((x & 0x00FF00FFu) << 8);
    return (x >> 16) | (x << 16);
}
}  // namespace

extern "C" uint32_t emu_fl2_div(uint32_t x, uint32_t q) {
    static const uint32_t MAGIC[64] = {SJ_FL2_MAGIC_VALUES};
    return fl2_div(x, MAGIC[q]);
}
extern "C" uint32_t emu_drop_high_bits(uint32_t w, uint32_t r) { return drop_high_bits(w, r); }

extern "C" int32_t emu_flatten_unit(const uint32_t *w, uint32_t value_base, uint32_t cap_indexes, uint32_t *out, uint32_t *count) {
    static const uint32_t MAGIC[64] = {SJ_FL2_MAGIC_VALUES};
    const uint32_t SENTINEL = 128;
    uint32_t n[32], e[32], px[128], wrev[129], next[129];
    uint32_t K = 0;
    for (int t = 0; t < 32; t++) {
        e[t] = K;
        n[t] = 0;
        for (int j = 0; j < 4; j++) {
            px[4 * t + j] = K;
            K += (uint32_t)popc32(w[4 * t + j]);
        }
        n[t] = K - e[t];
    }
    *count = K;
    if (K > cap_indexes) return 1;
    if (K == 0) return 0;
    // entries: the word owners link the non-empty words (within the lane, then to the first one of the next lane that has any)
    for (int t = 0; t < 32; t++) {
        uint32_t after = SENTINEL;
        for (int s = t + 1; s < 32 && after == SENTINEL; s++)
            for (int j = 0; j < 4; j++)
                if (w[4 * s + j]) {
                    after = (uint32_t)(4 * s + j);
                    break;
                }
        uint32_t nx = after;
        for (int j = 3; j >= 0; j--) {
            wrev[4 * t + j] = brev32(w[4 * t + j]);
            next[4 * t + j] = nx;
            if (w[4 * t + j]) nx = (uint32_t)(4 * t + j);
        }
    }
    wrev[SENTINEL] = 0xFFFFFFFFu;
    next[SENTINEL] = SENTINEL;
    const uint32_t q = fl2_share(K);
    uint32_t tab[32];
    for (int u = 0; u < 32; u++) tab[u] = 0xFFFFFFFFu;
    for (int t = 0; t < 32; t++) {
        const uint32_t u_hi = fl2_div(e[t] + n[t] + q - 1u, MAGIC[q]);
        for (uint32_t u = fl2_div(e[t] + q - 1u, MAGIC[q]); u < u_hi; u++) {
            if (u >= 32 || tab[u] != 0xFFFFFFFFu) return -1;   // every share is claimed exactly once
            tab[u] = (uint32_t)t;
        }
    }
    std::vector<uint32_t> stage(32 * q, 0xFFFFFFFFu);
    for (uint32_t u = 0; u < 32; u++) {
        const uint32_t j0 = u * q;
        uint32_t cur = 0, vb = 0, nxt = SENTINEL;
        if (j0 < K) {
            const uint32_t t = tab[u];
            if (t >= 32) return -2;
            uint32_t j = 0;
            for (uint32_t i = 1; i < 4; i++)
                if (px[4 * t + i] <= j0) j = i;
            const uint32_t k = 4 * t + j;
            if (j0 - px[k] >= (uint32_t)popc32(w[k])) return -3;   // the start word holds output j0
            cur = drop_high_bits(wrev[k], j0 - px[k]);
            nxt = next[k];
            vb = value_base + 32u * k + 31u;
        }
        for (uint32_t trip = 0; trip < q; trip++) {
            if (cur == 0) {
                const uint32_t k = nxt;
                cur = wrev[k];
                nxt = next[k];
                vb = value_base + 32u * k + 31u;
            }
            const uint32_t h = 31u - (uint32_t)clz32(cur);
            cur ^= 1u << h;
            stage[j0 + trip] = vb - h;
        }
    }
    for (uint32_t i = 0; i < K; i++) out[i] = stage[i];
    return 0;
}
