// stage1_core.cuh -- per-lane / per-warp arithmetic of the B200 stage-1 structural indexer.
//
// Everything in this header is a pure function of registers, written once and compiled twice:
// by nvcc into the sm_100a kernel (stage1_kernel.cu) and by g++ into the host-side lane emulator
// used by the CPU tests (tests/emu/emulate_stage1.cpp) so that every bit trick is checked against
// the oracle without a GPU.  Nothing here touches memory.
//
// What it replaces in the reference (paths relative to /root/reference/src/mojo_simdjson/):
//   eq / pack_bits byte compares            stuff.mojo:6-9
//   classify (whitespace / op nibble tables) haswell.mojo:22-74, generic/json_character_block.mojo:22-23
//   escape scanner                           generic/stage1/json_escape_scanner.mojo:18-45
//   prefix_xor / in_string                   stuff.mojo:21-28, generic/stage1/json_string_scanner.mojo:55-69
//   structural_start / follows               generic/stage1/json_scanner.mojo:24-49,64-79
//   unescaped control characters             generic/stage1/json_structural_indexer.mojo:129-145
//   Utf8Checker (a stub in the reference)    generic/stage1/json_structural_indexer.mojo:16-30
//
// Design: one lane owns 64 consecutive input bytes (16 x u32).  The bytes are transposed into eight
// bit planes (plane k, bit i = bit k of byte i) with a 4x4 byte transpose (PRMT) followed by a
// three-stage nibble/pair/bit butterfly; every character class is then a handful of LOP3s evaluated
// for 32 bytes per instruction, and the class masks come out directly as the 64-bit words that the
// escape / in-string / structural algebra needs.  No per-byte compares, no ballots for classification.
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define SJ_HD __host__ __device__ __forceinline__
#else
#define SJ_HD inline
#endif

namespace sjb200 {

// ------------------------------------------------------------------------------------------------
// portable intrinsics
// ------------------------------------------------------------------------------------------------
SJ_HD uint32_t prmt(uint32_t a, uint32_t b, uint32_t sel) {
#if defined(__CUDA_ARCH__)
    return __byte_perm(a, b, sel);
#else
    uint64_t both = ((uint64_t)b << 32) | a;
    uint32_t r = 0;
    for (int i = 0; i < 4; i++) {
        uint32_t s = (sel >> (4 * i)) & 7;
        r |= (uint32_t)((both >> (8 * s)) & 0xFF) << (8 * i);
    }
    return r;
#endif
}
SJ_HD int popc32(uint32_t x) {
#if defined(__CUDA_ARCH__)
    return __popc(x);
#else
    return __builtin_popcount(x);
#endif
}
SJ_HD int popc64(uint64_t x) {
#if defined(__CUDA_ARCH__)
    return __popcll(x);
#else
    return __builtin_popcountll(x);
#endif
}
SJ_HD int clz32(uint32_t x) {  // clz32(0) == 32
#if defined(__CUDA_ARCH__)
    return __clz((int)x);
#else
    return x ? __builtin_clz(x) : 32;
#endif
}
SJ_HD int clz64(uint64_t x) {  // clz64(0) == 64
#if defined(__CUDA_ARCH__)
    return __clzll((long long)x);
#else
    return x ? __builtin_clzll(x) : 64;
#endif
}
SJ_HD int ffs32(uint32_t x) {  // 1-based, 0 if none
#if defined(__CUDA_ARCH__)
    return __ffs((int)x);
#else
    return x ? __builtin_ctz(x) + 1 : 0;
#endif
}

// ------------------------------------------------------------------------------------------------
// bytes -> bit planes (32 bytes = 8 words at a time)
// ------------------------------------------------------------------------------------------------
// rows a,b,c,d (4 bytes each) -> o_k = [a.k, b.k, c.k, d.k]
SJ_HD void byte_transpose4(uint32_t a, uint32_t b, uint32_t c, uint32_t d, uint32_t &o0, uint32_t &o1, uint32_t &o2,
                           uint32_t &o3) {
    uint32_t t0 = prmt(a, b, 0x5140);  // a0 b0 a1 b1
    uint32_t t1 = prmt(a, b, 0x7362);  // a2 b2 a3 b3
    uint32_t t2 = prmt(c, d, 0x5140);  // c0 d0 c1 d1
    uint32_t t3 = prmt(c, d, 0x7362);  // c2 d2 c3 d3
    o0 = prmt(t0, t2, 0x5410);
    o1 = prmt(t0, t2, 0x7632);
    o2 = prmt(t1, t3, 0x5410);
    o3 = prmt(t1, t3, 0x7632);
}

// (a & m) | (b & ~m) in ONE LOP3 (nvcc splits it in two when m is an immediate)
SJ_HD uint32_t bitselect(uint32_t a, uint32_t b, uint32_t m) {
#if defined(__CUDA_ARCH__)
    uint32_t d;
    asm("lop3.b32 %0, %1, %2, %3, 0xE4;" : "=r"(d) : "r"(a), "r"(b), "r"(m));
    return d;
#else
    return (a & m) | (b & ~m);
#endif
}
// x >> s on the FMA pipe (IMAD.HI): the ALU pipe is the one this kernel saturates (profiles/b200_pipe_throughput_ubench.txt)
SJ_HD uint32_t shr_fma(uint32_t x, int s) {
#if defined(__CUDA_ARCH__)
    return __umulhi(x, 1u << (32 - s));
#else
    return x >> s;
#endif
}

// exchange the bit-field selected by ~m in a with the field selected by m in b (delta swap across regs)
SJ_HD void field_swap(uint32_t &a, uint32_t &b, uint32_t m, int s) {
    const uint32_t na = bitselect(a, b << s, m);
    const uint32_t nb = bitselect(shr_fma(a, s), b, m);
    a = na;
    b = nb;
}

// w[0..7]: 32 consecutive bytes (little endian words).  p[k] bit i = bit k of byte i.
SJ_HD void bitplanes32(const uint32_t w[8], uint32_t p[8]) {
    // byte transpose so that register i, byte b holds input byte 8b+i
    byte_transpose4(w[0], w[2], w[4], w[6], p[0], p[1], p[2], p[3]);
    byte_transpose4(w[1], w[3], w[5], w[7], p[4], p[5], p[6], p[7]);
    // 8x8 bit transpose inside every byte lane, across the 8 registers
    field_swap(p[0], p[4], 0x0F0F0F0Fu, 4);
    field_swap(p[1], p[5], 0x0F0F0F0Fu, 4);
    field_swap(p[2], p[6], 0x0F0F0F0Fu, 4);
    field_swap(p[3], p[7], 0x0F0F0F0Fu, 4);
    field_swap(p[0], p[2], 0x33333333u, 2);
    field_swap(p[1], p[3], 0x33333333u, 2);
    field_swap(p[4], p[6], 0x33333333u, 2);
    field_swap(p[5], p[7], 0x33333333u, 2);
    field_swap(p[0], p[1], 0x55555555u, 1);
    field_swap(p[2], p[3], 0x55555555u, 1);
    field_swap(p[4], p[5], 0x55555555u, 1);
    field_swap(p[6], p[7], 0x55555555u, 1);
}

// ------------------------------------------------------------------------------------------------
// character classes on planes (32 bytes per instruction)
// ------------------------------------------------------------------------------------------------
struct Classes32 {
    uint32_t bs;   // '\\'
    uint32_t rq;   // '"' (raw, before escape resolution)
    uint32_t op;   // , : [ ] { } and the reference's 0x0C / 0x1A artefacts (haswell.mojo:44-69)
    uint32_t ws;   // 0x20 0x09 0x0A 0x0D
    uint32_t ctl;  // <= 0x1F
};
struct Utf8Pre32 {
    uint32_t hi;    // >= 0x80
    uint32_t cont;  // 10xxxxxx
    uint32_t A;     // >= 0xC0 (any lead)
    uint32_t B;     // >= 0xE0 (3/4-byte lead)
    uint32_t C;     // >= 0xF0 (4-byte lead, incl. the invalid F5..FF)
    uint32_t bad;   // C0 C1 F5..FF
    uint32_t U;     // E0 | F0: next byte must have a minimum value
    uint32_t V;     // ED | F4: next byte must have a maximum value
    uint32_t W;     // F0 | F4: selects the 4-byte variant of U / V
    uint32_t p5, p4;
};

// Any function of three words in ONE LOP3.  LUT = the function evaluated on the constants TA, TB, TC (the usual truth-table
// encoding); the host version evaluates the same table, so the emulator checks exactly what the kernel computes.
static const uint32_t TA = 0xF0u, TB = 0xCCu, TC = 0xAAu;
template <uint32_t LUT>
SJ_HD uint32_t lop3(uint32_t a, uint32_t b, uint32_t c) {
#if defined(__CUDA_ARCH__)
    uint32_t d;
    asm("lop3.b32 %0, %1, %2, %3, %4;" : "=r"(d) : "r"(a), "r"(b), "r"(c), "n"(LUT & 0xFFu));
    return d;
#else
    uint32_t r = 0;
    for (uint32_t i = 0; i < 8; i++)
        if ((LUT >> i) & 1u) r |= ((i & 4u) ? a : ~a) & ((i & 2u) ? b : ~b) & ((i & 1u) ? c : ~c);
    return r;
#endif
}

// the JSON classes of 32 bytes (reference json_character_block.mojo / haswell.mojo:44-69) as 19 three-input functions of the
// planes (a plain nibble-by-nibble formulation costs 28):
//   op  : (b | 0x20) == table[b & 15], i.e. low nibble C with high nibble 0|2, A with 1|3, B or D with 5|7 (this includes the
//         reference's 0x0C / 0x1A artefacts).  In all four low nibbles p3 = 1 and p2 != p1; then p0 = 0 pairs with p6 = 0 and
//         p2 != p4 (C: p2 = 1, p4 = 0; A: p2 = 0, p4 = 1), p0 = 1 pairs with p6 = p4 = 1.
//   ws  : 0x20 | 0x09 0x0A 0x0D: high nibble 0|2 with p4 = 0, p3 != p5, and the low three bits 000 (p5 = 1) or one of
//         001 010 101 (p5 = 0), which is (p1 != p0) and not (p2 and p1).
SJ_HD void classify_json32(const uint32_t p[8], Classes32 &c) {
    const uint32_t p0 = p[0], p1 = p[1], p2 = p[2], p3 = p[3], p4 = p[4], p5 = p[5], p6 = p[6], p7 = p[7];
    c.ctl = lop3<(~TA & ~TB & ~TC)>(p7, p6, p5);                              // 000x xxxx
    const uint32_t w2 = lop3<(~TA & ~TB & ~TC)>(p7, p6, p4);                  // high nibble 0 or 2
    // op
    const uint32_t a1 = lop3<((TA ^ TB) & TC)>(p2, p1, p3);
    const uint32_t b1 = lop3<(TA & TB & TC)>(p0, p6, p4);
    const uint32_t b2 = lop3<((TA ^ TB) & ~TC)>(p2, p4, p0);
    const uint32_t b3 = lop3<((TA & ~TB) | TC)>(b2, p6, b1);
    c.op = lop3<(TA & ~TB & TC)>(a1, p7, b3);
    // whitespace
    const uint32_t w1 = lop3<((TB ^ TC) & ~(TA & TB))>(p2, p1, p0);          // low three bits 001 010 101
    const uint32_t z = lop3<(~TA & ~TB & ~TC)>(p2, p1, p0);                   // low three bits 000
    const uint32_t y = lop3<((TA & TB) | (~TA & TC))>(p5, z, w1);
    const uint32_t t = lop3<((TA ^ TB) & TC)>(p3, p5, y);
    c.ws = w2 & t;
    // '"' = 0010 0010
    const uint32_t q1 = lop3<(~TA & TB & ~TC)>(p2, p1, p0);
    const uint32_t q2 = lop3<(TA & ~TB & TC)>(p5, p3, q1);
    c.rq = w2 & q2;
    // '\\' = 0101 1100
    const uint32_t x = lop3<(TA & TB & ~TC)>(p6, p4, p0);
    const uint32_t yb = lop3<(~TA & ~TB & ~TC)>(p7, p5, p1);
    const uint32_t l2 = lop3<(TA & TB & TC)>(p3, p2, x);
    c.bs = l2 & yb;
}
// the UTF-8 lead / continuation classes of the same 32 bytes; only needed when some byte is >= 0x80
SJ_HD void utf8_pre32(const uint32_t p[8], Utf8Pre32 &u8) {
    const uint32_t p0 = p[0], p1 = p[1], p2 = p[2], p3 = p[3], p4 = p[4], p5 = p[5], p6 = p[6], p7 = p[7];
    const uint32_t A = p7 & p6, B = A & p5, C = B & p4;
    const uint32_t L3 = B & ~p4;
    const uint32_t q = ~p3 & ~p1 & ~p0;   // low nibble 0 or 4
    const uint32_t lo0 = q & ~p2, lo4 = q & p2;
    const uint32_t loD = p3 & p2 & ~p1 & p0;
    u8.hi = p7;
    u8.cont = p7 & ~p6;
    u8.A = A;
    u8.B = B;
    u8.C = C;
    u8.bad = (A & ~p5 & ~p4 & ~p3 & ~p2 & ~p1) | (C & (p3 | (p2 & (p1 | p0))));
    u8.U = B & lo0;                    // E0, F0 (also F8..: already bad)
    u8.V = (L3 & loD) | (C & lo4);     // ED, F4
    u8.W = C & q;                      // F0, F4
    u8.p5 = p5;
    u8.p4 = p4;
}
template <bool UTF8>
SJ_HD void classify32(const uint32_t p[8], Classes32 &c, Utf8Pre32 &u8) {
    classify_json32(p, c);
    if (UTF8) utf8_pre32(p, u8);
}

SJ_HD uint64_t join64(uint32_t lo, uint32_t hi) { return ((uint64_t)hi << 32) | lo; }

// ------------------------------------------------------------------------------------------------
// UTF-8 (RFC 3629) in bit-sliced form.  Same error classes as the Keiser-Lemire lookup tables
// (TOO_SHORT / TOO_LONG / TWO_CONTS = "must be continuation" xor "is continuation"; OVERLONG_2 = C0,C1;
// OVERLONG_3 = E0 + 80..9F; SURROGATE = ED + A0..BF; OVERLONG_4 = F0 + 80..8F; TOO_LARGE = F4 + 90..BF,
// F5..FF), evaluated on the planes the classifier already has instead of three nibble lookups per byte.
// ------------------------------------------------------------------------------------------------
struct Utf8Carry {       // what the three bytes before this lane's chunk demand of its first bytes
    uint32_t must;       // bit j: byte j of the chunk must be a continuation (j = 0..2)
    uint32_t u, v, w;    // bit 0: byte -1 was E0|F0 / ED|F4 / F0|F4
};

// prev = the 4 bytes preceding the chunk, little endian (byte -1 is the top byte)
SJ_HD Utf8Carry utf8_carry_from_prev_word(uint32_t prev) {
    Utf8Carry c;
    const uint32_t x1 = prev >> 24, x2 = (prev >> 16) & 0xFF, x3 = (prev >> 8) & 0xFF;
    uint32_t k = 0;                       // number of leading bytes of the chunk that must continue
    if (x3 >= 0xF0) k = 1;
    if (x2 >= 0xE0) k = 1;
    if (x2 >= 0xF0) k = 2;
    if (x1 >= 0xC0) k = k > 1 ? k : 1;
    if (x1 >= 0xE0) k = 2;
    if (x1 >= 0xF0) k = 3;
    c.must = (1u << k) - 1u;
    c.u = (x1 == 0xE0) | (x1 == 0xF0);
    c.v = (x1 == 0xED) | (x1 == 0xF4);
    c.w = (x1 == 0xF0) | (x1 == 0xF4);
    // F5..FF / C0 C1 in the previous bytes were already reported by the lane that owns them
    return c;
}

// returns non-zero iff this chunk (given what precedes it) violates UTF-8; *tail_must = number of
// continuation bytes still owed after the last byte of the chunk (for the end-of-input check)
SJ_HD uint64_t utf8_errors64(const Utf8Pre32 &l, const Utf8Pre32 &h, const Utf8Carry &cin, uint32_t *tail_must) {
    const uint64_t A = join64(l.A, h.A), B = join64(l.B, h.B), C = join64(l.C, h.C);
    const uint64_t cont = join64(l.cont, h.cont), bad = join64(l.bad, h.bad);
    const uint64_t U = join64(l.U, h.U), V = join64(l.V, h.V), W = join64(l.W, h.W);
    const uint64_t p5 = join64(l.p5, h.p5), p4 = join64(l.p4, h.p4);
    const uint64_t must = (A << 1) | (B << 2) | (C << 3) | cin.must;
    const uint64_t Us = (U << 1) | cin.u, Vs = (V << 1) | cin.v, Ws = (W << 1) | cin.w;
    const uint64_t w4 = Ws & p4;
    const uint64_t err = (must ^ cont) | bad | (Us & ~p5 & ~w4) | (Vs & (p5 | w4));
    *tail_must = (uint32_t)((A >> 63) | (B >> 62) | (C >> 61));
    return err;
}

// ------------------------------------------------------------------------------------------------
// escapes, quotes, strings
// ------------------------------------------------------------------------------------------------
// Positions escaped by a backslash, given that the chunk's first byte is (e_in=1) or is not escaped
// by the previous chunk.  Add-carry formulation of upstream simdjson's escape scanner as used by the
// reference (json_escape_scanner.mojo:18-45): within a run of backslashes the ones at even distance
// from the run start are escapes, the bytes right after them are escaped.
SJ_HD uint64_t escaped_mask(uint64_t bs, uint64_t e_in) {
    const uint64_t ODD = 0xAAAAAAAAAAAAAAAAull;
    const uint64_t potential = bs & ~e_in;
    const uint64_t code = (((potential << 1) | ODD) - potential) ^ ODD;
    return code ^ (bs | e_in);
}

// prefix xor of a 64-bit word, done on its two halves (the left shifts of 32-bit words run on the FMA pipe as multiplications;
// a 64-bit shift would cost a funnel shift on the ALU pipe per step); the parity of the low half then flips the high half
SJ_HD uint64_t prefix_xor64(uint64_t x) {
    uint32_t lo = (uint32_t)x, hi = (uint32_t)(x >> 32);
    lo ^= lo << 1;
    hi ^= hi << 1;
    lo ^= lo << 2;
    hi ^= hi << 2;
    lo ^= lo << 4;
    hi ^= hi << 4;
    lo ^= lo << 8;
    hi ^= hi << 8;
    lo ^= lo << 16;
    hi ^= hi << 16;
#if defined(__CUDA_ARCH__)
    hi ^= (uint32_t)__mulhi((int)lo, 2);        // all ones iff bit 31 of lo is set (IMAD.HI)
#else
    hi ^= 0u - (lo >> 31);
#endif
    return ((uint64_t)hi << 32) | lo;
}

// ------------------------------------------------------------------------------------------------
// Carries.  The reference threads three 1-bit carries through its 64-byte blocks (SURVEY.md 3.2):
//   e = the first byte is escaped, p = the previous byte is a non-quote scalar, s = inside a string.
// e and p depend only on the few bytes just before a position, so every lane / warp / tile resolves
// them LOCALLY by looking at the preceding bytes (they are in shared memory anyway); only when a
// backslash run covers the whole look-behind window does it ask its predecessor.  The single carry
// that needs a global scan is s, the parity of all unescaped quotes before the position.
// ------------------------------------------------------------------------------------------------
SJ_HD uint32_t byte_is_scalar(uint32_t c) {  // !(op | whitespace), reference json_character_block.mojo:22-23
    // 128-bit membership table of the whitespace and op bytes (all < 0x80): 09 0A 0C 0D 1A | 20 2C 3A | 5B 5D | 7B 7D
    const uint32_t t0 = (1u << 0x09) | (1u << 0x0A) | (1u << 0x0C) | (1u << 0x0D) | (1u << 0x1A);
    const uint32_t t1 = (1u << 0x00) | (1u << 0x0C) | (1u << 0x1A);
    uint32_t w = (1u << 0x1B) | (1u << 0x1D);  // 0x40..0x7F: 5B 5D and 7B 7D share one pattern
    if (c < 0x40) w = t1;
    if (c < 0x20) w = t0;
    if (c >= 0x80) w = 0;
    return ((w >> (c & 31u)) & 1u) ^ 1u;
}

struct PrevState {
    uint32_t e, p;       // carries entering the position
    uint32_t unresolved; // bit0: e needs more look-behind, bit1: p needs more look-behind
};
// bsm: bit i set iff the byte at distance i+1 before the position is a backslash (i < nvalid, higher bits 0);
// c1: the byte just before the position.
SJ_HD PrevState prev_state(uint32_t bsm, int nvalid, uint32_t c1) {
    PrevState r;
    const int r1 = ffs32(~bsm) - 1;            // backslash run ending at byte -1   (32 if bsm is all ones)
    const int r2 = ffs32(~(bsm >> 1)) - 1;     // backslash run ending at byte -2
    r.e = (uint32_t)r1 & 1u;
    r.unresolved = (r1 < 0 || r1 >= nvalid) ? 1u : 0u;
    if (c1 == 0x22) {
        r.p = (uint32_t)r2 & 1u;               // an escaped quote is an ordinary scalar character
        if (r2 < 0 || r2 >= nvalid - 1) r.unresolved |= 2u;
    } else {
        r.p = byte_is_scalar(c1);
    }
    return r;
}

// Slow path: walk back over a long backslash run.  before[-1] is the last byte of the run, at most `limit`
// bytes may be read.  Returns the run length (== limit if it covers everything readable).
SJ_HD uint32_t backslash_run_before(const uint8_t *before, uint32_t limit) {
    uint32_t r = 0;
    while (r < limit && before[-(int)(r + 1)] == 0x5C) r++;
    return r;
}
// escapedness of the byte following a run of `run` backslashes whose first backslash has escapedness e0
SJ_HD uint32_t escaped_after_run(uint32_t run, uint32_t e0) { return (run & 1u) ^ e0; }

// ------------------------------------------------------------------------------------------------
// In-warp escape resolution from two ballots
//   A = ballot(lane is all backslashes), O = ballot(parity of the lane's trailing backslash run)
// ------------------------------------------------------------------------------------------------
SJ_HD bool lane_all_backslash(uint64_t bs) { return bs == ~0ull; }
SJ_HD uint32_t lane_trailing_run_parity(uint64_t bs) { return (uint32_t)clz64(~bs) & 1u; }

// e_in of `lane` (0..32; 32 = the carry leaving the warp) given the warp's own e_in.
// A lane made only of backslashes passes its e_in through (64 is even).
SJ_HD uint32_t warp_lane_e_in(uint32_t A, uint32_t O, int lane, uint32_t e_warp) {
    const uint32_t below = ~A & (lane >= 32 ? 0xFFFFFFFFu : ((1u << lane) - 1u));
    if (below == 0) return e_warp & 1u;
    const int j = 31 - clz32(below);
    return (O >> j) & 1u;
}

// ------------------------------------------------------------------------------------------------
// Lane results.  Everything is exact relative to the start of the warp except the in-string parity:
// the structural mask is produced for both values of "the warp starts inside a string".
// ------------------------------------------------------------------------------------------------
struct LaneMasks {
    uint64_t bs, rq, op, ws, ctl;
};
struct LaneQuotes {
    uint64_t quote;  // unescaped quotes
    uint64_t ps;     // prefix xor of quote: in_string relative to the chunk start
    uint64_t nqs;    // non-quote scalar
};
SJ_HD LaneQuotes lane_quotes(const LaneMasks &m, uint32_t e_in) {
    LaneQuotes q;
    const uint64_t esc = escaped_mask(m.bs, (uint64_t)(e_in & 1));
    q.quote = m.rq & ~esc;
    q.ps = prefix_xor64(q.quote);
    q.nqs = ~(m.op | m.ws) & ~q.quote;
    return q;
}
struct LaneDual {
    uint64_t m0, m1;      // structural bits if the warp starts outside / inside a string
    uint32_t u0, u1;      // unescaped control character inside a string, same two cases
};
// rel = parity of the unescaped quotes of the earlier lanes of the warp; p_in = previous byte is a non-quote scalar
SJ_HD LaneDual lane_structurals_dual(const LaneMasks &m, const LaneQuotes &q, uint32_t rel, uint32_t p_in) {
    const uint64_t in0 = q.ps ^ (0 - (uint64_t)(rel & 1));   // in_string if the warp starts outside a string
    const uint64_t scalar = ~(m.op | m.ws);
    const uint64_t follows = (q.nqs << 1) | (p_in & 1);
    const uint64_t pot = m.op | (scalar & ~follows);         // json_scanner.mojo:24-49
    const uint64_t tail0 = in0 ^ q.quote;                     // string_tail, json_string_scanner.mojo:41-44
    LaneDual d;
    d.m0 = pot & ~tail0;
    d.m1 = pot & tail0;                                       // in_string complemented => string_tail complemented
    d.u0 = (m.ctl & in0) != 0;
    d.u1 = (m.ctl & ~in0) != 0;
    return d;
}

// ------------------------------------------------------------------------------------------------
// Arithmetic of the balanced flatten kernel (stage1_split.cuh: stage1_flatten2_kernel), shared with the host emulator.
// ------------------------------------------------------------------------------------------------
// floor(x / q) = (x * FL2_MAGIC_VALUES[q]) >> 20 for 0 < q < 64 and x <= 34 q, x < 4200 (32-bit product; the kernel divides
// prefix counts of a unit of at most 32 q indexes; tests/test_core_emulation.py checks every pair)
#define SJ_FL2_MAGIC_VALUES 0, 1048577, 524289, 349526, 262145, 209716, 174763, 149797, 131073, 116509, 104858, 95326, 87382, 80660, 74899, 69906, 65537, 61681, 58255, 55189, 52429, 49933, 47663, 45591, 43691, 41944, 40330, 38837, 37450, 36158, 34953, 33826, 32769, 31776, 30841, 29960, 29128, 28340, 27595, 26887, 26215, 25576, 24967, 24386, 23832, 23302, 22796, 22311, 21846, 21400, 20972, 20561, 20165, 19785, 19419, 19066, 18725, 18397, 18079, 17773, 17477, 17190, 16913, 16645
SJ_HD uint32_t fl2_div(uint32_t x, uint32_t magic) { return (x * magic) >> 20; }
// every lane's share of a unit of K indexes: q consecutive outputs, q odd (the staging stores of the 32 lanes, stride q, then
// never share a bank)
SJ_HD uint32_t fl2_share(uint32_t K) { return ((K + 31u) >> 5) | 1u; }
// w (bit-reversed mask word) without its r highest set bits, r < popc(w): a binary descent to the largest `pos` whose top
// `pos` bits hold exactly r set bits
SJ_HD uint32_t drop_high_bits(uint32_t w, uint32_t r) {
    uint32_t ws = w, pos = 0;   // ws = w << pos
    for (int s = 16; s; s >>= 1) {
        const uint32_t c = (uint32_t)popc32(ws >> (32 - s));   // set bits among the next s bits from the top
        if (c <= r) {
            r -= c;
            ws <<= s;
            pos += s;
        }
    }
    return w & (0xFFFFFFFFu >> pos);
}

// ------------------------------------------------------------------------------------------------
// Tile descriptors for the single-pass look-back (one 64-bit word per tile, generation tagged).
//   AGG    : what the tile contributes, for both values of "the tile starts inside a string"
//   PREFIX : the state after the tile and the number of indexes produced up to and including it
// ------------------------------------------------------------------------------------------------
static const uint32_t DESC_AGG = 1, DESC_PREFIX = 2;
static const uint32_t EF_UNESCAPED = 1, EF_UTF8 = 2;
static const uint32_t GEN_MASK = 0xFFFFFu;  // 20-bit generation

struct TileAgg {
    uint32_t par;        // parity of the tile's unescaped quotes
    uint32_t e_out, p_out;
    uint32_t un[2];      // unescaped control character inside a string, if the tile starts outside / inside a string
    uint32_t u8;         // UTF-8 violation
    uint32_t c[2];       // structural count, same two cases (<= 2^17)
};
struct TilePrefix {
    uint32_t s_out, e_out, p_out;
    uint32_t err;        // EF_* accumulated over all tiles so far
    uint32_t count;      // indexes produced so far
};
SJ_HD uint64_t desc_pack_agg(uint32_t gen, const TileAgg &a) {
    const uint64_t hi = ((uint64_t)(gen & GEN_MASK) << 8) | (DESC_AGG << 6) | ((a.par & 1) << 5) | ((a.e_out & 1) << 4) |
                        ((a.p_out & 1) << 3) | ((a.un[0] & 1) << 2) | ((a.un[1] & 1) << 1) | (a.u8 & 1);
    return (hi << 36) | ((uint64_t)(a.c[1] & 0x3FFFFu) << 18) | (uint64_t)(a.c[0] & 0x3FFFFu);
}
SJ_HD uint64_t desc_pack_prefix(uint32_t gen, const TilePrefix &p) {
    const uint64_t hi = ((uint64_t)(gen & GEN_MASK) << 8) | (DESC_PREFIX << 6) | ((p.s_out & 1) << 5) | ((p.e_out & 1) << 4) |
                        ((p.p_out & 1) << 3) | ((p.err & 3) << 1);
    return (hi << 36) | (uint64_t)p.count;  // bits [35:32] unused
}
SJ_HD uint32_t desc_gen(uint64_t d) { return (uint32_t)(d >> 44) & GEN_MASK; }
SJ_HD uint32_t desc_status(uint64_t d) { return (uint32_t)(d >> 42) & 3u; }
SJ_HD TileAgg desc_unpack_agg(uint64_t d) {
    TileAgg a;
    const uint32_t f = (uint32_t)(d >> 36);
    a.par = (f >> 5) & 1;
    a.e_out = (f >> 4) & 1;
    a.p_out = (f >> 3) & 1;
    a.un[0] = (f >> 2) & 1;
    a.un[1] = (f >> 1) & 1;
    a.u8 = f & 1;
    a.c[0] = (uint32_t)d & 0x3FFFFu;
    a.c[1] = (uint32_t)(d >> 18) & 0x3FFFFu;
    return a;
}
SJ_HD TilePrefix desc_unpack_prefix(uint64_t d) {
    TilePrefix p;
    const uint32_t f = (uint32_t)(d >> 36);
    p.s_out = (f >> 5) & 1;
    p.e_out = (f >> 4) & 1;
    p.p_out = (f >> 3) & 1;
    p.err = (f >> 1) & 3;
    p.count = (uint32_t)d;  // low 32 bits; the 4 bits [35:32] are unused
    return p;
}

// A run of tiles seen as a function of "starts inside a string" (s): parity, counts and error flags.
struct SpanAcc {
    uint32_t par, c[2], un[2], u8;
};
SJ_HD SpanAcc span_empty() {
    SpanAcc a = {0, {0, 0}, {0, 0}, 0};
    return a;
}
// older happens first, then newer
SJ_HD SpanAcc span_concat(const SpanAcc &older, const SpanAcc &newer) {
    SpanAcc r;
    r.par = older.par ^ newer.par;
    const bool flip = (older.par & 1u) != 0;  // no dynamic indexing: these live in registers
    r.c[0] = older.c[0] + (flip ? newer.c[1] : newer.c[0]);
    r.c[1] = older.c[1] + (flip ? newer.c[0] : newer.c[1]);
    r.un[0] = older.un[0] | (flip ? newer.un[1] : newer.un[0]);
    r.un[1] = older.un[1] | (flip ? newer.un[0] : newer.un[1]);
    r.u8 = older.u8 | newer.u8;
    return r;
}

}  // namespace sjb200
