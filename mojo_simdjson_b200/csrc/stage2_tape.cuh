// stage2_tape.cuh -- SURVEY.md section 8(f) rank 4, first slice: the reference's stage-2 WALK (grammar verdict + tape) as
// data-parallel kernels over the structural index array.  Included at the end of capi.cu, after stage2_primitives.cuh.
//
// The reference walks the structurals with a state machine (JsonIterator.walk_document, generic/stage2/json_iterator.mojo:40-254)
// that keeps a stack of open containers (dom_parser_implementation.mojo:12-16, is_array / open_containers) and appends tape
// words as it goes (tape_builder.mojo, tape_writer.mojo:33-47).  Nothing in that walk needs to be sequential:
//
//   what the walk knows at token k          how it is obtained here
//   --------------------------------------  -----------------------------------------------------------------------------
//   depth, and whether the innermost open   ONE ordered scan with the "bounded bit stack" monoid: an element says "pop p, then
//   container is an array or an object      push these l bits"; composition is associative, the stack is 128 bits because the
//                                           reference refuses depth > 100 (DEPTH_ERROR) long before it could overflow
//   the state (object_begin / _field /      a function of the previous one or two token types and that container type: every
//   _continue, array_value / _continue ..)  transition of the state machine is a LOCAL rule once the container type is known
//   the error it returns                    the first token (lowest index) whose local rule fails, atomicMin over (index, check, code);
//                                           per token: position errors (TAPE_ERROR) before DEPTH_ERROR before the primitive's own
//                                           error (stage2_primitives.cuh) before CAPACITY (count > 0xFFFFFF), the walk's order
//   where a tape word goes                  exclusive prefix sum of the words each token appends (0, 1 or 2)
//   the matching bracket, element counts    stable multisplit of brackets and commas by depth: in the list of one depth an
//                                           open is followed by its direct commas and then by its close
//
// The verdict is the reference's, restated in oracle/stage2_oracle.c (oracle_stage2_walk), oddities included: a root-level
// empty container is never consumed (TAPE_ERROR), arrays hit DEPTH_ERROR one level before objects.  The tape is the format the
// reference's comments describe (upstream simdjson's) -- its own tape_builder is unfinished (no END words, byte offsets used
// as element indexes, doubles stored with a numeric cast; see the oracle's header) -- so tape parity is UNPINNED and checked
// against the oracle and, independently, against python's json.  Doubles: exact (Clinger's fast path: <= 19 significant
// digits that fit 2^53, |decimal exponent| <= 22) or flagged inexact in the summary; nothing else is approximated.
#pragma once

namespace {

enum : uint8_t { TK_LBRACE = 0, TK_RBRACE, TK_LBRACK, TK_RBRACK, TK_COLON, TK_COMMA, TK_STR, TK_VAL, TK_BAD, TK_NONE };
enum : uint8_t { S2E_DEPTH = 4, S2E_CAPACITY = 1 };
constexpr uint32_t S2_MAX_DEPTH = 100;   // dom_parser_implementation.mojo:40

__device__ __forceinline__ uint8_t s2_token(uint32_t c) {
    switch (c) {
    case '{': return TK_LBRACE;
    case '}': return TK_RBRACE;
    case '[': return TK_LBRACK;
    case ']': return TK_RBRACK;
    case ':': return TK_COLON;
    case ',': return TK_COMMA;
    case '"': return TK_STR;
    case '-': case 't': case 'f': case 'n': return TK_VAL;
    default: return (c - '0' <= 9u) ? TK_VAL : TK_BAD;
    }
}
__device__ __forceinline__ bool tk_open(uint8_t t) { return t == TK_LBRACE || t == TK_LBRACK; }
__device__ __forceinline__ bool tk_close(uint8_t t) { return t == TK_RBRACE || t == TK_RBRACK; }
__device__ __forceinline__ bool tk_value_start(uint8_t t) { return t == TK_LBRACE || t == TK_LBRACK || t == TK_STR || t == TK_VAL; }

// ---- the bounded bit stack monoid: "pop `pop` entries, then push `len` entries" (bit 0 of lo = the last one pushed; 1 = array)
struct Stk {
    uint32_t pop, len;
    uint64_t lo, hi;
};
__device__ __forceinline__ Stk stk_identity() { return Stk{0u, 0u, 0ull, 0ull}; }
__device__ __forceinline__ Stk stk_of(uint8_t t) {
    if (t == TK_LBRACE) return Stk{0u, 1u, 0ull, 0ull};
    if (t == TK_LBRACK) return Stk{0u, 1u, 1ull, 0ull};
    if (tk_close(t)) return Stk{1u, 0u, 0ull, 0ull};
    return stk_identity();
}
__device__ __forceinline__ void shr128(uint64_t &lo, uint64_t &hi, uint32_t s) {
    if (s >= 128u) { lo = hi = 0; }
    else if (s >= 64u) { lo = hi >> (s - 64u); hi = 0; }
    else if (s) { lo = (lo >> s) | (hi << (64u - s)); hi >>= s; }
}
__device__ __forceinline__ void shl128(uint64_t &lo, uint64_t &hi, uint32_t s) {
    if (s >= 128u) { lo = hi = 0; }
    else if (s >= 64u) { hi = lo << (s - 64u); lo = 0; }
    else if (s) { hi = (hi << s) | (lo >> (64u - s)); lo <<= s; }
}
// a happens first, then b
__device__ __forceinline__ Stk stk_concat(const Stk &a, const Stk &b) {
    Stk r;
    if (b.pop <= a.len) {
        uint64_t lo = a.lo, hi = a.hi;
        shr128(lo, hi, b.pop);
        shl128(lo, hi, b.len);
        r.pop = a.pop;
        r.len = a.len - b.pop + b.len;
        r.lo = lo | b.lo;
        r.hi = hi | b.hi;
    } else {
        r.pop = a.pop + (b.pop - a.len);
        r.len = b.len;
        r.lo = b.lo;
        r.hi = b.hi;
    }
    return r;
}
// Document streams: a document starts at every token of global bracket depth 0, and its walk must not see the stack of the
// document before it (after a stray close that stack never empties again).  The scans then run over (flag, Stk) with
// (fa, a) + (fb, b) = (fa | fb, fb ? b : a then b); the flag rides in the top bit of `pop`, which never reaches 2^30 (n < 2^30),
// and stk_concat carries a's flag through unchanged when b has none.
constexpr uint32_t STK_DOC_START = 0x80000000u;
template <bool SEG>
__device__ __forceinline__ Stk stk_combine(const Stk &a, const Stk &b) {
    if (SEG && (b.pop & STK_DOC_START)) return b;
    return stk_concat(a, b);
}
__device__ __forceinline__ Stk stk_shfl_up(const Stk &a, int d) {
    Stk r;
    r.pop = __shfl_up_sync(0xFFFFFFFFu, a.pop, d);
    r.len = __shfl_up_sync(0xFFFFFFFFu, a.len, d);
    r.lo = __shfl_up_sync(0xFFFFFFFFu, a.lo, d);
    r.hi = __shfl_up_sync(0xFFFFFFFFu, a.hi, d);
    return r;
}
template <bool SEG>
__device__ __forceinline__ Stk stk_warp_inclusive(Stk a, int lane) {
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const Stk o = stk_shfl_up(a, d);
        if (lane >= d) a = stk_combine<SEG>(o, a);
    }
    return a;
}

constexpr int TAPE_THREADS = 256, TAPE_PER_THREAD = 8, TAPE_BLOCK = TAPE_THREADS * TAPE_PER_THREAD;

// inclusive scan over the CTA's 256 threads; returns this thread's EXCLUSIVE prefix inside the CTA, `total` = the CTA's
template <bool SEG>
__device__ __forceinline__ Stk stk_block_exclusive(const Stk mine, Stk *s_w /* [8] */, Stk &total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const Stk incl = stk_warp_inclusive<SEG>(mine, lane);
    if (lane == 31) s_w[warp] = incl;
    __syncthreads();
    Stk before = stk_identity(), all = stk_identity();
    for (int q = 0; q < TAPE_THREADS / 32; q++) {
        if (q < warp) before = stk_combine<SEG>(before, s_w[q]);
        all = stk_combine<SEG>(all, s_w[q]);
    }
    total = all;
    __syncthreads();
    Stk prev = stk_shfl_up(incl, 1);            // the warp-inclusive value of the lane before = this lane's exclusive in-warp prefix
    if (lane == 0) prev = stk_identity();
    return stk_combine<SEG>(before, prev);
}

__device__ __forceinline__ uint8_t token_at(const uint8_t *buf, uint64_t len, const uint32_t *idx, uint64_t n, int64_t k) {
    if (k < 0 || (uint64_t)k >= n) return TK_NONE;
    const uint64_t i = idx[k];
    return s2_token(i < len ? (uint32_t)__ldg(buf + i) : 0x20u);
}

// the element of token k: stk_of(token), flagged where a document starts (stream mode only)
template <bool STREAM>
__device__ __forceinline__ Stk stk_elem(uint8_t t, const uint8_t *starts, uint64_t k) {
    Stk e = stk_of(t);
    if (STREAM && starts[k]) e.pop |= STK_DOC_START;
    return e;
}

template <bool STREAM>
__global__ void __launch_bounds__(TAPE_THREADS) tape_stack_totals_kernel(const uint8_t *__restrict__ buf, uint64_t len, const uint32_t *__restrict__ idx, uint64_t n,
                                                                         Stk *__restrict__ block_total, const uint8_t *__restrict__ starts) {
    __shared__ Stk s_w[TAPE_THREADS / 32];
    const uint64_t k0 = (uint64_t)blockIdx.x * TAPE_BLOCK + (uint64_t)threadIdx.x * TAPE_PER_THREAD;
    Stk mine = stk_identity();
#pragma unroll
    for (int j = 0; j < TAPE_PER_THREAD; j++)
        if (k0 + j < n) mine = stk_combine<STREAM>(mine, stk_elem<STREAM>(token_at(buf, len, idx, n, (int64_t)(k0 + j)), starts, k0 + j));
    Stk total;
    stk_block_exclusive<STREAM>(mine, s_w, total);
    if (threadIdx.x == 0) block_total[blockIdx.x] = total;
}
// one CTA: block_total[b] <- the stack operations of everything before block b (exclusive scan, in place)
template <bool STREAM>
__global__ void __launch_bounds__(1024) tape_stack_scan_kernel(Stk *block_total, uint32_t nblocks) {
    __shared__ Stk s_w[32];
    __shared__ Stk s_carry;
    if (threadIdx.x == 0) s_carry = stk_identity();
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (uint32_t b0 = 0; b0 < nblocks; b0 += 1024u) {
        const uint32_t b = b0 + threadIdx.x;
        const Stk v = b < nblocks ? block_total[b] : stk_identity();
        const Stk incl = stk_warp_inclusive<STREAM>(v, lane);
        if (lane == 31) s_w[warp] = incl;
        __syncthreads();
        Stk before = s_carry;
        for (int q = 0; q < warp; q++) before = stk_combine<STREAM>(before, s_w[q]);
        Stk prev = stk_shfl_up(incl, 1);
        if (lane == 0) prev = stk_identity();
        const Stk excl = stk_combine<STREAM>(before, prev);
        if (b < nblocks) block_total[b] = excl;
        __syncthreads();
        if (threadIdx.x == 1023) s_carry = stk_combine<STREAM>(excl, v);
        __syncthreads();
    }
}

// Stream mode (document streams): where documents start, the document of every token, the first token of every document
// (doc_first[d], d <= n_docs, doc_first[n_docs] = n), where every document's tape slice starts, and one status word per document
struct StreamArgs {
    const uint8_t *starts;
    const uint32_t *doc_of;
    const uint32_t *doc_first;
    const uint64_t *doc_tape;
    unsigned long long *doc_status;
};

// per-token outputs of the grammar pass
//   words[k]  tape words the token appends (0, 1, 2)
//   cls[k]    multisplit class: 0 = none; else 1 + min(depth, 126), bit 7 set for commas (brackets: depth of the container's inside)
// STREAM: every rule that reads the document's first token, second token, last token or length reads those of the token's own
// document, the stack restarts empty at every document start, and errors go to the document's status word with the index
// relative to its first token.
template <bool STREAM>
__global__ void __launch_bounds__(TAPE_THREADS) tape_grammar_kernel(const uint8_t *__restrict__ buf, uint64_t len, const uint32_t *__restrict__ idx, uint64_t n,
                                                                    const uint8_t *__restrict__ prim_kind, const uint8_t *__restrict__ prim_err,
                                                                    const Stk *__restrict__ block_before, uint32_t *__restrict__ words, uint8_t *__restrict__ cls,
                                                                    unsigned long long *__restrict__ first_err, const StreamArgs sa) {
    __shared__ Stk s_w[TAPE_THREADS / 32];
    const uint64_t k0 = (uint64_t)blockIdx.x * TAPE_BLOCK + (uint64_t)threadIdx.x * TAPE_PER_THREAD;
    uint8_t tok[TAPE_PER_THREAD];
    Stk mine = stk_identity();
#pragma unroll
    for (int j = 0; j < TAPE_PER_THREAD; j++) {
        tok[j] = token_at(buf, len, idx, n, (int64_t)(k0 + j));
        if (k0 + j < n) mine = stk_combine<STREAM>(mine, stk_elem<STREAM>(tok[j], sa.starts, k0 + j));
    }
    Stk total;
    Stk st = stk_combine<STREAM>(block_before[blockIdx.x], stk_block_exclusive<STREAM>(mine, s_w, total));   // the stack before this thread's first token
    if (STREAM) st.pop &= ~STK_DOC_START;
    uint8_t p1 = token_at(buf, len, idx, n, (int64_t)k0 - 1), p2 = token_at(buf, len, idx, n, (int64_t)k0 - 2);
    unsigned long long worst = ~0ull;
    const uint8_t first_tok = token_at(buf, len, idx, n, 0), last_tok = token_at(buf, len, idx, n, (int64_t)n - 1);
#pragma unroll
    for (int j = 0; j < TAPE_PER_THREAD; j++) {
        const uint64_t k = k0 + j;
        if (k >= n) break;
        const uint8_t t = tok[j];
        const uint8_t nxt = (j + 1 < TAPE_PER_THREAD) ? tok[j + 1] : token_at(buf, len, idx, n, (int64_t)k + 1);
        // the token's index in its document, the document's length, first and last token
        uint64_t kl = k, nl = n;
        uint8_t ft = first_tok, lt = last_tok;
        uint32_t doc = 0;
        if (STREAM) {
            if (sa.starts[k]) st = stk_identity();
            doc = sa.doc_of[k];
            const uint32_t f = sa.doc_first[doc];
            kl = k - f;
            nl = (uint64_t)sa.doc_first[doc + 1] - f;
            ft = kl == 1 ? p1 : TK_NONE;                                                  // only read at the second token
            lt = kl == 0 ? token_at(buf, len, idx, n, (int64_t)(f + nl - 1)) : TK_NONE;   // only read at the first
        }
        const bool underflow = st.pop != 0;
        const uint32_t depth = st.len;
        const int ctx = depth == 0 ? 0 : ((st.lo & 1ull) ? 2 : 1);   // 0 root, 1 object, 2 array
        uint8_t e = 0, prio = 0;   // at one token the walk checks the position first, then the depth, then the primitive, then the count
        // ---- is this token allowed here?  (the walk's position checks: TAPE_ERROR)
        bool ok;
        if (underflow) {
            ok = false;
        } else if (ctx == 0) {
            ok = (kl == 0) && tk_value_start(t);                      // document_start: one value; anything after it is trailing content
            if (kl == 0 && ok) {
                if (t == TK_LBRACE && lt != TK_RBRACE) ok = false;         // json_iterator.mojo:54-59
                if (t == TK_LBRACK && lt != TK_RBRACK) ok = false;
            }
        } else if (ctx == 2) {
            if (p1 == TK_LBRACK) ok = t == TK_RBRACK || tk_value_start(t);                 // array_begin / empty array
            else if (p1 == TK_COMMA) ok = tk_value_start(t);                                  // array_value
            else ok = t == TK_COMMA || t == TK_RBRACK;                                        // array_continue (p1 ends a value)
        } else {
            const bool p1_is_key = p1 == TK_STR && (p2 == TK_LBRACE || p2 == TK_COMMA);
            if (p1 == TK_LBRACE) ok = t == TK_RBRACE || t == TK_STR;                          // object_begin / empty object
            else if (p1 == TK_COMMA) ok = t == TK_STR;                                        // the next key
            else if (p1_is_key) ok = t == TK_COLON;                                           // object_field
            else if (p1 == TK_COLON) ok = tk_value_start(t);
            else ok = t == TK_COMMA || t == TK_RBRACE;                                        // object_continue
        }
        if (!ok) e = S2E_TAPE;
        // a root-level empty container is never consumed by the walk (json_iterator.mojo:61-65, 72-76): the index check at the end fails
        if (!e && kl == 1 && depth == 1 && tk_close(t) && nl >= 2 && ((ft == TK_LBRACE && t == TK_RBRACE) || (ft == TK_LBRACK && t == TK_RBRACK))) e = S2E_TAPE;
        // ---- depth (object_begin / array_begin, not for empty containers)
        if (!e && tk_open(t)) {
            const bool empty = (t == TK_LBRACE && nxt == TK_RBRACE) || (t == TK_LBRACK && nxt == TK_RBRACK);
            if (!empty) {
                const uint32_t nd = depth + 1;
                if (t == TK_LBRACE ? nd > S2_MAX_DEPTH : nd >= S2_MAX_DEPTH) {
                    e = S2E_DEPTH;
                    prio = 1;
                }
            }
        }
        // ---- the primitive itself
        if (!e && (t == TK_STR || t == TK_VAL || t == TK_BAD)) {
            e = prim_err[k];
            prio = 2;
        }
        if (e) {
            const unsigned long long cand = ((unsigned long long)kl << 16) | ((unsigned long long)prio << 8) | e;
            if (STREAM) atomicMin(sa.doc_status + doc, cand);   // a thread's tokens may belong to several documents
            else worst = cand < worst ? cand : worst;
        }
        // ---- what the token appends, and its multisplit class
        uint32_t w = 0;
        uint8_t c = 0;
        if (t == TK_STR || tk_open(t) || tk_close(t)) w = 1;
        else if (t == TK_VAL) w = (prim_kind[k] == S2_INT || prim_kind[k] == S2_FLOAT) ? 2 : 1;
        if (tk_open(t)) c = (uint8_t)(1u + (depth + 1u < 126u ? depth + 1u : 126u));
        else if (tk_close(t)) c = (uint8_t)(1u + (depth < 126u ? depth : 126u));
        else if (t == TK_COMMA) c = (uint8_t)(0x80u | (1u + (depth < 126u ? depth : 126u)));
        words[k] = w;
        cls[k] = c;
        st = stk_concat(st, stk_of(t));
        p2 = p1;
        p1 = t;
        // the walk of a document runs off its end with containers still open: TAPE_ERROR at the document's length
        if (STREAM && kl + 1 == nl && st.pop == 0 && st.len != 0) atomicMin(sa.doc_status + doc, ((unsigned long long)nl << 16) | S2E_TAPE);
    }
    // the walk runs off the end with containers still open: the state that reads the trailer fails (TAPE_ERROR at index n)
    if (!STREAM && k0 <= n - 1 && n - 1 < k0 + TAPE_PER_THREAD && st.pop == 0 && st.len != 0) {
        const unsigned long long cand = ((unsigned long long)n << 16) | S2E_TAPE;
        worst = cand < worst ? cand : worst;
    }
    if (worst != ~0ull) atomicMin(first_err, worst);
}

// ---- stable multisplit by class: rank of every bracket among the brackets of its class (B), and among brackets + commas (A)
constexpr int MS_TILE = 2048, MS_CLASSES = 128;
// hist layout: [class][tile] for B, then the same for A
__global__ void __launch_bounds__(32) tape_multisplit_hist_kernel(const uint8_t *__restrict__ cls, uint64_t n, uint32_t ntiles, uint32_t *__restrict__ hist) {
    __shared__ uint32_t cb[MS_CLASSES], ca[MS_CLASSES];
    const int lane = threadIdx.x;
    for (int c = lane; c < MS_CLASSES; c += 32) cb[c] = ca[c] = 0;
    __syncwarp();
    const uint64_t t0 = (uint64_t)blockIdx.x * MS_TILE;
    for (int s = 0; s < MS_TILE / 32; s++) {
        const uint64_t k = t0 + (uint64_t)s * 32 + lane;
        const uint8_t c = k < n ? cls[k] : 0;
        if (c) {
            atomicAdd(&ca[c & 0x7F], 1u);
            if (!(c & 0x80)) atomicAdd(&cb[c & 0x7F], 1u);
        }
    }
    __syncwarp();
    for (int c = lane; c < MS_CLASSES; c += 32) {
        hist[(size_t)c * ntiles + blockIdx.x] = cb[c];
        hist[(size_t)(MS_CLASSES + c) * ntiles + blockIdx.x] = ca[c];
    }
}
// after the exclusive scan of hist (B part and A part scanned as one array each): global ranks, and the sorted bracket list
__global__ void __launch_bounds__(32) tape_multisplit_rank_kernel(const uint8_t *__restrict__ cls, uint64_t n, uint32_t ntiles, const uint32_t *__restrict__ hist,
                                                                  uint32_t a_base, uint32_t *__restrict__ slot_b, uint32_t *__restrict__ rank_a,
                                                                  uint32_t *__restrict__ sorted_b) {
    __shared__ uint32_t cb[MS_CLASSES], ca[MS_CLASSES];
    const int lane = threadIdx.x;
    for (int c = lane; c < MS_CLASSES; c += 32) {
        cb[c] = hist[(size_t)c * ntiles + blockIdx.x];
        ca[c] = hist[(size_t)(MS_CLASSES + c) * ntiles + blockIdx.x] - a_base;
    }
    __syncwarp();
    const uint64_t t0 = (uint64_t)blockIdx.x * MS_TILE;
    const uint32_t lt = (1u << lane) - 1u;
    for (int s = 0; s < MS_TILE / 32; s++) {
        const uint64_t k = t0 + (uint64_t)s * 32 + lane;
        const uint8_t c = k < n ? cls[k] : 0;
        const uint32_t key = c ? (uint32_t)(c & 0x7F) : 0xFFFFu;
        const uint32_t peers_a = __match_any_sync(0xFFFFFFFFu, key);
        const uint32_t is_b = __ballot_sync(0xFFFFFFFFu, c && !(c & 0x80));
        const uint32_t peers_b = peers_a & is_b;
        uint32_t ra = 0, rb = 0;
        if (c) {
            ra = ca[key] + (uint32_t)__popc(peers_a & lt);
            rb = cb[key] + (uint32_t)__popc(peers_b & lt);
        }
        __syncwarp();
        if (c && (peers_a & lt) == 0) {   // the first lane of every class group advances the counters
            ca[key] += (uint32_t)__popc(peers_a);
            cb[key] += (uint32_t)__popc(peers_b);
        }
        __syncwarp();
        if (c && !(c & 0x80)) {
            slot_b[k] = rb;
            rank_a[k] = ra;
            sorted_b[rb] = (uint32_t)k;
        }
    }
}

// decimal token -> IEEE-754 double, exact when Clinger's fast path applies; *inexact set otherwise (value then approximated)
__device__ __forceinline__ uint64_t s2_double_bits(const DocBytes &at, uint64_t i, bool &inexact) {
    const bool neg = at(i) == '-';
    uint64_t p = i + (neg ? 1u : 0u);
    uint64_t mant = 0;
    int digits = 0, dropped = 0, frac = 0;
    bool seen_nonzero = false;
    uint32_t c = at(p);
    auto take = [&](uint32_t ch, bool is_frac) {
        if (ch != '0') seen_nonzero = true;
        if (seen_nonzero) {
            if (digits < 19) {
                mant = mant * 10u + (ch - '0');
                digits++;
                if (is_frac) frac++;
            } else {
                if (ch != '0') inexact = true;
                if (!is_frac) dropped++;
            }
        } else if (is_frac) {
            frac++;
        }
    };
    while (c - '0' <= 9u) { take(c, false); c = at(++p); }
    if (c == '.') {
        c = at(++p);
        while (c - '0' <= 9u) { take(c, true); c = at(++p); }
    }
    int e10 = 0;
    if (c == 'e' || c == 'E') {
        c = at(++p);
        const bool eneg = c == '-';
        if (c == '+' || c == '-') c = at(++p);
        int ev = 0;
        while (c - '0' <= 9u) { if (ev < 100000) ev = ev * 10 + (int)(c - '0'); c = at(++p); }
        e10 = eneg ? -ev : ev;
    }
    e10 += dropped - frac;
    static const double P10[23] = {1e0, 1e1, 1e2, 1e3, 1e4, 1e5, 1e6, 1e7, 1e8, 1e9, 1e10, 1e11, 1e12, 1e13, 1e14, 1e15, 1e16, 1e17, 1e18, 1e19, 1e20, 1e21, 1e22};
    double d;
    if (mant == 0) {
        d = 0.0;
    } else if (mant < (1ull << 53) && e10 >= -22 && e10 <= 22) {
        d = (double)mant;
        d = e10 < 0 ? d / P10[-e10] : d * P10[e10];
    } else {
        inexact = true;
        d = (double)mant;
        int e = e10;
        while (e > 0) { const int s = e > 22 ? 22 : e; d *= P10[s]; e -= s; }
        while (e < 0) { const int s = -e > 22 ? 22 : -e; d /= P10[s]; e += s; }
    }
    if (neg) d = -d;
    return (uint64_t)__double_as_longlong(d);
}

// summary[3]: number of doubles whose value is not guaranteed exact
// STREAM: token k of document d writes at 1 + pos[k] + 2 d (two root words per document before it), and the tape indexes it
// stores are relative to the start of its document's slice, doc_tape[d]
template <bool STREAM>
__global__ void __launch_bounds__(256) tape_emit_kernel(const uint8_t *__restrict__ buf, uint64_t len, const uint32_t *__restrict__ idx, uint64_t n,
                                                        const uint8_t *__restrict__ prim_kind, const int64_t *__restrict__ prim_value,
                                                        const uint64_t *__restrict__ str_off, const uint32_t *__restrict__ pos, const uint8_t *__restrict__ cls,
                                                        const uint32_t *__restrict__ slot_b, const uint32_t *__restrict__ rank_a, const uint32_t *__restrict__ sorted_b,
                                                        uint32_t nbrackets, uint64_t *__restrict__ tape, uint64_t tape_cap, unsigned long long *__restrict__ summary,
                                                        const StreamArgs sa) {
    const DocBytes at = {buf, len};
    for (uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t i = idx[k];
        const uint32_t ch = at(i);
        const uint8_t t = s2_token(ch);
        uint32_t doc = 0, shift = 0;                  // STREAM: absolute position = slice-relative position + shift
        if (STREAM && (tk_open(t) || tk_close(t))) {
            doc = sa.doc_of[k];
            shift = (uint32_t)sa.doc_tape[doc] - 2u * doc;
        }
        const uint64_t p = 1ull + pos[k] + (STREAM ? 2ull * sa.doc_of[k] : 0ull);   // word 0 is the root
        if (t == TK_STR) {
            if (p < tape_cap) tape[p] = ((uint64_t)'"' << 56) | str_off[k];
        } else if (t == TK_VAL) {
            const uint8_t kd = prim_kind[k];
            if (kd == S2_INT) {
                if (p + 1 < tape_cap) {
                    tape[p] = (uint64_t)'l' << 56;
                    tape[p + 1] = (uint64_t)prim_value[k];
                }
            } else if (kd == S2_FLOAT) {
                bool inexact = false;
                const uint64_t bits = s2_double_bits(at, i, inexact);
                if (inexact) atomicAdd(summary + 3, 1ull);
                if (p + 1 < tape_cap) {
                    tape[p] = (uint64_t)'d' << 56;
                    tape[p + 1] = bits;
                }
            } else if (p < tape_cap) {
                tape[p] = (uint64_t)ch << 56;             // 't' 'f' 'n'
            }
        } else if (tk_open(t) || tk_close(t)) {
            const uint32_t s = slot_b[k];
            const bool open = tk_open(t);
            const uint32_t other_slot = open ? s + 1u : s - 1u;
            const uint32_t o = other_slot < nbrackets ? sorted_b[other_slot] : 0xFFFFFFFFu;   // the matching bracket (garbage in a broken document:
            if ((uint64_t)o < n && (open ? o > k : o < k)) {                                    //  its verdict is already an error, only stay in bounds)
                const uint32_t ko = open ? (uint32_t)k : o, kc = open ? o : (uint32_t)k;
                if (open) {
                    const uint64_t count = (kc == ko + 1u) ? 0ull : (uint64_t)(rank_a[kc] - rank_a[ko] - 1u) + 1ull;
                    if (p < tape_cap) tape[p] = ((uint64_t)ch << 56) | ((count & 0xFFFFFFull) << 32) | (uint64_t)(1u + pos[kc] + 1u - shift);
                } else {
                    const uint64_t count = (kc == ko + 1u) ? 0ull : (uint64_t)(rank_a[kc] - rank_a[ko] - 1u) + 1ull;
                    if (count > 0xFFFFFFull) {   // tape_builder.mojo:239-241
                        if (STREAM) atomicMin(sa.doc_status + doc, ((unsigned long long)(k - sa.doc_first[doc]) << 16) | (3ull << 8) | S2E_CAPACITY);
                        else atomicMin(summary, ((unsigned long long)k << 16) | (3ull << 8) | S2E_CAPACITY);
                    }
                    if (p < tape_cap) tape[p] = ((uint64_t)ch << 56) | (uint64_t)(1u + pos[ko] - shift);
                }
            }
        }
    }
}
__global__ void tape_roots_kernel(uint64_t *tape, uint64_t tape_cap, const unsigned long long *total_words, unsigned long long *summary) {
    const uint64_t N = *total_words + 2ull;      // both root words
    if (0 < tape_cap) tape[0] = ((uint64_t)'r' << 56) | N;
    if (N - 1 < tape_cap) tape[N - 1] = (uint64_t)'r' << 56;
    summary[2] = N;
}

// ---- document streams ----
// flags[k] = starts[k] (the exclusive scan of flags then numbers the documents)
__global__ void __launch_bounds__(256) stream_flags_kernel(const uint8_t *__restrict__ starts, uint64_t n, uint32_t *__restrict__ flags) {
    for (uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += (uint64_t)gridDim.x * blockDim.x) flags[k] = starts[k];
}
// doc_of[k] (in place over the scanned flags) and doc_first[d]; doc_first[n_docs] = n
__global__ void __launch_bounds__(256) stream_docs_kernel(const uint8_t *__restrict__ starts, uint64_t n, uint32_t *__restrict__ doc_of,
                                                          uint32_t *__restrict__ doc_first, const unsigned long long *__restrict__ n_docs) {
    for (uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t before = doc_of[k];
        if (starts[k]) {
            doc_first[before] = (uint32_t)k;
            doc_of[k] = before;
        } else {
            doc_of[k] = before - 1u;
        }
        if (k == 0) doc_first[*n_docs] = (uint32_t)n;
    }
}
// doc_tape[d] = words of the tokens before document d + its 2 d root words before it; both root words of every document;
// summary[2] = the whole tape's length
__global__ void __launch_bounds__(256) stream_roots_kernel(const uint32_t *__restrict__ doc_first, const uint32_t *__restrict__ pos, uint64_t n,
                                                           const unsigned long long *__restrict__ n_docs, const unsigned long long *__restrict__ total_words,
                                                           uint64_t *__restrict__ doc_tape, uint64_t *__restrict__ tape, uint64_t tape_cap,
                                                           unsigned long long *__restrict__ summary) {
    const uint64_t nd = *n_docs, N = *total_words + 2ull * nd;
    for (uint64_t d = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; d < nd; d += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t off = (uint64_t)pos[doc_first[d]] + 2ull * d;
        const uint64_t end = d + 1 < nd ? (uint64_t)pos[doc_first[d + 1]] + 2ull * (d + 1) : N;
        doc_tape[d] = off;
        if (off < tape_cap) tape[off] = ((uint64_t)'r' << 56) | (end - off);
        if (end - 1 < tape_cap) tape[end - 1] = (uint64_t)'r' << 56;
        if (d == 0) {
            doc_tape[nd] = N;
            summary[2] = N;
        }
    }
}
// summary[1] = documents whose status is not SUCCESS
__global__ void __launch_bounds__(256) stream_failed_kernel(const unsigned long long *__restrict__ doc_status, unsigned long long *__restrict__ summary) {
    const uint64_t nd = summary[0];
    for (uint64_t d0 = (uint64_t)blockIdx.x * blockDim.x; d0 < nd; d0 += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t d = d0 + threadIdx.x;
        const int c = __syncthreads_count(d < nd && doc_status[d] != ~0ull);
        if (threadIdx.x == 0 && c) atomicAdd(summary + 1, (unsigned long long)c);
    }
}

// The walk over a single document (STREAM false) or a stream of documents: the buffers and the launch sequence of both
// modes, with the steps only a stream needs behind `if constexpr`.  The caller has checked the arguments and initialised
// the summary (and, STREAM, the document status words).
template <bool STREAM>
int32_t stage2_walk(sjb200_ctx *c, const uint8_t *d_buf, uint64_t len, const uint32_t *d_idx, uint64_t n, const uint8_t *d_kind, const uint8_t *d_err,
                    const int64_t *d_value, const uint64_t *d_str_off, uint64_t *d_tape, uint64_t tape_capacity, unsigned long long *summary,
                    uint32_t *d_doc_first, uint64_t *d_doc_tape, unsigned long long *doc_status) {
    cudaStream_t s = c->stream;
    const uint64_t nblk = (n + TAPE_BLOCK - 1) / TAPE_BLOCK, dblk = (n + DEPTH_BLOCK - 1) / DEPTH_BLOCK;
    const uint32_t ntiles = (uint32_t)((n + MS_TILE - 1) / MS_TILE);
    const uint64_t hist_half = (uint64_t)MS_CLASSES * ntiles;   // hist: the B part, then the A part
    PoolBuffers tmp(c);
    Stk *d_stk = tmp.get<Stk>(nblk);
    uint32_t *d_words = tmp.get<uint32_t>(n);
    uint8_t *d_cls = tmp.get<uint8_t>(n);
    uint32_t *d_slot = tmp.get<uint32_t>(n), *d_rank = tmp.get<uint32_t>(n), *d_sorted = tmp.get<uint32_t>(n), *d_hist = tmp.get<uint32_t>(2 * hist_half);
    unsigned long long *d_tot = tmp.get<unsigned long long>(4);
    uint32_t *d_doc = STREAM ? tmp.get<uint32_t>(n) : nullptr;
    uint8_t *d_bytes = STREAM ? tmp.get<uint8_t>(n) : nullptr, *d_starts = STREAM ? tmp.get<uint8_t>(n) : nullptr;
    int32_t *d_depth = STREAM ? tmp.get<int32_t>(dblk) : nullptr;
    if (tmp.failed) return SJB200_MEMALLOC;
    const unsigned grid = grid_256(c, n);
    StreamArgs sa{};
    int32_t rc;
    if constexpr (STREAM) {
        // where documents start: the bracket depth over the structural bytes
        rc = sjb200_structural_bytes_device_async(c, d_buf, len, d_idx, n, d_bytes);
        if (rc == SJB200_SUCCESS) rc = sjb200_document_starts_device_async(c, d_bytes, n, d_starts, d_depth, dblk);
        if (rc != SJB200_SUCCESS) return rc;
        // the document of every token, and the first token of every document
        stream_flags_kernel<<<grid, 256, 0, s>>>(d_starts, n, d_doc);
        c->launches += 1;
        rc = scan_exclusive(d_doc, n, summary, c);
        if (rc != SJB200_SUCCESS) return rc;
        stream_docs_kernel<<<grid, 256, 0, s>>>(d_starts, n, d_doc, d_doc_first, summary);
        c->launches += 1;
        sa = StreamArgs{d_starts, d_doc, d_doc_first, d_doc_tape, doc_status};
    }
    // depth / container type (inside each document): the bit-stack scan; then the grammar, the words and the multisplit classes
    tape_stack_totals_kernel<STREAM><<<(unsigned)nblk, TAPE_THREADS, 0, s>>>(d_buf, len, d_idx, n, d_stk, sa.starts);
    tape_stack_scan_kernel<STREAM><<<1, 1024, 0, s>>>(d_stk, (uint32_t)nblk);
    tape_grammar_kernel<STREAM><<<(unsigned)nblk, TAPE_THREADS, 0, s>>>(d_buf, len, d_idx, n, d_kind, d_err, d_stk, d_words, d_cls, STREAM ? nullptr : summary, sa);
    c->launches += 3;
    // where every token's words go; their total is summary[1] of the single walk (the stream's [1] counts failing documents)
    rc = scan_exclusive(d_words, n, STREAM ? d_tot + 2 : summary + 1, c);
    if (rc != SJB200_SUCCESS) return rc;
    if constexpr (STREAM) {
        stream_roots_kernel<<<grid, 256, 0, s>>>(d_doc_first, d_words, n, summary, d_tot + 2, d_doc_tape, d_tape, tape_capacity, summary);
        c->launches += 1;
    }
    // brackets and commas by depth: two class-major histograms, each scanned on its own, then the ranks
    tape_multisplit_hist_kernel<<<ntiles, 32, 0, s>>>(d_cls, n, ntiles, d_hist);
    c->launches += 1;
    rc = scan_exclusive(d_hist, hist_half, d_tot, c);                                            // B: total = number of brackets
    if (rc == SJB200_SUCCESS) rc = scan_exclusive(d_hist + hist_half, hist_half, d_tot + 1, c);   // A
    if (rc != SJB200_SUCCESS) return rc;
    tape_multisplit_rank_kernel<<<ntiles, 32, 0, s>>>(d_cls, n, ntiles, d_hist, 0u, d_slot, d_rank, d_sorted);
    tape_emit_kernel<STREAM><<<grid, 256, 0, s>>>(d_buf, len, d_idx, n, d_kind, d_value, d_str_off, d_words, d_cls, d_slot, d_rank, d_sorted, (uint32_t)n,
                                                  d_tape, tape_capacity, summary, sa);
    if constexpr (STREAM) stream_failed_kernel<<<grid, 256, 0, s>>>(doc_status, summary);
    else tape_roots_kernel<<<1, 1, 0, s>>>(d_tape, tape_capacity, summary + 1, summary);
    c->launches += 3;
    return cuda_err(cudaGetLastError());
}

// What a host-to-host call reads back: the summary of sjb200_stage2_primitives_device_async, then the walk's
struct Stage2Summary {
    uint64_t first_primitive_error, strbuf_len, primitives_unused[2];
    union {
        uint64_t verdict;   // single walk: first error, all ones = SUCCESS
        uint64_t n_docs;    // stream walk
    };
    union {
        uint64_t token_words;
        uint64_t n_failed;
    };
    uint64_t tape_len, inexact_doubles;
};
static_assert(sizeof(Stage2Summary) == 64, "two summaries of 4 words");

// The device results of a host-to-host call, in buffers of the caller's PoolBuffers
struct ResidentStage2 {
    uint8_t *strbuf = nullptr;
    uint64_t *tape = nullptr, *doc_tape = nullptr, *doc_status = nullptr;
    uint32_t *doc_first = nullptr;
    Stage2Summary sum = {};
};

// The part the host-to-host calls share: primitives and the walk over the document the preceding successful sjb200_stage1 on
// this context left on the device (no second copy of the input), then both summaries read back.  Synchronous.
template <bool STREAM>
int32_t stage2_resident(sjb200_ctx *c, PoolBuffers &tmp, ResidentStage2 &r) {
    if (c->resident_len == 0 || c->resident_n == 0) return SJB200_UNINITIALIZED;   // no successful stage 1 before this call
    const uint64_t len = c->resident_len, n = c->resident_n;
    CK(cudaSetDevice(c->device));
    const uint64_t sb_cap = len + 2 * n + 64, tp_cap = STREAM ? 4 * n : 2 * n + 2;
    uint8_t *d_kind = tmp.get<uint8_t>(n), *d_err = tmp.get<uint8_t>(n);
    int64_t *d_val = tmp.get<int64_t>(n);
    uint64_t *d_off = tmp.get<uint64_t>(n);
    r.strbuf = tmp.get<uint8_t>(sb_cap);
    r.tape = tmp.get<uint64_t>(tp_cap);
    uint64_t *d_sum = tmp.get<uint64_t>(8);
    if (STREAM) {
        r.doc_first = tmp.get<uint32_t>(n + 1);
        r.doc_tape = tmp.get<uint64_t>(n + 1);
        r.doc_status = tmp.get<uint64_t>(n);
    }
    if (tmp.failed) return SJB200_MEMALLOC;
    int32_t rc = sjb200_stage2_primitives_device_async(c, c->d_in, len, c->d_out, n, d_kind, d_err, d_val, d_off, r.strbuf, sb_cap, d_sum);
    if (rc != SJB200_SUCCESS) return rc;
    if constexpr (STREAM)
        rc = sjb200_stage2_stream_device_async(c, c->d_in, len, c->d_out, n, d_kind, d_err, d_val, d_off, r.tape, tp_cap, r.doc_first, r.doc_tape, r.doc_status,
                                               d_sum + 4);
    else
        rc = sjb200_stage2_tape_device_async(c, c->d_in, len, c->d_out, n, d_kind, d_err, d_val, d_off, r.tape, tp_cap, d_sum + 4);
    if (rc != SJB200_SUCCESS) return rc;
    CK(cudaMemcpyAsync(&r.sum, d_sum, sizeof r.sum, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    return SJB200_SUCCESS;
}

}  // namespace

#pragma GCC visibility push(default)
extern "C" {

int32_t sjb200_stage2_tape_device_async(sjb200_ctx *c, const uint8_t *d_buf, uint64_t len, const uint32_t *d_idx, uint64_t n, const uint8_t *d_kind,
                                        const uint8_t *d_err, const int64_t *d_value, const uint64_t *d_str_off, uint64_t *d_tape, uint64_t tape_capacity,
                                        uint64_t *d_summary) {
    if (!c) return SJB200_UNINITIALIZED;
    if (!d_buf || !d_idx || !d_kind || !d_err || !d_value || !d_str_off || !d_tape || !d_summary) return SJB200_UNINITIALIZED;
    if (len > 0xFFFFFFFFull || n > 0x7FFFFFF0ull) return SJB200_CAPACITY;   // tape positions are 32 bit: 2 n + 2 words must fit
    if (n == 0) return SJB200_EMPTY;   // json_iterator.mojo:45-46 (at_eof)
    CK(cudaSetDevice(c->device));
    // summary: [0] first error as (index << 16 | rank of the check at that token << 8 | code), all ones = SUCCESS; [1] tape words of the tokens; [2] tape length; [3] inexact doubles
    CK(cudaMemsetAsync(d_summary, 0xFF, 8, c->stream));
    CK(cudaMemsetAsync(d_summary + 1, 0, 24, c->stream));
    return stage2_walk<false>(c, d_buf, len, d_idx, n, d_kind, d_err, d_value, d_str_off, d_tape, tape_capacity,
                              reinterpret_cast<unsigned long long *>(d_summary), nullptr, nullptr, nullptr);
}

// Stage 2 over a stream of documents (include/simdjson_b200.h): the same launches as the single-document walk, on the
// segmented stack scan, plus the document split (structural bytes and the depth scan of sjb200_document_starts_device_async),
// the document numbering, the roots of every slice and the count of failing documents.
int32_t sjb200_stage2_stream_device_async(sjb200_ctx *c, const uint8_t *d_buf, uint64_t len, const uint32_t *d_idx, uint64_t n, const uint8_t *d_kind,
                                          const uint8_t *d_err, const int64_t *d_value, const uint64_t *d_str_off, uint64_t *d_tape, uint64_t tape_capacity,
                                          uint32_t *d_doc_first, uint64_t *d_doc_tape, uint64_t *d_doc_status, uint64_t *d_summary) {
    if (!c) return SJB200_UNINITIALIZED;
    if (!d_buf || !d_idx || !d_kind || !d_err || !d_value || !d_str_off || !d_tape || !d_doc_first || !d_doc_tape || !d_doc_status || !d_summary)
        return SJB200_UNINITIALIZED;
    if (len > 0xFFFFFFFFull || n >= (1ull << 30)) return SJB200_CAPACITY;   // tape positions are 32 bit: up to 4 n words
    if (n == 0) return SJB200_EMPTY;
    CK(cudaSetDevice(c->device));
    // summary: [0] documents, [1] failing documents, [2] tape length, [3] inexact doubles
    CK(cudaMemsetAsync(d_summary, 0, 32, c->stream));
    CK(cudaMemsetAsync(d_doc_status, 0xFF, n * 8, c->stream));
    return stage2_walk<true>(c, d_buf, len, d_idx, n, d_kind, d_err, d_value, d_str_off, d_tape, tape_capacity,
                             reinterpret_cast<unsigned long long *>(d_summary), d_doc_first, d_doc_tape,
                             reinterpret_cast<unsigned long long *>(d_doc_status));
}

// Host-to-host stage 2 over a stream of documents: sjb200_stage2's counterpart for NDJSON and concatenated JSON.
int32_t sjb200_stage2_stream(sjb200_ctx *c, uint64_t *tape_out, uint64_t tape_capacity, uint8_t *strbuf_out, uint64_t strbuf_capacity, uint32_t *doc_first,
                             uint64_t *doc_tape, uint64_t *doc_status, uint64_t max_docs, uint64_t *n_docs, uint64_t *n_failed, uint64_t *tape_len,
                             uint64_t *strbuf_len, uint64_t *inexact_doubles) {
    if (!c || !tape_out || !strbuf_out || !doc_first || !doc_tape || !doc_status) return SJB200_UNINITIALIZED;
    PoolBuffers tmp(c);
    ResidentStage2 r;
    const int32_t rc = stage2_resident<true>(c, tmp, r);
    if (rc != SJB200_SUCCESS) return rc;
    const uint64_t nd = r.sum.n_docs, tl = r.sum.tape_len, sb = r.sum.strbuf_len;
    if (n_docs) *n_docs = nd;
    if (n_failed) *n_failed = r.sum.n_failed;
    if (tape_len) *tape_len = tl;
    if (strbuf_len) *strbuf_len = sb;
    if (inexact_doubles) *inexact_doubles = r.sum.inexact_doubles;
    if (nd > max_docs || tl > tape_capacity || sb > strbuf_capacity) return SJB200_CAPACITY;
    cudaStream_t s = c->stream;
    CK(cudaMemcpyAsync(tape_out, r.tape, tl * 8, cudaMemcpyDeviceToHost, s));
    if (sb) CK(cudaMemcpyAsync(strbuf_out, r.strbuf, sb, cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(doc_first, r.doc_first, (nd + 1) * 4, cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(doc_tape, r.doc_tape, (nd + 1) * 8, cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(doc_status, r.doc_status, nd * 8, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    return SJB200_SUCCESS;
}

// Host-to-host stage 2, the drop-in for DomParserImplementation.stage2 (include/generic/dom_parser_implementation.mojo:71-83):
// walks the document the preceding sjb200_stage1 call on this context left on the device (no second copy of the input),
// copies the tape and the string buffer back.  Returns the walk's verdict.
int32_t sjb200_stage2(sjb200_ctx *c, uint64_t *tape_out, uint64_t tape_capacity, uint8_t *strbuf_out, uint64_t strbuf_capacity, uint64_t *tape_len,
                      uint64_t *strbuf_len, uint64_t *inexact_doubles) {
    if (!c || !tape_out || !strbuf_out) return SJB200_UNINITIALIZED;
    PoolBuffers tmp(c);
    ResidentStage2 r;
    int32_t rc = stage2_resident<false>(c, tmp, r);
    if (rc != SJB200_SUCCESS) return rc;
    const uint64_t tl = r.sum.tape_len, sb = r.sum.strbuf_len;
    if (tape_len) *tape_len = tl;
    if (strbuf_len) *strbuf_len = sb;
    if (inexact_doubles) *inexact_doubles = r.sum.inexact_doubles;
    rc = r.sum.verdict == ~0ull ? SJB200_SUCCESS : (int32_t)(r.sum.verdict & 0xFF);
    if (rc == SJB200_SUCCESS && (tl > tape_capacity || sb > strbuf_capacity)) rc = SJB200_CAPACITY;
    if (rc != SJB200_SUCCESS) return rc;
    cudaStream_t s = c->stream;
    CK(cudaMemcpyAsync(tape_out, r.tape, tl * 8, cudaMemcpyDeviceToHost, s));
    if (sb) CK(cudaMemcpyAsync(strbuf_out, r.strbuf, sb, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    return SJB200_SUCCESS;
}

}  // extern "C"
#pragma GCC visibility pop
