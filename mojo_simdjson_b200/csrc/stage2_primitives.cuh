// stage2_primitives.cuh -- SURVEY.md section 8(f) rank 3, first slice: the per-primitive half of mojo-simdjson's stage 2 as
// data-parallel kernels over the structural index array stage 1 leaves in HBM.  Included at the end of capi.cu.
//
// The reference walks the structurals one at a time (generic/stage2/json_iterator.mojo:40-254) and, at every value or key,
// calls one of
//   parse_string            generic/stage2/string_parsing.mojo:334-386 (+ handle_unicode_codepoint :263-331, escape_map :7-260)
//   is_valid_*_atom         include/generic/atom_parsing.mojo:34-80
//   parse_number            include/generic/number_parsing.mojo:22-80
// selected by the first byte (visit_primitive, json_iterator.mojo:306-329).  None of these depends on anything but the bytes
// at and after the structural, so here every structural is one thread:
//
//   primitives_kernel   kind, error code, value (integers), unescaped length (strings) per structural; the first error
//                       in index order (the one the sequential walk would have returned, grammar errors aside) by atomicMin
//   scan (3 launches)   exclusive prefix sum of the string records (4 + length bytes each) -> offset of every record
//   strings_kernel      every string unescaped into the string buffer, in the reference's layout: uint32 length, bytes,
//                       no terminator (generic/stage2/tape_builder.mojo:268-301)
//
// Semantics follow oracle/stage2_oracle.c (its header lists the two places where the reference cannot be restated as
// written: the 8-byte load / 32-byte advance of its string scanner -- implemented as intended, every byte examined -- and
// the standard-library number conversions -- integer value and float syntax as restated there, float value not produced).
// Bytes at or beyond the end of the document read as 0x20, stage 1's tail padding.
// First slice: one thread walks one string byte by byte; a document that is one enormous string is correct but slow.
#pragma once

#include <vector>

namespace {

enum : uint8_t { S2_NONE = 0, S2_STRING = 1, S2_INT = 2, S2_FLOAT = 3, S2_TRUE = 4, S2_FALSE = 5, S2_NULL = 6, S2_BAD = 7 };
enum : uint8_t { S2E_TAPE = 3, S2E_STRING = 5, S2E_T_ATOM = 6, S2E_F_ATOM = 7, S2E_N_ATOM = 8, S2E_NUMBER = 9 };

struct DocBytes {
    const uint8_t *buf;
    uint64_t len;
    __device__ __forceinline__ uint32_t operator()(uint64_t i) const { return i < len ? (uint32_t)__ldg(buf + i) : 0x20u; }
};

__device__ __forceinline__ bool s2_structural_or_ws(uint32_t c) {   // internal/jsoncharutils_tables.mojo:5-16
    return c == 0x09u || c == 0x0Au || c == 0x0Du || c == 0x20u || c == ',' || c == ':' || c == '[' || c == ']' || c == '{' || c == '}';
}
__device__ __forceinline__ uint32_t s2_escape(uint32_t c) {          // string_parsing.mojo:7-260
    switch (c) {
    case '"': return 0x22u;
    case '/': return 0x2Fu;
    case '\\': return 0x5Cu;
    case 'b': return 0x08u;
    case 'f': return 0x0Cu;
    case 'n': return 0x0Au;
    case 'r': return 0x0Du;
    case 't': return 0x09u;
    default: return 0u;
    }
}
__device__ __forceinline__ uint32_t s2_hex(uint32_t c) {
    if (c - '0' <= 9u) return c - '0';
    const uint32_t l = c | 0x20u;
    if (l - 'a' <= 5u) return l - 'a' + 10u;
    return 0xFFFFFFFFu;
}
__device__ __forceinline__ uint32_t s2_hex4(const DocBytes &at, uint64_t i) {   // jsoncharutils.mojo:33-45
    const uint32_t a = s2_hex(at(i)), b = s2_hex(at(i + 1)), c = s2_hex(at(i + 2)), d = s2_hex(at(i + 3));
    if ((a | b | c | d) & 0xFFFF0000u) return 0xFFFFFFFFu;
    return (a << 12) | (b << 8) | (c << 4) | d;
}
// jsoncharutils.mojo:48-81; dst == nullptr: length only
__device__ __forceinline__ uint32_t s2_utf8(uint32_t cp, uint8_t *dst) {
    if (cp <= 0x7Fu) {
        if (dst) dst[0] = (uint8_t)cp;
        return 1;
    }
    if (cp <= 0x7FFu) {
        if (dst) {
            dst[0] = (uint8_t)((cp >> 6) + 192u);
            dst[1] = (uint8_t)((cp & 63u) + 128u);
        }
        return 2;
    }
    if (cp <= 0xFFFFu) {
        if (dst) {
            dst[0] = (uint8_t)((cp >> 12) + 224u);
            dst[1] = (uint8_t)(((cp >> 6) & 63u) + 128u);
            dst[2] = (uint8_t)((cp & 63u) + 128u);
        }
        return 3;
    }
    if (cp <= 0x10FFFFu) {
        if (dst) {
            dst[0] = (uint8_t)((cp >> 18) + 240u);
            dst[1] = (uint8_t)(((cp >> 12) & 63u) + 128u);
            dst[2] = (uint8_t)(((cp >> 6) & 63u) + 128u);
            dst[3] = (uint8_t)((cp & 63u) + 128u);
        }
        return 4;
    }
    return 0;
}

// parse_string with every byte examined: src = index after the opening quote.  Returns the unescaped length or -1.
// WRITE: also stores the bytes at dst.
template <bool WRITE>
__device__ __forceinline__ int64_t s2_parse_string(const DocBytes &at, uint64_t src, uint8_t *dst) {
    uint64_t d = 0;
    for (;;) {
        const uint32_t c = at(src);
        if (c == '"') return (int64_t)d;
        if (src >= at.len) return -1;            // ran off the document (stage 1 would have said UNCLOSED_STRING)
        if (c != '\\') {
            if (WRITE) dst[d] = (uint8_t)c;
            d++;
            src++;
            continue;
        }
        const uint32_t e = at(src + 1);
        if (e == 'u') {
            uint32_t cp = s2_hex4(at, src + 2);
            src += 6;
            if (cp >= 0xD800u && cp < 0xDC00u) {
                if (!(at(src) == '\\' && at(src + 1) == 'u')) return -1;
                const uint32_t low = s2_hex4(at, src + 2) - 0xDC00u;
                if (low >> 10) return -1;
                cp = (((cp - 0xD800u) << 10) | low) + 0x10000u;
                src += 6;
            } else if (cp >= 0xDC00u && cp <= 0xDFFFu) {
                return -1;
            }
            const uint32_t n = s2_utf8(cp, WRITE ? dst + d : nullptr);
            if (n == 0) return -1;
            d += n;
        } else {
            const uint32_t r = s2_escape(e);
            if (r == 0) return -1;
            if (WRITE) dst[d] = (uint8_t)r;
            d++;
            src += 2;
        }
    }
}

// number_parsing.mojo:22-80 as restated in oracle/stage2_oracle.c
__device__ __forceinline__ uint8_t s2_parse_number(const DocBytes &at, uint64_t i, bool &is_float, int64_t &value) {
    const bool neg = at(i) == '-';
    uint64_t p = i + (neg ? 1u : 0u);
    uint64_t acc = 0, digits = 0;
    uint32_t c = at(p);
    while (c - '0' <= 9u) {
        acc = acc * 10u + (c - '0');
        digits++;
        c = at(++p);
    }
    is_float = false;
    value = 0;
    if (c == '.' || c == 'e' || c == 'E') {
        is_float = true;
        uint64_t q = p, mant = digits;
        if (at(q) == '.') {
            q++;
            while (at(q) - '0' <= 9u) {
                q++;
                mant++;
            }
        }
        bool ok = mant != 0;
        if (ok && (at(q) == 'e' || at(q) == 'E')) {
            q++;
            if (at(q) == '+' || at(q) == '-') q++;
            uint64_t ed = 0;
            while (at(q) - '0' <= 9u) {
                q++;
                ed++;
            }
            ok = ed != 0;
        }
        while (!s2_structural_or_ws(at(p))) p++;     // the token runs to the next structural or whitespace byte
        value = (int64_t)(p - i);
        return (ok && q == p) ? 0 : S2E_NUMBER;
    }
    if (!s2_structural_or_ws(c) || digits == 0) return S2E_NUMBER;
    value = (int64_t)(neg ? (uint64_t)0 - acc : acc);
    return 0;
}

__device__ __forceinline__ bool s2_four(const DocBytes &at, uint64_t i, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    return at(i) == a && at(i + 1) == b && at(i + 2) == c && at(i + 3) == d;
}

// summary[0]: (k << 8 | error) of the first failing primitive (all ones: none); [1]: bytes of string records; [2]: strings
__global__ void __launch_bounds__(256) stage2_primitives_kernel(const uint8_t *__restrict__ buf, uint64_t len, const uint32_t *__restrict__ idx, uint64_t n,
                                                                uint8_t *__restrict__ kind, uint8_t *__restrict__ err, int64_t *__restrict__ value,
                                                                uint64_t *__restrict__ rec_len, unsigned long long *__restrict__ summary) {
    const DocBytes at = {buf, len};
    for (uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t i = idx[k];
        const uint32_t c = at(i);
        uint8_t kd = S2_NONE, e = 0;
        int64_t v = 0;
        uint64_t rl = 0;
        if (c == '"') {
            kd = S2_STRING;
            int64_t l = s2_parse_string<false>(at, i + 1, nullptr);
            if (l < 0) {
                e = S2E_STRING;
                l = 0;
            }
            v = l;
            rl = 4u + (uint64_t)l;
        } else if (c == '-' || c - '0' <= 9u) {
            bool isf;
            e = s2_parse_number(at, i, isf, v);
            kd = isf ? S2_FLOAT : S2_INT;
        } else if (c == 't') {
            kd = S2_TRUE;
            e = (s2_four(at, i, 't', 'r', 'u', 'e') && s2_structural_or_ws(at(i + 4))) ? 0 : S2E_T_ATOM;
        } else if (c == 'f') {
            kd = S2_FALSE;
            e = (s2_four(at, i + 1, 'a', 'l', 's', 'e') && s2_structural_or_ws(at(i + 5))) ? 0 : S2E_F_ATOM;
        } else if (c == 'n') {
            kd = S2_NULL;
            e = (s2_four(at, i, 'n', 'u', 'l', 'l') && s2_structural_or_ws(at(i + 4))) ? 0 : S2E_N_ATOM;
        } else if (!(c == '{' || c == '}' || c == '[' || c == ']' || c == ':' || c == ',')) {
            kd = S2_BAD;
            e = S2E_TAPE;
        }
        kind[k] = kd;
        err[k] = e;
        value[k] = v;
        rec_len[k] = rl;
        if (e) atomicMin(summary, (unsigned long long)((k << 8) | e));
    }
}

// ---- exclusive prefix sum (in place), three launches: per-block totals, one CTA over the totals, per-block scan ----
constexpr int SCAN_THREADS = 256, SCAN_PER_THREAD = 8, SCAN_BLOCK = SCAN_THREADS * SCAN_PER_THREAD;

template <typename T>
__device__ __forceinline__ T scan_block_exclusive(T mine, T *s_w, T &total) {   // over the CTA's 256 threads
    T incl = mine;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const T o = __shfl_up_sync(0xFFFFFFFFu, incl, d);
        if ((int)(threadIdx.x & 31) >= d) incl += o;
    }
    if ((threadIdx.x & 31) == 31) s_w[threadIdx.x >> 5] = incl;
    __syncthreads();
    T before = 0, all = 0;
    for (int q = 0; q < SCAN_THREADS / 32; q++) {
        if (q < (int)(threadIdx.x >> 5)) before += s_w[q];
        all += s_w[q];
    }
    total = all;
    __syncthreads();
    return before + incl - mine;
}
template <typename T>
__global__ void __launch_bounds__(SCAN_THREADS) scan_totals_kernel(const T *__restrict__ x, uint64_t n, uint64_t *__restrict__ block_total) {
    __shared__ T s_w[SCAN_THREADS / 32];
    const uint64_t k0 = (uint64_t)blockIdx.x * SCAN_BLOCK + (uint64_t)threadIdx.x * SCAN_PER_THREAD;
    T mine = 0;
#pragma unroll
    for (int j = 0; j < SCAN_PER_THREAD; j++)
        if (k0 + j < n) mine += x[k0 + j];
    T total;
    scan_block_exclusive(mine, s_w, total);
    if (threadIdx.x == 0) block_total[blockIdx.x] = total;
}
__global__ void __launch_bounds__(1024) scan_of_totals_kernel(uint64_t *block_total, uint32_t nblocks, unsigned long long *grand_total) {
    __shared__ uint64_t s_w[32];
    __shared__ uint64_t s_carry;
    if (threadIdx.x == 0) s_carry = 0;
    __syncthreads();
    for (uint32_t b0 = 0; b0 < nblocks; b0 += 1024u) {
        const uint32_t b = b0 + threadIdx.x;
        const uint64_t v = b < nblocks ? block_total[b] : 0;
        uint64_t incl = v;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint64_t o = __shfl_up_sync(0xFFFFFFFFu, incl, d);
            if ((int)(threadIdx.x & 31) >= d) incl += o;
        }
        if ((threadIdx.x & 31) == 31) s_w[threadIdx.x >> 5] = incl;
        __syncthreads();
        uint64_t before_warp = 0;
        for (int q = 0; q < (int)(threadIdx.x >> 5); q++) before_warp += s_w[q];
        const uint64_t carry = s_carry;
        if (b < nblocks) block_total[b] = carry + before_warp + incl - v;
        __syncthreads();
        if (threadIdx.x == 1023) s_carry = carry + before_warp + incl;
        __syncthreads();
    }
    if (threadIdx.x == 0) *grand_total = s_carry;
}
template <typename T>
__global__ void __launch_bounds__(SCAN_THREADS) scan_apply_kernel(T *__restrict__ x, uint64_t n, const uint64_t *__restrict__ block_before) {
    __shared__ T s_w[SCAN_THREADS / 32];
    const uint64_t k0 = (uint64_t)blockIdx.x * SCAN_BLOCK + (uint64_t)threadIdx.x * SCAN_PER_THREAD;
    T v[SCAN_PER_THREAD], mine = 0;
#pragma unroll
    for (int j = 0; j < SCAN_PER_THREAD; j++) {
        v[j] = k0 + j < n ? x[k0 + j] : 0;
        mine += v[j];
    }
    T total;
    T run = (T)block_before[blockIdx.x] + scan_block_exclusive(mine, s_w, total);
#pragma unroll
    for (int j = 0; j < SCAN_PER_THREAD; j++) {
        if (k0 + j < n) x[k0 + j] = run;
        run += v[j];
    }
}

// The temporaries of one call, from the context's stream-ordered pool.  Hands out buffers until an allocation fails (from
// then on nullptr, with `failed` set and the CUDA error cleared); frees everything it handed out, stream ordered, when it
// goes out of scope.
struct PoolBuffers {
    explicit PoolBuffers(sjb200_ctx *c) : pool(c->pool), s(c->stream) {}
    PoolBuffers(const PoolBuffers &) = delete;
    PoolBuffers &operator=(const PoolBuffers &) = delete;
    ~PoolBuffers() {
        for (void *p : bufs) cudaFreeAsync(p, s);
    }
    template <typename T>
    T *get(uint64_t count) {
        void *p = nullptr;
        if (failed) return nullptr;
        if (cudaMallocFromPoolAsync(&p, count * sizeof(T), pool, s) != cudaSuccess) {
            failed = true;
            cudaGetLastError();
            return nullptr;
        }
        bufs.push_back(p);
        return static_cast<T *>(p);
    }
    cudaMemPool_t pool;
    cudaStream_t s;
    std::vector<void *> bufs;
    bool failed = false;
};

// exclusive scan of x[0 .. n) in place on the context's stream; *d_total (device) receives the grand total
template <typename T>
int32_t scan_exclusive(T *x, uint64_t n, unsigned long long *d_total, sjb200_ctx *c) {
    const uint64_t nblocks = (n + SCAN_BLOCK - 1) / SCAN_BLOCK;
    PoolBuffers tmp(c);
    uint64_t *d_totals = tmp.get<uint64_t>(nblocks);
    if (tmp.failed) return SJB200_MEMALLOC;
    scan_totals_kernel<<<(unsigned)nblocks, SCAN_THREADS, 0, c->stream>>>(x, n, d_totals);
    scan_of_totals_kernel<<<1, 1024, 0, c->stream>>>(d_totals, (uint32_t)nblocks, d_total);
    scan_apply_kernel<<<(unsigned)nblocks, SCAN_THREADS, 0, c->stream>>>(x, n, d_totals);
    c->launches += 3;
    return cuda_err(cudaGetLastError());
}

// the grid of a grid-stride kernel of 256 threads over n items: one thread per item, at most 32 CTAs per SM
unsigned grid_256(const sjb200_ctx *c, uint64_t n) {
    const uint64_t blocks = (n + 255) / 256, cap = (uint64_t)c->sm_count * 32;
    return (unsigned)(blocks < cap ? blocks : cap);
}

// every string's record {uint32 length, bytes} at strbuf + off[k]; a string that failed gets length 0
__global__ void __launch_bounds__(256) stage2_strings_kernel(const uint8_t *__restrict__ buf, uint64_t len, const uint32_t *__restrict__ idx, uint64_t n,
                                                             const uint8_t *__restrict__ kind, const uint8_t *__restrict__ err, const int64_t *__restrict__ value,
                                                             const uint64_t *__restrict__ off, uint8_t *__restrict__ strbuf, uint64_t cap) {
    const DocBytes at = {buf, len};
    for (uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += (uint64_t)gridDim.x * blockDim.x) {
        if (kind[k] != S2_STRING) continue;
        const uint64_t o = off[k];
        const uint32_t l = err[k] ? 0u : (uint32_t)value[k];
        if (o + 4u + l > cap) continue;   // the caller's buffer is too small: reported through the summary, nothing written past it
        strbuf[o] = (uint8_t)l;
        strbuf[o + 1] = (uint8_t)(l >> 8);
        strbuf[o + 2] = (uint8_t)(l >> 16);
        strbuf[o + 3] = (uint8_t)(l >> 24);
        if (l) s2_parse_string<true>(at, (uint64_t)idx[k] + 1u, strbuf + o + 4);
    }
}

}  // namespace

#pragma GCC visibility push(default)
extern "C" {

int32_t sjb200_stage2_primitives_device_async(sjb200_ctx *c, const uint8_t *d_buf, uint64_t len, const uint32_t *d_idx, uint64_t n, uint8_t *d_kind,
                                              uint8_t *d_err, int64_t *d_value, uint64_t *d_str_off, uint8_t *d_strbuf, uint64_t strbuf_capacity,
                                              uint64_t *d_summary) {
    if (!c) return SJB200_UNINITIALIZED;
    if (!d_buf || !d_idx || !d_kind || !d_err || !d_value || !d_str_off || !d_summary) return SJB200_UNINITIALIZED;
    if (len > 0xFFFFFFFFull) return SJB200_CAPACITY;
    CK(cudaSetDevice(c->device));
    cudaStream_t s = c->stream;
    // summary: {first error (k << 8 | code; all ones = none), bytes of string records, 0, 0}
    CK(cudaMemsetAsync(d_summary, 0xFF, 8, s));
    CK(cudaMemsetAsync(d_summary + 1, 0, 24, s));
    if (n == 0) return SJB200_SUCCESS;
    const unsigned grid = grid_256(c, n);
    stage2_primitives_kernel<<<grid, 256, 0, s>>>(d_buf, len, d_idx, n, d_kind, d_err, d_value, d_str_off, reinterpret_cast<unsigned long long *>(d_summary));
    CK(cudaGetLastError());
    c->launches += 1;
    const int32_t rc = scan_exclusive(d_str_off, n, reinterpret_cast<unsigned long long *>(d_summary + 1), c);
    if (rc != SJB200_SUCCESS) return rc;
    if (d_strbuf) {
        stage2_strings_kernel<<<grid, 256, 0, s>>>(d_buf, len, d_idx, n, d_kind, d_err, d_value, d_str_off, d_strbuf, strbuf_capacity);
        CK(cudaGetLastError());
        c->launches += 1;
    }
    return SJB200_SUCCESS;
}

}  // extern "C"
#pragma GCC visibility pop
