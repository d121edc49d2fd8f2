// stage2_pointer.cuh -- JSON Pointer (RFC 6901) lookups on the tapes stage 2 leaves in device memory: for K pointers and D
// documents, K columns of D cells (type, code, value).  Included at the end of capi.cu, after stage2_tape.cuh.
//
// The rule table (what every cell holds) is this project's definition; it is in include/simdjson_b200.h and DESIGN.md §7.2,
// and tests/pointer_oracle.py restates it.  It follows upstream simdjson's DOM element::at_pointer on well-formed pointers.
//
//   host    the pointers are checked and unescaped into one flat program: per pointer its tokens, per token its bytes and
//           what it means at an array (an index, or the code it produces there); the program goes to the device with one
//           copy into a buffer from the context's pool
//   device  one thread per (pointer, document) cell, adjacent threads on adjacent documents of one pointer; a block copies
//           its pointer's tokens and bytes to shared memory, so that the threads of a warp read the same addresses.  The
//           walk is a chain of hops over the document's tape slice: an object member is a key word then a value; a value is
//           skipped by one word (" t f n), two (l d) or a jump to the open word's "index after the matching close" ({ [).
//
// Cost: O(members or elements skipped) per cell -- element i of one array costs about i dependent loads (DESIGN.md §8).
// Every tape read stays inside the document's slice and every string read inside strbuf_len, whatever the caller passes.
#pragma once

#include <vector>

namespace {

constexpr uint32_t PTR_THREADS = 256;
constexpr uint64_t PTR_PAYLOAD = (1ull << 56) - 1;
enum : uint8_t { PE_CAPACITY = 1, PE_TAPE = 3, PE_INCORRECT_TYPE = 17, PE_INDEX_OUT_OF_BOUNDS = 19, PE_NO_SUCH_FIELD = 20, PE_INVALID_POINTER = 22 };

// One token of the program: x = offset of its unescaped bytes within its pointer's bytes | length << 16;
// y = code at an array << 24 | array index (saturated at 0xFFFFFF: no successful document has an array that long).
// The device program: uint32 tok_first[K + 1], uint32 byte_first[K + 1], uint2 tokens[tok_first[K]], uint8 bytes[].
struct PtrProgram {
    std::vector<uint32_t> words;   // the program, as 32-bit words (the bytes padded to a whole word)
    uint32_t smem = 0;             // shared memory of the largest pointer: 8 bytes per token + its bytes
};

int32_t ptr_compile(const uint8_t *p, const uint64_t *off, uint64_t k_count, PtrProgram &prog) {
    if (k_count > SJB200_POINTER_MAX_COUNT) return SJB200_CAPACITY;
    for (uint64_t k = 0; k < k_count; k++)
        if (off[k + 1] < off[k]) return SJB200_INVALID_JSON_POINTER;
    if (off[k_count] - off[0] > SJB200_POINTER_MAX_BYTES) return SJB200_CAPACITY;
    std::vector<uint32_t> tok_first(1, 0), byte_first(1, 0);
    std::vector<uint32_t> toks;
    std::vector<uint8_t> bytes;
    for (uint64_t k = 0; k < k_count; k++) {
        const uint8_t *s = p + off[k];
        const uint64_t n = off[k + 1] - off[k];
        if (n && s[0] != '/') return SJB200_INVALID_JSON_POINTER;   // also "#/..." (URI fragments are not accepted)
        const uint32_t pb = (uint32_t)bytes.size();
        uint64_t i = 0;
        while (i < n) {
            i++;   // the '/'
            const uint32_t tb = (uint32_t)bytes.size() - pb;
            while (i < n && s[i] != '/') {
                if (s[i] == '~') {   // ~0 -> '~', ~1 -> '/', left to right: "~01" is "~1"
                    if (i + 1 >= n || (s[i + 1] != '0' && s[i + 1] != '1')) return SJB200_INVALID_JSON_POINTER;
                    bytes.push_back(s[i + 1] == '0' ? '~' : '/');
                    i += 2;
                } else {
                    bytes.push_back(s[i++]);
                }
            }
            const uint8_t *t = bytes.data() + pb + tb;
            const uint32_t len = (uint32_t)bytes.size() - pb - tb;
            // what the token means at an array, checked in this order
            uint32_t code = 0, index = 0;
            bool digits = true;
            for (uint32_t j = 0; j < len; j++) digits &= (uint32_t)(t[j] - '0') <= 9u;
            if (len == 1 && t[0] == '-') code = PE_INDEX_OUT_OF_BOUNDS;        // the element after the last one
            else if (len == 0) code = PE_INVALID_POINTER;
            else if (!digits) code = PE_INCORRECT_TYPE;
            else if (len > 1 && t[0] == '0') code = PE_INVALID_POINTER;         // leading zero
            else
                for (uint32_t j = 0; j < len; j++) {
                    index = index * 10 + (t[j] - '0');
                    if (index > 0xFFFFFFu) index = 0xFFFFFFu;   // saturates: 20 digits cannot overflow
                }
            toks.push_back(tb | len << 16);
            toks.push_back(code << 24 | index);
        }
        tok_first.push_back((uint32_t)toks.size() / 2);
        byte_first.push_back((uint32_t)bytes.size());
        const uint32_t ntok = tok_first[k + 1] - tok_first[k], nb = byte_first[k + 1] - byte_first[k];
        const uint32_t need = 8 * ntok + ((nb + 7) & ~7u);
        if (need > prog.smem) prog.smem = need;
    }
    bytes.resize((bytes.size() + 3) & ~(size_t)3);
    prog.words = tok_first;
    prog.words.insert(prog.words.end(), byte_first.begin(), byte_first.end());
    prog.words.insert(prog.words.end(), toks.begin(), toks.end());
    const size_t w0 = prog.words.size();
    prog.words.resize(w0 + bytes.size() / 4);
    if (!bytes.empty()) memcpy(prog.words.data() + w0, bytes.data(), bytes.size());
    return SJB200_SUCCESS;
}

__device__ __forceinline__ uint32_t ptr_load_u32(const uint8_t *p) {
    return (uint32_t)p[0] | (uint32_t)p[1] << 8 | (uint32_t)p[2] << 16 | (uint32_t)p[3] << 24;
}

// the index after the value at j, which must end at or before lim; 0 if the words say otherwise
__device__ __forceinline__ uint64_t ptr_skip(const uint64_t *w, uint64_t j, uint64_t lim) {
    if (j >= lim) return 0;
    const uint64_t word = w[j];
    switch ((uint32_t)(word >> 56)) {
    case '"': case 't': case 'f': case 'n': return j + 1;
    case 'l': case 'd': return j + 2 <= lim ? j + 2 : 0;
    case '{': case '[': {
        const uint64_t e = word & 0xFFFFFFFFull;
        return e > j + 1 && e <= lim ? e : 0;
    }
    default: return 0;
    }
}

// the length of the string record at `off`, or -1 if the record reaches past the buffer
__device__ __forceinline__ int64_t ptr_record(const uint8_t *sb, uint64_t sb_len, uint64_t off) {
    if (off > sb_len || sb_len - off < 4) return -1;
    const uint32_t len = ptr_load_u32(sb + off);
    return sb_len - off - 4 >= len ? (int64_t)len : -1;
}

// One cell: the walk of one pointer over one successful document's slice w[0 .. m).  Returns the code; type and value on success.
__device__ __forceinline__ uint8_t ptr_walk(const uint64_t *w, uint64_t m, const uint8_t *sb, uint64_t sb_len, const uint2 *tok, uint32_t ntok, const uint8_t *bytes,
                                            uint8_t *type, int64_t *value) {
    if (m < 3) return PE_TAPE;
    const uint64_t last = m - 1;   // the closing root: every value lies in [1, last)
    uint64_t i = 1;
    for (uint32_t t = 0; t < ntok; t++) {
        const uint64_t word = w[i];
        const uint32_t ty = (uint32_t)(word >> 56);
        if (ty == '{' || ty == '[') {
            const uint64_t end = word & 0xFFFFFFFFull;   // one past the matching close
            if (end <= i + 1 || end > last) return PE_TAPE;
            const uint64_t close = end - 1;
            const uint2 tk = tok[t];
            if (ty == '{') {
                const uint32_t klen = tk.x >> 16;
                const uint8_t *key = bytes + (tk.x & 0xFFFF);
                uint64_t j = i + 1;
                for (;;) {
                    if (j + 1 >= close) {   // no member left: a clean end, or a key without a value
                        if (j != close) return PE_TAPE;
                        return PE_NO_SUCH_FIELD;
                    }
                    const uint64_t kw = w[j];
                    if ((kw >> 56) != '"') return PE_TAPE;
                    const int64_t len = ptr_record(sb, sb_len, kw & PTR_PAYLOAD);
                    if (len < 0) return PE_CAPACITY;
                    if (len == klen) {   // the length first, then the bytes
                        const uint8_t *kb = sb + (kw & PTR_PAYLOAD) + 4;
                        uint32_t b = 0;
                        while (b < klen && kb[b] == key[b]) b++;
                        if (b == klen) break;   // the first match in tape order
                    }
                    j = ptr_skip(w, j + 1, close);
                    if (!j) return PE_TAPE;
                }
                i = j + 1;
            } else {
                if (tk.y >> 24) return (uint8_t)(tk.y >> 24);
                const uint32_t index = tk.y & 0xFFFFFF, count = (uint32_t)(word >> 32) & 0xFFFFFF;
                if (index >= count) return PE_INDEX_OUT_OF_BOUNDS;
                uint64_t j = i + 1;
                for (uint32_t e = 0; e < index; e++) {
                    j = ptr_skip(w, j, close);
                    if (!j) return PE_TAPE;
                }
                if (j >= close) return PE_TAPE;
                i = j;
            }
        } else if (ty == '"' || ty == 'l' || ty == 'd' || ty == 't' || ty == 'f' || ty == 'n') {
            return PE_NO_SUCH_FIELD;   // a token left, and a scalar to apply it to
        } else {
            return PE_TAPE;
        }
    }
    const uint64_t word = w[i];
    const uint32_t ty = (uint32_t)(word >> 56);
    switch (ty) {
    case 'l': case 'd':
        if (i + 1 >= last) return PE_TAPE;
        *value = (int64_t)w[i + 1];
        break;
    case 't': *value = 1; break;
    case 'f': case 'n': *value = 0; break;
    case '"': {
        if (ptr_record(sb, sb_len, word & PTR_PAYLOAD) < 0) return PE_CAPACITY;
        *value = (int64_t)(word & PTR_PAYLOAD);
        break;
    }
    case '{': case '[': *value = (int64_t)i; break;
    default: return PE_TAPE;
    }
    *type = (uint8_t)ty;
    return 0;
}

// grid (ceil(D / PTR_THREADS), K); dynamic shared memory: the largest pointer's tokens and bytes (PtrProgram::smem)
__global__ void __launch_bounds__(PTR_THREADS) at_pointer_kernel(const uint64_t *__restrict__ tape, uint64_t tape_len, const uint8_t *__restrict__ sb,
                                                                 uint64_t sb_len, const uint64_t *__restrict__ doc_tape,
                                                                 const uint64_t *__restrict__ doc_status, uint64_t n_docs,
                                                                 const uint32_t *__restrict__ prog, uint32_t n_ptr, uint8_t *__restrict__ out_type,
                                                                 uint8_t *__restrict__ out_code, int64_t *__restrict__ out_value) {
    extern __shared__ uint2 s_tok[];
    const uint32_t k = blockIdx.y;
    const uint32_t t0 = prog[k], ntok = prog[k + 1] - t0;
    const uint32_t b0 = prog[n_ptr + 1 + k], nb = prog[n_ptr + 2 + k] - b0;
    const uint2 *g_tok = reinterpret_cast<const uint2 *>(prog + 2 * (n_ptr + 1));   // 8-byte aligned: 2 (K + 1) words precede it
    const uint8_t *g_bytes = reinterpret_cast<const uint8_t *>(g_tok + prog[n_ptr]);
    uint8_t *s_bytes = reinterpret_cast<uint8_t *>(s_tok + ntok);
    for (uint32_t x = threadIdx.x; x < ntok; x += blockDim.x) s_tok[x] = g_tok[t0 + x];
    for (uint32_t x = threadIdx.x; x < nb; x += blockDim.x) s_bytes[x] = g_bytes[b0 + x];
    __syncthreads();
    const uint64_t d = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (d >= n_docs) return;
    uint8_t type = 0, code;
    int64_t value = 0;
    const uint64_t status = doc_status[d];
    if (status != ~0ull) {
        code = (uint8_t)(status & 0xFF);   // a failing document: its own code, and its slice is never read
    } else {
        const uint64_t lo = doc_tape[d], hi = doc_tape[d + 1];
        if (hi < lo || hi > tape_len) code = PE_CAPACITY;
        else code = ptr_walk(tape + lo, hi - lo, sb, sb_len, s_tok, ntok, s_bytes, &type, &value);
        if (code) type = 0, value = 0;
    }
    const uint64_t cell = (uint64_t)k * n_docs + d;
    out_type[cell] = type;
    out_code[cell] = code;
    out_value[cell] = value;
}

// sjb200_at_pointers_device_async after the compilation of its pointers
int32_t at_pointers_enqueue(sjb200_ctx *c, const PtrProgram &prog, uint64_t n_pointers, const uint64_t *d_tape, uint64_t tape_len, const uint8_t *d_strbuf,
                            uint64_t strbuf_len, const uint64_t *d_doc_tape, const uint64_t *d_doc_status, uint64_t n_docs, uint8_t *d_type, uint8_t *d_code,
                            int64_t *d_value) {
    if (n_docs == 0 || n_pointers == 0) return SJB200_SUCCESS;
    if (!d_tape || !d_strbuf || !d_doc_tape || !d_doc_status || !d_type || !d_code || !d_value) return SJB200_UNINITIALIZED;
    if (n_docs >= (1ull << 40)) return SJB200_CAPACITY;
    CK(cudaSetDevice(c->device));
    cudaStream_t s = c->stream;
    const size_t bytes = prog.words.size() * 4;
    PoolBuffers tmp(c);
    uint32_t *d_prog = tmp.get<uint32_t>(prog.words.size());
    if (tmp.failed) return SJB200_MEMALLOC;
    // pageable source: the copy has taken the bytes when it returns, so `prog` may go out of scope
    CK(cudaMemcpyAsync(d_prog, prog.words.data(), bytes, cudaMemcpyHostToDevice, s));
    if (prog.smem > 48 * 1024) CK(cudaFuncSetAttribute(at_pointer_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)prog.smem));
    const dim3 grid((unsigned)((n_docs + PTR_THREADS - 1) / PTR_THREADS), (unsigned)n_pointers);
    at_pointer_kernel<<<grid, PTR_THREADS, prog.smem, s>>>(d_tape, tape_len, d_strbuf, strbuf_len, d_doc_tape, d_doc_status, n_docs, d_prog, (uint32_t)n_pointers,
                                                          d_type, d_code, d_value);
    c->launches += 1;
    return cuda_err(cudaGetLastError());
}

}  // namespace

#pragma GCC visibility push(default)
extern "C" {

int32_t sjb200_at_pointers_device_async(sjb200_ctx *c, const uint64_t *d_tape, uint64_t tape_len, const uint8_t *d_strbuf, uint64_t strbuf_len,
                                        const uint64_t *d_doc_tape, const uint64_t *d_doc_status, uint64_t n_docs, const uint8_t *pointers,
                                        const uint64_t *pointer_offsets, uint64_t n_pointers, uint8_t *d_type, uint8_t *d_code, int64_t *d_value) {
    if (!c || !pointer_offsets || (!pointers && n_pointers)) return SJB200_UNINITIALIZED;
    PtrProgram prog;
    const int32_t rc = ptr_compile(pointers, pointer_offsets, n_pointers, prog);
    if (rc != SJB200_SUCCESS) return rc;
    return at_pointers_enqueue(c, prog, n_pointers, d_tape, tape_len, d_strbuf, strbuf_len, d_doc_tape, d_doc_status, n_docs, d_type, d_code, d_value);
}

// Host to host: the stream walk of the document the preceding sjb200_stage1 left resident, then the lookups; only the cells
// (and, on request, the string buffer) come back.
int32_t sjb200_stage2_stream_at_pointers(sjb200_ctx *c, const uint8_t *pointers, const uint64_t *pointer_offsets, uint64_t n_pointers, uint8_t *type_out,
                                         uint8_t *code_out, int64_t *value_out, uint64_t cells_capacity, uint8_t *strbuf_out, uint64_t strbuf_capacity,
                                         uint64_t *n_docs, uint64_t *strbuf_len) {
    if (!c || !pointer_offsets || (!pointers && n_pointers)) return SJB200_UNINITIALIZED;
    if (n_pointers && (!type_out || !code_out || !value_out)) return SJB200_UNINITIALIZED;
    PtrProgram prog;   // compiled once, and first: a bad pointer is refused before any device work
    int32_t rc = ptr_compile(pointers, pointer_offsets, n_pointers, prog);
    if (rc != SJB200_SUCCESS) return rc;
    PoolBuffers tmp(c);
    ResidentStage2 r;
    rc = stage2_resident<true>(c, tmp, r);
    if (rc != SJB200_SUCCESS) return rc;
    const uint64_t nd = r.sum.n_docs, sb = r.sum.strbuf_len, cells = n_pointers * nd;
    if (n_docs) *n_docs = nd;
    if (strbuf_len) *strbuf_len = sb;
    if (cells > cells_capacity || (strbuf_out && sb > strbuf_capacity)) return SJB200_CAPACITY;
    cudaStream_t s = c->stream;
    if (cells) {
        // [K][D] codes, then types, then values (8-byte aligned at 2 cells bytes rounded up)
        const uint64_t voff = (2 * cells + 7) & ~7ull;
        uint8_t *d_cells = tmp.get<uint8_t>(voff + 8 * cells);
        if (tmp.failed) return SJB200_MEMALLOC;
        rc = at_pointers_enqueue(c, prog, n_pointers, r.tape, r.sum.tape_len, r.strbuf, sb, r.doc_tape, r.doc_status, nd, d_cells + cells, d_cells,
                                 reinterpret_cast<int64_t *>(d_cells + voff));
        if (rc != SJB200_SUCCESS) return rc;
        CK(cudaMemcpyAsync(code_out, d_cells, cells, cudaMemcpyDeviceToHost, s));
        CK(cudaMemcpyAsync(type_out, d_cells + cells, cells, cudaMemcpyDeviceToHost, s));
        CK(cudaMemcpyAsync(value_out, d_cells + voff, 8 * cells, cudaMemcpyDeviceToHost, s));
    }
    if (strbuf_out && sb) CK(cudaMemcpyAsync(strbuf_out, r.strbuf, sb, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    return SJB200_SUCCESS;
}

}  // extern "C"
#pragma GCC visibility pop
