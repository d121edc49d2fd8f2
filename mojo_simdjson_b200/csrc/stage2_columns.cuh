// stage2_columns.cuh -- the string cells of K pointer columns (sjb200_at_pointers_device_async) as K string columns in the
// offsets + bytes layout (Arrow, cuDF, torch nested tensors).  Included at the end of capi.cu, after stage2_pointer.cuh.
//
//   lengths   one thread per cell: the length word of the string record a '"' cell points at (after ptr_record's guard),
//             0 for every other cell; then scan_exclusive over the K·D + 1 lengths gives the offsets and the total
//   copy      balanced by output bytes, not by cells: CTAs grid-stride over windows of 4 KiB of output, aligned to the
//             destination's 16-byte boundaries.  A window finds its first and last cell by binary search in the offsets
//             (the largest i with offsets[i] <= x lands on the non-empty cell even inside a run of empty ones); each thread
//             assembles 16 consecutive output bytes, finds its starting cell by a search narrowed to the window's cells,
//             crosses cell boundaries by a galloping search (so a run of empty cells costs its logarithm, not its length),
//             and writes one 16-byte vector -- byte stores only at the head and tail of the data and at the capacity cut.
//
// The work of a CTA is one window of output bytes plus logarithmic searches, whatever the lengths: one 64 MiB string, a
// million 1-byte strings and long runs of empty cells between them cost the same per output byte.  The total exists only on
// the device after the scan, so the copy grid is sized from the SM count and the kernel reads the total itself.
//
// Compiler output (nvcc 12.9, sm_100a, -O3, -Xptxas -v): string_lengths_kernel 23 registers; string_copy_kernel 40 registers,
// 128 bytes of shared memory as ptxas reports it (16 are s_cells); no spills, no stack frames.  The SASS of the 46 kernels
// the library had before is unchanged.
#pragma once

namespace {

constexpr uint32_t COL_THREADS = 256, COL_VEC = 16, COL_WINDOW = COL_THREADS * COL_VEC;   // 4 KiB of output per window

// one thread per cell: lengths[i] = the cell's string length (0 for non-strings and for records past sb_len); lengths[n] = 0
__global__ void __launch_bounds__(256) string_lengths_kernel(const uint8_t *__restrict__ type, const int64_t *__restrict__ value, uint64_t n,
                                                             const uint8_t *__restrict__ sb, uint64_t sb_len, uint64_t *__restrict__ lengths,
                                                             unsigned long long *__restrict__ n_bad) {
    uint32_t bad = 0;
    const uint64_t first = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    for (uint64_t i = first; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        uint64_t l = 0;
        if (type[i] == '"') {
            const int64_t r = ptr_record(sb, sb_len, (uint64_t)value[i]);
            if (r < 0) bad++;
            else l = (uint64_t)r;
        }
        lengths[i] = l;
    }
    if (first == 0) lengths[n] = 0;
    bad = __reduce_add_sync(0xFFFFFFFFu, bad);
    if ((threadIdx.x & 31) == 0 && bad) atomicAdd(n_bad, (unsigned long long)bad);
}

// the largest i in [lo, hi] with off[i] <= x, given off[lo] <= x
__device__ __forceinline__ uint64_t col_last_le(const uint64_t *off, uint64_t lo, uint64_t hi, uint64_t x) {
    while (lo < hi) {
        const uint64_t mid = lo + (hi - lo + 1) / 2;
        if (off[mid] <= x) lo = mid;
        else hi = mid - 1;
    }
    return lo;
}

// the same, galloping up from lo: O(log (result - lo)) loads
__device__ __forceinline__ uint64_t col_gallop(const uint64_t *off, uint64_t lo, uint64_t hi, uint64_t x) {
    uint64_t step = 1;
    while (step <= hi - lo && off[lo + step] <= x) {
        lo += step;
        step <<= 1;
    }
    return col_last_le(off, lo, step - 1 < hi - lo ? lo + step - 1 : hi, x);
}

// grid: a multiple of the SM count; grid-stride over the windows of min(summary[0], cap) output bytes
__global__ void __launch_bounds__(COL_THREADS) string_copy_kernel(const int64_t *__restrict__ value, uint64_t n, const uint8_t *__restrict__ sb,
                                                                  const uint64_t *__restrict__ off, const unsigned long long *__restrict__ summary,
                                                                  uint8_t *__restrict__ data, uint64_t cap) {
    __shared__ uint64_t s_cells[2];
    const uint64_t total = summary[0] < cap ? summary[0] : cap;
    const uint64_t mis = (uint64_t)(uintptr_t)data & (COL_VEC - 1);   // window w starts at output byte w * COL_WINDOW - mis
    const uint64_t n_windows = (total + mis + COL_WINDOW - 1) / COL_WINDOW;
    for (uint64_t w = blockIdx.x; w < n_windows; w += gridDim.x) {
        const uint64_t ws = w * COL_WINDOW, we = ws + COL_WINDOW;          // in "output byte + mis" coordinates
        const uint64_t xs = (ws > mis ? ws - mis : 0), xe = (we - mis < total ? we - mis : total) - 1;   // the window's bytes
        if (threadIdx.x < 2) s_cells[threadIdx.x] = col_last_le(off, 0, n - 1, threadIdx.x ? xe : xs);
        __syncthreads();
        const uint64_t c0 = s_cells[0], c1 = s_cells[1];
        __syncthreads();   // s_cells is rewritten by the next window
        const uint64_t p = ws + threadIdx.x * COL_VEC;                      // this thread's 16 bytes: [p - mis, p - mis + 16)
        const uint64_t lo = p > mis ? p - mis : 0, hi = p + COL_VEC - mis < total ? p + COL_VEC - mis : total;
        if (lo >= hi) continue;
        uint64_t cell = col_last_le(off, c0, c1, lo);
        uint64_t next = off[cell + 1];
        const uint8_t *src = sb + (uint64_t)value[cell] + 4 - off[cell];   // src[x] = byte x of the output, inside this cell
        uint32_t word[4] = {0, 0, 0, 0};
#pragma unroll
        for (uint32_t b = 0; b < COL_VEC; b++) {
            const uint64_t x = p - mis + b;   // wraps below 0 in the first window: excluded by the range check
            if (x < lo || x >= hi) continue;
            if (x >= next) {
                cell = col_gallop(off, cell + 1, c1, x);
                next = off[cell + 1];
                src = sb + (uint64_t)value[cell] + 4 - off[cell];
            }
            word[b / 4] |= (uint32_t)__ldg(src + x) << (8 * (b % 4));
        }
        if (hi - lo == COL_VEC) {
            *reinterpret_cast<uint4 *>(data + lo) = make_uint4(word[0], word[1], word[2], word[3]);
        } else {
#pragma unroll
            for (uint32_t b = 0; b < COL_VEC; b++) {
                const uint64_t x = p - mis + b;
                if (x >= lo && x < hi) data[x] = (uint8_t)(word[b / 4] >> (8 * (b % 4)));
            }
        }
    }
}

}  // namespace

#pragma GCC visibility push(default)
extern "C" {

int32_t sjb200_string_columns_device_async(sjb200_ctx *c, const uint8_t *d_type, const int64_t *d_value, uint64_t n_columns, uint64_t n_docs,
                                           const uint8_t *d_strbuf, uint64_t strbuf_len, int64_t *d_offsets, uint8_t *d_data,
                                           uint64_t data_capacity, uint64_t *d_summary) {
    if (!c || !d_offsets || !d_summary) return SJB200_UNINITIALIZED;
    const bool empty = n_columns == 0 || n_docs == 0;
    if (!empty && (!d_type || !d_value || !d_strbuf)) return SJB200_UNINITIALIZED;
    if (!empty && n_docs > (1ull << 40) / n_columns) return SJB200_CAPACITY;
    CK(cudaSetDevice(c->device));
    cudaStream_t s = c->stream;
    CK(cudaMemsetAsync(d_summary, 0, 16, s));
    if (empty) {
        CK(cudaMemsetAsync(d_offsets, 0, 8, s));
        return SJB200_SUCCESS;
    }
    const uint64_t n = n_columns * n_docs;
    uint64_t *off = reinterpret_cast<uint64_t *>(d_offsets);   // lengths, then their exclusive sum: never negative
    unsigned long long *sum = reinterpret_cast<unsigned long long *>(d_summary);
    string_lengths_kernel<<<grid_256(c, n), 256, 0, s>>>(d_type, d_value, n, d_strbuf, strbuf_len, off, sum + 1);
    CK(cudaGetLastError());
    c->launches += 1;
    const int32_t rc = scan_exclusive(off, n + 1, sum, c);
    if (rc != SJB200_SUCCESS || !d_data) return rc;
    string_copy_kernel<<<(unsigned)c->sm_count * 8, COL_THREADS, 0, s>>>(d_value, n, d_strbuf, off, sum, d_data, data_capacity);
    c->launches += 1;
    return cuda_err(cudaGetLastError());
}

}  // extern "C"
#pragma GCC visibility pop
