/*
 * simdjson_b200.h -- C ABI of libsimdjson_b200.so: the B200 (sm_100a) stage-1 structural indexer that sits
 * behind mojo-simdjson's stage-1 API ("input buffer in -> uint32 structural index array + error code out").
 *
 * Flat C only (pointers and fixed-width integers; no structs by value, no callbacks, no exceptions) so that
 * Mojo's sys.ffi.DLHandle.get_function / external_call, Python ctypes or any other FFI can bind it.
 * Every function returns a simdjson error code (reference src/mojo_simdjson/errors.mojo:2-34) as int32_t.
 *
 * Reference interface each entry point replaces (paths relative to the reference's src/mojo_simdjson/):
 *   sjb200_stage1            -> DomParserImplementation.stage1(Span[UInt8])
 *                               include/generic/dom_parser_implementation.mojo:65-69, i.e. the call
 *                               JsonStructuralIndexer.index[128](buffer, self) at :69
 *                               (generic/stage1/json_structural_indexer.mojo:81-186)
 *   sjb200_ctx_create        -> DomParserImplementation.__init__ + allocate()
 *                               include/generic/dom_parser_implementation.mojo:29-39, 85-89
 *   output contract          -> structural_indexes[0..n) ascending byte offsets, [n] = [n+1] = len, [n+2] = 0,
 *                               n_structural_indexes = n, next_structural_index = 0
 *                               (json_structural_indexer.mojo:160-174; consumed by
 *                               generic/stage2/json_iterator.mojo:28-38,256-288)
 *   sjb200_batch_*           -> no reference counterpart (the reference has no NDJSON / multi-document mode,
 *                               generic/stage2/tape_builder.mojo:25 "TODO: add streaming"); parity is defined
 *                               as "the reference called once per line-aligned segment"
 *
 * Differences from the reference that a caller must know:
 *   - the index array needs capacity >= n + 3 entries; the reference sizes it to len entries and writes the
 *     trailer out of bounds whenever n + 3 > len (dom_parser_implementation.mojo:85-89 vs
 *     json_structural_indexer.mojo:167-173).  Too small -> SJB200_CAPACITY instead of a wild write.
 *   - the reference's Utf8Checker is a stub (json_structural_indexer.mojo:16-30), so it never returns
 *     UTF8_ERROR.  Here the UTF-8 verdict is always computed and reported separately; it is folded into the
 *     return code only when SJB200_FLAG_VALIDATE_UTF8 is set (default off = reference-exact verdicts).
 *   - on UNCLOSED_STRING / UNESCAPED_CHARS the reference returns before assigning n_structural_indexes
 *     (:151-158); *n_out is likewise left untouched (the indexes written so far are still delivered).
 */
#ifndef SIMDJSON_B200_H
#define SIMDJSON_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SJB200_ABI_VERSION 1

/* error codes (subset of reference errors.mojo that stage 1 can return) */
#define SJB200_SUCCESS 0
#define SJB200_CAPACITY 1
#define SJB200_MEMALLOC 2
#define SJB200_UTF8_ERROR 11
#define SJB200_UNINITIALIZED 12
#define SJB200_EMPTY 13
#define SJB200_UNESCAPED_CHARS 14
#define SJB200_UNCLOSED_STRING 15
#define SJB200_UNEXPECTED_ERROR 24
/* codes of the JSON Pointer lookups (sjb200_at_pointers_device_async) */
#define SJB200_TAPE_ERROR 3
#define SJB200_INCORRECT_TYPE 17
#define SJB200_INDEX_OUT_OF_BOUNDS 19
#define SJB200_NO_SUCH_FIELD 20
#define SJB200_INVALID_JSON_POINTER 22

/* flags */
#define SJB200_FLAG_VALIDATE_UTF8 1u /* return UTF8_ERROR (lowest priority) when the input is not valid UTF-8 */
#define SJB200_FLAG_NO_UTF8 4u       /* do not even compute the UTF-8 verdict (utf8_err_out = -1) */
#define SJB200_FLAG_TIMING 8u        /* record CUDA events around the kernel (sjb200_last_elapsed_ms) */

typedef struct sjb200_ctx sjb200_ctx;

/* ABI version of the loaded library. */
int32_t sjb200_version(void);

/* Number of CUDA devices visible (0 if none / no driver). */
int32_t sjb200_device_count(void);

/*
 * Creates a parser context on `device`: a stream, look-back descriptors and a mapped result slot sized for
 * documents up to max_len bytes (< 2^32), and -- unless max_len_host == 0 -- device input/output buffers for the
 * host-to-host entry point (input max_len_host bytes, output max_len_host + 3 entries).
 * MEMALLOC on allocation failure, CAPACITY if max_len >= 2^32, UNEXPECTED_ERROR on any other CUDA error.
 */
int32_t sjb200_ctx_create(int32_t device, uint64_t max_len, uint64_t max_len_host, uint32_t flags, sjb200_ctx **ctx);
int32_t sjb200_ctx_destroy(sjb200_ctx *ctx);

/* Run all work of this context on an existing CUDA stream (cudaStream_t as void*), e.g. torch's current stream. */
int32_t sjb200_ctx_set_stream(sjb200_ctx *ctx, void *cuda_stream);
/* Force the tile shape of the PERSISTENT / SPLIT organisations: warps per tile in {2,4,8,16,24} (2 KiB per warp; SPLIT: 8 or
 * 16), 0 = choose from the document size.  A shape the selected organisation does not have makes the next stage-1 call
 * return UNEXPECTED_ERROR (never a silently different shape). */
int32_t sjb200_ctx_set_warps(sjb200_ctx *ctx, int32_t warps);
/*
 * Force the kernel organisation (tuning / test knob; every choice produces identical results):
 *   AUTO        chosen from the document size: PERSISTENT below 24 MiB and for the chunked host path, SPLIT from 24 MiB,
 *               STREAM from 80 MiB on
 *   PERSISTENT  persistent CTAs of compute warps + a scan warp over tiles, classify and flatten of a tile fused, decoupled
 *               look-back between tiles; needs no scratch
 *   SPLIT       two launches: classify (masks + per-chunk carries to L2 / HBM), then flatten
 *   STREAM      four launches, no waiting anywhere: classify with one private bulk-copy pipeline per warp (UTF-8 of sparse
 *               non-ASCII lanes validated by the same warp, 32 lanes at a time), two scan kernels over the chunk summaries,
 *               flatten
 * STREAM resolves the escape state entering a chunk from a 32-byte look-behind and, if a backslash run fills it, a walk
 * back through global memory of up to 64 KiB; a longer run makes the PERSISTENT kernel, enqueued behind the pipeline on
 * every call and otherwise returning at once, redo the document (same results).
 * SPLIT / STREAM use scratch in device memory (0.26 bytes per input byte: mask planes, chunk summaries, carry words),
 * allocated with the stream-ordered allocator on first use and grown when a larger document arrives (no call synchronises
 * for it); sjb200_ctx_reserve allocates it ahead of time.  If the allocation fails an explicit choice returns MEMALLOC, the
 * automatic choice stays with PERSISTENT.
 * Values 1, 3 and 6 named organisations that were measured, rejected and removed (one tile per CTA, in-CTA dataflow,
 * fused single launch; profiles/r2_overlap_experiments.txt): UNEXPECTED_ERROR.
 */
#define SJB200_KERNEL_AUTO 0
#define SJB200_KERNEL_PERSISTENT 2
#define SJB200_KERNEL_SPLIT 4
#define SJB200_KERNEL_STREAM 5
int32_t sjb200_ctx_set_kernel(sjb200_ctx *ctx, int32_t kind);
/* Allocates the scratch for documents of up to `len` bytes now (flags: reserved, pass 0), so that
 * no later call has to.  MEMALLOC if it cannot be had. */
int32_t sjb200_ctx_reserve(sjb200_ctx *ctx, uint64_t len, uint32_t flags);
/* Chunk size (bytes, >= 4096) of the streaming host path of sjb200_stage1: the document travels to the device in chunks
 * of this size, each indexed as soon as it has arrived.  Default 32 MiB. */
int32_t sjb200_ctx_set_chunk_bytes(sjb200_ctx *ctx, uint64_t bytes);

/*
 * Host-to-host drop-in for DomParserImplementation.stage1: copies buf to the device, indexes it, copies the
 * n + 3 entries into idx_out.  Synchronous.  idx_capacity is in entries.
 *   len == 0 -> EMPTY; len >= 2^32 or len > max_len_host -> CAPACITY; n + 3 > idx_capacity -> CAPACITY.
 * utf8_err_out (may be NULL): 1 iff the input is not valid UTF-8, -1 if not computed.
 */
int32_t sjb200_stage1(sjb200_ctx *ctx, const uint8_t *buf, uint64_t len, uint32_t *idx_out, uint64_t idx_capacity,
                      uint32_t *n_out, int32_t *utf8_err_out, uint32_t flags);

/*
 * Device-resident variant (what the roofline metric times): d_buf and d_idx are device pointers, any alignment
 * for d_buf, 4-byte alignment for d_idx.  _async only enqueues on the context's stream; _finish waits and returns
 * the verdict of the most recent _async call.  sjb200_stage1_device = _async + _finish.
 */
int32_t sjb200_stage1_device_async(sjb200_ctx *ctx, const uint8_t *d_buf, uint64_t len, uint32_t *d_idx,
                                   uint64_t idx_capacity, uint32_t flags);
int32_t sjb200_stage1_finish(sjb200_ctx *ctx, uint32_t *n_out, uint32_t *n_written_out, int32_t *utf8_err_out);
int32_t sjb200_stage1_device(sjb200_ctx *ctx, const uint8_t *d_buf, uint64_t len, uint32_t *d_idx,
                             uint64_t idx_capacity, uint32_t *n_out, int32_t *utf8_err_out, uint32_t flags);

/* Waits for everything enqueued on the context's stream. */
int32_t sjb200_sync(sjb200_ctx *ctx);

/* Kernel-only device time (ms) of the last call made with SJB200_FLAG_TIMING; negative if none. */
float sjb200_last_elapsed_ms(sjb200_ctx *ctx);
/* Number of kernels this context has launched so far. */
uint64_t sjb200_launch_count(sjb200_ctx *ctx);

/* Pinned host memory for callers that want full-speed DMA; device memory helpers for FFI callers without CUDA. */
int32_t sjb200_pinned_alloc(uint64_t bytes, void **p);
int32_t sjb200_pinned_free(void *p);
int32_t sjb200_device_alloc(sjb200_ctx *ctx, uint64_t bytes, void **p);
int32_t sjb200_device_free(sjb200_ctx *ctx, void *p);
int32_t sjb200_copy_to_device(sjb200_ctx *ctx, void *d_dst, const void *h_src, uint64_t bytes);
int32_t sjb200_copy_to_host(sjb200_ctx *ctx, void *h_dst, const void *d_src, uint64_t bytes);

/*
 * Side output for stage 2 (SURVEY.md section 8(f), rank 2): d_bytes[k] = d_buf[d_idx[k]] for k < n, the byte every
 * structural index points at.  The reference's stage 2 reads `buffer[next_structural[k]]` once per step
 * (generic/stage2/json_iterator.mojo:256-262: a dependent random read); with this array the walk reads two sequential
 * streams.  Asynchronous on the context's stream, after the stage-1 call that produced d_idx (n = its n_out; the trailer
 * entries are not included).  An index >= len yields 0.  Any alignment of d_idx / d_bytes (16-byte-aligned d_idx with
 * 4-byte-aligned d_bytes takes the vector path).
 */
int32_t sjb200_structural_bytes_device_async(sjb200_ctx *ctx, const uint8_t *d_buf, uint64_t len, const uint32_t *d_idx,
                                             uint64_t n, uint8_t *d_bytes);

/*
 * Second side output for stage 2 (SURVEY.md section 8(f), rank 2): where top-level documents start in a stream of
 * structurals -- NDJSON or any concatenation of documents indexed by ONE stage-1 call (the reference has no document
 * stream mode: generic/stage2/tape_builder.mojo:25 "TODO: add streaming").  With depth(k) = #('{' '[') - #('}' ']') among
 * the structural bytes [0, k), d_starts[k] = 1 if depth(k) == 0, else 0: structural k opens a document (a top-level
 * scalar is a document of one structural).  d_bytes is the output of sjb200_structural_bytes_device_async (n entries).
 * d_scratch: int32[scratch_entries], at least ceil(n / 4096) entries (CAPACITY otherwise); on return it holds the depth
 * before every block of 4096 structurals.  Unbalanced input is not an error here (depths may go negative; stage 2
 * diagnoses that).  Asynchronous on the context's stream.
 */
int32_t sjb200_document_starts_device_async(sjb200_ctx *ctx, const uint8_t *d_bytes, uint64_t n, uint8_t *d_starts,
                                            int32_t *d_scratch, uint64_t scratch_entries);

/*
 * NDJSON / multi-document batches.  A batch is cut at '\n' into segments; every segment is an independent stage-1 call
 * with segment-relative indexes, its own trailer and verdict -- exactly what the reference would produce if called once
 * per segment.
 *
 * The cut rule (seg_bytes in [1, 2^31 - 1]): the batch has ncuts = ceil(len / seg_bytes) windows; cut k is the position
 * right after the last '\n' among the bytes [k * seg_bytes, (k + 1) * seg_bytes), or len itself once
 * (k + 1) * seg_bytes >= len.  Segments run from one cut to the next, so every segment but the last ends in '\n' and is
 * at most 2 * seg_bytes - 1 bytes long.  A line longer than seg_bytes is accepted unless it leaves a whole window without
 * a newline: with seg_bytes = 1000, a 1500-byte line at offset 500 becomes the segment [500, 2000), while a 1001-byte
 * line at offset 0 is refused.  Blank lines are not skipped: a segment of nothing but newlines is indexed and reports
 * EMPTY.  CAPACITY if seg_bytes is 0 or larger than 2^31 - 1, if ncuts > max_segments, or if a window other than the
 * last holds no '\n'.
 *
 * sjb200_batch_split_device: finds the cut points of a device-resident batch.  seg_offsets must hold
 * max_segments + 1 entries; on return seg_offsets[0..*n_segments] are byte offsets (last one == len).  The device
 * splitter also refuses more than 4096 windows (CAPACITY).  sjb200_batch_split_host applies the same rule on the host,
 * without that limit.
 */
int32_t sjb200_batch_split_device(sjb200_ctx *ctx, const uint8_t *d_buf, uint64_t len, uint64_t seg_bytes,
                                  uint64_t *seg_offsets, uint32_t max_segments, uint32_t *n_segments);
int32_t sjb200_batch_split_host(const uint8_t *buf, uint64_t len, uint64_t seg_bytes, uint64_t *seg_offsets,
                                uint32_t max_segments, uint32_t *n_segments);
/*
 * Indexes segments [first, first+count) of a device-resident batch back to back on this context's stream.
 * Segment s writes its indexes (+ trailer) at d_idx + idx_offsets[s] (entries; caller-chosen, typically
 * seg_offsets[s] - seg_offsets[first] + 3 * (s - first)); seg_counts[s] / seg_errors[s] / seg_utf8[s] receive n,
 * the verdict and the UTF-8 verdict.  Returns the worst (numerically largest) per-segment error.
 */
int32_t sjb200_batch_run_device(sjb200_ctx *ctx, const uint8_t *d_buf, const uint64_t *seg_offsets, uint32_t first,
                                uint32_t count, uint32_t *d_idx, const uint64_t *idx_offsets, uint64_t idx_capacity,
                                uint32_t *seg_counts, int32_t *seg_errors, int32_t *seg_utf8, uint32_t flags);

/*
 * Same, without waiting: only enqueues.  If d_status is not NULL, segment first+i also leaves {error, n} as two
 * int32 at d_status[2*i] in device memory, so that the verdict exchange between GPUs (NCCL all-reduce of error
 * flags, all-gather of counts) can be enqueued behind it with no host round trip.  Returns the worst launch error.
 */
int32_t sjb200_batch_run_device_async(sjb200_ctx *ctx, const uint8_t *d_buf, const uint64_t *seg_offsets,
                                      uint32_t first, uint32_t count, uint32_t *d_idx, const uint64_t *idx_offsets,
                                      uint64_t idx_capacity, int32_t *d_status, uint32_t flags);

/*
 * Multi-GPU batch driver (SURVEY.md section 8(b) / 8(e)): owns one context per GPU and the NCCL communicators.  The batch
 * is cut at '\n' into one shard per GPU and every shard into segments of < 2 * seg_bytes (the rule above; each segment = one reference
 * stage-1 call, dom_parser_implementation.mojo:65-69, on that byte range).  Per pass the GPUs exchange ONE NCCL all-gather
 * of the {error, n} rows of their segments -- the only inter-GPU traffic; the worst error is the maximum over the rows.
 * NCCL is loaded at run time (libnccl.so.2, or the path in SJB200_NCCL_LIB) and only when more than one GPU takes part.
 *
 * sjb200_batch_create: ONE process drives `ngpus` devices (devices == NULL: 0 .. ngpus-1; communicators from
 *   ncclCommInitAll).  max_shard_bytes > 0 also allocates, per GPU, staging for the host-batch entry point sjb200_batch_run.
 * sjb200_batch_create_rank: one process PER GPU (torchrun / MPI): rank `rank` of `world` on `device`; nccl_id = the 128
 *   bytes sjb200_batch_unique_id produced on rank 0, carried to the other ranks by the caller (ncclCommInitRank inside).
 * max_segments: rows per GPU in the exchange (<= 256).
 */
typedef struct sjb200_batch sjb200_batch;
int32_t sjb200_batch_unique_id(void *id128);
int32_t sjb200_batch_create(int32_t ngpus, const int32_t *devices, uint64_t max_shard_bytes, uint64_t seg_bytes,
                            uint32_t max_segments, uint32_t flags, sjb200_batch **batch);
int32_t sjb200_batch_create_rank(int32_t device, int32_t rank, int32_t world, const void *nccl_id, uint64_t max_shard_bytes,
                                 uint64_t seg_bytes, uint32_t max_segments, uint32_t flags, sjb200_batch **batch);
int32_t sjb200_batch_destroy(sjb200_batch *batch);
/* GPUs this process drives, and the context of one of them (e.g. to put it on an existing stream). */
int32_t sjb200_batch_local_gpus(sjb200_batch *batch);
int32_t sjb200_batch_ctx(sjb200_batch *batch, int32_t local_gpu, sjb200_ctx **ctx);
/*
 * Host batch in, host indexes out (single-process mode): shards [0, len) over the GPUs by line ranges, copies every shard
 * to its GPU, indexes its segments, exchanges the verdicts, copies every segment's n + 3 entries back.  On return
 * seg_offsets[0 .. *n_segments] are the byte offsets of the segments in buf, seg_idx_offsets[s] the entry of idx_out where
 * segment s starts (= seg_offsets[s] + 3 * s), seg_counts / seg_errors the per-segment n and verdict (may be NULL),
 * *global_error the worst verdict over the whole batch.  CAPACITY if a shard exceeds max_shard_bytes, the batch needs more
 * than max_total_segments segments, or idx_capacity < len + 3 * segments.
 */
int32_t sjb200_batch_run(sjb200_batch *batch, const uint8_t *buf, uint64_t len, uint32_t *idx_out, uint64_t idx_capacity,
                         uint64_t *seg_offsets, uint64_t *seg_idx_offsets, uint32_t *seg_counts, int32_t *seg_errors,
                         uint32_t max_total_segments, uint32_t *n_segments, int32_t *global_error, uint32_t flags);
/*
 * Device-resident shards (what the scaling benchmark times).  plan: cuts the shard that is resident on local GPU
 * `local_gpu` into segments (device-side newline search; seg_offsets / idx_offsets: max_segments + 1 entries, may be NULL).
 * run_resident_async: one pass -- per local GPU its segments back to back into d_idx[g] (segment s at idx_offsets[s]),
 * then the all-gather on an internal stream, so that it runs beside the kernels of the next pass; never blocks the host.
 * finish: waits for everything in flight; all_rows (may be NULL): int32 [world][max_segments][2] = {error, n} of every
 * segment of every rank after the most recent pass ({-1, -1}: no such segment); *global_error: the worst of them.
 */
int32_t sjb200_batch_plan_resident(sjb200_batch *batch, int32_t local_gpu, const uint8_t *d_shard, uint64_t shard_len,
                                   uint64_t *seg_offsets, uint64_t *idx_offsets, uint32_t *n_segments);
int32_t sjb200_batch_run_resident_async(sjb200_batch *batch, uint32_t *const *d_idx, const uint64_t *idx_capacities, uint32_t flags);
int32_t sjb200_batch_finish(sjb200_batch *batch, int32_t *all_rows, int32_t *global_error);

/*
 * SURVEY.md section 8(f) rank 3, first slice -- the per-primitive half of stage 2 over the index array stage 1 left on the
 * device.  For every structural k < n, as the reference's visit_primitive (generic/stage2/json_iterator.mojo:306-329)
 * would treat the byte it points at:
 *   kind[k]    0 structural character, 1 string, 2 integer, 3 float, 4 true, 5 false, 6 null, 7 anything else
 *   err[k]     simdjson error code of that primitive: 0, STRING_ERROR 5 (parse_string, string_parsing.mojo:334-386),
 *              T/F/N_ATOM_ERROR 6/7/8 (atom_parsing.mojo:34-80), NUMBER_ERROR 9 (number_parsing.mojo:22-80), TAPE_ERROR 3
 *   value[k]   strings: unescaped length; integers: the value; floats: token length
 *   str_off[k] strings: offset of the string's record in strbuf
 *   strbuf     (may be NULL) every string unescaped, in index order, as the reference's string buffer holds it: uint32
 *              length, then the bytes, no terminator (tape_builder.mojo:268-301); a string that fails gets length 0
 *   summary    4 x uint64 on the device: [0] = (k << 8 | error) of the first failing primitive in index order, all ones if
 *              none -- the error the sequential walk would have returned, grammar (TAPE / DEPTH) errors aside; [1] = bytes
 *              of string records (what strbuf must hold; records that do not fit strbuf_capacity are not written)
 * Stream ordered on the context's stream; nothing is copied to the host.  Semantics: oracle/stage2_oracle.c, whose header
 * lists the two places where the reference cannot be restated as written (string scanner stride, standard-library number
 * conversions).  Bytes at or beyond len read as 0x20.
 */
int32_t sjb200_stage2_primitives_device_async(sjb200_ctx *ctx, const uint8_t *d_buf, uint64_t len, const uint32_t *d_idx, uint64_t n,
                                              uint8_t *d_kind, uint8_t *d_err, int64_t *d_value, uint64_t *d_str_off, uint8_t *d_strbuf,
                                              uint64_t strbuf_capacity, uint64_t *d_summary);

/*
 * SURVEY.md section 8(f) rank 4, first slice -- the stage-2 walk: the verdict JsonIterator.walk_document would return
 * (generic/stage2/json_iterator.mojo:40-254, restated in oracle/stage2_oracle.c: oracle_stage2_walk) and the tape, computed
 * in parallel over the index array (d_idx holds n indexes; the trailer is not read).  d_kind / d_err / d_value / d_str_off are
 * the outputs of sjb200_stage2_primitives_device_async for the same document.
 *   tape     64-bit words, type character in the top byte (include/internal/tape_type.mojo): 'r' | N ... 'r' | 0 roots,
 *            '{' '[' | count << 32 | index after the matching close, '}' ']' | index of the matching open, '"' | offset of
 *            the string record, 'l' | 0 + int64, 'd' | 0 + IEEE-754 bits, 't' 'f' 'n' | 0; at most 2 n + 2 words
 *   summary  4 x uint64 on the device: [0] all ones = SUCCESS, else index << 16 | check << 8 | error code of the first failing
 *            token (TAPE_ERROR 3, DEPTH_ERROR 4 -- depth limit 100, dom_parser_implementation.mojo:40 --, the primitive's own
 *            code, CAPACITY 1 for a container of more than 0xFFFFFF elements); [1] words appended by the tokens; [2] N;
 *            [3] doubles whose bits are not guaranteed exact (outside the exact fast path: > 15 digits or |exponent| > 22)
 * The tape is meaningful only when [0] says SUCCESS.  EMPTY if n == 0.  Tape parity with the reference is UNPINNED: its own
 * tape_builder is unfinished (see the oracle's header); the format is the one its comments describe.
 */
int32_t sjb200_stage2_tape_device_async(sjb200_ctx *ctx, const uint8_t *d_buf, uint64_t len, const uint32_t *d_idx, uint64_t n,
                                        const uint8_t *d_kind, const uint8_t *d_err, const int64_t *d_value, const uint64_t *d_str_off,
                                        uint64_t *d_tape, uint64_t tape_capacity, uint64_t *d_summary);

/*
 * Host-to-host stage 2: replaces DomParserImplementation.stage2 (include/generic/dom_parser_implementation.mojo:71-83, which
 * sizes the document's tape and string buffer and calls TapeBuilder.parse_document).  Walks the document that the preceding,
 * successful sjb200_stage1 call on this context left resident on the device -- primitives, then the walk -- and copies the
 * tape (<= 2 n + 2 words) and the string buffer (<= len + 2 n bytes) back.  Returns the walk's verdict (SUCCESS, TAPE_ERROR,
 * DEPTH_ERROR, STRING_ERROR, T/F/N_ATOM_ERROR, NUMBER_ERROR, CAPACITY); UNINITIALIZED without such a stage-1 call; CAPACITY
 * also when an output does not fit.  On an error verdict the outputs are not written.  Synchronous.
 */
int32_t sjb200_stage2(sjb200_ctx *ctx, uint64_t *tape_out, uint64_t tape_capacity, uint8_t *strbuf_out, uint64_t strbuf_capacity,
                      uint64_t *tape_len, uint64_t *strbuf_len, uint64_t *inexact_doubles);

/*
 * Stage 2 over a stream of documents (NDJSON, or JSON documents simply concatenated), indexed by ONE stage-1 call: a
 * verdict and a tape for every document, in one device pass.  Upstream simdjson calls this parse_many; the reference has
 * no stream mode (generic/stage2/tape_builder.mojo:25 "TODO: add streaming").
 *
 * Documents.  Structural k starts a document iff the bracket depth over the structurals before it ('{' '[' +1, '}' ']' -1)
 * is 0 -- the rule of sjb200_document_starts_device_async.  Document d is the tokens [doc_first[d], doc_first[d + 1]),
 * doc_first[n_docs] = n.  Consequences: scalars separated by whitespace are separate documents (`1 2`, `"a" "b"`,
 * `[1] 2` are two each); documents need no separator (`[1][2]`, `{}{}`); a document left unclosed swallows the rest of
 * the stream; a stray close is a document of its own that fails, and everything after it up to where the depth returns
 * to 0 belongs to it.  On well-formed input this separates documents the way parse_many does.  Lines play no part.
 *
 * Verdicts.  doc_status[d] is exactly the verdict the single-document walk (sjb200_stage2_tape_device_async, oracle
 * oracle_stage2_walk) gives on document d alone, i.e. on its index sub-array followed by the trailer len, len, 0, in the
 * same encoding: all ones = SUCCESS, else k << 16 | check << 8 | code with k relative to doc_first[d] (an unclosed last
 * document fails at k = its length).  The reference's oddities hold per document: a root-level {} or [] is TAPE_ERROR,
 * arrays hit DEPTH_ERROR one level before objects, more than 0xFFFFFF elements is CAPACITY.  A document's verdict never
 * depends on any other document.
 *
 * Tape.  One tape for the stream; document d owns the words [doc_tape[d], doc_tape[d + 1]): 2 root words plus, per token,
 * 1 word for strings, brackets and t f n, 2 for numbers, 0 for ':' ','.  The slice length does not depend on the verdict;
 * the whole tape is at most 2 n + 2 n_docs <= 4 n words.  The slice of a successful document is the tape the
 * single-document walk produces for it, with its root words and container indexes relative to the slice; its string words
 * hold offsets into the stream's ONE string buffer, the one sjb200_stage2_primitives_device_async writes for all tokens in
 * index order.  The words inside a failing document's slice are unspecified; nothing is written outside a document's slice.
 *
 * sjb200_stage2_stream_device_async: d_kind / d_err / d_value / d_str_off are the outputs of
 * sjb200_stage2_primitives_device_async for the same indexes.  d_doc_first and d_doc_tape hold n + 1 entries, d_doc_status n
 * (there are at most n documents); d_summary 4 x uint64: [0] documents, [1] failing documents, [2] tape words, [3] doubles
 * not guaranteed exact.  Writes past tape_capacity are dropped; [2] still reports the full length.  EMPTY if n == 0,
 * CAPACITY if len >= 2^32 or n >= 2^30.  Stream ordered on the context's stream; temporaries from its pool.
 *
 * sjb200_stage2_stream: host to host, after a successful sjb200_stage1 on this context (the resident copy, like
 * sjb200_stage2).  doc_first and doc_tape hold max_docs + 1 entries, doc_status max_docs.  Returns the call's status, not
 * the documents': SUCCESS when the outputs were delivered, also when documents fail (their verdicts are in doc_status);
 * CAPACITY when n_docs > max_docs or the tape or the strings do not fit (nothing is copied, the sizes are set so that the
 * caller can retry); UNINITIALIZED without such a stage-1 call.  Synchronous.
 */
int32_t sjb200_stage2_stream_device_async(sjb200_ctx *ctx, const uint8_t *d_buf, uint64_t len, const uint32_t *d_idx, uint64_t n,
                                          const uint8_t *d_kind, const uint8_t *d_err, const int64_t *d_value, const uint64_t *d_str_off,
                                          uint64_t *d_tape, uint64_t tape_capacity, uint32_t *d_doc_first, uint64_t *d_doc_tape,
                                          uint64_t *d_doc_status, uint64_t *d_summary);
int32_t sjb200_stage2_stream(sjb200_ctx *ctx, uint64_t *tape_out, uint64_t tape_capacity, uint8_t *strbuf_out, uint64_t strbuf_capacity,
                             uint32_t *doc_first, uint64_t *doc_tape, uint64_t *doc_status, uint64_t max_docs, uint64_t *n_docs,
                             uint64_t *n_failed, uint64_t *tape_len, uint64_t *strbuf_len, uint64_t *inexact_doubles);

/*
 * JSON Pointer (RFC 6901) lookups on the device tapes: for K pointers and D documents, K columns of D cells.  The rules
 * below are this project's definition (restated in tests/pointer_oracle.py, DESIGN.md section 7.2).  They follow upstream
 * simdjson's DOM element::at_pointer on well-formed pointers; where upstream releases differ (a token applied to a scalar)
 * this table pins the choice.
 *
 * Input: a tape with one slice per document, its string buffer, each document's slice bounds doc_tape[d] .. doc_tape[d + 1]
 * and status word doc_status[d] -- the outputs of sjb200_stage2_stream_device_async.  One document from
 * sjb200_stage2_tape_device_async is the case D = 1: doc_tape = {0, summary[2]}, doc_status = {summary[0]}.
 *
 * Pointers.  Pointer k is the bytes pointers[pointer_offsets[k] .. pointer_offsets[k + 1]) (UTF-8 by convention).  It is
 * empty (the root value, slice word 1) or a sequence of '/'-prefixed tokens; in a token "~1" becomes '/' and "~0" becomes
 * '~', left to right ("~01" is "~1").  A pointer that is not empty and does not start with '/' ("#/..." URI fragments
 * included), a '~' not followed by '0' or '1', or decreasing offsets: INVALID_JSON_POINTER for the whole call, nothing
 * written.  More than SJB200_POINTER_MAX_COUNT pointers or more than SJB200_POINTER_MAX_BYTES pointer bytes in all: CAPACITY.
 *
 * Cells.  The walk starts at the root value and applies one token at a time:
 *   object     the FIRST member in tape order whose unescaped key bytes equal the token's (upstream's DOM at_key; python's
 *              json keeps the last); none: NO_SUCH_FIELD
 *   array      of c elements (exact: a successful document has none of 2^24 or more), checked in this order:
 *              token "-": INDEX_OUT_OF_BOUNDS; empty token: INVALID_JSON_POINTER; a byte outside 0-9: INCORRECT_TYPE ("0a");
 *              more than one digit with a leading 0: INVALID_JSON_POINTER; value >= c (saturating, no overflow):
 *              INDEX_OUT_OF_BOUNDS; else element value
 *   scalar     a token left: NO_SUCH_FIELD
 * A failing document (status not all ones) gives every cell its own code status & 0xFF; its slice is never read.
 * Guards against caller-supplied arrays (a tape this library writes never triggers them): a slice that reaches past
 * tape_len, or a string record the walk reads that reaches past strbuf_len: CAPACITY; a tape word that points outside the
 * slice or its container, or a word of the wrong type: TAPE_ERROR.  Every read stays inside the slice and strbuf_len.
 *
 * Outputs, pointer-major ([K][D], cell k * n_docs + d; each column contiguous):
 *   type   uint8: the tape type character of the value found ('{' '[' '"' 'l' 'd' 't' 'f' 'n'), 0 when code != SUCCESS
 *   code   uint8: SUCCESS, or the code from the rules above
 *   value  int64: 'l' the integer; 'd' the IEEE-754 bits (the tape's payload, with its inexactness caveat); 't' 1, 'f' 'n' 0;
 *          '"' the offset of the string's {uint32 length, bytes} record in the string buffer; '{' '[' the slice-relative
 *          index of the container's open word.  0 when code != SUCCESS.
 * Cost: a cell costs O(members or elements skipped); element i of one array costs about i dependent loads.
 *
 * sjb200_at_pointers_device_async: pointers and pointer_offsets (K + 1 entries) are host memory, everything else device
 * memory.  Stream ordered on the context's stream.  n_docs == 0 or K == 0: SUCCESS, nothing written.  Nothing is written
 * outside the K x D cells.
 *
 * sjb200_stage2_stream_at_pointers: host to host, over the document the preceding successful sjb200_stage1 on this context
 * left resident (like sjb200_stage2_stream): the primitives, the stream walk and the lookups run on the device; only the
 * K x D cells come back, plus the string buffer if strbuf_out is not NULL (to read string cells).  cells_capacity is in
 * cells.  CAPACITY when the cells or the strings do not fit (nothing copied; *n_docs and *strbuf_len are set so that the
 * caller can retry); UNINITIALIZED without such a stage-1 call.  Synchronous.
 */
#define SJB200_POINTER_MAX_COUNT 1024
#define SJB200_POINTER_MAX_BYTES 16384
int32_t sjb200_at_pointers_device_async(sjb200_ctx *ctx, const uint64_t *d_tape, uint64_t tape_len, const uint8_t *d_strbuf, uint64_t strbuf_len,
                                        const uint64_t *d_doc_tape, const uint64_t *d_doc_status, uint64_t n_docs, const uint8_t *pointers,
                                        const uint64_t *pointer_offsets, uint64_t n_pointers, uint8_t *d_type, uint8_t *d_code, int64_t *d_value);
int32_t sjb200_stage2_stream_at_pointers(sjb200_ctx *ctx, const uint8_t *pointers, const uint64_t *pointer_offsets, uint64_t n_pointers,
                                         uint8_t *type_out, uint8_t *code_out, int64_t *value_out, uint64_t cells_capacity, uint8_t *strbuf_out,
                                         uint64_t strbuf_capacity, uint64_t *n_docs, uint64_t *strbuf_len);

/*
 * String columns from pointer cells: the string cells of K columns of D cells (the type and value outputs of
 * sjb200_at_pointers_device_async, [K][D], pointer-major) become K string columns in the offsets + bytes layout (Arrow,
 * cuDF, torch nested tensors), on the device.
 *
 * Input: d_type and d_value (K x D cells each) and the string buffer the cells point into, strbuf_len bytes of it.  A cell
 * with type '"' is a string: its bytes are those of the {uint32 length, bytes} record at d_strbuf + value.  Every other cell,
 * found or not, contributes 0 bytes.
 *
 * Outputs:
 *   d_offsets  K·D + 1 int64 (8-byte aligned): one exclusive prefix sum of the cell lengths over all K·D cells in cell order,
 *              d_offsets[K·D] = total bytes.  Cell i's bytes are d_data[d_offsets[i] .. d_offsets[i + 1]); column k is
 *              d_offsets[k·D .. k·D + D] inclusive (neighbouring columns share an endpoint), one contiguous slice of d_data.
 *   d_data     every string's unescaped bytes exactly as its record holds them: no length words, no terminators.  Any
 *              alignment.  Bytes at or past data_capacity are never written; every byte below min(total, data_capacity) is.
 *              May be NULL: then only the offsets and the summary are written, so that a caller can size the buffer first.
 *   d_summary  2 x uint64: [0] total bytes (the full figure, also when it exceeds data_capacity); [1] the number of string
 *              cells whose record does not lie inside strbuf_len (the guard of the pointer lookups).  Those cells get length
 *              0; cells sjb200_at_pointers_device_async wrote over the same buffer never trigger it.
 * Every read stays inside d_type, d_value, d_offsets and strbuf_len, whatever the caller passes.
 *
 * UNINITIALIZED for a NULL ctx, d_offsets or d_summary, or, when K·D > 0, a NULL d_type, d_value or d_strbuf.  CAPACITY
 * when K·D > 2^40.  K·D == 0: SUCCESS, d_offsets[0] = 0, summary zeroed.  Stream ordered on the context's stream, no host
 * synchronisation; temporaries from its pool.  The copy is balanced by output bytes, not by cells: its cost does not
 * depend on how the bytes are spread over the cells.
 */
int32_t sjb200_string_columns_device_async(sjb200_ctx *ctx, const uint8_t *d_type, const int64_t *d_value, uint64_t n_columns, uint64_t n_docs,
                                           const uint8_t *d_strbuf, uint64_t strbuf_len, int64_t *d_offsets, uint8_t *d_data,
                                           uint64_t data_capacity, uint64_t *d_summary);

#ifdef __cplusplus
}
#endif
#endif /* SIMDJSON_B200_H */
