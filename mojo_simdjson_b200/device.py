"""Device-resident stage 1 over torch tensors (torch supplies device memory and streams; the compute is ours).

This is the path the roofline metric times: input already in HBM, indexes left in HBM.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

import torch

from . import _native, errors


@dataclass
class DeviceResult:
    error: int
    n: int | None       # None where the reference leaves n_structural_indexes untouched
    n_written: int
    utf8_error: int


def pointer_program(pointers) -> tuple[bytes, "C.Array"]:
    """The pointers (str or bytes) as the flat byte string and the K + 1 offsets the C entry points take."""
    raw = [p.encode("utf-8") if isinstance(p, str) else bytes(p) for p in pointers]
    offs = [0]
    for p in raw:
        offs.append(offs[-1] + len(p))
    return b"".join(raw), (C.c_uint64 * len(offs))(*offs)


@dataclass
class PointerColumns:
    """K columns of D cells from Stage1Context.at_pointers, each a [K, D] device tensor (include/simdjson_b200.h,
    sjb200_at_pointers_device_async): type (uint8, the tape type character or 0), code (uint8, 0 = found), value (int64)."""
    type: torch.Tensor
    code: torch.Tensor
    value: torch.Tensor

    def int64(self, k: int) -> tuple[torch.Tensor, torch.Tensor]:
        """(values, mask) of column k: the integers of 'l' cells, 0 elsewhere."""
        mask = self.type[k] == ord("l")
        return torch.where(mask, self.value[k], torch.zeros_like(self.value[k])), mask

    def float64(self, k: int) -> tuple[torch.Tensor, torch.Tensor]:
        """(values, mask) of column k: 'd' cells bit-cast, 'l' cells converted as float(int) would (nearest), 0 elsewhere."""
        t, v = self.type[k], self.value[k]
        is_d, is_l = t == ord("d"), t == ord("l")
        out = torch.where(is_d, v.view(torch.float64), v.to(torch.float64))
        mask = is_d | is_l
        return torch.where(mask, out, torch.zeros_like(out)), mask

    def boolean(self, k: int) -> tuple[torch.Tensor, torch.Tensor]:
        """(values, mask) of column k: True for 't' cells, False for 'f' cells and everywhere else."""
        t = self.type[k]
        return t == ord("t"), (t == ord("t")) | (t == ord("f"))


@dataclass
class StringColumns:
    """K string columns of D cells from Stage1Context.string_columns, in the offsets + bytes layout (include/simdjson_b200.h,
    sjb200_string_columns_device_async): offsets (int64 [K·D + 1], one prefix sum over every cell, column k is
    offsets[k·D .. k·D + D]), data (uint8 [total], the strings' bytes back to back), mask (bool [K, D], True for string
    cells).  Every non-string cell is empty."""
    offsets: torch.Tensor
    data: torch.Tensor
    mask: torch.Tensor
    bounds: list[int]   # offsets[k·D] for k = 0 .. K, on the host: where each column's bytes start and end

    def column(self, k: int) -> tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
        """(offsets int64 [D + 1] rebased to 0, data uint8 view of the column's bytes, mask bool [D]) of column k."""
        d = self.mask.shape[1]
        return self.offsets[k * d : k * d + d + 1] - self.bounds[k], self.data[self.bounds[k] : self.bounds[k + 1]], self.mask[k]

    def to_list(self, k: int) -> list:
        """Column k on the host: bytes for string cells, None for every other cell."""
        off, data, mask = (t.cpu() for t in self.column(k))
        off, raw = off.tolist(), data.numpy().tobytes()
        return [raw[off[d] : off[d + 1]] if m else None for d, m in enumerate(mask.tolist())]


class Stage1Context:
    """One parser context per GPU; runs on torch's current stream of that device by default."""

    def __init__(self, device: int | torch.device = 0, max_len: int = (1 << 32) - 1, max_len_host: int = 0,
                 use_torch_stream: bool = True):
        self._lib = _native.lib()
        dev = torch.device("cuda", device) if isinstance(device, int) else device
        if not torch.cuda.is_available():
            raise RuntimeError("no CUDA device: the stage-1 path has no CPU fallback")
        self.device = dev
        self._ctx = C.c_void_p()
        rc = self._lib.sjb200_ctx_create(dev.index or 0, max_len, max_len_host, 0, C.byref(self._ctx))
        if rc != errors.SUCCESS:
            raise RuntimeError(f"sjb200_ctx_create failed: {errors.NAMES.get(rc, rc)}")
        if use_torch_stream:
            self.use_stream(torch.cuda.current_stream(dev))

    @classmethod
    def borrow(cls, ctx_ptr: C.c_void_p, device: torch.device) -> "Stage1Context":
        """Wraps a context that something else owns (the in-library batch driver's): close() leaves it alone."""
        self = cls.__new__(cls)
        self._lib = _native.lib()
        self.device = device
        self._ctx = ctx_ptr
        self._borrowed = True
        return self

    def use_stream(self, stream: torch.cuda.Stream) -> None:
        self._stream = stream
        self._lib.sjb200_ctx_set_stream(self._ctx, C.c_void_p(stream.cuda_stream))

    def set_warps(self, warps: int) -> None:
        rc = self._lib.sjb200_ctx_set_warps(self._ctx, warps)
        if rc != errors.SUCCESS:
            raise ValueError("warps must be 0, 2, 4, 8, 16 or 24")

    KERNELS = {"auto": 0, "persistent": 2, "split": 4, "stream": 5}

    def reserve(self, length: int, stream_pipeline: bool = False) -> None:
        """Allocate the scratch for documents of up to `length` bytes now (otherwise: on first use, stream ordered)."""
        rc = self._lib.sjb200_ctx_reserve(self._ctx, length, 1 if stream_pipeline else 0)
        if rc != errors.SUCCESS:
            raise RuntimeError(f"sjb200_ctx_reserve failed: {errors.NAMES.get(rc, rc)}")

    def set_kernel(self, kind) -> None:
        """Force the kernel organisation (include/simdjson_b200.h, SJB200_KERNEL_*); results do not depend on it."""
        rc = self._lib.sjb200_ctx_set_kernel(self._ctx, self.KERNELS[kind] if isinstance(kind, str) else int(kind))
        if rc != errors.SUCCESS:
            raise ValueError(f"unknown kernel kind {kind!r}")

    def close(self):
        if self._ctx:
            if not getattr(self, "_borrowed", False):
                self._lib.sjb200_ctx_destroy(self._ctx)
            self._ctx = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- single document -------------------------------------------------------------------------
    def enqueue(self, buf: torch.Tensor, out: torch.Tensor, flags: int = 0, length: int | None = None) -> int:
        """Enqueue stage 1 of buf[:length] into out (uint32/int32 tensor).  Returns the launch status."""
        assert buf.is_cuda and buf.dtype == torch.uint8 and buf.is_contiguous()
        assert out.is_cuda and out.element_size() == 4 and out.is_contiguous()
        n = buf.numel() if length is None else length
        return self._lib.sjb200_stage1_device_async(self._ctx, buf.data_ptr(), n, out.data_ptr(), out.numel(), flags)

    def finish(self) -> DeviceResult:
        n = C.c_uint32(0xFFFFFFFF)
        nw = C.c_uint32(0)
        u8 = C.c_int32(0)
        rc = self._lib.sjb200_stage1_finish(self._ctx, C.byref(n), C.byref(nw), C.byref(u8))
        return DeviceResult(rc, None if n.value == 0xFFFFFFFF else n.value, nw.value, u8.value)

    def index(self, buf: torch.Tensor, out: torch.Tensor, flags: int = 0, length: int | None = None) -> DeviceResult:
        rc = self.enqueue(buf, out, flags, length)
        if rc != errors.SUCCESS:
            return DeviceResult(rc, None, 0, 0)
        return self.finish()

    def structural_bytes(self, buf: torch.Tensor, idx: torch.Tensor, n: int, out: torch.Tensor | None = None) -> torch.Tensor:
        """out[k] = buf[idx[k]] for k < n (the byte each structural index points at), enqueued on the context's stream."""
        assert buf.is_cuda and buf.dtype == torch.uint8 and buf.is_contiguous()
        assert idx.is_cuda and idx.element_size() == 4 and idx.is_contiguous() and idx.numel() >= n
        if out is None:
            out = torch.empty(n, dtype=torch.uint8, device=buf.device)
        assert out.is_cuda and out.dtype == torch.uint8 and out.is_contiguous() and out.numel() >= n
        rc = self._lib.sjb200_structural_bytes_device_async(self._ctx, buf.data_ptr(), buf.numel(), idx.data_ptr(), n, out.data_ptr())
        if rc != errors.SUCCESS:
            raise RuntimeError(f"structural byte gather failed: {errors.NAMES.get(rc, rc)}")
        return out

    def document_starts(self, structural_bytes: torch.Tensor, n: int, out: torch.Tensor | None = None) -> torch.Tensor:
        """out[k] = 1 iff structural k opens a top-level document (bracket depth before it is 0); see the C header."""
        assert structural_bytes.is_cuda and structural_bytes.dtype == torch.uint8 and structural_bytes.numel() >= n
        if out is None:
            out = torch.empty(n, dtype=torch.uint8, device=structural_bytes.device)
        scratch = torch.empty(max(1, -(-n // 4096)), dtype=torch.int32, device=structural_bytes.device)
        rc = self._lib.sjb200_document_starts_device_async(self._ctx, structural_bytes.data_ptr(), n, out.data_ptr(),
                                                           scratch.data_ptr(), scratch.numel())
        if rc != errors.SUCCESS:
            raise RuntimeError(f"document start scan failed: {errors.NAMES.get(rc, rc)}")
        self._depth_scratch = scratch  # keep it alive until the stream has used it
        return out

    def stage2_primitives(self, buf: torch.Tensor, idx: torch.Tensor, n: int, want_strings: bool = True):
        """The per-primitive half of stage 2 over a stage-1 index array (include/simdjson_b200.h,
        sjb200_stage2_primitives_device_async).  Returns a dict of device tensors: kind, error (uint8 [n]), value (int64 [n]),
        str_off (int64 [n]), string_buf (uint8, the reference's {uint32 length, bytes} records; None unless want_strings),
        summary (int64 [4]: first failing primitive as k << 8 | error or -1, bytes of string records)."""
        assert buf.is_cuda and buf.dtype == torch.uint8 and buf.is_contiguous()
        assert idx.is_cuda and idx.element_size() == 4 and idx.is_contiguous() and idx.numel() >= n
        dev = buf.device
        kind = torch.empty(max(n, 1), dtype=torch.uint8, device=dev)
        err = torch.empty(max(n, 1), dtype=torch.uint8, device=dev)
        value = torch.empty(max(n, 1), dtype=torch.int64, device=dev)
        off = torch.empty(max(n, 1), dtype=torch.int64, device=dev)
        summary = torch.empty(4, dtype=torch.int64, device=dev)
        # every unescaped string is no longer than its source, and every string costs at least its two quotes: len + 2 n bounds the records
        cap = buf.numel() + 2 * n + 64 if want_strings else 0
        sbuf = torch.empty(cap, dtype=torch.uint8, device=dev) if want_strings else None
        rc = self._lib.sjb200_stage2_primitives_device_async(self._ctx, buf.data_ptr(), buf.numel(), idx.data_ptr(), n, kind.data_ptr(), err.data_ptr(),
                                                             value.data_ptr(), off.data_ptr(), sbuf.data_ptr() if want_strings else None, cap,
                                                             summary.data_ptr())
        if rc != errors.SUCCESS:
            raise RuntimeError(f"stage-2 primitives failed: {errors.NAMES.get(rc, rc)}")
        return {"kind": kind[:n], "error": err[:n], "value": value[:n], "str_off": off[:n], "string_buf": sbuf, "summary": summary}

    def stage2_tape(self, buf: torch.Tensor, idx: torch.Tensor, n: int, prims: dict):
        """The stage-2 walk over a stage-1 index array: verdict + tape (include/simdjson_b200.h, sjb200_stage2_tape_device_async).
        `prims` = the result of stage2_primitives for the same document.  Returns (tape int64 [2 n + 2] on the device, summary
        int64 [4] on the device: first error or -1, token words, tape length, inexact doubles)."""
        dev = buf.device
        tape = torch.zeros(2 * n + 2, dtype=torch.int64, device=dev)
        summary = torch.empty(4, dtype=torch.int64, device=dev)
        rc = self._lib.sjb200_stage2_tape_device_async(self._ctx, buf.data_ptr(), buf.numel(), idx.data_ptr(), n, prims["kind"].data_ptr(),
                                                       prims["error"].data_ptr(), prims["value"].data_ptr(), prims["str_off"].data_ptr(), tape.data_ptr(),
                                                       tape.numel(), summary.data_ptr())
        if rc != errors.SUCCESS:
            raise RuntimeError(f"stage-2 tape failed: {errors.NAMES.get(rc, rc)}")
        return tape, summary

    def stage2_stream(self, buf: torch.Tensor, idx: torch.Tensor, n: int, prims: dict, tape_capacity: int | None = None):
        """Stage 2 over a stream of documents (NDJSON or concatenated JSON; include/simdjson_b200.h,
        sjb200_stage2_stream_device_async): one verdict and one tape slice per document.  `prims` = the result of
        stage2_primitives for the same indexes; its string buffer is the one the string words point into.  Returns a dict of
        device tensors: tape (int64, 4 n words unless tape_capacity is given), doc_first (int32 [n_docs + 1]), doc_tape
        (int64 [n_docs + 1]), doc_status (int64 [n_docs], -1 = SUCCESS), summary (int64 [4]: documents, failing documents,
        tape length, inexact doubles).  Synchronises to learn n_docs."""
        dev = buf.device
        tape = torch.zeros(4 * n if tape_capacity is None else max(tape_capacity, 1), dtype=torch.int64, device=dev)
        first = torch.empty(n + 1, dtype=torch.int32, device=dev)
        doc_tape = torch.empty(n + 1, dtype=torch.int64, device=dev)
        status = torch.empty(max(n, 1), dtype=torch.int64, device=dev)
        summary = torch.empty(4, dtype=torch.int64, device=dev)
        rc = self._lib.sjb200_stage2_stream_device_async(self._ctx, buf.data_ptr(), buf.numel(), idx.data_ptr(), n, prims["kind"].data_ptr(),
                                                         prims["error"].data_ptr(), prims["value"].data_ptr(), prims["str_off"].data_ptr(),
                                                         tape.data_ptr(), tape.numel() if tape_capacity is None else tape_capacity,
                                                         first.data_ptr(), doc_tape.data_ptr(), status.data_ptr(), summary.data_ptr())
        if rc != errors.SUCCESS:
            raise RuntimeError(f"stage-2 stream walk failed: {errors.NAMES.get(rc, rc)}")
        nd = int(summary[0].item())
        return {"tape": tape, "doc_first": first[: nd + 1], "doc_tape": doc_tape[: nd + 1], "doc_status": status[:nd], "summary": summary}

    def at_pointers(self, pointers, tape: torch.Tensor, string_buf: torch.Tensor, doc_tape: torch.Tensor, doc_status: torch.Tensor) -> PointerColumns:
        """JSON Pointer lookups (RFC 6901) on device tapes, one column per pointer over every document (include/simdjson_b200.h,
        sjb200_at_pointers_device_async, for the rules).  `pointers`: str or bytes.  Enqueued on the context's stream; the
        tape stays on the device.  Over a stream of documents:

            prims = ctx.stage2_primitives(buf, idx, n)
            s = ctx.stage2_stream(buf, idx, n, prims)
            cols = ctx.at_pointers(["/user/id", "/text"], s["tape"], prims["string_buf"], s["doc_tape"], s["doc_status"])
            ids, found = cols.int64(0)

        Over one document (D = 1):

            tape, summary = ctx.stage2_tape(buf, idx, n, prims)
            doc_tape = torch.stack([torch.zeros_like(summary[2]), summary[2]])
            cols = ctx.at_pointers(["/a/0"], tape, prims["string_buf"], doc_tape, summary[:1])

        The whole `tape` and `string_buf` tensors bound the reads.  Raises ValueError for an invalid pointer or one over the
        limits (SJB200_POINTER_MAX_COUNT, SJB200_POINTER_MAX_BYTES)."""
        for t, dt in ((tape, torch.int64), (doc_tape, torch.int64), (doc_status, torch.int64), (string_buf, torch.uint8)):
            assert t.is_cuda and t.dtype == dt and t.is_contiguous()
        n_docs = doc_status.numel()
        assert doc_tape.numel() >= n_docs + 1
        raw, offs = pointer_program(pointers)
        k = len(offs) - 1
        dev = tape.device
        cols = PointerColumns(torch.zeros((k, n_docs), dtype=torch.uint8, device=dev), torch.zeros((k, n_docs), dtype=torch.uint8, device=dev),
                              torch.zeros((k, n_docs), dtype=torch.int64, device=dev))
        rc = self._lib.sjb200_at_pointers_device_async(self._ctx, tape.data_ptr(), tape.numel(), string_buf.data_ptr(), string_buf.numel(),
                                                       doc_tape.data_ptr(), doc_status.data_ptr(), n_docs, raw, offs, k, cols.type.data_ptr(),
                                                       cols.code.data_ptr(), cols.value.data_ptr())
        if rc in (errors.INVALID_JSON_POINTER, errors.CAPACITY):
            raise ValueError(f"pointer lookup refused: {errors.NAMES[rc]}")
        if rc != errors.SUCCESS:
            raise RuntimeError(f"pointer lookup failed: {errors.NAMES.get(rc, rc)}")
        return cols

    def string_columns(self, cols: PointerColumns, string_buf: torch.Tensor) -> StringColumns:
        """The string cells of pointer columns as device string columns, offsets + bytes (include/simdjson_b200.h,
        sjb200_string_columns_device_async).  `string_buf` is the buffer the cells point into.  The whole chain stays on the
        device:

            prims = ctx.stage2_primitives(buf, idx, n)
            s = ctx.stage2_stream(buf, idx, n, prims)
            cols = ctx.at_pointers(["/text", "/lang"], s["tape"], prims["string_buf"], s["doc_tape"], s["doc_status"])
            strs = ctx.string_columns(cols, prims["string_buf"])
            offsets, data, mask = strs.column(0)

        Synchronises once to learn the total size: the offsets are computed first without the data, then the bytes are
        gathered into a buffer of exactly that size.  Raises RuntimeError if a string cell's record lies outside
        `string_buf` (cells at_pointers wrote over the same buffer never do)."""
        assert string_buf.is_cuda and string_buf.dtype == torch.uint8 and string_buf.is_contiguous()
        assert cols.type.is_contiguous() and cols.value.is_contiguous() and cols.type.shape == cols.value.shape
        k, d = cols.type.shape
        dev = cols.type.device
        offsets = torch.empty(k * d + 1, dtype=torch.int64, device=dev)
        summary = torch.empty(2, dtype=torch.int64, device=dev)

        def call(data: torch.Tensor | None) -> None:
            rc = self._lib.sjb200_string_columns_device_async(self._ctx, cols.type.data_ptr(), cols.value.data_ptr(), k, d, string_buf.data_ptr(),
                                                              string_buf.numel(), offsets.data_ptr(), None if data is None else data.data_ptr(),
                                                              0 if data is None else data.numel(), summary.data_ptr())
            if rc != errors.SUCCESS:
                raise RuntimeError(f"string columns failed: {errors.NAMES.get(rc, rc)}")

        call(None)
        total, bad = summary.tolist()
        if bad:
            raise RuntimeError(f"string columns: {bad} string cells point outside the string buffer")
        bounds = offsets[::d].tolist() if d else [0] * (k + 1)
        data = torch.empty(total, dtype=torch.uint8, device=dev)
        if total:
            call(data)
        return StringColumns(offsets, data, cols.type == ord('"'), bounds)

    def last_elapsed_ms(self) -> float:
        return float(self._lib.sjb200_last_elapsed_ms(self._ctx))

    def launch_count(self) -> int:
        return int(self._lib.sjb200_launch_count(self._ctx))

    def sync(self) -> None:
        self._lib.sjb200_sync(self._ctx)

    # -- NDJSON batches --------------------------------------------------------------------------
    def split(self, buf: torch.Tensor, seg_bytes: int, max_segments: int = 4096) -> list[int]:
        assert buf.is_cuda and buf.dtype == torch.uint8 and buf.is_contiguous()
        offs = (C.c_uint64 * (max_segments + 1))()
        nseg = C.c_uint32(0)
        rc = self._lib.sjb200_batch_split_device(self._ctx, buf.data_ptr(), buf.numel(), seg_bytes, offs, max_segments,
                                                 C.byref(nseg))
        if rc != errors.SUCCESS:
            raise RuntimeError(f"batch split failed: {errors.NAMES.get(rc, rc)}")
        return [int(offs[i]) for i in range(nseg.value + 1)]

    def run_segments(self, buf: torch.Tensor, seg_offsets: list[int], out: torch.Tensor, flags: int = 0,
                     first: int = 0, count: int | None = None):
        """Index segments [first, first+count) back to back.  Segment s writes at out[idx_offsets[s]:]."""
        nseg = len(seg_offsets) - 1
        if count is None:
            count = nseg - first
        offs = (C.c_uint64 * (nseg + 1))(*seg_offsets)
        idx_offsets = [0] * (nseg + 1)
        for s in range(first, first + count):
            idx_offsets[s + 1] = idx_offsets[s] + (seg_offsets[s + 1] - seg_offsets[s]) + 3
        ioffs = (C.c_uint64 * (nseg + 1))(*idx_offsets)
        counts = (C.c_uint32 * nseg)()
        errs = (C.c_int32 * nseg)()
        u8 = (C.c_int32 * nseg)()
        worst = self._lib.sjb200_batch_run_device(self._ctx, buf.data_ptr(), offs, first, count, out.data_ptr(), ioffs,
                                                  out.numel(), counts, errs, u8, flags)
        sl = slice(first, first + count)
        return worst, list(counts)[sl], list(errs)[sl], list(u8)[sl], idx_offsets[first:first + count + 1]

    def run_segments_async(self, buf: torch.Tensor, seg_offsets: list[int], out: torch.Tensor, status: torch.Tensor,
                           flags: int = 0) -> int:
        """Enqueue every segment without waiting; segment s leaves (error, n) at status[s] (int32 [nseg, 2], device)."""
        nseg = len(seg_offsets) - 1
        assert status.is_cuda and status.dtype == torch.int32 and status.numel() >= 2 * nseg and status.is_contiguous()
        key = (tuple(seg_offsets), out.numel())
        cached = getattr(self, "_seg_cache", None)
        if cached is None or cached[0] != key:
            offs = (C.c_uint64 * (nseg + 1))(*seg_offsets)
            idx_offsets = [0] * (nseg + 1)
            for s in range(nseg):
                idx_offsets[s + 1] = idx_offsets[s] + (seg_offsets[s + 1] - seg_offsets[s]) + 3
            ioffs = (C.c_uint64 * (nseg + 1))(*idx_offsets)
            self._seg_cache = (key, offs, ioffs, idx_offsets)
        _, offs, ioffs, _ = self._seg_cache
        return self._lib.sjb200_batch_run_device_async(self._ctx, buf.data_ptr(), offs, 0, nseg, out.data_ptr(), ioffs,
                                                       out.numel(), status.data_ptr(), flags)
