"""Host-side mirror of the reference's parser facade.

Reference: src/mojo_simdjson/include/generic/dom_parser_implementation.mojo:15-89.  Same field names, same
calls (`stage1(buffer) -> ErrorType`, `stage2() -> ErrorType`), same error behaviour; the line that called
JsonStructuralIndexer.index[128] (:69) calls libsimdjson_b200.so instead, and so does the one that called
TapeBuilder.parse_document (:83).  A consumer that walks the index array itself reads `buf`, `length`,
`structural_indexes[0 .. n+2]`, `n_structural_indexes` and `next_structural_index` exactly as the reference's
JsonIterator does (json_iterator.mojo:28-38,256-288).
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _native, errors

DEFAULT_MAX_LEN = 64 << 20

JSON_VALUE_MASK = (1 << 56) - 1


class Document:
    """The reference's Document (include/dom/document.mojo:13-19): a tape and a string buffer."""

    def __init__(self):
        self.tape = np.zeros(0, dtype=np.uint64)
        self.string_buf = np.zeros(0, dtype=np.uint8)
        self.inexact_doubles = 0      # doubles outside the exact decimal -> binary fast path (not in the reference)

    def string_at(self, offset: int) -> bytes:
        n = int.from_bytes(self.string_buf[offset : offset + 4].tobytes(), "little")
        return self.string_buf[offset + 4 : offset + 4 + n].tobytes()

    def dump_raw_tape(self):
        """The listing of include/dom/document.mojo:48-162, one line per tape word.  Returns (text, ok)."""
        t = [int(x) for x in self.tape]
        if not t or t[0] >> 56 != ord("r"):
            return "", False
        how_many = t[0] & JSON_VALUE_MASK
        out = [f"0 : r\t// pointing to {how_many} (right after last node)"]
        i = 1
        while i < how_many - 1:
            ty, payload = chr(t[i] >> 56), t[i] & JSON_VALUE_MASK
            if ty == '"':
                out.append(f'{i} : string "{self.string_at(payload).decode("utf-8", "replace")}"')
            elif ty == "l":
                v = t[i + 1]
                out.append(f"{i} : integer {v - (1 << 64) if v >> 63 else v}")
                i += 1
            elif ty == "d":
                out.append(f"{i} : float {float(np.array([t[i + 1]], dtype=np.uint64).view(np.float64)[0])}")
                i += 1
            elif ty in "tfn":
                out.append(f"{i} : {dict(t='true', f='false', n='null')[ty]}")
            elif ty in "{[":
                out.append(f"{i} : {ty}\t// pointing to next tape location {payload & 0xFFFFFFFF} (first node after the scope),  saturated count "
                           f"{(payload >> 32) & 0xFFFFFF}")
            elif ty in "}]":
                out.append(f"{i} : {ty}\t// pointing to previous tape location {payload & 0xFFFFFFFF} (start of the scope)")
            else:
                return "\n".join(out), False
            i += 1
        out.append(f"{how_many - 1} : r\t// pointing to {t[how_many - 1] & JSON_VALUE_MASK} (start root)")
        return "\n".join(out) + "\n", True


class DocumentStream:
    """The documents of one stream (NDJSON or concatenated JSON) after DomParserImplementation.stage2_stream(): one tape with
    a slice per document, one string buffer, one verdict per document (include/simdjson_b200.h, sjb200_stage2_stream)."""

    def __init__(self, tape, string_buf, doc_first, doc_tape, doc_status, n_failed: int, inexact_doubles: int):
        self.tape = tape                    # uint64, every document's slice back to back
        self.string_buf = string_buf        # uint8, the records every slice's string words point into
        self.doc_first = doc_first          # uint32 [len + 1]: first structural of every document
        self.doc_tape = doc_tape            # uint64 [len + 1]: where every document's slice starts
        self.doc_status = doc_status        # uint64 [len]: all ones = SUCCESS, else k << 16 | check << 8 | code
        self.n_failed = n_failed
        self.inexact_doubles = inexact_doubles

    def __len__(self) -> int:
        return int(self.doc_status.size)

    def error(self, d: int) -> int:
        """The error code of document d (0 = SUCCESS)."""
        s = int(self.doc_status[d])
        return 0 if s == (1 << 64) - 1 else s & 0xFF

    def document(self, d: int) -> Document:
        """Document d as a Document: a view of its tape slice and the stream's string buffer.  Meaningful when error(d) == 0."""
        doc = Document()
        doc.tape = self.tape[int(self.doc_tape[d]) : int(self.doc_tape[d + 1])]
        doc.string_buf = self.string_buf
        return doc


class PointerCells:
    """The result of DomParserImplementation.at_pointers(): K columns of D cells as numpy arrays [K, D] (include/simdjson_b200.h,
    sjb200_stage2_stream_at_pointers), and the stream's string buffer that string cells point into."""

    def __init__(self, type_, code, value, string_buf):
        self.type = type_           # uint8: the tape type character of the value found, 0 if not found
        self.code = code            # uint8: 0 = found, else the simdjson error code
        self.value = value          # int64: integer, double bits, 1/0 for true/false/null, string record offset, container index
        self.string_buf = string_buf

    def strings(self, k: int) -> list:
        """Column k as bytes for string cells, None for every other cell."""
        sb = self.string_buf
        out = []
        for t, off in zip(self.type[k].tolist(), self.value[k].tolist()):
            if t == ord('"'):
                n = int.from_bytes(sb[off : off + 4].tobytes(), "little")
                out.append(sb[off + 4 : off + 4 + n].tobytes())
            else:
                out.append(None)
        return out


class DomParserImplementation:
    """Stage-1 half of the reference's DomParserImplementation, backed by the B200 kernel."""

    def __init__(self, device: int = 0, max_len: int = DEFAULT_MAX_LEN, validate_utf8: bool = False, chunk_bytes: int | None = None):
        self._lib = _native.lib()
        if self._lib.sjb200_device_count() <= 0:
            raise RuntimeError("no CUDA device: the stage-1 path has no CPU fallback")
        self.buf: np.ndarray | None = None          # buffer passed to stage 1 (kept alive for stage 2)
        self.length = 0
        self.n_structural_indexes = 0
        self.structural_indexes = np.zeros(0, dtype=np.uint32)
        self.next_structural_index = 0
        self.document = Document()
        self.stream: DocumentStream | None = None    # stage2_stream()'s result
        self.pointer_cells: PointerCells | None = None   # at_pointers()'s result
        self.utf8_error = 0                          # not in the reference: its Utf8Checker is a stub
        self._capacity = 0
        self._max_depth = 100
        self._max_len = max_len
        self._flags = _native.FLAG_VALIDATE_UTF8 if validate_utf8 else 0
        self._ctx = C.c_void_p()
        rc = self._lib.sjb200_ctx_create(device, max_len, max_len, 0, C.byref(self._ctx))
        if rc != errors.SUCCESS:
            raise RuntimeError(f"sjb200_ctx_create failed: {errors.NAMES.get(rc, rc)}")
        if chunk_bytes is not None and self._lib.sjb200_ctx_set_chunk_bytes(self._ctx, chunk_bytes) != errors.SUCCESS:
            raise ValueError("chunk_bytes must be >= 4096")

    def close(self):
        if getattr(self, "_ctx", None) is not None and self._ctx:
            self._lib.sjb200_ctx_destroy(self._ctx)
            self._ctx = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def max_depth(self) -> int:
        return self._max_depth

    def capacity(self) -> int:
        return self._capacity

    def allocate(self, amount: int) -> None:
        # reference :85-89 resizes to `amount` entries and then writes the 3-entry trailer past the end;
        # we allocate the 3 extra entries the trailer needs
        if self.structural_indexes.size < amount + 3:
            self.structural_indexes = np.zeros(amount + 3, dtype=np.uint32)
        self._capacity = amount

    def stage1(self, buffer) -> int:
        """reference :59-69 -- accepts str / bytes / uint8 ndarray, returns the error code."""
        if isinstance(buffer, str):
            buffer = buffer.encode("utf-8")
        if isinstance(buffer, (bytes, bytearray, memoryview)):
            buffer = np.frombuffer(bytes(buffer), dtype=np.uint8)
        buffer = np.ascontiguousarray(buffer, dtype=np.uint8)
        n_bytes = int(buffer.size)
        if n_bytes > self._max_len:     # before allocate(): an oversize input must not cost 4 * len bytes of host memory first
            return errors.CAPACITY
        self.allocate(n_bytes)
        self.buf = buffer
        self.length = n_bytes
        n = C.c_uint32(self.n_structural_indexes)
        u8 = C.c_int32(0)
        rc = self._lib.sjb200_stage1(self._ctx, buffer.ctypes.data if n_bytes else None, n_bytes,
                                     self.structural_indexes.ctypes.data, self.structural_indexes.size,
                                     C.byref(n), C.byref(u8), self._flags)
        self.utf8_error = int(u8.value)
        if rc in (errors.SUCCESS, errors.EMPTY, errors.UTF8_ERROR) and n_bytes:
            # the reference assigns these only past its early returns (json_structural_indexer.mojo:160-174)
            self.n_structural_indexes = int(n.value)
            self.next_structural_index = 0
        return rc

    def stage2(self) -> int:
        """reference :71-83 -- sizes the document's tape and string buffer, walks the structurals.  The walk runs on the
        device over the copy of the document that stage1() left there; returns the error code."""
        n, length = int(self.n_structural_indexes), int(self.length)
        if self.buf is None or n == 0:
            return errors.UNINITIALIZED
        tape = np.zeros(2 * n + 2, dtype=np.uint64)
        sbuf = np.zeros(length + 2 * n + 64, dtype=np.uint8)
        tl, sl, inexact = C.c_uint64(0), C.c_uint64(0), C.c_uint64(0)
        rc = self._lib.sjb200_stage2(self._ctx, tape.ctypes.data, tape.size, sbuf.ctypes.data, sbuf.size, C.byref(tl), C.byref(sl), C.byref(inexact))
        if rc == errors.SUCCESS:
            self.document.tape = tape[: tl.value]
            self.document.string_buf = sbuf[: sl.value]
            self.document.inexact_doubles = int(inexact.value)
        return rc

    def stage2_stream(self) -> int:
        """Stage 2 over a stream of documents (NDJSON or concatenated JSON) that stage1() indexed: one verdict and one tape
        slice per document, in `self.stream` (a DocumentStream).  Returns the call's code: SUCCESS when the outputs were
        delivered, also when documents fail; the documents' verdicts are in self.stream."""
        n, length = int(self.n_structural_indexes), int(self.length)
        if self.buf is None or n == 0:
            return errors.UNINITIALIZED
        tape = np.zeros(4 * n, dtype=np.uint64)
        sbuf = np.zeros(length + 2 * n + 64, dtype=np.uint8)
        first = np.zeros(n + 1, dtype=np.uint32)
        doc_tape = np.zeros(n + 1, dtype=np.uint64)
        status = np.zeros(n, dtype=np.uint64)
        nd, nf, tl, sl, inexact = (C.c_uint64(0) for _ in range(5))
        rc = self._lib.sjb200_stage2_stream(self._ctx, tape.ctypes.data, tape.size, sbuf.ctypes.data, sbuf.size, first.ctypes.data, doc_tape.ctypes.data,
                                            status.ctypes.data, n, C.byref(nd), C.byref(nf), C.byref(tl), C.byref(sl), C.byref(inexact))
        if rc == errors.SUCCESS:
            d = int(nd.value)
            self.stream = DocumentStream(tape[: tl.value], sbuf[: sl.value], first[: d + 1], doc_tape[: d + 1], status[:d], int(nf.value), int(inexact.value))
        return rc

    def at_pointers(self, pointers) -> int:
        """JSON Pointer lookups over every document of the stream stage1() indexed (include/simdjson_b200.h for the rules): the
        walk and the lookups run on the device and only the cells and the string buffer come back, into `self.pointer_cells`
        (a PointerCells).  `pointers`: str or bytes.  Returns the call's code: SUCCESS also when cells hold errors;
        INVALID_JSON_POINTER or CAPACITY for pointers the call refuses."""
        from .device import pointer_program

        n, length = int(self.n_structural_indexes), int(self.length)
        if self.buf is None or n == 0:
            return errors.UNINITIALIZED
        raw, offs = pointer_program(pointers)
        k = len(offs) - 1
        docs = int(np.count_nonzero(self.buf == 0x0A)) + 1    # a first guess; the call reports the real count
        sb_cap = length + 2 * n + 64
        nd, sl = C.c_uint64(0), C.c_uint64(0)
        for _ in range(2):
            cells = max(k * docs, 1)
            ty, code, val = np.zeros(cells, np.uint8), np.zeros(cells, np.uint8), np.zeros(cells, np.int64)
            sbuf = np.zeros(sb_cap, dtype=np.uint8)
            rc = self._lib.sjb200_stage2_stream_at_pointers(self._ctx, raw, offs, k, ty.ctypes.data, code.ctypes.data, val.ctypes.data, cells,
                                                            sbuf.ctypes.data, sbuf.size, C.byref(nd), C.byref(sl))
            if rc != errors.CAPACITY or k * int(nd.value) <= cells and int(sl.value) <= sb_cap:
                break
            docs, sb_cap = int(nd.value), int(sl.value)
        if rc == errors.SUCCESS:
            d = int(nd.value)
            self.pointer_cells = PointerCells(ty[: k * d].reshape(k, d), code[: k * d].reshape(k, d), val[: k * d].reshape(k, d), sbuf[: sl.value])
        return rc
