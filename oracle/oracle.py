"""ctypes wrapper around oracle/liboracle_stage1.so.

TEST INFRASTRUCTURE, NOT PRODUCT CODE: only tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / --impl reference legs import this module.  The product path
(mojo_simdjson_b200) never does.
"""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile
from dataclasses import dataclass

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))

SUCCESS, CAPACITY, UTF8_ERROR, EMPTY, UNESCAPED_CHARS, UNCLOSED_STRING, UNEXPECTED_ERROR = 0, 1, 11, 13, 14, 15, 24
FLAG_VALIDATE_UTF8 = 1


def _cpu_signature() -> str:
    """The host's CPU feature flags: a -march=native build must not be carried to a machine with different ones."""
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.startswith("flags"):
                    return hashlib.sha1(line.encode()).hexdigest()
    except OSError:
        pass
    return "unknown"


def _build_native(src: str) -> str:
    """The -march=native build goes to a per-user temporary directory, never into the tree: bench.py must run from a
    read-only checkout, and a build for one CPU must not travel with the tree to another.  The file name carries a digest
    of the source, the Makefile and the CPU's feature flags, so a different checkout or host never picks up a stale build."""
    h = hashlib.sha1(_cpu_signature().encode())
    for p in (src, os.path.join(_HERE, "Makefile")):
        with open(p, "rb") as f:
            h.update(f.read())
    d = os.path.join(tempfile.gettempdir(), f"sjb200-oracle-{os.getuid()}")
    path = os.path.join(d, f"liboracle_stage1_native-{h.hexdigest()[:16]}.so")
    if not os.path.exists(path):
        os.makedirs(d, mode=0o700, exist_ok=True)
        tmp = f"{path}.{os.getpid()}.tmp"   # concurrent ranks each build their own, then rename atomically
        subprocess.check_call(["make", "-s", "-C", _HERE, f"NATIVE_OUT={tmp}", tmp])
        os.replace(tmp, path)
    return path


def build(native: bool = False) -> str:
    src = os.path.join(_HERE, "stage1_oracle.c")
    if native:
        return _build_native(src)
    path = os.path.join(_HERE, "liboracle_stage1.so")
    if not os.path.exists(path) or os.path.getmtime(path) < os.path.getmtime(src):
        if os.path.exists(path):
            os.remove(path)
        subprocess.check_call(["make", "-s", "-C", _HERE, "liboracle_stage1.so"])
    return path


_libs: dict[bool, C.CDLL] = {}


def lib(native: bool = False) -> C.CDLL:
    if native not in _libs:
        L = C.CDLL(build(native))
        u8p, u32p, u64p, i32p = C.c_void_p, C.c_void_p, C.POINTER(C.c_uint64), C.POINTER(C.c_int32)
        for name in ("oracle_stage1_ref", "oracle_stage1_spec"):
            f = getattr(L, name)
            f.restype = C.c_int32
            f.argtypes = [u8p, C.c_uint64, u32p, C.c_uint64, C.POINTER(C.c_uint32), u64p, i32p, C.c_uint32]
        L.oracle_stage1_fast.restype = C.c_int32
        L.oracle_stage1_fast.argtypes = [u8p, C.c_uint64, u32p, C.c_uint64, C.POINTER(C.c_uint32), u64p, C.c_uint32]
        L.oracle_stage1_ref_trace.restype = C.c_int32
        L.oracle_stage1_ref_trace.argtypes = [u8p, C.c_uint64, u32p, C.c_uint64, C.POINTER(C.c_uint32), C.c_char_p]
        for name in ("oracle_utf8_valid_dfa", "oracle_utf8_valid_kl"):
            f = getattr(L, name)
            f.restype = C.c_int32
            f.argtypes = [u8p, C.c_uint64]
        L.oracle_index_digest.restype = None
        L.oracle_index_digest.argtypes = [u32p, C.c_uint64, u64p, u64p]
        L.oracle_set_shuffle_variant.restype = None
        L.oracle_set_shuffle_variant.argtypes = [C.c_int]
        _libs[native] = L
    return _libs[native]


@dataclass
class Stage1Result:
    error: int
    n: int | None          # n_structural_indexes as the reference would have assigned it (None: not assigned)
    n_written: int         # entries the indexer wrote (also on the early-return error paths)
    indexes: np.ndarray    # uint32, n_written entries (+3 trailer entries when the trailer was written)
    utf8_error: int        # 1 iff the input is not valid UTF-8 (always computed)
    trailer_written: bool


def _as_u8(data) -> np.ndarray:
    if isinstance(data, np.ndarray):
        assert data.dtype == np.uint8
        return np.ascontiguousarray(data)
    if isinstance(data, str):
        data = data.encode("utf-8")
    return np.frombuffer(bytes(data), dtype=np.uint8)


def stage1(data, flags: int = 0, impl: str = "ref", cap: int | None = None, native: bool = False) -> Stage1Result:
    """Run the oracle.  impl: 'ref' (block restatement), 'spec' (per-byte closed form), 'fast'."""
    L = lib(native)
    a = _as_u8(data)
    n_bytes = int(a.size)
    if cap is None:
        cap = n_bytes + 3
    out = np.full(max(cap, 1), 0xDEADBEEF, dtype=np.uint32)
    n = C.c_uint32(0xFFFFFFFF)
    nw = C.c_uint64(0)
    u8 = C.c_int32(0)
    ptr = a.ctypes.data if n_bytes else None
    if impl == "fast":
        err = L.oracle_stage1_fast(ptr, n_bytes, out.ctypes.data, cap, C.byref(n), C.byref(nw), flags)
        u8.value = 0 if L.oracle_utf8_valid_dfa(ptr, n_bytes) else 1
        if (flags & 1) and err == SUCCESS and u8.value:
            err = UTF8_ERROR  # same priority slot as oracle_stage1_ref: only a would-be SUCCESS turns into UTF8_ERROR
    else:
        f = L.oracle_stage1_ref if impl == "ref" else L.oracle_stage1_spec
        err = f(ptr, n_bytes, out.ctypes.data, cap, C.byref(n), C.byref(nw), C.byref(u8), flags)
    assigned = n.value != 0xFFFFFFFF
    trailer = assigned
    count = int(nw.value)
    keep = min(count + (3 if trailer else 0), cap)
    return Stage1Result(err, n.value if assigned else None, count, out[:keep].copy(), int(u8.value), trailer)


_simd = None


def simd_lib() -> C.CDLL:
    """liboracle_stage1_simd.so: the AVX-512 / AVX2 "cpu_simd" baseline (oracle/stage1_simd.c)."""
    global _simd
    if _simd is None:
        path = os.path.join(_HERE, "liboracle_stage1_simd.so")
        src = os.path.join(_HERE, "stage1_simd.c")
        if not os.path.exists(path) or os.path.getmtime(path) < os.path.getmtime(src):
            subprocess.check_call(["make", "-s", "-C", _HERE, "liboracle_stage1_simd.so"])
        L = C.CDLL(path)
        L.simd_stage1_level.restype = C.c_int
        L.simd_stage1_level.argtypes = []
        L.simd_stage1.restype = C.c_int32
        L.simd_stage1.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint32), C.POINTER(C.c_uint64),
                                  C.POINTER(C.c_int32), C.c_uint32, C.c_int]
        _simd = L
    return _simd


def simd_level() -> int:
    """2 = AVX-512 + pclmulqdq, 1 = AVX2 + pclmulqdq, 0 = this CPU has neither."""
    return int(simd_lib().simd_stage1_level())


def stage1_simd(data, flags: int = 0, cap: int | None = None, level: int = 0) -> Stage1Result:
    """The cpu_simd baseline with the oracle's result shape (tests compare it with the oracle bit for bit)."""
    L = simd_lib()
    a = _as_u8(data)
    n_bytes = int(a.size)
    if cap is None:
        cap = n_bytes + 3 + 8
    out = np.full(max(cap, 1), 0xDEADBEEF, dtype=np.uint32)
    n = C.c_uint32(0xFFFFFFFF)
    nw = C.c_uint64(0)
    u8 = C.c_int32(0)
    err = L.simd_stage1(a.ctypes.data if n_bytes else None, n_bytes, out.ctypes.data, cap, C.byref(n), C.byref(nw), C.byref(u8), flags, level)
    if err < 0:
        raise RuntimeError("this CPU has neither AVX-512 nor AVX2 with pclmulqdq")
    assigned = n.value != 0xFFFFFFFF
    count = int(nw.value)
    keep = min(count + (3 if assigned else 0), cap)
    return Stage1Result(err, n.value if assigned else None, count, out[:keep].copy(), int(u8.value), assigned)


def utf8_valid(data, impl: str = "dfa") -> bool:
    L = lib()
    a = _as_u8(data)
    f = L.oracle_utf8_valid_dfa if impl == "dfa" else L.oracle_utf8_valid_kl
    return bool(f(a.ctypes.data if a.size else None, int(a.size)))


def index_digest(idx: np.ndarray) -> tuple[int, int]:
    L = lib()
    a = np.ascontiguousarray(idx, dtype=np.uint32)
    d0, d1 = C.c_uint64(0), C.c_uint64(0)
    L.oracle_index_digest(a.ctypes.data if a.size else None, int(a.size), C.byref(d0), C.byref(d1))
    return d0.value, d1.value


def structural_bytes(data, indexes) -> np.ndarray:
    """Side output for stage 2 (SURVEY.md section 8(f) rank 2): the byte each structural index points at.

    Restates what the reference's stage-2 walk reads at every step, `self.buf[self.next_structural[0]]` and its
    `peek` variants (generic/stage2/json_iterator.mojo:256-262, :28-38): out[k] = data[indexes[k]]; an index at or
    beyond len(data) -- the trailer entries are -- reads as 0 (the reference's buffer is zero padded there)."""
    a = _as_u8(data)
    idx = np.asarray(indexes, dtype=np.uint32).astype(np.int64)
    out = np.zeros(idx.size, dtype=np.uint8)
    ok = idx < a.size
    out[ok] = a[idx[ok]]
    return out


def document_starts(structural_byte_values) -> np.ndarray:
    """Side output for stage 2 (SURVEY.md section 8(f) rank 2): out[k] = 1 iff structural k opens a top-level document,
    i.e. the bracket depth over the structural bytes before it is 0.  The reference has no document-stream mode
    (generic/stage2/tape_builder.mojo:25 "TODO: add streaming"); the depth bookkeeping restated here is the one its
    stage-2 walk does one container at a time (generic/stage2/json_iterator.mojo:40-254: depth += 1 at '{' / '[',
    depth -= 1 at '}' / ']', a document is finished when depth returns to 0)."""
    b = np.asarray(structural_byte_values, dtype=np.uint8)
    step = np.zeros(b.size, dtype=np.int64)
    step[(b == ord("{")) | (b == ord("["))] = 1
    step[(b == ord("}")) | (b == ord("]"))] = -1
    before = np.cumsum(step) - step
    return (before == 0).astype(np.uint8)


# ------------------------------------------------------------------------------------------------
# stage 2, per-primitive half (oracle/stage2_oracle.c): strings, atoms, numbers
# ------------------------------------------------------------------------------------------------
TAPE_ERROR, STRING_ERROR, T_ATOM_ERROR, F_ATOM_ERROR, N_ATOM_ERROR, NUMBER_ERROR = 3, 5, 6, 7, 8, 9
KIND_NONE, KIND_STRING, KIND_INT, KIND_FLOAT, KIND_TRUE, KIND_FALSE, KIND_NULL, KIND_BAD = range(8)

_stage2 = None


def stage2_lib() -> C.CDLL:
    global _stage2
    if _stage2 is None:
        path = os.path.join(_HERE, "liboracle_stage2.so")
        src = os.path.join(_HERE, "stage2_oracle.c")
        if not os.path.exists(path) or os.path.getmtime(path) < os.path.getmtime(src):
            subprocess.check_call(["make", "-s", "-C", _HERE, "liboracle_stage2.so"])
        L = C.CDLL(path)
        L.oracle_parse_string.restype = C.c_int64
        L.oracle_parse_string.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_void_p, C.c_uint32, C.POINTER(C.c_uint64)]
        for name in ("oracle_is_valid_true_atom", "oracle_is_valid_false_atom", "oracle_is_valid_null_atom"):
            f = getattr(L, name)
            f.restype = C.c_int32
            f.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64]
        L.oracle_parse_number.restype = C.c_int32
        L.oracle_parse_number.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.POINTER(C.c_int32), C.POINTER(C.c_int64), C.POINTER(C.c_uint32)]
        L.oracle_stage2_primitives.restype = C.c_int32
        L.oracle_stage2_primitives.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                               C.c_void_p, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.POINTER(C.c_int32)]
        L.oracle_stage2_walk.restype = C.c_int32
        L.oracle_stage2_walk.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64), C.c_void_p,
                                         C.POINTER(C.c_uint64)]
        _stage2 = L
    return _stage2


def parse_string(data, start: int, advance: int = 8):
    """parse_string of the reference (generic/stage2/string_parsing.mojo:334-386) on the bytes after an opening quote at
    data[start - 1].  Returns (unescaped bytes or None on STRING_ERROR, index of the closing quote).  advance = 32 restates
    BYTES_PROCESSED as written (see stage2_oracle.c); gaps it never copies stay zero, like the reference's zero-filled buffer."""
    L = stage2_lib()
    a = _as_u8(data)
    dst = np.zeros(a.size + 128, dtype=np.uint8)
    end = C.c_uint64(0)
    n = L.oracle_parse_string(a.ctypes.data, a.size, start, dst.ctypes.data, advance, C.byref(end))
    return (None, None) if n < 0 else (bytes(dst[:n]), int(end.value))


def parse_number(data, start: int = 0):
    """(error, is_float, integer value, token length) of number_parsing.mojo:22-80 at data[start]."""
    L = stage2_lib()
    a = _as_u8(data)
    isf, iv, tl = C.c_int32(0), C.c_int64(0), C.c_uint32(0)
    err = L.oracle_parse_number(a.ctypes.data, a.size, start, C.byref(isf), C.byref(iv), C.byref(tl))
    return int(err), bool(isf.value), int(iv.value), int(tl.value)


def atom_valid(data, start: int, which: str) -> bool:
    L = stage2_lib()
    a = _as_u8(data)
    f = {"true": L.oracle_is_valid_true_atom, "false": L.oracle_is_valid_false_atom, "null": L.oracle_is_valid_null_atom}[which]
    return bool(f(a.ctypes.data, a.size, start))


@dataclass
class Stage2Primitives:
    kind: np.ndarray        # uint8 [n]   KIND_*
    error: np.ndarray       # uint8 [n]   simdjson error code of that primitive (0 = fine)
    value: np.ndarray       # int64 [n]   strings: unescaped length; integers: value; floats: token length
    str_off: np.ndarray     # uint64 [n]  strings: offset of the record (uint32 length + bytes) in string_buf
    string_buf: np.ndarray  # uint8
    first_error_index: int  # n if none
    first_error: int


def stage2_primitives(data, indexes) -> Stage2Primitives:
    """Every structural of a stage-1 index array as the reference's visit_primitive would treat it (stage2_oracle.c)."""
    L = stage2_lib()
    a = _as_u8(data)
    idx = np.ascontiguousarray(indexes, dtype=np.uint32)
    n = int(idx.size)
    kind = np.zeros(max(n, 1), dtype=np.uint8)
    err = np.zeros(max(n, 1), dtype=np.uint8)
    val = np.zeros(max(n, 1), dtype=np.int64)
    off = np.zeros(max(n, 1), dtype=np.uint64)
    sbuf = np.zeros(a.size + 4 * n + 64, dtype=np.uint8)
    slen, fei, fe = C.c_uint64(0), C.c_uint64(0), C.c_int32(0)
    L.oracle_stage2_primitives(a.ctypes.data if a.size else None, a.size, idx.ctypes.data if n else None, n, kind.ctypes.data, err.ctypes.data,
                               val.ctypes.data, off.ctypes.data, sbuf.ctypes.data, C.byref(slen), C.byref(fei), C.byref(fe))
    return Stage2Primitives(kind[:n], err[:n], val[:n], off[:n], sbuf[: slen.value].copy(), int(fei.value), int(fe.value))


DEPTH_ERROR = 4


@dataclass
class Stage2Tape:
    error: int              # what walk_document returns (generic/stage2/json_iterator.mojo:40-254)
    tape: np.ndarray        # uint64, the words appended until the walk returned
    string_buf: np.ndarray  # uint8, {uint32 length, bytes} records in walk order


def stage2_walk(data, indexes_with_trailer, n: int) -> Stage2Tape:
    """The reference's stage-2 walk over a stage-1 result (indexes incl. the 3-entry trailer), restated in stage2_oracle.c."""
    L = stage2_lib()
    a = _as_u8(data)
    idx = np.ascontiguousarray(indexes_with_trailer, dtype=np.uint32)
    assert idx.size >= n + 3
    tape = np.zeros(2 * n + 8, dtype=np.uint64)
    sbuf = np.zeros(a.size + 4 * n + 64, dtype=np.uint8)
    tl, sl = C.c_uint64(0), C.c_uint64(0)
    err = L.oracle_stage2_walk(a.ctypes.data if a.size else None, a.size, idx.ctypes.data, n, tape.ctypes.data, tape.size, C.byref(tl), sbuf.ctypes.data,
                               C.byref(sl))
    return Stage2Tape(int(err), tape[: min(int(tl.value), tape.size)].copy(), sbuf[: sl.value].copy())


def decode_tape(tape: np.ndarray, string_buf: np.ndarray):
    """The document a tape describes, as python objects (objects as lists of (key, value) pairs so that order and duplicate keys
    survive); checks the structure words on the way: start -> one past the matching end, end -> its start, counts, both roots."""
    t = [int(x) for x in tape]
    sb = bytes(string_buf)
    N = len(t)
    assert N >= 2 and t[0] >> 56 == ord("r") and (t[0] & ((1 << 56) - 1)) == N and t[N - 1] == ord("r") << 56

    def string_at(off):
        n = int.from_bytes(sb[off : off + 4], "little")
        return sb[off + 4 : off + 4 + n].decode("utf-8", "surrogatepass")

    def value(i):
        w = t[i]
        ty, payload = chr(w >> 56), w & ((1 << 56) - 1)
        if ty == '"':
            return string_at(payload), i + 1
        if ty == "l":
            v = t[i + 1]
            return (v - (1 << 64) if v >> 63 else v), i + 2
        if ty == "d":
            return float(np.array([t[i + 1]], dtype=np.uint64).view(np.float64)[0]), i + 2
        if ty in "tfn":
            return {"t": True, "f": False, "n": None}[ty], i + 1
        if ty in "[{":
            end_next, count = payload & 0xFFFFFFFF, (payload >> 32) & 0xFFFFFF
            close = "]" if ty == "[" else "}"
            assert t[end_next - 1] >> 56 == ord(close) and (t[end_next - 1] & ((1 << 56) - 1)) == i
            items, j = [], i + 1
            while j < end_next - 1:
                if ty == "{":
                    k, j = value(j)
                    assert isinstance(k, str)
                    v, j = value(j)
                    items.append((k, v))
                else:
                    v, j = value(j)
                    items.append(v)
            assert j == end_next - 1 and count == min(len(items), 0xFFFFFF)
            return (items if ty == "[" else ("object", items)), end_next
        raise AssertionError(f"unexpected tape word {w:#x} at {i}")

    v, j = value(1)
    assert j == N - 1
    return v
