"""Builds and loads the host-side lane emulator (test infrastructure)."""
import ctypes as C
import os
import subprocess
from dataclasses import dataclass

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "emulate_stage1.cpp")
_CORE = os.path.join(_HERE, "..", "..", "mojo_simdjson_b200", "csrc", "stage1_core.cuh")
_SO = os.path.join(_HERE, "libemu_stage1.so")
_lib = None


def lib():
    global _lib
    if _lib is None:
        newest = max(os.path.getmtime(_SRC), os.path.getmtime(_CORE))
        if not os.path.exists(_SO) or os.path.getmtime(_SO) < newest:
            subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wall", "-o", _SO, _SRC])
        L = C.CDLL(_SO)
        L.emu_stage1.restype = C.c_int32
        L.emu_stage1.argtypes = [C.c_void_p, C.c_uint64, C.c_uint32, C.c_int, C.c_void_p, C.c_uint64,
                                 C.POINTER(C.c_uint32), C.POINTER(C.c_uint64), C.POINTER(C.c_int32), C.c_uint32]
        L.emu_stage1_stream.restype = C.c_int32
        L.emu_stage1_stream.argtypes = [C.c_void_p, C.c_uint64, C.c_uint32, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint32),
                                        C.POINTER(C.c_uint64), C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.c_uint32]
        L.emu_stage1_stream_sched.restype = C.c_int32
        L.emu_stage1_stream_sched.argtypes = [C.c_void_p, C.c_uint64, C.c_uint32, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint32),
                                              C.POINTER(C.c_uint64), C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.c_uint32,
                                              C.c_uint32, C.c_uint64, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p]
        L.emu_straddle_gate_misses.restype = C.c_uint64
        L.emu_straddle_gate_misses.argtypes = [C.POINTER(C.c_uint64)]
        L.emu_bitplanes32.restype = None
        L.emu_bitplanes32.argtypes = [C.c_void_p, C.c_void_p]
        L.emu_fl2_div.restype = C.c_uint32
        L.emu_fl2_div.argtypes = [C.c_uint32, C.c_uint32]
        L.emu_drop_high_bits.restype = C.c_uint32
        L.emu_drop_high_bits.argtypes = [C.c_uint32, C.c_uint32]
        L.emu_flatten_unit.restype = C.c_int32
        L.emu_flatten_unit.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.POINTER(C.c_uint32)]
        _lib = L
    return _lib


def stage1(data: bytes, mis: int = 0, warps: int = 8, flags: int = 0, cap=None):
    L = lib()
    a = np.frombuffer(bytes(data), dtype=np.uint8)
    n_bytes = int(a.size)
    if cap is None:
        cap = n_bytes + 3
    out = np.full(max(cap, 1), 0xDEADBEEF, dtype=np.uint32)
    n = C.c_uint32(0xFFFFFFFF)
    nw = C.c_uint64(0)
    u8 = C.c_int32(0)
    err = L.emu_stage1(a.ctypes.data if n_bytes else None, n_bytes, mis, warps, out.ctypes.data, cap,
                       C.byref(n), C.byref(nw), C.byref(u8), flags)
    assigned = n.value != 0xFFFFFFFF
    keep = min(int(nw.value) + (3 if assigned else 0), cap)
    return err, (n.value if assigned else None), int(nw.value), out[:keep].copy(), int(u8.value)


def stage1_stream(data: bytes, mis: int = 0, flags: int = 0, cap=None):
    """The stream pipeline's arithmetic on the host.  Returns (err, n, n_written, out, utf8, gave_up)."""
    L = lib()
    a = np.frombuffer(bytes(data), dtype=np.uint8)
    n_bytes = int(a.size)
    if cap is None:
        cap = n_bytes + 3
    out = np.full(max(cap, 1), 0xDEADBEEF, dtype=np.uint32)
    n = C.c_uint32(0xFFFFFFFF)
    nw = C.c_uint64(0)
    u8 = C.c_int32(0)
    spec = C.c_int32(0)
    err = L.emu_stage1_stream(a.ctypes.data if n_bytes else None, n_bytes, mis, out.ctypes.data, cap,
                              C.byref(n), C.byref(nw), C.byref(u8), C.byref(spec), flags)
    assigned = n.value != 0xFFFFFFFF
    keep = min(int(nw.value) + (3 if assigned else 0), cap)
    return err, (n.value if assigned else None), int(nw.value), out[:keep].copy(), int(u8.value), bool(spec.value)


SKIPPED, INLINE, PARKED = 0, 1, 2
MID_RUN, END_OF_WARP = 1, 2


@dataclass
class Probe:
    """How the lane holding one byte was validated: kind SKIPPED / INLINE / PARKED; for PARKED the warp, the slot of its
    ring and the flush (MID_RUN / END_OF_WARP) that validated it, else None."""
    kind: int
    warp: int | None
    slot: int | None
    flush: int | None


@dataclass
class StreamRun:
    err: int
    n: int | None
    n_written: int
    out: np.ndarray
    utf8: int
    gave_up: bool
    mid_run_flushes: int
    end_of_warp_flushes: int
    max_fill: int            # the largest fill of a ring at a flush
    slots_reached: int       # bit s: some lane was parked in slot s
    inline_chunks: int
    probes: list


def stage1_stream_sched(data, mis: int = 0, flags: int = 0, cap=None, warps: int = 4736, seed: int = 0, probes=()):
    """The stream pipeline with the classify kernel's UTF-8 deferral: `warps` warps in the grid, runs past the first
    4 * warps chunks handed out in an order drawn from `seed`.  `probes`: document byte positions to report on."""
    L = lib()
    a = np.frombuffer(bytes(data), dtype=np.uint8) if not isinstance(data, np.ndarray) else np.ascontiguousarray(data, dtype=np.uint8)
    n_bytes = int(a.size)
    if cap is None:
        cap = n_bytes + 3
    out = np.full(max(cap, 1), 0xDEADBEEF, dtype=np.uint32)
    n = C.c_uint32(0xFFFFFFFF)
    nw = C.c_uint64(0)
    u8 = C.c_int32(0)
    spec = C.c_int32(0)
    stats = np.zeros(5, dtype=np.int64)
    pp = np.ascontiguousarray(np.asarray(list(probes), dtype=np.uint64))
    po = np.zeros(max(4 * pp.size, 1), dtype=np.int32)
    err = L.emu_stage1_stream_sched(a.ctypes.data if n_bytes else None, n_bytes, mis, out.ctypes.data, cap, C.byref(n), C.byref(nw),
                                    C.byref(u8), C.byref(spec), flags, warps, seed, stats.ctypes.data,
                                    pp.ctypes.data if pp.size else None, pp.size, po.ctypes.data)
    assert err > -100, f"emulator invariant broken: {err}"
    assigned = n.value != 0xFFFFFFFF
    keep = min(int(nw.value) + (3 if assigned else 0), cap)
    pr = []
    for i in range(pp.size):
        k, w, s, f = (int(x) for x in po[4 * i : 4 * i + 4])
        pr.append(Probe(k, None if w < 0 else w, None if s < 0 else s, None if f < 0 else f))
    return StreamRun(err, n.value if assigned else None, int(nw.value), out[:keep].copy(), int(u8.value), bool(spec.value),
                     int(stats[0]), int(stats[1]), int(stats[2]), int(stats[3]), int(stats[4]), pr)


def straddle_gate_misses():
    """(values of the 3 bytes before a lane for which the inline path's straddle gate is closed but the carry it skips is not
    zero, values for which the gate is closed)"""
    closed = C.c_uint64(0)
    miss = lib().emu_straddle_gate_misses(C.byref(closed))
    return int(miss), int(closed.value)


def flatten_unit(words: np.ndarray, value_base: int = 0, cap: int = 768):
    """The balanced flatten kernel's steps for one unit of 128 mask words.  Returns (rc, indexes)."""
    L = lib()
    w = np.ascontiguousarray(words, dtype=np.uint32)
    assert w.size == 128
    out = np.zeros(4096, dtype=np.uint32)
    count = C.c_uint32(0)
    rc = L.emu_flatten_unit(w.ctypes.data, value_base, cap, out.ctypes.data, C.byref(count))
    return rc, out[: count.value].copy()
