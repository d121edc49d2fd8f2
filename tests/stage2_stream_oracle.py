"""ctypes wrapper of tests/stage2_stream_oracle.c: stage 2 over a stream of documents, restated on the CPU with the
reference's walk (oracle/stage2_oracle.c) run on every document alone.  The library is built into a per-user temporary
directory, named after a digest of its sources, so that the tree stays untouched."""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile
from dataclasses import dataclass

import numpy as np

from oracle import oracle

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "stage2_stream_oracle.c")
_DEPS = [_SRC, os.path.join(os.path.dirname(_HERE), "oracle", "stage2_oracle.c")]
_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        h = hashlib.sha1()
        for p in _DEPS:
            with open(p, "rb") as f:
                h.update(f.read())
        d = os.path.join(tempfile.gettempdir(), f"sjb200-oracle-{os.getuid()}")
        path = os.path.join(d, f"liboracle_stage2_stream-{h.hexdigest()[:16]}.so")
        if not os.path.exists(path):
            os.makedirs(d, mode=0o700, exist_ok=True)
            tmp = f"{path}.{os.getpid()}.tmp"
            subprocess.check_call([os.environ.get("CC", "cc"), "-O2", "-std=c11", "-fPIC", "-shared", "-o", tmp, _SRC])
            os.replace(tmp, path)
        L = C.CDLL(path)
        L.oracle_stage2_walk_stream.restype = C.c_int64
        L.oracle_stage2_walk_stream.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p,
                                                C.c_void_p]
        _lib = L
    return _lib


@dataclass
class StreamWalk:
    doc_first: np.ndarray   # uint32 [n_docs + 1]
    doc_tape: np.ndarray    # uint64 [n_docs + 1]
    doc_error: np.ndarray   # int32 [n_docs], 0 = SUCCESS
    tape: np.ndarray        # uint64 [doc_tape[-1]]; a failing document's slice is unspecified
    string_buf: np.ndarray  # uint8, every string's record in index order (oracle.stage2_primitives)

    def slice(self, d: int) -> np.ndarray:
        return self.tape[int(self.doc_tape[d]) : int(self.doc_tape[d + 1])]


def stage2_walk_stream(data, indexes, n: int) -> StreamWalk:
    a = np.frombuffer(bytes(data), dtype=np.uint8) if not isinstance(data, np.ndarray) else data
    idx = np.ascontiguousarray(np.asarray(indexes)[:n], dtype=np.uint32)
    cap = 4 * n + 2
    tape = np.zeros(cap, dtype=np.uint64)
    first = np.zeros(n + 1, dtype=np.uint32)
    off = np.zeros(n + 1, dtype=np.uint64)
    err = np.zeros(max(n, 1), dtype=np.int32)
    nd = lib().oracle_stage2_walk_stream(a.ctypes.data if a.size else None, a.size, idx.ctypes.data if n else None, n, tape.ctypes.data, cap,
                                         first.ctypes.data, off.ctypes.data, err.ctypes.data)
    assert nd >= 0
    sbuf = oracle.stage2_primitives(a, idx).string_buf
    return StreamWalk(first[: nd + 1].copy(), off[: nd + 1].copy(), err[:nd].copy(), tape[: int(off[nd])].copy(), sbuf)
