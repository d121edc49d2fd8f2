"""JSON Pointer lookups on stage-2 tapes, restated in Python: the rule table of include/simdjson_b200.h
(sjb200_at_pointers_device_async) over a tape slice and a string buffer, guards included."""
from __future__ import annotations

import numpy as np

SUCCESS, CAPACITY, TAPE_ERROR = 0, 1, 3
INCORRECT_TYPE, INDEX_OUT_OF_BOUNDS, NO_SUCH_FIELD, INVALID_JSON_POINTER = 17, 19, 20, 22
ALL_ONES = (1 << 64) - 1
PAYLOAD = (1 << 56) - 1
MAX_COUNT, MAX_BYTES = 1024, 16384
SCALARS = set(b'"ldtfn')


class InvalidPointer(ValueError):
    pass


def tokens(p: bytes) -> list[bytes]:
    """The unescaped reference tokens of one pointer; InvalidPointer if the call would refuse it."""
    if not p:
        return []
    if p[:1] != b"/":
        raise InvalidPointer(p)
    out = []
    for raw in p[1:].split(b"/"):
        tok, i = bytearray(), 0
        while i < len(raw):
            if raw[i] == 0x7E:   # '~'
                if raw[i + 1 : i + 2] not in (b"0", b"1"):
                    raise InvalidPointer(p)
                tok += b"~" if raw[i + 1] == 0x30 else b"/"
                i += 2
            else:
                tok.append(raw[i])
                i += 1
        out.append(bytes(tok))
    return out


def array_rule(tok: bytes) -> tuple[int, int]:
    """(code, index) of a token applied to an array: the checks in the header's order; the index saturates."""
    if tok == b"-":
        return INDEX_OUT_OF_BOUNDS, 0
    if not tok:
        return INVALID_JSON_POINTER, 0
    if any(not 0x30 <= b <= 0x39 for b in tok):
        return INCORRECT_TYPE, 0
    if len(tok) > 1 and tok[0] == 0x30:
        return INVALID_JSON_POINTER, 0
    return SUCCESS, min(int(tok), 0xFFFFFF)


def check_call(pointers: list[bytes]) -> int:
    """The call-level verdict: SUCCESS, INVALID_JSON_POINTER or CAPACITY."""
    if len(pointers) > MAX_COUNT or sum(len(p) for p in pointers) > MAX_BYTES:
        return CAPACITY
    try:
        for p in pointers:
            tokens(p)
    except InvalidPointer:
        return INVALID_JSON_POINTER
    return SUCCESS


def _record(sb: bytes, sb_len: int, off: int):
    """The bytes of the string record at off, or None if it reaches past sb_len."""
    if off > sb_len or sb_len - off < 4:
        return None
    n = int.from_bytes(sb[off : off + 4], "little")
    return sb[off + 4 : off + 4 + n] if sb_len - off - 4 >= n else None


def _skip(w, j: int, lim: int) -> int:
    """Index after the value at j, which must end at or before lim; 0 if the words say otherwise."""
    if j >= lim:
        return 0
    ty = w[j] >> 56
    if ty in b'"tfn':
        return j + 1
    if ty in b"ld":
        return j + 2 if j + 2 <= lim else 0
    if ty in b"{[":
        e = w[j] & 0xFFFFFFFF
        return e if j + 1 < e <= lim else 0
    return 0


def lookup(w, sb: bytes, sb_len: int, toks: list[bytes]) -> tuple[int, int, int]:
    """(type, code, value) of one pointer over one successful document's slice w (a list of ints)."""
    m = len(w)
    if m < 3:
        return 0, TAPE_ERROR, 0
    last = m - 1
    i = 1
    for tok in toks:
        word = w[i]
        ty = word >> 56
        if ty in b"{[":
            end = word & 0xFFFFFFFF
            if end <= i + 1 or end > last:
                return 0, TAPE_ERROR, 0
            close = end - 1
            if ty == ord("{"):
                j = i + 1
                while True:
                    if j + 1 >= close:
                        return 0, (TAPE_ERROR if j != close else NO_SUCH_FIELD), 0
                    if w[j] >> 56 != ord('"'):
                        return 0, TAPE_ERROR, 0
                    key = _record(sb, sb_len, w[j] & PAYLOAD)
                    if key is None:
                        return 0, CAPACITY, 0
                    if key == tok:   # the first match in tape order
                        break
                    j = _skip(w, j + 1, close)
                    if not j:
                        return 0, TAPE_ERROR, 0
                i = j + 1
            else:
                code, index = array_rule(tok)
                if code:
                    return 0, code, 0
                if index >= (word >> 32) & 0xFFFFFF:
                    return 0, INDEX_OUT_OF_BOUNDS, 0
                j = i + 1
                for _ in range(index):
                    j = _skip(w, j, close)
                    if not j:
                        return 0, TAPE_ERROR, 0
                if j >= close:
                    return 0, TAPE_ERROR, 0
                i = j
        elif ty in SCALARS:
            return 0, NO_SUCH_FIELD, 0
        else:
            return 0, TAPE_ERROR, 0
    word = w[i]
    ty = word >> 56
    if ty in b"ld":
        if i + 1 >= last:
            return 0, TAPE_ERROR, 0
        v = w[i + 1]
        return ty, SUCCESS, v - (1 << 64) if v >> 63 else v
    if ty == ord("t"):
        return ty, SUCCESS, 1
    if ty in b"fn":
        return ty, SUCCESS, 0
    if ty == ord('"'):
        if _record(sb, sb_len, word & PAYLOAD) is None:
            return 0, CAPACITY, 0
        return ty, SUCCESS, word & PAYLOAD
    if ty in b"{[":
        return ty, SUCCESS, i
    return 0, TAPE_ERROR, 0


def cells(pointers, tape, string_buf, doc_tape, doc_status, tape_len: int | None = None, strbuf_len: int | None = None):
    """The K x D cells: (type uint8 [K, D], code uint8 [K, D], value int64 [K, D]).  doc_status: uint64 words (all ones =
    SUCCESS) or int64 (-1).  Raises InvalidPointer for a pointer the call refuses."""
    pointers = [p.encode() if isinstance(p, str) else bytes(p) for p in pointers]
    toks = [tokens(p) for p in pointers]
    t = [int(x) for x in np.asarray(tape).view(np.uint64)]
    sb = bytes(np.asarray(string_buf, dtype=np.uint8))
    tape_len = len(t) if tape_len is None else tape_len
    sb_len = len(sb) if strbuf_len is None else strbuf_len
    dt = [int(x) for x in np.asarray(doc_tape).astype(np.uint64)]
    st = [int(x) & ALL_ONES for x in np.asarray(doc_status).astype(np.int64).view(np.uint64)]
    k_n, d_n = len(pointers), len(st)
    ty, code, val = np.zeros((k_n, d_n), np.uint8), np.zeros((k_n, d_n), np.uint8), np.zeros((k_n, d_n), np.int64)
    for d in range(d_n):
        lo, hi = dt[d], dt[d + 1]
        w = t[lo:hi] if lo <= hi <= tape_len else None
        for k in range(k_n):
            if st[d] != ALL_ONES:
                ty[k, d], code[k, d], val[k, d] = 0, st[d] & 0xFF, 0
            elif w is None:
                ty[k, d], code[k, d], val[k, d] = 0, CAPACITY, 0
            else:
                ty[k, d], code[k, d], val[k, d] = lookup(w, sb, sb_len, toks[k])
    return ty, code, val
