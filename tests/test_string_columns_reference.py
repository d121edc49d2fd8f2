"""String columns from pointer cells (sjb200_string_columns_device_async), restated in Python, and pinned against Python's
json on generated streams.

expected_string_columns() is the definition the GPU tests (tests/test_gpu_string_columns.py) compare the device with, bit for
bit: one exclusive prefix sum of the cell lengths over all K·D cells, the strings' record bytes back to back, and the
summary (total bytes, string cells whose record does not lie inside strbuf_len).  Here it runs over the cells the restated
pointer rules give on the CPU stream oracle's tapes, and every string cell must be what json.loads reads at that pointer."""
from __future__ import annotations

import json
import random

import numpy as np

from tests import pointer_oracle as po
from tests.test_json_differential import corpus, oracle_stream, pointer_set
from tests.test_pointer_oracle import FAILING, RULES, stream_tapes

ALL_ONES = (1 << 64) - 1


def expected_string_columns(type_, value, strbuf, strbuf_len: int | None = None):
    """(offsets int64 [K·D + 1], data bytes, summary [total, cells whose record lies outside strbuf_len]) of the cells
    type_ / value ([K, D] or flat, in cell order) over the string buffer's first strbuf_len bytes."""
    ty = np.asarray(type_, dtype=np.uint8).ravel()
    val = np.asarray(value, dtype=np.int64).ravel()
    sb = bytes(np.asarray(strbuf, dtype=np.uint8))
    sb_len = len(sb) if strbuf_len is None else strbuf_len
    offsets = np.zeros(ty.size + 1, dtype=np.int64)
    parts, bad = [], 0
    for i in range(ty.size):
        rec = b""
        if ty[i] == ord('"'):
            r = po._record(sb, sb_len, int(val[i]) & ALL_ONES)   # the lookups' guard: the whole record inside sb_len
            if r is None:
                bad += 1
            else:
                rec = r
        parts.append(rec)
        offsets[i + 1] = offsets[i] + len(rec)
    return offsets, b"".join(parts), [int(offsets[-1]), bad]


def column_lists(offsets, data: bytes, type_) -> list[list]:
    """Per column: bytes for string cells, None elsewhere (PointerCells.strings' shape)."""
    ty = np.asarray(type_)
    k_n, d_n = ty.shape
    return [[data[offsets[k * d_n + d] : offsets[k * d_n + d + 1]] if ty[k, d] == ord('"') else None for d in range(d_n)] for k in range(k_n)]


def first_wins(pairs):
    """json.loads' object hook that keeps the first of repeated keys, as the pointer rules do."""
    out = {}
    for k, v in pairs:
        out.setdefault(k, v)
    return out


def resolve(v, toks):
    """RFC 6901 over a json.loads value; None if the pointer does not lead to a value."""
    for t in toks:
        t = t.decode("utf-8")
        if isinstance(v, dict):
            if t not in v:
                return None
            v = v[t]
        elif isinstance(v, list):
            if not t.isdigit() or (len(t) > 1 and t[0] == "0") or int(t) >= len(v):
                return None
            v = v[int(t)]
        else:
            return None
    return v


def test_against_json_loads_on_generated_streams():
    data, docs, _, g = corpus(0x57C0, 150, "lf", templated=300)
    _, s = oracle_stream(data)
    assert not s.doc_error.any()
    pointers = pointer_set(docs, random.Random(11), k=300, max_bytes=4000)
    status = np.full(len(docs), ALL_ONES, dtype=np.uint64)
    ty, code, val = po.cells(pointers, s.tape, s.string_buf, s.doc_tape, status)
    offsets, out, summary = expected_string_columns(ty, val, s.string_buf)
    assert summary == [len(out), 0] and int(offsets[-1]) == len(out) and (np.diff(offsets) >= 0).all()
    values = [json.loads(d.data, object_pairs_hook=first_wins) for d in docs]
    toks = [po.tokens(p) for p in pointers]
    d_n = len(docs)
    strings = []
    for k in range(len(pointers)):
        for d in range(d_n):
            i = k * d_n + d
            cell = out[offsets[i] : offsets[i + 1]]
            if ty[k, d] != ord('"'):
                assert cell == b"", (k, d)
                continue
            v = resolve(values[d], toks[k])
            assert isinstance(v, str) and cell == v.encode("utf-8"), (pointers[k][:40], d)
            strings.append(cell)
    # what the streams hold: escapes, surrogate pairs, \u0000, CJK, emoji, empty strings, repeated keys
    for feature in ("surrogate_pair", "u_0000", "esc_n", "esc_\\", 'esc_"', "utf8_3", "utf8_4", "key_dup"):
        assert g.counts[feature] >= 5, feature
    assert len(strings) > 500
    assert any(x == b"" for x in strings) and any(b"\x00" in x for x in strings)
    assert any("中".encode() in x for x in strings) and any("😀".encode() in x for x in strings)
    assert any(b'"' in x or b"\\" in x or b"\n" in x for x in strings)
    assert any(len(x.decode("utf-8")) < len(x) - 2 and any(ord(c) > 0xFFFF for c in x.decode("utf-8")) for x in strings)


def test_against_pointer_cells_strings():
    """The columns as lists are PointerCells.strings: the record's bytes where the cell is a string, None elsewhere."""
    from mojo_simdjson_b200.dom_parser_implementation import PointerCells

    docs = list(dict.fromkeys(d for d, _, _ in RULES))
    stream = []
    for i, d in enumerate(docs):
        stream += [d, FAILING[i % len(FAILING)]]
    pointers = [p for _, p, _ in RULES]
    tape, sb, doc_tape, status = stream_tapes(b"\n".join(stream))
    ty, code, val = po.cells(pointers, tape, sb, doc_tape, status)
    offsets, out, summary = expected_string_columns(ty, val, sb)
    cells = PointerCells(ty, code, val, np.asarray(sb, dtype=np.uint8))
    lists = column_lists(offsets, out, ty)
    assert lists == [cells.strings(k) for k in range(len(pointers))]
    assert summary == [len(out), 0] and sum(x is not None for row in lists for x in row) >= 2
    assert any(x == b"str" for row in lists for x in row)


def test_guard_and_non_string_cells():
    tape, sb, doc_tape, status = stream_tapes(b'{"a":"xyz","b":"","c":1,"d":"long string"}')
    ty, code, val = po.cells([b"/a", b"/b", b"/c", b"/d", b"/zz"], tape, sb, doc_tape, status)
    offsets, out, summary = expected_string_columns(ty, val, sb)
    assert out == b"xyzlong string" and offsets.tolist() == [0, 3, 3, 3, 14, 14] and summary == [14, 0]
    # records in index order: "a" 0, "xyz" 5, "b" 12, "" 17, "c" 21, "d" 26, "long string" 31: cut inside "xyz"'s record
    o2, out2, s2 = expected_string_columns(ty, val, sb, strbuf_len=7)
    assert out2 == b"" and s2 == [0, 3] and o2.tolist() == [0] * 6
    o3, out3, s3 = expected_string_columns(ty, val, sb, strbuf_len=41)   # "long string" ends at 46
    assert out3 == b"xyz" and s3 == [3, 1]
    # only '"' cells count: other types with any value, found or not, are empty; a string cell's value is a byte offset
    # read as unsigned, so a negative one is past every buffer
    t = np.array([ord("l"), ord("{"), 0, ord('"'), ord('"')], dtype=np.uint8)
    v = np.array([5, 1 << 40, -1, -1, 5], dtype=np.int64)
    o4, out4, s4 = expected_string_columns(t, v, sb)
    assert out4 == b"xyz" and s4 == [3, 1] and o4.tolist() == [0, 0, 0, 0, 0, 3]
