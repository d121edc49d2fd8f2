"""Differential tests of the CPU oracles against Python's json on streams from tests/jsongen.py, and the helpers the GPU
differential tests (tests/test_gpu_json_differential.py) share with them.

Stage 1 of the oracle, then the stream oracle (tests/stage2_stream_oracle.c) on generated NDJSON (LF and CRLF) and
concatenated streams: every document is SUCCESS, its tape slice decodes to what json.loads says, and its first token sits at
the byte offset the generator recorded.  The pointer cells expected from the generated values (RFC 6901, the first of
repeated keys) are checked against the restated pointer rules over the same tapes.  Each documented difference from
json.loads is pinned with a known answer."""
from __future__ import annotations

import json
import random
import struct

import numpy as np
import pytest

from oracle import oracle
from tests import jsongen as jg
from tests import pointer_oracle as po
from tests import stage2_stream_oracle as so
from tests.test_pointer_oracle import decode_at, resolve_decoded
from tests.test_stage2_oracle import python_document

ALL_ONES = (1 << 64) - 1
MODES = ("lf", "crlf", "concat")


# ---- shared helpers --------------------------------------------------------------------------------------------------------

def corpus(seed: int, n_docs: int, mode: str, templated: int = 0, **gen_kw):
    """(stream bytes, docs, start offsets, generator): n_docs random documents and `templated` templated ones, shuffled."""
    g = jg.Gen(seed, **gen_kw)
    docs = [g.document() for _ in range(n_docs)] + (g.templated(templated) if templated else [])
    g.r.shuffle(docs)
    data, starts = jg.stream(docs, g.r, mode, g.counts)
    return data, docs, starts, g


def oracle_stream(data: bytes):
    """(stage-1 result, stream walk) of the CPU oracles."""
    w = oracle.stage1(data, impl="fast" if len(data) > 20000 else "ref")
    assert w.error == 0, data[:60]
    return w, so.stage2_walk_stream(np.frombuffer(data, dtype=np.uint8), w.indexes[: w.n], w.n)


def check_split(idx: np.ndarray, doc_first: np.ndarray, docs, starts):
    """The documents split where the generator put them: their count, token counts and the byte offset of every first token."""
    first = np.asarray(doc_first, dtype=np.int64)
    assert first.size == len(docs) + 1
    assert np.array_equal(np.diff(first), [d.tokens for d in docs])
    assert np.array_equal(np.asarray(idx, dtype=np.int64)[first[:-1]], starts)


def bits(x: float) -> int:
    return struct.unpack("<Q", struct.pack("<d", x))[0]


def kernel_double(f: jg.Float) -> float:
    """The double the device writes for a token (test_gpu_stage2_scale.restated): float() itself on the exact fast path."""
    from tests.test_gpu_stage2_scale import restated

    b, _ = restated(f.tok)
    return struct.unpack("<d", struct.pack("<Q", b))[0]


def as_kernel(v):
    """A generated value with every double replaced by the one the device writes."""
    if isinstance(v, jg.Float):
        return kernel_double(v)
    if isinstance(v, tuple):
        return ("object", [(k, as_kernel(x)) for k, x in v[1]])
    if isinstance(v, list):
        return [as_kernel(x) for x in v]
    return v


def check_exact_doubles(docs):
    """Every token the restated kernel conversion calls exact converts to float()'s bits."""
    from tests.test_gpu_stage2_scale import restated

    n = 0
    for d in docs:
        for f in floats_of(d.value):
            b, inexact = restated(f.tok)
            if not inexact:
                assert b == bits(float(f.tok)), f.tok
                n += 1
    return n


def floats_of(v):
    if isinstance(v, jg.Float):
        yield v
    elif isinstance(v, tuple):
        for _, x in v[1]:
            yield from floats_of(x)
    elif isinstance(v, list):
        for x in v:
            yield from floats_of(x)


def check_documents(docs, tape: np.ndarray, doc_tape: np.ndarray, string_buf: np.ndarray, which=None, kernel: bool = False):
    """decode_tape of every document's slice (or of those in `which`) equals its value: json.loads' value, with the device's
    doubles where kernel=True."""
    sb = bytes(np.asarray(string_buf))   # once: decode_tape takes bytes as they are
    tape = np.asarray(tape).view(np.uint64)
    for d in range(len(docs)) if which is None else which:
        got = oracle.decode_tape(tape[int(doc_tape[d]) : int(doc_tape[d + 1])].tolist(), sb)
        assert got == (as_kernel(docs[d].value) if kernel else docs[d].value), (d, docs[d].data[:80])


def node_at(v, path):
    for t in path:
        if isinstance(t, int):
            v = v[t]
        else:
            v = next(x for k, x in v[1] if k == t)   # the first of repeated keys
    return v


def pointer_set(docs, r: random.Random, k: int = po.MAX_COUNT, max_bytes: int = po.MAX_BYTES):
    """Up to k pointers, max_bytes in all: paths sampled from the documents and variants of them that miss (a missing key,
    index = count, '-', a leading zero, '0a', a token applied to a scalar)."""
    out, used = {b"": None}, 0
    tries = 0
    while len(out) < k and tries < 50 * k:
        tries += 1
        d = r.choice(docs)
        path = r.choice(d.paths)
        p = jg.pointer(path)
        node = node_at(d.value, path)
        cands = [p]
        if isinstance(node, list):
            cands += [jg.pointer(path + [len(node)]), p + b"/-", p + b"/00", p + b"/01", p + b"/0a"]
        elif isinstance(node, tuple):
            cands += [jg.pointer(path + ["no such key"]), jg.pointer(path + ["0"])]
        else:
            cands += [p + b"/0", p + b"/a"]
        q = cands[0] if r.random() < 0.6 else r.choice(cands)
        room = (max_bytes - used) / (k - len(out))   # bytes per pointer still to come: long ones only now and then
        if q in out or used + len(q) > max_bytes or (len(q) > room and r.random() < 0.9):
            continue
        out[q] = None
        used += len(q)
    return list(out)


def type_of(v) -> int:
    if v is True:
        return ord("t")
    if v is False:
        return ord("f")
    if v is None:
        return ord("n")
    if isinstance(v, int):
        return ord("l")
    if isinstance(v, float):
        return ord("d")
    if isinstance(v, str):
        return ord('"')
    return ord("[") if isinstance(v, list) else ord("{")


def expected_cells(pointers, docs, status=None):
    """[k][d] -> (code, value or None): RFC 6901 over the generated values, the first of repeated keys, the array rules of
    pointer_oracle.array_rule.  A failing document (status word not all ones) gives its own code in every cell."""
    toks = [po.tokens(p) for p in pointers]
    out = []
    for t in toks:
        row = []
        for d, doc in enumerate(docs):
            if status is not None and int(status[d]) != ALL_ONES:
                row.append((int(status[d]) & 0xFF, None))
            else:
                row.append(resolve_decoded(doc.value, t))
        out.append(row)
    return out


def check_cells(want, ty, code, val, tape, doc_tape, string_buf, kernel: bool):
    """Device or oracle cells against expected_cells: code and type, and the value: 'l' the integer, 'd' the double's bits
    (the device's where kernel=True), '"' the record, '{' and '[' the subtree at the slice index, 't' 'f' 'n' 1 0 0."""
    sb = bytes(np.asarray(string_buf))
    ty, code, val = np.asarray(ty), np.asarray(code), np.asarray(val)
    slices = {}
    found = 0
    for k, row in enumerate(want):
        for d, (c, v) in enumerate(row):
            assert int(code[k, d]) == c, (k, d)
            if c:
                assert int(ty[k, d]) == 0 and int(val[k, d]) == 0, (k, d)
                continue
            found += 1
            t, x = int(ty[k, d]), int(val[k, d])
            assert t == type_of(v), (k, d)
            if t == ord("l"):
                assert x == v, (k, d)
            elif t == ord("d"):
                assert x & ALL_ONES == bits(kernel_double(v) if kernel else float(v)), (k, d)
            elif t == ord('"'):
                n = int.from_bytes(sb[x : x + 4], "little")
                assert sb[x + 4 : x + 4 + n] == v.encode("utf-8"), (k, d)
            elif t in b"tfn":
                assert x == (1 if t == ord("t") else 0), (k, d)
            else:
                if d not in slices:
                    slices[d] = [int(w) for w in np.asarray(tape)[int(doc_tape[d]) : int(doc_tape[d + 1])].view(np.uint64)]
                assert decode_at(slices[d], sb, x) == (as_kernel(v) if kernel else v), (k, d)
    return found


# ---- the tests -------------------------------------------------------------------------------------------------------------

def test_depth_limits_are_the_walks():
    from tests.test_gpu_at_pointer import deepest

    assert deepest(b"[", b"]", b"7") == jg.MAX_ARRAY_LEVEL
    assert deepest(b'{"k":', b"}", b"7") == jg.MAX_OBJECT_LEVEL


@pytest.mark.parametrize("mode", MODES)
def test_streams_against_json_loads(mode):
    data, docs, starts, g = corpus(0xD1FF + MODES.index(mode), 500, mode, templated=200)
    w, s = oracle_stream(data)
    assert not s.doc_error.any()
    check_split(w.indexes, s.doc_first, docs, starts)
    for d, doc in enumerate(docs):   # json.loads first: the generator's value is what Python's json reads
        assert python_document(doc.data) == doc.value, doc.data[:80]
    check_documents(docs, s.tape, s.doc_tape, s.string_buf)
    assert check_exact_doubles(docs) > 200


def test_feature_counts():
    """What the generator writes at the sizes the tests use, so that the coverage cannot quietly shrink."""
    counts = {}
    for mode in MODES:
        _, _, _, g = corpus(0xD1FF + MODES.index(mode), 500, mode, templated=200)
        for key, v in g.counts.items():
            counts[key] = counts.get(key, 0) + v
    at_least = {"documents": 1500, "templated": 600, "root_scalar": 100, "true": 100, "false": 100, "null": 100, "empty_array": 100,
                "empty_object": 100, "wide_array": 1, "wide_object": 1, "max_depth_array": 2, "max_depth_object": 2,
                "str_gt64": 100, "str_gt2k": 10, "surrogate_pair": 1000, "surrogate_pair_max": 100, "u_lower": 1000, "u_upper": 1000,
                "key_empty": 50, "key_slash": 50, "key_tilde": 50, "key_numeric": 50, "key_dup": 50, "int64_min": 20, "int64_max": 20,
                "int_neg_zero": 20, "float_neg_zero": 20, "exp_e": 100, "exp_E": 100, "exp_sign_+": 100, "exp_sign_-": 100,
                "exp_sign_none": 100, "exp_near22": 100, "exp_near308": 100, "exp_beyond": 100, "ws_space": 100, "ws_tab": 100,
                "ws_lf": 100, "ws_cr": 100, "sep_lf": 500, "sep_crlf": 500, "blank_line": 10, "concat_after_brace": 20,
                "concat_after_bracket": 20, "concat_after_quote": 5}
    at_least.update({"esc_" + e[1:].decode(): 100 for e in jg.SHORT_ESCAPES})
    at_least.update({"u_%04x" % cp: 100 for cp in jg.U_EDGES})
    at_least.update({"utf8_%d" % n: 100 for n in (1, 2, 3, 4)})
    at_least.update({"int_digits_%d" % n: 20 for n in range(1, 20)})
    at_least.update({"mant_%d" % n: 50 for n in range(15, 21)})
    short = {k: (counts.get(k, 0), v) for k, v in at_least.items() if counts.get(k, 0) < v}
    assert not short, short


def test_expected_cells_against_the_restated_rules():
    """The cells the GPU tests expect, from the generated values, equal the restated pointer rules over the oracle's tapes."""
    data, docs, starts, g = corpus(0x9017, 150, "lf", templated=250)
    w, s = oracle_stream(data)
    assert not s.doc_error.any()
    pointers = pointer_set(docs, random.Random(5))
    assert len(pointers) > 800 and sum(map(len, pointers)) <= po.MAX_BYTES and max(map(len, pointers)) > 100
    status = np.full(len(docs), ALL_ONES, dtype=np.uint64)
    ty, code, val = po.cells(pointers, s.tape, s.string_buf, s.doc_tape, status)
    want = expected_cells(pointers, docs)
    found = check_cells(want, ty, code, val, s.tape, s.doc_tape, s.string_buf, kernel=False)
    assert found > 3000
    codes = set(np.unique(code).tolist())
    assert {0, po.NO_SUCH_FIELD, po.INDEX_OUT_OF_BOUNDS, po.INCORRECT_TYPE, po.INVALID_JSON_POINTER} <= codes
    assert set(np.unique(ty).tolist()) >= set(b'{["ldtfn')


def walk_one(data: bytes):
    w = oracle.stage1(data)
    assert w.error == 0
    return w, so.stage2_walk_stream(np.frombuffer(data, dtype=np.uint8), w.indexes[: w.n], w.n)


def test_documented_differences_from_json_loads():
    # a root-level empty container: TAPE_ERROR here, accepted by json.loads
    for doc in (b"{}", b"[]"):
        assert json.loads(doc) in ({}, [])
        _, s = walk_one(doc)
        assert s.doc_error.tolist() == [oracle.TAPE_ERROR]
    # an integer past int64: the decimal value mod 2^64 as a signed 'l'; json.loads keeps every digit
    for tok in (b"9223372036854775808", b"18446744073709551617", b"-9223372036854775809", b"99999999999999999999"):
        _, s = walk_one(b"[" + tok + b"]")
        assert s.doc_error.tolist() == [0]
        t = s.slice(0)
        v = (int(tok) % (1 << 64))
        assert int(t[2]) >> 56 == ord("l") and int(t[3]) == v, tok
        assert json.loads(tok) == int(tok)
    # a leading zero: accepted as 1 here, refused by json.loads
    _, s = walk_one(b"[01]")
    assert s.doc_error.tolist() == [0] and oracle.decode_tape(s.slice(0), s.string_buf) == [1]
    with pytest.raises(json.JSONDecodeError):
        json.loads(b"[01]")
    # a lone surrogate escape: STRING_ERROR here, accepted by json.loads
    for doc in (b'["\\ud800"]', b'["\\uDC00"]', b'["\\ud800\\u0041"]', b'["\\ud800x"]'):
        _, s = walk_one(doc)
        assert s.doc_error.tolist() == [oracle.STRING_ERROR], doc
        json.loads(doc)
    # a number with a string right after it: one document, NUMBER_ERROR; json.loads refuses the pair
    w, s = walk_one(b'1"a"')
    assert w.n == 1 and s.doc_error.tolist() == [oracle.NUMBER_ERROR]
    with pytest.raises(json.JSONDecodeError):
        json.loads(b'1"a"')
    # repeated keys: the tape keeps every member, pointers take the first, json.loads keeps the last
    doc = b'{"a":1,"b":2,"a":3}'
    _, s = walk_one(doc)
    assert oracle.decode_tape(s.slice(0), s.string_buf) == ("object", [("a", 1), ("b", 2), ("a", 3)])
    st = np.array([ALL_ONES], dtype=np.uint64)
    _, code, val = po.cells([b"/a"], s.tape, s.string_buf, s.doc_tape, st)
    assert int(code[0, 0]) == 0 and int(val[0, 0]) == 1 and json.loads(doc)["a"] == 3
    # nesting: objects fail past depth 100, arrays one level earlier; json.loads takes both
    for depth, want in ((jg.MAX_ARRAY_LEVEL, 0), (jg.MAX_ARRAY_LEVEL + 1, oracle.DEPTH_ERROR)):
        doc = b"[" * depth + b"1" + b"]" * depth
        assert walk_one(doc)[1].doc_error.tolist() == [want]
        json.loads(doc)
    for depth, want in ((jg.MAX_OBJECT_LEVEL, 0), (jg.MAX_OBJECT_LEVEL + 1, oracle.DEPTH_ERROR)):
        doc = b'{"k":' * depth + b"1" + b"}" * depth
        assert walk_one(doc)[1].doc_error.tolist() == [want]
        json.loads(doc)
