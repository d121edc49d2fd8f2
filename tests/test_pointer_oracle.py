"""Pins tests/pointer_oracle.py, the restated JSON Pointer rules, three ways: a hand-written rule table, an independent
composition over oracle.decode_tape's ordered (key, value) lists, and 2,000 fuzzed documents against json.loads plus a
plain RFC 6901 resolver.  The tapes come from the CPU stream oracle (tests/stage2_stream_oracle.c)."""
import json
import random
import struct

import numpy as np
import pytest

from oracle import oracle
from tests import pointer_oracle as po
from tests import stage2_stream_oracle as so

ALL_ONES = (1 << 64) - 1


def stream_tapes(data: bytes):
    """(tape, string_buf, doc_tape, doc_status) of a stream from the CPU oracles; doc_status as uint64 words."""
    w = oracle.stage1(data)
    assert w.error == 0, data[:60]
    s = so.stage2_walk_stream(data, w.indexes[: w.n], w.n)
    status = np.array([ALL_ONES if e == 0 else int(e) for e in s.doc_error.tolist()], dtype=np.uint64)
    return s.tape, s.string_buf, s.doc_tape, status


def decode_at(w, sb: bytes, i: int):
    """The value at slice index i as python objects (objects as ("object", [(key, value), ...]))."""
    ty, p = chr(w[i] >> 56), w[i] & po.PAYLOAD
    if ty == '"':
        n = int.from_bytes(sb[p : p + 4], "little")
        return sb[p + 4 : p + 4 + n].decode("utf-8", "surrogatepass")
    if ty == "l":
        return w[i + 1] - (1 << 64) if w[i + 1] >> 63 else w[i + 1]
    if ty == "d":
        return struct.unpack("<d", struct.pack("<Q", w[i + 1]))[0]
    if ty in "tfn":
        return {"t": True, "f": False, "n": None}[ty]
    end, items, j = p & 0xFFFFFFFF, [], i + 1
    while j < end - 1:
        if ty == "{":
            k = decode_at(w, sb, j)
            j += 1
        v = decode_at(w, sb, j)
        j = po._skip(w, j, end - 1)
        items.append((k, v) if ty == "{" else v)
    return ("object", items) if ty == "{" else items


def cell_value(w, sb: bytes, ty: int, value: int):
    """A found cell as the python value it stands for."""
    if ty == ord("l"):
        return value
    if ty == ord("d"):
        return struct.unpack("<d", struct.pack("<q", value))[0]
    if ty in b"tfn":
        assert value == (1 if ty == ord("t") else 0)
        return {ord("t"): True, ord("f"): False, ord("n"): None}[ty]
    if ty == ord('"'):
        n = int.from_bytes(sb[value : value + 4], "little")
        return sb[value + 4 : value + 4 + n].decode("utf-8", "surrogatepass")
    assert ty in b"{[" and w[value] >> 56 == ty
    return decode_at(w, sb, value)


def run_cells(docs: list[bytes], pointers):
    data = b"\n".join(docs)
    tape, sb, doc_tape, status = stream_tapes(data)
    assert status.size == len(docs)
    ty, code, val = po.cells(pointers, tape, sb, doc_tape, status)
    slices = [[int(x) for x in tape[int(doc_tape[d]) : int(doc_tape[d + 1])]] for d in range(len(docs))]
    return ty, code, val, slices, bytes(sb), status


# ---- 1. the rule table ---------------------------------------------------------------------------------------------------

DOC_KEYS = (b'{"a~b":1,"a/b":2,"~1":3,"":4,"a":{"":5},"ab":6,"a\\/c":7,"\xc3\xa9":8,"x":[10,20,30],"s":"str","t":true,"f":false,'
            b'"n":null,"d":1.5,"dup":1,"dup":2,"e":[],"o":{}}')
LONG = {n: b"k" * n for n in (31, 32, 33, 5000)}
DOC_LONG = b'{"":0,' + b",".join(b'"%s":%d' % (LONG[n], n) for n in (31, 32, 33, 5000)) + b"}"
NSF, IOB, BAD, ITY = po.NO_SUCH_FIELD, po.INDEX_OUT_OF_BOUNDS, po.INVALID_JSON_POINTER, po.INCORRECT_TYPE

# (document, pointer, expected): an error code, or (type character, python value); containers by their slice index too
RULES = [
    (DOC_KEYS, b"/a~0b", ("l", 1)), (DOC_KEYS, b"/a~1b", ("l", 2)), (DOC_KEYS, b"/~01", ("l", 3)), (DOC_KEYS, b"/~1", NSF),
    (DOC_KEYS, b"/~0", NSF), (DOC_KEYS, b"/", ("l", 4)), (DOC_KEYS, b"/a/", ("l", 5)), (DOC_KEYS, b"/ab", ("l", 6)),
    (DOC_KEYS, b"/a", ("{", ("object", [("", 5)]))), (DOC_KEYS, b"/a~1c", ("l", 7)), (DOC_KEYS, b"/a\\/c", NSF),
    (DOC_KEYS, "/é".encode(), ("l", 8)), (DOC_KEYS, b"/x/0", ("l", 10)), (DOC_KEYS, b"/x/2", ("l", 30)), (DOC_KEYS, b"/x/3", IOB),
    (DOC_KEYS, b"/x/-", IOB), (DOC_KEYS, b"/x/00", BAD), (DOC_KEYS, b"/x/01", BAD), (DOC_KEYS, b"/x/0a", ITY), (DOC_KEYS, b"/x/", BAD),
    (DOC_KEYS, b"/x/a", ITY), (DOC_KEYS, b"/x/-1", ITY), (DOC_KEYS, b"/x/+1", ITY), (DOC_KEYS, b"/x/99999999999999999999", IOB),
    (DOC_KEYS, b"/x/16777215", IOB), (DOC_KEYS, b"/e/0", IOB), (DOC_KEYS, b"/e/-", IOB), (DOC_KEYS, b"/e/", BAD), (DOC_KEYS, b"/o/", NSF),
    (DOC_KEYS, b"/x", ("[", [10, 20, 30])), (DOC_KEYS, b"/s", ('"', "str")), (DOC_KEYS, b"/s/0", NSF), (DOC_KEYS, b"/t", ("t", True)),
    (DOC_KEYS, b"/f", ("f", False)), (DOC_KEYS, b"/n", ("n", None)), (DOC_KEYS, b"/n/x", NSF), (DOC_KEYS, b"/d", ("d", 1.5)),
    (DOC_KEYS, b"/d/0", NSF), (DOC_KEYS, b"/x/0/y", NSF), (DOC_KEYS, b"/x/1/0", NSF), (DOC_KEYS, b"/t/", NSF), (DOC_KEYS, b"/dup", ("l", 1)),
    (DOC_KEYS, b"/missing", NSF), (DOC_KEYS, b"/A", NSF), (DOC_KEYS, b"/a/b", NSF), (DOC_KEYS, b"/x/0a/b", ITY),
    (DOC_LONG, b"/", ("l", 0)), (DOC_LONG, b"/" + LONG[31], ("l", 31)), (DOC_LONG, b"/" + LONG[32], ("l", 32)), (DOC_LONG, b"/" + LONG[33], ("l", 33)),
    (DOC_LONG, b"/" + LONG[5000], ("l", 5000)), (DOC_LONG, b"/" + b"k" * 34, NSF), (DOC_LONG, b"/" + b"k" * 4999, NSF), (DOC_LONG, b"/k", NSF),
    (b'[1,{"a":2}]', b"", ("[", [1, ("object", [("a", 2)])])), (b'[1,{"a":2}]', b"/1/a", ("l", 2)), (b'[1,{"a":2}]', b"/0", ("l", 1)),
    (b'[1,{"a":2}]', b"/2", IOB), (b'[1,{"a":2}]', b"/a", ITY), (b'"abc"', b"", ('"', "abc")), (b'"abc"', b"/x", NSF), (b'"abc"', b"/0", NSF),
    (b"-5", b"", ("l", -5)), (b"-5", b"/", NSF), (b"true", b"", ("t", True)), (b"null", b"/-", NSF),
    (b'[[[[7]]]]', b"/0/0/0/0", ("l", 7)), (b'[[[[7]]]]', b"/0/0/0/1", IOB), (b'{"a":{"b":{"c":[true]}}}', b"/a/b/c/0", ("t", True)),
]
FAILING = [b'{"a":tru}', b"[1,]", b'{"a" 1}', b'{"a":"\\x"}', b"[12x]", b'{"a":1,}', b"[" * 101 + b"]" * 101]


def check_cell(w, sb, got, want, where):
    ty, code, val = got
    if isinstance(want, int):
        assert (ty, code, val) == (0, want, 0), where
    else:
        assert code == 0 and ty == ord(want[0]), where
        assert cell_value(w, sb, ty, val) == want[1], where


def test_rule_table():
    docs = list(dict.fromkeys(d for d, _, _ in RULES))
    for doc in docs:
        rows = [(p, e) for d, p, e in RULES if d == doc]
        ty, code, val, slices, sb, _ = run_cells([doc], [p for p, _ in rows])
        for k, (p, e) in enumerate(rows):
            check_cell(slices[0], sb, (int(ty[k, 0]), int(code[k, 0]), int(val[k, 0])), e, (doc[:40], p[:40]))


def test_rule_table_container_indexes():
    # slice words: 0 r, 1 [, 2 l, 3 1, 4 {, 5 "a", 6 l, 7 2, 8 }, 9 ], 10 r
    ty, code, val, _, _, _ = run_cells([b'[1,{"a":2}]'], [b"", b"/1"])
    assert (int(ty[0, 0]), int(val[0, 0])) == (ord("["), 1) and (int(ty[1, 0]), int(val[1, 0])) == (ord("{"), 4)
    # in a stream the index is relative to the document's own slice
    ty, code, val, _, _, _ = run_cells([b"[0,0,0]", b'[1,{"a":2}]'], [b"/1"])
    assert (int(ty[0, 1]), int(val[0, 1])) == (ord("{"), 4)


def test_rule_table_as_one_stream_with_failing_documents():
    """Every document of the table in one stream, with failing documents between them: each failing document's cells carry
    its own code, and its neighbours' cells are what they are alone."""
    docs = list(dict.fromkeys(d for d, _, _ in RULES))
    stream = []
    for i, d in enumerate(docs):
        stream.append(d)
        stream.append(FAILING[i % len(FAILING)])
    pointers = [p for _, p, _ in RULES]
    ty, code, val, slices, sb, status = run_cells(stream, pointers)
    for i, doc in enumerate(stream):
        if doc in FAILING:
            c = int(status[i]) & 0xFF
            assert int(status[i]) != ALL_ONES and c != 0, doc
            assert (ty[:, i] == 0).all() and (code[:, i] == c).all() and (val[:, i] == 0).all(), doc
            continue
        for k, (d, p, e) in enumerate(RULES):
            if d == doc:
                check_cell(slices[i], sb, (int(ty[k, i]), int(code[k, i]), int(val[k, i])), e, (doc[:40], p[:40]))


def test_call_level_checks():
    assert po.check_call([b"", b"/a"]) == 0
    for bad in (b"a", b"#/a", b"/a~", b"/a~2", b"/~a", b"//~"):
        assert po.check_call([b"/a", bad]) == po.INVALID_JSON_POINTER, bad
    assert po.check_call([b"/a"] * 1024) == 0 and po.check_call([b"/a"] * 1025) == po.CAPACITY
    assert po.check_call([b"/" + b"a" * 16383]) == 0 and po.check_call([b"/" + b"a" * 16384]) == po.CAPACITY
    assert po.tokens(b"/~01") == [b"~1"] and po.tokens(b"/~10") == [b"/0"] and po.tokens(b"//") == [b"", b""]


def test_guards():
    tape, sb, doc_tape, status = stream_tapes(b'{"a":[1,2],"b":"xyz"}')
    t = tape.copy()
    ty, code, val = po.cells([b"/b", b"/a/1"], t, sb, doc_tape, status)
    assert code.tolist() == [[0], [0]]
    # a slice past tape_len, a string record past strbuf_len
    assert po.cells([b"/a/1"], t, sb, doc_tape, status, tape_len=int(doc_tape[1]) - 1)[1].tolist() == [[po.CAPACITY]]
    assert po.cells([b"/b"], t, sb, doc_tape, status, strbuf_len=len(sb) - 1)[1].tolist() == [[po.CAPACITY]]
    assert po.cells([b"/a/1"], t, sb, doc_tape, status, strbuf_len=len(sb) - 1)[1].tolist() == [[0]]
    # a container word that points past its slice
    t[1] = (t[1] & ~np.uint64(0xFFFFFFFF)) | np.uint64(int(doc_tape[1]) + 5)
    assert po.cells([b"/a/1", b""], t, sb, doc_tape, status)[1].tolist() == [[po.TAPE_ERROR], [0]]


# ---- 2. independent composition over decode_tape ------------------------------------------------------------------------

def resolve_decoded(v, toks):
    """The rules over oracle.decode_tape's python objects; returns (code, value)."""
    for tok in toks:
        if isinstance(v, tuple):
            hits = [x for k, x in v[1] if k.encode("utf-8", "surrogatepass") == tok]
            if not hits:
                return po.NO_SUCH_FIELD, None
            v = hits[0]
        elif isinstance(v, list):
            code, i = po.array_rule(tok)
            if code or i >= len(v):
                return code or po.INDEX_OUT_OF_BOUNDS, None
            v = v[i]
        else:
            return po.NO_SUCH_FIELD, None
    return 0, v


def paths(v, prefix=b"", out=None, depth=0):
    out = [] if out is None else out
    out.append(prefix)
    if depth < 6:
        if isinstance(v, tuple):
            for k, x in v[1][:6]:
                paths(x, prefix + b"/" + k.encode("utf-8", "surrogatepass").replace(b"~", b"~0").replace(b"/", b"~1"), out, depth + 1)
        elif isinstance(v, list):
            for i, x in list(enumerate(v))[:3] + list(enumerate(v))[-1:]:
                paths(x, prefix + b"/%d" % i, out, depth + 1)
            out.append(prefix + b"/%d" % len(v))
    return out


def test_composition_with_decode_tape():
    from mojo_simdjson_b200 import synth
    from tests.test_stage2_stream_oracle import WALK_TABLE

    data = bytes(synth.ndjson(64 << 10))
    tape, sb, doc_tape, status = stream_tapes(data)
    docs = [oracle.decode_tape(tape[int(doc_tape[d]) : int(doc_tape[d + 1])], sb) if int(status[d]) == ALL_ONES else None for d in range(status.size)]
    pointers = sorted(set(p for v in docs[:8] if v is not None for p in paths(v)))[:400]
    pointers += [b"/user/id", b"/entities/hashtags/0/text", b"/missing", b"/id/0", b"/entities/urls/-"]
    ty, code, val = po.cells(pointers, tape, sb, doc_tape, status)
    sbb = bytes(sb)
    for d, v in enumerate(docs):
        w = [int(x) for x in tape[int(doc_tape[d]) : int(doc_tape[d + 1])]]
        for k, p in enumerate(pointers):
            c, want = resolve_decoded(v, po.tokens(p))
            assert int(code[k, d]) == c, (d, p)
            if c == 0:
                assert cell_value(w, sbb, int(ty[k, d]), int(val[k, d])) == want, (d, p)
    assert len(WALK_TABLE) > 0   # the walk table's documents, which include failing ones
    for doc in WALK_TABLE:
        w1 = oracle.stage1(doc)
        if w1.error or w1.n == 0:
            continue
        s = so.stage2_walk_stream(doc, w1.indexes[: w1.n], w1.n)
        st = np.array([ALL_ONES if e == 0 else int(e) for e in s.doc_error.tolist()], dtype=np.uint64)
        ty, code, val = po.cells([b"", b"/0", b"/a"], s.tape, s.string_buf, s.doc_tape, st)
        for d in range(st.size):
            if s.doc_error[d]:
                assert (code[:, d] == s.doc_error[d]).all()
                continue
            v = oracle.decode_tape(s.slice(d), s.string_buf)
            for k, p in enumerate([b"", b"/0", b"/a"]):
                c, want = resolve_decoded(v, po.tokens(p))
                assert int(code[k, d]) == c, (doc, p)
                if c == 0:
                    w = [int(x) for x in s.slice(d)]
                    assert cell_value(w, bytes(s.string_buf), int(ty[k, d]), int(val[k, d])) == want


# ---- 3. fuzzing against json.loads and a plain RFC 6901 resolver ---------------------------------------------------------

def rfc6901(doc, pointer: str):
    """RFC 6901 over json.loads' objects, with this project's array rules; returns (code, value)."""
    if pointer == "":
        return 0, doc
    for raw in pointer[1:].split("/"):
        tok = raw.replace("~1", "/").replace("~0", "~")
        if isinstance(doc, dict):
            if tok not in doc:
                return po.NO_SUCH_FIELD, None
            doc = doc[tok]
        elif isinstance(doc, list):
            code, i = po.array_rule(tok.encode())
            if code or i >= len(doc):
                return code or po.INDEX_OUT_OF_BOUNDS, None
            doc = doc[i]
        else:
            return po.NO_SUCH_FIELD, None
    return 0, doc


KEY_CHARS = ["a", "b", "/", "~", "0", "1", "é", "中", " ", '"', "\\"]


def rand_value(r: random.Random, depth: int):
    c = r.random()
    if depth < 4 and c < 0.25:
        return {"".join(r.choice(KEY_CHARS) for _ in range(r.randint(0, 4))): rand_value(r, depth + 1) for _ in range(r.randint(0, 5))}
    if depth < 4 and c < 0.45:
        return [rand_value(r, depth + 1) for _ in range(r.randint(0, 12))]
    return r.choice([lambda: r.randint(-10**12, 10**12), lambda: round(r.uniform(-1e3, 1e3), 3), lambda: "".join(r.choice(KEY_CHARS) for _ in range(r.randint(0, 6))),
                     lambda: True, lambda: False, lambda: None])()


def json_paths(v, prefix=""):
    yield prefix
    if isinstance(v, dict):
        for k, x in v.items():
            yield from json_paths(x, prefix + "/" + k.replace("~", "~0").replace("/", "~1"))
    elif isinstance(v, list):
        for i, x in enumerate(v):
            yield from json_paths(x, prefix + f"/{i}")
        yield prefix + f"/{len(v)}"
        yield prefix + f"/{len(v) + 7}"


def to_python(v):
    if isinstance(v, tuple):
        return {k: to_python(x) for k, x in v[1]}
    if isinstance(v, list):
        return [to_python(x) for x in v]
    return v


def test_fuzz_against_json_loads():
    r = random.Random(0x501E7)
    values = []
    while len(values) < 2000:
        v = rand_value(r, 0)
        if v not in ({}, []):   # a root-level empty container is a TAPE_ERROR document (the reference's walk)
            values.append(v)
    docs = [json.dumps(v, ensure_ascii=r.random() < 0.5).encode() for v in values]
    tape, sb, doc_tape, status = stream_tapes(b"\n".join(docs))
    assert status.size == len(docs) and (status == ALL_ONES).all()
    sbb = bytes(sb)
    checked = 0
    for d, v in enumerate(values):
        ps = list(json_paths(v))
        picks = r.sample(ps, min(len(ps), 6))
        for p in list(picks):   # siblings with one byte changed
            if p:
                b = bytearray(p.encode())
                i = r.randrange(1, len(b)) if len(b) > 1 else 0
                b[i] = ord(r.choice("ab01/~-"))
                try:
                    picks.append(b.decode())
                except UnicodeDecodeError:
                    pass
        picks = [p for p in picks if po.check_call([p.encode()]) == 0]
        w = [int(x) for x in tape[int(doc_tape[d]) : int(doc_tape[d + 1])]]
        lo, hi = int(doc_tape[d]), int(doc_tape[d + 1])
        ty, code, val = po.cells([p.encode() for p in picks], tape[lo:hi], sb, np.array([0, hi - lo]), status[d : d + 1])
        for k, p in enumerate(picks):
            c, want = rfc6901(v, p)
            assert int(code[k, 0]) == c, (docs[d][:80], p)
            if c == 0:
                assert to_python(cell_value(w, sbb, int(ty[k, 0]), int(val[k, 0]))) == want, (docs[d][:80], p)
            checked += 1
    assert checked > 8000
