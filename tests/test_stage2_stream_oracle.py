"""CPU checks of the stream oracle (tests/stage2_stream_oracle.c): stage 2 over a stream of documents, split by bracket
depth, every document walked alone.  It must equal an independent composition in Python -- oracle.document_starts, then
oracle.stage2_walk per document with its trailer, string words rebased onto the stream's string buffer -- and hold the
points of the definition in include/simdjson_b200.h (sjb200_stage2_stream)."""
import random

import numpy as np

from oracle import oracle
from tests import stage2_stream_oracle as so

T, D = oracle.TAPE_ERROR, oracle.DEPTH_ERROR

# the single-document walk's error table (tests/test_stage2_oracle.py, test_walk_error_codes) and a few deeper documents
WALK_TABLE = [b"{}", b"[]", b"[1]", b'{"a":1}', b"[1,]", b"[,1]", b"[1 2]", b'{"a" 1}', b'{"a":}', b"{1:2}", b'{"a":1,}', b'{"a":1 "b":2}', b"[1}",
              b'{"a":1]', b"[1] 2", b"1 2", b'"a" "b"', b"[[1]", b"[1]]", b'{"a":[}', b"[1,2", b'{"a":1', b"@", b"[@]", b"[tru]", b"[fals]", b"[nul]",
              b"[12x]", b'["\\q"]', b'{"\\q":1}', b"[1, tru, 12x]", b"[12x, tru]", b"[12x 3]", b"[1 12x]", b"tru", b"-", b'[{"a":[1,{"b":[]}]}]',
              b"[[],[]]", b"[{},{}]", b'{"a":{},"b":[]}', b"[1,[2,[3]],4]", b'{"a":"b","c":"d"}', b":", b",", b"]", b"}", b"[:]", b'{"a"::1}',
              b'{"a":1,,"b":2}', b"[1,,2]", b'[{"a":1},]', b"[" * 100 + b"1" + b"]" * 100, b'{"k":' * 101 + b"1" + b"}" * 101,
              b"[" * 99 + b'{"k":1}' + b"]" * 99, b"[" * 99 + b"[1]" + b"]" * 99]


def index(data: bytes):
    w = oracle.stage1(data, impl="fast" if len(data) > 20000 else "ref")
    assert w.error == 0 and w.n, data[:60]
    return w.indexes, w.n


def token_words(data: bytes, idx) -> np.ndarray:
    a = np.frombuffer(data, dtype=np.uint8)
    b = oracle.structural_bytes(a, idx)
    w = np.zeros(b.size, dtype=np.int64)
    w[np.isin(b, np.frombuffer(b'"{}[]tfn', dtype=np.uint8))] = 1
    w[np.isin(b, np.frombuffer(b"-0123456789", dtype=np.uint8))] = 2
    return w


def composed(data: bytes, idx, n: int):
    """The independent composition: (first, tape_off, errors, {d: slice of a successful document}, string buffer)."""
    idx = np.asarray(idx[:n], dtype=np.uint32)
    starts = oracle.document_starts(oracle.structural_bytes(data, idx))
    first = np.append(np.nonzero(starts)[0], n).astype(np.int64)
    words = token_words(data, idx)
    cw = np.concatenate([[0], np.cumsum(words)])
    nd = first.size - 1
    off = cw[first] + 2 * np.arange(nd + 1)
    p = oracle.stage2_primitives(data, idx)
    errs, slices = [], {}
    for d in range(nd):
        f, e = int(first[d]), int(first[d + 1])
        sub = np.concatenate([idx[f:e], np.array([len(data), len(data), 0], dtype=np.uint32)])
        w = oracle.stage2_walk(data, sub, e - f)
        errs.append(w.error)
        if w.error == 0:
            s = w.tape.copy()
            strs = [k for k in range(f, e) if p.kind[k] == oracle.KIND_STRING]
            base = int(p.str_off[strs[0]]) if strs else 0
            j = 1
            while j < s.size - 1:
                ty = int(s[j]) >> 56
                if ty == ord('"'):
                    s[j] += np.uint64(base)
                j += 2 if ty in (ord("l"), ord("d")) else 1
            assert s.size == off[d + 1] - off[d]
            slices[d] = s
    return first, off, errs, slices, p.string_buf


def check(data: bytes):
    idx, n = index(data)
    got = so.stage2_walk_stream(data, idx, n)
    first, off, errs, slices, sbuf = composed(data, idx, n)
    assert np.array_equal(got.doc_first.astype(np.int64), first), data[:80]
    assert np.array_equal(got.doc_tape.astype(np.int64), off), data[:80]
    assert got.doc_error.tolist() == errs, data[:80]
    for d, s in slices.items():
        assert np.array_equal(got.slice(d), s), (data[:80], d)
    assert np.array_equal(got.string_buf, sbuf)
    return got


def test_error_table_joined_three_ways():
    for a in WALK_TABLE:
        for b in WALK_TABLE[:20]:
            check(a + b"\n" + b + b"\n" + b'{"ok":[1,"s"]}')
            check(b'"x"' + b" " + a + b" " + b)
            if a[-1:] in (b"]", b"}", b'"') or b[:1] in (b"[", b"{", b'"'):   # no separator where the tokens stay apart
                check(a + b + b'["z"]')


def test_fuzzed_streams():
    rng = random.Random(11)
    atoms = ['1', '-2', '3.5', 'true', 'false', 'null', '"s"', '"k"', '12x', 'tru', '"\\\\q"', '{}', '[]']

    def gen(depth):
        r = rng.random()
        if depth > 4 or r < 0.35:
            return rng.choice(atoms)
        if r < 0.7:
            return "[" + ",".join(gen(depth + 1) for _ in range(rng.randrange(0, 5))) + "]"
        return "{" + ",".join('"k%d":%s' % (i, gen(depth + 1)) for i in range(rng.randrange(0, 4))) + "}"

    mut = [",", ":", "[", "]", "{", "}", '"x"', "1", " ", ""]
    done = 0
    while done < 2000:
        docs = []
        for _ in range(rng.randrange(1, 6)):
            s = gen(0)
            for _ in range(rng.randrange(0, 2)):
                p = rng.randrange(0, len(s) + 1)
                s = s[:p] + rng.choice(mut) + s[p + rng.randrange(0, 2):]
            docs.append(s)
        data = rng.choice(["\n", " ", ""]).join(docs).encode()
        w = oracle.stage1(data)
        if w.error != 0 or not w.n:
            continue
        check(data)
        done += 1


def test_definition_points():
    g = check(b"1 2")
    assert g.doc_first.tolist() == [0, 1, 2] and g.doc_error.tolist() == [0, 0]
    g = check(b"[1][2]")
    assert g.doc_first.tolist() == [0, 3, 6] and g.doc_error.tolist() == [0, 0]
    g = check(b"{}\n[1]")
    assert g.doc_error.tolist() == [T, 0]
    assert oracle.decode_tape(g.slice(1), g.string_buf) == [1]
    g = check(b"[1] ] [2] 3")                  # a stray close starts a failing document; the depth is -1 until the next '['
    assert g.doc_first.tolist() == [0, 3, 5, 6, 8] and g.doc_error.tolist() == [0, T, 0, T]
    g = check(b'[1] ] 2 [ "s"')                 # everything up to where the depth returns to 0 belongs to the stray close
    assert g.doc_first.tolist() == [0, 3, 6, 7] and g.doc_error.tolist() == [0, T, 0]
    g = check(b'"a" [1, [2')                     # an unclosed last document swallows the rest
    assert g.doc_first.tolist() == [0, 1, 6] and g.doc_error.tolist() == [0, T]
    deep = b"[" * 101 + b"1" + b"]" * 101
    g = check(b'{"a":1}\n' + deep + b'\n["x", {"y": null}]')
    assert g.doc_error.tolist() == [0, D, 0]
    assert oracle.decode_tape(g.slice(2), g.string_buf) == ["x", ("object", [("y", None)])]
    assert oracle.decode_tape(g.slice(0), g.string_buf) == ("object", [("a", 1)])
    # slice lengths do not depend on the verdict
    assert int(g.doc_tape[2] - g.doc_tape[1]) == 2 + 2 * 101 + 2
