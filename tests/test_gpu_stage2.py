"""GPU parity tests of the per-primitive half of stage 2 (sjb200_stage2_primitives_device_async, SURVEY.md 8(f) rank 3)
against oracle/stage2_oracle.c: kind, error code, value, string-record offsets, the string buffer and the first error,
bit for bit, on the reference's stage-2 fixtures, the synthetic documents and corpora of corner-case tokens."""
import json
import os

import numpy as np
import pytest

from oracle import oracle
from tests import test_gpu_stage2_scale as scale
from tests import test_stage2_oracle as cpu

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")


@pytest.fixture(scope="module")
def dev():
    from mojo_simdjson_b200 import device

    ctx = device.Stage1Context(0, max_len=(1 << 32) - 1)
    yield ctx
    ctx.close()


def check(dev, data: bytes, mis: int = 0):
    """stage 1 on the device, then the primitives kernel on its index array; everything compared with the oracle."""
    a = np.frombuffer(data, dtype=np.uint8)
    store = torch.full((mis + a.size + 64,), 0x22, dtype=torch.uint8, device="cuda")   # hostile bytes around the document
    d_in = store[mis : mis + a.size]
    d_in.copy_(torch.from_numpy(a.copy()))
    d_idx = torch.empty(a.size + 8, dtype=torch.int32, device="cuda")
    res = dev.index(d_in, d_idx)
    w = oracle.stage1(data, impl="fast" if a.size > 20000 else "ref")
    assert res.error == w.error
    n = res.n_written if res.n is None else res.n
    assert n == (w.n if w.n is not None else w.n_written)
    want = oracle.stage2_primitives(data, w.indexes[:n])
    got = dev.stage2_primitives(d_in, d_idx, n)
    torch.cuda.synchronize()
    assert np.array_equal(got["kind"].cpu().numpy(), want.kind)
    assert np.array_equal(got["error"].cpu().numpy(), want.error)
    assert np.array_equal(got["value"].cpu().numpy(), want.value)
    is_str = want.kind == oracle.KIND_STRING
    assert np.array_equal(got["str_off"].cpu().numpy().astype(np.uint64)[is_str], want.str_off[is_str])
    summary = got["summary"].cpu().numpy()
    if want.first_error == 0:
        assert summary[0] == -1
    else:
        assert int(summary[0]) == (want.first_error_index << 8 | want.first_error)
    assert int(summary[1]) == want.string_buf.size
    assert np.array_equal(got["string_buf"][: want.string_buf.size].cpu().numpy(), want.string_buf)
    return want


def test_reference_stage2_fixtures(dev):
    for name, data in cpu._fixture_inputs().items():
        want = check(dev, data)
        assert want.first_error == 0, name   # what tests/test_stage_2.mojo asserts


def test_synthetic_documents(dev):
    from mojo_simdjson_b200 import synth

    for doc in (synth.twitter_like(), synth.status_array(2 << 20), synth.ndjson(1 << 20)):
        for mis in (0, 3):
            want = check(dev, bytes(doc), mis)
            assert want.first_error == 0
    # and against python's json, end to end on the GPU output
    data = bytes(synth.twitter_like())
    want = check(dev, data)
    assert cpu._strings_of(want) == [s.encode("utf-8", "surrogatepass") for s in cpu.strings_in_document_order(data)]


def test_string_corner_cases(dev):
    toks = [b'""', b'"a"', b'"\\n"', b'"\\u0041"', b'"\\ud83d\\ude00"', b'"\\uD83D\\uDE00x"', b'"\\\\"', b'"\\""', b'"\\/"', b'"\\b\\f\\n\\r\\t"',
            b'"\\u0000"', b'"\\udbff\\udfff"', "\"日本語\"".encode(), b'"' + b"x" * 300 + b'"', b'"' + b"\\\\" * 100 + b'"',
            b'"' + b"\\u00e9" * 50 + b'"', b'"abc\\u20acdef"']
    bad = [b'"\\x"', b'"\\u12G4"', b'"\\ud800"', b'"\\ud800\\n"', b'"\\udc00"', b'"\\udfff\\ud800"', b'"\\a"', b'"\\U0041"', b'"\\ud800\\ud800"',
           b'"\\u00"']
    want = check(dev, b"[" + b", ".join(toks) + b"]")
    assert want.first_error == 0 and (want.kind == oracle.KIND_STRING).sum() == len(toks)
    for k, b in enumerate(bad):
        items = toks[:k] + [b] + toks[k:]
        want = check(dev, b"[" + b",".join(items) + b"]", mis=k % 5)
        assert want.first_error == oracle.STRING_ERROR and (want.error != 0).sum() == 1
    want = check(dev, b"[" + b",".join(toks + bad) + b"]")
    assert (want.error == oracle.STRING_ERROR).sum() == len(bad)
    # a string that ends at the very end of the buffer, and one that is cut off (stage 1 says UNCLOSED_STRING; the kernel must not read on)
    check(dev, b'"abc"')
    check(dev, b'["abc')
    check(dev, b'["abc\\')
    check(dev, b'["abc\\u12')


def test_numbers_and_atoms(dev):
    toks = [t.encode() for t in cpu.number_tokens()]
    for sep in (b",", b" ,", b"\n,"):
        want = check(dev, b"[" + sep.join(toks) + b"]")
        assert (want.kind == oracle.KIND_INT).sum() + (want.kind == oracle.KIND_FLOAT).sum() >= len(toks) // 2
    atoms = [b"true", b"false", b"null", b"tru", b"truex", b"falsey", b"fals", b"nul", b"nulll", b"t", b"f", b"n", b"txue", b"fxlse", b"nxll", b"True",
             b"@", b"abc", b"\xc3\xa9", b"-", b"+1", b".5"]
    want = check(dev, b"[" + b", ".join(atoms) + b"]")
    assert (want.kind == oracle.KIND_BAD).sum() >= 5
    for t in (b"true", b"false", b"null", b"tru", b"nul", b"12", b"-", b"1.5", b"1e", b'"x"'):   # the primitive is the whole document / its tail
        check(dev, t)
        check(dev, b"[" + t)


def test_first_error_is_the_first_in_index_order(dev):
    from mojo_simdjson_b200 import synth

    doc = bytearray(bytes(synth.status_array(1 << 20)))
    w = oracle.stage1(bytes(doc), impl="fast")
    idx = w.indexes[: w.n]
    p = oracle.stage2_primitives(bytes(doc), idx)
    strs = np.nonzero(p.kind == oracle.KIND_STRING)[0]
    # break an early and a late string's first character into a bogus escape; the early one must be reported
    for k in (strs[len(strs) // 3], strs[len(strs) // 2], strs[-5]):
        i = int(idx[k]) + 1
        if doc[i] != ord('"') and doc[i + 1] not in (ord('"'), ord("\\")):
            doc[i] = ord("\\")
            doc[i + 1] = ord("q")
    want = check(dev, bytes(doc))
    assert want.first_error == oracle.STRING_ERROR and (want.error != 0).sum() >= 2
    assert want.first_error_index == int(np.nonzero(want.error)[0][0])


def test_empty_index_array(dev):
    d_in = torch.full((64,), 0x20, dtype=torch.uint8, device="cuda")
    d_idx = torch.zeros(8, dtype=torch.int32, device="cuda")
    got = dev.stage2_primitives(d_in, d_idx, 0)
    torch.cuda.synchronize()
    assert got["summary"].cpu().tolist()[:2] == [-1, 0]


# ------------------------------------------------------------------------------------------------
# the walk (SURVEY.md 8(f) rank 4): verdict of walk_document and the tape, against oracle_stage2_walk and python's json
# ------------------------------------------------------------------------------------------------
def run_walk(dev, data: bytes, mis: int = 0):
    a = np.frombuffer(data, dtype=np.uint8)
    store = torch.full((mis + a.size + 64,), 0x22, dtype=torch.uint8, device="cuda")
    d_in = store[mis : mis + a.size]
    d_in.copy_(torch.from_numpy(a.copy()))
    d_idx = torch.empty(a.size + 8, dtype=torch.int32, device="cuda")
    res = dev.index(d_in, d_idx)
    w = oracle.stage1(data, impl="fast" if a.size > 20000 else "ref")
    assert res.error == w.error == 0 and res.n == w.n, data[:60]
    want = oracle.stage2_walk(data, w.indexes, w.n)
    prims = dev.stage2_primitives(d_in, d_idx, res.n)
    tape, summary = dev.stage2_tape(d_in, d_idx, res.n, prims)
    torch.cuda.synchronize()
    s = summary.cpu().numpy()
    got_err = 0 if s[0] == -1 else int(s[0]) & 0xFF
    assert got_err == want.error, (data[:80], got_err, want.error, int(s[0]) >> 16)
    if want.error == 0:
        assert int(s[2]) == want.tape.size
        got = tape[: want.tape.size].cpu().numpy().view(np.uint64)
        # double payloads: the kernel's conversion, restated bit for bit (python's float() where it is exact)
        p = oracle.stage2_primitives(data, w.indexes[: w.n])
        exp, n_inexact, _ = scale.expected_tape(a, w.indexes[: w.n], p, want)
        assert np.array_equal(got, exp), data[:80]
        assert int(s[3]) == n_inexact, data[:80]
        assert np.array_equal(prims["string_buf"][: want.string_buf.size].cpu().numpy(), want.string_buf)
        return got, prims["string_buf"][: want.string_buf.size].cpu().numpy(), int(s[3])
    return None, None, 0


def test_walk_error_codes_on_the_gpu(dev):
    T, D = oracle.TAPE_ERROR, oracle.DEPTH_ERROR
    docs = [b"{}", b"[]", b"[1]", b'{"a":1}', b"[1,]", b"[,1]", b"[1 2]", b'{"a" 1}', b'{"a":}', b"{1:2}", b'{"a":1,}', b'{"a":1 "b":2}', b"[1}", b'{"a":1]',
            b"[1] 2", b"1 2", b'"a" "b"', b"[[1]", b"[1]]", b'{"a":[}', b"[1,2", b'{"a":1', b"@", b"[@]", b"[tru]", b"[fals]", b"[nul]", b"[12x]", b'["\\q"]',
            b'{"\\q":1}', b"[1, tru, 12x]", b"[12x, tru]", b"[12x 3]", b"[1 12x]", b"tru", b"-", b'[{"a":[1,{"b":[]}]}]', b"[[],[]]", b"[{},{}]",
            b'{"a":{},"b":[]}', b"[1,[2,[3]],4]", b'{"a":"b","c":"d"}', b":", b",", b"]", b"}", b"[:]", b'{"a"::1}', b'{"a":1,,"b":2}', b"[1,,2]",
            b'[{"a":1},]', b"{} }", b"[] ]", b'[{"a" "b"}]', b'{"a":{"b":1 2}}', b'[[1,2],[3 4]]', b'{"a":[1,2,{"b":]}]}', b'[1,{"a":1,"b"}]',
            b'["a":1]', b'{"a":1:2}', b"[[[[]]]]", b"[[[[]]]", b'[{"a":[{"b":[{"c":{}}]}]}]']
    for data in docs:
        run_walk(dev, data, mis=len(data) % 4)
    for depth in (98, 99, 100, 101, 130, 300):
        run_walk(dev, b"[" * depth + b"1" + b"]" * depth)
        run_walk(dev, b'{"k":' * depth + b"1" + b"}" * depth)
    run_walk(dev, b"[" * 99 + b'{"k":1}' + b"]" * 99)
    run_walk(dev, b"[" * 99 + b"[1]" + b"]" * 99)
    run_walk(dev, b"[" * 99 + b"[]" + b"]" * 99)      # an empty container does not count as a level


def test_walk_tapes_against_the_oracle_and_python(dev):
    from mojo_simdjson_b200 import synth

    docs = [b"[1, 2]", b'{ " hello " : " world " }', b'{"a": {"b": [1, 2, {"c": null}], "d": "x"}, "e": [[], {}, [[]], true, false, -7, 2.5e3]}',
            b'[[[[[[]]]]], {"k": {}}]', b'"just a string"', b"12345", b"-0", b"true", b"null", b'{"a":1,"a":2}', b"[0.1, 1e22, 123456789012345678, 1.5e-7, -2.25]",
            bytes(synth.twitter_like()), bytes(synth.status_array(3 << 20))]
    for data in docs:
        tape, sbuf, inexact = run_walk(dev, data)
        assert tape is not None, data[:60]
        if inexact == 0:
            assert oracle.decode_tape(tape, sbuf) == cpu.python_document(data), data[:60]
    for name, data in cpu._fixture_inputs().items():
        tape, _, _ = run_walk(dev, data)
        assert tape is not None, name        # tests/test_stage_2.mojo: error code 0
    # doubles outside the exact fast path are counted, never silently approximated
    _, _, inexact = run_walk(dev, b"[0.1234567890123456789, 1e300, 3.5]")
    assert inexact == 2


def test_walk_fuzz(dev):
    """Random token soups around valid documents: the GPU verdict must be the sequential walk's on every one of them."""
    import random

    rng = random.Random(7)
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
    while done < 500:
        s = gen(0)
        for _ in range(rng.randrange(0, 3)):
            p = rng.randrange(0, len(s) + 1)
            s = s[:p] + rng.choice(mut) + s[p + rng.randrange(0, 2):]
        data = s.encode()
        w = oracle.stage1(data)
        if w.error != 0 or not w.n:
            continue
        run_walk(dev, data)
        done += 1


def test_facade_stage1_then_stage2_like_the_reference_test():
    """tests/test_stage_2.mojo:27-44, on the same four fixtures: stage1 -> 0, stage2 -> 0, dump_raw_tape succeeds; here also:
    the tape decodes to what python's json parses (the reference test imports json.loads and stops there)."""
    from mojo_simdjson_b200 import synth
    from mojo_simdjson_b200.dom_parser_implementation import DomParserImplementation

    parser = DomParserImplementation(0, max_len=8 << 20)
    try:
        docs = dict(cpu._fixture_inputs())
        docs["twitter"] = bytes(synth.twitter_like())
        docs["statuses"] = bytes(synth.status_array(1 << 20))
        for name, data in docs.items():
            assert parser.stage1(data) == 0, name
            assert parser.stage2() == 0, name
            text, ok = parser.document.dump_raw_tape()
            assert ok and text.startswith("0 : r"), name
            if parser.document.inexact_doubles == 0:
                assert oracle.decode_tape(parser.document.tape, parser.document.string_buf) == cpu.python_document(data), name
            w = oracle.stage1(data, impl="fast")
            want = oracle.stage2_walk(data, w.indexes, w.n)
            assert np.array_equal(parser.document.tape, want.tape) and np.array_equal(parser.document.string_buf, want.string_buf), name
        # verdicts through the facade
        for data, want in ((b"[1,]", 3), (b'{"a":tru}', 6), (b"[" * 120 + b"]" * 120, 4), (b'["\\q"]', 5), (b"[12x]", 9), (b"{}", 3)):
            assert parser.stage1(data) == 0
            assert parser.stage2() == want, data
        assert parser.stage1(b'"abc') == 15          # stage 1 fails: stage 2 has nothing to walk
        assert parser.stage2() == 12
    finally:
        parser.close()
