"""CPU tests of oracle/stage2_oracle.c -- the per-primitive half of the reference's stage 2 (strings, atoms, numbers).

What the reference's own tests hold for this path is only "stage2() returns SUCCESS" on four fixtures
(/root/reference/tests/test_stage_2.mojo:27-63); those are reproduced from the committed stage-1 golden file.  Everything
else is pinned against independent statements of the same rules: Python's json module for string unescaping and the
JSON / reference grammar written as regular expressions for numbers."""
import json
import os
import random
import re

import numpy as np

from oracle import oracle

HERE = os.path.dirname(os.path.abspath(__file__))
STAGE2_FIXTURES = ["simple_json.json", "simple_strings.json", "escaping.json", "escaping_very_long.json"]


def _fixture_inputs():
    with open(os.path.join(HERE, "golden", "stage1_fixtures.json")) as f:
        items = json.load(f)["fixtures"]
    out = {}
    for it in items:
        name = os.path.basename(it["file"])
        if name in STAGE2_FIXTURES:
            out[name] = it["input"].encode("utf-8")
    return out


def _strings_of(p):
    out = []
    for k in np.nonzero(p.kind == oracle.KIND_STRING)[0]:
        o = int(p.str_off[k])
        n = int(np.frombuffer(p.string_buf[o : o + 4].tobytes(), dtype=np.uint32)[0])
        assert n == p.value[k]
        out.append(p.string_buf[o + 4 : o + 4 + n].tobytes())
    return out


def test_reference_stage2_fixtures_every_primitive_succeeds():
    """tests/test_stage_2.mojo asserts error code 0 for these four inputs: every primitive must come out SUCCESS, and the
    string scanner as written (advance 32) must agree with the one that examines every byte (advance 8) on them."""
    inputs = _fixture_inputs()
    assert sorted(inputs) == sorted(STAGE2_FIXTURES)
    for name, data in inputs.items():
        w = oracle.stage1(data)
        assert w.error == 0
        p = oracle.stage2_primitives(data, w.indexes[: w.n])
        assert p.first_error == 0 and p.first_error_index == w.n, name
        assert not p.error.any()
        for k in np.nonzero(p.kind == oracle.KIND_STRING)[0]:
            start = int(w.indexes[k]) + 1
            a, enda = oracle.parse_string(data, start, 8)
            b, endb = oracle.parse_string(data, start, 32)
            assert a is not None and a == b and enda == endb, (name, k)
    # the values of escaping.json, by hand: keys and strings in document order
    data = inputs["escaping.json"]
    w = oracle.stage1(data)
    p = oracle.stage2_primitives(data, w.indexes[: w.n])
    assert _strings_of(p) == [b'\\"Nam[{', b"\\\\", b"true", b"t", b'\\"']
    ints = [int(p.value[k]) for k in np.nonzero(p.kind == oracle.KIND_INT)[0]]
    assert ints == [116] and (p.kind == oracle.KIND_FLOAT).sum() == 1 and (p.kind == oracle.KIND_FALSE).sum() == 1


def test_string_scanner_as_written_skips_bytes():
    """The reference loads 8 bytes and advances 32 (stringparsing_defs.mojo:10,40; string_parsing.mojo:384-385): a closing
    quote in a skipped gap is missed.  Recorded here so that the divergence of the product (every byte examined) is explicit."""
    tok = b'"abcdefghijklmnop" , "x"'
    assert oracle.parse_string(tok, 1, 8) == (b"abcdefghijklmnop", 17)
    assert oracle.parse_string(tok, 1, 32) != (b"abcdefghijklmnop", 17)
    # strings whose first 8 bytes hold the closing quote or a backslash that leads to it behave identically
    for tok in (b'"abcdefg" ', b'"" ', b'"\\n\\t" ', b'"\\u00e9" ', b'"abc\\"d" '):
        assert oracle.parse_string(tok, 1, 8) == oracle.parse_string(tok, 1, 32)


_PAIR = object()


def _walk_strings(obj, out):
    if isinstance(obj, list) and obj and isinstance(obj[0], tuple) and len(obj[0]) == 2 and obj[0][0] is _PAIR:
        for _, (k, v) in obj:
            out.append(k)
            _walk_strings(v, out)
    elif isinstance(obj, list):
        for v in obj:
            _walk_strings(v, out)
    elif isinstance(obj, str):
        out.append(obj)


def strings_in_document_order(doc_bytes: bytes):
    """Every key and string value of a JSON document in the order the text holds them (python's json as the independent parser)."""
    parsed = json.loads(doc_bytes.decode("utf-8"), object_pairs_hook=lambda pairs: [(_PAIR, p) for p in pairs])
    out = []
    _walk_strings(parsed, out)
    return out


def test_strings_against_python_json_on_the_synthetic_documents():
    from mojo_simdjson_b200 import synth

    for doc in (synth.twitter_like(), synth.status_array(300_000)):
        data = bytes(doc)
        w = oracle.stage1(data, impl="fast")
        assert w.error == 0
        p = oracle.stage2_primitives(data, w.indexes[: w.n])
        assert p.first_error == 0
        want = strings_in_document_order(data)
        got = _strings_of(p)
        assert len(got) == len(want)
        for g, s in zip(got, want):
            assert g == s.encode("utf-8", "surrogatepass")
        # integers agree with python's
        for k in np.nonzero(p.kind == oracle.KIND_INT)[0][:2000]:
            i = int(w.indexes[k])
            tok = re.match(rb"-?\d+", data[i:]).group(0)
            assert int(tok) == int(p.value[k])


def test_string_fuzz_against_python_json():
    rng = random.Random(0)
    alphabet = ["a", "Z", "0", " ", '"', "\\", "/", "\b", "\f", "\n", "\r", "\t", "\u00e9", "\u20ac", "\u65e5", "\U0001f600", "\x00", "\x1f", "\x7f",
                "\ud7ff", "\ue000", "\uffff"]
    for _ in range(3000):
        s = "".join(rng.choice(alphabet) for _ in range(rng.randrange(0, 40)))
        for ensure_ascii in (True, False):
            tok = json.dumps(s, ensure_ascii=ensure_ascii).encode("utf-8")
            if rng.random() < 0.3:   # upper-case hex digits and \/ are legal too
                tok = re.sub(rb"\\u([0-9a-f]{4})", lambda m: b"\\u" + m.group(1).upper(), tok).replace(b"/", b"\\/")
            data = b"[" + tok + b"]"
            got, end = oracle.parse_string(data, 2, 8)
            assert got == s.encode("utf-8"), (s, tok)
            assert end == len(data) - 2


def test_string_errors():
    bad = [rb'"\x"', rb'"\u12"', rb'"\u12G4"', rb'"\ud800"', rb'"\ud800\n"', rb'"\ud800A"', rb'"\udc00"', rb'"\udfff\ud800"', rb'"\a"', rb'"\U0041"',
           rb'"\u"', rb'"abc\\\u00"', rb'"\ud800\ud800"', rb'"\ud800A"']
    for tok in bad:
        assert oracle.parse_string(tok + b" ", 1, 8) == (None, None), tok
    good = {rb'"\ud83d\ude00"': "\U0001f600".encode(), rb'"\uD83D\uDE00"': "\U0001f600".encode(), rb'"\u0000"': b"\x00", rb'"\\\""': b'\\"',
            rb'"\/"': b"/", rb'"\udbff\udfff"': "\U0010ffff".encode(), rb'"\u00e9\u20AC"': "\u00e9\u20ac".encode(), rb'"\b\f\n\r\t"': b"\b\f\n\r\t"}
    for tok, want in good.items():
        assert oracle.parse_string(tok + b" ", 1, 8)[0] == want, tok
    # an unterminated string runs off the document: an error, not a read past the end
    assert oracle.parse_string(b'"abc', 1, 8) == (None, None)


def test_atoms():
    cases = {b"true,": ("true", True), b"true]": ("true", True), b"true": ("true", True), b"truex": ("true", False), b"tru": ("true", False),
             b"trux ": ("true", False), b"true\n": ("true", True), b"true\x00": ("true", False), b"false}": ("false", True), b"false": ("false", True),
             b"fals ": ("false", False), b"falsey": ("false", False), b"fxlse ": ("false", False), b"null ": ("null", True), b"null": ("null", True),
             b"nul": ("null", False), b"nulll": ("null", False), b"null:": ("null", True), b"true\x0c": ("true", False)}
    for data, (which, ok) in cases.items():
        assert oracle.atom_valid(data, 0, which) == ok, data


NUMBER_INT = re.compile(rb"-?[0-9]+$")
NUMBER_FLOAT = re.compile(rb"-?(?:[0-9]+\.?[0-9]*|\.[0-9]+)(?:[eE][+-]?[0-9]+)?$")


def number_tokens():
    rng = random.Random(1)
    pieces = ["-", "0", "1", "9", "12", ".", "e", "E", "+", "x", "00"]
    tokens = {"0", "-0", "123", "-123", "0123", "1.5", "-1.5e10", "1e5", "1E+5", "1e-5", "1.", "1.e3", "-", "-.5", "1e", "1e+", "1.2.3", "1ee5", "12x",
              "1-2", "9223372036854775807", "-9223372036854775808", "9223372036854775808", "18446744073709551616", "1.5x", "0x10", "1e5.5", "--1", "1+1"}
    for _ in range(4000):
        tokens.add("".join(rng.choice(pieces) for _ in range(rng.randrange(1, 7))))
    return sorted(t for t in tokens if t[:1] == "-" or t[:1].isdigit())


def test_numbers_against_the_restated_grammar():
    enders = [b",", b"]", b"}", b" ", b"\n", b":", b""]
    for t in number_tokens():
        tb = t.encode()
        for end in enders:
            err, isf, iv, tl = oracle.parse_number(tb + end, 0)
            m = re.match(rb"-?[0-9]*", tb)
            after = tb[m.end() : m.end() + 1]
            want_float = after in (b".", b"e", b"E")
            assert isf == want_float, (t, end)
            if want_float:
                assert tl == len(tb)
                ok = NUMBER_FLOAT.match(tb) is not None
                assert (err == 0) == ok, (t, end, err)
            else:
                ok = NUMBER_INT.match(tb) is not None
                assert (err == 0) == ok, (t, end, err)
                if ok:
                    v = int(tb)
                    assert iv == ((v + (1 << 63)) % (1 << 64)) - (1 << 63)   # 64-bit two's complement, as restated


def test_primitive_dispatch_and_first_error():
    data = b'[true, flase, "a\\qb", 12x, nul, 7, @, {"k": "v"}]'
    w = oracle.stage1(data)
    p = oracle.stage2_primitives(data, w.indexes[: w.n])
    kinds = [int(k) for k in p.kind if k != oracle.KIND_NONE]
    assert kinds == [oracle.KIND_TRUE, oracle.KIND_FALSE, oracle.KIND_STRING, oracle.KIND_INT, oracle.KIND_NULL, oracle.KIND_INT, oracle.KIND_BAD,
                     oracle.KIND_STRING, oracle.KIND_STRING]
    errs = [int(e) for e, k in zip(p.error, p.kind) if k != oracle.KIND_NONE]
    assert errs == [0, oracle.F_ATOM_ERROR, oracle.STRING_ERROR, oracle.NUMBER_ERROR, oracle.N_ATOM_ERROR, 0, oracle.TAPE_ERROR, 0, 0]
    assert p.first_error == oracle.F_ATOM_ERROR and data[w.indexes[p.first_error_index] :].startswith(b"flase")


# ------------------------------------------------------------------------------------------------
# the walk (SURVEY.md 8(f) rank 4): error codes of walk_document, and the tape against python's json
# ------------------------------------------------------------------------------------------------
def _as_pairs(obj):
    """python's json result in the shape oracle.decode_tape returns (objects as ("object", [(k, v), ...]))."""
    if isinstance(obj, list) and obj and isinstance(obj[0], tuple) and len(obj[0]) == 2 and obj[0][0] is _PAIR:
        return ("object", [(k, _as_pairs(v)) for _, (k, v) in obj])
    if isinstance(obj, _EmptyObject):
        return ("object", [])
    if isinstance(obj, list):
        return [_as_pairs(v) for v in obj]
    return obj


class _EmptyObject:
    pass


def python_document(data: bytes):
    parsed = json.loads(data.decode("utf-8"), object_pairs_hook=lambda pairs: [(_PAIR, p) for p in pairs] if pairs else _EmptyObject())
    return _as_pairs(parsed)


def walk(data: bytes):
    w = oracle.stage1(data, impl="fast" if len(data) > 20000 else "ref")
    assert w.error == 0, data[:60]
    return oracle.stage2_walk(data, w.indexes, w.n)


def same_document(a, b):
    """Equal up to float formatting: python parses floats exactly, the oracle with strtod -- both correctly rounded."""
    return a == b


def test_walk_tape_decodes_to_what_python_parses():
    from mojo_simdjson_b200 import synth

    docs = [b'[1, 2]', b'{ " hello " : " world " }', b'{"a": {"b": [1, 2, {"c": null}], "d": "x"}, "e": [[], {}, [[]], true, false, -7, 2.5e3]}',
            b'[[[[[[]]]]], {"k": {}}]', b'"just a string"', b"12345", b"-0", b"true", b"null", b'{"a":1,"a":2}',
            bytes(synth.twitter_like()), bytes(synth.status_array(200_000))]
    for data in docs:
        t = walk(data)
        assert t.error == 0, data[:60]
        assert same_document(oracle.decode_tape(t.tape, t.string_buf), python_document(data)), data[:60]
    for name, data in _fixture_inputs().items():   # what tests/test_stage_2.mojo asserts: error code 0
        assert walk(data).error == 0, name


def test_walk_error_codes():
    """Derived by hand from json_iterator.mojo:40-254 (state by state); includes the reference's own oddities: a root-level
    empty container is not consumed (:61-65, :72-76), so `{}` and `[]` end in TAPE_ERROR; arrays hit DEPTH_ERROR one level
    before objects (:177-180 vs :86-88)."""
    T, D = oracle.TAPE_ERROR, oracle.DEPTH_ERROR
    table = {
        b"{}": T, b"[]": T, b"[1]": 0, b'{"a":1}': 0, b"[1,]": T, b"[,1]": T, b"[1 2]": T, b'{"a" 1}': T, b'{"a":}': T, b"{1:2}": T, b'{"a":1,}': T,
        b'{"a":1 "b":2}': T, b"[1}": T, b'{"a":1]': T, b"[1] 2": T, b"1 2": T, b'"a" "b"': T, b"[[1]": T, b"[1]]": T, b'{"a":[}': T,
        b"[1,2": T, b'{"a":1': T, b"@": T, b"[@]": T, b"[tru]": oracle.T_ATOM_ERROR, b"[fals]": oracle.F_ATOM_ERROR, b"[nul]": oracle.N_ATOM_ERROR,
        b"[12x]": oracle.NUMBER_ERROR, b'["\\q"]': oracle.STRING_ERROR, b'{"\\q":1}': oracle.STRING_ERROR, b"[1, tru, 12x]": oracle.T_ATOM_ERROR,
        b"[12x, tru]": oracle.NUMBER_ERROR, b"[12x 3]": oracle.NUMBER_ERROR, b"[1 12x]": T, b"tru": oracle.T_ATOM_ERROR, b"-": oracle.NUMBER_ERROR,
        b'[{"a":[1,{"b":[]}]}]': 0, b"[[],[]]": 0, b"[{},{}]": 0, b'{"a":{},"b":[]}': 0, b"[1,[2,[3]],4]": 0, b'{"a":"b","c":"d"}': 0,
        b":": T, b",": T, b"]": T, b"}": T, b"[:]": T, b'{"a"::1}': T, b'{"a":1,,"b":2}': T, b"[1,,2]": T, b'[{"a":1},]': T,
    }
    for data, want in table.items():
        assert walk(data).error == want, (data, walk(data).error, want)
    # depth: arrays fail at depth 100, objects at depth 101
    for depth, want in ((98, 0), (99, 0), (100, D), (101, D)):
        assert walk(b"[" * depth + b"1" + b"]" * depth).error == want, depth
    for depth, want in ((99, 0), (100, 0), (101, D), (102, D)):
        assert walk(b'{"k":' * depth + b"1" + b"}" * depth).error == want, depth
    # mixed: 99 arrays, then an object at depth 100 is fine, an array is not
    assert walk(b"[" * 99 + b'{"k":1}' + b"]" * 99).error == 0
    assert walk(b"[" * 99 + b"[1]" + b"]" * 99).error == D


def test_walk_doubles_of_any_token_length():
    """A float token has no length limit: the tape holds its correctly rounded value however long the token is."""
    import struct

    long = [b"5e" + b"0" * 600, b"1." + b"0" * 600, b"1" + b"2" * 599 + b".0", b"0." + b"0" * 600 + b"1", b"-" + b"9" * 600 + b".5",
            b"1" * 600 + b"e-590"]
    assert all(len(t) >= 600 for t in long)
    toks = long + [b"1.5"] + [b"2.5e" + b"0" * (k - 5) + b"1" for k in (511, 512, 513)]   # 511 to 513 bytes
    t = walk(b"[" + b",".join(toks) + b"]")
    assert t.error == 0
    m = len(toks)
    assert t.tape.size == 2 * m + 4          # root, '[', a 'd' word and its payload per token, ']', root
    assert [int(x) >> 56 for x in t.tape[2 : 2 + 2 * m : 2]] == [ord("d")] * m
    assert [int(x) for x in t.tape[3 : 3 + 2 * m : 2]] ==[struct.unpack("<Q", struct.pack("<d", float(tok)))[0] for tok in toks]
