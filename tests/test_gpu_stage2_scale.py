"""GPU tests of the stage-2 walk (csrc/stage2_primitives.cuh, csrc/stage2_tape.cuh) where small documents cannot reach:

  A  documents past one iteration of the single-CTA scans (more than 1024 blocks of 2048 tokens), past one iteration of the
     multisplit histogram scan (more than 16384 tiles of 2048 tokens), and the bracket stack carried across that boundary
  B  containers of 2^24 - 1 and 2^24 elements: the count field of an open word has 24 bits, one element more is CAPACITY
  C  short valid and invalid probes with their first token at every position around a CTA boundary of the grammar kernel
  D  every double payload bit for bit, against a restatement of s2_double_bits and python's correctly rounded float()
  E  caller buffers that are too small for the tape or the string records

Everything is compared strictly with oracle/stage2_oracle.c: the primitives arrays, the verdict, the tape word for word and
the string buffer; where a test plants an error, also the index of the token the kernel reports it at.  Large documents
assert the sizes they claim to cover, so that a change to a generator cannot shrink the coverage unnoticed."""
import ctypes as C
import random
import struct

import numpy as np
import pytest

from oracle import oracle

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

TAPE_BLOCK = 2048                 # tokens per CTA of the tape kernels and per block of the scans (256 threads x 8)
SCAN_ITER = 1024 * TAPE_BLOCK     # tokens one iteration of the single-CTA scans covers (tape_stack_scan_kernel, scan_of_totals_kernel)
MS_TILE = 2048                    # tokens per multisplit tile
MS_ITER_TILES = 16384             # the histogram scan covers 128 classes x ntiles entries, 1024 blocks of 2048 per iteration
MAX_COUNT = 0xFFFFFF              # largest element count the tape stores (tape_builder.mojo:239-241)
CAPACITY = 1


@pytest.fixture(scope="module")
def dev():
    from mojo_simdjson_b200 import device

    ctx = device.Stage1Context(0, max_len=(1 << 32) - 1)
    yield ctx
    ctx.close()


# ------------------------------------------------------------------------------------------------
# s2_double_bits (stage2_tape.cuh:335-388), restated
# ------------------------------------------------------------------------------------------------
_P10 = [float(10**i) for i in range(23)]   # P10[] of :372, 1e0 .. 1e22: every entry is exact in binary64


def _bits(d: float) -> int:
    return struct.unpack("<Q", struct.pack("<d", d))[0]


def s2_double_bits(tok: bytes) -> tuple[int, bool]:
    """(IEEE-754 bits, inexact) of a float token as the kernel computes them.  Exact where Clinger's fast path applies; the
    slow path is plain binary64 arithmetic (no FMA, no fast-math), which python's float arithmetic performs identically."""
    neg = tok[:1] == b"-"                                          # :336
    p, n = (1 if neg else 0), len(tok)
    mant = digits = dropped = frac = 0
    seen_nonzero = inexact = False

    def run(p, is_frac):                                           # take() of :342-356 over one digit run
        nonlocal mant, digits, dropped, frac, seen_nonzero, inexact
        while p < n and 48 <= tok[p] <= 57:
            ch = tok[p]
            if ch != 48:
                seen_nonzero = True
            if seen_nonzero:
                if digits < 19:                                    # the mantissa keeps 19 significant digits
                    mant = mant * 10 + ch - 48
                    digits += 1
                    if is_frac:
                        frac += 1
                else:                                              # later ones are dropped: inexact unless '0'
                    if ch != 48:
                        inexact = True
                    if not is_frac:
                        dropped += 1
            elif is_frac:                                          # leading zeros of the fraction shift the exponent
                frac += 1
            p += 1
        return p

    p = run(p, False)                                              # :357
    if p < n and tok[p] == 46:                                     # :358-361
        p = run(p + 1, True)
    e10 = 0
    if p < n and tok[p] in b"eE":                                  # :363-370
        p += 1
        eneg = tok[p : p + 1] == b"-"
        if tok[p : p + 1] in (b"+", b"-"):
            p += 1
        ev = 0
        while p < n and 48 <= tok[p] <= 57:
            if ev < 100000:                                        # the exponent clamp: stops growing once >= 100000
                ev = ev * 10 + tok[p] - 48
            p += 1
        e10 = -ev if eneg else ev
    e10 += dropped - frac                                          # :371
    if mant == 0:                                                  # :374-375
        d = 0.0
    elif mant < (1 << 53) and -22 <= e10 <= 22:                    # :376-378, the fast path: one correctly rounded operation
        d = float(mant)
        d = d / _P10[-e10] if e10 < 0 else d * _P10[e10]
    else:                                                          # :379-385, steps of at most 1e22
        inexact = True
        d = float(mant)                                            # (double) of a uint64: round to nearest even, as float(int)
        e = e10
        while e > 0 and d != float("inf"):                         # (inf and 0 are fixed points of the remaining steps)
            s = min(e, 22)
            d *= _P10[s]
            e -= s
        while e < 0 and d != 0.0:
            s = min(-e, 22)
            d /= _P10[s]
            e += s
    if neg:
        d = -d
    return _bits(d), inexact


_restated: dict[bytes, tuple[int, bool]] = {}


def restated(tok: bytes) -> tuple[int, bool]:
    r = _restated.get(tok)
    if r is None:
        r = _restated[tok] = s2_double_bits(tok)
    return r


def tape_positions(data: np.ndarray, idx: np.ndarray, p: "oracle.Stage2Primitives") -> np.ndarray:
    """Tape index of the first word of every token of a document that walks to SUCCESS (commas and colons append none)."""
    b = oracle.structural_bytes(data, idx)
    w = np.zeros(idx.size, dtype=np.int64)
    w[np.isin(b, np.frombuffer(b"[]{}", dtype=np.uint8))] = 1
    w[np.isin(p.kind, (oracle.KIND_STRING, oracle.KIND_TRUE, oracle.KIND_FALSE, oracle.KIND_NULL))] = 1
    w[np.isin(p.kind, (oracle.KIND_INT, oracle.KIND_FLOAT))] = 2
    return 1 + np.cumsum(w) - w


def expected_tape(data: np.ndarray, idx: np.ndarray, p: "oracle.Stage2Primitives", want: "oracle.Stage2Tape"):
    """The oracle's tape with every double payload replaced by the restated kernel's bits; also the number of doubles the
    restatement flags inexact and, per double, (token, restated bits, inexact).  Checks on the way that the oracle's payload
    (strtod) is python's float() of the token."""
    t = want.tape.copy()
    ks = np.nonzero(p.kind == oracle.KIND_FLOAT)[0]
    pos = tape_positions(data, idx, p)[ks]
    assert np.all(t[pos] == np.uint64(ord("d") << 56))
    doubles, n_inexact = [], 0
    for k, q in zip(ks.tolist(), pos.tolist()):
        i = int(idx[k])
        tok = data[i : i + int(p.value[k])].tobytes()
        bits, inexact = restated(tok)
        assert int(t[q + 1]) == _bits(float(tok)), tok
        t[q + 1] = bits
        n_inexact += inexact
        doubles.append((tok, bits, inexact))
    return t, n_inexact, doubles


# ------------------------------------------------------------------------------------------------
# one document through stage 1 and both halves of stage 2 on the device, everything compared with the oracle
# ------------------------------------------------------------------------------------------------
class Walked:
    def __init__(self, n, error, error_index, tape, doubles):
        self.n, self.error, self.error_index, self.tape, self.doubles = n, error, error_index, tape, doubles

    @property
    def ntiles(self):
        return -(-self.n // MS_TILE)


def walk_on_gpu(dev, data) -> Walked:
    a = np.frombuffer(data, dtype=np.uint8) if isinstance(data, (bytes, bytearray)) else data
    w = oracle.stage1(a, impl="fast")
    assert w.error == 0
    n = w.n
    d_in = torch.from_numpy(a if a.flags.writeable else a.copy()).to("cuda")
    d_idx = torch.empty(a.size + 8, dtype=torch.int32, device="cuda")
    res = dev.index(d_in, d_idx)
    assert res.error == 0 and res.n == n
    assert np.array_equal(d_idx[: n + 3].cpu().numpy().view(np.uint32), w.indexes)   # stage 2 is what is under test here
    prims = dev.stage2_primitives(d_in, d_idx, n)
    tape, summary = dev.stage2_tape(d_in, d_idx, n, prims)
    torch.cuda.synchronize()
    # the primitives: kind, error, value, string record offsets, first failing primitive, record bytes, the records
    p = oracle.stage2_primitives(a, w.indexes[:n])
    assert np.array_equal(prims["kind"].cpu().numpy(), p.kind)
    assert np.array_equal(prims["error"].cpu().numpy(), p.error)
    assert np.array_equal(prims["value"].cpu().numpy(), p.value)
    is_str = p.kind == oracle.KIND_STRING
    assert np.array_equal(prims["str_off"].cpu().numpy().view(np.uint64)[is_str], p.str_off[is_str])
    ps = prims["summary"].cpu().numpy()
    assert int(ps[0]) == (-1 if p.first_error == 0 else (p.first_error_index << 8 | p.first_error))
    assert int(ps[1]) == p.string_buf.size
    assert np.array_equal(prims["string_buf"][: p.string_buf.size].cpu().numpy(), p.string_buf)
    # the walk
    want = oracle.stage2_walk(a, w.indexes, n)
    s = summary.cpu().numpy()
    error = 0 if s[0] == -1 else int(s[0]) & 0xFF
    assert error == want.error, (error, want.error, int(s[0]) >> 16)
    if error:
        return Walked(n, error, int(s[0]) >> 16, None, None)
    N = want.tape.size
    assert int(s[2]) == N and int(s[1]) == N - 2
    exp, n_inexact, doubles = expected_tape(a, w.indexes[:n], p, want)
    got = tape[:N].cpu().numpy().view(np.uint64)
    assert np.array_equal(got, exp)
    assert int(s[3]) == n_inexact
    assert np.array_equal(want.string_buf, p.string_buf)   # on SUCCESS the walk's records are the primitives', in index order
    return Walked(n, 0, None, got, doubles)


# ------------------------------------------------------------------------------------------------
# A: past one scan iteration
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mib", [16, 256])
def test_status_array_past_one_scan_iteration(dev, mib):
    from mojo_simdjson_b200 import synth

    r = walk_on_gpu(dev, synth.status_array(mib << 20))
    assert r.error == 0
    assert r.n > SCAN_ITER                      # 16 MiB: about 2.70 M tokens, 1,320 blocks
    if mib == 256:
        assert r.ntiles > MS_ITER_TILES         # about 43 M tokens, 21,122 tiles
    assert len(r.doubles) > 10000


def _nest(depth: int, first_array: bool, body: int) -> list[bytes]:
    """Tokens of `depth` nested containers, alternately `[` and `{"k":`, around a flat body of `body` elements of the innermost
    container, then the matching closes."""
    kinds = [(j % 2 == 0) == first_array for j in range(depth)]   # True: array
    toks = []
    for arr in kinds:
        toks += [b"["] if arr else [b"{", b'"k"', b":"]
    toks.append(b"0")
    toks += ([b",", b"0"] if kinds[-1] else [b",", b'"k"', b":", b"0"]) * body
    toks += [b"]" if arr else b"}" for arr in reversed(kinds)]
    return toks


def _place(toks: list[bytes], anchor: int, at: int) -> bytes:
    """`[0,0,...,<toks>]` with toks[anchor] at token index `at` (filler tokens are one byte each; a leading `[]` element
    fixes the parity)."""
    head = at - anchor                       # tokens before toks[0]
    lead = (head - 1) % 2
    a = (head - 1 - 3 * lead) // 2
    assert a >= 0 and 1 + 3 * lead + 2 * a == head
    return b"[" + b"[]," * lead + b"0," * a + b"".join(toks) + b"]"


def _depth_before(toks: list[bytes], i: int) -> int:
    return 1 + sum(1 for t in toks[:i] if t in (b"[", b"{")) - sum(1 for t in toks[:i] if t in (b"]", b"}"))


NEST_DEPTH, NEST_BODY = 80, 50_000


def _nest_cases():
    """(name, first_array, where the boundary token is: ('open', j) / ('key', j) / ('colon', j) / ('body', 0) / ('close', c))"""
    cases = []
    for first_array in (True, False):
        for j in (1, 60, 61, 62, 63, 79):
            cases.append((first_array, "open", j))
        cases += [(first_array, "key", 61 if first_array else 60), (first_array, "colon", 61 if first_array else 60), (first_array, "body", 0)]
        for c in (0, 1, 10, 19):
            cases.append((first_array, "close", c))
    return cases


def _anchor(toks: list[bytes], first_array: bool, where: str, j: int) -> int:
    if where == "close":
        return len(toks) - NEST_DEPTH + j
    starts, i = [], 0
    for d in range(NEST_DEPTH):
        starts.append(i)
        i += 1 if (d % 2 == 0) == first_array else 3
    if where == "body":         # 100 tokens into the body: every open lies in the block before the boundary
        return i + 100
    return starts[j] + {"open": 0, "key": 1, "colon": 2}[where]


@pytest.mark.parametrize("first_array,where,j", _nest_cases())
def test_stack_carried_across_the_scan_iteration(dev, first_array, where, j):
    """Token 2^21 (the first one the second iteration of tape_stack_scan_kernel covers) at depth 60 to 80 of alternating
    arrays and objects, or at an open or close near there.  The opens and closes before the boundary lie in the last block of
    the first iteration, so its stack operations are part of the carry; a wrong carry gives the tokens after the boundary a
    wrong depth or container type, which changes the verdict or the tape."""
    toks = _nest(NEST_DEPTH, first_array, NEST_BODY)
    anchor = _anchor(toks, first_array, where, j)
    if where != "open" or j > 1:
        assert _depth_before(toks, anchor) + (1 if where in ("open", "key", "colon") else 0) >= 60
    r = walk_on_gpu(dev, _place(toks, anchor, SCAN_ITER))
    assert r.error == 0 and r.n > SCAN_ITER


@pytest.mark.parametrize("first_array", [True, False])
@pytest.mark.parametrize("plant", ["wrong close", "wrong close + 1", "comma after open", "comma after colon", "double comma"])
def test_error_just_after_the_scan_iteration(dev, first_array, plant):
    """A close of the wrong type or a stray `,` as the first or second token of the second scan iteration, at depth >= 60:
    TAPE_ERROR at that token."""
    toks = _nest(NEST_DEPTH, first_array, NEST_BODY)
    if plant.startswith("wrong close"):
        bad = len(toks) - NEST_DEPTH + 5
        toks[bad] = b"]" if toks[bad] == b"}" else b"}"
        at = SCAN_ITER + (1 if plant.endswith("+ 1") else 0)
    elif plant == "double comma":                      # `0,,0` in the body
        bad = next(i for i in range(len(toks) - NEST_DEPTH - 200, len(toks)) if toks[i - 1] == b",")
        toks.insert(bad, b",")
        at = SCAN_ITER
    else:                                              # `[,` or `{"k":,`
        want_arr = plant == "comma after open"
        bad = next(i + 1 for i in range(130, len(toks)) if toks[i] == (b"[" if want_arr else b":"))
        toks.insert(bad, b",")
        at = SCAN_ITER
    assert _depth_before(toks, bad) >= 60
    r = walk_on_gpu(dev, _place(toks, bad, at))
    assert r.error == oracle.TAPE_ERROR and r.error_index == at


# ------------------------------------------------------------------------------------------------
# B: the element-count limit
# ------------------------------------------------------------------------------------------------
def _array(m: int, last: bytes = b"0") -> bytes:
    return b"[" + b"0," * (m - 1) + last + b"]"


def _object(m: int) -> bytes:
    return b"{" + b'"a":0,' * (m - 1) + b'"a":0}'


def _count(word) -> int:
    return (int(word) >> 32) & 0xFFFFFF


@pytest.mark.parametrize("m", [MAX_COUNT, MAX_COUNT + 1])
def test_array_at_the_element_count_limit(dev, m):
    r = walk_on_gpu(dev, _array(m))
    assert r.n == 2 * m + 1
    if m == MAX_COUNT:                     # n = 33,554,431: 16,384 tiles, the last that one histogram scan iteration covers
        assert r.ntiles == MS_ITER_TILES
        assert r.error == 0 and chr(int(r.tape[1]) >> 56) == "[" and _count(r.tape[1]) == MAX_COUNT
    else:                                  # n = 33,554,433: 16,385 tiles; CAPACITY at the close
        assert r.ntiles == MS_ITER_TILES + 1
        assert r.error == CAPACITY and r.error_index == r.n - 1


@pytest.mark.parametrize("m", [MAX_COUNT, MAX_COUNT + 1])
def test_object_at_the_element_count_limit(dev, m):
    r = walk_on_gpu(dev, _object(m))
    assert r.n == 4 * m + 1 and r.ntiles > MS_ITER_TILES
    if m == MAX_COUNT:
        assert r.error == 0 and chr(int(r.tape[1]) >> 56) == "{" and _count(r.tape[1]) == MAX_COUNT
    else:
        assert r.error == CAPACITY and r.error_index == r.n - 1


@pytest.mark.parametrize("m", [MAX_COUNT, MAX_COUNT + 1])
def test_array_at_the_limit_inside_an_object(dev, m):
    r = walk_on_gpu(dev, b'{"k":' + _array(m) + b"}")
    assert r.n == 2 * m + 5
    if m == MAX_COUNT:                      # root, '{', '"k"', '[' ...
        assert r.error == 0 and chr(int(r.tape[3]) >> 56) == "[" and _count(r.tape[3]) == MAX_COUNT and _count(r.tape[1]) == 1
    else:
        assert r.error == CAPACITY and r.error_index == r.n - 2


def test_over_the_limit_atom_error_before_the_close_wins(dev):
    r = walk_on_gpu(dev, _array(MAX_COUNT + 1, last=b"tru"))
    assert r.error == oracle.T_ATOM_ERROR and r.error_index == r.n - 2


def test_over_the_limit_capacity_wins_over_trailing_content(dev):
    # (the trailer ends in `]`: a document that starts with `[` and ends otherwise fails at its first token)
    r = walk_on_gpu(dev, _array(MAX_COUNT + 1) + b" [0]")
    assert r.error == CAPACITY and r.error_index == r.n - 4


def test_element_count_limit_through_the_host_facade():
    from mojo_simdjson_b200.dom_parser_implementation import DomParserImplementation

    parser = DomParserImplementation(0, max_len=40 << 20)
    try:
        data = _array(MAX_COUNT)
        assert parser.stage1(data) == 0
        assert parser.stage2() == 0
        w = oracle.stage1(data, impl="fast")
        want = oracle.stage2_walk(data, w.indexes, w.n)
        assert np.array_equal(parser.document.tape, want.tape) and _count(parser.document.tape[1]) == MAX_COUNT
        assert parser.stage1(_array(MAX_COUNT + 1)) == 0
        assert parser.stage2() == CAPACITY
    finally:
        parser.close()


# ------------------------------------------------------------------------------------------------
# C: CTA and thread boundaries of the grammar kernel
# ------------------------------------------------------------------------------------------------
PROBES = {   # name: (tokens, offset of the token the error is reported at or None, verdict)
    "[]": ([b"[", b"]"], None, 0),
    "{}": ([b"{", b"}"], None, 0),
    '{"k":[]}': ([b"{", b'"k"', b":", b"[", b"]", b"}"], None, 0),
    "[[],{}]": ([b"[", b"[", b"]", b",", b"{", b"}", b"]"], None, 0),
    '{"k":0}': ([b"{", b'"k"', b":", b"0", b"}"], None, 0),
    "[1,]": ([b"[", b"1", b",", b"]"], 3, oracle.TAPE_ERROR),
    "[,1]": ([b"[", b",", b"1", b"]"], 1, oracle.TAPE_ERROR),
    '{"a" 1}': ([b"{", b'"a"', b" 1", b"}"], 2, oracle.TAPE_ERROR),
    '{"a":1,}': ([b"{", b'"a"', b":", b"1", b",", b"}"], 5, oracle.TAPE_ERROR),
    '{"a"::1}': ([b"{", b'"a"', b":", b":", b"1", b"}"], 3, oracle.TAPE_ERROR),
    "[1}": ([b"[", b"1", b"}"], 2, oracle.TAPE_ERROR),
    "tru": ([b"tru"], 0, oracle.T_ATOM_ERROR),
}


@pytest.mark.parametrize("m", [1, 1024])
@pytest.mark.parametrize("probe", list(PROBES))
def test_probe_at_every_position_around_a_cta_boundary(dev, probe, m):
    """The probe's first token at every k in 2048 m - 4 ... 2048 m + 4 of a flat array of `0`: the grammar kernel reads the two
    tokens before a thread's first token, the one after its last, and the stack state from the block scan across there.
    m = 1024 is also the first token of the second scan iteration."""
    toks, bad, code = PROBES[probe]
    for k in range(TAPE_BLOCK * m - 4, TAPE_BLOCK * m + 5):
        data = _place([b"0", b","] * 2 + toks + [b","] + [b"0", b","] * 40 + [b"0"], 4, k)
        r = walk_on_gpu(dev, data)
        assert r.error == code, (probe, k)
        if bad is not None:
            assert r.error_index == k + bad, (probe, k)


# ------------------------------------------------------------------------------------------------
# D: every double, bit for bit
# ------------------------------------------------------------------------------------------------
def _fast_path_tokens() -> list[bytes]:
    rng = random.Random(13)
    out = [b"-0.0", b"0.0", b"0e999", b"-0e-5", b"0.000", b"0." + b"0" * 21 + b"1", b"1e22", b"1E+22", b"1e-22", b"-1.5e-0",
           b"123456789012345e7", b"0.5", b"2.5E3", b"1.", b"-.5"]
    for _ in range(20000):
        k = rng.randint(1, 15)
        m = str(rng.randrange(10 ** (k - 1), 10**k))
        form = rng.randrange(4)
        e = rng.randint(-22, 22)
        ex = rng.choice(("e", "E", "e+", "E-" if e < 0 else "E+")) if form != 3 else ""
        exp = "" if form == 3 else (ex + str(abs(e)) if ex.endswith(("+", "-")) else ex + str(e))
        if form == 0:
            tok = m + exp                                    # integer mantissa
        elif form == 1:
            pnt = rng.randint(1, k)
            tok = m[:pnt] + "." + m[pnt:] + exp
        elif form == 2:                                      # leading zeros of the fraction
            z = rng.randint(0, 15 - k)
            tok = "0." + "0" * z + m + exp
        else:                                                # trailing zeros of the fraction
            pnt = rng.randint(1, k)
            tok = m[:pnt] + "." + m[pnt:] + "0" * rng.randint(0, 15 - k)
        out.append(("-" if rng.random() < 0.3 else "").encode() + tok.encode())
    return out


def _mantissa_edge_tokens() -> list[bytes]:
    out = []
    for m in (2**53 - 2, 2**53 - 1, 2**53, 2**53 + 1, 2**53 + 2, 2**53 + 3, 2**54 - 1, 2**54 + 1, 2**63 + 1):
        for e in (0, 1, -1, 15, -15, 22, -22, 23, -23):
            out.append(b"%de%d" % (m, e))
            out.append(b"-%de%d" % (m, e))
    for e in (22, -22, 23, -23):
        out += [b"1e%d" % e, b"1.5e%d" % e, b"4.9e%d" % e, b"123456789012345e%d" % e, b"9007199254740991e%d" % e]
    out += [b"9007199254740991.0", b"900719925474099.1e1", b"9007199254740993.", b"0.9007199254740993e16", b"9.007199254740993"]
    return out


def _digit_count_edge_tokens() -> list[bytes]:
    return [b"1234567890123456789e0", b"1234567890123456789.0", b"1234567890123456789.1", b"12345678901234567891e0",
            b"12345678901234567890e0", b"123456789012345678900000e-5", b"100000000000000000000000e-10", b"1" + b"0" * 30 + b".0",
            b"0.1234567890123456789", b"0.12345678901234567891", b"0.12345678901234567890", b"999999999999999999.9",
            b"9999999999999999999.9", b"99999999999999999999e-20", b"0.000000000000000000001234567890123456789e5", b"1.000000000000000000",
            b"123456789012345678e-30", b"1234567890123456789e-330", b"-98765432109876543210.5e3"]


def _exponent_extreme_tokens() -> list[bytes]:
    return [b"1e308", b"1.7976931348623157e308", b"1.7976931348623158e308", b"1.7976931348623159e308", b"1e309", b"-1e309",
            b"2.2250738585072014e-308", b"1e-307", b"1e-308", b"4.9406564584124654e-324", b"1e-324", b"2.5e-324", b"1e-325",
            b"9e-310", b"1E+308", b"1e99999", b"1e100000", b"1e100001", b"1e999999", b"1e1000000", b"1e-1000000", b"1e1234567890",
            b"1e-1234567890", b"0e1234567", b"1e0000000000000001", b"123e-0000000000005", b"5e-0000000000000000000000000000000324",
            b"1e+0000000308", b"0.000001e314", b"100000e-330"]


def _long_tokens() -> list[bytes]:
    return [b"5e" + b"0" * 600, b"1." + b"0" * 600, b"1" + b"2" * 599 + b".0", b"0." + b"0" * 600 + b"1", b"-" + b"9" * 600 + b".5",
            b"0." + b"0" * 530 + b"123e530", b"1" + b"0" * 600 + b"e-600", b"1" * 600 + b"e-590", b"2.5e" + b"0" * 600 + b"1"]


DOUBLE_CORPORA = {"fast path": _fast_path_tokens, "mantissa edges": _mantissa_edge_tokens, "digit-count edges": _digit_count_edge_tokens,
                  "exponent extremes": _exponent_extreme_tokens, "long tokens": _long_tokens}


@pytest.mark.parametrize("corpus", list(DOUBLE_CORPORA))
def test_every_double_bit_for_bit(dev, corpus):
    """One array per corpus (the inexact count is per document).  walk_on_gpu compares every payload with the restatement and
    summary[3] with the restated inexact count; here also: where the restated rule says exact, the payload is python's
    correctly rounded float() of the token."""
    toks = DOUBLE_CORPORA[corpus]()
    r = walk_on_gpu(dev, b"[" + b",".join(toks) + b"]")
    assert r.error == 0 and [t for t, _, _ in r.doubles] == toks
    for tok, bits, inexact in r.doubles:
        if not inexact:
            assert bits == _bits(float(tok)), tok
    n_exact = sum(not inexact for _, _, inexact in r.doubles)
    if corpus == "fast path":
        assert n_exact > 0.9 * len(toks)
    else:
        assert 0 < len(toks) - n_exact
    if corpus == "long tokens":
        assert min(len(t) for t in toks) > 512


# ------------------------------------------------------------------------------------------------
# E: caller buffers that are too small
# ------------------------------------------------------------------------------------------------
GUARD = 64
SENT64 = 0x5A5A5A5A5A5A5A5A
SENT8 = 0xA5


@pytest.fixture(scope="module")
def small_doc(dev):
    """A document with strings, integers and doubles, its stage-1 result and primitives on the device, and the oracle's walk."""
    from mojo_simdjson_b200 import synth

    a = synth.twitter_like()
    w = oracle.stage1(a, impl="fast")
    d_in = torch.from_numpy(a.copy()).to("cuda")
    d_idx = torch.empty(a.size + 8, dtype=torch.int32, device="cuda")
    assert dev.index(d_in, d_idx).n == w.n
    prims = dev.stage2_primitives(d_in, d_idx, w.n)
    p = oracle.stage2_primitives(a, w.indexes[: w.n])
    want = oracle.stage2_walk(a, w.indexes, w.n)
    assert want.error == 0
    exp, n_inexact, _ = expected_tape(a, w.indexes[: w.n], p, want)
    ks = np.nonzero(np.isin(p.kind, (oracle.KIND_INT, oracle.KIND_FLOAT)))[0]
    two_word = np.zeros(exp.size, dtype=bool)   # first words of the values that take two tape words
    two_word[tape_positions(a, w.indexes[: w.n], p)[ks]] = True
    assert (p.kind == oracle.KIND_STRING).sum() > 1000 and (p.kind == oracle.KIND_FLOAT).any() and (p.kind == oracle.KIND_INT).any()
    return dict(a=a, n=w.n, d_in=d_in, d_idx=d_idx, prims=prims, p=p, tape=exp, n_inexact=n_inexact, two_word=two_word)


def _tape_caps(two_word: np.ndarray) -> list[int]:
    N = two_word.size
    caps = [N - 1, N // 2, 1]
    q = int(np.nonzero(two_word[N // 2 :])[0][0]) + N // 2
    caps.append(q + 1)          # the type word of an integer or double would fit, its payload would not
    return caps


def test_tape_capacity_short(dev, small_doc):
    """Nothing is stored at or past the capacity, and nothing before the buffer; every word below it is the oracle's, except
    that a two-word value that does not fit whole is not written at all; the summary still reports the full tape."""
    sd = small_doc
    N = sd["tape"].size
    for cap in _tape_caps(sd["two_word"]):
        buf = torch.full((cap + 2 * GUARD,), SENT64, dtype=torch.int64, device="cuda")
        summary = torch.empty(4, dtype=torch.int64, device="cuda")
        pr = sd["prims"]
        rc = dev._lib.sjb200_stage2_tape_device_async(dev._ctx, sd["d_in"].data_ptr(), sd["d_in"].numel(), sd["d_idx"].data_ptr(), sd["n"],
                                                      pr["kind"].data_ptr(), pr["error"].data_ptr(), pr["value"].data_ptr(),
                                                      pr["str_off"].data_ptr(), buf.data_ptr() + 8 * GUARD, cap, summary.data_ptr())
        assert rc == 0
        torch.cuda.synchronize()
        got = buf.cpu().numpy().view(np.uint64)
        assert np.all(got[:GUARD] == np.uint64(SENT64)) and np.all(got[GUARD + cap :] == np.uint64(SENT64)), cap
        want = sd["tape"][:cap].copy()
        if sd["two_word"][cap - 1]:
            want[cap - 1] = SENT64
        assert np.array_equal(got[GUARD : GUARD + cap], want), cap
        assert summary.cpu().tolist() == [-1, N - 2, N, sd["n_inexact"]], cap


def test_string_capacity_short(dev, small_doc):
    """Records that do not fit whole are not written at all, nothing past the capacity changes, the primitives arrays and the
    record byte count are the full ones."""
    sd = small_doc
    p, n = sd["p"], sd["n"]
    total = p.string_buf.size
    ends = np.sort(p.str_off[p.kind == oracle.KIND_STRING].astype(np.int64) + 4 + p.value[p.kind == oracle.KIND_STRING])
    for cap in (total - 1, total // 2, 3, 0):
        sbuf = torch.full((cap + 2 * GUARD,), SENT8, dtype=torch.uint8, device="cuda")
        kind = torch.empty(n, dtype=torch.uint8, device="cuda")
        err = torch.empty(n, dtype=torch.uint8, device="cuda")
        value = torch.empty(n, dtype=torch.int64, device="cuda")
        off = torch.empty(n, dtype=torch.int64, device="cuda")
        summary = torch.empty(4, dtype=torch.int64, device="cuda")
        rc = dev._lib.sjb200_stage2_primitives_device_async(dev._ctx, sd["d_in"].data_ptr(), sd["d_in"].numel(), sd["d_idx"].data_ptr(), n,
                                                            kind.data_ptr(), err.data_ptr(), value.data_ptr(), off.data_ptr(),
                                                            sbuf.data_ptr() + GUARD, cap, summary.data_ptr())
        assert rc == 0
        torch.cuda.synchronize()
        assert np.array_equal(kind.cpu().numpy(), p.kind) and np.array_equal(err.cpu().numpy(), p.error)
        assert np.array_equal(value.cpu().numpy(), p.value)
        is_str = p.kind == oracle.KIND_STRING
        assert np.array_equal(off.cpu().numpy().view(np.uint64)[is_str], p.str_off[is_str])
        assert summary.cpu().tolist()[:2] == [-1, total]
        got = sbuf.cpu().numpy()
        assert np.all(got[:GUARD] == SENT8) and np.all(got[GUARD + cap :] == SENT8), cap
        fit = int(ends[ends <= cap][-1]) if (ends <= cap).any() else 0     # records are contiguous: the ones that fit are a prefix
        want = np.full(cap, SENT8, dtype=np.uint8)
        want[:fit] = p.string_buf[:fit]
        assert np.array_equal(got[GUARD : GUARD + cap], want), cap


def test_host_stage2_with_short_buffers(small_doc):
    """sjb200_stage2 returns CAPACITY and copies nothing when either host buffer is short; with exact sizes it succeeds."""
    from mojo_simdjson_b200.dom_parser_implementation import DomParserImplementation

    sd = small_doc
    N, SB = sd["tape"].size, sd["p"].string_buf.size
    parser = DomParserImplementation(0, max_len=1 << 20)
    try:
        assert parser.stage1(sd["a"]) == 0
        for tcap, scap, want_rc in ((N - 1, SB, CAPACITY), (N, SB - 1, CAPACITY), (1, 1, CAPACITY), (N, SB, 0)):
            tape = np.full(tcap + 2 * GUARD, SENT64, dtype=np.uint64)
            sbuf = np.full(scap + 2 * GUARD, SENT8, dtype=np.uint8)
            tl, sl, inexact = C.c_uint64(0), C.c_uint64(0), C.c_uint64(0)
            rc = parser._lib.sjb200_stage2(parser._ctx, tape.ctypes.data + 8 * GUARD, tcap, sbuf.ctypes.data + GUARD, scap, C.byref(tl), C.byref(sl),
                                           C.byref(inexact))
            assert rc == want_rc, (tcap, scap)
            assert (tl.value, sl.value, inexact.value) == (N, SB, sd["n_inexact"])
            assert np.all(tape[:GUARD] == np.uint64(SENT64)) and np.all(tape[GUARD + tcap :] == np.uint64(SENT64))
            assert np.all(sbuf[:GUARD] == SENT8) and np.all(sbuf[GUARD + scap :] == SENT8)
            if rc == CAPACITY:
                assert np.all(tape == np.uint64(SENT64)) and np.all(sbuf == SENT8)
            else:
                assert np.array_equal(tape[GUARD : GUARD + N], sd["tape"]) and np.array_equal(sbuf[GUARD : GUARD + SB], sd["p"].string_buf)
    finally:
        parser.close()
