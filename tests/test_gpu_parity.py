"""GPU parity tests: the CUDA stage 1 (through the C ABI) against the CPU oracle, bit-exact.

Run on a B200 with `pytest -m gpu`.  Indexes, n, trailer, verdicts and the UTF-8 verdict must all be identical
to the oracle's on the same inputs; at full size (1 GiB) the comparison is a digest of the index stream plus
size-independent properties.
"""
import ctypes as C
import os

import numpy as np
import pytest
from hypothesis import given, settings, strategies as st

from oracle import oracle
from tests import cases

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")


@pytest.fixture(scope="module")
def dev():
    from mojo_simdjson_b200 import device

    ctx = device.Stage1Context(0, max_len=(1 << 32) - 1)
    yield ctx
    ctx.close()


@pytest.fixture(scope="module")
def parser():
    from mojo_simdjson_b200.dom_parser_implementation import DomParserImplementation

    p = DomParserImplementation(0, max_len=8 << 20)
    yield p
    p.close()


class Scratch:
    """Reusable device buffers; inputs are placed at a chosen misalignment inside the allocation."""

    def __init__(self, nbytes):
        self.inp = torch.empty(nbytes + 256, dtype=torch.uint8, device="cuda")
        self.out = torch.empty(nbytes + 16, dtype=torch.int32, device="cuda")

    def put(self, data: bytes, mis: int):
        a = np.frombuffer(data, dtype=np.uint8)
        # hostile bytes around the document: the kernel must never let them leak in
        self.inp[: mis + len(data) + 64].fill_(0x22)
        view = self.inp[mis : mis + len(data)]
        view.copy_(torch.from_numpy(a.copy()))
        return view


@pytest.fixture(scope="module")
def scratch():
    return Scratch(4 << 20)


def run_device(dev, scratch, data: bytes, mis=0, flags=0, warps=0, cap=None, kernel="auto"):
    dev.set_warps(warps)
    dev.set_kernel(kernel)
    view = scratch.put(data, mis)
    out = scratch.out if cap is None else scratch.out[:cap]
    scratch.out[: len(data) + 8].fill_(-1)
    res = dev.index(view, out, flags)
    dev.set_warps(0)
    dev.set_kernel("auto")
    return res, scratch.out


def assert_same(res, out_t, want, cap=None):
    assert res.error == want.error
    assert res.n == want.n
    if want.error != oracle.CAPACITY:
        assert res.n_written == want.n_written
        keep = want.indexes.size
        got = out_t[:keep].cpu().numpy().view(np.uint32)
        assert np.array_equal(got, want.indexes)
    assert res.utf8_error == want.utf8_error


# ------------------------------------------------------------------------------------------------
# config 1: the reference's own fixtures, through the reference-shaped facade (host buffers)
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("fx", cases.golden_fixtures(), ids=lambda f: f["file"])
def test_reference_fixtures_through_facade(parser, fx):
    """tests/test_stage_1.mojo:85-96 + :43-82 restated against the drop-in."""
    err = parser.stage1(fx["input"])
    assert err == 0, "unexpected error code"
    n = parser.n_structural_indexes
    got = [int(x) for x in parser.structural_indexes[:n]]
    assert all(a < b for a, b in zip(got, got[1:]))
    mask = [" "] * len(fx["mask"])
    for i in got:
        mask[i] = "1"
    if fx["harness_negative"]:
        assert "".join(mask) != fx["mask"]
    else:
        assert "".join(mask) == fx["mask"]
    ln = len(fx["input"].encode("utf-8"))
    assert list(parser.structural_indexes[n : n + 3]) == [ln, ln, 0]
    assert parser.next_structural_index == 0


@pytest.mark.parametrize("case", cases.KNOWN_ANSWERS, ids=lambda c: repr(c)[:24])
def test_known_answers_through_facade(parser, case):
    data, err, n, idx = case
    parser.n_structural_indexes = 777  # sentinel: must survive the reference's early-return paths
    got = parser.stage1(data)
    assert got == err
    if n is None:
        assert parser.n_structural_indexes == 777
    else:
        assert parser.n_structural_indexes == n
        assert list(parser.structural_indexes[n : n + 3]) == [len(data), len(data), 0]
    if idx:
        assert [int(x) for x in parser.structural_indexes[: len(idx)]] == idx


def test_host_path_matches_oracle_on_corpus(parser):
    for name, data in cases.adversarial_cases(tile_bytes=(4096,))[::7]:
        want = oracle.stage1(data)
        parser.n_structural_indexes = 0xFFFFFFFF
        err = parser.stage1(data)
        assert err == want.error, name
        if want.n is not None:
            assert parser.n_structural_indexes == want.n, name
        assert np.array_equal(parser.structural_indexes[: want.indexes.size], want.indexes), name
        assert parser.utf8_error == want.utf8_error, name


def test_validate_utf8_flag_through_facade():
    from mojo_simdjson_b200.dom_parser_implementation import DomParserImplementation

    p = DomParserImplementation(0, max_len=1 << 20, validate_utf8=True)
    try:
        assert p.stage1(b'["\xc0\x80"]') == 11
        assert p.stage1(b'"\xff') == 15
        assert p.stage1(b'"\xff\x01"') == 14
        assert p.stage1('["héllo"]') == 0
    finally:
        p.close()


def test_host_path_streams_in_chunks():
    """sjb200_stage1 copies / indexes / copies back chunk by chunk (look-back state carried across launches)."""
    from mojo_simdjson_b200 import synth
    from mojo_simdjson_b200.dom_parser_implementation import DomParserImplementation

    size = (20 << 20) + 12345
    doc = synth.status_array(size)
    p = DomParserImplementation(0, max_len=size, chunk_bytes=1 << 20)
    try:
        want = oracle.stage1(doc, impl="fast")
        assert p.stage1(doc) == want.error == 0
        assert p.n_structural_indexes == want.n
        assert np.array_equal(p.structural_indexes[: want.n + 3], want.indexes)
        # verdicts that need the whole document, decided in the last chunk
        bad = doc.copy()
        bad[size // 2] = 0x22  # a stray quote in the middle flips every string after it
        want = oracle.stage1(bad, impl="fast")
        p.n_structural_indexes = 777
        assert p.stage1(bad) == want.error
        assert want.error in (14, 15) and p.n_structural_indexes == 777
        assert np.array_equal(p.structural_indexes[: want.n_written], want.indexes[: want.n_written])
        ndj = synth.ndjson(3 << 20)
        want = oracle.stage1(ndj, impl="fast")
        assert p.stage1(ndj) == 0 and np.array_equal(p.structural_indexes[: want.n + 3], want.indexes)
    finally:
        p.close()


# ------------------------------------------------------------------------------------------------
# config 5: adversarial set, device-resident path, every tile shape, aligned and misaligned input
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("warps", [2, 4, 8, 16, 24])
def test_adversarial_corpus_device(dev, scratch, warps):
    tiles = tuple(sorted({warps * 2048, 4096}))
    corpus = cases.adversarial_cases(tile_bytes=tiles)
    if warps != 2:
        corpus = corpus[::3]
    for k, (name, data) in enumerate(corpus):
        if not data:
            continue
        want = oracle.stage1(data, impl="fast" if len(data) > 20000 else "ref")
        for mis in ((0, 5) if k % 4 == 0 else (0,)):
            res, out = run_device(dev, scratch, data, mis=mis, warps=warps)
            try:
                assert_same(res, out, want)
            except AssertionError as e:  # pragma: no cover
                raise AssertionError(f"case {name} mis={mis} warps={warps}") from e


@pytest.mark.parametrize("kernel,warps", [("persistent", 2), ("persistent", 4), ("persistent", 8), ("persistent", 16), ("persistent", 24),
                                          ("split", 8), ("split", 16), ("stream", 8), ("stream", 2)])
def test_adversarial_corpus_every_kernel_organisation(dev, scratch, kernel, warps):
    """The same corpus through each kernel organisation (sjb200_ctx_set_kernel): results must not depend on it."""
    tiles = tuple(sorted({warps * 2048, 4096}))
    corpus = cases.adversarial_cases(tile_bytes=tiles)[::2]
    for k, (name, data) in enumerate(corpus):
        if not data:
            continue
        want = oracle.stage1(data, impl="fast" if len(data) > 20000 else "ref")
        for mis in ((0, 11) if k % 4 == 0 else (0,)):
            res, out = run_device(dev, scratch, data, mis=mis, warps=warps, kernel=kernel)
            try:
                assert_same(res, out, want)
            except AssertionError as e:  # pragma: no cover
                raise AssertionError(f"case {name} mis={mis} warps={warps} kernel={kernel}") from e


def test_stream_pipeline_speculation_and_fallback(dev, scratch):
    """A backslash run that covers the 32 bytes before a 2 KiB chunk is walked back through global memory (up to 64 KiB);
    only a longer one makes the stream pipeline give up, and the persistent kernel behind it must then produce the
    document (and must stay out of the way otherwise)."""
    for run in (0, 1, 30, 31, 32, 33, 64, 65, 511, 512, 513, 2047, 2048, 2049, 5000, 65535, 65536, 65537, 66047, 66048, 66049, 70001, 200000):
        for pad in (2048 - 2, 2048 - 1, 2048, 4096 - 33, 4096 - 1):
            lead = (pad - 2 - run) % 2048   # the run always ends `pad` mod 2 KiB
            head = b'["' + b"a" * lead
            data = head + b"\\" * 0 + b"\\"[:1] * run + b'"x", "y\\"", 1, {"k": "\\\\"}]' + b" " * 3000 + b"[]"
            want = oracle.stage1(data, impl="ref")
            for kernel in ("stream", "persistent"):
                res, out = run_device(dev, scratch, data, kernel=kernel, warps=8)
                try:
                    assert_same(res, out, want)
                except AssertionError as e:  # pragma: no cover
                    raise AssertionError(f"run={run} pad={pad} kernel={kernel}") from e
    # alternate documents that do / do not trigger the fallback: no state may leak between calls
    ok = b'{"a": [1, 2, 3], "b": "' + b"z" * 9000 + b'"}'
    bad = b'["' + b"a" * 2046 + b"\\"[:1] * (2048 * 40 + 1) + b'" ]'   # 80 KiB + 1 backslashes ending on a chunk boundary
    walk = b'["' + b"a" * 2040 + b"\\"[:1] * 200 + b'" ]'               # resolved by the walk
    wok, wbad, wwalk = oracle.stage1(ok), oracle.stage1(bad, impl="fast"), oracle.stage1(walk)
    for kernel in ("stream",):
        for _ in range(6):
            res, out = run_device(dev, scratch, ok, kernel=kernel)
            assert_same(res, out, wok)
            res, out = run_device(dev, scratch, bad, kernel=kernel)
            assert_same(res, out, wbad)
            res, out = run_device(dev, scratch, walk, kernel=kernel)
            assert_same(res, out, wwalk)
    # the walk must stop at the first byte of the document: backslashes in the memory before it are not input
    data = b"\\"[:1] * 4095 + b'"' + b'"abc"' + b" " * 3000 + b"[1]"
    want = oracle.stage1(data, impl="ref")
    for mis in (0, 1, 7, 15):
        for kernel in ("stream", "persistent"):
            dev.set_kernel(kernel)
            dev.set_warps(8)
            scratch.inp[: mis + len(data) + 64].fill_(0x5C)
            view = scratch.inp[mis : mis + len(data)]
            view.copy_(torch.from_numpy(np.frombuffer(data, dtype=np.uint8).copy()))
            scratch.out[: len(data) + 8].fill_(-1)
            res = dev.index(view, scratch.out)
            dev.set_kernel("auto")
            dev.set_warps(0)
            assert_same(res, scratch.out, want)


@pytest.mark.parametrize("kernel", ["stream", "split", "persistent"])
def test_chunks_without_structurals_at_every_output_phase(dev, scratch, kernel):
    """2 KiB chunks that contribute no index (inside a long string) at every 16-byte phase of the output cursor, and chunks
    that contribute 1, 2, 3 indexes: the flatten kernel's vector copy must not touch a neighbour's entries."""
    for k in range(0, 9):
        for tail_items in (0, 1, 2, 3, 5):
            data = b"[" + b"1," * k + b'"' + b"s" * 9000 + b'"' + b",2" * tail_items + b"]" + b" " * 2500 + b"\n[]"
            want = oracle.stage1(data, impl="ref")
            for mis in (0, 4, 8, 12):
                res, out = run_device(dev, scratch, data, mis=mis, warps=8, kernel=kernel)
                try:
                    assert_same(res, out, want)
                except AssertionError as e:  # pragma: no cover
                    raise AssertionError(f"k={k} tail_items={tail_items} mis={mis} kernel={kernel}") from e
    # output buffer at every 4-byte phase of a 16-byte line
    data = b"[" + b"1," * 5 + b'"' + b"s" * 5000 + b'",' + b"[]," * 700 + b"0]"
    want = oracle.stage1(data, impl="ref")
    inp = scratch.put(data, 0)
    for shift in range(4):
        scratch.out[: len(data) + 16].fill_(-1)
        dev.set_kernel(kernel)
        dev.set_warps(8)
        res = dev.index(inp, scratch.out[shift:])
        dev.set_kernel("auto")
        dev.set_warps(0)
        assert_same(res, scratch.out[shift:], want)
        assert int((scratch.out[:shift] != -1).sum()) == 0


@pytest.mark.parametrize("kernel", ["split", "stream"])
def test_split_pair_capacity_and_flags(dev, scratch, kernel):
    data = b'[' + b'1,' * 40000 + b'1]'
    want = oracle.stage1(data, impl="fast")
    for cap in (want.n + 3, want.n + 2, want.n, 1000, 3):
        res, out = run_device(dev, scratch, data, cap=cap, warps=8, kernel=kernel)
        if cap >= want.n + 3:
            assert_same(res, out, want)
        else:
            assert res.error == 1 and res.n is None, cap
            keep = min(cap, want.n)
            assert np.array_equal(out[:keep].cpu().numpy().view(np.uint32), want.indexes[:keep]), cap
            assert int((out[cap : len(data) + 8] != -1).sum()) == 0, "wrote past the capacity"
    bad = b'["\xc0\x80", "' + b"x" * 70000 + b'"]'
    for flags in (0, 1):
        w = oracle.stage1(bad, flags=flags, impl="ref")
        res, out = run_device(dev, scratch, bad, flags=flags, warps=16, kernel=kernel)
        assert_same(res, out, w)
        assert res.error == (11 if flags else 0)
    res, out = run_device(dev, scratch, bad, flags=4, warps=16, kernel=kernel)
    assert res.error == 0 and res.utf8_error == -1


def test_every_misalignment(dev, scratch):
    data = b'{"k":"v\\"x","a":[1,2,3],"u":"\xe2\x82\xac"}' * 300
    want = oracle.stage1(data)
    for mis in range(16):
        res, out = run_device(dev, scratch, data, mis=mis, warps=2)
        assert_same(res, out, want)


def test_stream_pipeline_at_every_start_in_a_line(dev, scratch):
    """The stream pipeline on documents that start anywhere inside a 128-byte line (a variant of its classify kernel with
    128-byte lanes on a swizzled layout, tried in round 2, depended on that; the test stayed): non-ASCII text in most lanes,
    an odd number of chunks, invalid UTF-8 in the middle and as the last bytes of a unit / an odd chunk."""
    from mojo_simdjson_b200 import synth
    docs = [c[1] for c in cases.adversarial_cases()][:40]
    docs.append(b'{"k":"v\\"x","a":[1,2,3],"u":"\xe2\x82\xac \xf0\x9f\x98\x80"}' * 4000)       # ~100 chunks, non-ASCII in most lanes
    docs.append(b"[" + b'"\xe4\xb8\xad\xe6\x96\x87 text \\\\ \\" end",' * 9000 + b"0]")
    docs.append(bytes(synth.status_array((3 << 20) + 4097)))                                      # odd number of chunks, ragged end
    bad = docs[-3]
    docs.append(bad[:70001] + b"\xe2\x82" + bad[70001:])      # a truncated sequence in the middle: UTF8_ERROR
    docs.append(bad[:4096 * 9 - 1] + b"\xc3")                  # ... and as the very last byte, right at the end of a unit
    docs.append(bad[:4096 * 9 + 2047] + b"\xf0\x9f")           # ... and at the end of an odd chunk
    for data in docs:
        want = oracle.stage1(data, impl="fast", flags=oracle.FLAG_VALIDATE_UTF8)
        for mis in (0, 5, 16, 64 + 3, 112, 127):
            res, out = run_device(dev, scratch, data, mis=mis, flags=oracle.FLAG_VALIDATE_UTF8, warps=8, kernel="stream")
            try:
                assert_same(res, out, want)
            except AssertionError as e:  # pragma: no cover
                raise AssertionError(f"len={len(data)} mis={mis}") from e


def test_flags(dev, scratch):
    bad = b'["\xc0\x80"]' * 10
    res, _ = run_device(dev, scratch, bad, flags=1)
    assert res.error == 11 and res.utf8_error == 1
    res, _ = run_device(dev, scratch, bad, flags=0)
    assert res.error == 0 and res.utf8_error == 1
    res, _ = run_device(dev, scratch, bad, flags=4)  # NO_UTF8: verdict not computed
    assert res.error == 0 and res.utf8_error == -1
    assert dev.index(scratch.inp[:0], scratch.out).error == 13  # len == 0 -> EMPTY, no launch


def test_capacity(dev, scratch):
    data = b"[1,2,3]"
    res, out = run_device(dev, scratch, data, cap=10)
    assert res.error == 0 and res.n == 7
    res, out = run_device(dev, scratch, data, cap=9)
    assert res.error == 1 and res.n is None
    # nothing may be written past the capacity
    big = b"[" + b"1," * 5000 + b"1]"
    scratch.out[:20000].fill_(-1)
    res, out = run_device(dev, scratch, big, cap=100)
    assert res.error == 1
    assert int((scratch.out[100:20000] != -1).sum()) == 0


@pytest.mark.parametrize("kernel", ["stream", "split"])
def test_flatten_units_of_every_density(dev, scratch, kernel):
    """The balanced flatten kernel works on units of two chunks (4 KiB): every lane extracts the same number of consecutive
    indexes.  Pieces of very different density side by side -- long strings (no index for kilobytes), one index every few
    hundred bytes (shares of 1..3 indexes, most mask words empty), the bench document's density, units just below and just
    above the staging capacity (768 indexes per unit: per-chunk fallback), everything structural -- at piece lengths that
    are not multiples of a chunk, with an odd number of chunks and with a clipped output capacity."""
    rng = np.random.default_rng(20261018)
    pieces = []
    for rep in range(200):
        kind = int(rng.choice(9, p=[0.1, 0.15, 0.15, 0.15, 0.15, 0.1, 0.08, 0.06, 0.06]))
        length = int(rng.integers(300, 9000))
        if kind == 0:
            piece = b'"' + b"s" * length + b'",'
        elif kind == 1:
            piece = b"".join(b'"' + b"x" * int(rng.integers(100, 700)) + b'",' for _ in range(length // 400 + 1))
        elif kind == 2:
            piece = b'"abcdefgh",' * (length // 11 + 1)    # 0.18 per byte: units just below the capacity
        elif kind == 3:
            piece = b"12345," * (length // 6 + 1)          # 0.17 per byte
        elif kind == 4:
            piece = b"123456789012," * (length // 13 + 1)  # 0.08 per byte
        elif kind == 5:
            piece = b'{"id":12345,"text":"hello \\"world\\"","tags":[]},' * (length // 50 + 1)
        elif kind == 6:
            piece = b"123,45," * (length // 7 + 1)         # 0.29 per byte: units above the capacity, chunks below 512 + 85
        elif kind == 7:
            piece = b"1," * (length // 2 + 1)              # 0.5 per byte
        else:
            piece = b"[]," * (length // 3 + 1)             # every byte structural
        pieces.append(piece)
    body = b"".join(pieces)
    for extra in (0, 1777, 2048 + 5):                      # odd / even chunk counts, ragged last chunk
        data = b"[" + body + b"0" * extra + b"]"
        want = oracle.stage1(data, impl="fast")
        assert want.error == 0
        for mis in (0, 4):
            res, out = run_device(dev, scratch, data, mis=mis, warps=8, kernel=kernel)
            assert_same(res, out, want)
    data = b"[" + body + b"0]"
    want = oracle.stage1(data, impl="fast")
    for cap in (want.n + 3, want.n - 1, want.n // 2 + 1, 777):
        res, out = run_device(dev, scratch, data, cap=cap, warps=8, kernel=kernel)
        if cap >= want.n + 3:
            assert_same(res, out, want)
        else:
            assert res.error == 1 and res.n is None, cap
            keep = min(cap, want.n)
            assert np.array_equal(out[:keep].cpu().numpy().view(np.uint32), want.indexes[:keep]), cap


def test_dense_tile_takes_direct_path(dev, scratch):
    data = b"[" + b"1," * 100000 + b"1]"  # every byte structural: > 0.5 per byte, bypasses staging
    want = oracle.stage1(data, impl="fast")
    for warps in (2, 8, 16, 24):
        res, out = run_device(dev, scratch, data, warps=warps)
        assert_same(res, out, want)
    for kernel in ("stream", "split"):
        res, out = run_device(dev, scratch, data, warps=8, kernel=kernel)
        assert_same(res, out, want)


@settings(max_examples=150, deadline=None)
@given(st.lists(st.sampled_from(list(cases.NASTY)), min_size=1, max_size=12000), st.integers(0, 15))
def test_fuzz_nasty_device(dev, scratch, xs, mis):
    data = bytes(xs)
    res, out = run_device(dev, scratch, data, mis=mis, warps=2)
    assert_same(res, out, oracle.stage1(data))


@settings(max_examples=100, deadline=None)
@given(st.binary(min_size=1, max_size=6000), st.integers(0, 15))
def test_fuzz_binary_device(dev, scratch, data, mis):
    res, out = run_device(dev, scratch, data, mis=mis, warps=2)
    assert_same(res, out, oracle.stage1(data))


def test_alternating_kernel_kinds_and_tile_shapes(dev, scratch):
    """Persistent launches alternate two ticket counters; launches of the other kernel in between must not disturb them."""
    a = b'{"a":"' + b"x" * 3000 + b'","b":[1,2,3]}'
    wa = oracle.stage1(a)
    for warps in (2, 24, 2, 2, 24, 24, 2, 16, 4, 24, 8, 2, 24, 2):
        res, out = run_device(dev, scratch, a, warps=warps)
        assert_same(res, out, wa)
    seq = [("split", 8), ("persistent", 2), ("stream", 2), ("split", 16), ("split", 8), ("stream", 8), ("stream", 8), ("split", 8),
           ("persistent", 16), ("stream", 4), ("stream", 4), ("split", 16), ("stream", 8), ("stream", 8), ("persistent", 4),
           ("stream", 2), ("persistent", 2), ("stream", 16), ("split", 8), ("stream", 4), ("stream", 24), ("persistent", 24)]
    for kernel, warps in seq:
        res, out = run_device(dev, scratch, a, warps=warps, kernel=kernel)
        assert_same(res, out, wa)


def test_repeated_calls_reuse_descriptors(dev, scratch):
    """Generation-tagged look-back descriptors: back-to-back calls with different inputs must not interfere."""
    a = (b'{"a":"' + b"x" * 5000 + b'"}') * 40
    b = b'"' + b"\\" * 70001 + b'" 1'
    wa, wb = oracle.stage1(a, impl="fast"), oracle.stage1(b, impl="fast")
    for _ in range(20):
        res, out = run_device(dev, scratch, a, warps=2)
        assert_same(res, out, wa)
        res, out = run_device(dev, scratch, b, warps=2)
        assert_same(res, out, wb)


# ------------------------------------------------------------------------------------------------
# configs 2-4: synthetic workloads
# ------------------------------------------------------------------------------------------------
def test_twitter_like_631k(dev):
    from mojo_simdjson_b200 import synth

    doc = synth.twitter_like()
    assert doc.size == 631_515
    want = oracle.stage1(doc, impl="fast")
    assert want.error == 0
    inp = torch.from_numpy(doc).cuda()
    out = torch.empty(doc.size + 3, dtype=torch.int32, device="cuda")
    for warps in (0, 2, 4, 8, 16, 24):
        dev.set_warps(warps)
        out.fill_(-1)
        res = dev.index(inp, out)
        assert_same(res, out, want)
    dev.set_warps(0)
    for kernel in ("stream", "split"):
        dev.set_kernel(kernel)
        out.fill_(-1)
        res = dev.index(inp, out)
        assert_same(res, out, want)
    dev.set_kernel("auto")


def test_document_64mib_full_compare(dev):
    from mojo_simdjson_b200 import synth

    size = 64 << 20
    doc = synth.status_array(size)
    want = oracle.stage1(doc, impl="fast", cap=size // 3)
    assert want.error == 0
    inp = torch.from_numpy(doc).cuda()
    out = torch.empty(size // 3, dtype=torch.int32, device="cuda")
    for kernel, warps in (("persistent", 2), ("persistent", 8), ("persistent", 16), ("persistent", 24), ("split", 0), ("stream", 0), ("auto", 0)):
        dev.set_kernel(kernel)
        dev.set_warps(warps)
        out.fill_(-1)
        res = dev.index(inp, out)
        assert_same(res, out, want)
    dev.set_warps(0)
    dev.set_kernel("auto")
    # error injected far into the document: verdict parity at scale
    bad = doc.copy()
    bad[size - 1000] = 0x22
    want = oracle.stage1(bad, impl="fast", cap=size // 3)
    inp.copy_(torch.from_numpy(bad))
    res = dev.index(inp, out)
    assert res.error == want.error and res.n == want.n and res.n_written == want.n_written


@pytest.mark.skipif(os.environ.get("SJB200_SKIP_1GIB") == "1", reason="SJB200_SKIP_1GIB=1")
def test_document_1gib_digest_and_properties(dev):
    """BASELINE.json config 3 at full size: digest of the index stream vs the oracle + domain properties."""
    from mojo_simdjson_b200 import synth

    size = 1 << 30
    doc = synth.status_array(size)
    cap = size // 4
    want = oracle.stage1(doc, impl="fast", cap=cap)
    assert want.error == 0
    inp = torch.from_numpy(doc).cuda()
    out = torch.empty(cap, dtype=torch.int32, device="cuda")
    res = dev.index(inp, out)
    assert res.error == 0 and res.n == want.n and res.utf8_error == 0
    n = res.n
    got = out[: n + 3].cpu().numpy().view(np.uint32)
    assert oracle.index_digest(got) == oracle.index_digest(want.indexes)
    # properties: strictly ascending, every index on a structural byte or a scalar/string start, trailer
    assert bool((got[1:n] > got[: n - 1]).all())
    assert list(got[n : n + 3]) == [size, size, 0]
    first_bytes = doc[got[:n]]
    assert not np.isin(first_bytes, np.frombuffer(b" \n\t\r", dtype=np.uint8)).any()
    # idempotence: a second run over the same buffer gives the same stream
    out2 = torch.empty(cap, dtype=torch.int32, device="cuda")
    res2 = dev.index(inp, out2)
    assert res2.n == n and bool(torch.equal(out[: n + 3], out2[: n + 3]))


def test_ndjson_batch_segments(dev):
    """Config 4 in miniature: cut at newlines, every segment == an independent reference call."""
    from mojo_simdjson_b200 import synth

    size = 48 << 20
    batch = synth.ndjson(size)
    inp = torch.from_numpy(batch).cuda()
    seg_bytes = 5 << 20
    offs = dev.split(inp, seg_bytes)
    assert offs[0] == 0 and offs[-1] == size
    host_offs = (C.c_uint64 * 64)()
    nseg = C.c_uint32(0)
    from mojo_simdjson_b200 import _native

    rc = _native.lib().sjb200_batch_split_host(batch.ctypes.data, size, seg_bytes, host_offs, 63, C.byref(nseg))
    assert rc == 0 and [int(host_offs[i]) for i in range(nseg.value + 1)] == offs
    for a, b in zip(offs, offs[1:]):
        assert b > a and b - a <= 2 * seg_bytes and batch[b - 1] == 0x0A
    out = torch.empty(size + 3 * len(offs), dtype=torch.int32, device="cuda")
    out.fill_(-1)
    worst, counts, errs, u8, idx_offs = dev.run_segments(inp, offs, out)
    assert worst == 0
    host = out.cpu().numpy().view(np.uint32)
    for s in range(len(offs) - 1):
        seg = batch[offs[s] : offs[s + 1]]
        want = oracle.stage1(seg, impl="fast")
        assert errs[s] == want.error == 0
        assert counts[s] == want.n
        assert u8[s] == 0
        got = host[idx_offs[s] : idx_offs[s] + want.n + 3]
        assert np.array_equal(got, want.indexes)


def test_ndjson_batch_driver_single_rank():
    """The in-library batch driver (sjb200_batch_create_rank, world 1): plan + passes alternating the two row-buffer sets +
    run(); then a re-plan with FEWER segments must not leave rows of segments that no longer exist (round-1 advisor finding)."""
    from mojo_simdjson_b200 import batch as batch_mod, synth

    size = 24 << 20
    data = synth.ndjson(size)
    inp = torch.from_numpy(data).cuda()
    drv = batch_mod.NdjsonBatchDriver(0, seg_bytes=4 << 20, max_segments=16)
    try:
        offs = drv.plan(inp)
        assert offs[0] == 0 and offs[-1] == size and len(offs) - 1 >= 3
        out = torch.empty(drv.index_capacity(), dtype=torch.int32, device="cuda")
        want = [oracle.stage1(data[a:b], impl="fast") for a, b in zip(offs, offs[1:])]
        for _ in range(3):
            out.fill_(-1)
            v = drv.run(out)
            assert v.worst_error == 0
            assert v.errors == [0] * (len(offs) - 1)
            assert v.counts == [[w.n for w in want]]
            host = out.cpu().numpy().view(np.uint32)
            for s, w in enumerate(want):
                o = drv.index_offsets()[s]
                assert np.array_equal(host[o : o + w.n + 3], w.indexes)
        # a broken segment shows up in the worst error and in this rank's per-segment errors
        bad = data.copy()
        bad[offs[1] + 10] = 0x22  # unbalances the quotes of segment 1
        wbad = oracle.stage1(bad[offs[1] : offs[2]], impl="fast")
        if wbad.error != 0:
            drv.plan(torch.from_numpy(bad).cuda())
            v = drv.run(out)
            assert v.worst_error == wbad.error
            assert v.errors[1] == wbad.error and v.errors[0] == 0
        # fewer segments than before: the rows of the vanished segments read "no such segment", the stale error is gone
        small = inp[: offs[2]]
        offs2 = drv.plan(small)
        assert len(offs2) - 1 == 2
        for _ in range(3):
            v = drv.run(out)
            assert v.worst_error == 0 and v.counts == [[want[0].n, want[1].n]] and v.errors == [0, 0]
    finally:
        drv.close()


def test_batch_host_entry_point_single_process():
    """sjb200_batch_run (host batch in, host indexes out) on one GPU: shards / segments cut at newlines, every segment ==
    an independent reference call on its byte range."""
    from mojo_simdjson_b200 import _native, synth

    L = _native.lib()
    size = 20 << 20
    data = synth.ndjson(size)
    b = C.c_void_p()
    assert L.sjb200_batch_create(1, None, size, 3 << 20, 32, 0, C.byref(b)) == 0
    try:
        idx = np.full(size + 3 * 32, 0xFFFFFFFF, dtype=np.uint32)
        seg_off = (C.c_uint64 * 33)()
        seg_idx = (C.c_uint64 * 33)()
        seg_n = (C.c_uint32 * 32)()
        seg_err = (C.c_int32 * 32)()
        nseg = C.c_uint32(0)
        worst = C.c_int32(-1)
        for _ in range(2):
            rc = L.sjb200_batch_run(b, data.ctypes.data, size, idx.ctypes.data, idx.size, seg_off, seg_idx, seg_n, seg_err, 32,
                                    C.byref(nseg), C.byref(worst), 0)
            assert rc == 0 and worst.value == 0 and nseg.value >= 3
            assert seg_off[0] == 0 and seg_off[nseg.value] == size
            for s in range(nseg.value):
                a, e = int(seg_off[s]), int(seg_off[s + 1])
                assert data[e - 1] == 0x0A
                want = oracle.stage1(data[a:e], impl="fast")
                assert seg_err[s] == want.error == 0 and seg_n[s] == want.n
                o = int(seg_idx[s])
                assert o == a + 3 * s
                assert np.array_equal(idx[o : o + want.n + 3], want.indexes)
        # too small an index array is refused up front
        rc = L.sjb200_batch_run(b, data.ctypes.data, size, idx.ctypes.data, size, seg_off, seg_idx, seg_n, seg_err, 32,
                                C.byref(nseg), C.byref(worst), 0)
        assert rc == 1
    finally:
        L.sjb200_batch_destroy(b)


def nccl_library_path():
    """The NCCL the image ships inside the torch wheel (the C++ test has no torch to pull it in)."""
    try:
        import nvidia.nccl

        p = os.path.join(list(nvidia.nccl.__path__)[0], "lib", "libnccl.so.2")
        return p if os.path.exists(p) else None
    except Exception:
        return None


def test_batch_driver_from_cpp_alone():
    """tests/cpp/batch_test: sjb200_batch_create / run / plan_resident / run_resident_async / finish driven from a C++
    binary (no Python, no torch in that process), on 2 GPUs when the box has them, checked there against the oracle."""
    import subprocess

    from mojo_simdjson_b200 import build

    exe = build.build_cpp_tests()
    gpus = 2 if torch.cuda.device_count() >= 2 else 1
    env = dict(os.environ)
    lib = nccl_library_path()
    if lib:
        env.setdefault("SJB200_NCCL_LIB", lib)
    r = subprocess.run([exe, str(gpus), "48", "2"], capture_output=True, text=True, timeout=600, env=env)
    assert r.returncode == 0 and r.stdout.strip().endswith("PASS"), r.stdout + r.stderr


@pytest.mark.parametrize("kernel", ["auto", "stream", "persistent"])
def test_maximum_length_document(kernel):
    """len = 2^32 - 1, the largest document the uint32 index format allows (reference include/base.mojo:2): index values
    above 2^31, chunk arithmetic at the top of the 32-bit range, trailer = len.  Built on the device, expected output
    known in closed form (a 4 GiB oracle run would take minutes)."""
    free, _ = torch.cuda.mem_get_info()
    if free < 12 << 30:
        pytest.skip("needs ~10 GiB of device memory")
    from mojo_simdjson_b200 import device

    L = (1 << 32) - 1
    ctx = device.Stage1Context(0, max_len=L)
    try:
        ctx.set_kernel(kernel)
        buf = torch.full((L,), 0x20, dtype=torch.uint8, device="cuda")
        buf[0] = ord("[")
        buf[L - 1] = ord("]")
        # a little structure at chosen offsets: `"k":1,` (6 bytes) -> structurals at +0 (quote), +3 (:), +4 (1), +5 (,)
        spots = [1, 2047, 2048 * 3 - 2, (1 << 31) - 3, (1 << 31) + 5, (3 << 30) + 2045, L - 4096 - 7, L - 8]
        pat = torch.tensor(list(b'"k":1,'), dtype=torch.uint8, device="cuda")
        want = [0]
        for p in spots:
            buf[p : p + 6] = pat
            want += [p, p + 3, p + 4, p + 5]
        want.append(L - 1)
        # one long string across many chunks near the top: its inside must contribute nothing
        s0, s1 = (7 << 29) + 11, (7 << 29) + 11 + 5_000_000
        buf[s0 + 1 : s1] = ord("{")
        buf[s0] = ord('"')
        buf[s1] = ord('"')
        want = sorted(want + [s0])
        out = torch.full((4096,), -1, dtype=torch.int32, device="cuda")
        res = ctx.index(buf, out)
        assert res.error == 0 and res.n == len(want)
        got = out[: len(want) + 3].cpu().numpy().view(np.uint32).astype(np.int64).tolist()
        assert got == want + [L, L, 0]
    finally:
        ctx.close()


@pytest.mark.parametrize("kernel", ["stream", "persistent"])
def test_utf8_verdicts_sparse_lanes(dev, scratch, kernel):
    """Valid and invalid UTF-8 sequences in otherwise ASCII documents, placed so that they straddle lane (64 B) and chunk
    (2 KiB) boundaries, sit at the very start / end of the document, or follow a lane that is pure ASCII: in the stream
    pipeline these are lanes the classify kernel parks in its warp's ring and validates at a flush (validate_parked_lanes,
    stage1_stream.cuh).  Every slot, both flushes and ticketed runs: tests/test_gpu_utf8_deferral.py."""
    seqs = list(cases.UTF8_VALID) + list(cases.UTF8_INVALID)
    for k, seq in enumerate(seqs):
        seq = seq if isinstance(seq, (bytes, bytearray)) else seq.encode("utf-8", "surrogatepass")
        for pos in (0, 1, 60, 62, 63, 64, 2044, 2046, 2047, 2048, 4095, 6000):
            body = bytearray(b"a" * 7000)
            body[pos:pos] = seq
            for data in (b'"' + bytes(body) + b'"', b'"' + bytes(body[: pos + len(seq)])):  # second one: ends right after the sequence
                want = oracle.stage1(data, flags=1, impl="ref")
                res, out = run_device(dev, scratch, data, flags=1, kernel=kernel, warps=8, mis=(k + pos) % 16)
                try:
                    assert_same(res, out, want)
                except AssertionError as e:  # pragma: no cover
                    raise AssertionError(f"seq={seq!r} pos={pos} len={len(data)} kernel={kernel}") from e
    # many flagged lanes in one chunk (more than the deferral limit) next to chunks with a single one
    data = b'["' + ("é" * 40 + "a" * 200).encode() * 30 + b'", "' + b"a" * 3000 + "€".encode() + b"a" * 3000 + b'\xc3"]'
    want = oracle.stage1(data, flags=1, impl="ref")
    res, out = run_device(dev, scratch, data, flags=1, kernel=kernel, warps=8)
    assert_same(res, out, want)
    assert want.utf8_error == 1


def test_structural_bytes_side_output(dev, scratch):
    """SURVEY 8(f) rank 2: out[k] = buf[idx[k]] on the device against the oracle, every alignment of idx / out."""
    from mojo_simdjson_b200 import synth

    docs = [b"[1]", b'{"a":[1,-2.5e3,true,null,"x\\"y"],"b":{}}', bytes(synth.twitter_like()), bytes(synth.status_array(3 << 20))]
    for data in docs:
        want = oracle.stage1(data, impl="fast" if len(data) > 20000 else "ref")
        assert want.error == 0
        wb = oracle.structural_bytes(data, want.indexes[: want.n])
        inp = torch.from_numpy(np.frombuffer(data, dtype=np.uint8).copy()).cuda()
        idx_buf = torch.full((len(data) + 16,), -1, dtype=torch.int32, device="cuda")
        out_buf = torch.full((len(data) + 64,), 0xEE, dtype=torch.uint8, device="cuda")
        for ishift in (0, 1, 2, 3):
            for oshift in (0, 1, 3, 4):
                idx = idx_buf[ishift:]
                res = dev.index(inp, idx)
                assert res.error == 0 and res.n == want.n
                out_buf.fill_(0xEE)
                out = out_buf[8 + oshift :]
                dev.structural_bytes(inp, idx, res.n, out)
                torch.cuda.synchronize()
                got = out[: res.n].cpu().numpy()
                assert np.array_equal(got, wb), (len(data), ishift, oshift)
                assert int(out_buf[7 + oshift]) == 0xEE and int(out[res.n]) == 0xEE, "wrote outside [0, n)"
    # the trailer entries (len, len, 0) read as 0, 0 and the first byte
    data = docs[1]
    inp = torch.from_numpy(np.frombuffer(data, dtype=np.uint8).copy()).cuda()
    idx = torch.empty(len(data) + 3, dtype=torch.int32, device="cuda")
    res = dev.index(inp, idx)
    got = dev.structural_bytes(inp, idx, res.n + 3).cpu().numpy()
    assert list(got[-3:]) == [0, 0, data[0]]


def test_document_starts_side_output(dev):
    """SURVEY 8(f) rank 2, second half: depth-0 structurals of a document stream, against the oracle's cumulative sum."""
    from mojo_simdjson_b200 import synth

    docs = [b"1", b'{"a":[1,2]}\n[3]\n4 "s"\n{"b":{}}', b"]]][[[", bytes(synth.ndjson(24 << 20)), bytes(synth.status_array(5 << 20))]
    for data in docs:
        want = oracle.stage1(data, impl="fast" if len(data) > 20000 else "ref")
        n = want.n_written
        sb = oracle.structural_bytes(data, want.indexes[:n])
        ws = oracle.document_starts(sb)
        for shift in (0, 1, 5, 16):
            buf = torch.full((n + 64,), 0x7B, dtype=torch.uint8, device="cuda")   # hostile bytes around: '{'
            view = buf[shift : shift + n]
            view.copy_(torch.from_numpy(sb))
            out_buf = torch.full((n + 64,), 0xEE, dtype=torch.uint8, device="cuda")
            out = out_buf[8 + shift :]
            dev.document_starts(view, n, out)
            torch.cuda.synchronize()
            assert np.array_equal(out[:n].cpu().numpy(), ws), (len(data), shift)
            assert int(out_buf[7 + shift]) == 0xEE and int(out[n]) == 0xEE, "wrote outside [0, n)"
    # the whole chain on the device: index -> bytes -> starts; an NDJSON batch has one start per line
    data = docs[3]
    inp = torch.from_numpy(np.frombuffer(data, dtype=np.uint8).copy()).cuda()
    idx = torch.empty(len(data) // 2, dtype=torch.int32, device="cuda")
    res = dev.index(inp, idx)
    assert res.error == 0
    sbytes = dev.structural_bytes(inp, idx, res.n)
    starts = dev.document_starts(sbytes, res.n)
    torch.cuda.synchronize()
    assert int(starts.sum().item()) == data.count(b"\n")


# ------------------------------------------------------------------------------------------------
# config 5 at its specified sizes (SURVEY.md section 8(d)): the heavy adversarial set through every kernel organisation,
# and the dense 64 MiB / 192 MiB buffers (digest + n + verdict + UTF-8 verdict against the oracle)
# ------------------------------------------------------------------------------------------------
def _heavy_only_cases():
    base = {name for name, _ in cases.adversarial_cases(tile_bytes=(4096, 8192, 16384))}
    return [(n, d) for n, d in cases.adversarial_cases(tile_bytes=(4096, 8192, 16384), heavy=True) if n not in base]


@pytest.mark.parametrize("kernel", ["stream", "split", "persistent"])
def test_adversarial_corpus_heavy(dev, scratch, kernel):
    """65535 / 65536 / 2^20+1 backslash runs at every offset and the larger fuzz set (cases.adversarial_cases(heavy=True))."""
    heavy = _heavy_only_cases()
    assert len(heavy) > 200 and any(name.startswith("bsrun:1048577@") for name, _ in heavy)
    for k, (name, data) in enumerate(heavy):
        want = oracle.stage1(data, impl="fast" if len(data) > 20000 else "ref")
        for mis in ((0, 7) if k % 5 == 0 else (0,)):
            res, out = run_device(dev, scratch, data, mis=mis, kernel=kernel)
            try:
                assert_same(res, out, want)
            except AssertionError as e:  # pragma: no cover
                raise AssertionError(f"case {name} mis={mis} kernel={kernel}") from e


def test_every_kernel_and_tile_shape_pair(dev, scratch):
    """Every (organisation, warps) pair sjb200_ctx_set_warps accepts either produces the oracle's result or is refused
    with UNEXPECTED_ERROR -- never a silently truncated index (round-1 advisor finding)."""
    from mojo_simdjson_b200 import synth

    data = bytes(synth.status_array(300_000)) + b" " * 777
    want = oracle.stage1(data, impl="fast")
    for kernel in ("auto", "persistent", "split", "stream"):
        for warps in (0, 2, 4, 8, 16, 24):
            res, out = run_device(dev, scratch, data, warps=warps, kernel=kernel)
            if kernel == "split" and warps in (2, 4, 24):
                assert res.error == 24 and res.n is None, (kernel, warps)
            else:
                assert_same(res, out, want)
    for bad in (1, 3, 12, 32, 64):
        with pytest.raises(ValueError):
            dev.set_warps(bad)
    for bad in (1, 3, 6, 7):
        with pytest.raises(ValueError):
            dev.set_kernel(bad)


def _dense_documents(size):
    """SURVEY.md 8(d) config 5(ii) at `size` bytes: quote-dense, escape-dense, all-CJK, all-bracket, and a document with a
    33-byte backslash run before a chunk boundary every MiB (the input that used to cost the stream pipeline a second pass)."""
    q = np.full(size, 0x22, dtype=np.uint8)
    e = np.empty(size, dtype=np.uint8)
    e[0::2] = 0x5C
    e[1::2] = 0x22
    e[0], e[1], e[-2], e[-1] = ord("["), ord('"'), ord('"'), ord("]")
    cjk_unit = np.frombuffer("日本語のテキスト€😀".encode("utf-8"), dtype=np.uint8)
    cjk = np.resize(cjk_unit, size).copy()
    cut = (size - 2) // cjk_unit.size * cjk_unit.size
    cjk[0], cjk[1] = ord("["), ord('"')
    cjk[2 : 2 + cut - cjk_unit.size] = np.resize(cjk_unit, cut - cjk_unit.size)
    cjk[2 + cut - cjk_unit.size :] = ord("a")
    cjk[-2], cjk[-1] = ord('"'), ord("]")
    br = np.full(size, ord("["), dtype=np.uint8)
    from mojo_simdjson_b200 import synth

    runs = synth.status_array(size).copy()
    return {"quotes": q, "escapes": e, "cjk": cjk, "brackets": br, "runs": runs}


@pytest.mark.parametrize("size_mib", [64, 192])
def test_dense_buffers_at_specified_sizes(dev, size_mib):
    size = size_mib << 20
    docs = _dense_documents(size)
    from mojo_simdjson_b200 import synth

    assert synth.plant_backslash_runs(docs["runs"]) >= size_mib - 8
    kernels = ("auto", "stream", "persistent") if size_mib == 64 else ("auto", "stream")
    out = torch.empty(size + 16, dtype=torch.int32, device="cuda")
    for name, doc in docs.items():
        want = oracle.stage1(doc, impl="fast", cap=size + 3, flags=1)
        inp = torch.from_numpy(doc).cuda()
        for kernel in kernels:
            dev.set_kernel(kernel)
            res = dev.index(inp, out, flags=1)
            dev.set_kernel("auto")
            assert (res.error, res.n, res.n_written, res.utf8_error) == (want.error, want.n, want.n_written, want.utf8_error), (name, kernel)
            keep = want.indexes.size
            got = out[:keep].cpu().numpy().view(np.uint32)
            assert oracle.index_digest(got) == oracle.index_digest(want.indexes), (name, kernel)
        del inp
