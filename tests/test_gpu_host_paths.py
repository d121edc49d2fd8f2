"""GPU tests of the two paths on which host code splits one job into several kernel launches and puts the results together:

  A  the chunked host entry point sjb200_stage1 (what DomParserImplementation.stage1 calls): a document larger than
     chunk_bytes is indexed by one persistent-kernel launch per chunk of tiles, all sharing one generation, so that the
     look-back carries parity and the output cursor from one launch into the next; every chunk's indexes travel back on a
     second stream, clamped to the caller's capacity
  B  NDJSON batches: the device splitter, sjb200_batch_run_device with segments of every verdict and of every kernel
     organisation in one call, the host batch entry point sjb200_batch_run and the resident driver (NdjsonBatchDriver)

Every result is compared with oracle.stage1 on the same bytes: the error, n (or the untouched sentinel where the reference
leaves n alone), the indexes the oracle delivers (trailer included) and the UTF-8 verdict.  Host arrays are larger than
the capacity passed and filled with 0xFFFFFFFF; whatever the oracle does not deliver must still hold that sentinel."""
import ctypes as C
import random

import numpy as np
import pytest

from oracle import oracle
from tests import cases
from tests.test_batch_split_rule import CAPACITY, check_plan, enumerated_cases, expected_cuts, host_split, random_batch

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

SENT = 0xFFFFFFFF
GUARD = 64                      # host-array entries past the capacity that must keep the sentinel
VALIDATE_UTF8, NO_UTF8 = 1, 4
EMPTY, UTF8_ERROR, UNESCAPED_CHARS, UNCLOSED_STRING = 13, 11, 14, 15
MAX_CHUNKS = 256                # launches the host path splits one document into at most
KERNEL_SPLIT, KERNEL_STREAM = 4, 5


def _u8(data) -> np.ndarray:
    return data if isinstance(data, np.ndarray) else np.frombuffer(bytes(data), dtype=np.uint8)


def want_of(data, flags=0, cap=None):
    a = _u8(data)
    return oracle.stage1(a, flags=flags & VALIDATE_UTF8, impl="fast" if a.size > 20000 else "ref", cap=cap)


# ------------------------------------------------------------------------------------------------
# A: the chunked host entry point
# ------------------------------------------------------------------------------------------------
def make_parser(max_len, chunk_bytes=None, warps=0):
    from mojo_simdjson_b200.dom_parser_implementation import DomParserImplementation

    p = DomParserImplementation(0, max_len=max_len, chunk_bytes=chunk_bytes)
    if warps:
        assert p._lib.sjb200_ctx_set_warps(p._ctx, warps) == 0
    return p


def launches(p) -> int:
    return int(p._lib.sjb200_launch_count(p._ctx))


def host_stage1(p, data, cap=None, flags=0):
    """sjb200_stage1 on the parser's context into a host array of cap + GUARD sentinel entries.
    Returns (error, n or None, utf8 verdict, the whole host array)."""
    a = _u8(data)
    if cap is None:
        cap = a.size + 3
    out = np.full(cap + GUARD, SENT, dtype=np.uint32)
    n = C.c_uint32(SENT)
    u8 = C.c_int32(-7)
    rc = p._lib.sjb200_stage1(p._ctx, a.ctypes.data, a.size, out.ctypes.data, cap, C.byref(n), C.byref(u8), flags)
    return rc, (None if n.value == SENT else n.value), u8.value, out


def check_host(got, want, label=""):
    rc, n, u8, out = got
    assert rc == want.error, label
    assert n == want.n, label
    k = want.indexes.size
    assert np.array_equal(out[:k], want.indexes), label
    assert np.all(out[k:] == SENT), f"{label}: entries past what the oracle delivers were written"
    assert u8 == want.utf8_error, label


def run_and_check(p, data, flags=0, cap=None, label=""):
    want = want_of(data, flags, cap)
    check_host(host_stage1(p, data, cap, flags), want, label)
    return want


def expected_chunks(length: int, tile: int, chunk_bytes: int) -> int:
    """Launches sjb200_stage1 makes for one document: chunks of whole tiles, re-chunked to at most 256."""
    ntiles = -(-length // tile)
    per = max(chunk_bytes // tile, 1)
    nchunks = -(-ntiles // per)
    if nchunks > MAX_CHUNKS:
        per = -(-ntiles // MAX_CHUNKS)
        nchunks = -(-ntiles // per)
    return nchunks


_want_cache: dict = {}


def cached_want(name, data, flags):
    key = (name, flags)
    if key not in _want_cache:
        _want_cache[key] = want_of(data, flags)
    return _want_cache[key]


def tile_edge_cases():
    """What the corpus lacks at tile edges of 8 and 16 KiB: 2-, 3- and 4-byte sequences, valid and invalid, starting 3 bytes
    before the edge through the edge itself; a control byte inside a string at edge - 1 and at the edge."""
    seqs = {"c3a9": b"\xc3\xa9", "e282ac": b"\xe2\x82\xac", "f09f9880": b"\xf0\x9f\x98\x80", "e0a080": b"\xe0\xa0\x80",
            "f48fbfbf": b"\xf4\x8f\xbf\xbf",
            "c080": b"\xc0\x80", "c2": b"\xc2", "e08080": b"\xe0\x80\x80", "eda080": b"\xed\xa0\x80", "e282": b"\xe2\x82",
            "f0808080": b"\xf0\x80\x80\x80", "f4908080": b"\xf4\x90\x80\x80", "f09f98": b"\xf0\x9f\x98", "80": b"\x80"}
    out = []
    for edge in (8192, 16384):
        for name, s in seqs.items():
            for start in range(edge - 3, edge + 1):
                body = b'["' + b"a" * (start - 2) + s + b"a" * 40 + b'", 1, "' + b"b" * 300 + b'"]'
                out.append((f"utf8:{name}@{edge}{start - edge:+d}", body))
        for c in (0x01, 0x1F, 0x0A):
            for at in (edge - 1, edge):
                body = b'["' + b"a" * (at - 2) + bytes([c]) + b"a" * 40 + b'", 2]'
                out.append((f"ctl-in:{c:02x}@{edge}{at - edge:+d}", body))
    return out


@pytest.mark.parametrize("warps", [2, 4, 8])
def test_carries_across_launches(warps):
    """chunk_bytes = 4096: every tile of 4, 8 or 16 KiB is its own launch, so every carry -- backslash runs, open strings,
    UTF-8 sequences, scalars -- that crosses a tile edge crosses a launch boundary."""
    tile = warps * 2048
    corpus = [(n, d) for n, d in cases.adversarial_cases(tile_bytes=(4096, 8192, 16384)) if len(d) > tile]
    assert len(corpus) >= {2: 600, 4: 250, 8: 130}[warps]
    corpus += [(n, d) for n, d in tile_edge_cases() if len(d) > tile]
    p = make_parser(1 << 20, chunk_bytes=4096, warps=warps)
    try:
        for name, data in corpus:
            for flags in (0, VALIDATE_UTF8):
                before = launches(p)
                check_host(host_stage1(p, data, flags=flags), cached_want(name, data, flags), f"{name} flags={flags}")
                assert launches(p) - before == -(-len(data) // tile), name
    finally:
        p.close()


@pytest.mark.parametrize("ntiles", [255, 256, 257, 511, 513])
def test_chunk_count_and_rechunking(ntiles):
    """4 KiB tiles, 4 KiB chunks: one launch per tile up to 256 tiles; from 257 tiles on the host re-chunks to
    ceil(T / 256) tiles per chunk."""
    from mojo_simdjson_b200 import synth

    tile = 4096
    p = make_parser(4 << 20, chunk_bytes=4096, warps=2)
    try:
        for size in (ntiles * tile, ntiles * tile - 777):
            doc = synth.status_array(size)
            before = launches(p)
            run_and_check(p, doc, label=f"{ntiles} tiles, {size} bytes")
            got = launches(p) - before
            assert got == expected_chunks(size, tile, 4096)
            assert got == {255: 255, 256: 256, 257: 129, 511: 256, 513: 171}[ntiles]
    finally:
        p.close()


@pytest.mark.parametrize("warps,chunk_tiles,extra,ntiles,tail", [
    (16, 0, 4096, 20, -5),        # chunk_bytes (4096) smaller than a 32 KiB tile: one tile per launch
    (4, 3, 1, 100, -5),           # 3 tiles + 1 byte: 3 tiles per chunk, a last chunk of one tile
    (8, 7, 0, 60, -1000),         # a prime number of tiles per chunk, a ragged last chunk of 4 tiles
    (2, 5, 0, 23, -4095),         # last tile of one byte
])
def test_chunk_geometry(warps, chunk_tiles, extra, ntiles, tail):
    from mojo_simdjson_b200 import synth

    tile = warps * 2048
    chunk = chunk_tiles * tile + extra
    size = ntiles * tile + tail
    p = make_parser(2 << 20, chunk_bytes=chunk, warps=warps)
    try:
        for doc in (synth.status_array(size), synth.ndjson(size)):
            before = launches(p)
            run_and_check(p, doc, label=f"warps={warps} chunk={chunk} size={size}")
            assert launches(p) - before == expected_chunks(size, tile, chunk)
        big = cases.adversarial_cases(tile_bytes=(tile,))
        for name, data in big:
            if len(data) > chunk:
                run_and_check(p, data, flags=VALIDATE_UTF8, label=name)
    finally:
        p.close()


def test_default_chunk_size_two_chunks():
    """The automatic tile shape (16 warps) at the default 32 MiB chunk: a document just over 32 MiB takes two launches."""
    from mojo_simdjson_b200 import synth

    size = (32 << 20) + 12345
    doc = synth.status_array(size)
    p = make_parser(40 << 20)
    try:
        before = launches(p)
        want = run_and_check(p, doc, label="32 MiB + 12345")
        assert launches(p) - before == 2 == expected_chunks(size, 16 * 2048, 32 << 20)
        assert want.error == 0
    finally:
        p.close()


def test_capacity_on_the_chunked_path():
    """idx_capacity below n + 3: the oracle's result for cap=, and nothing stored at or past the capacity."""
    from mojo_simdjson_b200 import synth

    size = 150_000
    doc = synth.status_array(size)
    tile, chunk = 4096, 4 * 4096
    p = make_parser(1 << 20, chunk_bytes=chunk, warps=2)
    try:
        full = run_and_check(p, doc, label="full")          # leaves the device index array full of this document's indexes
        n = full.n
        first_chunk = int(np.count_nonzero(full.indexes[:n] < chunk))
        assert 0 < first_chunk < n
        for cap in (n + 3, n + 2, first_chunk, first_chunk - 1, first_chunk + 1, n // 2, 1):
            run_and_check(p, doc, cap=cap, label=f"cap={cap}")
        # a document that ends with an error keeps the same clamp
        bad = doc.copy()
        bad[size // 2] = 0x22
        wbad = want_of(bad)
        assert wbad.error in (UNESCAPED_CHARS, UNCLOSED_STRING)
        for cap in (wbad.n_written + 3, wbad.n_written, first_chunk, 1):
            run_and_check(p, bad, cap=cap, label=f"bad cap={cap}")
    finally:
        p.close()


def string_doc(size: int, seed: int) -> bytes:
    """An array of strings of 'x' and of integers, no backslashes: a byte is inside a string iff an odd number of quotes
    precedes it."""
    rng = random.Random(seed)
    parts, n = [b"["], 1
    while n < size - 10:
        s = b'"' + b"x" * rng.randint(0, 300) + b'"' if rng.random() < 0.6 else str(rng.randint(0, 10**9)).encode()
        parts.append(s + b",")
        n += len(s) + 1
    parts.append(b"0]")
    return b"".join(parts)


def place_in_string(doc: bytes, pos: int) -> bytes:
    """doc shifted right by leading spaces so that byte `pos` is an 'x' inside a string."""
    for k in range(0, 400):
        q = pos - k
        if doc[q] == ord("x") and doc[:q].count(b'"') % 2 == 1:
            return b" " * k + doc
    raise AssertionError("no string near the position")


def test_verdicts_decided_at_the_end():
    """A stray quote, a control byte in a string and an invalid UTF-8 byte in chunk 0, in a middle chunk and in the last byte
    of a chunk: the oracle's verdict, n left alone where the reference leaves it, indexes[:n_written] delivered."""
    chunk = 2 * 4096
    base = string_doc(110_000, 7)
    p = make_parser(1 << 20, chunk_bytes=chunk, warps=2)
    try:
        for where, pos in (("chunk 0", 1000), ("middle chunk", 5 * chunk + 3000), ("last byte of chunk 2", 3 * chunk - 1),
                           ("first byte of chunk 7", 7 * chunk)):
            doc = bytearray(place_in_string(base, pos))
            ok = bytes(doc)
            run_and_check(p, ok, label=where)
            for kind, byte in (("stray quote", 0x22), ("control byte", 0x01), ("invalid utf-8", 0xFF)):
                doc[pos] = byte
                bad = bytes(doc)
                for flags in (0, VALIDATE_UTF8):
                    want = run_and_check(p, bad, flags=flags, label=f"{kind} at {where} flags={flags}")
                    expect = {"stray quote": (UNCLOSED_STRING,), "control byte": (UNESCAPED_CHARS,),
                              "invalid utf-8": (UTF8_ERROR,) if flags else (0,)}[kind]
                    assert want.error in expect, (kind, where, want.error)
                    if kind != "invalid utf-8":
                        assert want.n is None and want.n_written > 0
                doc[pos] = ord("x")
    finally:
        p.close()


def test_order_of_calls_on_one_context():
    """Large, small, large, an error, a valid one, twice over, at 4096-byte chunks on one context: a stale progress word,
    generation or ticket counter would show up here."""
    from mojo_simdjson_b200 import synth

    large = synth.status_array((3 << 20) + 123)
    small = b'{"a":[1,2,{"b":"c"}]}'
    large2 = synth.ndjson(2 << 20)
    err = large.copy()
    err[len(err) // 3] = 0x22
    valid = synth.twitter_like()
    seq = [("large", large), ("small", small), ("large2", large2), ("error", err), ("valid", valid), ("tiny", b"1"),
           ("blank", b" " * 9000)]
    p = make_parser(4 << 20, chunk_bytes=4096)
    try:
        for rep in range(2):
            for name, data in seq:
                run_and_check(p, data, label=f"{name} #{rep}")
                run_and_check(p, data, flags=VALIDATE_UTF8, label=f"{name} #{rep} utf8")
    finally:
        p.close()


@pytest.mark.parametrize("kernel", [KERNEL_SPLIT, KERNEL_STREAM])
def test_set_kernel_does_not_change_the_host_path(kernel):
    """The host path always indexes with the persistent kernel, one launch per chunk, whatever organisation is forced."""
    from mojo_simdjson_b200 import synth

    doc = synth.status_array((1 << 20) + 7)
    chunk = 64 << 10
    p = make_parser(2 << 20, chunk_bytes=chunk)
    try:
        assert p._lib.sjb200_ctx_set_kernel(p._ctx, kernel) == 0
        for warps in (0, 8, 16):
            assert p._lib.sjb200_ctx_set_warps(p._ctx, warps) == 0
            tile = (warps or 2) * 2048      # 1 MiB picks 2-warp tiles
            before = launches(p)
            run_and_check(p, doc, label=f"kernel={kernel} warps={warps}")
            assert launches(p) - before == expected_chunks(doc.size, tile, chunk)
    finally:
        p.close()


def test_stage2_after_chunked_stage1():
    """stage2() walks the document stage 1 indexed in several chunks: the oracle's tape (doubles restated bit for bit) and
    string buffer."""
    from mojo_simdjson_b200 import synth
    from tests.test_gpu_stage2_scale import expected_tape

    chunk = 64 << 10
    p = make_parser(8 << 20, chunk_bytes=chunk)
    try:
        for doc in (synth.twitter_like(), synth.status_array(3 << 20)):
            w = oracle.stage1(doc, impl="fast")
            assert w.error == 0 and doc.size > 4 * chunk
            before = launches(p)
            assert p.stage1(doc) == 0
            assert launches(p) - before > 1
            assert p.n_structural_indexes == w.n
            assert np.array_equal(p.structural_indexes[: w.n + 3], w.indexes)
            assert p.stage2() == 0
            want = oracle.stage2_walk(doc, w.indexes, w.n)
            assert want.error == 0
            prims = oracle.stage2_primitives(doc, w.indexes[: w.n])
            exp, n_inexact, _ = expected_tape(doc, w.indexes[: w.n], prims, want)
            assert np.array_equal(p.document.tape, exp)
            assert np.array_equal(p.document.string_buf, want.string_buf)
            assert p.document.inexact_doubles == n_inexact
    finally:
        p.close()


# ------------------------------------------------------------------------------------------------
# B: NDJSON batches
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def dev():
    from mojo_simdjson_b200 import device

    ctx = device.Stage1Context(0, max_len=(1 << 32) - 1)
    yield ctx
    ctx.close()


def to_device(data: bytes, mis=0, fill=0x0A):
    """`data` at byte offset `mis` of a device buffer whose other bytes are `fill` (newlines: a splitter that reads outside
    the batch would find them)."""
    buf = torch.full((len(data) + mis + 64,), fill, dtype=torch.uint8, device="cuda")
    view = buf[mis : mis + len(data)]
    if data:
        view.copy_(torch.from_numpy(np.frombuffer(bytes(data), dtype=np.uint8).copy()))
    return buf, view


def device_split(dev, data: bytes, seg, max_segments, mis=0):
    """sjb200_batch_split_device: the offsets, or the error code."""
    buf, view = to_device(data, mis)
    offs = (C.c_uint64 * (max_segments + 2))()
    nseg = C.c_uint32(SENT)
    rc = dev._lib.sjb200_batch_split_device(dev._ctx, view.data_ptr(), len(data), seg, offs, max_segments, C.byref(nseg))
    del buf
    if rc != 0:
        return rc
    return [int(offs[i]) for i in range(nseg.value + 1)]


def device_only_split_cases():
    out = []
    for g in (31, 32, 33, 64, 65):                       # gaps between newlines around the warp's 32-byte steps
        data = (b"x" * (g - 1) + b"\n") * 200 + b"x" * (g // 2)
        for seg in (31, 32, 33, 64, 65, 96, 100, 1000, 4095):
            out.append((f"gap{g}-seg{seg}", data, seg, 4096))
    for seg in (32, 33, 64, 1000):                       # the newline as the first / the last byte of every window
        first = bytearray(b"y" * (10 * seg + 5))
        last = bytearray(b"y" * (10 * seg + 5))
        for k in range(11):
            if k * seg < len(first):
                first[k * seg] = 0x0A
            if (k + 1) * seg - 1 < len(last):
                last[(k + 1) * seg - 1] = 0x0A
        out.append((f"first-byte-seg{seg}", bytes(first), seg, 4096))
        out.append((f"last-byte-seg{seg}", bytes(last), seg, 4096))
        out.append((f"first-byte-only-seg{seg}", bytes(first[: 3 * seg + 1]), seg, 4096))
    for seg, line in ((16, 10), (100, 37)):              # 4096 cuts fit the device splitter, 4097 do not
        for length in (4096 * seg, 4096 * seg + 1):
            data = (b"z" * (line - 1) + b"\n") * (length // line + 1)
            out.append((f"cuts-seg{seg}-len{length}", data[:length], seg, 5000))
    return out


def test_device_splitter_matches_the_rule(dev):
    rng = random.Random(99)
    inputs = [(n, d, s, m) for n, d, s, m in enumerated_cases()]
    inputs += [(f"random{k}", random_batch(rng), rng.choice([1, 7, 31, 32, 33, 64, 257, 1000]), 4096) for k in range(300)]
    inputs += device_only_split_cases()
    refused_by_device_only = 0
    for k, (name, data, seg, max_segments) in enumerate(inputs):
        want = expected_cuts(data, seg, max_segments, device=True)
        host = host_split(data, seg, max_segments)
        if want != CAPACITY:
            assert host == want, name
            check_plan(data, seg, want)
        elif host != CAPACITY:
            refused_by_device_only += 1
            assert -(-len(data) // seg) > 4096, name
        for mis in ((0, 1, 3, 7) if k % 3 == 0 or name.startswith(("gap", "first", "last", "cuts")) else (0,)):
            assert device_split(dev, data, seg, max_segments, mis) == want, f"{name} mis={mis}"
    assert refused_by_device_only == 2


def verdict_batch():
    """Segments of 256 bytes, each ending in a newline, then a short last one without: under seg_bytes = 256 every planted
    fault is a segment of its own."""
    seg = 256

    def part(body: bytes) -> bytes:
        assert len(body) < seg
        return body + b" " * (seg - 1 - len(body)) + b"\n"

    parts = [
        ("valid", part(b'{"a":1,"b":[1,2,3]}\n{"c":"d"}\n[true,false,null]')),
        ("blank lines", b"\n" * seg),
        ("unclosed string", part(b'{"a":1}\n{"s":"never closed')),
        ("control byte", part(b'{"a":"x\x01y"}\n[1]')),
        ("invalid utf-8", part(b'{"a":"\xff"}\n[2]')),
        ("truncated sequence", part(b"[1]\n[2]") [:-3] + b"\xe2\x82\n"),
        ("valid again", part('{"é":"€"}\n[3,4]'.encode())),
        ("truncated at the end", b'{"z":"end"}\n[5]\xf0\x9f'),
    ]
    data = b"".join(p for _, p in parts)
    bounds = np.cumsum([0] + [len(p) for _, p in parts]).tolist()
    return data, seg, parts, bounds


def test_per_segment_verdicts(dev):
    data, seg, parts, bounds = verdict_batch()
    buf, inp = to_device(data, 5)
    offs = dev.split(inp, seg)
    assert offs == bounds == host_split(data, seg, 64) == expected_cuts(data, seg, 64, device=True)
    nseg = len(offs) - 1
    plain = [want_of(data[a:b]) for a, b in zip(offs, offs[1:])]      # every planted fault is what it claims to be
    assert [w.error for w in plain] == [0, EMPTY, UNCLOSED_STRING, UNESCAPED_CHARS, 0, 0, 0, 0]
    assert [w.utf8_error for w in plain] == [0, 0, 0, 0, 1, 1, 0, 1]
    out_full = torch.full((len(data) + 3 * nseg + 64,), -1, dtype=torch.int32, device="cuda")
    for flags in (0, VALIDATE_UTF8, NO_UTF8):
        out_full.fill_(-1)
        worst, counts, errs, u8, idx_offs = dev.run_segments(inp, offs, out_full, flags)
        host = out_full.cpu().numpy().view(np.uint32)
        wants = [want_of(data[a:b], flags) for a, b in zip(offs, offs[1:])]
        for s, w in enumerate(wants):
            label = f"{parts[s][0]} flags={flags}"
            assert errs[s] == w.error, label
            assert counts[s] == (w.n if w.n is not None else 0), label
            assert u8[s] == (-1 if flags & NO_UTF8 else w.utf8_error), label
            o = idx_offs[s]
            assert np.array_equal(host[o : o + w.indexes.size], w.indexes), label
            assert np.all(host[o + w.indexes.size : idx_offs[s + 1]] == SENT), label
        assert worst == max(w.error for w in wants)
        if flags & VALIDATE_UTF8:
            assert errs[4] == errs[5] == errs[7] == UTF8_ERROR

    # too little index room for the last segment: CAPACITY there, the others unaffected, nothing past the room written
    last = nseg - 1
    wl = want_of(data[offs[last] :])
    room = wl.n + 2
    out_full.fill_(-1)
    view = out_full[: idx_offs[last] + room]
    worst, counts, errs, u8, idx_offs2 = dev.run_segments(inp, offs, view, 0)
    assert idx_offs2 == idx_offs
    host = out_full.cpu().numpy().view(np.uint32)
    wcap = want_of(data[offs[last] :], cap=room)
    assert errs[last] == CAPACITY == wcap.error and counts[last] == 0 and u8[last] == wcap.utf8_error
    assert np.array_equal(host[idx_offs[last] : idx_offs[last] + wcap.indexes.size], wcap.indexes)
    assert np.all(host[idx_offs[last] + wcap.indexes.size :] == SENT)
    for s in range(last):
        w = want_of(data[offs[s] : offs[s + 1]])
        assert (errs[s], counts[s], u8[s]) == (w.error, w.n or 0, w.utf8_error), parts[s][0]
        assert np.array_equal(host[idx_offs[s] : idx_offs[s] + w.indexes.size], w.indexes), parts[s][0]
    assert worst == max(errs)


def test_per_segment_verdicts_through_the_batch_entry_points():
    """The same batch through sjb200_batch_run (host batch) and NdjsonBatchDriver (resident shard): the gathered
    {error, n} rows and every segment's indexes."""
    from mojo_simdjson_b200 import _native
    from mojo_simdjson_b200 import batch as batch_mod

    data, seg, parts, bounds = verdict_batch()
    nseg = len(bounds) - 1
    a = np.frombuffer(data, dtype=np.uint8)
    L = _native.lib()
    for flags in (0, VALIDATE_UTF8):
        wants = [want_of(data[x:y], flags) for x, y in zip(bounds, bounds[1:])]
        b = C.c_void_p()
        assert L.sjb200_batch_create(1, None, len(data), seg, 16, 0, C.byref(b)) == 0
        try:
            idx = np.full(len(data) + 3 * nseg + GUARD, SENT, dtype=np.uint32)
            seg_off = (C.c_uint64 * 17)()
            seg_idx = (C.c_uint64 * 17)()
            seg_n = (C.c_uint32 * 16)()
            seg_err = (C.c_int32 * 16)()
            n_out = C.c_uint32(0)
            worst = C.c_int32(-1)
            rc = L.sjb200_batch_run(b, a.ctypes.data, a.size, idx.ctypes.data, len(data) + 3 * nseg, seg_off, seg_idx, seg_n, seg_err, 16,
                                    C.byref(n_out), C.byref(worst), flags)
            assert rc == 0 and n_out.value == nseg
            assert [int(seg_off[i]) for i in range(nseg + 1)] == bounds
            assert worst.value == max(w.error for w in wants)
            for s, w in enumerate(wants):
                assert (seg_err[s], seg_n[s]) == (w.error, w.n or 0), (parts[s][0], flags)
                o = int(seg_idx[s])
                assert o == bounds[s] + 3 * s
                assert np.array_equal(idx[o : o + w.indexes.size], w.indexes), (parts[s][0], flags)
            assert np.all(idx[len(data) + 3 * nseg :] == SENT)
        finally:
            L.sjb200_batch_destroy(b)

        drv = batch_mod.NdjsonBatchDriver(0, seg_bytes=seg, max_segments=16)
        try:
            buf, inp = to_device(data, 3)
            assert drv.plan(inp) == bounds
            out = torch.full((drv.index_capacity(),), -1, dtype=torch.int32, device="cuda")
            v = drv.run(out, flags)
            assert v.worst_error == max(w.error for w in wants)
            assert v.errors == [w.error for w in wants]
            assert v.counts == [[w.n or 0 for w in wants]]
            host = out.cpu().numpy().view(np.uint32)
            for s, w in enumerate(wants):
                o = drv.index_offsets()[s]
                assert np.array_equal(host[o : o + w.indexes.size], w.indexes), (parts[s][0], flags)
        finally:
            drv.close()


def test_mixed_organisations_in_one_call(dev):
    """Segments of about 1 MiB, 30 MiB, 2 KiB, 90 MiB and 1 MiB in one sjb200_batch_run_device call: the persistent kernel,
    the split pair, the persistent kernel, the stream pipeline (with its persistent fallback launch) and the persistent
    kernel again, back to back on shared scratch, generations and speculation flag.  Twice."""
    from mojo_simdjson_b200 import synth

    sizes = [1 << 20, 30 << 20, 2 << 10, 90 << 20, 1 << 20]
    total = sum(sizes) + (1 << 20)
    data = synth.ndjson(total)
    offs, pos = [0], 0
    for s in sizes:
        nl = np.flatnonzero(data[pos + s :] == 0x0A)    # the segment ends at the first line end at or after `s` bytes
        pos = pos + s + int(nl[0]) + 1
        offs.append(pos)
    assert offs[-1] < total
    wants = [oracle.stage1(data[a:b], impl="fast") for a, b in zip(offs, offs[1:])]
    assert all(w.error == 0 for w in wants)
    inp = torch.from_numpy(data).cuda()
    out = torch.empty(offs[-1] + 3 * len(sizes), dtype=torch.int32, device="cuda")
    dev.set_kernel("auto")
    dev.set_warps(0)
    for rep in range(2):
        out.fill_(-1)
        before = dev.launch_count()
        worst, counts, errs, u8, idx_offs = dev.run_segments(inp, offs, out)
        assert dev.launch_count() - before == 1 + 2 + 1 + 4 + 1     # the organisations this test claims to cover
        assert worst == 0
        host = out.cpu().numpy().view(np.uint32)
        for s, w in enumerate(wants):
            assert (errs[s], counts[s], u8[s]) == (0, w.n, 0), (rep, s)
            o = idx_offs[s]
            assert np.array_equal(host[o : o + w.n + 3], w.indexes), (rep, s)


def test_segment_count_limits(dev):
    """256 segments in one call run; 257 are refused with CAPACITY (one result slot per segment), and so is a batch driver
    created for more than 256 segments."""
    from mojo_simdjson_b200 import _native

    lines = [f'{{"k":{i},"v":[{"1," * (i % 7)}0]}}\n'.encode() for i in range(257)]
    data = b"".join(lines)
    offs = np.cumsum([0] + [len(x) for x in lines]).tolist()
    inp = torch.from_numpy(np.frombuffer(data, dtype=np.uint8).copy()).cuda()
    out = torch.full((len(data) + 3 * 257,), -1, dtype=torch.int32, device="cuda")
    worst, counts, errs, u8, idx_offs = dev.run_segments(inp, offs[:257], out)
    assert worst == 0
    host = out.cpu().numpy().view(np.uint32)
    for s in range(256):
        w = want_of(lines[s])
        assert (errs[s], counts[s], u8[s]) == (0, w.n, 0), s
        assert np.array_equal(host[idx_offs[s] : idx_offs[s] + w.n + 3], w.indexes), s
    worst, *_ = dev.run_segments(inp, offs, out)
    assert worst == CAPACITY
    L = _native.lib()
    for max_segments, want_rc in ((256, 0), (257, CAPACITY)):
        b = C.c_void_p()
        assert L.sjb200_batch_create(1, None, 0, 1 << 20, max_segments, 0, C.byref(b)) == want_rc
        L.sjb200_batch_destroy(b)
        b = C.c_void_p()
        assert L.sjb200_batch_create_rank(0, 0, 1, None, 0, 1 << 20, max_segments, 0, C.byref(b)) == want_rc
        L.sjb200_batch_destroy(b)
