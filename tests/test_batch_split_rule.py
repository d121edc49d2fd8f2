"""The rule that cuts an NDJSON batch into segments, restated in Python and checked against sjb200_batch_split_host.

Cut k is the position after the last '\\n' among the bytes [k * seg, (k + 1) * seg), or len once (k + 1) * seg >= len.  A
segment therefore runs from one cut to the next and is at most 2 * seg - 1 bytes long; a line longer than seg_bytes is
accepted unless it leaves a whole window without a newline, and the batch is refused (CAPACITY) only then, or when there
are more windows than max_segments.  No GPU is needed: the host splitter is plain C++ inside libsimdjson_b200.so.  The
device splitter is checked against the same function in tests/test_gpu_host_paths.py."""
import ctypes as C
import random

import pytest

from mojo_simdjson_b200 import _native, errors

CAPACITY = errors.CAPACITY
SEG_LIMIT = 0x7FFFFFFF     # largest seg_bytes either splitter accepts
DEVICE_CUTS = 4096         # cuts the device splitter can hold (its scratch array on the context)


def expected_cuts(data: bytes, seg_bytes: int, max_segments: int, device: bool = False):
    """Segment offsets [0, cut_1, ..., len] of `data`, or CAPACITY.  device=True adds the device splitter's own limit of
    4096 cuts."""
    n = len(data)
    if seg_bytes == 0 or seg_bytes > SEG_LIMIT:
        return CAPACITY
    ncuts = -(-n // seg_bytes)
    if ncuts > max_segments or (device and ncuts > DEVICE_CUTS):
        return CAPACITY
    cuts = [0]
    for k in range(ncuts):
        lo, hi = k * seg_bytes, (k + 1) * seg_bytes
        if hi >= n:
            cut = n
        else:
            p = data.rfind(b"\n", lo, hi)
            if p < 0:
                return CAPACITY
            cut = p + 1
        if cut > cuts[-1]:
            cuts.append(cut)
    return cuts


def host_split(data: bytes, seg_bytes: int, max_segments: int):
    """sjb200_batch_split_host: the offsets, or the error code."""
    L = _native.lib()
    offs = (C.c_uint64 * (max_segments + 2))()
    nseg = C.c_uint32(0xFFFFFFFF)
    rc = L.sjb200_batch_split_host(data, len(data), seg_bytes, offs, max_segments, C.byref(nseg))
    if rc != errors.SUCCESS:
        return rc
    return [int(offs[i]) for i in range(nseg.value + 1)]


def check_plan(data: bytes, seg_bytes: int, cuts):
    """An accepted plan tiles the input; every segment but the last ends in '\\n'; every segment is shorter than 2 * seg."""
    assert cuts[0] == 0 and cuts[-1] == len(data)
    for s, (a, b) in enumerate(zip(cuts, cuts[1:])):
        assert a < b, (s, a, b)
        assert b - a < 2 * seg_bytes, (s, a, b)
        if s + 2 < len(cuts):
            assert data[b - 1 : b] == b"\n", (s, b)


def enumerated_cases():
    """(name, data, seg_bytes, max_segments): the edges of the rule, each small enough to read."""
    out = []

    def add(name, data, seg, max_segments=4096):
        out.append((name, bytes(data), seg, max_segments))

    seg = 16
    for k in (1, 2, 3):
        for d in (-1, 0, 1):
            p = k * seg + d                              # the only newline up to 4 * seg
            data = bytearray(b"x" * (5 * seg))
            data[p] = 0x0A
            add(f"newline-at-{k}seg{d:+d}", data, seg)
            data2 = bytearray(b"x" * (5 * seg))
            for q in range(d % seg, len(data2), seg):     # one newline per window, always at the same phase
                data2[q] = 0x0A
            add(f"newline-every-seg-phase{d:+d}-k{k}", data2[: k * seg + 7], seg)
    add("no-trailing-newline", b'{"a":1}\n{"b":2}\n{"c":3}', 10)
    add("trailing-newline", b'{"a":1}\n{"b":2}\n{"c":3}\n', 10)
    for n in (seg - 1, seg, seg + 1):
        add(f"len-{n}-no-newline", b"x" * n, seg)
        add(f"len-{n}-newline-last", b"x" * (n - 1) + b"\n", seg)
        add(f"len-{n}-newline-first", b"\n" + b"x" * (n - 1), seg)
    add("empty", b"", seg)
    add("all-newlines-seg1", b"\n" * 40, 1)
    add("all-newlines-seg2", b"\n" * 41, 2)
    add("one-byte-seg1", b"x", 1)
    add("two-bytes-seg1", b"xy", 1)
    add("blank-lines", b'{"a":1}\n\n\n\n\n\n\n\n\n\n{"b":2}\n\n\n\n\n\n[3]\n', 8)
    add("only-blank-lines", b"\n" * 100, 7)
    add("crlf", b'{"a":1}\r\n{"bb":22}\r\n{"ccc":333}\r\n[4]\r\n' * 5, 12)
    add("crlf-cr-at-window-end", b"x" * 14 + b"\r\n" + b"y" * 14 + b"\r\n", 15)
    # long lines: a line of seg + 1 .. 2 * seg - 1 bytes is accepted when it starts right after a cut and some window after
    # it still holds a newline; it is refused when a whole window falls inside it
    seg = 1000
    add("line-1500@500", b"x" * 499 + b"\n" + b"y" * 1499 + b"\n" + b"z" * 300, seg)
    add("line-1001@0", b"y" * 1000 + b"\n" + b"z" * 300, seg)
    seg = 32
    for length in (seg + 1, seg + 2, 3 * seg // 2, 2 * seg - 2, 2 * seg - 1):
        for start in (1, seg // 2, seg - 1, seg):       # the line starts right after a newline at start - 1
            data = b"a" * (start - 1) + b"\n" + b"L" * (length - 1) + b"\n" + b"b" * (seg - 1) + b"\n" + b"c" * 5
            add(f"long-line-{length}@{start}", data, seg)
    for max_segments_delta in (0, -1):
        data = (b"[1,2]\n" * 40)
        ncuts = -(-len(data) // 20)
        add(f"max-segments{max_segments_delta:+d}", data, 20, ncuts + max_segments_delta)
    add("max-segments-1-one-window", b"[1]\n[2]\n", 100, 1)
    add("max-segments-0", b"[1]\n", 100, 0)
    add("max-segments-0-empty", b"", 100, 0)
    for seg in (0, (1 << 31) - 1, 1 << 31, 1 << 32, (1 << 64) - 1):
        add(f"seg-{seg}", b'{"a":1}\n{"b":2}\n', seg)
    return out


@pytest.mark.parametrize("name,data,seg,max_segments", enumerated_cases(), ids=[c[0] for c in enumerated_cases()])
def test_host_splitter_follows_the_rule(name, data, seg, max_segments):
    want = expected_cuts(data, seg, max_segments)
    got = host_split(data, seg, max_segments)
    assert got == want
    if want != CAPACITY:
        check_plan(data, seg, got)


def test_rule_pins_what_the_header_documents():
    """The examples the header comment gives, as numbers."""
    seg = 1000
    ok = b"x" * 499 + b"\n" + b"y" * 1499 + b"\n" + b"z" * 300
    cuts = host_split(ok, seg, 16)
    assert cuts == [0, 500, 2000, len(ok)]
    assert cuts[2] - cuts[1] == 1500 > seg                      # a segment longer than seg_bytes
    assert host_split(b"y" * 1000 + b"\n" + b"z" * 300, seg, 16) == CAPACITY   # window [0, 1000) holds no newline
    # the longest possible segment: 2 * seg - 1 bytes
    worst = b"\n" + b"w" * (2 * seg - 2) + b"\n" + b"v" * 10
    cuts = host_split(worst, seg, 16)
    assert cuts == [0, 1, 2 * seg, len(worst)] and cuts[2] - cuts[1] == 2 * seg - 1
    # blank lines are not skipped: a segment may be nothing but newlines
    assert host_split(b"\n" * 10, 3, 16) == [0, 3, 6, 9, 10]


def random_batch(rng: random.Random):
    """Lines of random length (empty ones included), CRLF or LF, with or without a final newline."""
    lines = []
    total = rng.choice([0, 1, 10, 100, 1000, 4000])
    long_bias = rng.random() < 0.3
    crlf = rng.random() < 0.2
    size = 0
    while size < total:
        if long_bias and rng.random() < 0.2:
            n = rng.randint(50, 400)
        else:
            n = rng.choice([0, 0, 1, 2, 5, 10, 30, 80])
        line = bytes(rng.choice(b'{}[]":,0123456789abc ') for _ in range(n)) + (b"\r\n" if crlf else b"\n")
        lines.append(line)
        size += len(line)
    data = b"".join(lines)
    if data and rng.random() < 0.4:
        data = data[: rng.randint(0, len(data))]       # cut anywhere: no trailing newline, or a ragged last line
    return data


def test_host_splitter_random_batches():
    rng = random.Random(20261021)
    accepted = refused = 0
    for it in range(3000):
        data = random_batch(rng)
        seg = rng.choice([1, 2, 3, 7, 8, 31, 32, 33, 64, 100, 257, 1000, 5000])
        ncuts = -(-len(data) // seg)
        max_segments = rng.choice([ncuts, ncuts + 1, max(ncuts - 1, 0), 4096])
        want = expected_cuts(data, seg, max_segments)
        got = host_split(data, seg, max_segments)
        assert got == want, (it, seg, max_segments, data[:200])
        if want == CAPACITY:
            refused += 1
        else:
            accepted += 1
            check_plan(data, seg, got)
    assert accepted > 500 and refused > 500        # both outcomes are exercised, not just one of them
