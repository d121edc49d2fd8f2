"""GPU tests of stage 2 over document streams (sjb200_stage2_stream_device_async, sjb200_stage2_stream,
DomParserImplementation.stage2_stream) against the stream oracle (tests/stage2_stream_oracle.c, which runs the reference's
walk on every document alone).

Per stream: the document count, doc_first, doc_tape, every document's error code, the summary, the string buffer, and
every successful document's slice word for word (double payloads through the restated kernel conversion of
test_gpu_stage2_scale).  The full status word (token index, check, code) of a failing document is compared with the
single-document walk's on that document alone: a document's verdict never depends on its neighbours."""
import ctypes as C

import numpy as np
import pytest

from oracle import oracle
from tests import stage2_stream_oracle as so
from tests import test_gpu_stage2_scale as scale
from tests.test_stage2_oracle import python_document
from tests.test_stage2_stream_oracle import WALK_TABLE

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

ALL_ONES = (1 << 64) - 1
TAPE_BLOCK = 2048


@pytest.fixture(scope="module")
def dev():
    from mojo_simdjson_b200 import device

    ctx = device.Stage1Context(0, max_len=(1 << 32) - 1)
    yield ctx
    ctx.close()


def u64(t: torch.Tensor) -> np.ndarray:
    return t.cpu().numpy().view(np.uint64)


def on_device(data: bytes, mis: int = 0):
    a = np.frombuffer(data, dtype=np.uint8)
    store = torch.full((mis + a.size + 64,), 0x22, dtype=torch.uint8, device="cuda")   # hostile bytes around the stream
    d_in = store[mis : mis + a.size]
    d_in.copy_(torch.from_numpy(a.copy()))
    return a, d_in


def expected_tape(a: np.ndarray, idx: np.ndarray, want: so.StreamWalk):
    """The oracle's stream tape with the double payloads of successful documents replaced by the restated kernel bits, and
    the number of doubles the kernel flags inexact (every float token of the stream counts, whatever its document's verdict)."""
    n = idx.size
    p = oracle.stage2_primitives(a, idx)
    t = want.tape.copy()
    ks = np.nonzero(p.kind == oracle.KIND_FLOAT)[0]
    first = want.doc_first.astype(np.int64)
    doc_of = np.searchsorted(first, np.arange(n), side="right") - 1
    pos = scale.tape_positions(a, idx, p) + 2 * doc_of
    ok = np.asarray(want.doc_error) == 0
    n_inexact = 0
    for k in ks.tolist():
        i = int(idx[k])
        bits, inexact = scale.restated(a[i : i + int(p.value[k])].tobytes())
        n_inexact += inexact
        if ok[doc_of[k]]:
            t[pos[k] + 1] = bits
    return t, n_inexact


def single_status(dev, d_in, d_idx_doc: torch.Tensor, m: int) -> tuple[int, np.ndarray]:
    """The single-document walk on one document's tokens: (summary[0], tape)."""
    prims = dev.stage2_primitives(d_in, d_idx_doc, m)
    tape, summary = dev.stage2_tape(d_in, d_idx_doc, m, prims)
    s = u64(summary)
    return int(s[0]), u64(tape)[: int(s[2])]


def run_stream(dev, data: bytes, mis: int = 0, single_check: bool = True, want=None):
    a, d_in = on_device(data, mis)
    d_idx = torch.empty(a.size + 8, dtype=torch.int32, device="cuda")
    res = dev.index(d_in, d_idx)
    w = oracle.stage1(data, impl="fast" if a.size > 20000 else "ref")
    assert res.error == w.error == 0 and res.n == w.n, data[:60]
    n = w.n
    idx = w.indexes[:n]
    if want is None:
        want = so.stage2_walk_stream(a, idx, n)
    prims = dev.stage2_primitives(d_in, d_idx, n)
    got = dev.stage2_stream(d_in, d_idx, n, prims)
    torch.cuda.synchronize()
    nd = want.doc_error.size
    s = u64(got["summary"])
    status = u64(got["doc_status"])
    codes = [0 if x == ALL_ONES else int(x) & 0xFF for x in status.tolist()]
    assert int(s[0]) == nd, data[:60]
    assert np.array_equal(got["doc_first"].cpu().numpy().astype(np.uint32), want.doc_first)
    assert np.array_equal(u64(got["doc_tape"]), want.doc_tape)
    assert codes == want.doc_error.tolist(), data[:80]
    assert int(s[1]) == int(np.count_nonzero(want.doc_error))
    assert int(s[2]) == int(want.doc_tape[-1])
    assert np.array_equal(prims["string_buf"][: want.string_buf.size].cpu().numpy(), want.string_buf)
    exp, n_inexact = expected_tape(a, idx, want)
    tape = u64(got["tape"])[: int(s[2])]
    for d in np.nonzero(want.doc_error == 0)[0].tolist():
        lo, hi = int(want.doc_tape[d]), int(want.doc_tape[d + 1])
        assert np.array_equal(tape[lo:hi], exp[lo:hi]), (data[:80], d)
    assert int(s[3]) == n_inexact
    if single_check:   # the full status word of every failing document is the single walk's on it alone
        for d in np.nonzero(want.doc_error)[0].tolist():
            f, e = int(want.doc_first[d]), int(want.doc_first[d + 1])
            st, _ = single_status(dev, d_in, d_idx[f:].clone(), e - f)
            assert int(status[d]) == st, (data[:80], d, hex(int(status[d])), hex(st))
    return got, want, tape, n_inexact


def test_synth_ndjson(dev):
    from mojo_simdjson_b200 import synth

    small = bytes(synth.ndjson(1 << 20))
    for mis in (0, 3):
        got, want, tape, n_inexact = run_stream(dev, small, mis)
        assert want.doc_error.size > 500 and not want.doc_error.any()
        if n_inexact == 0:
            lines = [ln for ln in small.split(b"\n") if ln.strip()]
            assert len(lines) == want.doc_error.size
            for d, ln in enumerate(lines):
                assert oracle.decode_tape(tape[int(want.doc_tape[d]) : int(want.doc_tape[d + 1])], want.string_buf) == python_document(ln), d
    big = bytes(synth.ndjson(64 << 20))
    w = oracle.stage1(big, impl="fast")
    assert w.n > (1 << 21) + 4 * TAPE_BLOCK      # past one iteration of the single-CTA scans
    want = so.stage2_walk_stream(np.frombuffer(big, dtype=np.uint8), w.indexes[: w.n], w.n)
    first = want.doc_first.astype(np.int64)
    assert np.count_nonzero((first[:-1] // TAPE_BLOCK) != ((first[1:] - 1) // TAPE_BLOCK)) > 100   # documents across CTA boundaries
    for mis in (0, 3):
        run_stream(dev, big, mis, want=want)


FAILING = [b"]\n[", b"[}", b"[1 2]", b"[tru]", b'["\\q"]', b"[" * 101 + b"1" + b"]" * 101, b"{}"]
GOOD = b'{"a":[1,"x",{"b":null}],"c":-2.5}'


def test_isolation_across_cta_boundaries(dev):
    """A valid line right after each kind of failing document, with the failing document's first token at 2048 m - 2 ...
    2048 m + 2: the line must be SUCCESS with an exact slice, the failing document must keep its own verdict."""
    for m in (1, 3):
        for bad in FAILING:
            for p in range(TAPE_BLOCK * m - 2, TAPE_BLOCK * m + 3):
                data = b"7\n" * p + bad + b"\n" + GOOD + b"\n" + b"8\n"
                got, want, _, _ = run_stream(dev, data, mis=p % 4)
                nd = want.doc_error.size
                assert int(want.doc_first[p]) == p and want.doc_error[p] != 0 and want.doc_error[p + 1] == 0 and nd == p + 3, (bad, p)
    # a container of 2^24 elements: CAPACITY at its close, the line after it untouched
    big = b"[" + b"0," * ((1 << 24) - 1) + b"0]"
    data = b"7\n" * (TAPE_BLOCK - 1) + big + b"\n" + GOOD + b"\n"
    got, want, _, _ = run_stream(dev, data)
    assert want.doc_error.tolist()[-2:] == [oracle.CAPACITY, 0]


def test_one_token_documents(dev):
    """About 3 M documents of one token: the most documents and the longest tape (4 n words) a stream can have."""
    data = b"1\n" * 3_000_000
    got, want, _, _ = run_stream(dev, data)
    assert want.doc_error.size == 3_000_000 and int(want.doc_tape[-1]) == 4 * 3_000_000


def test_single_document_streams_match_the_single_walk(dev):
    """A stream of exactly one document: the same status word as sjb200_stage2_tape_device_async and, on SUCCESS, the same tape."""
    docs = WALK_TABLE + [b'"just a string"', b"12345", b"-0", b"true", b"null", b"[0.1, 1e22, 123456789012345678, 1.5e-7, -2.25]"]
    for data in docs:
        w = oracle.stage1(data)
        if w.error != 0 or not w.n:
            continue
        want = so.stage2_walk_stream(np.frombuffer(data, dtype=np.uint8), w.indexes[: w.n], w.n)
        if want.doc_error.size != 1:
            continue
        got, _, tape, _ = run_stream(dev, data, single_check=False, want=want)
        a, d_in = on_device(data)
        d_idx = torch.from_numpy(w.indexes[: w.n].astype(np.int32)).cuda()
        st, single_tape = single_status(dev, d_in, d_idx, w.n)
        assert int(u64(got["doc_status"])[0]) == st, data
        if st == ALL_ONES:
            assert np.array_equal(tape, single_tape), data
    # an unclosed last document fails at its length, as the single walk fails at n (its first and last token must match,
    # or it fails at its first token)
    got, _, _, _ = run_stream(dev, b'"a" [[1], [2]')
    assert int(u64(got["doc_status"])[1]) == (8 << 16) | oracle.TAPE_ERROR
    got, _, _, _ = run_stream(dev, b'"a" [1, [2')
    assert int(u64(got["doc_status"])[1]) == oracle.TAPE_ERROR


def test_short_tape_buffers(dev):
    from mojo_simdjson_b200 import synth

    data = bytes(synth.ndjson(256 << 10))
    got, want, full, _ = run_stream(dev, data)
    N = int(want.doc_tape[-1])
    a, d_in = on_device(data)
    d_idx = torch.empty(a.size + 8, dtype=torch.int32, device="cuda")
    n = dev.index(d_in, d_idx).n
    prims = dev.stage2_primitives(d_in, d_idx, n)
    for cap in (N - 1, N // 2, 1):
        store = torch.full((cap + 16,), 0x5A5A5A5A5A5A5A5A, dtype=torch.int64, device="cuda")
        view = store[8 : 8 + cap]
        first = torch.empty(n + 1, dtype=torch.int32, device="cuda")
        doc_tape = torch.empty(n + 1, dtype=torch.int64, device="cuda")
        status = torch.empty(n, dtype=torch.int64, device="cuda")
        summary = torch.empty(4, dtype=torch.int64, device="cuda")
        rc = dev._lib.sjb200_stage2_stream_device_async(dev._ctx, d_in.data_ptr(), d_in.numel(), d_idx.data_ptr(), n, prims["kind"].data_ptr(),
                                                        prims["error"].data_ptr(), prims["value"].data_ptr(), prims["str_off"].data_ptr(),
                                                        view.data_ptr(), cap, first.data_ptr(), doc_tape.data_ptr(), status.data_ptr(), summary.data_ptr())
        torch.cuda.synchronize()
        assert rc == 0 and int(summary[2]) == N
        s = u64(store)
        assert np.all(s[:8] == 0x5A5A5A5A5A5A5A5A) and np.all(s[8 + cap :] == 0x5A5A5A5A5A5A5A5A), cap
        assert np.array_equal(s[8 : 8 + cap], full[:cap]), cap


def host_stream(parser, max_docs=None):
    lib = parser._lib
    n = int(parser.n_structural_indexes)
    tape = np.zeros(4 * n, dtype=np.uint64)
    sbuf = np.zeros(parser.length + 2 * n + 64, dtype=np.uint8)
    md = n if max_docs is None else max_docs
    first = np.full(md + 1, 0xFFFFFFFF, dtype=np.uint32)
    doc_tape = np.zeros(md + 1, dtype=np.uint64)
    status = np.zeros(max(md, 1), dtype=np.uint64)
    nd, nf, tl, sl, inexact = (C.c_uint64(0) for _ in range(5))
    rc = lib.sjb200_stage2_stream(parser._ctx, tape.ctypes.data, tape.size, sbuf.ctypes.data, sbuf.size, first.ctypes.data, doc_tape.ctypes.data,
                                  status.ctypes.data, md, C.byref(nd), C.byref(nf), C.byref(tl), C.byref(sl), C.byref(inexact))
    return rc, int(nd.value), int(tl.value), first


def test_host_path_and_facade():
    from mojo_simdjson_b200 import errors, synth
    from mojo_simdjson_b200.dom_parser_implementation import DomParserImplementation

    streams = [bytes(synth.ndjson(1 << 20)), b"{}\n[1]\n" + b"[" * 101 + b"]" * 101 + b'\n{"a":"b"} "c" [1][2]', b"[1] ] [2] 3"]
    for chunk in (None, 4096):
        parser = DomParserImplementation(0, max_len=8 << 20, chunk_bytes=chunk)
        try:
            for data in streams:
                assert parser.stage1(data) == 0
                w = oracle.stage1(data, impl="fast")
                want = so.stage2_walk_stream(np.frombuffer(data, dtype=np.uint8), w.indexes[: w.n], w.n)
                assert parser.stage2_stream() == 0
                st = parser.stream
                nd = want.doc_error.size
                assert len(st) == nd and st.n_failed == int(np.count_nonzero(want.doc_error))
                assert np.array_equal(st.doc_first, want.doc_first) and np.array_equal(st.doc_tape, want.doc_tape)
                assert [st.error(d) for d in range(nd)] == want.doc_error.tolist()
                assert np.array_equal(st.string_buf, want.string_buf)
                for d in range(nd):
                    if st.error(d) == 0:
                        doc = st.document(d)
                        text, ok = doc.dump_raw_tape()
                        assert ok and text.startswith("0 : r"), d
                        if st.inexact_doubles == 0:
                            assert np.array_equal(doc.tape, want.slice(d)), d
                # CAPACITY for max_docs one too small: nothing copied, the sizes set
                rc, got_nd, tl, first = host_stream(parser, max_docs=nd - 1)
                assert rc == errors.CAPACITY and got_nd == nd and tl == int(want.doc_tape[-1]) and np.all(first == 0xFFFFFFFF)
                rc, got_nd, _, first = host_stream(parser, max_docs=nd)
                assert rc == 0 and np.array_equal(first, want.doc_first)
            assert parser.stage1(b'"abc') == errors.UNCLOSED_STRING
            assert host_stream(parser)[0] == errors.UNINITIALIZED
            assert parser.stage2_stream() == errors.UNINITIALIZED
        finally:
            parser.close()


def test_batch_segment_through_the_device_entry_point(dev):
    """One segment of an NDJSON batch, walked in place: (d_buf + seg_offset, seg_len, d_idx + idx_offset, n)."""
    from mojo_simdjson_b200 import synth

    data = bytes(synth.ndjson(4 << 20))
    a, d_in = on_device(data)
    offs = dev.split(d_in, 1 << 20)
    assert len(offs) >= 4
    out = torch.empty(a.size + 3 * len(offs) + 8, dtype=torch.int32, device="cuda")
    worst, counts, errs, _, idx_offs = dev.run_segments(d_in, offs, out)
    assert worst == 0
    s = 2
    seg = data[offs[s] : offs[s + 1]]
    seg_buf = d_in[offs[s] : offs[s + 1]]
    seg_idx = out[idx_offs[s] :]
    n = counts[s]
    w = oracle.stage1(seg, impl="fast")
    assert w.n == n
    want = so.stage2_walk_stream(np.frombuffer(seg, dtype=np.uint8), w.indexes[:n], n)
    prims = dev.stage2_primitives(seg_buf, seg_idx, n)
    got = dev.stage2_stream(seg_buf, seg_idx, n, prims)
    torch.cuda.synchronize()
    assert np.array_equal(got["doc_first"].cpu().numpy().astype(np.uint32), want.doc_first)
    assert not want.doc_error.any() and u64(got["doc_status"]).tolist() == [ALL_ONES] * want.doc_error.size
    exp, _ = expected_tape(np.frombuffer(seg, dtype=np.uint8), w.indexes[:n], want)
    assert np.array_equal(u64(got["tape"])[: exp.size], exp)
    lines = [ln for ln in seg.split(b"\n") if ln.strip()]
    assert len(lines) == want.doc_error.size
