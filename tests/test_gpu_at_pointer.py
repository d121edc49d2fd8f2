"""GPU tests of the JSON Pointer lookups (sjb200_at_pointers_device_async, sjb200_stage2_stream_at_pointers,
Stage1Context.at_pointers, DomParserImplementation.at_pointers): every cell against the restated rules of
tests/pointer_oracle.py, over tapes from the CPU stream oracle or from the device walk, and against json.loads."""
import ctypes as C
import json
import struct

import numpy as np
import pytest

from mojo_simdjson_b200 import errors
from oracle import oracle
from tests import pointer_oracle as po
from tests import stage2_stream_oracle as so
from tests.test_pointer_oracle import FAILING, RULES, check_cell

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

ALL_ONES = (1 << 64) - 1


@pytest.fixture(scope="module")
def dev():
    from mojo_simdjson_b200 import device

    ctx = device.Stage1Context(0, max_len=(1 << 32) - 1)
    yield ctx
    ctx.close()


def walk(dev, data: bytes, single: bool = False):
    """Stage 1, the primitives and the stream walk (or the single-document walk) on the device.  Returns
    (tape, string_buf, doc_tape, doc_status) as device tensors."""
    a = np.frombuffer(data, dtype=np.uint8).copy()
    d_in = torch.from_numpy(a).cuda()
    d_idx = torch.empty(a.size + 8, dtype=torch.int32, device="cuda")
    r = dev.index(d_in, d_idx)
    assert r.error == 0, data[:60]
    prims = dev.stage2_primitives(d_in, d_idx, r.n)
    if single:
        tape, summary = dev.stage2_tape(d_in, d_idx, r.n, prims)
        doc_tape = torch.stack([torch.zeros_like(summary[2]), summary[2]])
        return tape, prims["string_buf"], doc_tape, summary[:1].clone()
    s = dev.stage2_stream(d_in, d_idx, r.n, prims)
    return s["tape"], prims["string_buf"], s["doc_tape"], s["doc_status"]


def host(t: torch.Tensor) -> np.ndarray:
    return t.cpu().numpy()


def expect(pointers, tape, sb, doc_tape, doc_status, **kw):
    return po.cells(pointers, host(tape).view(np.uint64), host(sb), host(doc_tape), host(doc_status), **kw)


def assert_cells(cols, want):
    ty, code, val = want
    assert np.array_equal(host(cols.code), code)
    assert np.array_equal(host(cols.type), ty)
    assert np.array_equal(host(cols.value), val)


def raw_call(dev, tape, tape_len, sb, sb_len, doc_tape, doc_status, n_docs, pointers, out_ty, out_code, out_val):
    from mojo_simdjson_b200.device import pointer_program

    raw, offs = pointer_program(pointers)
    rc = dev._lib.sjb200_at_pointers_device_async(dev._ctx, tape.data_ptr(), tape_len, sb.data_ptr(), sb_len, doc_tape.data_ptr(), doc_status.data_ptr(),
                                                  n_docs, raw, offs, len(offs) - 1, out_ty.data_ptr(), out_code.data_ptr(), out_val.data_ptr())
    torch.cuda.synchronize()
    return rc


def test_rule_table_as_one_stream(dev):
    docs = list(dict.fromkeys(d for d, _, _ in RULES))
    stream = []
    for i, d in enumerate(docs):
        stream += [d, FAILING[i % len(FAILING)]]
    data = b"\n".join(stream)
    pointers = [p for _, p, _ in RULES]
    tape, sb, doc_tape, status = walk(dev, data)
    assert status.numel() == len(stream)
    cols = dev.at_pointers(pointers, tape, sb, doc_tape, status)
    # the same cells as the restated rules over the CPU oracle's tapes
    w = oracle.stage1(data)
    s = so.stage2_walk_stream(data, w.indexes[: w.n], w.n)
    st = np.array([ALL_ONES if e == 0 else int(e) for e in s.doc_error.tolist()], dtype=np.uint64)
    assert np.array_equal(host(status).view(np.uint64) == ALL_ONES, st == ALL_ONES)
    assert_cells(cols, po.cells(pointers, s.tape, s.string_buf, s.doc_tape, st))
    # and what the table says, with every failing document's cells carrying its own code
    ty, code, val = host(cols.type), host(cols.code), host(cols.value)
    t, sbb = host(tape).view(np.uint64), host(sb).tobytes()
    for i, doc in enumerate(stream):
        if doc in FAILING:
            c = int(host(status)[i]) & 0xFF
            assert c and (code[:, i] == c).all() and (ty[:, i] == 0).all() and (val[:, i] == 0).all()
            continue
        sl = [int(x) for x in t[int(host(doc_tape)[i]) : int(host(doc_tape)[i + 1])]]
        for k, (d, p, e) in enumerate(RULES):
            if d == doc:
                check_cell(sl, sbb, (int(ty[k, i]), int(code[k, i]), int(val[k, i])), e, (doc[:40], p[:40]))


def test_rule_table_single_documents(dev):
    for doc in dict.fromkeys(d for d, _, _ in RULES):
        rows = [(p, e) for d, p, e in RULES if d == doc]
        tape, sb, doc_tape, status = walk(dev, doc, single=True)
        cols = dev.at_pointers([p for p, _ in rows], tape, sb, doc_tape, status)
        assert_cells(cols, expect([p for p, _ in rows], tape, sb, doc_tape, status))
        sl = [int(x) for x in host(tape).view(np.uint64)[: int(host(doc_tape)[1])]]
        for k, (p, e) in enumerate(rows):
            check_cell(sl, host(sb).tobytes(), (int(host(cols.type)[k, 0]), int(host(cols.code)[k, 0]), int(host(cols.value)[k, 0])), e, (doc[:40], p[:40]))


SYNTH_POINTERS = ["/id", "/text", "/user/id", "/user/name", "/user/ratio", "/user/verified", "/user/utc_offset", "/entities/hashtags/0/text",
                  "/entities/hashtags/0/indices/1", "/entities/hashtags/99", "/id/x", "/missing", "/user", "/entities/hashtags", "", "/truncated",
                  "/user/default_profile", "/user/geo_enabled"]


def test_synth_ndjson_4mib_against_oracle(dev):
    from mojo_simdjson_b200 import synth

    data = bytes(synth.ndjson(4 << 20))
    tape, sb, doc_tape, status = walk(dev, data)
    cols = dev.at_pointers(SYNTH_POINTERS, tape, sb, doc_tape, status)
    assert_cells(cols, expect(SYNTH_POINTERS, tape, sb, doc_tape, status))
    code = host(cols.code)
    assert (code == 0).any(axis=1).sum() >= 10 and (code == po.NO_SUCH_FIELD).any() and (code == po.INDEX_OUT_OF_BOUNDS).any()
    assert set(host(cols.type).ravel().tolist()) >= set(b'{["ldtfn')


def test_synth_ndjson_64mib_against_json_loads(dev):
    from mojo_simdjson_b200 import synth

    data = bytes(synth.ndjson(64 << 20))
    lines = data.split(b"\n")
    lines = [ln for ln in lines if ln]
    tape, sb, doc_tape, status = walk(dev, data)
    assert status.numel() == len(lines) and bool((status == -1).all())
    cols = dev.at_pointers(SYNTH_POINTERS, tape, sb, doc_tape, status)
    ty, code, val, sbb = host(cols.type), host(cols.code), host(cols.value), host(sb).tobytes()
    t = host(tape).view(np.uint64)
    dt = host(doc_tape)
    from tests.test_pointer_oracle import cell_value, rfc6901, to_python

    step = max(1, len(lines) // 4000)
    for d in range(0, len(lines), step):
        v = json.loads(lines[d])
        sl = None
        for k, p in enumerate(SYNTH_POINTERS):
            c, want = rfc6901(v, p)
            assert int(code[k, d]) == c, (d, p)
            if c:
                continue
            if int(ty[k, d]) == ord("d"):   # the tape's double bits: exact on the fast path, which synth's ratios take
                assert struct.unpack("<d", struct.pack("<q", int(val[k, d])))[0] == want, (d, p)
            elif int(ty[k, d]) in b"{[":
                sl = sl if sl is not None else [int(x) for x in t[int(dt[d]) : int(dt[d + 1])]]
                assert to_python(cell_value(sl, sbb, int(ty[k, d]), int(val[k, d]))) == want, (d, p)
            else:
                assert cell_value(None, sbb, int(ty[k, d]), int(val[k, d])) == want, (d, p)


def test_failing_documents_between_valid_ones(dev):
    good = b'{"a":[1,{"b":"x"}],"c":true}'
    stream = []
    for f in FAILING:
        stream += [good, f]
    stream.append(good)
    pointers = ["/a/1/b", "/c", "", "/a/2", "/zz"]
    tape, sb, doc_tape, status = walk(dev, b"\n".join(stream))
    cols = dev.at_pointers(pointers, tape, sb, doc_tape, status)
    assert_cells(cols, expect(pointers, tape, sb, doc_tape, status))
    code, st = host(cols.code), host(status)
    for i in range(len(stream)):
        if i % 2:
            assert st[i] != -1 and (code[:, i] == (int(st[i]) & 0xFF)).all()
        else:
            assert code[:, i].tolist() == [0, 0, 0, po.INDEX_OUT_OF_BOUNDS, po.NO_SUCH_FIELD]


def single_cells(dev, doc: bytes, pointers):
    tape, sb, doc_tape, status = walk(dev, doc, single=True)
    assert int(status[0]) == -1
    cols = dev.at_pointers(pointers, tape, sb, doc_tape, status)
    return cols, (tape, sb, doc_tape, status)


def test_wide_object_target_last(dev):
    doc = b"{" + b",".join(b'"k%d":%d' % (i, i) for i in range(100_000)) + b"}"
    cols, _ = single_cells(dev, doc, ["/k99999", "/k0", "/k100000", "/k9999"])
    assert host(cols.code)[:, 0].tolist() == [0, 0, po.NO_SUCH_FIELD, 0]
    assert host(cols.value)[:, 0].tolist() == [99999, 0, 0, 9999]


def deepest(open_: bytes, close: bytes, inner: bytes) -> int:
    d = 1
    while True:
        doc = open_ * (d + 1) + inner + close * (d + 1)
        w = oracle.stage1(doc)
        if oracle.stage2_walk(doc, w.indexes, w.n).error:
            return d
        d += 1


def test_deepest_nests(dev):
    do = deepest(b'{"k":', b"}", b"7")
    da = deepest(b"[", b"]", b"7")
    assert do == da + 1   # arrays hit DEPTH_ERROR one level before objects
    cols, _ = single_cells(dev, b'{"k":' * do + b"7" + b"}" * do, ["/k" * do, "/k" * (do - 1), "/k" * (do + 1)])
    assert host(cols.code)[:, 0].tolist() == [0, 0, po.NO_SUCH_FIELD] and int(host(cols.value)[0, 0]) == 7
    assert int(host(cols.type)[1, 0]) == ord("{")
    cols, _ = single_cells(dev, b"[" * da + b"7" + b"]" * da, ["/0" * da, "/0" * (da + 1), "/0" * (da - 1) + "/1"])
    assert host(cols.code)[:, 0].tolist() == [0, po.NO_SUCH_FIELD, po.INDEX_OUT_OF_BOUNDS] and int(host(cols.value)[0, 0]) == 7


def test_long_arrays(dev):
    n = 1 << 20
    doc = b"[" + b",".join(b"%d" % i for i in range(n)) + b"]"
    cols, t = single_cells(dev, doc, ["/0", f"/{n - 1}", f"/{n}", f"/{n - 2}"])
    assert host(cols.code)[:, 0].tolist() == [0, 0, po.INDEX_OUT_OF_BOUNDS, 0]
    assert host(cols.value)[:, 0].tolist() == [0, n - 1, 0, n - 2]
    m = (1 << 24) - 1
    doc = b"[" + b"0," * (m - 1) + b"0]"
    cols, t = single_cells(dev, doc, [f"/{m}", f"/{m - 1}", "/0"])
    assert host(cols.code)[:, 0].tolist() == [po.INDEX_OUT_OF_BOUNDS, 0, 0]


def test_outputs_inside_sentinels(dev):
    tape, sb, doc_tape, status = walk(dev, b'{"a":[1,2]}\n{"a":"x"}\n[3]')
    nd = status.numel()
    for pointers, n_docs in ((["/a/1", "/a"], nd), (["/a"] * po.MAX_COUNT, nd), (["/a/0"], 1), (["/a"], 0)):
        k = len(pointers)
        pad = 64
        ty = torch.full((k * n_docs + 2 * pad,), 0xA5, dtype=torch.uint8, device="cuda")
        code = torch.full_like(ty, 0x5A)
        val = torch.full((k * n_docs + 2 * pad,), -0x123456789, dtype=torch.int64, device="cuda")
        rc = raw_call(dev, tape, tape.numel(), sb, sb.numel(), doc_tape, status, n_docs, pointers, ty[pad:], code[pad:], val[pad:])
        assert rc == 0
        for t, s in ((ty, 0xA5), (code, 0x5A), (val, -0x123456789)):
            h = host(t)
            assert (h[:pad] == s).all() and (h[pad + k * n_docs :] == s).all(), (k, n_docs)
        if n_docs:
            want = expect(pointers, tape, sb, doc_tape[: n_docs + 1], status[:n_docs])
            assert np.array_equal(host(code)[pad : pad + k * n_docs], want[1].ravel())
            assert np.array_equal(host(ty)[pad : pad + k * n_docs], want[0].ravel())
            assert np.array_equal(host(val)[pad : pad + k * n_docs], want[2].ravel())


def test_call_level_errors_write_nothing(dev):
    tape, sb, doc_tape, status = walk(dev, b'{"a":1}')
    ty = torch.full((4096,), 0xA5, dtype=torch.uint8, device="cuda")
    code, val = torch.full_like(ty, 0x5A), torch.full((4096,), 7, dtype=torch.int64, device="cuda")
    cases = [(["/a", "a"], errors.INVALID_JSON_POINTER), (["#/a"], errors.INVALID_JSON_POINTER), (["/a~"], errors.INVALID_JSON_POINTER),
             (["/a~2b"], errors.INVALID_JSON_POINTER), (["/a"] * (po.MAX_COUNT + 1), errors.CAPACITY), (["/" + "a" * po.MAX_BYTES], errors.CAPACITY)]
    for pointers, want in cases:
        assert raw_call(dev, tape, tape.numel(), sb, sb.numel(), doc_tape, status, 1, pointers, ty, code, val) == want, pointers[0][:10]
        assert po.check_call([p.encode() for p in pointers]) == want
    assert (host(ty) == 0xA5).all() and (host(code) == 0x5A).all() and (host(val) == 7).all()
    assert raw_call(dev, tape, tape.numel(), sb, sb.numel(), doc_tape, status, 1, ["/" + "a" * (po.MAX_BYTES - 1)], ty, code, val) == 0
    assert host(code)[0] == po.NO_SUCH_FIELD
    # at the byte limit with one token per two bytes: the program of one pointer needs more than 48 KiB of shared memory
    for doc, pointers in ((b"[0]", ["/0" * (po.MAX_BYTES // 2)]), (b'{"a":1}', ["/a", "/" * (po.MAX_BYTES - 2)])):
        tape, sb, doc_tape, status = walk(dev, doc)
        cols = dev.at_pointers(pointers, tape, sb, doc_tape, status)
        assert_cells(cols, expect(pointers, tape, sb, doc_tape, status))
    with pytest.raises(ValueError):
        dev.at_pointers(["a"], tape, sb, doc_tape, status)


def test_guards(dev):
    doc = b'{"a":[1,{"b":"xyz"}],"c":"long string value"}'
    tape, sb, doc_tape, status = walk(dev, doc, single=True)
    m = int(doc_tape[1])
    # the slice in the middle of a larger tensor of valid-looking words, its container word pointing past the slice
    big = torch.zeros(3 * m + 16, dtype=torch.int64, device="cuda")
    big[m : 2 * m] = tape[:m]
    big[2 * m :] = tape[1]
    t = host(tape).view(np.uint64)[:m].copy()
    t[1] = (t[1] & np.uint64(~0xFFFFFFFF & (2**64 - 1))) | np.uint64(m + 3)
    big[m : 2 * m] = torch.from_numpy(t.view(np.int64)).cuda()
    dt = torch.tensor([m, 2 * m], dtype=torch.int64, device="cuda")
    pointers = ["/a/1/b", "", "/c"]
    cols = dev.at_pointers(pointers, big, sb, dt, status)
    assert host(cols.code)[:, 0].tolist() == [po.TAPE_ERROR, 0, po.TAPE_ERROR]
    assert_cells(cols, expect(pointers, big, sb, dt, status))
    # tape_len and strbuf_len cut short
    ty = torch.zeros(3, dtype=torch.uint8, device="cuda")
    code, val = torch.zeros_like(ty), torch.zeros(3, dtype=torch.int64, device="cuda")
    assert raw_call(dev, tape, m - 1, sb, sb.numel(), doc_tape, status, 1, pointers, ty, code, val) == 0
    assert host(code).tolist() == [po.CAPACITY] * 3
    sb_len = 12   # records in index order: "a" at 0, "b" at 5, "xyz" at 10: the keys fit, "xyz" and every later record do not
    want = expect(pointers, tape, sb, doc_tape, status, strbuf_len=sb_len)
    assert raw_call(dev, tape, tape.numel(), sb, sb_len, doc_tape, status, 1, pointers, ty, code, val) == 0
    assert host(code).tolist() == want[1][:, 0].tolist() and po.CAPACITY in host(code).tolist()
    assert host(val).tolist() == want[2][:, 0].tolist()


def test_host_path(dev):
    from mojo_simdjson_b200 import synth
    from mojo_simdjson_b200.dom_parser_implementation import DomParserImplementation

    data = bytes(synth.ndjson(1 << 20)) + b"\n" + b"\n".join(FAILING[:3]) + b"\n[1][2]{}{}"
    p = DomParserImplementation(0, max_len=4 << 20)
    try:
        assert p.at_pointers(["/id"]) == errors.UNINITIALIZED
        assert p.stage1(data) == 0
        # device path on the same bytes
        tape, sb, doc_tape, status = walk(dev, data)
        cols = dev.at_pointers(SYNTH_POINTERS, tape, sb, doc_tape, status)
        assert p.at_pointers(SYNTH_POINTERS) == 0
        r = p.pointer_cells
        assert np.array_equal(r.code, host(cols.code)) and np.array_equal(r.type, host(cols.type)) and np.array_equal(r.value, host(cols.value))
        # strings(k) against the oracle's string buffer
        w = oracle.stage1(data)
        s = so.stage2_walk_stream(data, w.indexes[: w.n], w.n)
        st = np.array([ALL_ONES if e == 0 else int(e) for e in s.doc_error.tolist()], dtype=np.uint64)
        oty, ocode, oval = po.cells(SYNTH_POINTERS, s.tape, s.string_buf, s.doc_tape, st)
        osb = s.string_buf.tobytes()
        for k in range(len(SYNTH_POINTERS)):
            want = [osb[v + 4 : v + 4 + int.from_bytes(osb[v : v + 4], "little")] if t == ord('"') else None for t, v in zip(oty[k].tolist(), oval[k].tolist())]
            assert r.strings(k) == want
        assert any(x is not None for x in r.strings(1))
        # INVALID_JSON_POINTER leaves the previous result alone
        assert p.at_pointers(["/id", "x"]) == errors.INVALID_JSON_POINTER and p.pointer_cells is r
        # CAPACITY, then a retry with the sizes the call reports
        L = p._lib
        from mojo_simdjson_b200.device import pointer_program

        raw, offs = pointer_program(["/id", "/text"])
        nd, sl = C.c_uint64(0), C.c_uint64(0)
        ty, code, val = np.zeros(8, np.uint8), np.full(8, 9, np.uint8), np.zeros(8, np.int64)
        sbuf = np.zeros(16, np.uint8)
        rc = L.sjb200_stage2_stream_at_pointers(p._ctx, raw, offs, 2, ty.ctypes.data, code.ctypes.data, val.ctypes.data, 8, sbuf.ctypes.data, 16,
                                                C.byref(nd), C.byref(sl))
        assert rc == errors.CAPACITY and (code == 9).all()
        assert nd.value == status.numel() and sl.value > 16
        cells = 2 * nd.value
        ty, code, val = np.zeros(cells, np.uint8), np.zeros(cells, np.uint8), np.zeros(cells, np.int64)
        sbuf = np.zeros(sl.value, np.uint8)
        rc = L.sjb200_stage2_stream_at_pointers(p._ctx, raw, offs, 2, ty.ctypes.data, code.ctypes.data, val.ctypes.data, cells, sbuf.ctypes.data, sbuf.size,
                                                C.byref(nd), C.byref(sl))
        assert rc == 0
        assert np.array_equal(code.reshape(2, -1), r.code[:2]) and np.array_equal(val.reshape(2, -1), r.value[:2])
        assert np.array_equal(sbuf, r.string_buf)
        # without a string buffer only the cells are copied
        rc = L.sjb200_stage2_stream_at_pointers(p._ctx, raw, offs, 2, ty.ctypes.data, code.ctypes.data, val.ctypes.data, cells, None, 0, C.byref(nd), C.byref(sl))
        assert rc == 0 and np.array_equal(code.reshape(2, -1), r.code[:2])
    finally:
        p.close()


def test_column_conversions(dev):
    doc = b"\n".join([b'{"v":1}', b'{"v":-9007199254740993}', b'{"v":2.5}', b'{"v":true}', b'{"v":false}', b'{"v":null}', b'{"v":"s"}', b'{"w":1}',
                      b'{"v":[1]}', b'{"v":tru}', b'{"v":9223372036854775807}', b'{"v":-0.0}'])
    tape, sb, doc_tape, status = walk(dev, doc)
    cols = dev.at_pointers(["/v", "/w"], tape, sb, doc_tape, status)
    ty, val = host(cols.type)[0], host(cols.value)[0]
    v, m = cols.int64(0)
    assert np.array_equal(host(m), ty == ord("l")) and np.array_equal(host(v), np.where(ty == ord("l"), val, 0))
    f, m = cols.float64(0)
    want = np.where(ty == ord("d"), val.view(np.float64), np.array([float(int(x)) for x in val]))
    want = np.where((ty == ord("d")) | (ty == ord("l")), want, 0.0)
    assert np.array_equal(host(m), (ty == ord("d")) | (ty == ord("l")))
    assert np.array_equal(host(f).view(np.int64), want.view(np.int64))
    b, m = cols.boolean(0)
    assert np.array_equal(host(m), (ty == ord("t")) | (ty == ord("f"))) and np.array_equal(host(b), ty == ord("t"))
    assert host(m).tolist() == [False, False, False, True, True, False, False, False, False, False, False, False]
    assert int(host(cols.code)[0, 9]) == 6   # T_ATOM_ERROR of the failing document
