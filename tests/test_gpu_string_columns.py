"""GPU tests of the string columns (sjb200_string_columns_device_async, Stage1Context.string_columns): offsets, bytes and
summary bit for bit against expected_string_columns (tests/test_string_columns_reference.py) over the device's own cells
and the CPU oracle's, against json.loads and PointerCells.strings on synth NDJSON, and on length distributions that would
unbalance a copy of one thread per cell."""
import json

import numpy as np
import pytest

from mojo_simdjson_b200 import errors
from oracle import oracle
from tests import pointer_oracle as po
from tests import stage2_stream_oracle as so
from tests.test_gpu_at_pointer import walk
from tests.test_pointer_oracle import FAILING, RULES, rfc6901
from tests.test_string_columns_reference import column_lists, expected_string_columns

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

ALL_ONES = (1 << 64) - 1
Q = ord('"')


@pytest.fixture(scope="module")
def dev():
    from mojo_simdjson_b200 import device

    ctx = device.Stage1Context(0, max_len=(1 << 32) - 1)
    yield ctx
    ctx.close()


def host(t: torch.Tensor) -> np.ndarray:
    return t.cpu().numpy()


def raw_call(dev, ty, val, k, d, sb, sb_len, offsets, data, cap, summary, ctx=True):
    rc = dev._lib.sjb200_string_columns_device_async(dev._ctx if ctx else None, ty.data_ptr(), val.data_ptr(), k, d, sb.data_ptr(), sb_len,
                                                     offsets.data_ptr(), None if data is None else data.data_ptr(), cap, summary.data_ptr())
    torch.cuda.synchronize()
    return rc


def assert_columns(sc, want_offsets, want_data: bytes, mask=None):
    assert np.array_equal(host(sc.offsets), want_offsets)
    assert host(sc.data).tobytes() == want_data
    if mask is not None:
        assert np.array_equal(host(sc.mask), mask)


def check_reference(dev, cols, sb):
    """string_columns over the device's cells equals the reference over the same cells, summary included."""
    sc = dev.string_columns(cols, sb)
    offsets, data, summary = expected_string_columns(host(cols.type), host(cols.value), host(sb))
    assert_columns(sc, offsets, data, host(cols.type) == Q)
    s = torch.full((2,), -1, dtype=torch.int64, device="cuda")
    off = torch.empty_like(sc.offsets)
    k, d = cols.type.shape
    assert raw_call(dev, cols.type, cols.value, k, d, sb, sb.numel(), off, None, 0, s) == 0
    assert host(s).tolist() == summary and np.array_equal(host(off), offsets)
    return sc


# ---- 1. the rule table, failing documents between -------------------------------------------------------------------------

def test_rule_table_and_failing_documents(dev):
    docs = list(dict.fromkeys(d for d, _, _ in RULES))
    stream = []
    for i, d in enumerate(docs):
        stream += [d, FAILING[i % len(FAILING)]]
    data = b"\n".join(stream)
    pointers = [p for _, p, _ in RULES]
    tape, sb, doc_tape, status = walk(dev, data)
    cols = dev.at_pointers(pointers, tape, sb, doc_tape, status)
    sc = check_reference(dev, cols, sb)
    # the same offsets and bytes as the reference over the CPU oracle's cells and string buffer
    w = oracle.stage1(data)
    s = so.stage2_walk_stream(data, w.indexes[: w.n], w.n)
    st = np.array([ALL_ONES if e == 0 else int(e) for e in s.doc_error.tolist()], dtype=np.uint64)
    oty, _, oval = po.cells(pointers, s.tape, s.string_buf, s.doc_tape, st)
    offsets, out, _ = expected_string_columns(oty, oval, s.string_buf)
    assert_columns(sc, offsets, out, oty == Q)
    # failing documents and non-string cells are empty and masked out
    d_n = len(stream)
    lens = np.diff(host(sc.offsets)).reshape(len(pointers), d_n)
    mask = host(sc.mask)
    for i, doc in enumerate(stream):
        if doc in FAILING:
            assert not mask[:, i].any() and (lens[:, i] == 0).all()
    assert (lens[~mask] == 0).all() and mask.sum() >= 2
    assert [sc.to_list(k) for k in range(len(pointers))] == column_lists(offsets, out, oty)


# ---- 2. synth NDJSON ------------------------------------------------------------------------------------------------------

SYNTH_STRINGS = ["/text", "/user/screen_name", "/user/description", "/lang", "/entities/hashtags/0/text", "/id", "/missing"]


def test_synth_ndjson_64mib(dev):
    from mojo_simdjson_b200 import synth
    from mojo_simdjson_b200.dom_parser_implementation import DomParserImplementation

    data = bytes(synth.ndjson(64 << 20))
    lines = [ln for ln in data.split(b"\n") if ln]
    tape, sb, doc_tape, status = walk(dev, data)
    assert status.numel() == len(lines) and bool((status == -1).all())
    cols = dev.at_pointers(SYNTH_STRINGS, tape, sb, doc_tape, status)
    sc = dev.string_columns(cols, sb)
    lists = [sc.to_list(k) for k in range(len(SYNTH_STRINGS))]
    step = max(1, len(lines) // 4000)
    for d in range(0, len(lines), step):
        v = json.loads(lines[d])
        for k, p in enumerate(SYNTH_STRINGS):
            c, want = rfc6901(v, p)
            if c == 0 and isinstance(want, str):
                assert lists[k][d] == want.encode("utf-8"), (d, p)
            else:
                assert lists[k][d] is None, (d, p)
    # every column found strings except /id (never a string) and /missing
    found = [sum(x is not None for x in col) for col in lists]
    assert all(f > 0 for f in found[:5]) and found[5:] == [0, 0]
    # the whole output against the host path on the same bytes
    p = DomParserImplementation(0, max_len=len(data) + (1 << 20))
    try:
        assert p.stage1(data) == 0 and p.at_pointers(SYNTH_STRINGS) == 0
        for k in range(len(SYNTH_STRINGS)):
            assert lists[k] == p.pointer_cells.strings(k), SYNTH_STRINGS[k]
    finally:
        p.close()
    column_offsets, column_data, column_mask = sc.column(3)
    assert int(column_offsets[0]) == 0 and int(column_offsets[-1]) == column_data.numel() and column_mask.numel() == len(lines)


# ---- 3. balance edge cases ------------------------------------------------------------------------------------------------

def synthetic_cells(lengths, gaps=None, k: int = 1, seed: int = 0):
    """Cells (type, value) of k columns over a string buffer built here: lengths[i] < 0 is a null cell, else a string of that
    many random bytes whose record starts gaps[i] bytes after the previous one.  Returns device (type, value, sb) and the
    expected offsets and data."""
    rng = np.random.default_rng(seed)
    lengths = np.asarray(lengths, dtype=np.int64)
    gaps = np.zeros(lengths.size, np.int64) if gaps is None else np.asarray(gaps, dtype=np.int64)
    is_str = lengths >= 0
    size = np.where(is_str, gaps + 4 + lengths, 0)
    end = np.cumsum(size)
    pos = end - np.where(is_str, 4 + lengths, 0)
    sb = rng.integers(0, 256, int(end[-1]) + 7, dtype=np.uint8)
    sl = np.where(is_str, lengths, 0)
    for b in range(4):
        sb[pos[is_str] + b] = (sl[is_str] >> (8 * b)) & 0xFF
    ty = np.where(is_str, Q, ord("n")).astype(np.uint8)
    val = np.where(is_str, pos, 0).astype(np.int64)
    offsets = np.zeros(lengths.size + 1, np.int64)
    offsets[1:] = np.cumsum(sl)
    if is_str.sum() < 1000:
        data = b"".join(sb[q + 4 : q + 4 + n].tobytes() for q, n in zip(pos[is_str], sl[is_str]))
    else:
        data = sb[np.repeat(pos + 4 - offsets[:-1], sl) + np.arange(int(offsets[-1]))].tobytes()
    d_n = lengths.size // k
    assert d_n * k == lengths.size
    t = lambda a: torch.from_numpy(a).cuda()   # noqa: E731
    return t(ty.reshape(k, d_n)), t(val.reshape(k, d_n)), t(sb), offsets, data


def check_synthetic(dev, lengths, gaps=None, k: int = 1, small: bool = False):
    from mojo_simdjson_b200.device import PointerColumns

    ty, val, sb, offsets, data = synthetic_cells(lengths, gaps, k)
    if small:   # the builder itself against the reference
        o, d, _ = expected_string_columns(host(ty), host(val), host(sb))
        assert np.array_equal(o, offsets) and d == data
    sc = dev.string_columns(PointerColumns(ty, torch.zeros_like(ty), val), sb)
    assert_columns(sc, offsets, data, host(ty) == Q)
    return sc


def test_one_huge_string_between_nulls(dev):
    n = 100_000
    check_synthetic(dev, [-1] * (n // 2) + [64 << 20] + [-1] * (n // 2))


def test_a_million_one_byte_strings(dev):
    check_synthetic(dev, [1] * (1 << 20))


def test_cell_starts_and_sources_at_every_residue(dev):
    lengths = [i % 71 for i in range(71 * 64)]                  # output cell starts at every residue mod 16
    check_synthetic(dev, lengths, small=True)
    check_synthetic(dev, lengths, gaps=[i % 16 for i in range(len(lengths))])   # records at every residue mod 16
    check_synthetic(dev, [i % 37 for i in range(37 * 48)], gaps=[(3 * i) % 16 for i in range(37 * 48)], small=True)


def test_null_columns_and_runs_of_empty_cells(dev):
    d_n = 5000
    lengths = [-1] * d_n + [(i * 7) % 100 if i % 500 == 0 else -1 for i in range(d_n)] + [-1] * d_n + [0] * d_n
    sc = check_synthetic(dev, lengths, k=4)
    for k in (0, 2, 3):
        off, data, _ = sc.column(k)
        assert int(off[-1]) == 0 and data.numel() == 0
    assert sc.to_list(3) == [b""] * d_n and sc.to_list(0) == [None] * d_n


def test_max_pointer_count(dev):
    docs = [b'{"a":"%s","b":%d,"c":"%s"}' % (b"x" * (i % 40), i, "é中😀".encode() * (i % 3)) for i in range(300)]
    tape, sb, doc_tape, status = walk(dev, b"\n".join(docs))
    pointers = (["/a", "/b", "/c", "/d"] * (po.MAX_COUNT // 4))[: po.MAX_COUNT]
    cols = dev.at_pointers(pointers, tape, sb, doc_tape, status)
    sc = check_reference(dev, cols, sb)
    assert sc.offsets.numel() == po.MAX_COUNT * 300 + 1
    assert sc.to_list(1022) == [("é中😀".encode() * (i % 3)) for i in range(300)]


def test_single_document_walk(dev):
    doc = b'{"s":"a\\u00e9\\ud83d\\ude00\\n","e":"","n":null,"arr":["x","yz"]}'
    tape, sb, doc_tape, status = walk(dev, doc, single=True)
    pointers = ["/s", "/e", "/n", "/arr/1", "/arr", "/zz"]
    cols = dev.at_pointers(pointers, tape, sb, doc_tape, status)
    sc = check_reference(dev, cols, sb)
    v = json.loads(doc)
    assert [sc.to_list(k)[0] for k in range(len(pointers))] == [v["s"].encode(), b"", None, b"yz", None, None]


def test_empty_string_versus_missing_field(dev):
    tape, sb, doc_tape, status = walk(dev, b'{"s":""}\n{"t":1}\n{"s":null}\n{"s":"x"}\n{"s":1}\n[tru]')
    cols = dev.at_pointers(["/s"], tape, sb, doc_tape, status)
    sc = check_reference(dev, cols, sb)
    assert sc.to_list(0) == [b"", None, None, b"x", None, None]
    assert host(sc.mask).tolist() == [[True, False, False, True, False, False]]
    assert host(sc.offsets).tolist() == [0, 0, 0, 0, 1, 1, 1]


# ---- 4. capacity, NULL data, call level -----------------------------------------------------------------------------------

def test_capacity_and_null_data(dev):
    ty, val, sb, offsets, data = synthetic_cells([(i * 13) % 50 - 3 for i in range(2000)], k=2, seed=3)
    total = len(data)
    n = ty.numel()
    summary = torch.full((2,), -1, dtype=torch.int64, device="cuda")
    for cap in (0, 1, 15, 16, 17, 4095, 4096, 4097, total // 2, total - 1):
        out = torch.full((total + 64,), 0xA5, dtype=torch.uint8, device="cuda")
        off = torch.full((n + 1,), -7, dtype=torch.int64, device="cuda")
        assert raw_call(dev, ty, val, 2, n // 2, sb, sb.numel(), off, out, cap, summary) == 0
        h = host(out)
        assert h[:cap].tobytes() == data[:cap] and (h[cap:] == 0xA5).all(), cap
        assert host(summary).tolist() == [total, 0] and np.array_equal(host(off), offsets)
    off = torch.full((n + 1,), -7, dtype=torch.int64, device="cuda")
    assert raw_call(dev, ty, val, 2, n // 2, sb, sb.numel(), off, None, 1 << 30, summary) == 0
    assert host(summary).tolist() == [total, 0] and np.array_equal(host(off), offsets)
    # call level: K·D == 0, NULL pointers, K·D past 2^40
    off = torch.full((4,), -7, dtype=torch.int64, device="cuda")
    for k, d in ((0, 5), (3, 0)):
        summary.fill_(-1)
        assert raw_call(dev, ty, val, k, d, sb, sb.numel(), off, None, 0, summary) == 0
        assert host(summary).tolist() == [0, 0] and host(off).tolist() == [0, -7, -7, -7]
    assert raw_call(dev, ty, val, 1, 1, sb, sb.numel(), off, None, 0, summary, ctx=False) == errors.UNINITIALIZED
    L = dev._lib
    for args in ((None, val.data_ptr(), sb.data_ptr(), off.data_ptr(), summary.data_ptr()), (ty.data_ptr(), None, sb.data_ptr(), off.data_ptr(), summary.data_ptr()),
                 (ty.data_ptr(), val.data_ptr(), None, off.data_ptr(), summary.data_ptr()), (ty.data_ptr(), val.data_ptr(), sb.data_ptr(), None, summary.data_ptr()),
                 (ty.data_ptr(), val.data_ptr(), sb.data_ptr(), off.data_ptr(), None)):
        rc = L.sjb200_string_columns_device_async(dev._ctx, args[0], args[1], 1, 1, args[2], sb.numel(), args[3], None, 0, args[4])
        assert rc == errors.UNINITIALIZED
    rc = L.sjb200_string_columns_device_async(dev._ctx, ty.data_ptr(), val.data_ptr(), 1 << 20, (1 << 20) + 1, sb.data_ptr(), sb.numel(), off.data_ptr(),
                                              None, 0, summary.data_ptr())
    assert rc == errors.CAPACITY
    torch.cuda.synchronize()


# ---- 5. sentinels ---------------------------------------------------------------------------------------------------------

def test_outputs_inside_sentinels(dev):
    ty, val, sb, offsets, data = synthetic_cells([(i * 11) % 90 - 5 for i in range(3000)], gaps=[i % 5 for i in range(3000)], k=3, seed=5)
    total, n = len(data), ty.numel()
    summary = torch.empty(2, dtype=torch.int64, device="cuda")
    for m in range(1, 16):
        out = torch.full((total + 64,), 0x5A, dtype=torch.uint8, device="cuda")
        off = torch.full((n + 1 + 32,), -0x123456789, dtype=torch.int64, device="cuda")
        for cap in (total, total - m, 1 << 40):
            out.fill_(0x5A)
            assert raw_call(dev, ty, val, 3, n // 3, sb, sb.numel(), off[m:], out[m:], cap, summary) == 0
            h, o = host(out), host(off)
            w = min(total, cap)
            assert (h[:m] == 0x5A).all() and h[m : m + w].tobytes() == data[:w] and (h[m + w :] == 0x5A).all(), (m, cap)
            assert (o[:m] == -0x123456789).all() and np.array_equal(o[m : m + n + 1], offsets) and (o[m + n + 1 :] == -0x123456789).all()


# ---- 6. guards ------------------------------------------------------------------------------------------------------------

def test_guards(dev):
    doc = b'{"a":[1,{"b":"xyz"}],"c":"long string value","d":""}'
    tape, sb, doc_tape, status = walk(dev, b"\n".join([doc] * 40))
    pointers = ["/a/1/b", "/c", "/d", "/a"]
    cols = dev.at_pointers(pointers, tape, sb, doc_tape, status)
    full = dev.string_columns(cols, sb)
    assert full.to_list(1) == [b"long string value"] * 40
    ty_h, val_h = host(cols.type), host(cols.value)
    k, d = ty_h.shape
    rec_end = int((val_h.ravel() + 4 + np.diff(host(full.offsets)))[ty_h.ravel() == Q].max())   # where the last record ends
    for cut in (0, 7, 12, int(val_h[1, 20]) + 10, rec_end - 1):
        offsets, data, summary = expected_string_columns(ty_h, val_h, host(sb), strbuf_len=cut)
        assert summary[1] > 0, cut
        off = torch.empty(k * d + 1, dtype=torch.int64, device="cuda")
        out = torch.full((max(len(data), 1) + 16,), 0xEE, dtype=torch.uint8, device="cuda")
        s = torch.empty(2, dtype=torch.int64, device="cuda")
        assert raw_call(dev, cols.type, cols.value, k, d, sb, cut, off, out, out.numel(), s) == 0
        assert host(s).tolist() == summary and np.array_equal(host(off), offsets)
        assert host(out)[: len(data)].tobytes() == data and (host(out)[len(data) :] == 0xEE).all()
        # the cells past the cut have length 0
        lens = np.diff(host(off))
        sb_end = val_h.ravel().astype(np.int64) + 4 + np.where(ty_h.ravel() == Q, np.diff(host(full.offsets)), 0)
        assert (lens[(ty_h.ravel() == Q) & (sb_end > cut)] == 0).all()
        with pytest.raises(RuntimeError):
            dev.string_columns(cols, sb[:cut])
