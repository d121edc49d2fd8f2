"""GPU differential tests of stage 2 and the pointer lookups on generated JSON (tests/jsongen.py): every result is compared
with Python's json first (the generated value, which tests/test_json_differential.py pins to json.loads) and with the C
stream oracle second (tests/stage2_stream_oracle.c, through tests/test_gpu_stage2_stream.run_stream: verdicts, the split,
every successful slice word for word with the device's doubles restated, the string buffer and the inexact count).

  - NDJSON (LF, CRLF) and concatenated streams through Stage1Context.index, stage2_primitives and stage2_stream at input
    misalignments 0 to 7, and the same documents in one array through the single-document walk
  - streams of more than 2^21 + 4 * 2048 tokens, past one iteration of the single-CTA scans, with documents placed at the
    2^21 boundary: starting at 2^21 - 1, 2^21 and 2^21 + 1, a document at the nesting limit whose opens straddle it, and a
    stray close and an over-deep document just before it followed by valid documents
  - up to 1024 pointers sampled from the documents, and variants that miss, against RFC 6901 over the generated values
  - the host paths (DomParserImplementation: plain and chunked stage 1, stage2_stream, at_pointers) and the segments of one
    NDJSON batch
  - near-valid streams: one mutation in some documents; those get the oracle's verdict, every other document is untouched"""
from __future__ import annotations

import json
import random
import struct

import numpy as np
import pytest

from oracle import oracle
from tests import jsongen as jg
from tests import pointer_oracle as po
from tests import stage2_stream_oracle as so
from tests import test_gpu_stage2_scale as scale
from tests.test_json_differential import (ALL_ONES, as_kernel, bits, check_cells, check_documents, check_split, corpus, expected_cells,
                                          kernel_double, oracle_stream, pointer_set, type_of)

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

from tests.test_gpu_at_pointer import host, walk  # noqa: E402
from tests.test_gpu_stage2_stream import expected_tape, on_device, run_stream, u64  # noqa: E402

TAPE_BLOCK = scale.TAPE_BLOCK
BOUNDARY = scale.SCAN_ITER   # 2^21 tokens: one iteration of the single-CTA scans


@pytest.fixture(scope="module")
def dev():
    from mojo_simdjson_b200 import device

    ctx = device.Stage1Context(0, max_len=(1 << 32) - 1)
    yield ctx
    ctx.close()


def depth(v) -> int:
    if isinstance(v, tuple):
        return 1 + max([depth(x) for _, x in v[1]], default=0)
    if isinstance(v, list):
        return 1 + max([depth(x) for x in v], default=0)
    return 0


def check_stream_documents(got, want, tape, docs, starts, data: bytes):
    """Every document SUCCESS, split where the generator put it, and decoding to its value with the device's doubles."""
    assert not want.doc_error.any() and (u64(got["doc_status"]) == ALL_ONES).all()
    w = oracle.stage1(data, impl="fast" if len(data) > 20000 else "ref")
    check_split(w.indexes, got["doc_first"].cpu().numpy().astype(np.int64), docs, starts)
    check_documents(docs, tape, want.doc_tape, want.string_buf, kernel=True)


# ---- the device path ---------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("mode", ["lf", "crlf", "concat"])
def test_streams_at_every_misalignment(dev, mode):
    data, docs, starts, _ = corpus(0x6E0 + len(mode), 300, mode, templated=150)
    w, want = oracle_stream(data)
    for mis in range(8):
        got, _, tape, _ = run_stream(dev, data, mis, want=want)
        check_stream_documents(got, want, tape, docs, starts, data)


def test_single_walk_of_the_documents_in_one_array(dev):
    """The same kind of documents as elements of one array (one level deeper, so none at the nesting limit)."""
    g = jg.Gen(0x5176)
    docs = [d for d in [g.document() for _ in range(400)] + g.templated(200) if depth(d.value) < jg.MAX_ARRAY_LEVEL - 1]
    data = b"[" + b",\n".join(d.data for d in docs) + b"]"
    walked = scale.walk_on_gpu(dev, data)   # verdict, tape word for word, string buffer and inexact count against the oracle
    assert walked.error == 0 and len(walked.doubles) > 500
    w = oracle.stage1(data, impl="fast")
    sb = oracle.stage2_walk(data, w.indexes, w.n).string_buf
    assert oracle.decode_tape(walked.tape, sb) == [as_kernel(d.value) for d in docs]
    for tok, b, inexact in walked.doubles:   # an exact double is float()'s, bit for bit
        if not inexact:
            assert b == bits(float(tok)), tok


# ---- past one scan iteration ---------------------------------------------------------------------------------------------

STRAY = jg.Doc(b"]\n[", None, [], 2)                                          # a stray close: TAPE_ERROR until the depth is 0 again
OVER_DEEP = jg.Doc(b"[" * 101 + b"1" + b"]" * 101, None, [], 203)            # DEPTH_ERROR
PAD = jg.Doc(b"0", 0, [[]], 1)


@pytest.fixture(scope="module")
def pool():
    g = jg.Gen(0x2021)
    docs = [g.document() for _ in range(2500)] + g.templated(1500)
    b, v, t = jg.Gen(0x2022).deep(1, limit_array=False)   # a chain of objects down to level 100
    return docs, jg.Doc(b, v, list(jg.paths(v)), t)


def scale_stream(pool_docs, nest: jg.Doc, variant: str, seed: int):
    """(docs, what was placed where): pool documents, shuffled, with documents placed around token 2^21.  variant: 'at-1',
    'at0', 'at+1' (a document of the pool starting at 2^21 + offset, after a stray close and an over-deep document just
    before), or 'nest' (the document at the nesting limit, its opens on both sides of 2^21)."""
    r = random.Random(seed)
    order = list(range(len(pool_docs)))
    r.shuffle(order)
    docs, placed = [], {}
    state = {"tok": 0, "next": 0}

    def add(d, name=None):
        if name:
            placed[name] = (len(docs), state["tok"])
        docs.append(d)
        state["tok"] += d.tokens

    def pool_next():
        d = pool_docs[order[state["next"] % len(order)]]
        return d

    def fill_to(target):
        while True:
            d = pool_next()
            if state["tok"] + d.tokens > target:
                break
            add(d)
            state["next"] += 1
        while state["tok"] < target:
            add(PAD)

    if variant == "nest":
        w = oracle.stage1(nest.data)
        b = oracle.structural_bytes(nest.data, w.indexes[: w.n])
        opens = np.nonzero((b == ord("{")) | (b == ord("[")))[0]
        fill_to(BOUNDARY - int(opens[opens.size // 2]))
        add(nest, "nest")
    else:
        off = {"at-1": -1, "at0": 0, "at+1": 1}[variant]
        fill_to(BOUNDARY - 600)
        small = [d for d in pool_docs if 3 <= d.tokens <= 50]
        add(STRAY, "stray")
        add(small[0], "after_stray")
        add(OVER_DEEP, "over_deep")
        add(small[1], "after_over_deep")
        fill_to(BOUNDARY + off)
        rich = next(d for d in pool_docs if 200 <= d.tokens <= 3000 and depth(d.value) >= 4)
        add(rich, "at")
    fill_to(BOUNDARY + 6 * TAPE_BLOCK)
    fill_to(state["tok"] + 4000)
    return docs, placed


@pytest.mark.parametrize("variant", ["at-1", "at0", "at+1", "nest"])
def test_stream_past_one_scan_iteration(dev, pool, variant):
    pool_docs, nest = pool
    docs, placed = scale_stream(pool_docs, nest, variant, seed=len(variant) + 3 * ord(variant[-1]))
    r = random.Random(variant)
    data, starts = jg.stream(docs, r, "concat" if variant == "at0" else "lf")
    got, want, tape, _ = run_stream(dev, data, mis=len(variant) % 4)
    first = want.doc_first.astype(np.int64)
    n = int(first[-1])
    # the sizes this test claims to cover
    assert n > BOUNDARY + 4 * TAPE_BLOCK
    assert np.count_nonzero((first[:-1] // TAPE_BLOCK) != ((first[1:] - 1) // TAPE_BLOCK)) > 500   # documents across CTA boundaries
    for name, (d, tok) in placed.items():
        assert int(first[d]) == tok, name
    if variant == "nest":
        d, tok = placed["nest"]
        w = oracle.stage1(nest.data)
        b = oracle.structural_bytes(nest.data, w.indexes[: w.n])
        opens = tok + np.nonzero((b == ord("{")) | (b == ord("[")))[0]
        assert (opens < BOUNDARY).sum() > 20 and (opens >= BOUNDARY).sum() > 20 and depth(nest.value) == jg.MAX_OBJECT_LEVEL
    else:
        d, tok = placed["at"]
        assert tok == BOUNDARY + {"at-1": -1, "at0": 0, "at+1": 1}[variant] and docs[d].tokens >= 200
        assert BOUNDARY - 600 <= placed["stray"][1] < placed["over_deep"][1] < BOUNDARY - 300
    # verdicts: the two failing documents and nothing else
    failing = {placed[k][0]: c for k, c in (("stray", oracle.TAPE_ERROR), ("over_deep", oracle.DEPTH_ERROR)) if k in placed}
    assert {int(d): int(want.doc_error[d]) for d in np.nonzero(want.doc_error)[0]} == failing
    assert (u64(got["doc_status"])[[d for d in range(len(docs)) if d not in failing]] == ALL_ONES).all()
    check_split(oracle.stage1(data, impl="fast").indexes, first, docs, starts)
    # every valid document against its value: at most 20,000 of them, always those across a CTA boundary or 2^21
    valid = [d for d in range(len(docs)) if d not in failing]
    across = [d for d in valid if first[d] // TAPE_BLOCK != (first[d + 1] - 1) // TAPE_BLOCK]
    rest = sorted(set(valid) - set(across))
    sample = sorted(set(across) | set(random.Random(1).sample(rest, max(0, min(len(rest), 20000 - len(across))))))
    assert len(sample) >= min(20000, len(valid))
    if variant in ("at-1", "nest"):
        assert any(first[d] < BOUNDARY <= first[d + 1] - 1 for d in sample)
    check_documents(docs, tape, want.doc_tape, want.string_buf, which=sample, kernel=True)


# ---- pointer columns -----------------------------------------------------------------------------------------------------

def test_pointer_columns(dev):
    data, docs, starts, _ = corpus(0x9017, 150, "crlf", templated=450)
    pointers = pointer_set(docs, random.Random(7))
    assert len(pointers) > 800
    tape, sb, doc_tape, status = walk(dev, data)
    assert status.numel() == len(docs) and bool((status == -1).all())
    cols = dev.at_pointers(pointers, tape, sb, doc_tape, status)
    ty, code, val = host(cols.type), host(cols.code), host(cols.value)
    want = expected_cells(pointers, docs)
    found = check_cells(want, ty, code, val, host(tape), host(doc_tape), host(sb), kernel=True)
    assert found > 5000 and set(np.unique(ty).tolist()) >= set(b'{["ldtfn')
    assert {0, po.NO_SUCH_FIELD, po.INDEX_OUT_OF_BOUNDS, po.INCORRECT_TYPE, po.INVALID_JSON_POINTER} <= set(np.unique(code).tolist())
    # the typed views of the columns, against the values
    hit = [k for k in range(len(pointers)) if any(c == 0 for c, _ in want[k])]
    for k in hit[:200]:
        ints, m_i = cols.int64(k)
        flts, m_f = cols.float64(k)
        bools, m_b = cols.boolean(k)
        row = [v if c == 0 else None for c, v in want[k]]
        is_l = [c == 0 and type_of(v) == ord("l") for c, v in want[k]]
        is_d = [c == 0 and type_of(v) == ord("d") for c, v in want[k]]
        is_b = [c == 0 and isinstance(v, bool) for c, v in want[k]]
        assert host(m_i).tolist() == is_l and host(ints).tolist() == [v if f else 0 for v, f in zip(row, is_l)]
        assert host(m_f).tolist() == [a or b for a, b in zip(is_l, is_d)]
        want_f = [float(v) if a else kernel_double(v) if b else 0.0 for v, a, b in zip(row, is_l, is_d)]
        assert host(flts).view(np.int64).tolist() == [struct.unpack("<q", struct.pack("<d", x))[0] for x in want_f], k
        assert host(m_b).tolist() == is_b and host(bools).tolist() == [v is True for v in row]


# ---- host paths ----------------------------------------------------------------------------------------------------------

def test_host_paths(dev):
    from mojo_simdjson_b200.dom_parser_implementation import DomParserImplementation

    data, docs, starts, _ = corpus(0x4057, 250, "lf", templated=150)
    pointers = pointer_set(docs, random.Random(11), k=300)
    tape, sb, doc_tape, status = walk(dev, data)
    cols = dev.at_pointers(pointers, tape, sb, doc_tape, status)
    d_tape, d_sb, d_dt = host(tape).view(np.uint64), host(sb), host(doc_tape).astype(np.uint64)
    want = expected_cells(pointers, docs)
    w = oracle.stage1(data, impl="fast")
    for chunk in (None, 64 << 10):
        p = DomParserImplementation(0, max_len=len(data) + 4096, chunk_bytes=chunk)
        try:
            assert p.stage1(data) == 0 and p.n_structural_indexes == w.n
            assert p.stage2_stream() == 0
            st = p.stream
            assert len(st) == len(docs) and st.n_failed == 0
            check_split(w.indexes, st.doc_first, docs, starts)
            assert np.array_equal(st.doc_tape, d_dt[: len(docs) + 1]) and np.array_equal(st.string_buf, d_sb[: st.string_buf.size])
            for d in range(len(docs)):
                assert np.array_equal(st.document(d).tape, d_tape[int(d_dt[d]) : int(d_dt[d + 1])]), d
            check_documents(docs, st.tape, st.doc_tape, st.string_buf, kernel=True)
            assert p.at_pointers(pointers) == 0
            r = p.pointer_cells
            assert np.array_equal(r.code, host(cols.code)) and np.array_equal(r.type, host(cols.type)) and np.array_equal(r.value, host(cols.value))
            for k in range(len(pointers)):
                assert r.strings(k) == [v.encode() if c == 0 and isinstance(v, str) else None for c, v in want[k]], k
        finally:
            p.close()


def test_ndjson_batch_segments(dev):
    """Every segment of one NDJSON batch (documents on one line each), walked as a stream in place."""
    data, docs, starts, _ = corpus(0xBA7C, 900, "lf", templated=300, ws_bytes=b" \t\r", wide=0.0)
    assert b"\n" not in b"".join(d.data for d in docs)
    a, d_in = on_device(data)
    offs = dev.split(d_in, 64 << 10)
    assert len(offs) >= 6
    out = torch.empty(a.size + 3 * len(offs) + 8, dtype=torch.int32, device="cuda")
    worst, counts, errs, _, idx_offs = dev.run_segments(d_in, offs, out)
    assert worst == 0
    starts = np.asarray(starts)
    seen = 0
    for s in range(len(offs) - 1):
        lo, hi = offs[s], offs[s + 1]
        seg = data[lo:hi]
        n = counts[s]
        w = oracle.stage1(seg, impl="fast")
        assert w.n == n
        want = so.stage2_walk_stream(np.frombuffer(seg, dtype=np.uint8), w.indexes[:n], n)
        prims = dev.stage2_primitives(d_in[lo:hi], out[idx_offs[s] :], n)
        got = dev.stage2_stream(d_in[lo:hi], out[idx_offs[s] :], n, prims)
        torch.cuda.synchronize()
        sel = np.nonzero((starts >= lo) & (starts < hi))[0]
        seg_docs = [docs[d] for d in sel]
        check_split(w.indexes, got["doc_first"].cpu().numpy().astype(np.int64), seg_docs, starts[sel] - lo)
        assert not want.doc_error.any() and (u64(got["doc_status"]) == ALL_ONES).all()
        exp, n_inexact = expected_tape(np.frombuffer(seg, dtype=np.uint8), w.indexes[:n], want)
        t = u64(got["tape"])[: exp.size]
        assert np.array_equal(t, exp) and int(got["summary"][3]) == n_inexact
        assert np.array_equal(prims["string_buf"][: want.string_buf.size].cpu().numpy(), want.string_buf)
        check_documents(seg_docs, t, want.doc_tape, want.string_buf, kernel=True)
        seen += len(seg_docs)
    assert seen == len(docs)


# ---- near-valid streams --------------------------------------------------------------------------------------------------

MUTATIONS = ("wrong_close", "missing_colon", "trailing_comma", "bad_escape", "lone_surrogate", "broken_atom")


def mutate(data: bytes, kind: str, r: random.Random):
    """One mutation of a valid document that keeps its bracket depth, so it stays one document; None if it has no place."""
    w = oracle.stage1(data)
    idx = w.indexes[: w.n].astype(np.int64)
    b = oracle.structural_bytes(data, idx)
    at = lambda cs: [int(i) for i, c in zip(idx, b) if c in cs]   # noqa: E731
    if kind == "wrong_close":
        cand = at(b"]}")
        if cand:
            i = r.choice(cand)
            return data[:i] + (b"}" if data[i : i + 1] == b"]" else b"]") + data[i + 1 :]
    elif kind == "missing_colon":
        cand = at(b":")
        if cand:
            i = r.choice(cand)
            return data[:i] + b" " + data[i + 1 :]
    elif kind == "trailing_comma":
        cand = [int(idx[k]) for k in range(1, len(idx)) if b[k] in b"]}" and b[k - 1] not in b"[{"]
        if cand:
            i = r.choice(cand)
            return data[:i] + b"," + data[i:]
    elif kind in ("bad_escape", "lone_surrogate"):
        cand = at(b'"')
        if cand:
            i = r.choice(cand) + 1
            return data[:i] + (b"\\q" if kind == "bad_escape" else r.choice((b"\\ud800x", b"\\uDBFF ", b"\\udc00", b"\\uD800\\u0041"))) + data[i:]
    elif kind == "broken_atom":
        cand = at(b"tfn")
        if cand:
            i = r.choice(cand)
            e = i + {ord("t"): 3, ord("f"): 4, ord("n"): 3}[data[i]]
            return data[:e] + data[e : e + 1].upper() + data[e + 1 :]
    return None


@pytest.mark.parametrize("mode", ["lf", "concat"])
def test_near_valid_streams(dev, mode):
    data0, docs, _, g = corpus(0x7EA2 + len(mode), 400, mode, templated=200, wide=0.0)
    r = random.Random(mode)
    mutated, kinds = {}, {}
    for d in range(len(docs)):
        if r.random() < 0.3:
            kind = r.choice(MUTATIONS)
            m = mutate(docs[d].data, kind, r)
            if m is not None:
                w = oracle.stage1(m)
                assert w.error == 0, m[:80]
                docs[d] = jg.Doc(m, None, [], w.n)
                mutated[d] = kind
                kinds[kind] = kinds.get(kind, 0) + 1
    assert all(kinds.get(k, 0) >= 5 for k in MUTATIONS), kinds
    data, starts = jg.stream(docs, r, mode)
    # run_stream: every document's code against the oracle, every failing document's full status word against the single walk
    got, want, tape, _ = run_stream(dev, data, mis=3)
    check_split(oracle.stage1(data, impl="fast").indexes, want.doc_first, docs, starts)
    err = want.doc_error
    for d, kind in mutated.items():
        assert err[d] != 0, (kind, docs[d].data[:80])
        if kind != "lone_surrogate":   # json.loads takes a lone surrogate
            with pytest.raises(ValueError):
                json.loads(docs[d].data)
    left = [d for d in range(len(docs)) if d not in mutated]
    assert not err[left].any() and (u64(got["doc_status"])[left] == ALL_ONES).all()
    check_documents(docs, tape, want.doc_tape, want.string_buf, which=left, kernel=True)
