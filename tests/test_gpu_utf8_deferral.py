"""GPU tests of the stream pipeline's deferred UTF-8 validation (csrc/stage1_stream.cuh): violations planted in every slot
of a warp's ring, validated by either flush, in fixed and in ticketed runs, at mixed densities, together with every other
verdict, in batch segments and across the wrap of the 20-bit document generation.

References, independent of each other: the verdict, n and the indexes come from the oracle (flags=1); utf8_error is
checked a second time against Python's strict UTF-8 decoder.  tests/utf8_plants.py builds the documents and plants;
tests/test_utf8_deferral_emulation.py shows on the CPU that each plant lands in the slot, flush and path named here."""
import time

import numpy as np
import pytest

from oracle import oracle
from tests import utf8_plants as up

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

VALIDATE_UTF8, NO_UTF8 = 1, 4


@pytest.fixture(scope="module")
def dev():
    from mojo_simdjson_b200 import device

    ctx = device.Stage1Context(0, max_len=(1 << 32) - 1)
    yield ctx
    ctx.close()


def grid_warps() -> int:
    """Warps of the stream classify kernel's grid, assumed to be 4 CTAs of 8 warps per SM: what the occupancy query gives for
    53760 B of shared memory and 64 registers per thread on a B200 (the library does not report it).  Only where the plants
    sit relative to the end of the fixed-run range depends on it, not their slots (uniform k), and
    utf8_plants.ticketed_plants puts plants on the 2 chunks either side of that end, so a grid that differs by a few
    CTAs still has plants near it."""
    return torch.cuda.get_device_properties(0).multi_processor_count * 4 * 8


class Doc:
    """A document on the device at misalignment `mis`, its oracle result and a host copy; plants are written into both and
    taken back out byte by byte."""

    def __init__(self, img: np.ndarray, mis: int, cap_extra: int = 8):
        self.mis = mis
        self.host = img[mis:].copy()
        self.len = self.host.size
        self.want = oracle.stage1(self.host, flags=VALIDATE_UTF8, impl="fast")
        self.base_valid = up.utf8_valid(self.host.tobytes())
        self.buf = torch.full((mis + self.len + 256,), 0x22, dtype=torch.uint8, device="cuda")
        self.view = self.buf[mis : mis + self.len]
        self.view.copy_(torch.from_numpy(self.host))
        assert self.view.data_ptr() % 16 == mis
        self.out = torch.empty(self.want.n_written + cap_extra + 3, dtype=torch.int32, device="cuda")
        self.want_idx = torch.from_numpy(self.want.indexes.view(np.int32)).cuda()

    def patch(self, patches):
        """aligned positions -> document positions; returns the patches that undo these"""
        undo = []
        for pos, b in patches:
            p = pos - self.mis
            undo.append((pos, self.host[p : p + len(b)].tobytes()))
            a = np.frombuffer(b, dtype=np.uint8)
            self.host[p : p + len(b)] = a
            self.view[p : p + len(b)].copy_(torch.from_numpy(a.copy()))
        return undo[::-1]

    def run(self, dev, flags=VALIDATE_UTF8, kernel="stream", cap=None):
        dev.set_kernel(kernel)
        try:
            self.out.fill_(-1)          # a run that leaves indexes unwritten must not pass on the previous run's
            out = self.out if cap is None else self.out[:cap]
            return dev.index(self.view, out, flags)
        finally:
            dev.set_kernel("auto")

    def check(self, res, valid, flags=VALIDATE_UTF8, label=""):
        """Compared with the base document's oracle result: a plant changes no index, only the UTF-8 verdict."""
        w = self.want
        assert w.error == 0 and w.utf8_error == 0, label
        want_err = oracle.UTF8_ERROR if (flags & VALIDATE_UTF8) and not valid else 0
        assert (res.error, res.n, res.n_written) == (want_err, w.n, w.n_written), label
        assert res.utf8_error == (-1 if flags & NO_UTF8 else int(not valid)), label
        assert torch.equal(self.out[: w.indexes.size], self.want_idx), label


def _flagged(doc, c):
    """the lanes of chunk c the kernel flags in the document as it now is"""
    return up.flagged_lanes(np.concatenate([np.zeros(doc.mis, np.uint8), doc.host]), doc.mis)[c]


# ------------------------------------------------------------------------------------------------
# every slot, fixed runs: a few hundred chunks, every warp works on its first run only
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [7, 8])
def test_every_slot_fixed_runs(dev, k):
    for layout in ("a", "b"):
        n, last, lanes_of = up.fixed_layout_a(k) if layout == "a" else up.fixed_layout_b(k)
        for mis in (0, 5):
            img = up.build_image(n, mis, lanes_of, last)
            f, cnt = up.lanes_of_doc(img, mis)
            assert (cnt[:-1] == k).all()
            doc = Doc(img, mis)
            assert doc.base_valid
            res = doc.run(dev)
            doc.check(res, True, label="base")
            slots = set()
            for slot, kind, c, lane, make in up.fixed_plants(k, layout, n):
                for valid in (False, True):
                    undo = doc.patch(make(valid))
                    assert np.array_equal(_flagged(doc, c), f[c])          # the plant flags no other lane
                    assert up.utf8_valid(doc.host.tobytes()) == valid
                    label = f"k={k} layout={layout} mis={mis} slot={slot} {kind} valid={valid}"
                    doc.check(doc.run(dev), valid, label=label)
                    if not valid:
                        for flags in (0, NO_UTF8):
                            doc.check(doc.run(dev, flags=flags), valid, flags, label=f"{label} flags={flags}")
                    doc.patch(undo)
                slots.add(slot)
            assert slots == set(range(4 * k))
            # truncated at the end of the document: the last chunk full (a: slot 4k-1, mid-run flush) or partial (b: slot
            # k-2, end-of-warp flush); only the parked end-of-document bit shows it
            for kind in ("3-byte", "1-byte"):
                for valid in (False, True):
                    undo = doc.patch(up.plant_end(img.size, valid, kind))
                    assert up.utf8_valid(doc.host.tobytes()) == valid
                    last_count = up.lanes_of_doc(np.concatenate([np.zeros(mis, np.uint8), doc.host]), mis)[1][-1]
                    assert last_count == k or (valid and kind == "1-byte" and last_count == k - 1)
                    doc.check(doc.run(dev), valid, label=f"end {kind} layout={layout} mis={mis} valid={valid}")
                    doc.patch(undo)
            doc.check(doc.run(dev), True, label="base again")


# ------------------------------------------------------------------------------------------------
# every slot, ticketed runs: 128 MiB, the stream pipeline chosen automatically
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [8, 7])
def test_every_slot_ticketed_runs(dev, k):
    nchunks = up.ticketed_chunks(128)
    n, last, lanes_of = up.ticketed_layout(k, nchunks)
    img = up.build_image(n, 3, lanes_of, last)
    assert (up.lanes_of_doc(img, 3)[1] == k).all()
    doc = Doc(img, 3)
    assert doc.base_valid
    before = dev.launch_count()
    doc.check(doc.run(dev, kernel="auto"), True, label="base")
    assert dev.launch_count() - before == 4           # classify, span scan, flatten, the persistent fallback
    plants = up.ticketed_plants(k, nchunks, 4 * grid_warps())
    assert {s for s, *_ in plants} == set(range(4 * k))
    for slot, c, lane, make in plants:
        for valid in (False, True):
            patches = make(valid)
            undo = doc.patch(patches)
            lo = patches[0][0] - doc.mis
            assert up.utf8_valid_around(doc.host, lo, lo + len(patches[0][1])) == valid
            doc.check(doc.run(dev, kernel="auto"), valid, label=f"k={k} slot={slot} chunk={c} lane={lane} valid={valid}")
            doc.patch(undo)
    doc.check(doc.run(dev, kernel="auto"), True, label="base again")


# ------------------------------------------------------------------------------------------------
# mixed densities: 256 MiB, k from 0..12 per chunk, rings carried partly filled from run to run
# ------------------------------------------------------------------------------------------------
def test_mixed_densities(dev):
    img, counts = up.mixed_density_image(256, 0)
    doc = Doc(img, 0)
    assert doc.base_valid
    assert (counts == 0).any() and (counts > 8).any() and ((counts >= 1) & (counts <= 8)).any()
    doc.check(doc.run(dev, kernel="auto"), True, label="base")
    plants = up.mixed_plants(counts.size, 200)
    for i, (c, lane, bad, good) in enumerate(plants):
        for valid, patches in ((False, bad), (True, good)):
            undo = doc.patch(patches)
            lo = patches[0][0]
            assert up.utf8_valid_around(doc.host, lo, lo + len(patches[0][1])) == valid
            doc.check(doc.run(dev, kernel="auto"), valid, label=f"plant {i} chunk={c} (k={counts[c]}) lane={lane} valid={valid}")
            doc.patch(undo)
    for path, (c, lane, patches) in up.three_path_plants(img, counts).items():
        undo = doc.patch(patches)
        assert not up.utf8_valid(doc.host.tobytes())
        for flags in (VALIDATE_UTF8, 0):
            doc.check(doc.run(dev, flags=flags, kernel="auto"), False, flags, label=f"{path} path flags={flags}")
        doc.patch(undo)
    doc.check(doc.run(dev, kernel="auto"), True, label="no violation")


# ------------------------------------------------------------------------------------------------
# the fold against every other verdict
# ------------------------------------------------------------------------------------------------
def _small_base(k=8, mis=0):
    n, last, lanes_of = up.fixed_layout_a(k)
    return up.build_image(n, mis, lanes_of, last)


def _run_raw(dev, data: np.ndarray, flags, kernel="stream", cap=None):
    buf = torch.full((data.size + 256,), 0x22, dtype=torch.uint8, device="cuda")
    buf[: data.size].copy_(torch.from_numpy(data))
    out = torch.full((data.size + 16 if cap is None else cap,), -1, dtype=torch.int32, device="cuda")
    dev.set_kernel(kernel)
    try:
        res = dev.index(buf[: data.size], out, flags)
    finally:
        dev.set_kernel("auto")
    return res, out


def _check_raw(res, out, data, flags, label):
    want = oracle.stage1(data, flags=flags & VALIDATE_UTF8, impl="fast", cap=out.numel())
    assert (res.error, res.n) == (want.error, want.n), label
    if want.error != oracle.CAPACITY:
        assert res.n_written == want.n_written, label
    keep = want.indexes.size
    assert np.array_equal(out[:keep].cpu().numpy().view(np.uint32), want.indexes), label
    py = 0 if up.utf8_valid(data.tobytes()) else 1
    assert res.utf8_error == (-1 if flags & NO_UTF8 else want.utf8_error), label
    if not flags & NO_UTF8:
        assert res.utf8_error == py, label
    return want


def test_fold_against_every_other_verdict(dev):
    img = _small_base()
    parked = up.plant_inside(100, 3)           # chunk 100 has 8 flagged lanes: parked in slot 3
    variants = {
        "unclosed string": [(250 * 2048 + 12, b"x")],
        "control byte after": [(250 * 2048 + 5, b"\x01")],
        "control byte before": [(20 * 2048 + 5, b"\x01")],
        "long backslash run": up.long_backslash_run(),     # the stream pipeline gives the document to the persistent kernel
    }
    for name, extra in variants.items():
        data = up.apply(img, parked + extra)
        assert up.lanes_of_doc(data, 0)[1][100] == 8
        for flags in (0, VALIDATE_UTF8, NO_UTF8):
            res, out = _run_raw(dev, data, flags)
            want = _check_raw(res, out, data, flags, f"{name} flags={flags}")
            if name == "long backslash run":
                assert want.error in (0, oracle.UTF8_ERROR)
            else:
                assert want.error in (oracle.UNCLOSED_STRING, oracle.UNESCAPED_CHARS)
    data = up.apply(img, parked)
    n = oracle.stage1(data, impl="fast").n
    for cap in (n + 2, n // 2):
        for flags in (0, VALIDATE_UTF8, NO_UTF8):
            res, out = _run_raw(dev, data, flags, cap=cap)
            want = _check_raw(res, out, data, flags, f"cap={cap} flags={flags}")
            assert want.error == oracle.CAPACITY


def test_nothing_leaks_between_calls(dev):
    """A deferred violation, a valid document, a violation in an inline chunk, a valid document, the split pair and the
    persistent kernel, back to back, twice."""
    img = _small_base()
    dense = up.build_image(up.FIXED_CHUNKS, 0, lambda c: range(12) if c == 150 else range(8))
    assert up.lanes_of_doc(dense, 0)[1][150] == 12
    seq = [("deferred", up.apply(img, up.plant_owed(60, 5)), "stream"),
           ("valid", img, "stream"),
           ("inline", up.apply(dense, up.plant_owed(150, 9)), "stream"),
           ("valid", img, "stream"),
           ("split pair", up.apply(img, up.plant_inside(7, 2)), "split"),
           ("persistent", img, "persistent"),
           ("deferred again", up.apply(img, up.plant_inside(299, 31, "surrogate")), "stream"),
           ("split valid", img, "split"),
           ("persistent invalid", up.apply(img, up.plant_owed(61, 1)), "persistent"),
           ("valid at last", img, "stream")]
    for rep in range(2):
        for name, data, kernel in seq:
            for flags in (VALIDATE_UTF8, 0):
                res, out = _run_raw(dev, data, flags, kernel=kernel)
                _check_raw(res, out, data, flags, f"{name} rep={rep} flags={flags}")


# ------------------------------------------------------------------------------------------------
# batch segments: a deferred violation in the 90 MiB segment of test_mixed_organisations_in_one_call
# ------------------------------------------------------------------------------------------------
def test_deferred_violation_in_a_batch_segment(dev):
    from mojo_simdjson_b200 import synth

    sizes = [1 << 20, 30 << 20, 2 << 10, 90 << 20, 1 << 20]
    total = sum(sizes) + (1 << 20)
    data = synth.ndjson(total)
    offs, pos = [0], 0
    for s in sizes:
        nl = np.flatnonzero(data[pos + s :] == 0x0A)
        pos = pos + s + int(nl[0]) + 1
        offs.append(pos)
    inp = torch.from_numpy(data).cuda()
    mis = (inp.data_ptr() + offs[3]) % 16
    seg = data[offs[3] : offs[4]]
    img = np.concatenate([np.zeros(mis, np.uint8), seg])
    f, cnt = up.lanes_of_doc(img, mis)
    # a parked lane in the middle of the segment holding a lead byte of a 3-byte sequence: its first continuation becomes 'a'
    hi = np.flatnonzero((seg >= 0xE0) & (seg < 0xF0))
    at = None
    for p in hi[hi.size // 2 :]:
        c, lane = divmod((int(p) + mis) // 64, 32)
        if 1 <= cnt[c] <= 8 and (int(p) + mis) % 64 < 48:
            at = int(p)
            break
    assert at is not None
    bad = data.copy()
    bad[offs[3] + at + 1] = ord("a")
    assert up.lanes_of_doc(np.concatenate([np.zeros(mis, np.uint8), bad[offs[3] : offs[4]]]), mis)[1][c] == cnt[c]
    wants = {flags: [oracle.stage1(bad[a:b], flags=flags, impl="fast") for a, b in zip(offs, offs[1:])] for flags in (0, VALIDATE_UTF8)}
    assert [w.utf8_error for w in wants[0]] == [0, 0, 0, 1, 0]
    assert not up.utf8_valid(bad[offs[3] : offs[4]].tobytes()) and up.utf8_valid(bad[offs[4] : offs[5]].tobytes())
    inp.copy_(torch.from_numpy(bad))
    out = torch.empty(offs[-1] + 3 * len(sizes), dtype=torch.int32, device="cuda")
    dev.set_kernel("auto")
    dev.set_warps(0)
    for rep in range(2):
        for flags in (VALIDATE_UTF8, 0):
            out.fill_(-1)
            before = dev.launch_count()
            worst, counts, errs, u8, idx_offs = dev.run_segments(inp, offs, out, flags)
            assert dev.launch_count() - before == 1 + 2 + 1 + 4 + 1
            assert errs[3] == (oracle.UTF8_ERROR if flags else 0) and u8[3] == 1
            assert (errs[4], u8[4]) == (0, 0)
            assert worst == (oracle.UTF8_ERROR if flags else 0)
            host = out.cpu().numpy().view(np.uint32)
            for s, w in enumerate(wants[flags]):
                assert (errs[s], counts[s], u8[s]) == (w.error, w.n, w.utf8_error), (rep, flags, s)
                assert np.array_equal(host[idx_offs[s] : idx_offs[s] + w.n + 3], w.indexes), (rep, flags, s)
            # the asynchronous entry point: the fold rewrites the segment's device status row
            status = torch.full((len(sizes), 2), -7, dtype=torch.int32, device="cuda")
            assert dev.run_segments_async(inp, offs, out, status, flags) == 0
            torch.cuda.synchronize()
            rows = status.cpu().tolist()
            assert rows == [[w.error, w.n] for w in wants[flags]], (rep, flags)


# ------------------------------------------------------------------------------------------------
# the wrap of the 20-bit generation (capi.cu, plan_document)
# ------------------------------------------------------------------------------------------------
GEN_MAX = (1 << 20) - 1     # generations run 1 .. GEN_MAX; the document after the one with GEN_MAX wraps back to 1


def gen_of(number: int) -> int:
    """The generation of the context's `number`-th planned document (1-based)"""
    return (number - 1) % GEN_MAX + 1


def test_generation_wrap():
    """Assumption, from plan_document: every document a context plans takes exactly one generation, whatever the entry point
    (one per segment of a batch call).  Calls of 256 tiny segments advance a fresh context to the wrap three times.

    The wrap must clear every generation-tagged word, or a document whose generation comes round again reads stale state
    as its own: the deferred-violation flag (spec_flag[1]), the span scan's block aggregates (block_sum) and the look-back
    descriptors (desc).  Early in a cycle a stream-pipeline document with a deferred violation (84 MiB, 11 span-scan
    blocks) and a split-pair document (26 MiB, 832 tiles) take generations g and g + 1; nothing until the wrap touches
    those words again (the documents right before the wrap are one span-scan block, or two tiles, long).  Just after the
    wrap a valid stream-pipeline document of other content takes generation g and a persistent document of other content
    g + 1: stale state gives them a UTF-8 error or wrong indexes.  Traps like this span the first wrap (between two calls)
    and the second (inside one batch call).  Around the third wrap (between calls) the four kinds -- a stream-pipeline
    document with a deferred violation, a valid one, a split-pair document and a persistent one -- are checked right
    before the wrap, at it and right after it.  About 3 x 2^20 documents: 31 s on a B200 at a 1000 W power limit."""
    from mojo_simdjson_b200 import device, synth

    t0 = time.time()
    stream_img = up.build_image(42 * 1024, 0, lambda c: [0, *range(25, 32)])      # 84 MiB: the stream pipeline
    docs = {
        "stream bad": up.apply(stream_img, up.plant_inside(30000, 27)),
        "stream valid": stream_img,
        "stream other": synth.status_array(84 << 20),                               # valid, other aggregates
        "split": synth.status_array(26 << 20),                                      # 26 MiB: the split pair
        "persistent other": synth.ndjson(20 << 20),                                 # 20 MiB: the persistent kernel, 640 tiles
        "persistent": np.frombuffer(b'["\xc3\xa9", ' + b'"\xe2\x82\xac",' * 3000 + b"1]", dtype=np.uint8),
        "split small": synth.status_array(40 << 10),                                # forced split pair: 2 tiles
        "stream small": synth.status_array(600 << 10),                              # forced stream pipeline: one block
    }
    kernel_of = {"split small": "split", "stream small": "stream"}
    wants = {k: oracle.stage1(v, flags=VALIDATE_UTF8, impl="fast") for k, v in docs.items()}
    assert wants["stream bad"].error == oracle.UTF8_ERROR and not up.utf8_valid(docs["stream bad"].tobytes())
    assert all(w.utf8_error == 0 for k, w in wants.items() if k != "stream bad")
    # one buffer: the tiny segments, then every document; the batch call below takes the consecutive segments `batch_order`
    tiny = np.frombuffer(b"[1]\n" * 256, dtype=np.uint8)
    batch_order = ["persistent", "split small", "persistent", "persistent", "stream other", "persistent other", "stream bad", "split"]
    names = batch_order + [k for k in docs if k not in batch_order]
    parts = [tiny] + [docs[k] for k in names]
    offs = np.cumsum([0] + [p.size for p in parts]).tolist()
    at = {k: (offs[1 + j], offs[2 + j]) for j, k in enumerate(names)}
    buf = torch.from_numpy(np.concatenate(parts)).cuda()
    tiny_offs = list(range(0, tiny.size + 1, 4))
    out = torch.empty(buf.numel() + 3 * 300, dtype=torch.int32, device="cuda")
    want_tiny = oracle.stage1(b"[1]\n", impl="ref")
    ctx = device.Stage1Context(0, max_len=(1 << 32) - 1)
    planned = 0
    log = []

    def advance_to(gen):
        """tiny documents until the next document planned takes generation `gen` of a later cycle"""
        nonlocal planned
        target = planned + ((gen - 1 - planned) % GEN_MAX)
        while planned < target:
            m = min(256, target - planned)
            worst, counts, errs, u8, _ = ctx.run_segments(buf, tiny_offs[: m + 1], out, VALIDATE_UTF8)
            assert worst == 0 and counts == [want_tiny.n] * m, planned
            planned += m
        assert gen_of(planned + 1) == gen

    def single(name):
        nonlocal planned
        a, b = at[name]
        ctx.set_kernel(kernel_of.get(name, "auto"))
        out[: b - a + 3].fill_(-1)
        res = ctx.index(buf[a:b], out, VALIDATE_UTF8)
        ctx.set_kernel("auto")
        planned += 1
        log.append((gen_of(planned), name))
        w = wants[name]
        label = (name, planned, gen_of(planned))
        assert (res.error, res.n, res.utf8_error) == (w.error, w.n, w.utf8_error), label
        assert np.array_equal(out[: w.indexes.size].cpu().numpy().view(np.uint32), w.indexes), label

    def batch():
        nonlocal planned
        segs = offs[1 : 2 + len(batch_order)]
        out.fill_(-1)
        worst, counts, errs, u8, idx_offs = ctx.run_segments(buf, segs, out, VALIDATE_UTF8)
        host = out.cpu().numpy().view(np.uint32)
        for s, name in enumerate(batch_order):
            log.append((gen_of(planned + 1 + s), name))
            w = wants[name]
            label = (name, planned + 1 + s, gen_of(planned + 1 + s))
            assert (errs[s], counts[s], u8[s]) == (w.error, w.n, w.utf8_error), label
            assert np.array_equal(host[idx_offs[s] : idx_offs[s] + w.n + 3], w.indexes), label
        planned += len(batch_order)

    try:
        # cycle 1: the traps at generations 1 and 2, then only documents that leave them alone
        single("stream bad")
        single("split")
        advance_to(GEN_MAX - 2)
        for name in ("persistent", "split small", "stream small"):              # right before the first wrap
            single(name)
        single("stream other")                                                  # at the wrap: generation 1
        single("persistent other")                                              # generation 2
        # cycle 2: the traps at generations 3 and 4 (the two documents after these)
        single("stream bad")
        single("split")
        for name in ("persistent", "split small", "stream small"):
            single(name)
        # the wrap inside one batch call: two persistent documents before it (the second one, 40 KiB, is not large enough
        # for the split pair), one at it, one after it, then the traps' victims at generations 3 and 4
        advance_to(GEN_MAX - 1)
        batch()
        assert log[-len(batch_order):] == [(GEN_MAX - 1, "persistent"), (GEN_MAX, "split small"), (1, "persistent"), (2, "persistent"),
                                           (3, "stream other"), (4, "persistent other"), (5, "stream bad"), (6, "split")]
        # cycle 3: the four kinds right before the third wrap, at it and right after it
        advance_to(GEN_MAX - 3)
        for name in ("stream bad", "stream valid", "split", "persistent") * 3:
            single(name)
        assert log[-8] == (1, "stream bad")
    finally:
        ctx.close()
    assert log[2:7] == [(GEN_MAX - 2, "persistent"), (GEN_MAX - 1, "split small"), (GEN_MAX, "stream small"),
                        (1, "stream other"), (2, "persistent other")]
    elapsed = time.time() - t0
    print(f"generation wrap test: {planned} documents planned in {elapsed:.1f} s")
