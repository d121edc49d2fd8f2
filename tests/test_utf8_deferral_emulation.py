"""CPU checks of the stream pipeline's deferred UTF-8 validation through the host emulator (tests/emu,
emu_stage1_stream_sched): the straddle gate of the inline path, the slots and flushes of the warps' rings under any
schedule of the ticket counter, the fold of a parked violation into the verdict, and that the documents of
tests/test_gpu_utf8_deferral.py put every planted violation in the slot, flush and path the GPU tests name."""
import numpy as np
import pytest

from oracle import oracle
from tests import cases, emu
from tests import utf8_plants as up

GRID_WARPS = 148 * 4 * 8          # the stream classify kernel's grid on a B200: 4 CTAs of 8 warps per SM
SCHEDULES = [(GRID_WARPS, 1), (64, 2), (5, 3)]


def _want(data, flags):
    return oracle.stage1(data, flags=flags, impl="fast" if len(data) > 20000 else "ref")


def _check(data, mis, flags, schedules=SCHEDULES):
    want = _want(data, flags)
    for warps, seed in schedules:
        r = emu.stage1_stream_sched(data, mis=mis, flags=flags, warps=warps, seed=seed)
        if r.gave_up:   # the device hands such a document to the persistent kernel (test_core_emulation covers when)
            return
        label = f"warps={warps} seed={seed} mis={mis} flags={flags}"
        assert (r.err, r.n, r.n_written, r.utf8) == (want.error, want.n, want.n_written, want.utf8_error), label
        assert np.array_equal(r.out, want.indexes), label


def test_schedule_model_agrees_with_oracle_on_corpus():
    for name, data in cases.adversarial_cases(tile_bytes=(2048, 4096, 16384)):
        if not data:
            continue
        for mis in (0, 5):
            try:
                _check(data, mis, 0)
                _check(data, mis, 1)
            except AssertionError as e:  # pragma: no cover
                raise AssertionError(f"case {name}") from e


def test_utf8_cases_at_every_lane_and_chunk_edge():
    """Every valid and invalid sequence of the corpus at the edges of a lane and a chunk, in few or many flagged lanes."""
    seqs = [s if isinstance(s, (bytes, bytearray)) else s.encode("utf-8", "surrogatepass") for s in list(cases.UTF8_VALID) + list(cases.UTF8_INVALID)]
    for k, seq in enumerate(seqs):
        for pos in (0, 1, 61, 62, 63, 64, 2045, 2046, 2047, 2048, 4095, 6000):
            body = bytearray(b"a" * 7000)
            body[pos:pos] = seq
            dense = bytearray("é".encode() * 1000) + body    # most lanes of the first chunk flagged: inline
            for data in (b'"' + bytes(body) + b'"', b'"' + bytes(body[: pos + len(seq)]), b'"' + bytes(dense[: pos + 2000 + len(seq)])):
                _check(data, (k + pos) % 16, 1, SCHEDULES[1:])


def test_straddle_gate_is_exact():
    """Over all 2^24 values of the three bytes before a lane: wherever the gate is closed, the carry it skips is zero."""
    miss, closed = emu.straddle_gate_misses()
    assert miss == 0
    assert closed == 192 ** 3          # closed exactly when none of the three bytes is >= 0xC0


@pytest.mark.parametrize("k", [7, 8])
def test_slot_determinism(k):
    """Every chunk with exactly k flagged lanes (any lanes): the lane of rank r in chunk c is parked in slot k (c mod 4) + r
    under every schedule, and the ring is flushed after the 4th chunk of every run, full (32) at k = 8."""
    rng = np.random.default_rng(k)
    nchunks = 4 * 40 + 2
    img = up.build_image_from_counts(np.full(nchunks, k), 3, rng)
    f, cnt = up.lanes_of_doc(img, 3)
    assert (cnt == k).all()
    ch, lane = np.nonzero(f)
    probes = [(int(c) * 32 + int(l)) * 64 + 30 - 3 for c, l in zip(ch, lane)]
    rank = np.concatenate([np.arange(k)] * nchunks)
    want = _want(img[3:], 1)
    for warps, seed in [(GRID_WARPS, 0), (16, 1), (7, 2), (3, 3), (1, 4)]:
        r = emu.stage1_stream_sched(img[3:], mis=3, flags=1, warps=warps, seed=seed, probes=probes)
        assert (r.err, r.n, r.utf8) == (want.error, want.n, 0)
        assert [p.kind for p in r.probes] == [emu.PARKED] * len(probes)
        assert [p.slot for p in r.probes] == [up.slot_uniform(k, int(c), int(q)) for c, q in zip(ch, rank)], (warps, seed)
        full_runs = nchunks // 4
        assert r.mid_run_flushes == full_runs
        assert r.end_of_warp_flushes == 1                  # the last run has 2 chunks
        assert r.max_fill == 4 * k
        flushes = [p.flush for p in r.probes]
        assert flushes == [emu.MID_RUN] * (full_runs * 4 * k) + [emu.END_OF_WARP] * (2 * k)


def test_fold_order():
    """A parked violation turns only SUCCESS into UTF8_ERROR (flag 1) and always sets utf8_error."""
    n, last, lanes = up.fixed_layout_a(8)
    img = up.build_image(n, 0, lanes, last)
    bad = up.apply(img, up.plant_inside(12, 3))
    variants = {
        "plain": bad,
        "unclosed string": up.apply(bad, [(20 * 2048 + 12, b"x")]),                 # an opening quote becomes a letter
        "control byte": up.apply(bad, [(30 * 2048 + 5, b"\x01")]),
        "control byte before": up.apply(bad, [(2 * 2048 + 5, b"\x01")]),
    }
    for name, data in variants.items():
        for flags in (0, 1):
            want = _want(data, flags)
            r = emu.stage1_stream_sched(data, flags=flags, probes=[12 * 2048 + 3 * 64 + up.INSIDE])
            assert r.probes[0].kind == emu.PARKED, name
            assert (r.err, r.n, r.utf8) == (want.error, want.n, want.utf8_error) == (r.err, r.n, 1), (name, flags)
    # the long backslash run the GPU test adds beside a parked violation: the speculation gives up on it
    r = emu.stage1_stream_sched(up.apply(bad, up.long_backslash_run()), flags=1)
    assert r.gave_up
    want = _want(bad, 1)
    for cap in (want.n + 2, want.n // 2):
        w = oracle.stage1(bad, flags=1, impl="fast", cap=cap)
        r = emu.stage1_stream_sched(bad, flags=1, cap=cap)
        assert (r.err, r.utf8) == (w.error, w.utf8_error) == (oracle.CAPACITY, 1)


# ------------------------------------------------------------------------------------------------
# the documents of tests/test_gpu_utf8_deferral.py reach what its tests claim
# ------------------------------------------------------------------------------------------------
def _probe_pos(c, lane, mis):
    return (c * 32 + lane) * 64 + up.INSIDE - mis


@pytest.mark.parametrize("k", [7, 8])
@pytest.mark.parametrize("layout", ["a", "b"])
def test_fixed_run_documents_reach_their_slots(k, layout):
    n, last, lanes_of = up.fixed_layout_a(k) if layout == "a" else up.fixed_layout_b(k)
    for mis in (0, 5):
        img = up.build_image(n, mis, lanes_of, last)
        f, cnt = up.lanes_of_doc(img, mis)
        assert (cnt[:-1] == k).all() and cnt[-1] == (k if layout == "a" else k - 1)
        plants = up.fixed_plants(k, layout, n)
        slots = set()
        for slot, kind, c, lane, make in plants:
            for valid in (False, True):
                data = up.apply(img, make(valid))
                f2, cnt2 = up.lanes_of_doc(data, mis)
                assert np.array_equal(f2, f), (slot, kind)        # the plant changes no lane's flag
                if valid:
                    continue
                want = _want(data[mis:], 1)
                r = emu.stage1_stream_sched(data[mis:], mis=mis, flags=1, probes=[_probe_pos(c, lane, mis)])
                p = r.probes[0]
                assert (p.kind, p.slot, p.flush) == (emu.PARKED, slot, emu.MID_RUN), (slot, kind)
                assert p.warp == c // 4                          # the warp's first run: fixed, not drawn
                assert (r.err, r.utf8) == (want.error, want.utf8_error) == (oracle.UTF8_ERROR, 1), (slot, kind)
                assert not up.utf8_valid(data[mis:])
                slots.add(slot)
        assert slots == set(range(4 * k))
        # the end of the document: the last lane of a full chunk (layout a) or of a partial one (layout b)
        end = up.plant_end(img.size)
        assert up.lanes_of_doc(up.apply(img, end), mis)[1][-1] == k
        r = emu.stage1_stream_sched(up.apply(img, end)[mis:], mis=mis, flags=1, probes=[img.size - 1 - mis])
        p = r.probes[0]
        if layout == "a":
            assert (p.kind, p.slot, p.flush) == (emu.PARKED, 4 * k - 1, emu.MID_RUN)
        else:
            assert (p.kind, p.slot, p.flush) == (emu.PARKED, k - 2, emu.END_OF_WARP)
        assert (r.err, r.utf8) == (oracle.UTF8_ERROR, 1)
        r = emu.stage1_stream_sched(up.apply(img, up.plant_end(img.size, valid=True))[mis:], mis=mis, flags=1)
        assert (r.err, r.utf8) == (0, 0)
        base = emu.stage1_stream_sched(img[mis:], mis=mis, flags=1)
        assert base.max_fill == 4 * k and base.slots_reached == (1 << 4 * k) - 1
        assert base.end_of_warp_flushes == (1 if layout == "b" else 0)


@pytest.mark.parametrize("k", [7, 8])
def test_ticketed_document_reaches_every_slot(k):
    nchunks = up.ticketed_chunks(128)
    n, last, lanes_of = up.ticketed_layout(k, nchunks)
    img = up.build_image(n, 0, lanes_of, last)
    f, cnt = up.lanes_of_doc(img, 0)
    assert (cnt == k).all()
    fixed_end = 4 * GRID_WARPS
    plants = up.ticketed_plants(k, nchunks, fixed_end)
    probes = [_probe_pos(c, lane, 0) for _, c, lane, _ in plants]
    for _, c, lane, make in plants:
        assert np.array_equal(up.lanes_of_doc(up.apply(img, make(False)), 0)[0][c - 1 : c + 2], f[c - 1 : c + 2])
    assert {s for s, *_ in plants} == set(range(4 * k))
    assert {c for _, c, _, _ in plants} >= {fixed_end - 1, fixed_end, nchunks - 1}
    for warps, seed in ((GRID_WARPS, 11), (GRID_WARPS, 12), (GRID_WARPS // 3, 13)):
        r = emu.stage1_stream_sched(img, flags=1, warps=warps, seed=seed, probes=probes)
        assert (r.err, r.utf8, r.max_fill) == (0, 0, 4 * k)
        assert [(p.kind, p.slot) for p in r.probes] == [(emu.PARKED, s) for s, *_ in plants]
        last_run = [p.flush for (_, c, _, _), p in zip(plants, r.probes) if c >= nchunks - nchunks % 4]
        assert last_run and set(last_run) == {emu.END_OF_WARP}
        assert r.end_of_warp_flushes == 1 and r.mid_run_flushes == nchunks // 4
    # a violation in a drawn run is caught whichever warp draws it
    slot, c, lane, make = plants[5]
    bad = up.apply(img, make(False))
    for warps, seed in ((GRID_WARPS, 21), (100, 22)):
        r = emu.stage1_stream_sched(bad, flags=1, warps=warps, seed=seed)
        assert (r.err, r.utf8) == (oracle.UTF8_ERROR, 1)


def test_mixed_density_document_reaches_every_path():
    """The mixed-density generator (k from 0..12 per chunk), at 16 MiB: rings carried partly filled from one run into the
    next, both flushes, inline chunks, and one planted violation in each of the skip, inline and park paths."""
    img, counts = up.mixed_density_image(16, 0)
    f, cnt = up.lanes_of_doc(img, 0)
    assert np.array_equal(cnt, counts)
    want = _want(img, 1)
    for warps, seed in ((GRID_WARPS, 1), (300, 2), (97, 3)):
        r = emu.stage1_stream_sched(img, flags=1, warps=warps, seed=seed)
        assert (r.err, r.n, r.utf8) == (want.error, want.n, 0)
        assert np.array_equal(r.out, want.indexes)
        assert r.mid_run_flushes > 0 and r.end_of_warp_flushes > 0 and r.inline_chunks > 0
        assert 24 < r.max_fill <= 32
    for path, (c, lane, patches) in up.three_path_plants(img, counts).items():
        bad = up.apply(img, patches)
        r = emu.stage1_stream_sched(bad, flags=1, probes=[_probe_pos(c, lane, 0)])
        assert r.probes[0].kind == {"skip": emu.PARKED, "inline": emu.INLINE, "park": emu.PARKED}[path], path
        assert cnt[c] == {"skip": 0, "inline": cnt[c], "park": cnt[c]}[path] and (path != "inline" or cnt[c] > 8)
        assert (r.err, r.utf8) == (oracle.UTF8_ERROR, 1), path
