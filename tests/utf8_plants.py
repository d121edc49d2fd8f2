"""Documents for testing the stream pipeline's deferred UTF-8 validation (csrc/stage1_stream.cuh), and UTF-8 violations
planted into them.

The classify kernel of the stream pipeline decides per warp and 2 KiB chunk how a lane (64 bytes) is validated: not at all
when no byte >= 0x80 is in the chunk or in the 4 bytes before any of its lanes; inline when more than 8 lanes are flagged;
otherwise each flagged lane parks in the next slot of its warp's 32-slot ring, validated later by a flush.  The documents
here control exactly which lanes are flagged, so that a test knows the slot and the flush of every planted violation.

Coordinates are aligned ones, as the kernel sees them: an image of mis + len bytes whose first `mis` bytes are not part of
the document (the document starts `mis` bytes past a 16-byte boundary); lane G covers image[64 G, 64 G + 64) and chunk c
the lanes 32 c .. 32 c + 31.

The image is a JSON array of 13-character strings with a period of 16 bytes: `abcdefghij","klm`.  Image offsets 13..15 and
0..9 modulo 16 are string content, so lane and chunk boundaries (multiples of 64) fall inside strings.  A flagged lane holds
one "é" at lane offsets 24-25.  The last lane of the image closes the last string and the array and ends with a bare
scalar of 61 letters, so that a truncated sequence can end the document while every verdict but UTF-8 stays SUCCESS.
Every plant replaces string content (or letters of that scalar) with bytes >= 0x80: the structural indexes never change."""
from __future__ import annotations

import numpy as np

LANE, CHUNK, LANES = 64, 2048, 32
PERIOD = b'abcdefghij","klm'
E_ACUTE = b"\xc3\xa9"
MID = 24                  # lane offset of the "é" that flags a lane
INSIDE = 46               # lane offset of a violation inside the lane: string content up to 4 bytes (46 mod 16 = 14)
RUN = 4                   # chunks per run of a warp
DEFER_MAX = 8             # flagged lanes a chunk parks at most
RING = 32                 # slots of a warp's ring

# violations inside one lane, each with a valid sequence of the same length
INSIDE_KINDS = {
    "overlong": (b"\xc0\x80", b"\xc2\x80"),
    "lone continuation": (b"\x80", b"a"),
    "surrogate": (b"\xed\xa0\x80", b"\xed\x9f\xbf"),
    "above U+10FFFF": (b"\xf4\x90\x80\x80", b"\xf4\x8f\xbf\xbf"),
}


def build_image(nchunks: int, mis: int, lanes_of, last_lanes: int = LANES) -> np.ndarray:
    """The aligned image: `nchunks` chunks, the last one `last_lanes` lanes long; lanes_of(c) = the lanes of chunk c to flag.
    The document is image[mis:] (0 <= mis <= 14)."""
    assert 0 <= mis <= 14 and 1 <= last_lanes <= LANES
    size = (nchunks - 1) * CHUNK + last_lanes * LANE
    img = np.resize(np.frombuffer(PERIOD, dtype=np.uint8), size).copy()
    img[:15] = ord(" ")
    img[mis] = ord("[")
    img[15] = ord('"')
    img[size - 64] = ord('"')
    img[size - 63] = ord("]")
    img[size - 62] = ord(" ")
    img[size - 61 :] = ord("z")
    for c in range(nchunks):
        for lane in lanes_of(c):
            g = (c * LANES + lane) * LANE + MID
            assert g + 2 <= size
            img[g : g + 2] = np.frombuffer(E_ACUTE, dtype=np.uint8)
    return img


def build_image_from_counts(counts: np.ndarray, mis: int, rng: np.random.Generator) -> np.ndarray:
    """A full-chunk image whose chunk c has counts[c] flagged lanes, chosen at random."""
    nchunks = int(counts.size)
    img = build_image(nchunks, mis, lambda c: ())
    sel = np.argsort(rng.random((nchunks, LANES)), axis=1)
    mask = np.arange(LANES)[None, :] < counts[:, None]
    chunk_idx, rank = np.nonzero(mask)
    lanes = sel[chunk_idx, rank]
    pos = (chunk_idx * LANES + lanes) * LANE + MID
    img[pos] = E_ACUTE[0]
    img[pos + 1] = E_ACUTE[1]
    return img


def flagged_lanes(img: np.ndarray, mis: int) -> np.ndarray:
    """[nchunks, 32] bool: the lanes the classify kernel flags (stage1_kernel.cuh, any_hi: a byte >= 0x80 among the lane's 64
    bytes or the 4 bytes before them; bytes outside the document read as 0x20)."""
    size = int(img.size)
    nl = -(-size // LANE)
    nchunks = -(-nl // LANES)
    hi = np.zeros(nchunks * LANES * LANE, dtype=bool)
    hi[mis:size] = img[mis:] >= 0x80
    hi = hi.reshape(nchunks * LANES, LANE)
    f = hi.any(axis=1)
    f[1:] |= hi[:-1, LANE - 4 :].any(axis=1)
    return f.reshape(nchunks, LANES)


def lanes_of_doc(img: np.ndarray, mis: int):
    """(flagged lanes per chunk as a [nchunks, 32] array, their count per chunk)"""
    f = flagged_lanes(img, mis)
    return f, f.sum(axis=1)


def slot_uniform(k: int, c: int, rank: int) -> int:
    """The slot of the lane of rank `rank` in chunk c when every chunk has exactly k in {7, 8} flagged lanes: a run starts with
    an empty ring (the previous run's 4th chunk left more than 24 slots in use) and its chunks fill k slots each."""
    assert k in (7, 8) and 0 <= rank < k
    return k * (c % RUN) + rank


# ---- plants: lists of (aligned position, bytes) ----
def plant_inside(c: int, lane: int, kind: str = "overlong", valid: bool = False):
    bad, good = INSIDE_KINDS[kind]
    return [((c * LANES + lane) * LANE + INSIDE, good if valid else bad)]


def plant_owed(c: int, lane: int, valid: bool = False):
    """The lane before ends in a lead byte; the continuation is missing at offset 0 of this lane (valid: present).  The
    violation belongs to this lane: only the carry from the 4 bytes before it shows it.  Lane 0 takes those bytes from the
    previous chunk's last lane."""
    g = (c * LANES + lane) * LANE
    assert g > 0
    return [(g - 1, E_ACUTE if valid else b"\xc3")]


def plant_owed_3(c: int, lane: int, valid: bool = False):
    """A 3-byte sequence whose lead sits 2 bytes before the lane: the lane owes 1 continuation and has none."""
    g = (c * LANES + lane) * LANE
    return [(g - 2, b"\xe2\x82\xac" if valid else b"\xe2\x82")]


def plant_end(img_size: int, valid: bool = False, kind: str = "3-byte"):
    """The document ends in the middle of a sequence at the last byte of its last lane: only the end-of-document bit shows it."""
    assert img_size % LANE == 0
    if kind == "3-byte":
        return [(img_size - 2, E_ACUTE if valid else b"\xe2\x82")]
    return [(img_size - 1, b"z" if valid else b"\xc3")]


def apply(img: np.ndarray, patches) -> np.ndarray:
    out = img.copy()
    for pos, b in patches:
        out[pos : pos + len(b)] = np.frombuffer(b, dtype=np.uint8)
    return out


def utf8_valid(data) -> bool:
    try:
        bytes(data).decode("utf-8")
        return True
    except UnicodeDecodeError:
        return False


def utf8_valid_around(doc: np.ndarray, lo: int, hi: int) -> bool:
    """Python's strict decoder on doc[lo:hi] widened to ASCII bytes on both sides.  For a document that was valid before
    bytes in [lo, hi) were replaced, this is the verdict of the whole document."""
    a = max(lo - 4, 0)
    while a > 0 and doc[a] >= 0x80:
        a -= 1
    b = min(hi + 4, doc.size)
    while b < doc.size and doc[b] >= 0x80:
        b += 1
    return utf8_valid(doc[a:b].tobytes())


# ---- the documents of tests/test_gpu_utf8_deferral.py ----
FIXED_CHUNKS = 300        # a few hundred chunks: every warp of the grid takes only its first run


def fixed_layout_a(k: int):
    """Every chunk: lanes 0 .. k-1 (a lane of rank r >= 1 follows a flagged lane), the last chunk of 300 (full): lanes
    32-k .. 31, so that its last lane ends the document."""
    n = FIXED_CHUNKS
    return n, LANES, lambda c: range(32 - k, 32) if c == n - 1 else range(k)


def fixed_layout_b(k: int):
    """Every chunk: lane 0 and lanes 33-k .. 31 (lane 0 follows the previous chunk's flagged lane 31); a 301st chunk of 20
    lanes, lanes 21-k .. 19: a run of one chunk at the end, flushed when its warp runs out of chunks.  (A byte >= 0x80 among
    the last 4 of the document also flags lane 20, past its end: the kernel reads the 4 bytes before every lane.  With
    plant_end the last chunk has k flagged lanes too.)"""
    n = FIXED_CHUNKS + 1
    return n, 20, lambda c: range(21 - k, 20) if c == n - 1 else [0, *range(33 - k, 32)]


def ticketed_chunks(mib: int = 128) -> int:
    return (mib << 20) // CHUNK + 3      # not a multiple of 4: the last run has 3 chunks


def ticketed_layout(k: int, nchunks: int):
    """Uniform k, layout b; the last chunk full with lanes 32-k .. 31."""
    return nchunks, LANES, lambda c: range(32 - k, 32) if c == nchunks - 1 else [0, *range(33 - k, 32)]


def fixed_plants(k: int, layout: str, nchunks: int):
    """For every slot reachable with k flagged lanes per chunk, the plants of each kind the layout allows:
    [(slot, kind, chunk, lane, patches(valid))].  Layout a: inside and owed at a lane boundary (rank >= 1).  Layout b:
    owed at the chunk boundary (rank 0, the previous chunk belongs to another warp's run), inside (every rank)."""
    out = []
    nruns = nchunks // RUN
    for slot in range(k * RUN):
        q, rank = divmod(slot, k)
        run = 1 + (slot * 7) % (nruns - 2)
        c = run * RUN + q
        if layout == "a":
            lane = rank
            out.append((slot, "inside", c, lane, lambda v, c=c, lane=lane, s=slot: plant_inside(c, lane, list(INSIDE_KINDS)[s % 4], v)))
            if rank >= 1:
                out.append((slot, "owed", c, lane, lambda v, c=c, lane=lane: plant_owed(c, lane, v)))
        else:
            lane = 0 if rank == 0 else 32 - k + rank
            if rank == 0:
                out.append((slot, "owed at a chunk boundary", c, lane, lambda v, c=c: plant_owed(c, 0, v)))
            out.append((slot, "inside", c, lane, lambda v, c=c, lane=lane, s=slot: plant_inside(c, lane, list(INSIDE_KINDS)[(s + 1) % 4], v)))
    return out


def ticketed_plants(k: int, nchunks: int, fixed_end: int):
    """Plants for the ticketed-run document: every slot at least once spread over the document, and around the end of the
    fixed-run range (chunk `fixed_end` = 4 x warps in the grid) and in the last chunks.  [(slot, chunk, lane, patches(valid))]"""
    def lane_of_rank(c, rank):
        if c == nchunks - 1:
            return 32 - k + rank
        return 0 if rank == 0 else 32 - k + rank

    picks = []
    for slot in range(k * RUN):
        q, rank = divmod(slot, k)
        run = (fixed_end // RUN) + 1 + (slot * 97) % ((nchunks - fixed_end) // RUN - 3)
        picks.append((run * RUN + q, rank))
    for c in (fixed_end - 2, fixed_end - 1, fixed_end, fixed_end + 1, 5, nchunks - 5, nchunks - 2):
        picks.append((c, k - 1))
        picks.append((c, 0))
    out = []
    for c, rank in picks:
        lane = lane_of_rank(c, rank)
        slot = slot_uniform(k, c, rank)
        if rank == 0 and c % RUN == 0 and c > 0 and c != nchunks - 1:
            out.append((slot, c, lane, lambda v, c=c: plant_owed(c, 0, v)))
        else:
            out.append((slot, c, lane, lambda v, c=c, lane=lane: plant_inside(c, lane, "overlong", v)))
    # the last chunk (its run has 3 chunks: flushed when the warp runs out of chunks)
    out.append((slot_uniform(k, nchunks - 1, k - 1), nchunks - 1, 31, lambda v: plant_end((nchunks) * CHUNK, v)))
    return out


MIXED_SEED = 20261022


def mixed_density_image(mib: int, mis: int, seed: int = MIXED_SEED):
    """Full chunks whose flagged-lane counts are drawn from 0..12: some chunks skip, some validate inline, and the parked
    ones leave rings partly filled at the end of a run.  Returns (image, counts)."""
    rng = np.random.default_rng(seed)
    counts = rng.integers(0, 13, (mib << 20) // CHUNK)
    return build_image_from_counts(counts, mis, rng), counts


def three_path_plants(img: np.ndarray, counts: np.ndarray):
    """One violation for each path: in a chunk with no flagged lane (the plant makes it park one), in an inline chunk (owed
    by the previous lane: only the carry the straddle gate lets through shows it) and in a parking chunk.
    {path: (chunk, lane, patches)}"""
    mid = counts.size // 2
    skip = mid + int(np.flatnonzero(counts[mid:] == 0)[0])
    inline = mid + int(np.flatnonzero(counts[mid:] >= 10)[0])
    park = mid + int(np.flatnonzero((counts[mid:] >= 1) & (counts[mid:] <= 8))[0])
    f = flagged_lanes(img, 0)
    park_lane = int(np.flatnonzero(f[park])[0])
    return {"skip": (skip, 5, plant_inside(skip, 5)),
            "inline": (inline, 17, plant_owed(inline, 17)),
            "park": (park, park_lane, plant_inside(park, park_lane, "surrogate"))}


def mixed_plants(nchunks: int, count: int, seed: int = MIXED_SEED + 1):
    """`count` single violations at seeded places, each with its valid twin: [(chunk, lane, bad patches, valid patches)]"""
    rng = np.random.default_rng(seed)
    out = []
    kinds = list(INSIDE_KINDS)
    for i in range(count):
        c = int(rng.integers(1, nchunks - 1))
        lane = int(rng.integers(0, LANES))
        how = i % 6
        if how < 4:
            out.append((c, lane, plant_inside(c, lane, kinds[how]), plant_inside(c, lane, kinds[how], True)))
        elif how == 4:
            out.append((c, lane, plant_owed(c, lane), plant_owed(c, lane, True)))
        else:
            out.append((c, lane, plant_owed_3(c, lane), plant_owed_3(c, lane, True)))
    return out


def long_backslash_run(chunk: int = 200, length: int = 80_000):
    """A backslash run of even length inside a string, ending 4 bytes past the start of `chunk`: the 32 bytes before that
    chunk are all backslashes and the run goes back further than the stream classify kernel walks (64 KiB), so the stream
    pipeline raises its speculation flag and the persistent kernel redoes the document."""
    return [(chunk * CHUNK - length + 4, b"\\" * length)]
