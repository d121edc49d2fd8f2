"""Device time of string columns from pointer cells (sjb200_string_columns_device_async), with CUDA events:

  synth arms, on synth.ndjson of --mib MiB (stage 1, the primitives and the stream walk run once, untimed):
    (a) lookups of /text, /user/screen_name, /user/description, /lang (sjb200_at_pointers_device_async)
    (b) (a) + their string columns
    (c) the string columns alone (lengths, scan, copy)
  balance arms, two seeded streams {"s": "..."} with the same number of documents and the same total string bytes; the
  walk and the lookup of /s run once, untimed, and the string columns alone are timed:
    (d) uniform lengths
    (e) heavy-tailed lengths: almost all 1-16 bytes, about 1 in 10^4 of 1 MiB

The arms of each group alternate within every repetition, after --warmup untimed rounds of each.  Prints the card, its
power limit, one line per arm (median and spread in ms), the bytes gathered, and the gather's modelled traffic over its time:
cells read (9 bytes each), the length words of the string records, the offsets written by the lengths pass, read and
written by the scan and read by the copy's searches (8 bytes per cell each), the source bytes read and the data written."""
import argparse
import os
import statistics
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from mojo_simdjson_b200 import _native, device, synth  # noqa: E402

POINTERS = ["/text", "/user/screen_name", "/user/description", "/lang"]


class Columns:
    """The walk and the lookups of one stream, run once; then timed calls of the lookups and of the string columns."""

    def __init__(self, ctx, doc: np.ndarray, pointers):
        self.ctx, self.L, self.c = ctx, _native.lib(), ctx._ctx
        d_in = torch.from_numpy(doc).cuda()
        d_idx = torch.empty(d_in.numel() + 8, dtype=torch.int32, device="cuda")
        r = ctx.index(d_in, d_idx)
        assert r.error == 0
        self.n_struct = r.n
        prims = ctx.stage2_primitives(d_in, d_idx, r.n)
        s = ctx.stage2_stream(d_in, d_idx, r.n, prims)
        self.sb, self.tape, self.doc_tape, self.status = prims["string_buf"], s["tape"], s["doc_tape"], s["doc_status"]
        self.n_docs, self.n_bytes = self.status.numel(), d_in.numel()
        del d_in, d_idx
        self.prog = device.pointer_program(pointers)
        self.k = len(pointers)
        self.cols = ctx.at_pointers(pointers, self.tape, self.sb, self.doc_tape, self.status)
        self.strs = ctx.string_columns(self.cols, self.sb)
        self.summary = torch.empty(2, dtype=torch.int64, device="cuda")
        self.string_cells = int(self.strs.mask.sum().item())
        self.total = self.strs.data.numel()

    def lookups(self) -> int:
        raw, offs = self.prog
        return self.L.sjb200_at_pointers_device_async(self.c, self.tape.data_ptr(), self.tape.numel(), self.sb.data_ptr(), self.sb.numel(),
                                                      self.doc_tape.data_ptr(), self.status.data_ptr(), self.n_docs, raw, offs, self.k,
                                                      self.cols.type.data_ptr(), self.cols.code.data_ptr(), self.cols.value.data_ptr())

    def gather(self) -> int:
        return self.L.sjb200_string_columns_device_async(self.c, self.cols.type.data_ptr(), self.cols.value.data_ptr(), self.k, self.n_docs,
                                                         self.sb.data_ptr(), self.sb.numel(), self.strs.offsets.data_ptr(), self.strs.data.data_ptr(),
                                                         self.total, self.summary.data_ptr())

    def traffic(self) -> int:
        n = self.k * self.n_docs
        return 9 * n + 4 * self.string_cells + 8 * (n + 1) * 5 + 2 * self.total


def timed(runs, reps: int, warmup: int) -> dict:
    times = {label: [] for label, _ in runs}
    for rep in range(warmup + reps):
        for label, fn in runs:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            rc = fn()
            e1.record()
            torch.cuda.synchronize()
            assert rc == 0, (label, rc)
            if rep >= warmup:
                times[label].append(e0.elapsed_time(e1))
    med = {}
    for label, _ in runs:
        t = sorted(times[label])
        med[label] = statistics.median(t)
        print(f"{label}: median {med[label]:.3f} ms (min {t[0]:.3f}, max {t[-1]:.3f}, {len(t)} runs)")
    return med


def balance_stream(lengths: np.ndarray) -> np.ndarray:
    """NDJSON of {"s": "<lengths[d] printable ASCII bytes>"} documents."""
    pool = (np.arange(int(lengths.max()) + 1, dtype=np.int64) * 7 % 90 + 33).astype(np.uint8)
    pool[pool == ord('"')] = ord("a")
    pool[pool == ord("\\")] = ord("b")
    text = pool.tobytes()
    return np.frombuffer(b"".join(b'{"s":"' + text[:n] + b'"}\n' for n in lengths.tolist()), dtype=np.uint8)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--mib", type=int, default=1024)
    ap.add_argument("--docs", type=int, default=1 << 20, help="documents of each balance stream")
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--warmup", type=int, default=2)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this script measures the GPU")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True).stdout.strip()
    print(f"card: {q or torch.cuda.get_device_name(0)}")
    ctx = device.Stage1Context(0)

    s = Columns(ctx, synth.ndjson(args.mib << 20), POINTERS)
    print(f"ndjson: {s.n_bytes} bytes, {s.n_struct} structurals, {s.n_docs} documents; {s.k} pointers, {s.string_cells} string cells, "
          f"{s.total} bytes gathered ({[int(x) for x in s.strs.mask.sum(dim=1).tolist()]} strings per pointer)")
    med = timed([("(a) lookups of 4 string pointers", s.lookups), ("(b) (a) + string columns", lambda: s.lookups() | s.gather()),
                 ("(c) string columns alone", s.gather)], args.reps, args.warmup)
    c = med["(c) string columns alone"]
    print(f"(b) - (a): {med['(b) (a) + string columns'] - med['(a) lookups of 4 string pointers']:.3f} ms; gather: {s.total / c / 1e6:.1f} GB/s of "
          f"data, {s.traffic() / c / 1e6:.1f} GB/s of modelled traffic ({s.traffic()} bytes)")
    del s
    torch.cuda.empty_cache()

    rng = np.random.default_rng(0x5EED)
    d = args.docs
    heavy = rng.integers(1, 17, d)
    heavy[rng.random(d) < 1e-4] = 1 << 20
    total = int(heavy.sum())
    uniform = np.full(d, total // d, dtype=np.int64)
    uniform[: total % d] += 1
    arms = {}
    for label, lengths in (("(d) uniform", uniform), ("(e) heavy-tailed", heavy)):
        arms[label] = Columns(ctx, balance_stream(lengths), ["/s"])
        b = arms[label]
        assert b.total == total and b.string_cells == d
        print(f"{label}: {d} documents, {total} string bytes, longest {int(lengths.max())}, {int((lengths >= 1 << 20).sum())} of 1 MiB")
    med = timed([(label + " string columns", b.gather) for label, b in arms.items()], args.reps, args.warmup)
    for label, b in arms.items():
        t = med[label + " string columns"]
        print(f"{label}: {b.total / t / 1e6:.1f} GB/s of data, {b.traffic() / t / 1e6:.1f} GB/s of modelled traffic")
    print(f"(e) / (d): {med['(e) heavy-tailed string columns'] / med['(d) uniform string columns']:.3f}")
    ctx.close()


if __name__ == "__main__":
    main()
