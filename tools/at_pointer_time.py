"""Device time of JSON Pointer lookups on the stream tapes, with CUDA events:

  (a) primitives + stream walk (sjb200_stage2_stream_device_async) on synth.ndjson of --mib MiB
  (b) (a) + lookups of 4 pointers (sjb200_at_pointers_device_async)
  (c) (a) + lookups of 16 pointers

Stage 1 runs once, untimed; inputs and outputs stay on the device.  The three arms alternate within every repetition,
after --warmup untimed rounds of each.  Prints the card, its power limit, one line per arm (median and spread in ms) and
the lookup time (b) - (a) and (c) - (a)."""
import argparse
import ctypes as C
import os
import statistics
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from mojo_simdjson_b200 import _native, device, synth  # noqa: E402

# top-level scalars, the nested user object, an array element inside entities, one missing field
POINTERS_4 = ["/id", "/user/followers_count", "/entities/hashtags/0/text", "/missing"]
POINTERS_16 = POINTERS_4 + ["/text", "/retweet_count", "/truncated", "/geo", "/user/id", "/user/screen_name", "/user/ratio", "/user/verified",
                            "/entities/hashtags/1/indices/0", "/entities/urls/0/url", "/metadata/iso_language_code", "/user/nope"]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--mib", type=int, default=1024)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--warmup", type=int, default=2)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this script measures the GPU")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True).stdout.strip()
    print(f"card: {q or torch.cuda.get_device_name(0)}")

    ctx = device.Stage1Context(0)
    L, c = _native.lib(), ctx._ctx
    doc = synth.ndjson(args.mib << 20)
    d_in = torch.from_numpy(np.asarray(doc)).cuda()
    d_idx = torch.empty(d_in.numel() + 8, dtype=torch.int32, device="cuda")
    r = ctx.index(d_in, d_idx)
    assert r.error == 0
    n = r.n
    o = dict(kind=torch.empty(n, dtype=torch.uint8, device="cuda"), err=torch.empty(n, dtype=torch.uint8, device="cuda"),
             val=torch.empty(n, dtype=torch.int64, device="cuda"), off=torch.empty(n, dtype=torch.int64, device="cuda"),
             sb=torch.empty(d_in.numel() + 2 * n + 64, dtype=torch.uint8, device="cuda"), psum=torch.empty(4, dtype=torch.int64, device="cuda"),
             tape=torch.empty(4 * n, dtype=torch.int64, device="cuda"), first=torch.empty(n + 1, dtype=torch.int32, device="cuda"),
             dtape=torch.empty(n + 1, dtype=torch.int64, device="cuda"), dstat=torch.empty(n, dtype=torch.int64, device="cuda"),
             sum=torch.empty(4, dtype=torch.int64, device="cuda"))

    def walk():
        rc = L.sjb200_stage2_primitives_device_async(c, d_in.data_ptr(), d_in.numel(), d_idx.data_ptr(), n, o["kind"].data_ptr(), o["err"].data_ptr(),
                                                     o["val"].data_ptr(), o["off"].data_ptr(), o["sb"].data_ptr(), o["sb"].numel(), o["psum"].data_ptr())
        rc |= L.sjb200_stage2_stream_device_async(c, d_in.data_ptr(), d_in.numel(), d_idx.data_ptr(), n, o["kind"].data_ptr(), o["err"].data_ptr(),
                                                  o["val"].data_ptr(), o["off"].data_ptr(), o["tape"].data_ptr(), o["tape"].numel(), o["first"].data_ptr(),
                                                  o["dtape"].data_ptr(), o["dstat"].data_ptr(), o["sum"].data_ptr())
        return rc

    walk()
    torch.cuda.synchronize()
    nd = int(o["sum"][0].item())
    print(f"ndjson: {d_in.numel()} bytes, {n} structurals, {nd} documents, {int(o['sum'][1].item())} failing")
    cells = {}
    for ps in (POINTERS_4, POINTERS_16):
        cells[len(ps)] = (device.pointer_program(ps), torch.empty((len(ps), nd), dtype=torch.uint8, device="cuda"),
                          torch.empty((len(ps), nd), dtype=torch.uint8, device="cuda"), torch.empty((len(ps), nd), dtype=torch.int64, device="cuda"))

    def lookups(k):
        (raw, offs), ty, code, val = cells[k]
        return L.sjb200_at_pointers_device_async(c, o["tape"].data_ptr(), o["tape"].numel(), o["sb"].data_ptr(), o["sb"].numel(), o["dtape"].data_ptr(),
                                                 o["dstat"].data_ptr(), nd, raw, offs, k, ty.data_ptr(), code.data_ptr(), val.data_ptr())

    runs = [("a primitives + stream walk", lambda: walk()), ("b (a) + 4 pointers", lambda: walk() | lookups(4)),
            ("c (a) + 16 pointers", lambda: walk() | lookups(16)), ("lookups of 4 pointers alone", lambda: lookups(4)),
            ("lookups of 16 pointers alone", lambda: lookups(16))]
    times = {r[0]: [] for r in runs}
    for rep in range(args.warmup + args.reps):
        for label, fn in runs:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            rc = fn()
            e1.record()
            torch.cuda.synchronize()
            assert rc == 0, (label, rc)
            if rep >= args.warmup:
                times[label].append(e0.elapsed_time(e1))
    med = {}
    for label, _ in runs:
        t = sorted(times[label])
        med[label] = statistics.median(t)
        print(f"{label}: median {med[label]:.3f} ms (min {t[0]:.3f}, max {t[-1]:.3f}, {len(t)} runs)")
    a = med["a primitives + stream walk"]
    print(f"(b) - (a): {med['b (a) + 4 pointers'] - a:.3f} ms; (c) - (a): {med['c (a) + 16 pointers'] - a:.3f} ms")
    for k in (4, 16):
        code = cells[k][2].cpu().numpy()
        print(f"{k} pointers: found per pointer {[int(x) for x in (code == 0).sum(axis=1)]}")


if __name__ == "__main__":
    main()
