"""Device time of stage 2 over a document stream against the single-document walk, with CUDA events:

  (a) primitives + stream walk (sjb200_stage2_stream_device_async) on synth.ndjson of --mib MiB
  (b) primitives + single-document walk (sjb200_stage2_tape_device_async) on synth.status_array of --mib MiB
  (c) (b) with another build of the library (--other-lib, e.g. one built from the parent commit), in the same process
  (d) (a) with that other build

Stage 1 runs once per input, untimed; the inputs and outputs stay on the device.  The runs of (a) to (d) alternate
within every repetition, after --warmup untimed rounds of each.  Prints the card, its power limit and one line per
measurement: median and spread in ms, and tokens per second."""
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


def bind(path):
    L = C.CDLL(path)
    for name, (res, args) in _native.SIGNATURES.items():
        if hasattr(L, name):
            getattr(L, name).restype = res
            getattr(L, name).argtypes = args
    ctx = C.c_void_p()
    assert L.sjb200_ctx_create(0, (1 << 32) - 1, 0, 0, C.byref(ctx)) == 0
    L.sjb200_ctx_set_stream(ctx, C.c_void_p(torch.cuda.current_stream().cuda_stream))
    return L, ctx


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--mib", type=int, default=1024)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--other-lib", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this script measures the GPU")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True).stdout.strip()
    print(f"card: {q or torch.cuda.get_device_name(0)}")

    s1 = device.Stage1Context(0)
    inputs = {}
    for name, gen in (("ndjson", synth.ndjson), ("status_array", synth.status_array)):
        doc = gen(args.mib << 20)
        d_in = torch.from_numpy(np.asarray(doc)).cuda()
        d_idx = torch.empty(d_in.numel() + 8, dtype=torch.int32, device="cuda")
        r = s1.index(d_in, d_idx)
        assert r.error == 0
        n = r.n
        out = dict(kind=torch.empty(n, dtype=torch.uint8, device="cuda"), err=torch.empty(n, dtype=torch.uint8, device="cuda"),
                   val=torch.empty(n, dtype=torch.int64, device="cuda"), off=torch.empty(n, dtype=torch.int64, device="cuda"),
                   sb=torch.empty(d_in.numel() + 2 * n + 64, dtype=torch.uint8, device="cuda"), psum=torch.empty(4, dtype=torch.int64, device="cuda"),
                   tape=torch.empty(4 * n, dtype=torch.int64, device="cuda"), first=torch.empty(n + 1, dtype=torch.int32, device="cuda"),
                   dtape=torch.empty(n + 1, dtype=torch.int64, device="cuda"), dstat=torch.empty(n, dtype=torch.int64, device="cuda"),
                   sum=torch.empty(4, dtype=torch.int64, device="cuda"))
        inputs[name] = (d_in, d_idx, n, out)
        print(f"{name}: {d_in.numel()} bytes, {n} structurals")

    def prims(L, ctx, d_in, d_idx, n, o):
        return L.sjb200_stage2_primitives_device_async(ctx, d_in.data_ptr(), d_in.numel(), d_idx.data_ptr(), n, o["kind"].data_ptr(), o["err"].data_ptr(),
                                                       o["val"].data_ptr(), o["off"].data_ptr(), o["sb"].data_ptr(), o["sb"].numel(), o["psum"].data_ptr())

    def stream(L, ctx):
        d_in, d_idx, n, o = inputs["ndjson"]
        rc = prims(L, ctx, d_in, d_idx, n, o)
        rc |= L.sjb200_stage2_stream_device_async(ctx, d_in.data_ptr(), d_in.numel(), d_idx.data_ptr(), n, o["kind"].data_ptr(), o["err"].data_ptr(),
                                                  o["val"].data_ptr(), o["off"].data_ptr(), o["tape"].data_ptr(), o["tape"].numel(), o["first"].data_ptr(),
                                                  o["dtape"].data_ptr(), o["dstat"].data_ptr(), o["sum"].data_ptr())
        return rc

    def single(L, ctx):
        d_in, d_idx, n, o = inputs["status_array"]
        rc = prims(L, ctx, d_in, d_idx, n, o)
        rc |= L.sjb200_stage2_tape_device_async(ctx, d_in.data_ptr(), d_in.numel(), d_idx.data_ptr(), n, o["kind"].data_ptr(), o["err"].data_ptr(),
                                                o["val"].data_ptr(), o["off"].data_ptr(), o["tape"].data_ptr(), o["tape"].numel(), o["sum"].data_ptr())
        return rc

    this = bind(_native.LIB_PATH)
    runs = [("a stream walk, ndjson", stream, this, "ndjson"), ("b single walk, status_array", single, this, "status_array")]
    if args.other_lib:
        other = bind(args.other_lib)
        runs.append(("c single walk, status_array, other build", single, other, "status_array"))
        runs.append(("d stream walk, ndjson, other build", stream, other, "ndjson"))
    times = {r[0]: [] for r in runs}
    for rep in range(args.warmup + args.reps):
        for label, fn, (L, ctx), _ in runs:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            rc = fn(L, ctx)
            e1.record()
            torch.cuda.synchronize()
            assert rc == 0, (label, rc)
            if rep >= args.warmup:
                times[label].append(e0.elapsed_time(e1))
    for label, _, _, name in runs:
        t = sorted(times[label])
        med = statistics.median(t)
        n = inputs[name][2]
        print(f"{label}: median {med:.2f} ms (min {t[0]:.2f}, max {t[-1]:.2f}, {len(t)} runs), {n / med / 1e6:.3f} G tokens/s")
    o = inputs["ndjson"][3]["sum"].cpu().tolist()
    print(f"ndjson stream: {o[0]} documents, {o[1]} failing, {o[2]} tape words")


if __name__ == "__main__":
    main()
