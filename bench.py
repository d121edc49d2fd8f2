#!/usr/bin/env python
"""bench.py -- stage-1 input GB/s on B200 (BASELINE.json metric), one JSON line on rank 0.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

Workload (synthetic, deterministic; mojo_simdjson_b200/synth/gen.c):
  N = 1 : BASELINE.json configs[2] -- ONE 1 GiB JSON document (array of minified twitter-like statuses).
          --config small : configs[1], the 631,515-byte twitter-like document (latency: us per launch with the L2 flushed
                           between launches, back to back, per synchronous call, host to host)
          --config cjk | dense | runs : configs[4] at 1 GiB -- an all-CJK string document (UTF-8 validation on every
                           lane), an escape-dense one (a backslash-quote pair repeated), and the bench document with a 33-byte backslash run
                           ending on a 2 KiB boundary every MiB (the input that used to cost the pipeline a second pass)
  N > 1 : configs[3] -- an 8 GiB NDJSON batch sharded by line ranges over the N GPUs (8/N GiB per GPU: 4 / 2 / 1 one-GiB
          segments per GPU at N = 2 / 4 / 8; a 256 MiB whole-line template, seed 0x5EED0003+rank, replicated on the
          device), through the in-library batch driver (sjb200_batch_*): after every pass the GPUs exchange ONE NCCL
          all-gather of the per-segment {error, n} rows -- the only inter-GPU traffic of this path.  Total work is fixed
          as N grows ("scaling": "strong").  Before timing every rank checks every one of its segments against the
          oracle (n, verdict, 128-bit digest of the index stream).
A step = one stage-1 pass over the rank's input.  `value` times it with the input resident in HBM (CUDA events on
the launching stream, max over ranks); `e2e` times the same pass through the host-buffer C-ABI call
(sjb200_stage1: H2D copy of the document from pinned memory + kernel + D2H copy of the n+3 indexes).
The input (>= 1 GiB per GPU) is larger than L2 (126 MB), so no L2 flush is needed between iterations; --config small
flushes it explicitly.

--impl reference times the CPU restatement of the reference's stage 1 (oracle/, kind "port": the reference is Mojo
and cannot be built in this image) on the host cores, on a bounded sample of the same workload (its size is printed in
`config`), and reports the AVX-512 / pclmulqdq "cpu_simd" stage 1 of the same specification beside it.

--dump-outputs DIR writes, after the timed steps, what the timed path computed in its last step: stage1_result.npy (the
verdict rows) and a fixed, seeded sample of the index stream with its positions (structural_indexes.npy,
structural_index_positions.npy), all float64, 32 MiB at most.  The inputs are generated from fixed seeds, so two builds run
with the same arguments can be compared file for file.  (--impl reference sizes its sample from a timing probe: its dumps
compare where `config.reference_sample_bytes_per_step` agrees.)
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import socket
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "stage1_input_throughput"
UNIT = "GB/s"
GIB = 1 << 30
HBM_FALLBACK_GBS = 6650.0  # /opt/skills/guides/B200_PROFILING.md fallback


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return HBM_FALLBACK_GBS, "fallback"


def ncu_traffic(kind: str):
    """Committed ncu capture of the kernel organisation `kind` ("stream" | "persistent"), if any: dram bytes per document
    pass (dram__bytes_read.sum + dram__bytes_write.sum over its launches) and the per-kernel shares."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            return json.load(f).get(kind) or {}
    except Exception:
        return {}


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons of one GPU during the timed region (NVML, ~4 ms period)."""

    def __init__(self, device_index: int):
        super().__init__(daemon=True)
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop_evt = threading.Event()
        self.ok = False
        try:
            import pynvml
            import torch

            pynvml.nvmlInit()
            uuid = str(torch.cuda.get_device_properties(device_index).uuid)
            if not uuid.startswith("GPU-"):
                uuid = "GPU-" + uuid
            try:
                self.h = pynvml.nvmlDeviceGetHandleByUUID(uuid.encode())
            except Exception:
                self.h = pynvml.nvmlDeviceGetHandleByIndex(device_index)
            self.nv = pynvml
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.ok = True
        except Exception:
            self.ok = False

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {
            0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
            0x80: "hw_power_brake_slowdown", 0x2: "applications_clocks_setting",
        }
        while not self._stop_evt.is_set():
            try:
                self.samples.append(int(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                r = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.004)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=2)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "samples": 0}
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2], "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(s)}


def free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="doc1g", choices=["doc1g", "small", "cjk", "dense", "runs"],
                    help="N = 1 only: which BASELINE.json configuration to time (default: the 1 GiB document)")
    ap.add_argument("--bytes-per-gpu", type=int, default=GIB, help="N = 1: document size")
    ap.add_argument("--total-bytes", type=int, default=8 * GIB, help="N > 1: size of the whole NDJSON batch")
    ap.add_argument("--seg-bytes", type=int, default=GIB, help="N > 1: segment size")
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--warps", type=int, default=0, help="force tile shape (2/4/8/16/24), 0 = auto")
    ap.add_argument("--kernel", default="auto", choices=["auto", "persistent", "split", "stream"],
                    help="force the kernel organisation (sjb200_ctx_set_kernel); auto = the library's choice")
    ap.add_argument("--no-utf8", action="store_true", help="skip UTF-8 validation (the reference validates nothing)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-sample-bytes", type=int, default=GIB)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the timed path computed in its last step to DIR/<name>.npy "
                         "(float64; the index stream as a fixed, seeded sample): compares two builds output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


# ------------------------------------------------------------------------------------------------
# workloads
# ------------------------------------------------------------------------------------------------
NDJSON_TEMPLATE = 256 << 20


def make_document(config: str, size: int, out):
    """The N = 1 documents, generated into `out` (a uint8 numpy view of pinned memory)."""
    import numpy as np

    from mojo_simdjson_b200 import synth

    if config in ("doc1g", "runs"):
        synth.status_array(size, synth.SEED_DOC, out=out)
        if config == "runs":
            synth.plant_backslash_runs(out[:size])
    elif config == "small":
        synth.twitter_like(size, synth.SEED_TWITTER, out=out)
    elif config == "cjk":      # ["<CJK / emoji text>"]: every lane holds multi-byte characters
        unit = np.frombuffer("日本語のテキスト€😀".encode("utf-8"), dtype=np.uint8)
        body = size - 4
        whole = body // unit.size * unit.size
        out[0], out[1] = ord("["), ord('"')
        out[2 : 2 + whole] = np.resize(unit, whole)
        out[2 + whole : size - 2] = ord("a")
        out[size - 2], out[size - 1] = ord('"'), ord("]")
    elif config == "dense":    # ["\"\"\"...\""]: every other byte an escaped quote
        out[0:size:2] = 0x5C
        out[1:size:2] = 0x22
        out[0], out[1], out[size - 2], out[size - 1] = ord("["), ord('"'), ord('"'), ord("]")
    return out[:size]


def workload_config(n_gpus: int, config: str, size: int, total: int = 0, seg_bytes: int = 0):
    l2 = "input larger than the 126 MB L2, no flush between iterations"
    if n_gpus > 1:
        per = total // n_gpus
        return {"workload": f"{total / GIB:g} GiB synthetic NDJSON batch (one status object per line; 256 MiB whole-line template, seed "
                            f"0x5EED0003+rank, replicated) sharded by line ranges over {n_gpus} B200: {per / GIB:g} GiB = "
                            f"{max(1, per // seg_bytes)} segment(s) of {seg_bytes / GIB:g} GiB per GPU; one NCCL all-gather of the "
                            "per-segment {error, n} rows per pass (in-library batch driver)",
                "bytes_per_gpu": per, "total_bytes": total, "segment_bytes": seg_bytes, "l2": l2}
    names = {
        "doc1g": f"single synthetic {size / GIB:g} GiB JSON document (array of minified twitter-like statuses, seed 0x5EED0002) on 1 B200",
        "small": f"single synthetic twitter-like document, pretty printed, {size} bytes (seed 0x5EED0001) on 1 B200: latency",
        "cjk": f"adversarial: {size / GIB:g} GiB document that is one string of CJK / emoji text (every lane validates UTF-8) on 1 B200",
        "dense": f"adversarial: {size / GIB:g} GiB escape-dense document (backslash-quote pairs inside one string) on 1 B200",
        "runs": f"adversarial: the {size / GIB:g} GiB bench document with a 33-byte backslash run ending on a 2 KiB boundary every MiB on 1 B200",
    }
    if config == "small":
        l2 = "L2 flushed (a 256 MB buffer rewritten) before every timed launch"
    return {"workload": names[config], "bytes_per_gpu": size, "l2": l2}


# ------------------------------------------------------------------------------------------------
# --dump-outputs: the last timed step's results, so that two builds can be compared output for output
# ------------------------------------------------------------------------------------------------
DUMP_ENTRIES = 2 << 20     # index entries sampled in all: values + positions in float64 = 32 MiB, under the 64 MiB limit
DUMP_SEED = 0x5EED0D06


def sample_positions(m: int, k: int):
    """Which entries of an m-entry index stream are dumped: all of them when m <= k; otherwise the first and the last k/4
    (the document's start, its end and the 3-entry trailer) and one seeded position in each of k/2 equal strata in
    between.  Depends on m alone, so two builds that agree on the count dump the same positions."""
    import numpy as np

    if m <= k:
        return np.arange(m, dtype=np.int64)
    edge = k // 4
    c, span = k - 2 * edge, m - 2 * edge
    lo = edge + np.arange(c, dtype=np.int64) * span // c
    hi = edge + (np.arange(c, dtype=np.int64) + 1) * span // c
    mid = lo + (np.random.default_rng(DUMP_SEED).random(c) * (hi - lo)).astype(np.int64)
    return np.concatenate([np.arange(edge, dtype=np.int64), mid, np.arange(m - edge, m, dtype=np.int64)])


def index_stream_sample(streams, k: int) -> dict:
    """A sample of the index streams of the last step (uint32 / int32 numpy arrays or device tensors, read as one
    concatenated stream) and the positions sampled."""
    import numpy as np
    import torch

    starts = np.cumsum([0] + [len(s) for s in streams])
    pos = sample_positions(int(starts[-1]), k)
    piece = np.searchsorted(starts, pos, side="right") - 1
    vals = []
    for i, s in enumerate(streams):
        p = pos[piece == i] - starts[i]
        v = s[p] if isinstance(s, np.ndarray) else s[torch.from_numpy(p).to(s.device)].cpu().numpy()
        vals.append(v.astype(np.int64) & 0xFFFFFFFF)
    return {"structural_indexes": np.concatenate(vals), "structural_index_positions": pos}


def write_outputs(out_dir: str, arrays: dict) -> None:
    """out_dir/<name>.npy in float64 for every array (indexes, counts and error codes are below 2^53: exact)."""
    import numpy as np

    arrays = {name: np.asarray(a, dtype=np.float64) for name, a in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > 64 << 20:
        raise RuntimeError(f"--dump-outputs: {total} bytes exceed the 64 MiB limit")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def dump_last_step(args, result, streams, suffix: str = "", k: int = DUMP_ENTRIES) -> None:
    """result: the last step's verdicts, one row per document: (error, n or -1, entries written, UTF-8 verdict), or the
    batch driver's {error, n} rows."""
    if args.dump_outputs:
        arrays = {"stage1_result": result, **index_stream_sample(streams, k)}
        write_outputs(args.dump_outputs, {name + suffix: a for name, a in arrays.items()})


def dump_last_device_step(args, ctx, d_out) -> None:
    """The last call enqueued on ctx (device-resident path): its verdict, and its index stream in d_out."""
    if args.dump_outputs:
        r = ctx.finish()
        n = -1 if r.n is None else r.n
        dump_last_step(args, [(r.error, n, r.n_written, r.utf8_error)], [d_out[: n + 3 if n >= 0 else r.n_written]])


# ------------------------------------------------------------------------------------------------
# CPU arm (oracle port of the reference) -- the only place besides tests/smoke that runs oracle/
# ------------------------------------------------------------------------------------------------
def _run_pieces(fn, threads: int, repeats: int):
    best = None
    for _ in range(repeats):
        t0 = time.perf_counter()
        if threads == 1:
            fn(0)
        else:
            ts = [threading.Thread(target=fn, args=(i,)) for i in range(threads)]
            [t.start() for t in ts]
            [t.join() for t in ts]
        dt = time.perf_counter() - t0
        best = dt if best is None or dt < best else best
    return best


def cpu_stage1_gbs(sample, threads: int, repeats: int = 1, impl: str = "port", last: list | None = None):
    """Times the CPU stage 1 on `sample`, split into `threads` independent pieces run concurrently (ctypes releases the
    GIL).  impl "port": oracle_stage1_ref, the block-for-block restatement of the reference incl. its 64-iteration
    prefix_xor; "simd": oracle/stage1_simd.c, AVX-512 / AVX2 + pclmulqdq stage 1 of the same specification.
    last (port only): receives, per piece, ((error, n or -1, entries written, UTF-8 verdict), index stream) of the last pass."""
    import numpy as np

    from oracle import oracle

    n_bytes = int(sample.size)
    piece = (n_bytes + threads - 1) // threads
    parts = [sample[i * piece : min(n_bytes, (i + 1) * piece)] for i in range(threads)]
    outs = [np.empty(p.size // 3 + 64, dtype=np.uint32) for p in parts]
    results = [None] * threads
    if impl == "port":
        L = oracle.lib(native=True)

        def work(i):
            n, nw, u8 = C.c_uint32(0xFFFFFFFF), C.c_uint64(0), C.c_int32(0)
            err = L.oracle_stage1_ref(parts[i].ctypes.data, parts[i].size, outs[i].ctypes.data, outs[i].size, C.byref(n), C.byref(nw),
                                      C.byref(u8), 0)
            results[i] = (err, -1 if n.value == 0xFFFFFFFF else n.value, nw.value, u8.value)
    else:
        L = oracle.simd_lib()

        def work(i):
            n, nw, u8 = C.c_uint32(0), C.c_uint64(0), C.c_int32(0)
            L.simd_stage1(parts[i].ctypes.data, parts[i].size, outs[i].ctypes.data, outs[i].size, C.byref(n), C.byref(nw), C.byref(u8), 0, 0)
    best = _run_pieces(work, threads, repeats)
    if last is not None:
        # the stream is n + 3 entries (the trailer) when n was assigned, else the entries written before the early return
        last[:] = [(r, outs[i][: r[1] + 3 if r[1] >= 0 else r[2]]) for i, r in enumerate(results)]
    return n_bytes / best / 1e9, best


def cpu_simd_report(sample, cores: int):
    """cpu_simd (SURVEY.md 8(d)): an upstream-quality CPU stage 1 of the same specification, 1 thread and all cores
    (independent pieces; a single document cannot be split that way -- the all-core figure is the NDJSON-style bound)."""
    try:
        from oracle import oracle

        level = oracle.simd_level()
        if level == 0:
            return {"unavailable": "this CPU has neither AVX-512 nor AVX2 with pclmulqdq"}
        one, _ = cpu_stage1_gbs(sample, 1, repeats=2, impl="simd")
        allc, _ = cpu_stage1_gbs(sample, cores, repeats=2, impl="simd")
        return {"kind": "cpu_simd", "isa": "AVX-512 + pclmulqdq" if level == 2 else "AVX2 + pclmulqdq", "gbs_1_thread": round(one, 3),
                "gbs_all_cores": round(allc, 3), "cores": cores, "sample_bytes": int(sample.size),
                "note": "oracle/stage1_simd.c: vpshufb classifier, add-carry escapes, clmul prefix xor, Keiser-Lemire UTF-8, "
                        "compress-store index extraction; bit-exact with the oracle (tests/test_oracle.py); all cores = independent pieces"}
    except Exception as e:  # pragma: no cover
        return {"unavailable": repr(e)[:200]}


def cpu_model():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


def run_reference(args):
    """Reference arm: rank 0 only.  Exactly --warmup untimed and --steps timed steps; a step is one pass of the CPU port over
    a bounded sample of the same workload, sized (from one probe pass) so that the whole run ends within a few minutes."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import numpy as np

    from mojo_simdjson_b200 import synth

    n_gpus = args.gpus
    cores = os.cpu_count() or 1
    # the reference is a single-threaded, sequential scan: one document can use one core; an NDJSON batch can use
    # one core per independent segment
    threads = 1 if n_gpus == 1 else min(cores, 64)
    probe_bytes = (8 << 20) * threads
    if n_gpus == 1:
        size = synth.TWITTER_BYTES if args.config == "small" else args.bytes_per_gpu
        full = np.empty(min(size, 64 << 20), dtype=np.uint8)
        probe = make_document(args.config if args.config == "small" else "doc1g", min(size, probe_bytes), full)
    else:
        size = args.total_bytes
        probe = synth.ndjson(probe_bytes, synth.SEED_NDJSON)
    gbs_probe, _ = cpu_stage1_gbs(probe, threads)
    budget_s = 120.0
    per_step = int(gbs_probe * 1e9 * budget_s / max(1, args.steps + args.warmup))
    per_step = max(1 << 20, min(per_step, (64 << 20) * threads, size))
    per_step -= per_step % 64 if per_step > 64 else 0
    if n_gpus == 1:
        if args.config == "small":
            per_step = size
            sample = make_document("small", size, np.empty(size, dtype=np.uint8))
        else:
            sample = make_document("doc1g" if args.config == "doc1g" else args.config, per_step, np.empty(per_step, dtype=np.uint8))
    else:
        sample = synth.ndjson(per_step, synth.SEED_NDJSON)
    # cpu_simd runs ~25x faster than the port: give it its own, larger sample (256 MiB) so that the all-core figure is not a
    # thread start-up measurement
    if n_gpus == 1 and args.config == "small":
        simd_sample = sample
    elif n_gpus == 1:
        simd_sample = make_document(args.config, min(size, 256 << 20), np.empty(min(size, 256 << 20), dtype=np.uint8))
    else:
        simd_sample = synth.ndjson(256 << 20, synth.SEED_NDJSON)
    for _ in range(args.warmup):
        cpu_stage1_gbs(sample, threads)
    t_total = 0.0
    last = []
    for _ in range(args.steps):
        _, dt = cpu_stage1_gbs(sample, threads, last=last)
        t_total += dt
    dump_last_step(args, [r for r, _ in last], [s for _, s in last])
    gbs = per_step * args.steps / t_total / 1e9
    sample_desc = (f"{per_step} bytes ({per_step / (1 << 20):.1f} MiB) of the same generator per step, {args.steps} timed steps after "
                   f"{args.warmup} warm-up steps, {threads} thread(s); CPU: {cpu_model()}, {cores} cores")
    cfg = workload_config(n_gpus, args.config, size if n_gpus == 1 else args.bytes_per_gpu, args.total_bytes, args.seg_bytes)
    cfg["reference_sample_bytes_per_step"] = per_step
    line = {
        "impl": "reference", "metric": METRIC, "value": round(gbs, 4), "unit": UNIT, "n_gpus": n_gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": round(1e3 * t_total / args.steps, 3), "higher_is_better": True,
        "scaling": "weak" if n_gpus == 1 else "strong", "vs_baseline": None, "dtype": "u8", "data": "synthetic", "config": cfg,
        "cpu_baseline": {"value": round(gbs, 4), "unit": UNIT, "cores": threads, "kind": "port", "sample": sample_desc,
                         "cpu_simd": cpu_simd_report(simd_sample, cores)},
        "e2e": {"value": round(gbs, 4), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "note": "CPU restatement of the reference's stage 1 (oracle/stage1_oracle.c, -O3 -march=native), a linear scan timed on a "
                "bounded sample of the workload named in config; the Mojo reference itself cannot be built in this image",
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
def kernel_kind_for(args, seg_bytes: int) -> str:
    """Which kernel organisation the library picks for a document of this size (capi.cu: SPLIT_MIN_BYTES / STREAM_MIN_BYTES)."""
    if args.kernel != "auto":
        return args.kernel
    return "stream" if seg_bytes >= (80 << 20) else "split" if seg_bytes >= (24 << 20) else "persistent"


KERNEL_NAMES = {
    "stream": "stage-1 stream pipeline, 4 launches per document: stage1_stream_classify_kernel -> stage1_span_scan_kernel -> "
              "stage1_flatten2_kernel (+ stage1_persistent_kernel as a no-op fallback)",
    "persistent": "stage1_persistent_kernel", "split": "stage1_classify_kernel + stage1_flatten2_kernel",
}


def roofline_object(args, kind, alg_bytes, k_ms, k_ms_check, density):
    peak, peak_kind = measured_peak()
    prof = ncu_traffic(kind) if args.config == "doc1g" else {}
    achieved = alg_bytes / (k_ms * 1e-3) / 1e9
    return {"bound": "hbm", "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s", "frac": round(achieved / peak, 4),
            "traffic": prof.get("dram_bytes_per_pass"), "traffic_source": prof.get("source"), "peak_source": f"of {peak_kind}",
            "kernel": KERNEL_NAMES[kind], "kernel_ms": round(k_ms, 4), "kernel_ms_second_loop": round(k_ms_check, 4),
            "algorithmic_bytes_per_launch": int(alg_bytes), "structural_density": round(density, 4),
            "note": "achieved = algorithmic bytes of one document pass / device time of ALL its launches (CUDA events)",
            "ncu_kernel_shares": prof.get("kernel_shares")}, peak


def run_small(args, torch, np, dev, local):
    """BASELINE.json configs[1]: the 631,515-byte document.  Launch-bound: the figures are microseconds."""
    from mojo_simdjson_b200 import _native, device, synth
    from oracle import oracle

    size = synth.TWITTER_BYTES
    h_in = torch.empty(size, dtype=torch.uint8, pin_memory=True)
    doc = make_document("small", size, h_in.numpy())
    d_in = h_in.to(dev)
    d_out = torch.empty(size + 16, dtype=torch.int32, device=dev)
    h_out = torch.empty(size + 16, dtype=torch.int32, pin_memory=True)
    ctx = device.Stage1Context(local, max_len=1 << 24, max_len_host=1 << 24)
    stream = torch.cuda.current_stream(dev)
    ctx.use_stream(stream)
    flags = _native.FLAG_NO_UTF8 if args.no_utf8 else 0
    want = oracle.stage1(doc, impl="fast")
    res = ctx.index(d_in, d_out, flags)
    assert res.error == want.error == 0 and res.n == want.n
    assert np.array_equal(d_out[: want.n + 3].cpu().numpy().view(np.uint32), want.indexes), "GPU index stream differs from the oracle"
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    for _ in range(max(args.warmup, 3)):
        ctx.enqueue(d_in, d_out, flags)
    torch.cuda.synchronize()
    sampler = ClockSampler(local)
    sampler.start()
    launches0 = ctx.launch_count()
    # (1) cold: L2 flushed before every launch, one event pair per launch
    cold = []
    for _ in range(args.steps):
        flush.fill_(1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        ctx.enqueue(d_in, d_out, flags)
        e1.record(stream)
        cold.append((e0, e1))
    torch.cuda.synchronize()
    cold_us = sorted(1e3 * a.elapsed_time(b) for a, b in cold)
    launches = ctx.launch_count() - launches0
    dump_last_device_step(args, ctx, d_out)   # the timed figure is the cold launches': their last one
    # (2) back to back (L2 warm), one event pair around K launches
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(args.steps):
        ctx.enqueue(d_in, d_out, flags)
    e1.record(stream)
    torch.cuda.synchronize()
    b2b_us = 1e3 * e0.elapsed_time(e1) / args.steps
    # (3) synchronous device-resident call (launch + kernel + verdict visible on the host), wall clock
    t0 = time.perf_counter()
    for _ in range(args.steps):
        ctx.index(d_in, d_out, flags)
    sync_us = (time.perf_counter() - t0) * 1e6 / args.steps
    # (4) host to host through sjb200_stage1 (pinned in, pinned out)
    L = _native.lib()
    n_out, u8 = C.c_uint32(0), C.c_int32(0)
    for _ in range(5):
        L.sjb200_stage1(ctx._ctx, h_in.data_ptr(), size, h_out.data_ptr(), h_out.numel(), C.byref(n_out), C.byref(u8), flags)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        rc = L.sjb200_stage1(ctx._ctx, h_in.data_ptr(), size, h_out.data_ptr(), h_out.numel(), C.byref(n_out), C.byref(u8), flags)
    h2h_us = (time.perf_counter() - t0) * 1e6 / args.steps
    clocks = sampler.stop()
    assert rc == 0 and n_out.value == want.n and np.array_equal(h_out[: want.n + 3].numpy().view(np.uint32), want.indexes)
    med = cold_us[len(cold_us) // 2]
    alg = size + 4 * (want.n + 3)
    roofline, _ = roofline_object(args, "persistent", alg, med * 1e-3, b2b_us * 1e-3, want.n / size)
    roofline["note"] = "launch-latency bound at this size; achieved = algorithmic bytes / median cold launch time"
    cpu = None
    if not args.no_cpu_baseline:
        gbs, secs = cpu_stage1_gbs(doc, 1, repeats=20)
        cpu = {"value": round(gbs, 4), "unit": UNIT, "cores": 1, "kind": "port",
               "sample": f"the whole document, best of 20 passes ({secs * 1e6:.0f} us); oracle_stage1_ref; CPU: {cpu_model()}, {os.cpu_count()} cores",
               "cpu_simd": cpu_simd_report(doc, 1), "parity_checked_indexes": int(want.n + 3)}
    line = {
        "metric": METRIC, "value": round(size / med / 1e3, 3), "unit": UNIT, "n_gpus": 1, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": round(med * 1e-3, 5), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8",
        "data": "synthetic", "config": workload_config(1, "small", size), "roofline": roofline, "cpu_baseline": cpu,
        "e2e": {"value": round(size / h2h_us / 1e3, 3), "unit": UNIT, "h2d_bytes_per_step": size, "d2h_bytes_per_step": 4 * (want.n + 3),
                "steps": args.steps, "ms_per_step": round(h2h_us * 1e-3, 5), "api": "sjb200_stage1 (pinned host in, pinned host out), wall clock"},
        "gpu_launches": int(launches), "clocks": clocks, "utf8_validation": not args.no_utf8,
        "latency_us": {"cold_l2_flushed_median": round(med, 2), "cold_l2_flushed_min": round(cold_us[0], 2),
                       "cold_l2_flushed_p90": round(cold_us[int(0.9 * (len(cold_us) - 1))], 2), "back_to_back_per_launch": round(b2b_us, 2),
                       "synchronous_device_call": round(sync_us, 2), "host_to_host_call": round(h2h_us, 2)},
    }
    print(json.dumps(line), flush=True)
    ctx.close()


def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    from mojo_simdjson_b200 import _native, batch, device, errors, synth

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the stage-1 path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world == 1 and args.config == "small":
        return run_small(args, torch, np, dev, local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    n_gpus = world
    flags = _native.FLAG_NO_UTF8 if args.no_utf8 else 0
    stream = torch.cuda.current_stream(dev)

    # ---- workload: generated straight into pinned host memory, then resident in HBM -------------------
    driver = None
    if n_gpus == 1:
        size = args.bytes_per_gpu
        h_in = torch.empty(size, dtype=torch.uint8, pin_memory=True)
        make_document(args.config, size, h_in.numpy())
        d_in = h_in.to(dev, non_blocking=True)
        ctx = device.Stage1Context(local, max_len=(1 << 32) - 1, max_len_host=size)
        ctx.use_stream(stream)
        seg_offsets, idx_offsets, nseg = [0, size], [0, size // 3 + 64], 1
        cap = size // 3 + 64 if args.config in ("doc1g", "runs") else size + 64
        idx_offsets = [0, cap]
    else:
        size = args.total_bytes // n_gpus                     # this rank's shard
        reps = max(1, size // NDJSON_TEMPLATE)
        size = reps * NDJSON_TEMPLATE
        h_in = torch.empty(size, dtype=torch.uint8, pin_memory=True)
        tpl = synth.ndjson(NDJSON_TEMPLATE, synth.SEED_NDJSON + rank, out=h_in.numpy()[:NDJSON_TEMPLATE])
        for r in range(1, reps):
            h_in.numpy()[r * NDJSON_TEMPLATE : (r + 1) * NDJSON_TEMPLATE] = tpl
        d_in = h_in.to(dev, non_blocking=True)
        driver = batch.NdjsonBatchDriver(local, seg_bytes=min(args.seg_bytes, 0x7FFFFFFF), max_segments=16, stream=stream)
        ctx = driver.ctx
        seg_offsets = driver.plan(d_in)
        idx_offsets = driver.index_offsets()
        nseg = len(seg_offsets) - 1
        cap = driver.index_capacity()
    d_out = torch.empty(cap, dtype=torch.int32, device=dev)
    if args.warps:
        ctx.set_warps(args.warps)
    if args.kernel != "auto":
        ctx.set_kernel(args.kernel)
    torch.cuda.synchronize()

    def step():
        if n_gpus == 1:
            rc = ctx.enqueue(d_in, d_out, flags)
            if rc != errors.SUCCESS:
                raise RuntimeError(f"launch failed: {errors.NAMES.get(rc, rc)}")
        else:
            # every segment's kernels, then (inside the library) the all-gather of the per-segment rows on the exchange
            # stream: no host round trip, and on the GPU it runs beside the kernels of the next pass
            driver.enqueue(d_out, flags)

    # ---- correctness gate before any timing: every segment against the oracle -----------------------------
    from oracle import oracle

    parity = {"segments": nseg, "checked_indexes": 0, "how": ""}
    if n_gpus == 1:
        res = ctx.index(d_in, d_out, flags)
        n_total = res.n
        if res.error != 0 or not n_total:
            raise RuntimeError(f"stage 1 failed on the bench document: {res}")
        tr = d_out[n_total : n_total + 3].cpu().numpy().view(np.uint32).tolist()
        assert tr == [size & 0xFFFFFFFF, size & 0xFFFFFFFF, 0], tr
        if args.config != "doc1g":   # the adversarial documents: whole-document digest (the default document: see cpu_baseline)
            want = oracle.stage1(h_in.numpy(), impl="fast", cap=cap, native=True, flags=0)
            got = d_out[: n_total + 3].cpu().numpy().view(np.uint32)
            if (want.error, want.n) != (0, n_total) or oracle.index_digest(got) != oracle.index_digest(want.indexes) or res.utf8_error != want.utf8_error:
                raise RuntimeError("GPU index stream differs from the oracle on the bench document")
            parity.update(checked_indexes=int(n_total + 3), how="n, verdict, UTF-8 verdict and 128-bit digest of the whole index stream vs oracle_stage1_fast")
    else:
        step()
        worst, rows = driver.finish()
        if worst != 0:
            raise RuntimeError(f"stage 1 failed on an NDJSON segment: {rows[rank].tolist()}")
        n_total = int(rows[rank, :nseg, 1].sum())
        assert rows.shape[0] == world and all(int(r[:, 0].max()) == 0 for r in rows)
        wants = {}
        for s in range(nseg):
            a, b = seg_offsets[s], seg_offsets[s + 1]
            key = (a % NDJSON_TEMPLATE, b - a)        # the shard is a replicated template: equal segments have equal answers
            if key not in wants:
                w = oracle.stage1(h_in.numpy()[a:b], impl="fast", cap=(b - a) // 3 + 64, native=True)
                wants[key] = (w.error, w.n, oracle.index_digest(w.indexes))
            werr, wn, wdig = wants[key]
            got = d_out[idx_offsets[s] : idx_offsets[s] + wn + 3].cpu().numpy().view(np.uint32)
            if (werr, wn) != (0, int(rows[rank, s, 1])) or oracle.index_digest(got) != wdig:
                raise RuntimeError(f"rank {rank} segment {s}: GPU index stream differs from the oracle")
            parity["checked_indexes"] += int(wn + 3)
        parity["how"] = "every segment of this rank: n, verdict and 128-bit digest of its index stream vs oracle_stage1_fast on the same bytes"
    density = n_total / size

    # ---- timed region: K passes, device-resident ----------------------------------------------------------
    for _ in range(args.warmup):
        step()
    if driver is not None:
        driver.finish()
    torch.cuda.synchronize()
    sampler = ClockSampler(local)   # NVML initialisation takes tens of ms with 8 processes: before the barrier, not after
    launches0 = ctx.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler.start()
    if world > 1:
        dist.barrier()
        torch.cuda.synchronize()
    # the last warm-up passes run right in front of the timed ones, stream ordered, so that the timed region does not start on
    # a GPU that sat idle while the clock sampler initialised (NVML takes tens of ms)
    for _ in range(min(args.warmup, 10)):
        step()
    launches0 = ctx.launch_count()   # (host-side counter: only the launches of the timed passes are reported)
    ev0.record(stream)
    t_host0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    host_enqueue_ms = (time.perf_counter() - t_host0) * 1e3 / args.steps   # CPU time to issue one pass (diagnostic)
    if driver is not None:
        _, last_rows = driver.finish()   # the last verdict exchanges belong to the timed region (the host waits for them, then records)
    ev1.record(stream)
    torch.cuda.synchronize()
    clocks = sampler.stop()
    if n_gpus == 1:
        dump_last_device_step(args, ctx, d_out)
    elif args.dump_outputs:
        # this rank's segments; every rank holds the all-gathered {error, n} rows of all of them
        rows = last_rows[rank, :nseg].tolist()
        streams = [d_out[idx_offsets[s] : idx_offsets[s] + (n + 3 if e == 0 else 0)] for s, (e, n) in enumerate(rows)]
        dump_last_step(args, last_rows.reshape(-1, 2), streams, suffix=f"_rank{rank}", k=DUMP_ENTRIES // world)
    if world > 1:
        dist.barrier()
        torch.cuda.synchronize()
    launches = ctx.launch_count() - launches0
    ms_total = ev0.elapsed_time(ev1)
    t = torch.tensor([ms_total], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        lt = torch.tensor([launches], dtype=torch.int64, device=dev)
        dist.all_reduce(lt, op=dist.ReduceOp.SUM)
        launches = int(lt.item())
    ms_step = float(t.item()) / args.steps
    value = n_gpus * size / (ms_step * 1e-3) / 1e9

    # ---- the document pass alone (same launches, CUDA events on its stream) for the roofline -------------------
    kev0, kev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    kreps = max(10, min(args.steps, 50))
    status = torch.empty((max(nseg, 1), 2), dtype=torch.int32, device=dev)
    torch.cuda.synchronize()
    kev0.record(stream)
    for _ in range(kreps):
        if n_gpus == 1:
            ctx.enqueue(d_in, d_out, flags)
        else:
            ctx.run_segments_async(d_in, seg_offsets, d_out, status, flags)
    kev1.record(stream)
    torch.cuda.synchronize()
    k_ms = kev0.elapsed_time(kev1) / kreps / nseg  # per document pass
    if n_gpus == 1:
        # at N = 1 a timed step IS one document pass (same launches, same stream, same events): report the roofline from
        # the timed region itself so that `value` and `roofline.achieved` can never disagree; the loop above is kept as a
        # cross-check
        k_ms_check, k_ms = k_ms, ms_step
    else:
        k_ms_check = k_ms
    alg_bytes = (size + 4 * (n_total + 3 * nseg)) / nseg  # per pass: input read once + every index written once
    kind = kernel_kind_for(args, size // nseg)
    roofline, peak = roofline_object(args, kind, alg_bytes, k_ms, k_ms_check, density)

    # ---- end to end through the host-buffer C-ABI call ------------------------------------------------------
    L = _native.lib()
    n_out = C.c_uint32(0)
    u8 = C.c_int32(0)
    e2e_cap = max(idx_offsets[s + 1] - idx_offsets[s] for s in range(nseg)) if n_gpus > 1 else cap
    e2e_cap = min(e2e_cap, (max(seg_offsets[s + 1] - seg_offsets[s] for s in range(nseg))) // 3 + 64) if args.config in ("doc1g", "runs") or n_gpus > 1 else e2e_cap
    h_out = torch.empty(e2e_cap, dtype=torch.int32, pin_memory=True)
    h_status = torch.zeros((nseg, 2), dtype=torch.int32)
    if n_gpus > 1:
        e2e_ctx = device.Stage1Context(local, max_len=(1 << 31) - 1, max_len_host=max(seg_offsets[s + 1] - seg_offsets[s] for s in range(nseg)))
        e2e_ctx.use_stream(stream)
    else:
        e2e_ctx = ctx

    def e2e_step():
        worst = 0
        for s in range(nseg):
            a, b = seg_offsets[s], seg_offsets[s + 1]
            rc = L.sjb200_stage1(e2e_ctx._ctx, h_in.data_ptr() + a, b - a, h_out.data_ptr(), e2e_cap, C.byref(n_out), C.byref(u8), flags)
            h_status[s, 0] = rc
            h_status[s, 1] = n_out.value
            worst = max(worst, rc)
        if world > 1:
            d_st = h_status.to(dev, non_blocking=True)
            batch.exchange_verdicts(d_st[:, 0], d_st[:, 1], 16)
        return worst

    e2e_step()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
        torch.cuda.synchronize()
    eev0, eev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    eev0.record(stream)
    for _ in range(args.e2e_steps):
        rc = e2e_step()
    eev1.record(stream)
    torch.cuda.synchronize()
    e_ms = torch.tensor([eev0.elapsed_time(eev1) / args.e2e_steps], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(e_ms, op=dist.ReduceOp.MAX)
    e2e_value = n_gpus * size / (float(e_ms.item()) * 1e-3) / 1e9
    got = h_out[: n_out.value + 3].numpy().view(np.uint32) if nseg == 1 else None
    e2e = {"value": round(e2e_value, 3), "unit": UNIT, "h2d_bytes_per_step": int(size),
           "d2h_bytes_per_step": int(4 * (n_total + 3 * nseg)), "steps": args.e2e_steps,
           "ms_per_step": round(float(e_ms.item()), 3), "api": "sjb200_stage1 (pinned host in, pinned host out), one call per segment"}
    if rc != 0:
        raise RuntimeError(f"e2e pass failed: {rc}")
    if got is not None:
        assert int(got[-3]) == size % (1 << 32) and int(got[-1]) == 0 and n_out.value == n_total

    # ---- CPU baseline beside it (rank 0, N = 1 only) ----------------------------------------------------------
    cpu = None
    if rank == 0 and n_gpus == 1 and not args.no_cpu_baseline:
        sample_bytes = min(size, args.cpu_sample_bytes)
        sample = h_in.numpy()[:sample_bytes]
        gbs, secs = cpu_stage1_gbs(sample, 1)
        # bit-exact check of the GPU stream against the oracle on that sample's prefix (default document; the others were
        # digested whole above)
        chk = min(sample_bytes, 64 << 20)
        want = oracle.stage1(h_in.numpy()[:chk], impl="fast", cap=chk + 16 if args.config in ("cjk", "dense") else chk // 3 + 16, native=True)
        k = want.n_written - 1  # the prefix is cut mid-document: compare the indexes that lie inside it
        mine = d_out[:k].cpu().numpy().view(np.uint32)
        if not bool(np.array_equal(mine, want.indexes[:k])):
            raise RuntimeError("GPU index stream differs from the oracle on the bench document")
        cpu = {"value": round(gbs, 4), "unit": UNIT, "cores": 1, "kind": "port",
               "sample": f"first {sample_bytes >> 20} MiB of the same document, one pass, {secs:.1f} s; oracle_stage1_ref "
                         f"(restatement of the reference incl. its 64-iteration prefix_xor), gcc -O3 -march=native; "
                         f"CPU: {cpu_model()}, {os.cpu_count()} cores",
               "parity_checked_indexes": int(max(k, parity["checked_indexes"])),
               "cpu_simd": cpu_simd_report(h_in.numpy()[: min(size, 256 << 20)], os.cpu_count() or 1)}

    # per-rank picture (N > 1): every rank's own pass time without the exchange, own timed-region time, own clocks and its
    # parity check -- the job-level number is the maximum over ranks, so one slower GPU shows up here
    per_rank = None
    if world > 1:
        mine = {"kernel_ms": round(k_ms * nseg, 4), "timed_ms_per_step": round(ms_total / args.steps, 4),
                "sm_mhz": clocks.get("sm_mhz"), "reasons": clocks.get("reasons"), "segments": nseg,
                "parity_checked_indexes": parity["checked_indexes"]}
        gathered = [None] * world
        dist.all_gather_object(gathered, mine)
        per_rank = gathered
    if rank == 0:
        line = {
            "metric": METRIC, "value": round(value, 2), "unit": UNIT, "n_gpus": n_gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": round(ms_step, 4), "higher_is_better": True, "scaling": "weak" if n_gpus == 1 else "strong",
            "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": workload_config(n_gpus, args.config, size, size * n_gpus, args.seg_bytes),
            "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks,
            "utf8_validation": not args.no_utf8, "segments_per_gpu": nseg, "host_enqueue_ms_per_step": round(host_enqueue_ms, 4),
            "parity": parity, "per_rank": per_rank,
            "frac_of_aggregate_hbm": round(value * (alg_bytes * nseg / size) / (peak * n_gpus), 4),
        }
        print(json.dumps(line), flush=True)
    if driver is not None:
        e2e_ctx.close()
        driver.close()
    else:
        ctx.close()
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse_args()
    world = int(os.environ.get("WORLD_SIZE", "0"))
    if args.gpus > 1 and world == 0:
        # plain `python bench.py --gpus N`: start one rank per GPU ourselves
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", str(free_port()), os.path.abspath(__file__)] + sys.argv[1:]
        raise SystemExit(subprocess.call(cmd))
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
