"""Checks of bench.py.  Without a GPU: `bench.py --impl reference` (the CPU restatement of the reference's stage 1 timed on
host cores) prints one JSON line with the agreed keys, and --dump-outputs writes its last step.  On a GPU: --dump-outputs
writes what the timed device path computed, equal to the oracle's answer on the same document."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference"
    assert line["metric"] == "stage1_input_throughput" and line["unit"] == "GB/s"
    assert line["higher_is_better"] is True and line["n_gpus"] == 1 and line["steps"] == 1
    assert line["value"] > 0 and line["ms_per_step"] > 0
    assert line["dtype"] == "u8" and line["data"] == "synthetic" and "workload" in line["config"]
    cb = line["cpu_baseline"]
    assert cb["kind"] in ("port", "reference") and cb["cores"] >= 1 and cb["value"] == line["value"] and cb["sample"]
    assert line["e2e"] == {"value": line["value"], "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert line["gpu_launches"] == 0


def _run_bench(*args):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    return json.loads(out.stdout.strip().splitlines()[-1])


def _check_dump(d, doc):
    """The dumped result and index sample against the oracle on the same document."""
    import numpy as np

    from oracle import oracle

    files = sorted(os.listdir(d))
    assert files == ["stage1_result.npy", "structural_index_positions.npy", "structural_indexes.npy"]
    arrays = {f[:-4]: np.load(os.path.join(d, f)) for f in files}
    assert all(a.dtype == np.float64 for a in arrays.values())
    assert sum(a.nbytes for a in arrays.values()) <= 64 << 20
    want = oracle.stage1(doc, impl="fast", cap=doc.size // 3 + 64)
    err, n, _, u8 = arrays["stage1_result"][0]
    assert want.error == 0 and (err, n, u8) == (0, want.n, 0)
    pos = arrays["structural_index_positions"].astype(np.int64)
    assert pos[0] == 0 and pos[-1] == want.n + 2 and bool((np.diff(pos) > 0).all())
    assert np.array_equal(arrays["structural_indexes"], want.indexes[pos].astype(np.float64))


def test_reference_arm_dumps_its_last_step(tmp_path):
    from mojo_simdjson_b200 import synth

    line = _run_bench("--impl", "reference", "--steps", "1", "--warmup", "0", "--dump-outputs", str(tmp_path))
    size = line["config"]["reference_sample_bytes_per_step"]
    _check_dump(tmp_path, synth.status_array(size, synth.SEED_DOC))


def test_dump_sample_positions_are_fixed():
    import importlib.util

    import numpy as np

    spec = importlib.util.spec_from_file_location("bench", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    assert np.array_equal(bench.sample_positions(10, 100), np.arange(10))
    a, b = bench.sample_positions(10**8, 1 << 12), bench.sample_positions(10**8, 1 << 12)
    assert np.array_equal(a, b) and a.size == 1 << 12 and bool((np.diff(a) > 0).all()) and a[0] == 0 and a[-1] == 10**8 - 1


def test_native_oracle_is_built_outside_the_tree():
    """bench.py runs from a read-only checkout: the -march=native oracle it times goes to a temporary directory."""
    from oracle import oracle

    path = oracle.build(native=True)
    assert os.path.exists(path) and not os.path.abspath(path).startswith(ROOT + os.sep)


@pytest.mark.gpu
def test_gpu_arm_dumps_its_last_step(tmp_path):
    from mojo_simdjson_b200 import synth

    size = 64 << 20
    line = _run_bench("--steps", "3", "--warmup", "1", "--bytes-per-gpu", str(size), "--no-cpu-baseline", "--e2e-steps", "1",
                      "--dump-outputs", str(tmp_path))
    assert line["steps"] == 3
    _check_dump(tmp_path, synth.status_array(size, synth.SEED_DOC))
