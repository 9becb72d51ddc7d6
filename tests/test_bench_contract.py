"""CPU tests of bench.py's contract: the reference arm's JSON line (keys the driver reads) and the refusal of the B200 arm to
run without a CUDA device (no CPU fallback on the measured path); --dump-outputs, end to end on a GPU."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*args, env=None):
    e = dict(os.environ, **(env or {}))
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, cwd=ROOT, env=e,
                          timeout=600)


def test_reference_arm_prints_one_json_line_with_the_contract_keys():
    p = _run("--impl", "reference", "--workload", "c3", "--steps", "1", "--warmup", "0")
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "gll_fwd_bwd_calls_per_sec" and d["unit"] == "calls/s"
    assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["steps"] == 1 and d["value"] > 0
    assert d["config"]["workload"].startswith("c3")
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and abs(cb["value"] - d["value"]) < 1e-12 and cb["sample"]
    e2e = d["e2e"]
    assert e2e["h2d_bytes_per_step"] == 0 and e2e["d2h_bytes_per_step"] == 0 and abs(e2e["value"] - d["value"]) < 1e-12
    assert d["gpu_launches"] == 0


def test_reference_arm_other_ranks_exit_quietly():
    """Under torchrun only rank 0 times the CPU arm; the other ranks print nothing and exit 0."""
    p = _run("--impl", "reference", "--workload", "c3", "--steps", "1", "--warmup", "0", "--gpus", "2",
             env={"RANK": "1", "LOCAL_RANK": "1", "WORLD_SIZE": "2", "MASTER_ADDR": "127.0.0.1", "MASTER_PORT": "29571"})
    assert p.returncode == 0, p.stderr[-2000:]
    assert not [l for l in p.stdout.splitlines() if l.startswith("{")]


def test_b200_arm_refuses_to_run_without_cuda():
    import torch

    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    p = _run("--steps", "1", "--warmup", "0")
    assert p.returncode != 0
    assert "no CPU fallback" in (p.stderr + p.stdout)


def _bench_module():
    import importlib.util

    spec = importlib.util.spec_from_file_location("bench", os.path.join(ROOT, "bench.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_dump_outputs_writes_small_arrays_whole_and_samples_large_ones(tmp_path):
    import numpy as np
    import torch

    bench = _bench_module()
    rows = bench.DUMP_BYTES_PER_ARRAY // (64 * 4) + 1000
    big = torch.arange(rows * 64, dtype=torch.float32).reshape(rows, 64)
    small = torch.randn(7, 3, dtype=torch.float64)
    bench.dump_outputs(str(tmp_path / "a"), {"dX": big, "pred": small, "loss": torch.tensor(0.5, dtype=torch.float64)})
    bench.dump_outputs(str(tmp_path / "b"), {"dX": big})
    a = {n: np.load(tmp_path / "a" / (n + ".npy")) for n in ("dX", "pred", "loss")}
    assert np.array_equal(a["pred"], small.numpy()) and a["loss"].dtype == np.float64 and float(a["loss"]) == 0.5
    assert a["dX"].dtype == np.float32 and a["dX"].nbytes <= bench.DUMP_BYTES_PER_ARRAY and a["dX"].shape[1] == 64
    picked = a["dX"][:, 0].astype(np.int64) // 64  # the row each sampled row came from, in increasing order
    assert np.all(np.diff(picked) > 0) and np.array_equal(a["dX"], big.numpy()[picked])
    assert np.array_equal(np.load(tmp_path / "b" / "dX.npy"), a["dX"])  # the same sample every time


def test_dump_outputs_is_refused_for_the_reference_arm(tmp_path):
    p = _run("--impl", "reference", "--steps", "1", "--warmup", "0", "--dump-outputs", str(tmp_path / "out"))
    assert p.returncode != 0 and "--dump-outputs" in p.stderr
    assert not (tmp_path / "out").exists()


@pytest.mark.gpu
def test_b200_arm_dumps_the_outputs_of_its_last_timed_step(tmp_path):
    import numpy as np
    import torch

    from oracle import gll_oracle as O

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    out = tmp_path / "dump"
    p = _run("--workload", "c1", "--steps", "2", "--warmup", "1", "--no-cpu-baseline", "--no-large-graph", "--no-sharded",
             "--dump-outputs", str(out))
    assert p.returncode == 0, p.stderr[-2000:]
    d = json.loads([l for l in p.stdout.splitlines() if l.startswith("{")][-1])
    assert d["steps"] == 2
    pred, loss, dX = (np.load(out / (n + ".npy")) for n in ("pred", "loss", "dX"))
    assert pred.dtype == np.float64 and pred.shape == (1000, 10) and dX.dtype == np.float32 and dX.shape == (2000, 128)
    X, Y, _, yq = O.synth_inputs(1000, 1000, 1000, 128, 10, 3.0)  # bench.py: seed 1000, WORKLOADS["c1"]
    f, loss_ref, _, bw = O.fwd_bwd(X, Y, yq, 0.0, 1.0, solver="lu")
    assert O.max_rel(pred, f.pred) < 1e-5 and O.max_rel(dX, bw.dX) < 1e-5
    assert abs(float(loss) - loss_ref) < 1e-5 * max(1.0, abs(loss_ref))
