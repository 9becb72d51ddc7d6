"""B independent graphs: B sequential LaplaceLearningSparseHard fwd+bwd calls against one LaplaceLearningSparseHardBatched call.
Run on the GPU box:

    python tools/batched_bench.py [--out FILE.json] [--reps 20]

Shapes: the C1 graph (1000 labeled + 1000 unlabeled rows, d = 128) x 8, 4096 + 512 at d = 512 x 4, and 25 + 75 at d = 64 x 64
(episodic few-shot size).  Each variant is timed eagerly and as one replayed CUDA graph (the B sequential calls captured
together), with CUDA events around `reps` calls after warm-up; inputs stay resident in L2 (all below 126 MB), as they would
in a training step.  Per-stage times come from one separately profiled eager call of each variant (gll_profile_*), and the
kNN work from gll_knn_segments_units: tensor-core units the segmented search issues against the uniform grid over the
same rows.  The card's name and power limit are read in the same run.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import graphlearninglayer_b200 as pkg  # noqa: E402
from graphlearninglayer_b200 import _lib  # noqa: E402
from graphlearninglayer_b200.synth import synth_inputs  # noqa: E402

# (name, B, k_lab, m, d, l, cluster spread): the spreads of bench.py's c1 and c3 workloads; at d = 512 a smaller spread makes the
# predictions one-hot to the last bit and the gradient pure rounding noise
SHAPES = [("c1x8", 8, 1000, 1000, 128, 10, 3.0), ("4096+512_d512x4", 4, 4096, 512, 512, 10, 4.5),
          ("25+75_d64x64", 64, 25, 75, 64, 5, 2.0)]


def gpu_identity():
    out = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30)
        out["power_limit_and_max_sm_clock"] = q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unavailable"
    except (OSError, subprocess.SubprocessError):
        out["power_limit_and_max_sm_clock"] = "unavailable"
    return out


def loss_of(pred, oh):
    return -torch.sum(oh * torch.log(pred + 1e-8)) / pred.shape[-2]


def time_ms(fn, reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def graphed(fn):
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(2):
            fn()
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        fn()
    return g.replay


def profiled(fn):
    fn()
    torch.cuda.synchronize()
    _lib.profile_collect()
    _lib.lib.gll_profile_enable(1)
    try:
        fn()
        torch.cuda.synchronize()
        return {k: {"ms": round(v[0], 4), "launches": v[1]} for k, v in _lib.profile_collect().items()}
    finally:
        _lib.lib.gll_profile_enable(0)


def case(name, B, k_lab, m, d, l, sigma, reps):
    Xs, Ys, ys = [], [], []
    for b in range(B):
        X, Y, _, yq = synth_inputs(1000 + b, k_lab, m, d, l, sigma)
        Xs.append(X)
        Ys.append(Y)
        ys.append(yq)
    X = torch.as_tensor(np.stack(Xs)).cuda().requires_grad_(True)
    Y = torch.as_tensor(np.stack(Ys)).cuda()
    oh = torch.nn.functional.one_hot(torch.as_tensor(np.stack(ys)).cuda(), l).double()
    Xb = [X[b].detach().clone().requires_grad_(True) for b in range(B)]

    def sequential():
        for b in range(B):
            Xb[b].grad = None
            loss_of(pkg.LaplaceLearningSparseHard.apply(Xb[b], Y[b], 0.0, "auto"), oh[b]).backward()

    def batched():
        X.grad = None
        loss_of(pkg.LaplaceLearningSparseHardBatched.apply(X, Y, 0.0, "auto"), oh).backward()

    for f in (sequential, batched):
        f()
    torch.cuda.synchronize()
    dev = max(float((X.grad[b] - Xb[b].grad).abs().max() / Xb[b].grad.abs().max()) for b in range(B))
    out = {"shape": name, "B": B, "k_lab": k_lab, "m": m, "d": d, "l": l, "sigma": sigma, "max_rel_dX_batched_vs_sequential": dev}
    n = k_lab + m
    seg = _lib.seg_ptr_array([b * n for b in range(B + 1)])
    su, uu = ctypes.c_longlong(), ctypes.c_longlong()
    _lib.lib.gll_knn_segments_units(B * n, d, seg, B, ctypes.byref(su), ctypes.byref(uu))
    out["knn_units"] = {"segmented": su.value, "uniform_grid": uu.value}
    out["stages_sequential"] = profiled(sequential)
    out["stages_batched"] = profiled(batched)
    out["ms_sequential_eager"] = time_ms(sequential, reps)
    out["ms_batched_eager"] = time_ms(batched, reps)
    out["ms_sequential_graph"] = time_ms(graphed(sequential), reps)
    out["ms_batched_graph"] = time_ms(graphed(batched), reps)
    out["speedup_eager"] = out["ms_sequential_eager"] / out["ms_batched_eager"]
    out["speedup_graph"] = out["ms_sequential_graph"] / out["ms_batched_graph"]
    print(json.dumps({k: v for k, v in out.items() if not k.startswith("stages")}), flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="")
    ap.add_argument("--reps", type=int, default=20)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("batched_bench.py needs a CUDA device")
    torch.cuda.set_device(0)
    res = {"gpu": gpu_identity(), "reps": a.reps, "cases": [case(*s, a.reps) for s in SHAPES]}
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
