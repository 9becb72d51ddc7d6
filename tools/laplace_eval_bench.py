"""Laplace-learning evaluation at the reference's real size (SURVEY 3.4: 10 000 labeled + 60 000 unlabeled rows, k = 50):
the device path laplace_learning() against the numpy/scipy wrapper path (knn_sym_dist + scipy assembly + stable_conjgrad,
utils.py:570-593).  Run on the GPU box:

    python tools/laplace_eval_bench.py [--out FILE.json] [--reps 5]

Device call: CUDA events around each call, after warm-up; a 256 MB buffer is overwritten between calls so that no input
(X is below the 126 MB L2) is served from L2.  Per-kernel times come from a separate profiled call (gll_profile_*), the CG
kernel that ran from a torch.profiler trace of one more call.  The wrapper path is timed with the host clock around one
synchronised call.
"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import scipy.sparse as sparse  # noqa: E402
import torch  # noqa: E402

import graphlearninglayer_b200 as pkg  # noqa: E402
from graphlearninglayer_b200 import _lib  # noqa: E402
from graphlearninglayer_b200.laplace_eval import last_eval_info  # noqa: E402
from graphlearninglayer_b200.synth import synth_inputs  # noqa: E402

K_LAB, M, L, K = 10000, 60000, 10, 50


def gpu_identity():
    out = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30)
        out["power_limit_and_max_sm_clock"] = q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unavailable"
    except (OSError, subprocess.SubprocessError):
        out["power_limit_and_max_sm_clock"] = "unavailable"
    return out


def wrapper_path(X, Y, tau):
    W = pkg.knn_sym_dist(X, K, "auto")[0]
    Lap = sparse.csgraph.laplacian(W).tocsr()
    Luu = Lap[K_LAB:, K_LAB:]
    Lul = Lap[K_LAB:, :K_LAB]
    m = Luu.shape[0]
    Luu = Luu + sparse.spdiags(tau * np.ones(m), 0, m, m).tocsr()
    Ms = sparse.spdiags(1 / np.sqrt(Luu.diagonal() + 1e-10), 0, m, m).tocsr()
    return Ms * pkg.stable_conjgrad(Ms * Luu * Ms, -Ms * Lul @ Y.astype(np.float64))


def case(d, sigma, tau, reps):
    X, Y, _, yq = synth_inputs(0, K_LAB, M, d, L, sigma)
    Xt, Yt, tt = torch.as_tensor(X).cuda(), torch.as_tensor(Y).cuda(), torch.as_tensor(yq).cuda()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def call():
        return pkg.laplace_learning(Xt, Yt, k=K, epsilon="auto", tau=tau, targets=tt)

    for _ in range(2):
        res = call()
    torch.cuda.synchronize()
    info = last_eval_info()
    times = []
    for _ in range(reps):
        flush.fill_(1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        call()
        e1.record()
        torch.cuda.synchronize()
        times.append(e0.elapsed_time(e1))
    _lib.lib.gll_profile_enable(1)
    _lib.profile_collect()
    flush.fill_(1)
    call()
    prof = _lib.profile_collect()
    _lib.lib.gll_profile_enable(0)
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as tp:
        call()
        torch.cuda.synchronize()
    cg_kernels = sorted({e.name for e in tp.events() if "cg_" in e.name and e.device_type == torch.autograd.DeviceType.CUDA})

    pred = res.pred.cpu().numpy()
    labels = res.labels.cpu().numpy()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    ref = np.asarray(wrapper_path(X, Y, tau))
    torch.cuda.synchronize()
    t_wrap = (time.perf_counter() - t0) * 1e3
    return dict(d=d, sigma=sigma, tau=tau, n=K_LAB + M, k=K, l=L,
                device_ms=dict(median=float(np.median(times)), min=float(min(times)), max=float(max(times)), calls=reps),
                device_kernel_ms={kk: dict(ms=round(v[0], 4), launches=v[1]) for kk, v in sorted(prof.items())},
                cg_kernels=cg_kernels, cg_iters_first=info["cg_iters_first"], round_iters=info["round_iters"],
                rounds=info["rounds"], scaled_resid_first=info["resid_first"], scaled_resid_final=info["resid"], status=info["status"],
                nnz=info["nnz"], wrapper_ms=t_wrap, speedup=t_wrap / float(np.median(times)),
                pred_max_rel_diff=float(np.abs(pred - ref).max() / np.abs(ref).max()),
                argmax_agreement=float((labels == ref.argmax(axis=1)).mean()),
                accuracy_device=int(res.correct) / M, accuracy_wrapper=float((ref.argmax(axis=1) == yq).mean()))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("laplace_eval_bench.py needs a CUDA device")
    out = dict(gpu=gpu_identity(), workload=f"synth_inputs(0, {K_LAB}, {M}, d, {L}, sigma), k={K}, epsilon='auto', tol=1e-10",
               l2_flush="256 MB buffer overwritten before every timed device call", cases=[])
    for d, sigma in ((128, 3.0), (512, 4.5)):
        for tau in (0.0, 1e-8):
            out["cases"].append(case(d, sigma, tau, a.reps))
            print(json.dumps(out["cases"][-1]), flush=True)
    text = json.dumps(out, indent=1)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
