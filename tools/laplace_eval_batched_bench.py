"""B independent graphs evaluated with Laplace learning: B sequential laplace_learning calls against one laplace_learning_batched
call, k = 50.  Run on the GPU box:

    python tools/laplace_eval_batched_bench.py [--out FILE.json] [--reps 20]

Shapes: 25 + 75 at d = 64, l = 5, x 64 (episodic few-shot size), 200 + 1800 at d = 128, l = 10, x 16, and 1000 + 9000 at
d = 128, l = 10, x 4.  A single 100-row graph cannot take k = 50 (k > 33 needs 256 rows per gll_knn call), so the few-shot shape
compares both variants at k = 33 and also times the batched call at k = 50, where only the batch reaches 256 rows.  Each variant
is timed eagerly and as one replayed CUDA graph (the B sequential calls captured together), with CUDA events around `reps`
calls after warm-up; the inputs stay resident in L2, as they would in an evaluation loop.  Per-stage times come from one
separately profiled eager call of each variant (gll_profile_*), the kNN work from gll_knn_segments_units.  Per shape the
largest pred difference against the sequential calls (max-relative), whether the labels are identical and whether the correct
counts are equal are recorded.  The card's name and power limit are read in the same run.
"""
import argparse
import ctypes
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)
import numpy as np  # noqa: E402
import torch  # noqa: E402

import graphlearninglayer_b200 as pkg  # noqa: E402
from batched_bench import gpu_identity, graphed, profiled, time_ms  # noqa: E402
from graphlearninglayer_b200 import _lib  # noqa: E402
from graphlearninglayer_b200.laplace_eval import last_eval_info  # noqa: E402
from graphlearninglayer_b200.synth import synth_inputs  # noqa: E402

# (name, B, k_lab, m, d, l, k of the comparison)
SHAPES = [("25+75_d64x64", 64, 25, 75, 64, 5, 33), ("200+1800_d128x16", 16, 200, 1800, 128, 10, 50),
          ("1000+9000_d128x4", 4, 1000, 9000, 128, 10, 50)]
SIGMA = 2.0


def case(name, B, k_lab, m, d, l, k, reps):
    Xs, Ys, ys = [], [], []
    for b in range(B):
        X, Y, _, yq = synth_inputs(2000 + b, k_lab, m, d, l, SIGMA)
        Xs.append(X)
        Ys.append(Y)
        ys.append(yq)
    X = torch.as_tensor(np.stack(Xs)).cuda()
    Y = torch.as_tensor(np.stack(Ys)).cuda()
    T = torch.as_tensor(np.stack(ys).astype(np.int64)).cuda()
    seq_out, bat_out = [None] * B, [None]

    def sequential():
        for b in range(B):
            seq_out[b] = pkg.laplace_learning(X[b], Y[b], k=k, targets=T[b])

    def batched(kk=k):
        bat_out[0] = pkg.laplace_learning_batched(X, Y, k=kk, targets=T)

    sequential()
    batched()
    torch.cuda.synchronize()
    res = bat_out[0]
    pred_s = torch.stack([r.pred for r in seq_out])
    lab_s = torch.stack([r.labels for r in seq_out])
    cor_s = torch.stack([r.correct for r in seq_out])
    out = {"shape": name, "B": B, "k_lab": k_lab, "m": m, "d": d, "l": l, "k": k, "sigma": SIGMA,
           "max_rel_pred_batched_vs_sequential": float((res.pred - pred_s).abs().max() / pred_s.abs().max()),
           "labels_identical": bool(torch.equal(res.labels, lab_s)), "correct_equal": bool(torch.equal(res.correct, cor_s)),
           "accuracy_batched": float(res.correct.sum()) / (B * m)}
    info = last_eval_info()
    out["batched_info"] = {kk: info[kk] for kk in ("rounds", "cg_iters_first", "cg_iters_correction", "round_iters", "resid")}
    out["batched_resid_per_graph_max"] = max(info["resid_per_graph"])
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
    if k < 50:  # the batch alone reaches the 256 rows k = 50 needs
        out["ms_batched_eager_k50"] = time_ms(lambda: batched(50), reps)
        out["ms_batched_graph_k50"] = time_ms(graphed(lambda: batched(50)), reps)
    print(json.dumps({kk: v for kk, v in out.items() if not kk.startswith("stages")}), flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="")
    ap.add_argument("--reps", type=int, default=20)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("laplace_eval_batched_bench.py needs a CUDA device")
    torch.cuda.set_device(0)
    res = {"gpu": gpu_identity(), "reps": a.reps, "cases": [case(*s, a.reps) for s in SHAPES]}
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
