"""Repeated Laplace-learning trials on one set of features: T sequential laplace_learning calls on permuted features (each trial's
labeled rows first, as laplace_learning needs them) against one laplace_learning_trials call, k = 50.  Run on the GPU box:

    python tools/laplace_eval_trials_bench.py [--out FILE.json] [--reps 5]

Shapes: n = 70 000 (the reference's evaluation size) at d = 128, l = 10, T in {1, 10, 100} with 10 and 50 labeled rows per
trial; n = 10 000 at d = 128, T in {4, 64}; n = 2 000 at d = 128, T = 64 (50 labeled rows each).  Each variant is timed eagerly and
as one replayed CUDA graph (the T sequential calls captured together), with CUDA events around `reps` rounds after warm-up; the
permuted copies of the features are made once, outside the timed window.  Per-stage times come from one separately profiled
eager call of each variant (gll_profile_*).  Per shape the largest pred difference against the sequential calls (max-relative,
over the unlabeled rows), whether the labels agree and whether the hit counts are identical are recorded.  The card's name and
power limit are read in the same run.
"""
import argparse
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
from graphlearninglayer_b200.laplace_eval import last_eval_info  # noqa: E402
from graphlearninglayer_b200.synth import synth_inputs  # noqa: E402

# (n, d, l, T, labeled rows per trial)
SHAPES = [(70000, 128, 10, T, kl) for kl in (10, 50) for T in (1, 10, 100)] + \
         [(10000, 128, 10, 4, 50), (10000, 128, 10, 64, 50), (2000, 128, 10, 64, 50)]
SIGMA, K = 3.0, 50


def case(n, d, l, T, k_lab, reps):
    X, _, yb, yq = synth_inputs(3000 + n + T, l, n - l, d, l, SIGMA)
    y = np.concatenate([yb, yq]).astype(np.int64)
    rng = np.random.default_rng(n + T + k_lab)
    idx = np.stack([rng.choice(n, k_lab, replace=False) for _ in range(T)]).astype(np.int64)
    Ys = np.eye(l, dtype=np.float32)[y[idx]]
    perms = [np.concatenate([idx[t], np.setdiff1d(np.arange(n), idx[t])]) for t in range(T)]
    Xt, It, Yt, tt = (torch.as_tensor(v).cuda() for v in (X, idx, Ys, y))
    Xp = [Xt[torch.as_tensor(p).cuda()].contiguous() for p in perms]
    Yp = [Yt[t].contiguous() for t in range(T)]
    tp = [tt[torch.as_tensor(p[k_lab:]).cuda()].contiguous() for p in perms]
    seq_out, tri_out = [None] * T, [None]

    def sequential():
        for t in range(T):
            seq_out[t] = pkg.laplace_learning(Xp[t], Yp[t], k=K, targets=tp[t])

    def trials():
        tri_out[0] = pkg.laplace_learning_trials(Xt, It, Yt, k=K, targets=tt)

    sequential()
    trials()
    torch.cuda.synchronize()
    info = last_eval_info()
    res = tri_out[0]
    worst, labels_agree, hits_equal = 0.0, True, True
    for t in range(T):
        U = torch.as_tensor(perms[t][k_lab:]).cuda()
        ref = seq_out[t]
        worst = max(worst, float((res.pred[t, U] - ref.pred).abs().max() / ref.pred.abs().max()))
        labels_agree &= bool(torch.equal(res.labels[t, U], ref.labels))
        hits_equal &= int(res.correct[t]) == int(ref.correct)
    out = {"n": n, "d": d, "l": l, "T": T, "k_lab": k_lab, "k": K, "sigma": SIGMA,
           "max_rel_pred_trials_vs_sequential": worst, "labels_identical": labels_agree, "correct_equal": hits_equal,
           "accuracy_trials": float(res.correct.sum()) / (T * (n - k_lab)),
           "trials_info": {kk: info[kk] for kk in ("rounds", "cg_iters_first", "cg_iters_correction", "round_iters", "resid")},
           "trials_resid_per_trial_max": max(info["resid_per_trial"])}
    r = reps if n * T <= 1000000 else 2  # a 100-trial sequential set at n = 70 000 takes over a second per round
    out["reps"] = r
    out["stages_sequential"] = profiled(sequential)
    out["stages_trials"] = profiled(trials)
    out["ms_sequential_eager"] = time_ms(sequential, r)
    out["ms_trials_eager"] = time_ms(trials, r)
    out["ms_sequential_graph"] = time_ms(graphed(sequential), r)
    out["ms_trials_graph"] = time_ms(graphed(trials), r)
    out["speedup_eager"] = out["ms_sequential_eager"] / out["ms_trials_eager"]
    out["speedup_graph"] = out["ms_sequential_graph"] / out["ms_trials_graph"]
    print(json.dumps({kk: v for kk, v in out.items() if not kk.startswith("stages")}), flush=True)
    del Xp, seq_out
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="")
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("laplace_eval_trials_bench.py needs a CUDA device")
    torch.cuda.set_device(0)
    res = {"gpu": gpu_identity(), "reps": a.reps, "cases": [case(*s, a.reps) for s in SHAPES]}
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
