"""Poisson learning against Laplace learning on the same trials at one label per class (k_lab = l), k = 50.  Run on the GPU box:

    python tools/poisson_eval_bench.py [--out FILE.json] [--reps 7]

Shapes: those of tools/laplace_eval_trials_bench.py at the low label rate Poisson learning is for: n = 70 000 (the reference's
evaluation size) at d = 128, l = 10, T in {100, 10}; n = 10 000, T = 4; n = 2 000, T = 64.  Each trial labels one row of every
class, drawn with a seeded generator.  Per shape: the time of one poisson_learning call and of one laplace_learning_trials call on
the same draw (CUDA events around each call after a warm-up call, median of `reps` calls), the first-solve and correction CG
iterations of each, their mean accuracy over the unlabeled rows, and the per-stage times of one separately profiled call
(gll_profile_*).  The card's name and power limit are read in the same run.
"""
import argparse
import json
import os
import statistics
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)
import numpy as np  # noqa: E402
import torch  # noqa: E402

import graphlearninglayer_b200 as pkg  # noqa: E402
from batched_bench import gpu_identity, profiled  # noqa: E402
from graphlearninglayer_b200.laplace_eval import last_eval_info  # noqa: E402
from graphlearninglayer_b200.synth import synth_inputs  # noqa: E402

# (n, d, l, T)
SHAPES = [(70000, 128, 10, 100), (70000, 128, 10, 10), (10000, 128, 10, 4), (2000, 128, 10, 64)]
SIGMA, K = 3.0, 50


def median_ms(fn, reps):
    fn()  # warm-up
    times = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        times.append(e0.elapsed_time(e1))
    return statistics.median(times)


def case(n, d, l, T, reps):
    X, _, yb, yq = synth_inputs(3000 + n + T, l, n - l, d, l, SIGMA)
    y = np.concatenate([yb, yq]).astype(np.int64)
    rng = np.random.default_rng(n + T)
    idx = np.stack([[rng.choice(np.flatnonzero(y == c)) for c in range(l)] for _ in range(T)]).astype(np.int64)
    Ys = np.eye(l, dtype=np.float32)[y[idx]]
    Xt, It, Yt, tt = (torch.as_tensor(v).cuda() for v in (X, idx, Ys, y))
    out = {"n": n, "d": d, "l": l, "T": T, "k_lab": l, "k": K, "sigma": SIGMA, "reps": reps}
    for name, fn in (("poisson", pkg.poisson_learning), ("laplace_trials", pkg.laplace_learning_trials)):
        res = fn(Xt, It, Yt, k=K, targets=tt)
        torch.cuda.synchronize()
        info = last_eval_info()
        out[name] = {"accuracy": float(res.correct.sum()) / (T * (n - l)),
                     "info": {kk: info[kk] for kk in ("status", "rounds", "cg_iters_first", "cg_iters_correction", "round_iters", "resid")},
                     "resid_per_trial_max": max(info["resid_per_trial"]),
                     "ms_call": median_ms(lambda: fn(Xt, It, Yt, k=K, targets=tt), reps),
                     "stages": profiled(lambda: fn(Xt, It, Yt, k=K, targets=tt))}
        del res
    print(json.dumps({kk: ({a: b for a, b in v.items() if a != "stages"} if isinstance(v, dict) else v) for kk, v in out.items()}),
          flush=True)
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="")
    ap.add_argument("--reps", type=int, default=7)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("poisson_eval_bench.py needs a CUDA device")
    torch.cuda.set_device(0)
    res = {"gpu": gpu_identity(), "reps": a.reps, "cases": [case(*s, a.reps) for s in SHAPES]}
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
