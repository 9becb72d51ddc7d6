"""Laplace-learning evaluation on the device: the reference's ``utils.laplace`` (utils.py:570-593), as ``test_GL_NP``
(utils.py:637-660) runs it on base + train + test features, in one call on features that are already on the GPU.

    res = laplace_learning(features, label_matrix, k=50, epsilon='auto', tau=0.0, tol=1e-10, targets=None)
    res.pred      (m, l) float64   harmonic extension on the unlabeled rows (m = n - k_lab)
    res.labels    (m,) int64       argmax, first maximal column on ties
    res.correct   0-dim int64      rows with targets >= 0 and labels == targets (None without targets)

Same graph as the layer (kNN -> union graph -> weights, with this k); the system L_uu + tau I is solved in fp32 and refined
in fp64 until every class column meets the reference's stop rule ||M (b - A x)||_2 <= tol with M = diag(A + 1e-10)^(-1/2)
(see gll_laplace_eval in include/gll_b200.h, including the row-sum degree).  Everything is enqueued on the current stream:
no host sync, no host round trip, so the call can be captured into a CUDA graph.  Status ('max iter reached' when tol is
unmet, epsilon ~ 0) goes through the same deferred check as the layer.  Knob: GLL_B200_CG_MAXIT (iterations per CG solve).

    res = laplace_learning_batched(features, label_matrix, k=50, epsilon='auto', tau=0.0, tol=1e-10, targets=None)

B independent graphs of the same shape in one call (features (B, n, d), label_matrix (B, k_lab, l), targets (B, m)); pred
(B, m, l), labels (B, m), correct (B,).  Every graph meets the stop rule on its own; the solver's step lengths are shared by
the graphs, so pred matches per-graph laplace_learning calls to solver accuracy (bit for bit at B = 1).  See
gll_laplace_eval_batched in include/gll_b200.h.

    res = laplace_learning_trials(features, train_idx, label_matrix, k=50, epsilon='auto', tau=0.0, tol=1e-10, targets=None)

T labeled sets on ONE set of features (n, d) in any row order: train_idx (T, k_lab) lists the labeled rows of each trial,
label_matrix (T, k_lab, l) their labels, targets (n,); pred (T, n, l), labels (T, n), correct (T,) over the rows not labeled in
that trial.  The graph is built once; all T l class columns are solved against it with each trial's labeled rows masked out of
its own columns, every column with its own step lengths.  A trial with an index outside [0, n) or a repeated index is invalid:
pred NaN, labels -1, correct -1 and a warning; the other trials are unaffected.  See gll_laplace_eval_trials in
include/gll_b200.h.
"""
from __future__ import annotations

from typing import NamedTuple, Optional

import numpy as np
import torch

from . import _lib
from .GLL import _bytes, _cg_maxit, _check_status, _require_cuda, _stream_ptr, as_features, decode_info, parse_epsilon
from ._lib import lib

__all__ = ["laplace_learning", "laplace_learning_batched", "laplace_learning_trials", "LaplaceResult", "last_eval_info"]


class LaplaceResult(NamedTuple):
    pred: torch.Tensor
    labels: torch.Tensor
    correct: Optional[torch.Tensor]


_last_info: Optional[torch.Tensor] = None
_last_resid: Optional[tuple] = None  # (key, per-group residuals) of the last call when it was batched or a trials call


def _check_args(n, d, k_lab, l, k, epsilon, tol, total_rows, rows_name):
    """The size, epsilon and tol checks the entry points share; returns (eps_auto, eps_fixed)."""
    if not (0 < k_lab < n):
        raise ValueError(f"need 0 < k_lab < n (k_lab={k_lab}, n={n}); labeled rows come first (GLL.py:11)")
    if l < 1 or d < 1:
        raise ValueError("need at least one class column and one feature")
    if not (2 <= k <= 64) or k > n or (k > 33 and total_rows < 256):
        raise ValueError(f"k must be in [2, 64] and <= n, with {rows_name} >= 256 when k > 33 (k={k}, n={n})")
    eps = parse_epsilon(epsilon)
    if not tol > 0:
        raise ValueError("tol must be > 0")
    return eps


def _run(name, features, label_matrix, targets, lead, ws_sizes, pred_shape, groups, eps, tau, tol, resid_key=None):
    """Converts the inputs, allocates the outputs and the workspace, runs gll_<name> on the current stream and records its info
    for last_eval_info().  lead(X, Y) gives the arguments in front of eps_auto, with X and Y the converted features and labels;
    groups is the shape of correct and of the residuals reported under resid_key."""
    _require_cuda(features, "features")
    dev = features.device
    Xc = as_features(features)
    Y = label_matrix.detach().to(device=dev, dtype=torch.float32).contiguous()
    tg = None if targets is None else targets.detach().to(device=dev, dtype=torch.int64).contiguous()
    with torch.cuda.device(dev):
        ws_bytes = getattr(lib, f"gll_{name}_workspace_bytes")(*ws_sizes)
        ws = _bytes(ws_bytes, dev)
        pred = torch.empty(pred_shape, dtype=torch.float64, device=dev)
        labels = torch.empty(pred_shape[:-1], dtype=torch.int64, device=dev)
        correct = None if tg is None else torch.empty(groups, dtype=torch.int64, device=dev)
        resid = None if resid_key is None else torch.empty(groups, dtype=torch.float64, device=dev)
        info = torch.empty(_lib.INFO_WORDS, dtype=torch.int32, device=dev)
        outs = [None if t is None else t.data_ptr() for t in (pred, labels, tg, correct)] + ([] if resid is None else [resid.data_ptr()])
        rc = getattr(lib, f"gll_{name}")(*lead(Xc.data_ptr(), Y.data_ptr()), *eps, float(tau), float(tol), _cg_maxit(), *outs,
                                         info.data_ptr(), ws.data_ptr(), ws_bytes, _stream_ptr(dev))
    _lib.check(rc, f"gll_{name}")
    global _last_info, _last_resid
    _last_info, _last_resid = info, None if resid is None else (resid_key, resid)
    _check_status(info, "Laplace-learning")
    return LaplaceResult(pred, labels, correct)


def laplace_learning(features: torch.Tensor, label_matrix: torch.Tensor, k: int = 50, epsilon="auto", tau: float = 0.0,
                     tol: float = 1e-10, targets: Optional[torch.Tensor] = None) -> LaplaceResult:
    """features (n, d) CUDA tensor with the k_lab labeled rows FIRST (GLL.py:11); label_matrix (k_lab, l) one-hot float32 or
    int64; targets (m,) int64 or None, a negative target is not counted."""
    if features.dim() != 2:
        raise ValueError("features must be (n, d)")
    if label_matrix.dim() != 2:
        raise ValueError("label_matrix must be (k_lab, l)")
    n, d = features.shape
    k_lab, l = label_matrix.shape
    k = int(k)
    eps = _check_args(n, d, k_lab, l, k, epsilon, tol, n, "n")
    m = n - k_lab
    if targets is not None and tuple(targets.shape) != (m,):
        raise ValueError(f"targets must be ({m},), got {tuple(targets.shape)}")
    return _run("laplace_eval", features, label_matrix, targets, lambda X, Y: (X, Y, n, d, k, l, k_lab), (n, d, k, l, k_lab), (m, l),
                (), eps, tau, tol)


def laplace_learning_batched(features: torch.Tensor, label_matrix: torch.Tensor, k: int = 50, epsilon="auto", tau: float = 0.0,
                             tol: float = 1e-10, targets: Optional[torch.Tensor] = None) -> LaplaceResult:
    """laplace_learning over B independent graphs of the same shape.  features (B, n, d) CUDA tensor, each graph's k_lab labeled
    rows FIRST; label_matrix (B, k_lab, l) one-hot float32 or int64; targets (B, m) int64 or None, a negative target is not
    counted.  Returns pred (B, m, l) float64, labels (B, m) int64 and correct (B,) int64 (None without targets)."""
    if features.dim() != 3:
        raise ValueError("features must be (B, n, d)")
    if label_matrix.dim() != 3:
        raise ValueError("label_matrix must be (B, k_lab, l)")
    B, n, d = features.shape
    if B < 1 or label_matrix.shape[0] != B:
        raise ValueError(f"label_matrix must be (B, k_lab, l) with B = {B} >= 1, got {tuple(label_matrix.shape)}")
    if B * n >= 2 ** 31:
        raise ValueError(f"B n must be < 2^31 (B={B}, n={n})")
    _, k_lab, l = label_matrix.shape
    k = int(k)
    eps = _check_args(n, d, k_lab, l, k, epsilon, tol, B * n, "B n")
    m = n - k_lab
    if targets is not None and tuple(targets.shape) != (B, m):
        raise ValueError(f"targets must be ({B}, {m}), got {tuple(targets.shape)}")
    return _run("laplace_eval_batched", features, label_matrix, targets, lambda X, Y: (X, Y, B, n, d, k, l, k_lab),
                (B, n, d, k, l, k_lab), (B, m, l), (B,), eps, tau, tol, "resid_per_graph")


def laplace_learning_trials(features: torch.Tensor, train_idx: torch.Tensor, label_matrix: torch.Tensor, k: int = 50, epsilon="auto",
                            tau: float = 0.0, tol: float = 1e-10, targets: Optional[torch.Tensor] = None) -> LaplaceResult:
    """T labeled sets on one graph.  features (n, d) CUDA tensor in any row order; train_idx (T, k_lab) int64 or int32, the labeled
    rows of trial t (read on the device: no host copy); label_matrix (T, k_lab, l) one-hot float32 or int64, row s of trial t
    labels row train_idx[t, s]; targets (n,) int64 or None, a negative target is not counted.  Returns pred (T, n, l) float64,
    labels (T, n) int64 and correct (T,) int64 (None without targets), counting the rows not labeled in that trial.  A labeled
    row gets its label row and that row's argmax.  Trial t equals laplace_learning on features[perm_t], perm_t = [train_idx[t],
    the other rows in natural order], on its unlabeled rows; the graph is built once in natural order, so on exact distance ties
    the kNN tie-break follows natural order rather than perm_t."""
    if features.dim() != 2:
        raise ValueError("features must be (n, d)")
    if train_idx.dim() != 2:
        raise ValueError("train_idx must be (T, k_lab)")
    if train_idx.dtype not in (torch.int64, torch.int32):
        raise ValueError(f"train_idx must be int64 or int32, got {train_idx.dtype}")
    if label_matrix.dim() != 3:
        raise ValueError("label_matrix must be (T, k_lab, l)")
    n, d = features.shape
    T, k_lab = train_idx.shape
    if T < 1 or tuple(label_matrix.shape[:2]) != (T, k_lab):
        raise ValueError(f"label_matrix must be (T, k_lab, l) = ({T}, {k_lab}, l) with T >= 1, got {tuple(label_matrix.shape)}")
    l = label_matrix.shape[2]
    k = int(k)
    eps = _check_args(n, d, k_lab, l, k, epsilon, tol, n, "n")
    lpad = lib.gll_padded_classes(l)
    if n * T * lpad >= 2 ** 31:
        raise ValueError(f"n T lpad must be < 2^31 (n={n}, T={T}, lpad={lpad})")
    if T * l > 65535 * 32:  # the refinement grid's column chunks (gridDim.y)
        raise ValueError(f"T l must be <= 2097120 (T={T}, l={l})")
    if targets is not None and tuple(targets.shape) != (n,):
        raise ValueError(f"targets must be ({n},), got {tuple(targets.shape)}")
    _require_cuda(features, "features")  # before train_idx is copied anywhere
    idx = train_idx.detach().to(device=features.device).contiguous()
    return _run("laplace_eval_trials", features, label_matrix, targets,
                lambda X, Y: (X, n, d, k, idx.data_ptr(), int(idx.dtype == torch.int64), Y, T, k_lab, l), (n, d, k, l, T, k_lab),
                (T, n, l), (T,), eps, tau, tol, "resid_per_trial")


def last_eval_info() -> dict:
    """Device status block of the most recent laplace_learning, laplace_learning_batched or laplace_learning_trials call
    (synchronises).  Keys follow GLL_INFO_* in include/gll_b200.h; after a batched call the residuals are the maximum over graphs,
    the iteration counts those of the whole batch, and resid_per_graph lists each graph's largest column norm of the last round.
    After a trials call the same holds over the valid trials, and resid_per_trial lists each trial's (NaN for an invalid one)."""
    if _last_info is None:
        return {}
    v = _last_info.cpu().numpy()
    f = v.view(np.float32)
    u = v.view(np.uint32)
    round_iters = [int((u[_lib.INFO_LAPLACE_ROUND_ITERS + r // 2] >> (16 * (r % 2))) & 0xFFFF) for r in range(4)]
    return dict(decode_info(v), cg_iters_first=int(v[_lib.INFO_CG_ITERS_FWD]), rounds=int(v[_lib.INFO_LAPLACE_ROUNDS]),
                cg_iters_correction=int(v[_lib.INFO_LAPLACE_CG_ITERS]), round_iters=round_iters, resid_first=float(f[_lib.INFO_LAPLACE_RESID0]),
                resid=float(f[_lib.INFO_LAPLACE_RESID]),
                **({} if _last_resid is None else {_last_resid[0]: [float(x) for x in _last_resid[1].cpu().numpy()]}))
