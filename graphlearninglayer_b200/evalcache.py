"""Evaluation loops over a FIXED base set (SURVEY.md 8f-4).

The reference's ``test_network`` (utils.py:596-621) calls the layer once per test batch on ``[base; batch]`` with the
model in ``eval()`` mode: the base rows and their labels are the same in every call, only the batch rows change.
``BaseSetEvaluator`` does the base-base part of the kNN search once and per batch searches only the batch rows against
all columns and the base rows against the batch columns; everything downstream (exact re-rank, completeness proof, graph,
weights, CG) is the layer's own forward, so the predictions are bit-identical to
``LaplaceLearningSparseHard.apply(torch.cat((base, batch)), label_matrix, tau, epsilon)``.

    ev = BaseSetEvaluator(base_features, label_matrix, tau=opt.temp, epsilon=opt.epsilon)
    for images, labels in test_loader:                      # utils.py:607
        _, feat = model(images.cuda())
        pred = ev(feat)                                     # (len(batch), n_classes) float64, like the layer's output
        correct += (pred.argmax(1) == labels.cuda()).sum()

Forward only (evaluation); CUDA tensors only; needs at least 256 base rows.
"""
from __future__ import annotations

import torch

from . import _lib
from ._lib import lib
from .GLL import K_NEIGHBOURS, GraphStages, _bytes, _cg_maxit, _cg_tol, _require_cuda, _stream_ptr, as_features, parse_epsilon, pred_dtype


def _uu_hint(k: int, m: int, n: int) -> float:
    """gll_forward's sparsity hint, uu_degree_hint in csrc/api.cu, in the same float32 arithmetic: 1.2f * (k - 1) * m / n."""
    import numpy as np

    return float(np.float32(1.2) * np.float32(k - 1) * np.float32(m) / np.float32(n))


class BaseSetEvaluator:
    def __init__(self, base_features: torch.Tensor, label_matrix: torch.Tensor, tau: float = 0.0, epsilon="auto",
                 k: int = K_NEIGHBOURS):
        _require_cuda(base_features, "base features")
        parse_epsilon(epsilon)
        self.base = as_features(base_features)
        self.Y = label_matrix.detach().to(device=self.base.device, dtype=torch.float32).contiguous()
        self.n_base, self.d = self.base.shape
        if self.Y.shape[0] != self.n_base:
            raise ValueError("label_matrix must have one row per base row (labeled rows first, GLL.py:11)")
        if self.n_base < 256:
            raise ValueError("the base-set cache needs at least 256 base rows")
        self.l = self.Y.shape[1]
        self.tau, self.epsilon, self.k = float(tau), epsilon, int(k)
        dev = self.base.device
        with torch.cuda.device(dev):
            self.cache = _bytes(lib.gll_base_cache_bytes(self.n_base), dev)
            wsb = lib.gll_base_cache_workspace_bytes(self.n_base, self.d)
            ws = _bytes(wsb, dev)
            _lib.check(lib.gll_base_cache_build(self.base.data_ptr(), self.n_base, self.d, self.cache.data_ptr(), ws.data_ptr(), wsb,
                                                _stream_ptr(dev)), "gll_base_cache_build")
        self.info = None
        self.knn_idx = None

    def __call__(self, batch_features: torch.Tensor) -> torch.Tensor:
        """Prediction for the batch rows: what the layer returns for [base; batch] (GLL.py:53,73)."""
        _require_cuda(batch_features, "batch features")
        dev = self.base.device
        b = batch_features.detach().to(device=dev, dtype=torch.float32)
        if b.dim() != 2 or b.shape[1] != self.d:
            raise ValueError(f"batch features must be (m, {self.d})")
        X = torch.cat((self.base, b), dim=0)
        return self._forward(X)

    def _forward(self, X: torch.Tensor) -> torch.Tensor:
        dev = X.device
        n, d, k, l, k_lab = X.shape[0], self.d, self.k, self.l, self.n_base
        m = n - k_lab
        s = _stream_ptr(dev)
        with torch.cuda.device(dev):
            info = torch.zeros(_lib.INFO_WORDS, dtype=torch.int32, device=dev)
            knn_idx = torch.empty((n, k), dtype=torch.int32, device=dev)
            knn_dist = torch.empty((n, k), dtype=torch.float32, device=dev)
            wsb = max(lib.gll_knn_cached_workspace_bytes(n, d, k, k_lab), lib.gll_graph_workspace_bytes(n, k),
                      lib.gll_weights_workspace_bytes(n, k), lib.gll_cg_workspace_bytes(m, l))
            ws = _bytes(wsb, dev)
            _lib.check(lib.gll_knn_cached(X.data_ptr(), n, d, k, k_lab, self.cache.data_ptr(), knn_idx.data_ptr(), knn_dist.data_ptr(),
                                          info.data_ptr(), ws.data_ptr(), wsb, s), "gll_knn_cached")
            g = GraphStages(knn_idx, knn_dist, self.Y, n, self.tau, self.epsilon, info, ws)
            u = g.ut[k_lab:]
            # the same sparsity hint as gll_forward passes, so that the same solver kernel runs: bit-identical predictions
            _lib.check(lib.gll_cg_solve_hint(g.uu_ptr.data_ptr(), g.uu_col.data_ptr(), g.uu_val.data_ptr(), g.diag.data_ptr(),
                                             g.rhs.data_ptr(), m, l, _cg_tol(), _cg_maxit(), u.data_ptr(),
                                             info[_lib.INFO_CG_ITERS_FWD:].data_ptr(), info[_lib.INFO_CG_RESID_FWD:].data_ptr(),
                                             info[_lib.INFO_STATUS:].data_ptr(), ws.data_ptr(), wsb, s, _uu_hint(k, m, n)),
                       "gll_cg_solve")
            pred = torch.empty((m, l), dtype=pred_dtype(), device=dev)
            _lib.check(lib.gll_unpack_pred(u.data_ptr(), m, l, pred.data_ptr(), int(pred.dtype == torch.float64), s), "gll_unpack_pred")
        self.info, self.knn_idx, self.knn_dist = info, knn_idx, knn_dist
        return pred
