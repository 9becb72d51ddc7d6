"""Host side of the B200 GraphLearningLayer hot path: the same three names the reference module exports
(``/root/reference/GLL.py``; ``utils.py:25`` imports all three), backed by libgll_b200.so.

    LaplaceLearningSparseHard.apply(X, label_matrix, tau=0, epsilon='auto')   GLL.py:10-177
    LaplaceLearningSparseHardBatched.apply(X, label_matrix, tau, epsilon)    B independent graphs, X (B, n, d)
    knn_sym_dist(data, k=25, epsilon='auto')                                  GLL.py:180-244
    stable_conjgrad(A, b, x0=None, max_iter=1e5, tol=1e-10)                   GLL.py:247-276

PyTorch is plumbing here (device memory, the current CUDA stream, autograd registration); every number is
produced by the sm_100a kernels in csrc/.  There is no CPU path: CPU tensors raise.

Knobs (environment, read at call time):
    GLL_B200_CG_TOL       absolute 2-norm residual per class column (default 1e-7; forward), and relative to the
                          largest column norm of grad_output for the adjoint solve
    GLL_B200_CG_MAXIT     default 5000
    GLL_B200_PRED_DTYPE   'float64' (default: the reference returns float64, GLL.py:66) or 'float32'
    GLL_B200_CHECK        '1': read the device status word after every call (one host sync) and warn like the
                          reference does (GLL.py:240-241 epsilon ~ 0; GLL.py:273-274 'max iter reached').
                          Default: DEFERRED -- the status word is copied to pinned memory behind the call and looked at
                          when a later call finds the copy complete (no host sync; the warning comes one call late).
                          '0': never (also skipped while a CUDA graph is being captured).
"""
from __future__ import annotations

import os
import warnings
from typing import Optional, Tuple, Union

import numpy as np
import torch

from . import _lib
from ._lib import lib

K_NEIGHBOURS = 25  # hard-coded in the reference at GLL.py:27

__all__ = ["LaplaceLearningSparseHard", "LaplaceLearningSparseHardNormalized", "LaplaceLearningSparseHardBatched", "knn_sym_dist", "stable_conjgrad", "last_info"]


def _env_float(name: str, default: float) -> float:
    v = os.environ.get(name)
    return float(v) if v else default


def _cg_tol() -> float:
    return _env_float("GLL_B200_CG_TOL", 1e-7)


def _cg_maxit() -> int:
    return int(_env_float("GLL_B200_CG_MAXIT", 5000))


def _stream_ptr(device: torch.device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def _bytes(nbytes: int, device: torch.device) -> torch.Tensor:
    # PyTorch's caching allocator owns every byte the library touches (the library never allocates).
    return torch.empty(int(nbytes), dtype=torch.uint8, device=device)


def _require_cuda(t: torch.Tensor, what: str) -> None:
    if not t.is_cuda:
        raise RuntimeError(f"graphlearninglayer_b200: {what} must be a CUDA tensor (this build has no CPU path; "
                           "the reference /root/reference/GLL.py is the CPU implementation)")


def parse_epsilon(epsilon) -> Tuple[int, float]:
    """(eps_auto, eps_fixed) of the C ABI: 'auto' (GLL.py:205) or a fixed bandwidth (GLL.py:226)."""
    if isinstance(epsilon, str):
        if epsilon != "auto":
            raise ValueError("epsilon must be a float or 'auto'")
        return 1, 0.0
    return 0, float(epsilon)


def pred_dtype() -> torch.dtype:
    """dtype of the predictions (GLL_B200_PRED_DTYPE; float64 like the reference, GLL.py:66)."""
    return torch.float32 if os.environ.get("GLL_B200_PRED_DTYPE", "float64") == "float32" else torch.float64


def as_features(X: torch.Tensor) -> torch.Tensor:
    """X detached as the float32, contiguous matrix the kernels read (no copy when it already is one)."""
    X = X.detach()
    if X.dtype != torch.float32:
        X = X.float()
    return X.contiguous()


def decode_info(v: np.ndarray) -> dict:
    """The keys every status block reports, from its host copy (int32 words, GLL_INFO_* in include/gll_b200.h)."""
    return dict(status=int(v[_lib.INFO_STATUS]), nnz=int(v[_lib.INFO_NNZ]), nnz_uu=int(v[_lib.INFO_NNZ_UU]),
                knn_fallback_rows=int(v[_lib.INFO_KNN_FALLBACK_ROWS]))


_last_info: Optional[torch.Tensor] = None


def last_info() -> dict:
    """Device status block of the most recent forward/backward (synchronises).  Keys follow GLL_INFO_* in
    include/gll_b200.h."""
    if _last_info is None:
        return {}
    v = _last_info.cpu().numpy()
    f = v.view(np.float32)
    return dict(decode_info(v), cg_iters_fwd=int(v[_lib.INFO_CG_ITERS_FWD]), cg_iters_bwd=int(v[_lib.INFO_CG_ITERS_BWD]),
                cg_resid_fwd=float(f[_lib.INFO_CG_RESID_FWD]), cg_resid_bwd=float(f[_lib.INFO_CG_RESID_BWD]))


def _warn_from_status(info: torch.Tensor, where: str) -> None:
    st = int(info[_lib.INFO_STATUS].item())
    if st & _lib.STATUS_EPS_TINY:
        warnings.warn("Epsilon in KNN is very close to zero.")  # GLL.py:240-241
    if st & _lib.STATUS_CG_NOT_CONVERGED:
        warnings.warn(f"max iter reached in the {where} CG solve")  # GLL.py:273-274 prints
    if st & _lib.STATUS_NONFINITE:
        warnings.warn(f"non-finite values in the {where} solve (singular L_uu or epsilon = 0)")
    if st & _lib.STATUS_BAD_INDEX:
        warnings.warn(f"{where}: a trial's labeled-row indices are out of range or repeated; that trial is invalid (NaN / -1)")


class _DeferredStatus:
    """One pinned slot per device: the previous call's status word, copied asynchronously; read when its event has completed."""
    slots: dict = {}

    def __init__(self):
        self.host = torch.zeros(_lib.INFO_WORDS, dtype=torch.int32).pin_memory()
        self.event: Optional[torch.cuda.Event] = None
        self.where = ""


def _check_status(info: torch.Tensor, where: str) -> None:
    mode = os.environ.get("GLL_B200_CHECK", "")
    if mode == "1":
        _warn_from_status(info, where)
        return
    if mode == "0" or torch.cuda.is_current_stream_capturing():
        return
    key = (info.device.index, torch.cuda.current_stream(info.device).cuda_stream)
    slot = _DeferredStatus.slots.get(key)
    if slot is None:
        slot = _DeferredStatus.slots[key] = _DeferredStatus()
    if slot.event is not None:
        if not slot.event.query():
            return  # the previous copy has not landed yet: keep it, look again at the next call
        _warn_from_status(slot.host, slot.where)
    slot.host.copy_(info, non_blocking=True)
    slot.where = where
    slot.event = torch.cuda.Event()
    slot.event.record(torch.cuda.current_stream(info.device))


class _State:
    """Buffers kept between forward and backward (replaces the scipy objects on ctx, GLL.py:69-70)."""
    __slots__ = ("buf", "layout", "n", "d", "k", "l", "k_lab", "eps_auto")

    def view(self, name: str, dtype: torch.dtype, count: int) -> torch.Tensor:
        off = getattr(self.layout, name)
        item = torch.empty((), dtype=dtype).element_size()
        return self.buf[off:off + count * item].view(dtype)


def _forward_impl(X: torch.Tensor, label_matrix: torch.Tensor, tau, epsilon, k: int = K_NEIGHBOURS):
    _require_cuda(X, "features")
    if X.dim() != 2:
        raise ValueError("features must be (n, d)")
    dev = X.device
    Xc = as_features(X)
    Y = label_matrix.detach().to(device=dev, dtype=torch.float32).contiguous()  # int64 one-hot allowed (t_a_a.py:545)
    if Y.dim() != 2:
        raise ValueError("label_matrix must be (k_lab, l)")
    n, d = Xc.shape
    k_lab, l = Y.shape
    if not (0 < k_lab < n):
        raise ValueError(f"need 0 < k_lab < n (k_lab={k_lab}, n={n}); labeled rows come first (GLL.py:11)")
    if n < k:
        raise ValueError(f"need at least k={k} nodes, got {n}")
    eps_auto, eps_fixed = parse_epsilon(epsilon)
    m = n - k_lab
    st = _State()
    st.layout = _lib.state_layout(n, k, l, k_lab)
    st.n, st.d, st.k, st.l, st.k_lab, st.eps_auto = n, d, k, l, k_lab, eps_auto
    with torch.cuda.device(dev):
        st.buf = _bytes(st.layout.total, dev)
        ws_bytes = lib.gll_workspace_bytes(n, d, k, l, k_lab)
        ws = _bytes(ws_bytes, dev)
        pred = torch.empty((m, l), dtype=pred_dtype(), device=dev)
        rc = lib.gll_forward(Xc.data_ptr(), Y.data_ptr(), n, d, k, l, k_lab, eps_auto, eps_fixed, float(tau), _cg_tol(),
                             _cg_maxit(), st.buf.data_ptr(), pred.data_ptr(), int(pred.dtype == torch.float64), ws.data_ptr(),
                             ws_bytes, _stream_ptr(dev))
    _lib.check(rc, "gll_forward")
    global _last_info
    _last_info = st.view("info", torch.int32, _lib.INFO_WORDS)
    _check_status(_last_info, "forward")
    return pred, st, Xc


def _backward_impl(st: _State, Xc: torch.Tensor, grad_output: torch.Tensor, scale: Optional[torch.Tensor] = None) -> torch.Tensor:
    """dX for d loss / d Pred = grad_output (times the 0-dim device tensor `scale`, if given: read by the kernel, no host sync)."""
    dev = Xc.device
    g = grad_output.detach().to(device=dev)
    if g.dtype not in (torch.float32, torch.float64):
        g = g.float()
    g = g.contiguous()
    m = st.n - st.k_lab
    if tuple(g.shape) != (m, st.l):
        raise ValueError(f"grad_output must be ({m}, {st.l}), got {tuple(g.shape)}")
    with torch.cuda.device(dev):
        dX = torch.empty((st.n, st.d), dtype=torch.float32, device=dev)
        ws_bytes = lib.gll_workspace_bytes(st.n, st.d, st.k, st.l, st.k_lab)
        ws = _bytes(ws_bytes, dev)
        # negative tolerance = relative to the largest column norm of the right-hand side (see gll_cg_solve)
        sc = None
        if scale is not None:
            sc = scale.detach().to(device=dev)
            if sc.dtype not in (torch.float32, torch.float64):
                sc = sc.float()
            sc = sc.reshape(1).contiguous()
        rc = lib.gll_backward_scaled(Xc.data_ptr(), g.data_ptr(), int(g.dtype == torch.float64),
                                     sc.data_ptr() if sc is not None else None, int(sc is not None and sc.dtype == torch.float64),
                                     st.n, st.d, st.k, st.l, st.k_lab, st.eps_auto, -_cg_tol(), _cg_maxit(), st.buf.data_ptr(),
                                     dX.data_ptr(), ws.data_ptr(), ws_bytes, _stream_ptr(dev))
    _lib.check(rc, "gll_backward")
    _check_status(st.view("info", torch.int32, _lib.INFO_WORDS), "adjoint")
    return dX


class LaplaceLearningSparseHard(torch.autograd.Function):
    """Drop-in for ``GLL.LaplaceLearningSparseHard`` (GLL.py:10-177).

    forward(X, label_matrix, tau=0, epsilon='auto'): X is (n, d) with the k_lab labeled ("base") rows FIRST
    (GLL.py:11,32-38), label_matrix is (k_lab, l) one-hot (float32 or int64); returns the (n-k_lab, l) harmonic
    extension, float64 like the reference (GLL.py:66,73), as a fresh tensor callers may mutate (adversarial.py:691).
    backward returns (dX, None, None, None) with dX (n, d) in X's dtype, non-zero on base rows too (GLL.py:159,177).
    """

    @staticmethod
    def forward(ctx, X, label_matrix, tau=0, epsilon="auto"):
        pred, st, Xc = _forward_impl(X, label_matrix, tau, epsilon)
        ctx.gll_state = st
        ctx.x_dtype = X.dtype
        ctx.save_for_backward(Xc)
        ctx.set_materialize_grads(True)
        return pred

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, grad_output):
        (Xc,) = ctx.saved_tensors
        dX = _backward_impl(ctx.gll_state, Xc, grad_output)
        if dX.dtype != ctx.x_dtype:
            dX = dX.to(ctx.x_dtype)
        return dX, None, None, None


class LaplaceLearningSparseHardNormalized(torch.autograd.Function):
    """`LaplaceLearningSparseHard.apply(F.normalize(feat, dim=1), label_matrix, tau, epsilon)` in one autograd node
    (SURVEY 8f-3): every caller normalises the encoder output right before the layer (networks/BuildNet.py:101,
    FullySup.py:122,156).  The rows are normalised by one kernel and the normalisation's backward,
    d feat = (d xn - xn <xn, d xn>) / |feat|, by another -- instead of PyTorch's ~10 small kernels for the pair."""

    @staticmethod
    def forward(ctx, feat, label_matrix, tau=0, epsilon="auto"):
        _require_cuda(feat, "features")
        f = as_features(feat)
        n, d = f.shape
        xn = torch.empty_like(f)
        inv = torch.empty(n, dtype=torch.float32, device=f.device)
        with torch.cuda.device(f.device):
            _lib.check(lib.gll_normalize_rows(f.data_ptr(), n, d, 1e-12, xn.data_ptr(), inv.data_ptr(), _stream_ptr(f.device)),
                       "gll_normalize_rows")
        pred, st, _ = _forward_impl(xn, label_matrix, tau, epsilon)
        ctx.gll_state = st
        ctx.x_dtype = feat.dtype
        ctx.save_for_backward(xn, inv)
        ctx.set_materialize_grads(True)
        return pred

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, grad_output):
        xn, inv = ctx.saved_tensors
        dxn = _backward_impl(ctx.gll_state, xn, grad_output)
        dx = torch.empty_like(dxn)
        n, d = xn.shape
        with torch.cuda.device(xn.device):
            _lib.check(lib.gll_normalize_rows_backward(xn.data_ptr(), inv.data_ptr(), dxn.data_ptr(), n, d, dx.data_ptr(),
                                                       _stream_ptr(xn.device)), "gll_normalize_rows_backward")
        if dx.dtype != ctx.x_dtype:
            dx = dx.to(ctx.x_dtype)
        return dx, None, None, None


def labeled_first(X: torch.Tensor, k_lab: int) -> torch.Tensor:
    """(B, n, d) -> (B n, d) in the batched layer's row order: all graphs' labeled rows, then all graphs' unlabeled rows."""
    d = X.shape[2]
    return torch.cat((X[:, :k_lab].reshape(-1, d), X[:, k_lab:].reshape(-1, d)))


def natural_order(Xg: torch.Tensor, B: int, k_lab: int) -> torch.Tensor:
    """Inverse of labeled_first: (B n, d) -> (B, n, d)."""
    d = Xg.shape[1]
    m = Xg.shape[0] // B - k_lab
    return torch.cat((Xg[:B * k_lab].reshape(B, k_lab, d), Xg[B * k_lab:].reshape(B, m, d)), dim=1)


def _batched_forward_impl(X: torch.Tensor, label_matrix: torch.Tensor, tau, epsilon, k: int = K_NEIGHBOURS):
    if X.dim() != 3:
        raise ValueError("features must be (B, n, d)")
    B, n, d = X.shape
    if label_matrix.dim() != 3 or label_matrix.shape[0] != B:
        raise ValueError(f"label_matrix must be (B, k_lab, l) with B = {B}, got {tuple(label_matrix.shape)}")
    _, k_lab, l = label_matrix.shape
    if k_lab < 1 or n - k_lab < 1 or l < 1 or d < 1:
        raise ValueError(f"need 1 <= k_lab < n, l >= 1 and d >= 1 (k_lab={k_lab}, n={n}, l={l}, d={d}); labeled rows come first")
    if n < k:
        raise ValueError(f"every graph needs at least k={k} nodes, got n={n}")
    eps_auto, eps_fixed = parse_epsilon(epsilon)
    _require_cuda(X, "features")
    dev = X.device
    Xc = as_features(X)
    Y = label_matrix.detach().to(device=dev, dtype=torch.float32).contiguous()  # int64 one-hot allowed
    st = _State()
    st.layout = _lib.state_layout(B * n, k, l, B * k_lab)
    st.n, st.d, st.k, st.l, st.k_lab, st.eps_auto = B * n, d, k, l, B * k_lab, eps_auto
    with torch.cuda.device(dev):
        st.buf = _bytes(st.layout.total, dev)
        ws_bytes = lib.gll_batched_workspace_bytes(B, n, d, k, l, k_lab)
        ws = _bytes(ws_bytes, dev)
        pred = torch.empty((B, n - k_lab, l), dtype=pred_dtype(), device=dev)
        rc = lib.gll_forward_batched(Xc.data_ptr(), Y.data_ptr(), B, n, d, k, l, k_lab, eps_auto, eps_fixed, float(tau), _cg_tol(),
                                     _cg_maxit(), st.buf.data_ptr(), pred.data_ptr(), int(pred.dtype == torch.float64), ws.data_ptr(),
                                     ws_bytes, _stream_ptr(dev))
        _lib.check(rc, "gll_forward_batched")
        Xg = labeled_first(Xc, k_lab)  # the backward's rows, in the order of the block-diagonal graph
    global _last_info
    _last_info = st.view("info", torch.int32, _lib.INFO_WORDS)
    _check_status(_last_info, "forward")
    return pred, st, Xg


class LaplaceLearningSparseHardBatched(torch.autograd.Function):
    """B independent graphs of the same shape in one call: ``LaplaceLearningSparseHard`` applied to each ``X[b]`` with
    ``label_matrix[b]``.

    forward(X, label_matrix, tau=0, epsilon='auto'): X is (B, n, d) with each graph's k_lab labeled rows first,
    label_matrix (B, k_lab, l) one-hot (float32 or int64); returns (B, n - k_lab, l) in the layer's prediction dtype.
    backward gives dX (B, n, d) in X's dtype.

    The B graphs are solved as one block-diagonal graph: the kNN search never crosses graphs, and the kNN lists, the graph,
    epsilon, the weights and the degrees are bit-identical to per-graph calls.  One multi-right-hand-side CG solves all B
    systems, so its step lengths are shared across graphs and each class column stops when its residual over all graphs
    meets the tolerance (which bounds every graph's residual): predictions and gradients agree with per-graph calls to the
    solver tolerance, not bit for bit when B > 1, and iteration counts in last_info() are the batch's.  B = 1 is
    bit-identical to LaplaceLearningSparseHard.
    """

    @staticmethod
    def forward(ctx, X, label_matrix, tau=0, epsilon="auto"):
        pred, st, Xg = _batched_forward_impl(X, label_matrix, tau, epsilon)
        ctx.gll_state = st
        ctx.x_dtype = X.dtype
        ctx.batch = (X.shape[0], label_matrix.shape[1])
        ctx.save_for_backward(Xg)
        ctx.set_materialize_grads(True)
        return pred

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, grad_output):
        (Xg,) = ctx.saved_tensors
        B, k_lab = ctx.batch
        dXg = _backward_impl(ctx.gll_state, Xg, grad_output.reshape(-1, grad_output.shape[-1]))
        dX = natural_order(dXg, B, k_lab)
        if dX.dtype != ctx.x_dtype:
            dX = dX.to(ctx.x_dtype)
        return dX, None, None, None


# ------------------------------------------------------------------------------------------------------------
# numpy / scipy compatibility wrappers used by the reference's evaluation code (utils.py:570-593)
# ------------------------------------------------------------------------------------------------------------
def _device() -> torch.device:
    if not torch.cuda.is_available():
        raise RuntimeError("graphlearninglayer_b200 needs a CUDA device (no CPU path)")
    return torch.device("cuda", torch.cuda.current_device())


class GraphStages:
    """K2 + K3 (gll_graph_build, gll_edge_weights) on kNN lists the caller searched: the graph (row_ptr, col, dist), its
    weights (eps, kappa, w, deg) and the unlabeled block's system (uu_ptr, uu_col, uu_val, diag, rhs) as device tensors, and
    ut whose first k_lab rows hold Y.  knn_idx / knn_dist may have more than n rows (never read); ws is a byte tensor of at
    least the graph and weights workspaces (None: one is allocated); ut is zero-filled when zero_ut."""

    def __init__(self, knn_idx: torch.Tensor, knn_dist: torch.Tensor, Y: torch.Tensor, n: int, tau: float, epsilon,
                 info: torch.Tensor, ws: Optional[torch.Tensor] = None, zero_ut: bool = False):
        dev = knn_idx.device
        k = knn_idx.shape[1]
        k_lab, l = Y.shape
        m, lp, emax = n - k_lab, lib.gll_padded_classes(l), lib.gll_max_edges(n, k)
        self.n, self.k, self.l, self.k_lab, self.m, self.lp = n, k, l, k_lab, m, lp
        self.eps_auto, eps_fixed = parse_epsilon(epsilon)
        self.knn_idx, self.knn_dist, self.info = knn_idx, knn_dist, info
        i32, f32 = torch.int32, torch.float32
        self.row_ptr = torch.empty(n + 1, dtype=i32, device=dev)
        self.col = torch.empty(emax, dtype=i32, device=dev)
        self.dist = torch.empty(emax, dtype=f32, device=dev)
        self.eps = torch.empty(n, dtype=f32, device=dev)
        self.kappa = torch.empty(n, dtype=i32, device=dev)
        self.w = torch.empty(emax, dtype=f32, device=dev)
        self.deg = torch.empty(n, dtype=f32, device=dev)
        self.uu_ptr = torch.empty(m + 1, dtype=i32, device=dev)
        self.uu_col = torch.empty(emax, dtype=i32, device=dev)
        self.uu_val = torch.empty(emax, dtype=f32, device=dev)
        self.diag = torch.empty(m, dtype=f32, device=dev)
        self.rhs = torch.empty((m, lp), dtype=f32, device=dev)
        self.ut = (torch.zeros if zero_ut else torch.empty)((n, lp), dtype=f32, device=dev)
        if ws is None:
            ws = _bytes(max(lib.gll_graph_workspace_bytes(n, k), lib.gll_weights_workspace_bytes(n, k)), dev)
        s = _stream_ptr(dev)
        _lib.check(lib.gll_graph_build(knn_idx.data_ptr(), knn_dist.data_ptr(), n, k, self.row_ptr.data_ptr(), self.col.data_ptr(),
                                       self.dist.data_ptr(), info.data_ptr(), ws.data_ptr(), ws.numel(), s), "gll_graph_build")
        _lib.check(lib.gll_edge_weights(knn_idx.data_ptr(), knn_dist.data_ptr(), self.row_ptr.data_ptr(), self.col.data_ptr(),
                                        self.dist.data_ptr(), Y.data_ptr(), n, k, l, k_lab, self.eps_auto, eps_fixed, float(tau),
                                        self.eps.data_ptr(), self.kappa.data_ptr(), self.w.data_ptr(), self.deg.data_ptr(),
                                        self.uu_ptr.data_ptr(), self.uu_col.data_ptr(), self.uu_val.data_ptr(),
                                        self.diag.data_ptr(), self.rhs.data_ptr(), self.ut.data_ptr(), info.data_ptr(),
                                        ws.data_ptr(), ws.numel(), s), "gll_edge_weights")


def knn_sym_dist(data, k=K_NEIGHBOURS, epsilon="auto"):
    """Same contract as the reference ``knn_sym_dist`` (GLL.py:180-244): numpy (n, d) in, scipy CSR out.

    Returns ``(W, V, mod_V, C, knn_ind)``; for a fixed epsilon ``mod_V`` and ``C`` are the integer 0, the reference's
    placeholders (GLL.py:229-230; its backward tests ``isinstance(C, int)``, GLL.py:124).  For 'auto', ``C`` is
    returned as a sparse CSR with C[kappa(i), i] = 1 (the reference builds the same matrix through a dense n x n
    array, GLL.py:209-213).  kNN, symmetrisation and the exp() run on the GPU; V and mod_V are the closed-form
    multiples of W (GLL.py:217-218) formed in fp64 on the host for the caller.
    """
    import scipy.sparse as sp

    dev = _device()
    Xc = torch.as_tensor(np.ascontiguousarray(data, dtype=np.float32)).to(dev)
    n, d = Xc.shape
    k = int(k)
    knn_idx = torch.empty((n, k), dtype=torch.int32, device=dev)
    knn_dist = torch.empty((n, k), dtype=torch.float32, device=dev)
    info = torch.zeros(_lib.INFO_WORDS, dtype=torch.int32, device=dev)
    wsb = max(lib.gll_knn_workspace_bytes(n, d, k), lib.gll_graph_workspace_bytes(n, k), lib.gll_weights_workspace_bytes(n, k))
    ws = _bytes(wsb, dev)
    _lib.check(lib.gll_knn(Xc.data_ptr(), n, d, k, knn_idx.data_ptr(), knn_dist.data_ptr(), info.data_ptr(), ws.data_ptr(), wsb,
                           _stream_ptr(dev)), "gll_knn")
    # the weights stage also emits the unlabeled-block system; with a 1-row dummy label block it is just ignored
    g = GraphStages(knn_idx, knn_dist, torch.zeros((1, 1), dtype=torch.float32, device=dev), n, 0.0, epsilon, info, ws)
    indptr = g.row_ptr.cpu().numpy()
    E = int(indptr[-1])
    cols = g.col[:E].cpu().numpy()
    dist = g.dist[:E].cpu().numpy().astype(np.float64)
    w = g.w[:E].cpu().numpy().astype(np.float64)
    eps = g.eps.cpu().numpy().astype(np.float64)
    if int(info[_lib.INFO_STATUS].item()) & _lib.STATUS_EPS_TINY:
        warnings.warn("Epsilon in KNN is very close to zero.")  # GLL.py:240-241
    rows = np.repeat(np.arange(n), np.diff(indptr))
    with np.errstate(divide="ignore", invalid="ignore"):
        v = -8.0 * w / eps[rows] / eps[cols]
    W = sp.csr_matrix((w, cols, indptr), shape=(n, n))
    V = sp.csr_matrix((v, cols.copy(), indptr.copy()), shape=(n, n))
    knn_ind = knn_idx.cpu().numpy().astype(np.int64)
    if isinstance(epsilon, str):
        with np.errstate(divide="ignore", invalid="ignore"):
            mv = dist * dist * v / (eps[rows] ** 2) / 2.0
        mod_V = sp.csr_matrix((mv, cols.copy(), indptr.copy()), shape=(n, n))
        kappa = g.kappa.cpu().numpy().astype(np.int64)
        Cm = sp.csr_matrix((np.ones(n), (kappa, np.arange(n))), shape=(n, n))
        return W, V, mod_V, Cm, knn_ind
    return W, V, 0, 0, knn_ind  # placeholders of GLL.py:229-230


def stable_conjgrad(A, b, x0=None, max_iter=1e5, tol=1e-10):
    """Same contract as the reference ``stable_conjgrad`` (GLL.py:247-276): scipy sparse SPD ``A``, numpy ``b``
    (m,) or (m, l) -> numpy solution with max_c ||b_c - A x_c||_2 <= tol (absolute), or 'max iter reached'.

    The solves run in the persistent fp32 CG kernel (gll_cg_solve); tolerances below what fp32 can reach are met by
    fp64 iterative refinement around it (residual b - A x by an fp64 CSR kernel, correction solved by the CG kernel), so
    the reference's default tol=1e-10 (utils.py:589-591) is honoured.  The ``p = r`` alias of GLL.py:254 is not
    reproduced (it only costs the reference iterations).
    """
    import scipy.sparse as sp

    dev = _device()
    A = sp.csr_matrix(A)
    A.sort_indices()
    b_np = np.asarray(b, dtype=np.float64)
    one_d = b_np.ndim == 1
    B = b_np[:, None] if one_d else b_np
    m, l_all = B.shape
    dg = A.diagonal()
    off = (A - sp.diags(dg)).tocsr()
    off.eliminate_zeros()
    off.sort_indices()
    i32, f32, f64 = torch.int32, torch.float32, torch.float64
    ptr = torch.as_tensor(off.indptr.astype(np.int32)).to(dev)
    col = torch.as_tensor(off.indices.astype(np.int32)).to(dev)
    val = torch.as_tensor((-off.data).astype(np.float32)).to(dev)  # kernel applies diag*p - sum val*p
    diag = torch.as_tensor(dg.astype(np.float32)).to(dev)
    # fp64 copy of the full matrix for the refinement residual r = b - A x (gll_csr_residual_f64)
    a_ptr = torch.as_tensor(A.indptr.astype(np.int32)).to(dev)
    a_col = torch.as_tensor(A.indices.astype(np.int32)).to(dev)
    a_val = torch.as_tensor(A.data.astype(np.float64)).to(dev)

    def residual(bb, x):
        r = torch.empty_like(bb)
        _lib.check(lib.gll_csr_residual_f64(a_ptr.data_ptr(), a_col.data_ptr(), a_val.data_ptr(), x.data_ptr(), bb.data_ptr(), m,
                                            bb.shape[1], r.data_ptr(), _stream_ptr(dev)), "gll_csr_residual_f64")
        return r

    X = np.zeros_like(B) if x0 is None else np.array(np.asarray(x0, dtype=np.float64).reshape(B.shape))
    maxit = int(max_iter)
    s = _stream_ptr(dev)
    total_it = 0
    converged = True
    for c0 in range(0, l_all, 128):  # the kernel handles up to 128 class columns per launch
        c1 = min(l_all, c0 + 128)
        l = c1 - c0
        lp = lib.gll_padded_classes(l)
        wsb = lib.gll_cg_workspace_bytes(m, l)
        ws = _bytes(wsb, dev)
        x = torch.as_tensor(X[:, c0:c1]).to(dev, f64).contiguous()
        bb = torch.as_tensor(B[:, c0:c1]).to(dev, f64).contiguous()
        rhs = torch.zeros((m, lp), dtype=f32, device=dev)
        corr = torch.empty((m, lp), dtype=f32, device=dev)
        stat = torch.zeros(4, dtype=i32, device=dev)
        ok = False
        for _ in range(12):
            r = residual(bb, x)
            rn = float(torch.linalg.vector_norm(r, dim=0).max().item())
            if rn <= tol or total_it >= maxit:
                ok = rn <= tol
                break
            scale = rn
            rhs[:, :l] = (r / scale).to(f32)
            inner_tol = max(1e-6, min(1e-3, 0.1 * tol / scale))
            _lib.check(lib.gll_cg_solve(ptr.data_ptr(), col.data_ptr(), val.data_ptr(), diag.data_ptr(), rhs.data_ptr(), m, l,
                                        inner_tol, max(1, maxit - total_it), corr.data_ptr(), stat.data_ptr(), 0,
                                        stat[1:].data_ptr(), ws.data_ptr(), wsb, s), "gll_cg_solve")
            total_it += int(stat[0].item())
            x += corr[:, :l].to(f64) * scale
        else:
            r = residual(bb, x)
            ok = float(torch.linalg.vector_norm(r, dim=0).max().item()) <= tol
        converged &= ok
        X[:, c0:c1] = x.cpu().numpy()
    if not converged:
        print("max iter reached")  # GLL.py:273-274
    return X[:, 0] if one_d else X
