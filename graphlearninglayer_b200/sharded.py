"""One large graph on N GPUs (BASELINE.json configs[4]: n = 1M nodes, d = 256, 100 classes; SURVEY.md 8e).

    pred = ShardedLaplaceLearning.apply(X, label_matrix, tau, epsilon)        # same call as the single-GPU layer

Every rank holds the full feature matrix X (the encoder output is all-gathered by the trainer, like the reference's
nn.DataParallel gather, utils.py:547-548).  Inside the layer the path is cut along its natural shards:

  rows      kNN search (K1) and the backward gather (K5/K6): rank r owns a block of nodes                [NCCL all-gather]
  columns   both CG solves (K4), default: rank r owns a block of the l class columns.  Columns of the multi-RHS CG are
            independent (per-column alpha/beta, GLL.py:262-269), so there is NO communication inside the solver
                                                                                                         [NCCL all-gather]
  rows      both CG solves, `cg_partition="rows"` (or GLL_B200_SHARD_CG=rows) -- the partition BASELINE.json's north star
            names: rank r owns a block of the unlabeled rows of x, r, p, s; every iteration exchanges the iterate with one
            all-gather and the three dot products with one all-reduce        [NCCL all-gather + all-reduce per iteration]
            `cg_partition="rows-p2p"`: the same partition with both exchanges fused into the kernels over NVLink peer
            memory (torch symmetric memory for the mapping; P2P stores + epoch flags, no NCCL inside the loop)
  replicated graph symmetrisation and weights (K2, K3): O(E) integer/byte work, a few ms at 1M nodes

Collectives per call: forward 2 all-gathers (kNN lists; U column blocks), backward 3 (w column blocks; b; dX row blocks).
`world` virtual ranks can also be executed one after the other in ONE process (`emulate=N`): that is how the slicing is
tested on a single GPU; the arithmetic is identical to the N-process run.
"""
from __future__ import annotations

import os
from typing import List, Optional

import torch
import torch.distributed as dist

from . import _lib
from ._lib import lib
from .GLL import K_NEIGHBOURS, GraphStages, _bytes, _cg_maxit, _cg_tol, _require_cuda, _stream_ptr, as_features, decode_info, pred_dtype

ROW_ALIGN = 128  # row blocks start on a tensor-core row tile


def row_block(n: int, rank: int, world: int):
    """Rows owned by `rank`: equal blocks of ceil(n/world) rounded up to ROW_ALIGN (the last blocks may be short/empty)."""
    per = -(-n // world)
    per = -(-per // ROW_ALIGN) * ROW_ALIGN
    lo = min(n, rank * per)
    hi = min(n, lo + per)
    return lo, hi, per


def col_block(l: int, rank: int, world: int):
    """Class columns owned by `rank`: equal blocks of ceil(l/world)."""
    per = -(-l // world)
    lo = min(l, rank * per)
    hi = min(l, lo + per)
    return lo, hi, per


class _Comm:
    """all_gather over real ranks (torch.distributed, NCCL) or over virtual ranks executed in this process."""

    def __init__(self, group=None, emulate: int = 0):
        self.group = group
        if emulate:
            self.world, self.ranks, self.real = emulate, list(range(emulate)), False
        elif dist.is_available() and dist.is_initialized():
            self.world, self.ranks, self.real = dist.get_world_size(group), [dist.get_rank(group)], True
        else:
            self.world, self.ranks, self.real = 1, [0], False

    def all_gather(self, parts: dict, like: torch.Tensor) -> List[torch.Tensor]:
        """parts: {rank: equally shaped tensor} for the ranks executed here -> list over all ranks."""
        if not self.real:
            return [parts[r] for r in range(self.world)]
        (mine,) = parts.values()
        out = torch.empty((self.world,) + tuple(mine.shape), dtype=mine.dtype, device=mine.device)
        dist.all_gather_into_tensor(out, mine.contiguous(), group=self.group)
        return list(out.unbind(0))


    def all_gather_blocks_(self, full: torch.Tensor, per: int) -> None:
        """In place: block r of `full` (rows [r*per, (r+1)*per)) is rank r's contribution.  Virtual ranks share `full`."""
        if self.real:
            r = self.ranks[0]
            dist.all_gather_into_tensor(full, full[r * per:(r + 1) * per], group=self.group)

    def all_reduce_sum_(self, parts: dict) -> None:
        """parts: {rank: tensor}; every tensor becomes the sum over all ranks (fixed rank order when emulated)."""
        if self.real:
            (mine,) = parts.values()
            dist.all_reduce(mine, op=dist.ReduceOp.SUM, group=self.group)
        elif self.world > 1:
            total = parts[0].clone()
            for r in range(1, self.world):
                total += parts[r]
            for r in range(self.world):
                parts[r].copy_(total)


def _forward(X: torch.Tensor, Y: torch.Tensor, tau: float, epsilon, comm: _Comm, k: int = K_NEIGHBOURS,
             cg_partition: str = "columns"):
    dev = X.device
    n, d = X.shape
    s = _stream_ptr(dev)
    info = torch.zeros(_lib.INFO_WORDS, dtype=torch.int32, device=dev)

    # ---- K1, rows: every rank searches its block of nodes against all n columns ----
    _, _, per = row_block(n, 0, comm.world)
    idx_parts, dist_parts = {}, {}
    knn_idx = torch.empty((comm.world * per, k), dtype=torch.int32, device=dev)
    knn_dist = torch.empty((comm.world * per, k), dtype=torch.float32, device=dev)
    for r in comm.ranks:
        lo, hi, _ = row_block(n, r, comm.world)
        if hi > lo:
            wsb = lib.gll_knn_rows_workspace_bytes(n, d, k, lo, hi)
            ws = _bytes(wsb, dev)
            _lib.check(lib.gll_knn_rows(X.data_ptr(), n, d, k, lo, hi, knn_idx.data_ptr(), knn_dist.data_ptr(), info.data_ptr(),
                                        ws.data_ptr(), wsb, s), "gll_knn_rows")
        idx_parts[r] = knn_idx[r * per:(r + 1) * per]
        dist_parts[r] = knn_dist[r * per:(r + 1) * per]
    if comm.real:  # (emulation wrote every block into the shared arrays already)
        knn_idx = torch.cat(comm.all_gather(idx_parts, knn_idx), 0)
        knn_dist = torch.cat(comm.all_gather(dist_parts, knn_dist), 0)

    # ---- K2, K3 replicated (kNN rows >= n are padding and never read) ----
    g = GraphStages(knn_idx, knn_dist, Y, n, tau, epsilon, info, zero_ut=True)
    g.d, g.cg_partition = d, cg_partition
    rhs, g.rhs = g.rhs, None  # the backward packs its own right-hand side

    # ---- K4, columns: each rank solves its block of class columns ----
    g.iters_fwd = torch.zeros(comm.world, dtype=torch.int32, device=dev)
    _solve(g, rhs, g.ut[g.k_lab:], _cg_tol(), comm, g.iters_fwd)
    pred = torch.empty((g.m, g.l), dtype=pred_dtype(), device=dev)
    _lib.check(lib.gll_unpack_pred(g.ut[g.k_lab:].data_ptr(), g.m, g.l, pred.data_ptr(), int(pred.dtype == torch.float64), s),
               "gll_unpack_pred")
    return pred, g


def _solve_columns(g, rhs: torch.Tensor, out: torch.Tensor, tol: float, comm: _Comm, iters: torch.Tensor):
    """out[:, cols] = A^-1 rhs[:, cols], cols split over the ranks; out and rhs are m x lp."""
    dev = rhs.device
    f32 = torch.float32
    s = _stream_ptr(dev)
    _, _, cper = col_block(g.l, 0, comm.world)
    lp_loc = lib.gll_padded_classes(cper)
    parts = {}
    for r in comm.ranks:
        c0, c1, _ = col_block(g.l, r, comm.world)
        cnt = c1 - c0
        x_loc = torch.zeros((g.m, lp_loc), dtype=f32, device=dev)
        if cnt > 0:
            b_loc = torch.empty((g.m, lp_loc), dtype=f32, device=dev)
            _lib.check(lib.gll_pack_columns(rhs.data_ptr(), g.m, g.lp, c0, cnt, b_loc.data_ptr(), lp_loc, s), "gll_pack_columns")
            # always solve `cper` columns (layout m x padded(cper)); columns beyond cnt have a zero right-hand side and
            # are frozen from the first iteration (GLL.py:262-263)
            wsb = lib.gll_cg_workspace_bytes(g.m, cper)
            ws = _bytes(wsb, dev)
            _lib.check(lib.gll_cg_solve(g.uu_ptr.data_ptr(), g.uu_col.data_ptr(), g.uu_val.data_ptr(), g.diag.data_ptr(),
                                        b_loc.data_ptr(), g.m, cper, tol, _cg_maxit(), x_loc.data_ptr(), iters[r:].data_ptr(), 0,
                                        g.info[_lib.INFO_STATUS:].data_ptr(), ws.data_ptr(), wsb, s), "gll_cg_solve")
        parts[r] = x_loc
    blocks = comm.all_gather(parts, out)
    for r, xb in enumerate(blocks):
        c0, c1, _ = col_block(g.l, r, comm.world)
        if c1 > c0:
            _lib.check(lib.gll_unpack_columns(xb.data_ptr(), g.m, lp_loc, c0, c1 - c0, out.data_ptr(), g.lp, s),
                       "gll_unpack_columns")


class _StopPoll:
    """Stop test of the host-driven CG loops without stalling the device: after every iteration the stop flag is copied
    into pinned host memory (async, own event); the host looks at the copy made `lag` iterations earlier, whose event has
    normally completed already.  Every rank looks at the copy of the SAME iteration, so all ranks leave the loop after the
    same number of launches (and collectives); iterations enqueued after the stop are no-ops on the device."""

    def __init__(self, lag: int):
        self.lag = max(0, lag)
        self.ring = torch.zeros(self.lag + 2, dtype=torch.int32).pin_memory()
        self.events = [None] * (self.lag + 2)

    def push(self, it: int, flag: torch.Tensor) -> None:
        slot = it % len(self.events)
        self.ring[slot:slot + 1].copy_(flag, non_blocking=True)
        ev = torch.cuda.Event()
        ev.record()
        self.events[slot] = ev

    def stopped(self, it: int, last: bool = False) -> bool:
        """True once the copy of iteration it - lag (of iteration it itself when `last`) shows the stop flag."""
        look = it if last else it - self.lag
        if look < 0:
            return False
        slot = look % len(self.events)
        self.events[slot].synchronize()
        return int(self.ring[slot]) != 0


def m_block(m: int, rank: int, world: int):
    """Unlabeled rows owned by `rank` in the row-partitioned CG: equal blocks of ceil(m/world) rounded up to 32."""
    per = -(-m // world)
    per = -(-per // 32) * 32
    lo = min(m, rank * per)
    hi = min(m, lo + per)
    return lo, hi, per


def _solve_rows(g, rhs: torch.Tensor, out: torch.Tensor, tol: float, comm: _Comm, iters: torch.Tensor):
    """out = A^-1 rhs with the ROWS of the system split over the ranks (csrc/cg_rows.cu): per iteration one all-gather of
    the iterate u (m x lp fp32) and one all-reduce of 3*lp fp64 dot products; out and rhs are m x lp."""
    dev = rhs.device
    s = _stream_ptr(dev)
    _, _, per = m_block(g.m, 0, comm.world)
    u_full = torch.zeros((comm.world * per, g.lp), dtype=torch.float32, device=dev)
    x_full = torch.zeros((comm.world * per, g.lp), dtype=torch.float32, device=dev)
    resid = torch.zeros(1, dtype=torch.float32, device=dev)
    st = {}
    for r in comm.ranks:
        lo, hi, _ = m_block(g.m, r, comm.world)
        wsb = lib.gll_cg_rows_workspace_bytes(max(hi - lo, 1), g.l)
        ws = _bytes(wsb, dev)
        sums = torch.zeros(3 * g.lp, dtype=torch.float64, device=dev)
        ctrl = torch.zeros(4, dtype=torch.int32, device=dev)
        st[r] = (lo, hi, ws, wsb, sums, ctrl)
        _lib.check(lib.gll_cg_rows_init(g.diag.data_ptr(), rhs.data_ptr(), g.m, g.l, lo, hi, x_full.data_ptr(), u_full.data_ptr(),
                                        ws.data_ptr(), wsb, s), "gll_cg_rows_init")
    maxit = _cg_maxit()
    first = comm.ranks[0]
    poll = _StopPoll(int(os.environ.get("GLL_B200_ROWS_STOP_LAG", "1")))  # every extra iteration costs an all-gather here
    for it in range(maxit + 1):
        comm.all_gather_blocks_(u_full, per)
        for r in comm.ranks:
            lo, hi, ws, wsb, sums, ctrl = st[r]
            _lib.check(lib.gll_cg_rows_spmv(g.uu_ptr.data_ptr(), g.uu_col.data_ptr(), g.uu_val.data_ptr(), g.diag.data_ptr(), g.m,
                                            g.l, lo, hi, u_full.data_ptr(), sums.data_ptr(), ws.data_ptr(), wsb, s),
                       "gll_cg_rows_spmv")
        comm.all_reduce_sum_({r: st[r][4] for r in comm.ranks})
        for r in comm.ranks:
            lo, hi, ws, wsb, sums, ctrl = st[r]
            _lib.check(lib.gll_cg_rows_update(g.diag.data_ptr(), g.m, g.l, lo, hi, sums.data_ptr(), it, maxit, tol,
                                              x_full.data_ptr(), u_full.data_ptr(), ctrl.data_ptr(), resid.data_ptr(),
                                              ws.data_ptr(), wsb, s), "gll_cg_rows_update")
        # the stop flag is identical on every rank (same reduced sums)
        poll.push(it, st[first][5][0:1])
        if poll.stopped(it, last=it == maxit):
            break
    comm.all_gather_blocks_(x_full, per)
    out.copy_(x_full[:g.m])
    ctrl = st[first][5]
    for r in comm.ranks:
        iters[r:r + 1].copy_(ctrl[1:2])
    g.info[_lib.INFO_STATUS:_lib.INFO_STATUS + 1] |= ctrl[2:3]
    g.cg_rows_resid = resid


_P2P_BLOCKS = {}  # (device index, world, rows, lp) -> symmetric u array, mailbox / flag block, peer table, next epoch


def _p2p_block(dev: torch.device, rows_total: int, lp: int, comm: _Comm):
    """Symmetric-memory buffers of the peer-memory CG (allocated and exchanged once per shape, collectively)."""
    import ctypes

    import torch.distributed._symmetric_memory as symm_mem

    key = (dev.index, comm.world, rows_total, lp)
    blk = _P2P_BLOCKS.get(key)
    if blk is None:
        grp = comm.group if comm.group is not None else dist.group.WORLD
        mail_b = lib.gll_cg_rows_peer_mail_bytes()
        u = symm_mem.empty((rows_total, lp), dtype=torch.float32, device=dev)
        ctl = symm_mem.empty((mail_b + lib.gll_cg_rows_peer_flag_bytes() + 256,), dtype=torch.uint8, device=dev)
        u.zero_()
        ctl.zero_()
        hu, hc = symm_mem.rendezvous(u, grp), symm_mem.rendezvous(ctl, grp)
        torch.cuda.synchronize(dev)
        dist.barrier(grp)  # every rank's flags are zero before anybody can raise one
        P = _lib.Peers()
        P.world, P.rank = comm.world, comm.ranks[0]
        for r in range(comm.world):
            P.u[r] = ctypes.c_void_p(int(hu.buffer_ptrs[r]))
            P.mail[r] = ctypes.c_void_p(int(hc.buffer_ptrs[r]))
            P.flags[r] = ctypes.c_void_p(int(hc.buffer_ptrs[r]) + mail_b)
        blk = dict(u=u, ctl=ctl, hu=hu, hc=hc, P=P, epoch=1)
        _P2P_BLOCKS[key] = blk
    return blk


def _solve_rows_p2p(g, rhs: torch.Tensor, out: torch.Tensor, tol: float, comm: _Comm, iters: torch.Tensor):
    """Row-partitioned CG with BOTH collectives fused into the kernels over NVLink peer memory (csrc/cg_rows.cu, peer-memory
    mode): the update kernel stores the new iterate into every rank's copy, the SpMV kernel's last CTA stores the partial
    dot products into every rank's mailbox; epoch flags in peer memory order the kernels across GPUs.  No NCCL call and no
    host stall inside the loop (the stop flag is polled through pinned memory, two iterations behind); one all-gather of x at the end."""
    import ctypes

    dev = rhs.device
    s = _stream_ptr(dev)
    rank = comm.ranks[0]
    _, _, per = m_block(g.m, 0, comm.world)
    blk = _p2p_block(dev, comm.world * per, g.lp, comm)
    P = ctypes.byref(blk["P"])
    x_full = torch.zeros((comm.world * per, g.lp), dtype=torch.float32, device=dev)
    resid = torch.zeros(1, dtype=torch.float32, device=dev)
    lo, hi, _ = m_block(g.m, rank, comm.world)
    wsb = lib.gll_cg_rows_workspace_bytes(max(hi - lo, 1), g.l)
    ws = _bytes(wsb, dev)
    ctrl = torch.zeros(4, dtype=torch.int32, device=dev)
    maxit = _cg_maxit()
    e0 = blk["epoch"]
    blk["epoch"] = e0 + maxit + 4  # flags only grow: the next solve starts above everything this one can publish
    _lib.check(lib.gll_cg_rows_init_p2p(g.diag.data_ptr(), rhs.data_ptr(), g.m, g.l, lo, hi, x_full.data_ptr(), P, e0,
                                        ws.data_ptr(), wsb, s), "gll_cg_rows_init_p2p")
    poll = _StopPoll(int(os.environ.get("GLL_B200_ROWS_STOP_LAG", "2")))
    for it in range(maxit + 1):
        _lib.check(lib.gll_cg_rows_spmv_p2p(g.uu_ptr.data_ptr(), g.uu_col.data_ptr(), g.uu_val.data_ptr(), g.diag.data_ptr(), g.m,
                                            g.l, lo, hi, P, e0 + it, ctrl.data_ptr(), ws.data_ptr(), wsb, s),
                   "gll_cg_rows_spmv_p2p")
        _lib.check(lib.gll_cg_rows_update_p2p(g.diag.data_ptr(), g.m, g.l, lo, hi, it, maxit, tol, x_full.data_ptr(), P, e0 + it,
                                              ctrl.data_ptr(), resid.data_ptr(), ws.data_ptr(), wsb, s),
                   "gll_cg_rows_update_p2p")
        poll.push(it, ctrl[0:1])
        if poll.stopped(it, last=it == maxit):
            break
    comm.all_gather_blocks_(x_full, per)
    out.copy_(x_full[:g.m])
    iters[rank:rank + 1].copy_(ctrl[1:2])
    g.info[_lib.INFO_STATUS:_lib.INFO_STATUS + 1] |= ctrl[2:3]


def _solve(g, rhs, out, tol, comm, iters):
    ev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))  # solve incl. its collectives
    ev[0].record()
    if g.cg_partition == "rows-p2p" and comm.real and comm.world > 1:
        _solve_rows_p2p(g, rhs, out, tol, comm, iters)
    elif g.cg_partition in ("rows", "rows-p2p"):   # rows-p2p needs real ranks with peer access; otherwise the NCCL form
        _solve_rows(g, rhs, out, tol, comm, iters)
    else:
        _solve_columns(g, rhs, out, tol, comm, iters)
    ev[1].record()
    g.solve_events = getattr(g, "solve_events", []) + [ev]


def _backward(g, X: torch.Tensor, grad_output: torch.Tensor, comm: _Comm) -> torch.Tensor:
    dev = X.device
    f32 = torch.float32
    s = _stream_ptr(dev)
    n, d, l, m, k_lab = g.n, g.d, g.l, g.m, g.k_lab
    gout = grad_output.detach().to(dev)
    if gout.dtype not in (torch.float32, torch.float64):
        gout = gout.float()
    gout = gout.contiguous()
    rhs = torch.empty((m, g.lp), dtype=f32, device=dev)
    _lib.check(lib.gll_pack_grad(gout.data_ptr(), int(gout.dtype == torch.float64), m, l, rhs.data_ptr(), s), "gll_pack_grad")
    wt = torch.zeros((n, g.lp), dtype=f32, device=dev)  # GLL.py:104: zero rows for the labeled nodes
    g.iters_bwd = torch.zeros(comm.world, dtype=torch.int32, device=dev)
    _solve(g, rhs, wt[k_lab:], -_cg_tol(), comm, g.iters_bwd)
    g.wt = wt  # [0; adjoint solution], GLL.py:104 (kept for inspection, like ut)

    # ---- K5 rows -> all-gather b -> K6 rows -> all-gather dX ----
    _, _, per = row_block(n, 0, comm.world)
    emax = g.col.numel()
    gv = torch.empty(emax, dtype=f32, device=dev)
    bvec = torch.zeros(comm.world * per, dtype=f32, device=dev)
    dX = torch.empty((comm.world * per, d), dtype=f32, device=dev)

    def edges(r, phases):
        lo, hi, _ = row_block(n, r, comm.world)
        _lib.check(lib.gll_backward_edges_rows(X.data_ptr(), n, d, l, k_lab, g.eps_auto, g.row_ptr.data_ptr(), g.col.data_ptr(),
                                               g.dist.data_ptr(), g.w.data_ptr(), g.eps.data_ptr(), g.kappa.data_ptr(),
                                               g.ut.data_ptr(), wt.data_ptr(), gv.data_ptr(), bvec.data_ptr(), dX.data_ptr(),
                                               lo, hi, phases, s), "gll_backward_edges_rows")

    for r in comm.ranks:
        edges(r, 1)
    if comm.real and g.eps_auto:
        parts = {r: bvec[r * per:(r + 1) * per] for r in comm.ranks}
        bvec.copy_(torch.cat(comm.all_gather(parts, bvec), 0))
    for r in comm.ranks:
        edges(r, 2)
    if comm.real:
        parts = {r: dX[r * per:(r + 1) * per] for r in comm.ranks}
        dX = torch.cat(comm.all_gather(parts, dX), 0)
    return dX[:n]


class ShardedLaplaceLearning(torch.autograd.Function):
    """`LaplaceLearningSparseHard` (GLL.py:10-177) for ONE graph spread over the ranks of a process group.

    forward(X, label_matrix, tau=0, epsilon='auto', group=None, emulate=0, cg_partition=None): every rank passes the SAME X
    and labels and receives the same full prediction; backward returns the full dX on every rank.  cg_partition: "columns"
    (default; or GLL_B200_SHARD_CG) / "rows" -- how the two CG solves are split (module docstring)."""

    @staticmethod
    def forward(ctx, X, label_matrix, tau=0, epsilon="auto", group=None, emulate=0, cg_partition=None):
        _require_cuda(X, "features")
        Xc = as_features(X)
        Y = label_matrix.detach().to(device=X.device, dtype=torch.float32).contiguous()
        if not (0 < Y.shape[0] < Xc.shape[0]):
            raise ValueError("need 0 < k_lab < n; labeled rows come first (GLL.py:11)")
        comm = _Comm(group, emulate)
        part = cg_partition or os.environ.get("GLL_B200_SHARD_CG", "columns")
        if part not in ("columns", "rows", "rows-p2p"):
            raise ValueError("cg_partition must be 'columns', 'rows' or 'rows-p2p'")
        with torch.cuda.device(X.device):
            pred, g = _forward(Xc, Y, float(tau), epsilon, comm, cg_partition=part)
        global _last_graph
        _last_graph = g
        ctx.gll_graph, ctx.gll_comm, ctx.x_dtype = g, comm, X.dtype
        ctx.save_for_backward(Xc)
        return pred

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, grad_output):
        (Xc,) = ctx.saved_tensors
        with torch.cuda.device(Xc.device):
            dX = _backward(ctx.gll_graph, Xc, grad_output, ctx.gll_comm)
        return dX.to(ctx.x_dtype), None, None, None, None, None, None


_last_graph = None


def last_info() -> dict:
    """Status block of the most recent sharded call on this rank (synchronises); same keys as GLL.last_info()."""
    g = _last_graph
    if g is None:
        return {}
    solve_ms = [a.elapsed_time(b) for a, b in getattr(g, "solve_events", [])]
    return dict(decode_info(g.info.cpu().numpy()), cg_partition=g.cg_partition, cg_solve_ms=solve_ms,
                cg_iters_fwd=int(g.iters_fwd.max().item()),
                cg_iters_bwd=int(g.iters_bwd.max().item()) if hasattr(g, "iters_bwd") else 0,
                cg_resid_fwd=float("nan"), cg_resid_bwd=float("nan"))
