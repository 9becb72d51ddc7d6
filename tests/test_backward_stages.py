"""Stage tests of the backward edge pass -- K5 `edge_grad_kernel` and every K6 `row_gather_kernel` instantiation
(csrc/backward.cu) -- and of the row normalisation pair (`gll_normalize_rows` / `_backward`, csrc/api.cu), each against a
plain fp64 restatement of the same operation on the same fp32 inputs.

The per-edge reference (GLL.py:104-159, as in test_gpu_parity._stagewise_fp64_check), over a CSR (row_ptr, col, dist, w):
    wt[:k_lab] := 0
    G_e  = -<wt_i - wt_j, ut_i - ut_j>,   V_e = -8 w_e / (eps_i eps_j),   gv_e = G_e V_e
    b_i  = sum_e G_e dist_e^2 V_e / (2 eps_i^2)                                     (eps = 'auto' only)
    t_e  = gv_e - [j == kappa_i] b_i - [kappa_j == i] b_j                           (fixed eps: t = gv)
    dX_i = sum_e t_e (x_i - x_j)
It is pinned to the oracle's backward (and through it to the reference fixtures) by the CPU test below.  The GPU tests build
their stage inputs on the host, so that a failure points at K5/K6 and nothing upstream.  Bounds come from rounding analysis
(u = 2^-24); every check prints its worst error as a fraction of its bound (`pytest -s`).
"""
import ctypes as C

import numpy as np
import pytest
import scipy.sparse as sp

from oracle import gll_oracle as O

U = 2.0 ** -24
K = 25


# ----------------------------------------------------------------------------------------------------------------
# fp64 reference
# ----------------------------------------------------------------------------------------------------------------
def edge_ref(row_ptr, col, dist, w, eps, kappa, ut, wt, k_lab):
    """Per-edge fp64 K5 and K6 edge weights from the given arrays (widened to fp64; kappa None: fixed eps).  Also returns the
    magnitudes the bounds are built from: S_e = |V_e| sum_c |dwt_c| |dut_c|, bS_i = sum_e |G_e modV_e| and
    tabs_e = |gv_e| + |b_i| [j == kappa_i] + |b_j| [kappa_j == i]."""
    row_ptr = np.asarray(row_ptr, dtype=np.int64)
    col = np.asarray(col, dtype=np.int64)
    n = len(row_ptr) - 1
    rows = np.repeat(np.arange(n), np.diff(row_ptr))
    dist, w, eps = (np.asarray(a, dtype=np.float64) for a in (dist, w, eps))
    ut = np.asarray(ut, dtype=np.float64)
    wt = np.array(wt, dtype=np.float64)
    wt[:k_lab] = 0.0
    du = ut[rows] - ut[col]
    dw = wt[rows] - wt[col]
    G = -np.einsum("ij,ij->i", dw, du)
    V = -8.0 * w / eps[rows] / eps[col]
    gv = G * V
    r = dict(rows=rows, G=G, gv=gv, S=np.abs(V) * np.einsum("ij,ij->i", np.abs(dw), np.abs(du)))
    if kappa is None:
        r.update(b=np.zeros(n), bS=np.zeros(n), t=gv, tabs=np.abs(gv))
        return r
    kappa = np.asarray(kappa, dtype=np.int64)
    Gm = G * (dist * dist * V / eps[rows] ** 2 / 2.0)
    b = np.bincount(rows, weights=Gm, minlength=n)
    ci, cj = col == kappa[rows], kappa[col] == rows
    r.update(b=b, bS=np.bincount(rows, weights=np.abs(Gm), minlength=n), t=gv - ci * b[rows] - cj * b[col],
             tabs=np.abs(gv) + ci * np.abs(b[rows]) + cj * np.abs(b[col]))
    return r


def edge_sum(X, row_ptr, col, coef):
    """(sum_e c_e (x_i - x_j), sum_e |c_e| |x_i - x_j|) for every row i, in fp64, edge blocks of about 4M elements."""
    X = np.asarray(X, dtype=np.float64)
    row_ptr = np.asarray(row_ptr, dtype=np.int64)
    col = np.asarray(col, dtype=np.int64)
    coef = np.asarray(coef, dtype=np.float64)
    n, d = X.shape
    out, mag = np.zeros((n, d)), np.zeros((n, d))
    step = max(1, (1 << 22) // d)
    r0 = 0
    while r0 < n:
        r1 = max(r0 + 1, int(np.searchsorted(row_ptr, row_ptr[r0] + step, side="right")) - 1)
        r1 = min(r1, n)
        e0, e1 = row_ptr[r0], row_ptr[r1]
        rr = np.repeat(np.arange(r1 - r0), np.diff(row_ptr[r0:r1 + 1]))
        diff = X[r0 + rr] - X[col[e0:e1]]
        S = sp.csr_matrix((coef[e0:e1], (rr, np.arange(e1 - e0))), shape=(r1 - r0, e1 - e0))
        out[r0:r1] = S @ diff
        S.data = np.abs(S.data)
        mag[r0:r1] = S @ np.abs(diff)
        r0 = r1
    return out, mag


def within(case, err, bound):
    """err <= bound elementwise (NaN fails); prints the worst err / bound."""
    err = np.asarray(err, dtype=np.float64)
    bound = np.asarray(bound, dtype=np.float64)
    ok = err <= bound
    with np.errstate(divide="ignore", invalid="ignore"):
        frac = np.where(bound > 0, err / bound, np.where(err == 0, 0.0, np.inf))
    worst = float(np.nanmax(frac, initial=0.0)) if ok.all() else float("inf")
    print(f"bound {case}: worst err/bound {worst:.3g}")
    assert ok.all(), f"{case}: {int((~ok).sum())} of {ok.size} outside the bound; first at {np.argwhere(~ok)[0]}"
    return worst


@pytest.mark.parametrize("seed,k_lab,m,d,l,sigma,eps", [(0, 300, 500, 64, 10, 2.0, "auto"), (3, 37, 91, 19, 3, 1.0, "auto"),
                                                        (0, 300, 500, 64, 10, 2.0, 1.0)])
def test_edge_reference_matches_oracle_backward(seed, k_lab, m, d, l, sigma, eps):
    """The per-edge restatement reproduces the oracle's backward (Laplacian products and the kappa scatter of GLL.py:126-159)."""
    X, Y, _, yq = O.synth_inputs(seed, k_lab, m, d, l, sigma)
    f, _, _, bw = O.fwd_bwd(X, Y, yq, 0.0, eps, solver="lu")
    g = f.graph
    ut = np.concatenate([Y, f.pred])
    wt = np.concatenate([np.full(Y.shape, np.nan), bw.w])  # the labeled head is never read
    R = edge_ref(g.dist.indptr, g.dist.indices, g.dist.data, g.W.data, g.eps, g.kappa, ut, wt, k_lab)
    dX, _ = edge_sum(X, g.dist.indptr, g.dist.indices, R["t"])
    assert O.max_rel(dX, bw.dX) < 1e-13
    if g.kappa is not None:
        assert O.max_rel(R["b"], bw.b) < 1e-13
    # and edge_sum itself against a plain per-edge loop
    i = int(np.argmax(np.diff(g.dist.indptr)))
    e0, e1 = g.dist.indptr[i], g.dist.indptr[i + 1]
    Xd = X.astype(np.float64)
    ref_i = sum(R["t"][e] * (Xd[i] - Xd[g.dist.indices[e]]) for e in range(e0, e1))
    assert np.allclose(dX[i], ref_i, rtol=1e-14, atol=1e-14 * np.abs(ref_i).max())


# ----------------------------------------------------------------------------------------------------------------
# stage inputs (host) and the device call
# ----------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def gll():
    torch = pytest.importorskip("torch")
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from test_gpu_parity import dev_t

    import graphlearninglayer_b200 as pkg
    from graphlearninglayer_b200 import _lib

    return torch, pkg, _lib, dev_t


class Stage:
    """fp32 / int32 inputs of K5 and K6 as the device reads them, and the fp64 reference built from the same arrays."""

    def __init__(self, X, row_ptr, col, dist, w, eps, kappa, k_lab, l, seed=0, Y=None):
        self.X = np.ascontiguousarray(X, dtype=np.float32)
        self.n, self.d = self.X.shape
        self.row_ptr = np.asarray(row_ptr, dtype=np.int32)
        self.col = np.asarray(col, dtype=np.int32)
        self.E = int(self.row_ptr[-1])
        self.dist = np.asarray(dist, dtype=np.float32)
        self.w = np.asarray(w, dtype=np.float32)
        self.eps = np.asarray(eps, dtype=np.float32)
        self.kappa = None if kappa is None else np.asarray(kappa, dtype=np.int32)
        assert self.w.min() > 1e-20, "weights near fp32 underflow make every check trivial"
        self.k_lab, self.l = k_lab, l
        self.lp = (l + 3) // 4 * 4
        rng = np.random.default_rng(seed)
        if Y is None:
            Y = np.zeros((k_lab, l), dtype=np.float32)
            Y[np.arange(k_lab), rng.integers(0, l, size=k_lab)] = 1.0
        self.ut = np.zeros((self.n, self.lp), dtype=np.float32)
        self.ut[:k_lab, :l] = Y
        self.ut[k_lab:, :l] = rng.random((self.n - k_lab, l))
        self.wt = np.zeros((self.n, self.lp), dtype=np.float32)
        self.wt[:k_lab] = np.nan  # the labeled head of the adjoint solution is never read
        self.wt[k_lab:, :l] = rng.standard_normal((self.n - k_lab, l))
        self.ref = edge_ref(self.row_ptr, self.col, self.dist, self.w, self.eps, self.kappa, self.ut, self.wt, k_lab)

    @classmethod
    def from_graph(cls, X, k_lab, l, eps, seed=0, Y=None):
        g = O.build_graph(X, K, eps)
        D = g.dist
        return cls(X, D.indptr, D.indices, D.data, g.W.data, g.eps, g.kappa, k_lab, l, seed, Y)

    @property
    def auto(self):
        return self.kappa is not None


def run_edges(gll, S, phases=3, rows=None, out=None, shift=0):
    """gll_backward_edges (rows None) or gll_backward_edges_rows on S's inputs.  out: host (gv, bvec, dX) the device buffers
    start from (default NaN).  shift: X and dX start that many floats past a 16-byte boundary.  Returns host copies of
    (gv, bvec, dX)."""
    torch, _, _lib, dev_t = gll
    f32, i32 = torch.float32, torch.int32

    def dev_shifted(a, k):
        buf = torch.empty(a.size + k, dtype=f32, device="cuda")
        assert buf.data_ptr() % 16 == 0
        buf[k:] = dev_t(a, f32).ravel()
        return buf[k:].view(a.shape)

    if out is None:
        out = (np.full(S.E, np.nan, np.float32), np.full(S.n, np.nan, np.float32), np.full((S.n, S.d), np.nan, np.float32))
    gv, bvec = (dev_t(a, f32) for a in out[:2])
    X, dX = dev_shifted(S.X, shift), dev_shifted(out[2], shift)
    rp, col = dev_t(S.row_ptr, i32), dev_t(S.col, i32)
    dist, w, eps, ut, wt = (dev_t(a, f32) for a in (S.dist, S.w, S.eps, S.ut, S.wt))
    kappa = dev_t(S.kappa, i32) if S.auto else None
    args = (X.data_ptr(), S.n, S.d, S.l, S.k_lab, int(S.auto), rp.data_ptr(), col.data_ptr(), dist.data_ptr(), w.data_ptr(),
            eps.data_ptr(), kappa.data_ptr() if S.auto else None, ut.data_ptr(), wt.data_ptr(), gv.data_ptr(), bvec.data_ptr(),
            dX.data_ptr())
    stream = torch.cuda.current_stream().cuda_stream
    if rows is None:
        assert phases == 3
        _lib.check(_lib.lib.gll_backward_edges(*args, stream), "gll_backward_edges")
    else:
        _lib.check(_lib.lib.gll_backward_edges_rows(*args, rows[0], rows[1], phases, stream), "gll_backward_edges_rows")
    torch.cuda.synchronize()
    return gv.cpu().numpy(), bvec.cpu().numpy(), dX.cpu().numpy()


def check_k5(S, gv, bvec, case):
    R = S.ref
    within(f"{case} gv", np.abs(gv.astype(np.float64) - R["gv"]), U * np.abs(R["gv"]) + 1e-13 * R["S"])
    if S.auto:
        within(f"{case} b", np.abs(bvec.astype(np.float64) - R["b"]), U * np.abs(R["b"]) + 1e-13 * R["bS"])


def check_k6(S, gv, bvec, dX, case):
    """Tight: the device's own gv / b, t formed in fp32 as the kernel forms it, the sum in fp64.  Accuracy: the all-fp64
    reference, with a bound for what fp32 gv / b / t cost."""
    rows, col = S.ref["rows"], S.col.astype(np.int64)
    tc = gv.astype(np.float32).copy()
    if S.auto:
        kap = S.kappa.astype(np.int64)
        ci, cj = col == kap[rows], kap[col] == rows
        tc[ci] = tc[ci] - bvec[rows[ci]]
        tc[cj] = tc[cj] - bvec[col[cj]]
    dXd = dX.astype(np.float64)
    ref, mag = edge_sum(S.X, S.row_ptr, col, tc)
    within(f"{case} dX tight", np.abs(dXd - ref), 2.0 ** -23 * (np.abs(ref) + mag))
    ref64, _ = edge_sum(S.X, S.row_ptr, col, S.ref["t"])
    _, mag64 = edge_sum(S.X, S.row_ptr, col, S.ref["tabs"])
    within(f"{case} dX accuracy", np.abs(dXd - ref64), 4 * U * mag64 + U * np.abs(ref64))


def gaussian_points(seed, n, d):
    """Rows of N(0, I/d): kNN distances of order one at every d, so that W = exp(-4 d^2 / eps_i eps_j) stays normal in fp32."""
    return (np.random.default_rng(seed).standard_normal((n, d)) / np.sqrt(d)).astype(np.float32)


# ----------------------------------------------------------------------------------------------------------------
# 1. K5 on its own
# ----------------------------------------------------------------------------------------------------------------
# l = 1, 10, 130: 1, 3 and 33 float4 chunks of a row of ut / wt; (900, 60): most edges join two labeled rows
@pytest.mark.gpu
@pytest.mark.parametrize("eps", ["auto", 1.0])
@pytest.mark.parametrize("k_lab,m,l", [(150, 350, 1), (150, 350, 10), (150, 350, 130), (900, 60, 10)])
def test_edge_grad_vs_reference(gll, k_lab, m, l, eps):
    X, *_ = O.synth_inputs(11 + l, k_lab, m, 16, l, 1.0)
    S = Stage.from_graph(X, k_lab, l, eps, seed=l)
    if k_lab == 900:
        lab = S.ref["rows"] < k_lab
        assert np.mean(lab & (S.col < k_lab)) > 0.8
    gv, bvec, dX = run_edges(gll, S, phases=1, rows=(0, S.n))
    check_k5(S, gv, bvec, f"K5 l={l} k_lab={k_lab} eps={eps}")
    assert np.isnan(dX).all()  # phase 1 writes no dX
    if not S.auto:
        assert np.isnan(bvec).all()  # fixed eps: no b


# ----------------------------------------------------------------------------------------------------------------
# 2. K6 on every variant
# ----------------------------------------------------------------------------------------------------------------
# row_gather_kernel<W, NV>, column passes of 32 NV chunks of W floats.  d % 4 != 0 -> W = 1: 1 / 3 / 19 -> NV 1, 99 -> NV 4,
# 130 -> NV 8, 515 -> NV 16 two passes, 2051 -> five.  Otherwise W = 4: 128 -> NV 1, 132 / 256 -> NV 2, 260 / 512 -> NV 4
# one pass, 516 -> two passes, 2048 -> four.
@pytest.mark.gpu
@pytest.mark.parametrize("eps", ["auto", 1.0])
@pytest.mark.parametrize("d", [1, 3, 19, 99, 128, 130, 132, 256, 260, 512, 515, 516, 2048, 2051])
def test_row_gather_every_variant(gll, d, eps):
    X = gaussian_points(100 + d, 320, d)
    S = Stage.from_graph(X, 64, 5, eps, seed=d)
    gv, bvec, dX = run_edges(gll, S)
    check_k5(S, gv, bvec, f"K5 d={d} eps={eps}")
    check_k6(S, gv, bvec, dX, f"K6 d={d} eps={eps}")


@pytest.mark.gpu
@pytest.mark.parametrize("eps", ["auto", 1.0])
def test_row_gather_misaligned_rows(gll, eps):
    """d % 4 == 0 with X and dX one float past a 16-byte boundary: float chunks (W = 1), not float4 loads."""
    d = 512
    X = gaussian_points(100 + d, 320, d)
    S = Stage.from_graph(X, 64, 5, eps, seed=d)
    gv, bvec, dX = run_edges(gll, S, shift=1)
    check_k5(S, gv, bvec, f"K5 d={d} misaligned eps={eps}")
    check_k6(S, gv, bvec, dX, f"K6 d={d} misaligned eps={eps}")


# ----------------------------------------------------------------------------------------------------------------
# 3. structure edges
# ----------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("eps", ["auto", 1.0])
@pytest.mark.parametrize("hub", ["labeled", "unlabeled"])
@pytest.mark.parametrize("d", [2048, 2051])
def test_row_gather_planted_hub(gll, d, hub, eps):
    """Unit-sphere points and the origin, every row's nearest neighbour: the origin's row has n - 1 edges (twenty 32-edge
    ballots of row_gather_kernel, each column pass)."""
    n, k_lab = 641, 100
    X = gaussian_points(7 + d, n, d)
    X /= np.linalg.norm(X, axis=1, keepdims=True)
    h = 0 if hub == "labeled" else n - 1
    X[h] = 0.0
    S = Stage.from_graph(X, k_lab, 10, eps, seed=d)
    assert np.diff(S.row_ptr)[h] == n - 1
    gv, bvec, dX = run_edges(gll, S)
    case = f"hub d={d} {hub} eps={eps}"
    check_k5(S, gv, bvec, case)
    check_k6(S, gv, bvec, dX, case)


def hand_built_csr(n, seed):
    """Symmetric CSR with what a kNN graph cannot have: rows without edges, rows of exactly 32, 33, 128 and 129 edges, and one
    row (the 128-edge one) that is kappa of all of its neighbours.  Returns (row_ptr, col, dist, w, eps, kappa, special)."""
    rng = np.random.default_rng(seed)
    empty = [3, 99, 100, n - 2]
    special = {40: 32, 170: 33, 260: 128, n - 1: 129}  # labeled rows are [0, 120)
    others = np.array([i for i in range(n) if i not in special and i not in empty])
    pairs = set()
    for i in others:
        for j in rng.choice(others, size=3, replace=False):
            if i != j:
                pairs.add((min(i, j), max(i, j)))
    for i, deg in special.items():
        for j in rng.choice(others, size=deg, replace=False):
            pairs.add((min(i, j), max(i, j)))
    p = np.array(sorted(pairs))
    r = np.concatenate([p[:, 0], p[:, 1]])
    c = np.concatenate([p[:, 1], p[:, 0]])
    dval = np.tile(rng.uniform(0.2, 1.5, size=len(p)), 2)
    A = sp.csr_matrix((dval, (r, c)), shape=(n, n))
    A.sort_indices()
    deg = np.diff(A.indptr)
    assert all(deg[i] == v for i, v in special.items()) and all(deg[i] == 0 for i in empty)
    eps = rng.uniform(0.5, 2.0, size=n).astype(np.float32)
    rows = np.repeat(np.arange(n), deg)
    w = np.exp(-4.0 * A.data ** 2 / eps[rows] / eps[A.indices])
    kappa = np.array([A.indices[A.indptr[i] + rng.integers(deg[i])] if deg[i] else i for i in range(n)])
    hub = 260
    kappa[A.indices[A.indptr[hub]:A.indptr[hub + 1]]] = hub
    return A.indptr, A.indices, A.data, w, eps, kappa, special, empty


@pytest.mark.gpu
@pytest.mark.parametrize("eps", ["auto", "fixed"])
@pytest.mark.parametrize("d", [19, 516])
def test_row_gather_hand_built_csr(gll, d, eps):
    n, k_lab = 400, 120
    row_ptr, col, dist, w, epsv, kappa, special, empty = hand_built_csr(n, 5)
    if eps == "fixed":
        epsv, kappa = np.full(n, 0.75, np.float32), None
        w = np.exp(-4.0 * np.asarray(dist) ** 2 / 0.75 ** 2)
    S = Stage(gaussian_points(d, n, d), row_ptr, col, dist, w, epsv, kappa, k_lab, 6, seed=d)
    gv, bvec, dX = run_edges(gll, S)
    case = f"hand-built CSR d={d} eps={eps}"
    check_k5(S, gv, bvec, case)
    check_k6(S, gv, bvec, dX, case)
    assert np.all(dX[empty] == 0.0)
    if S.auto:
        assert np.all(bvec[empty] == 0.0)
        assert np.count_nonzero(S.kappa == 260) >= 128


# ----------------------------------------------------------------------------------------------------------------
# 4. row ranges and phases (sharded.py:_backward)
# ----------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("eps", ["auto", 1.0])
@pytest.mark.parametrize("d", [19, 64])
def test_backward_edges_rows_and_phases(gll, d, eps):
    X = gaussian_points(300 + d, 400, d)
    S = Stage.from_graph(X, 90, 7, eps, seed=d)
    full = run_edges(gll, S)
    again = run_edges(gll, S)
    for a, b in zip(full, again):
        assert a.tobytes() == b.tobytes()
    ranges = [(0, 1), (1, 130), (130, S.n)]
    # phase 1 over all ranges, then phase 2 over all ranges == one call
    out = None
    for r in ranges:
        out = run_edges(gll, S, phases=1, rows=r, out=out)
    for r in ranges:
        out = run_edges(gll, S, phases=2, rows=r, out=out)
    for a, b in zip(full, out):
        assert a.tobytes() == b.tobytes()
    # one range at a time: phase 1 writes that range's edges and b rows only, phase 2 that range's dX rows only
    rp = S.row_ptr
    for lo, hi in ranges:
        gv, bvec, dX = run_edges(gll, S, phases=1, rows=(lo, hi))
        e = np.zeros(S.E, bool)
        e[rp[lo]:rp[hi]] = True
        assert gv[e].tobytes() == full[0][e].tobytes() and np.isnan(gv[~e]).all()
        r = np.zeros(S.n, bool)
        r[lo:hi] = S.auto
        assert bvec[r].tobytes() == full[1][r].tobytes() and np.isnan(bvec[~r]).all()
        assert np.isnan(dX).all()
        dX0 = np.full((S.n, S.d), np.nan, np.float32)
        gv2, bvec2, dX2 = run_edges(gll, S, phases=2, rows=(lo, hi), out=(full[0], full[1], dX0))
        assert gv2.tobytes() == full[0].tobytes() and bvec2.tobytes() == full[1].tobytes()
        assert dX2[lo:hi].tobytes() == full[2][lo:hi].tobytes()
        assert np.isnan(dX2[:lo]).all() and np.isnan(dX2[hi:]).all()


# ----------------------------------------------------------------------------------------------------------------
# 5. the fused driver runs exactly the stage
# ----------------------------------------------------------------------------------------------------------------
def _state_stage(torch, st, Xc, l, Y):
    """The layer's state as a Stage (its own fp32 arrays; the wt head poisoned) plus its raw ut / wt."""
    n, k_lab, lp = st.n, st.k_lab, (l + 3) // 4 * 4
    row_ptr = st.view("row_ptr", torch.int32, n + 1).cpu().numpy()
    E = int(row_ptr[-1])
    col = st.view("col", torch.int32, E).cpu().numpy()
    dist = st.view("dist", torch.float32, E).cpu().numpy()
    w = st.view("w", torch.float32, E).cpu().numpy()
    eps = st.view("eps", torch.float32, n).cpu().numpy()
    kappa = st.view("kappa", torch.int32, n).cpu().numpy() if st.eps_auto else None
    ut = st.view("ut", torch.float32, n * lp).reshape(n, lp).cpu().numpy()
    wt = st.view("wt", torch.float32, n * lp).reshape(n, lp).cpu().numpy()
    S = Stage(Xc.cpu().numpy(), row_ptr, col, dist, w, eps, kappa, k_lab, l, Y=Y)
    S.ut = ut.copy()
    S.wt = wt.copy()
    S.wt[:k_lab] = np.nan
    S.ref = edge_ref(row_ptr, col, dist, w, eps, kappa, S.ut, S.wt, k_lab)
    return S, ut, wt


@pytest.mark.gpu
@pytest.mark.parametrize("eps,tau", [("auto", 0.0), (1.0, 0.07)])
@pytest.mark.parametrize("path,code", [("streaming", 0), ("resident", 1), ("small", 2), ("cluster", 3)])
def test_fused_backward_is_the_stage(gll, monkeypatch, path, code, eps, tau):
    torch, pkg, _lib, _ = gll
    from graphlearninglayer_b200 import GLL

    monkeypatch.setenv("GLL_B200_CG_PATH", path)
    k_lab, m, d, l = 200, 400, 64, 10
    n = k_lab + m
    hint = np.float32(1.2) * np.float32(K - 1) * np.float32(m) / np.float32(n)  # api.cu uu_degree_hint
    assert _lib.lib.gll_cg_kernel(m, l, float(hint)) == code
    X, Y, *_ = O.synth_inputs(61, k_lab, m, d, l, 2.0)
    pred, st, Xc = GLL._forward_impl(torch.as_tensor(X).cuda(), torch.as_tensor(Y).cuda(), tau, eps)
    g = np.random.default_rng(3).standard_normal((m, l))
    dX = GLL._backward_impl(st, Xc, torch.as_tensor(g).cuda()).cpu().numpy()
    S, ut, wt = _state_stage(torch, st, Xc, l, Y)
    assert np.array_equal(ut[:k_lab, :l], Y)
    assert np.all(ut[:, l:] == 0) and np.all(wt[k_lab:, l:] == 0)  # K5 reads all lp columns
    assert np.isfinite(ut).all() and np.isfinite(wt[k_lab:]).all()
    gv, bvec, dX2 = run_edges(gll, S)
    assert dX2.tobytes() == dX.tobytes()
    case = f"layer cg={path} eps={eps}"
    check_k5(S, gv, bvec, case)
    check_k6(S, gv, bvec, dX, case)


# ----------------------------------------------------------------------------------------------------------------
# 6. float32 predictions
# ----------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("eps,tau", [("auto", 0.0), (1.0, 0.07)])
def test_float32_predictions_and_gradients(gll, monkeypatch, eps, tau):
    """pred in float32 is the float64 pred's fp32 solution; a grad_output that fp32 represents gives the same dX whether it
    comes as float32 or float64 (both are rounded to the same fp32 right-hand side)."""
    torch, pkg, _, _ = gll
    X, Y, *_ = O.synth_inputs(71, 150, 450, 48, 7, 2.0)
    g32 = np.random.default_rng(4).standard_normal((450, 7)).astype(np.float32)
    res = {}
    for dt, gnp in (("float64", g32.astype(np.float64)), ("float32", g32)):
        monkeypatch.setenv("GLL_B200_PRED_DTYPE", dt)
        Xt = torch.as_tensor(X).cuda().requires_grad_(True)
        pred = pkg.LaplaceLearningSparseHard.apply(Xt, torch.as_tensor(Y).cuda(), tau, eps)
        assert pred.dtype == getattr(torch, dt)
        g = torch.as_tensor(gnp).cuda()
        assert g.dtype == pred.dtype
        pred.backward(g)
        torch.cuda.synchronize()
        res[dt] = (pred.detach(), Xt.grad.clone())
    assert torch.equal(res["float32"][0], res["float64"][0].float())
    assert torch.equal(res["float32"][1], res["float64"][1])


# ----------------------------------------------------------------------------------------------------------------
# 7. the normalisation pair
# ----------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("d", [1, 31, 32, 33, 513, 2048])
def test_normalize_rows_pair_vs_torch_fp64(gll, d):
    """One warp per row, eight rows per CTA: n = 77 leaves a partial last CTA.  Rows: zero and |x| = 1e-13 (both clamped at
    eps = 1e-12: inv_norm carries the sign bit, dx = dxn / eps), |x| = 1e-11 and |x| = 1e30."""
    torch, _, _lib, dev_t = gll
    n = 77
    rng = np.random.default_rng(d)
    X = rng.standard_normal((n, d)) * rng.uniform(0.1, 10.0, size=(n, 1))
    unit = lambda v: v / np.linalg.norm(v)
    scaled = {1: 0.0, 2: 1e-13, 3: 1e-11, 4: 1e30, n - 1: 1e-13, n - 2: 1e30, n - 3: 0.0}
    for r, s in scaled.items():
        X[r] = s * unit(X[r])
    X = X.astype(np.float32)
    G = rng.standard_normal((n, d)).astype(np.float32)
    clamped = np.linalg.norm(X.astype(np.float64), axis=1) <= 1e-12
    assert clamped.sum() == 4
    f32 = torch.float32
    Xd, Gd = dev_t(X, f32), dev_t(G, f32)
    xn = torch.empty_like(Xd)
    inv = torch.empty(n, dtype=f32, device="cuda")
    dx = torch.empty_like(Xd)
    s = torch.cuda.current_stream().cuda_stream
    _lib.check(_lib.lib.gll_normalize_rows(Xd.data_ptr(), n, d, C.c_float(1e-12), xn.data_ptr(), inv.data_ptr(), s), "normalize")
    _lib.check(_lib.lib.gll_normalize_rows_backward(xn.data_ptr(), inv.data_ptr(), Gd.data_ptr(), n, d, dx.data_ptr(), s),
               "normalize backward")
    torch.cuda.synchronize()
    xn, inv, dx = xn.cpu().numpy().astype(np.float64), inv.cpu().numpy(), dx.cpu().numpy().astype(np.float64)
    x64 = torch.as_tensor(X.astype(np.float64)).requires_grad_(True)
    ref = torch.nn.functional.normalize(x64, dim=1, eps=1e-12)
    ref.backward(torch.as_tensor(G.astype(np.float64)))
    ref, ref_dx = ref.detach().numpy(), x64.grad.numpy()
    within(f"normalize d={d} xn", np.abs(xn - ref), 4 * U * np.abs(ref))
    assert np.array_equal(np.signbit(inv), clamped)
    # dx = (g - xn_f <xn_f, g>) inv_f from the ROUNDED xn_f = xn (1 + th)(1 + de_c) and inv_f = inv (1 + th), |th| <= 2u,
    # |de_c| <= u.  The per-element de_c do not cancel in the dot product: they cost u |xn_c| sum_k |xn_k g_k|, which can be
    # ~sqrt(d) times |xn_c| |<xn, g>|.  The common th enters three times and <xn, g> is rounded once; subtraction and
    # product round once each:  |dx - ref| <= u inv (4 |g| + 10 |xn| |<xn, g>| + |xn| sum_k |xn_k g_k|)   (first order)
    G64 = G.astype(np.float64)
    inv_ref = 1.0 / np.maximum(np.linalg.norm(X.astype(np.float64), axis=1), 1e-12)
    proj = np.abs(ref) * np.abs(np.einsum("ij,ij->i", ref, G64))[:, None]
    dot_abs = np.abs(ref) * np.einsum("ij,ij->i", np.abs(ref), np.abs(G64))[:, None]
    within(f"normalize d={d} dx", np.abs(dx - ref_dx), U * (4 * np.abs(G64) + 10 * proj + dot_abs) * inv_ref[:, None])
    within(f"normalize d={d} dx clamped", np.abs(dx[clamped] - G64[clamped] / 1e-12), 4 * U * np.abs(G64[clamped]) / 1e-12)
