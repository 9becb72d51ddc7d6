"""poisson_learning (gll_poisson_eval): Poisson learning of T labeled sets on one graph -- L u = b on all n rows with the centred
source of each trial's labeled rows, u with zero degree-weighted mean per class column.

Without a GPU: the exports, the C argument checks (they return before any CUDA call), the Python validation, and a numpy model
of the PoissonRows policy (its residual against scipy, its centred solution against the bordered system) and of the GLL_LAPLACE_*
schedule on the singular system.  On a GPU: every trial against an fp64 host reference on the device's own W, eps auto and
fixed, l = 8 and 37, the chunked CG (T lpad > 128) and every on-chip CG kernel, trial slices against T = 1 calls, a zero source,
an invalid trial next to valid ones, determinism and CUDA-graph replay, the max-iteration warning and an inconsistent source on a
graph of two far-apart clusters.
"""
import ctypes
import inspect
import os
import re
import warnings

import numpy as np
import pytest
import scipy.sparse as sp
import scipy.sparse.linalg as spla

from oracle import gll_oracle as O

torch = pytest.importorskip("torch")

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ERR_ARG = -1


@pytest.fixture(scope="module")
def libmod():
    from graphlearninglayer_b200 import build

    build.build()
    from graphlearninglayer_b200 import _lib

    return _lib


@pytest.fixture(scope="module")
def gpu(libmod):
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    torch.cuda.set_device(0)
    import graphlearninglayer_b200 as pkg

    return pkg


# ---------------------------------------------------------------------------------------------------- without a GPU
def test_signature_and_exports(libmod):
    import graphlearninglayer_b200 as pkg
    from graphlearninglayer_b200 import laplace_eval

    sig = inspect.signature(pkg.poisson_learning)
    assert list(sig.parameters) == ["features", "train_idx", "label_matrix", "k", "epsilon", "tol", "targets"]
    d = {p.name: p.default for p in sig.parameters.values()}
    assert d["k"] == 50 and d["epsilon"] == "auto" and d["tol"] == 1e-10 and d["targets"] is None
    assert "poisson_learning" in pkg.__all__ and "poisson_learning" in laplace_eval.__all__
    assert pkg.poisson_learning is laplace_eval.poisson_learning
    raw = ctypes.CDLL(libmod.LIB_PATH)
    for nm in ("gll_poisson_eval_workspace_bytes", "gll_poisson_eval"):
        assert hasattr(raw, nm) and nm in libmod.EXPORTS
        assert re.search(r"\b%s\(" % nm, open(os.path.join(ROOT, "include", "gll_b200.h")).read())
    names = libmod.kernel_names()
    assert names[-2:] == ["poisson_mean", "poisson_center"]
    assert names.index("laplace_trials_setup") == len(names) - 3  # existing ids keep their values


def test_c_argument_checks(libmod):
    lib = libmod.lib
    buf = ctypes.c_void_p(16)  # never dereferenced: the checks fail first

    def call(X=buf, n=300, d=8, k=50, idx=buf, Y=buf, T=4, k_lab=30, l=3, tol=1e-10, maxit=100, pred=buf, labels=buf, info=buf, ws=buf):
        return lib.gll_poisson_eval(X, n, d, k, idx, 1, Y, T, k_lab, l, 1, 0.0, tol, maxit, pred, labels, None, None, None, info, ws,
                                    1 << 30, None)

    bad = (dict(X=None), dict(idx=None), dict(Y=None), dict(pred=None), dict(labels=None), dict(info=None), dict(ws=None),
           dict(T=0), dict(n=1 << 20, T=1 << 10, l=3),
           dict(k=1), dict(k=65), dict(n=40, k=41, k_lab=10), dict(n=255, k=34),
           dict(k_lab=0), dict(k_lab=300), dict(l=0), dict(d=0),
           dict(tol=0.0), dict(tol=-1.0), dict(maxit=0),
           dict(T=1 << 19, l=4), dict(n=40, k=20, k_lab=10, T=1 << 16, l=33))
    for kw in bad:
        assert call(**kw) == ERR_ARG, kw
    wsb = lib.gll_poisson_eval_workspace_bytes  # (n, d, k, l, T, k_lab)
    for args in ((300, 8, 50, 3, 0, 30), (1 << 20, 8, 25, 3, 1 << 10, 30), (300, 8, 1, 3, 4, 30), (300, 8, 65, 3, 4, 30),
                 (40, 8, 41, 3, 4, 10), (255, 8, 34, 3, 4, 10), (300, 8, 50, 3, 4, 0), (300, 8, 50, 3, 4, 300),
                 (300, 8, 50, 0, 4, 30), (300, 0, 50, 3, 4, 30), (300, 8, 50, 4, 1 << 19, 30), (40, 8, 20, 33, 1 << 16, 10)):
        assert wsb(*args) == 0, args
    for args in ((300, 8, 50, 3, 4, 30), (2000, 64, 50, 37, 4, 74), (40, 8, 20, 1, 65535 * 32, 10)):
        # the trials' buffers plus the source means, the column means and a second half of the refinement partials
        assert wsb(*args) > lib.gll_laplace_eval_trials_workspace_bytes(*args) > 0, args


@pytest.mark.parametrize("kwargs, exc, match", [
    (dict(), RuntimeError, "no CPU path"),
    (dict(X=torch.zeros(2, 300, 8)), ValueError, "features"), (dict(I=torch.zeros(30, dtype=torch.long)), ValueError, "train_idx"),
    (dict(I=torch.zeros(2, 30)), ValueError, "int64 or int32"), (dict(Y=torch.zeros(30, 3)), ValueError, "label_matrix"),
    (dict(Y=torch.zeros(2, 29, 3)), ValueError, "label_matrix"),
    (dict(I=torch.zeros(0, 30, dtype=torch.long), Y=torch.zeros(0, 30, 3)), ValueError, "T >= 1"),
    (dict(k=1), ValueError, "k must be"), (dict(X=torch.zeros(200, 8), k=34), ValueError, "n >= 256"),
    (dict(I=torch.zeros(2, 300, dtype=torch.long), Y=torch.zeros(2, 300, 3)), ValueError, "k_lab"),
    (dict(Y=torch.zeros(2, 30, 0)), ValueError, "class column"), (dict(epsilon="knn"), ValueError, "epsilon"),
    (dict(tol=0.0), ValueError, "tol"), (dict(targets=torch.zeros(270, dtype=torch.long)), ValueError, "targets"),
    (dict(I=torch.zeros(1, 30, dtype=torch.long).expand(1 << 19, 30), Y=torch.zeros(1, 30, 4).expand(1 << 19, 30, 4)), ValueError,
     "T l must be")])
def test_python_validation_before_any_device_call(libmod, kwargs, exc, match):
    import graphlearninglayer_b200 as pkg

    X = kwargs.pop("X", torch.zeros(300, 8))  # CPU tensors: every argument check must come first
    idx = kwargs.pop("I", torch.zeros(2, 30, dtype=torch.long))
    Y = kwargs.pop("Y", torch.zeros(2, 30, 3))
    with pytest.raises(exc, match=match):
        pkg.poisson_learning(X, idx, Y, **kwargs)


# ---------------------------------------------------------------------------------------------------- model of the policy
def schedule():
    text = open(os.path.join(ROOT, "include", "gll_b200.h")).read()

    def val(name):
        return float(re.search(r"#define\s+%s\s+(\S+)" % name, text).group(1))

    return int(val("GLL_LAPLACE_ROUNDS")), val("GLL_LAPLACE_CG_RTOL0"), val("GLL_LAPLACE_CG_RTOL")


def poisson_source(idx, Ys, n):
    """b (T, n, l): row idx[t, s] of trial t gets Y[t, s] - mean_s Y[t, s], every other row 0"""
    T, _, l = Ys.shape
    b = np.zeros((T, n, l))
    Y = Ys.astype(np.float64)
    for t in range(T):
        b[t, idx[t]] = Y[t] - Y[t].mean(axis=0)
    return b


def policy_residual(W, dg, idx, Ys, x):
    """PoissonRows' residual as laplace_refine forms it, row by row: r_i = b_i + sum_j w_ij (x_j - x_i), b_i from the slot table,
    Y and ybar (x: (T, n, l))"""
    T, k_lab, l = Ys.shape
    n = W.shape[0]
    slot = -np.ones((n, T), dtype=np.int64)
    for t in range(T):
        slot[idx[t], t] = np.arange(k_lab)
    ybar = Ys.astype(np.float64).mean(axis=1)
    r = np.zeros_like(x)
    for i in range(n):
        js, ws = W.indices[W.indptr[i]:W.indptr[i + 1]], W.data[W.indptr[i]:W.indptr[i + 1]]
        for t in range(T):
            s = (ws[:, None] * (x[t, js] - x[t, i])).sum(axis=0)
            if slot[i, t] >= 0:
                s = s + (Ys[t, slot[i, t]].astype(np.float64) - ybar[t])
            r[t, i] = s
    return r


def bordered_solve(W, b):
    """the centred solution of L u = b: [[L, D 1], [(D 1)^T, 0]] [u; lam] = [b; 0] (b: (n, l))"""
    n = W.shape[0]
    dg = np.asarray(W.sum(axis=1)).ravel()
    L = sp.diags(dg) - W
    K = sp.bmat([[L, sp.csr_matrix(dg[:, None])], [sp.csr_matrix(dg[None, :]), None]]).tocsc()
    sol = spla.splu(K).solve(np.vstack([b, np.zeros((1, b.shape[1]))]))
    return sol[:n], sol[n]


def pcg(W, dg, b, rel, f32=True, maxit=5000):
    """cg_run's Jacobi-PCG without a mask on the full-graph system (per-column step lengths, fp64 dots): x (n, C), iterations"""
    ft = np.float32 if f32 else np.float64
    Wf, dgf = W.astype(ft), dg.astype(ft)
    dinv = (ft(1) / dgf)[:, None]
    r = b.astype(ft)
    x = np.zeros_like(r)
    z = r * dinv
    p = z.copy()

    def dot(a, c):
        return np.einsum("ij,ij->j", a.astype(np.float64), c.astype(np.float64))

    rz, rr = dot(r, z), dot(r, r)
    tol2 = rel * rel * rr.max()
    it = 0
    while rr.max() > tol2 and it < maxit:
        it += 1
        ap = (dgf[:, None] * p - (Wf @ p).astype(ft)).astype(ft)
        pap = dot(p, ap)
        live = rr > tol2
        al = np.where(live, rz / np.where(pap != 0, pap, 1), 0).astype(ft)
        x = x + al * p
        r = r - al * ap
        z = r * dinv
        rzn, rrn = dot(r, z), dot(r, r)
        be = np.where((rrn > tol2) & (rz != 0), rzn / np.where(rz != 0, rz, 1), 0).astype(ft)
        p = z + be * p
        rz, rr = rzn, rrn
    return x.astype(np.float64), it


def refine_model(W, idx, Ys, rounds, rtol0, rtol, tol=1e-10):
    """gll_poisson_eval on the host: the first solve from laplace_refine's x = 0 pass, then `rounds` fp64 residual rounds with
    fp32 correction solves while a column is above tol, then the centring.  Returns (norms per round (T, l), iterations, u (T, n,
    l))."""
    W = sp.csr_matrix(W).astype(np.float32).astype(np.float64)
    n = W.shape[0]
    T, _, l = Ys.shape
    dg = np.asarray(W.sum(axis=1)).ravel()
    b = poisson_source(idx, Ys, n).transpose(1, 0, 2).reshape(n, T * l)
    x, it0 = pcg(W, dg, b, rtol0)
    e = np.zeros_like(x)
    norms, iters = [], [it0]
    for _ in range(rounds):
        x = x + e
        r = b - (dg[:, None] * x - W @ x)
        cn = np.sqrt((r * r / (dg[:, None] + 1e-10)).sum(axis=0)).reshape(T, l)
        norms.append(cn)
        if not cn.max() <= tol:
            e, it = pcg(W, dg, r, rtol)
        else:
            e, it = np.zeros_like(x), 0
        iters.append(it)
    u = x + e
    u = u - (dg @ u) / dg.sum()
    return norms, iters, u.reshape(n, T, l).transpose(1, 0, 2)


def model_data(seed, n=600, l=5, far=8, gap=0.7):
    """l Gaussian classes plus a small far cluster that reaches the rest only through weak edges (the smallest nonzero eigenvalue of
    D^-1/2 L D^-1/2 is about 1e-4).  The trials' model data puts that cluster 3.0 away, where its edges' weights (1e-18 and less)
    vanish next to fp32 rounding: for Poisson learning that graph is numerically two components, and a labeled row in the far
    cluster makes the source inconsistent (the disconnected case the header leaves unspecified)."""
    X, _, yb, yq = O.synth_inputs(seed, l, n - l - far, 16, l, 1.5)
    rng = np.random.default_rng(seed)
    X = np.concatenate([X, (X.mean(axis=0) + gap + 0.05 * rng.standard_normal((far, X.shape[1]))).astype(np.float32)])
    y = np.concatenate([yb, yq, np.zeros(far, dtype=np.int64)])
    return X, y


def draw_trials(seed, y, l, T, per_class):
    """T labeled sets of per_class rows of every class, one-hot labels"""
    rng = np.random.default_rng(seed)
    idx = np.stack([np.concatenate([rng.choice(np.flatnonzero(y == c), per_class, replace=False) for c in range(l)])
                    for t in range(T)])
    return idx.astype(np.int64), np.eye(l, dtype=np.float32)[y[idx]]


def test_policy_residual_and_centred_solution():
    X, y = model_data(3, n=300)
    W = sp.csr_matrix(O.build_graph(X, 20, "auto").W).astype(np.float32).astype(np.float64)
    n = W.shape[0]
    dg = np.asarray(W.sum(axis=1)).ravel()
    L = (sp.diags(dg) - W).tocsr()
    idx, Ys = draw_trials(4, y, 5, 3, 2)
    Ys[2] = Ys[2] * 0.5 + 0.1  # not one-hot
    b = poisson_source(idx, Ys, n)
    assert np.abs(b.sum(axis=1)).max() < 1e-14  # the centred source is consistent on a connected graph
    x = np.random.default_rng(5).standard_normal((3, n, 5))
    r = policy_residual(W, dg, idx, Ys, x)
    for t in range(3):
        np.testing.assert_allclose(r[t], b[t] - L @ x[t], rtol=1e-12, atol=1e-12)
    # the centred solution: L u = b, sum_i D_i u_i = 0, and it is the bordered system's solution with multiplier 0
    for t in range(3):
        u, lam = bordered_solve(W, b[t])
        assert np.abs(lam).max() < 1e-10
        assert np.abs(L @ u - b[t]).max() < 1e-10
        assert np.abs(dg @ u).max() < 1e-10 * (dg @ np.abs(u)).max()
        # any solution of L u = b, centred, is u
        v = spla.lsqr(L, b[t][:, 0], atol=1e-14, btol=1e-14, iter_lim=20000)[0] + 3.0
        v = v - (dg @ v) / dg.sum()
        assert O.max_rel(v, u[:, 0]) < 1e-6


@pytest.mark.parametrize("T", [1, 16, 64])
def test_refinement_meets_every_column_with_a_round_to_spare(T):
    rounds, rtol0, rtol = schedule()
    X, y = model_data(10 + T)
    W = O.build_graph(X, 20, "auto").W
    idx, Ys = draw_trials(T, y, 5, T, 2)
    norms, iters, u = refine_model(W, idx, Ys, rounds, rtol0, rtol)
    first = next((i for i, nv in enumerate(norms) if nv.max() <= 1e-10), None)
    assert first is not None and first <= rounds - 2, (T, [float(nv.max()) for nv in norms])
    assert all(it == 0 for it in iters[1 + first:])
    assert np.all(norms[first] <= 1e-10)  # every column of every trial
    if T == 16:  # the far cluster is labeled in some trials: the hard case is exercised
        assert np.isin(idx, np.arange(592, 600)).any()
    Wd = sp.csr_matrix(W).astype(np.float32).astype(np.float64)
    b = poisson_source(idx, Ys, X.shape[0])
    for t in range(min(T, 4)):
        ref, _ = bordered_solve(Wd, b[t])
        assert O.max_rel(u[t], ref) < 1e-6, t


# ---------------------------------------------------------------------------------------------------- on the GPU
def _data(seed, n, d, l, sigma=2.0):
    X, _, yb, yq = O.synth_inputs(seed, l, n - l, d, l, sigma)
    return X, np.concatenate([yb, yq]).astype(np.int64)


def _info():
    from graphlearninglayer_b200.laplace_eval import last_eval_info

    return last_eval_info()


def _run(pkg, X, idx, Ys, y=None, **kw):
    return pkg.poisson_learning(torch.as_tensor(X).cuda(), torch.as_tensor(idx).cuda(), torch.as_tensor(Ys).cuda(),
                                targets=None if y is None else torch.as_tensor(y).cuda(), **kw)


def _per_class(seed, y, l, T, per):
    rng = np.random.default_rng(seed)
    idx = np.stack([np.concatenate([rng.choice(np.flatnonzero(y == c), per, replace=False) for c in range(l)]) for _ in range(T)])
    return idx.astype(np.int64), np.eye(l, dtype=np.float32)[y[idx]]


def _check(pkg, X, idx, Ys, y, k, eps, res, trials=None):
    """every trial against the bordered fp64 solve on the device's own W: stop rule, centring, values, labels, hits"""
    n = X.shape[0]
    W = sp.csr_matrix(pkg.knn_sym_dist(X, k, eps)[0]).astype(np.float64)
    dg = np.asarray(W.sum(axis=1)).ravel()
    L = (sp.diags(dg) - W).tocsr()
    pred, labels = res.pred.cpu().numpy(), res.labels.cpu().numpy()
    correct = None if res.correct is None else res.correct.cpu().numpy()
    resid = _info()["resid_per_trial"]
    for t in (range(idx.shape[0]) if trials is None else trials):
        b = poisson_source(idx[t:t + 1], Ys[t:t + 1], n)  # trial t only: an invalid trial's indices may be out of range
        r = b[0] - L @ pred[t]
        assert np.all(np.sqrt((r * r / (dg[:, None] + 1e-10)).sum(axis=0)) <= 1e-10 * (1 + 1e-6)), t
        assert resid[t] <= 1e-10, (t, resid[t])
        assert np.all(np.abs(dg @ pred[t]) <= 1e-12 * (dg @ np.abs(pred[t]))), t
        ref, _ = bordered_solve(W, b[0])
        err = O.max_rel(pred[t], ref)
        assert err <= 1e-6, (t, err)
        top = np.sort(ref, axis=1)
        sure = top[:, -1] - top[:, -2] > 2 * err * np.abs(ref).max()
        assert np.array_equal(labels[t][sure], ref.argmax(axis=1)[sure]), t
        if correct is not None:
            unl = np.setdiff1d(np.arange(n), idx[t])
            hits = int((labels[t, unl] == y[unl]).sum())
            assert int(correct[t]) == hits, t


# (n, per class, d, l, T), (eps, CG path)
SHAPES = [((3000, 1, 64, 10, 8), ("auto", "")), ((3000, 3, 64, 8, 8), (1.0, "")), ((2000, 1, 64, 10, 64), ("auto", "")),
          ((1500, 2, 32, 37, 4), ("auto", "")),
          ((400, 2, 16, 4, 2), ("auto", "small")), ((1200, 2, 16, 4, 4), ("auto", "cluster")),
          ((1200, 2, 16, 4, 4), ("auto", "resident")), ((1200, 2, 16, 4, 4), ("auto", "streaming"))]


@pytest.mark.gpu
@pytest.mark.parametrize("shape, et", SHAPES, ids=["3000x8-auto", "3000x8-l8-eps1", "2000x64-chunked", "1500x4-l37-chunked",
                                                   "400-small", "1200-cluster", "1200-resident", "1200-streaming"])
def test_trials_match_the_bordered_fp64_solve(gpu, shape, et, monkeypatch):
    n, per, d, l, T = shape
    eps, path = et
    if path:
        monkeypatch.setenv("GLL_B200_CG_PATH", path)
    X, y = _data(n + T, n, d, l)
    idx, Ys = _per_class(T, y, l, T, per)
    k = 50 if n >= 1000 else 20
    res = _run(gpu, X, idx, Ys, y, k=k, epsilon=eps)
    torch.cuda.synchronize()
    assert res.pred.shape == (T, n, l) and res.pred.dtype == torch.float64
    assert res.labels.shape == (T, n) and res.correct.shape == (T,) and res.correct.dtype == torch.int64
    info = _info()
    assert info["status"] & ~8 == 0 and info["resid"] <= 1e-10 and len(info["resid_per_trial"]) == T
    _check(gpu, X, idx, Ys, y, k, eps, res)


@pytest.mark.gpu
def test_a_trial_equals_a_one_trial_call(gpu):
    X, y = _data(7, 2000, 64, 10)
    idx, Ys = _per_class(8, y, 10, 6, 2)
    res = _run(gpu, X, idx, Ys, y)
    for t in (0, 5):
        one = _run(gpu, X, idx[t:t + 1], Ys[t:t + 1], y)
        torch.cuda.synchronize()
        a, b = res.pred[t].cpu().numpy(), one.pred[0].cpu().numpy()
        err = O.max_rel(a, b)
        assert err < 1e-6, t
        top = np.sort(b, axis=1)
        sure = top[:, -1] - top[:, -2] > 2 * err * np.abs(b).max()
        assert np.array_equal(res.labels[t].cpu().numpy()[sure], one.labels[0].cpu().numpy()[sure])
        flips = int((res.labels[t] != one.labels[0]).sum())
        assert abs(int(res.correct[t]) - int(one.correct[0])) <= flips


@pytest.mark.gpu
def test_zero_source_and_invalid_trials(gpu, monkeypatch):
    n, l = 1500, 5
    X, y = _data(9, n, 32, l)
    idx, Ys = _per_class(10, y, l, 5, 2)
    Ys[1] = np.eye(l, dtype=np.float32)[3]  # every labeled row of trial 1 has label 3: b = 0
    idx[3, 4] = idx[3, 1]  # a repeat
    idx[4, 0] = n  # out of range
    monkeypatch.setenv("GLL_B200_CHECK", "1")
    with warnings.catch_warnings(record=True) as rec:
        warnings.simplefilter("always")
        res = _run(gpu, X, idx, Ys, y)
        torch.cuda.synchronize()
    assert any("labeled-row indices" in str(w.message) for w in rec)
    info = _info()
    assert info["status"] & 16 and info["status"] & 1 == 0
    pred, labels, correct = res.pred.cpu().numpy(), res.labels.cpu().numpy(), res.correct.cpu().numpy()
    assert np.all(pred[1] == 0.0) and np.all(labels[1] == 0) and info["resid_per_trial"][1] == 0.0
    for t in (3, 4):
        assert np.all(np.isnan(pred[t])) and np.all(labels[t] == -1) and correct[t] == -1
        assert np.isnan(info["resid_per_trial"][t])
    _check(gpu, X, idx, Ys, y, 50, "auto", res, trials=[0, 2])
    alone = _run(gpu, X, idx[[0, 2]], Ys[[0, 2]], y)
    torch.cuda.synchronize()
    assert O.max_rel(pred[[0, 2]], alone.pred.cpu().numpy()) < 1e-6


@pytest.mark.gpu
def test_deterministic_and_graph_capturable(gpu):
    n, l = 2000, 10
    X, y = _data(11, n, 64, l)
    X2, _ = _data(12, n, 64, l)
    idx, Ys = _per_class(13, y, l, 16, 1)  # T lpad = 192: the chunked solve
    Xt, It, Yt, tt = (torch.as_tensor(v).cuda() for v in (X, idx, Ys, y))
    a = gpu.poisson_learning(Xt, It, Yt, targets=tt)
    b = gpu.poisson_learning(Xt, It, Yt, targets=tt)
    ref = gpu.poisson_learning(torch.as_tensor(X2).cuda(), It, Yt, targets=tt)
    torch.cuda.synchronize()
    assert torch.equal(a.pred, b.pred) and torch.equal(a.labels, b.labels) and torch.equal(a.correct, b.correct)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        gpu.poisson_learning(Xt, It, Yt, targets=tt)
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        c = gpu.poisson_learning(Xt, It, Yt, targets=tt)
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(c.pred, a.pred) and torch.equal(c.labels, a.labels) and torch.equal(c.correct, a.correct)
    Xt.copy_(torch.as_tensor(X2).cuda())  # replay on new inputs
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(c.pred, ref.pred) and torch.equal(c.labels, ref.labels) and torch.equal(c.correct, ref.correct)


@pytest.mark.gpu
def test_max_iter_warning(gpu, monkeypatch):
    X, y = _data(14, 1000, 64, 10)
    idx, Ys = _per_class(15, y, 10, 4, 1)
    monkeypatch.setenv("GLL_B200_CG_MAXIT", "1")
    monkeypatch.setenv("GLL_B200_CHECK", "1")
    with warnings.catch_warnings(record=True) as rec:
        warnings.simplefilter("always")
        _run(gpu, X, idx, Ys)
        torch.cuda.synchronize()
    assert any("max iter reached" in str(w.message) for w in rec)
    info = _info()
    assert info["status"] & 1 and max(info["resid_per_trial"]) > 1e-10


@pytest.mark.gpu
def test_inconsistent_source_on_two_components_warns(gpu, monkeypatch):
    """two clusters far apart (no edge between them), class 0 labeled in one and class 1 in the other: neither component's source
    sums to zero"""
    rng = np.random.default_rng(16)
    X = np.concatenate([rng.standard_normal((300, 8)), 1000.0 + rng.standard_normal((300, 8))]).astype(np.float32)
    idx = np.array([[0, 1, 300, 301]], dtype=np.int64)
    Ys = np.eye(2, dtype=np.float32)[[0, 0, 1, 1]][None]
    monkeypatch.setenv("GLL_B200_CHECK", "1")
    with warnings.catch_warnings(record=True) as rec:
        warnings.simplefilter("always")
        res = _run(gpu, X, idx, Ys, k=10)
        torch.cuda.synchronize()
    assert any("max iter reached" in str(w.message) or "non-finite" in str(w.message) for w in rec)
    assert _info()["status"] & (1 | 4)
    assert res.pred.shape == (1, 600, 2)
