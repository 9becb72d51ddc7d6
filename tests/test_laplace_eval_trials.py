"""laplace_learning_trials (gll_laplace_eval_trials): T labeled sets on one graph, solved against one full-graph system with each
trial's labeled rows masked out of its own class columns.

Without a GPU: the exports, the C argument checks (they return before any CUDA call), the Python validation, and a numpy model of
the masked formulation -- the masked operator against each trial's compact L_uu + tau I, the masked CG against the compact one,
and the GLL_LAPLACE_* refinement schedule on the masked fp32 solves.  On a GPU: every trial against laplace_learning on the
permuted features and against the reference's stop rule recomputed on the host, the chunked solve (T lpad > 128), T = 1 against
laplace_learning, overlapping and repeated labeled sets, invalid trials next to valid ones, determinism and CUDA-graph replay, and
the max-iteration warning.
"""
import ctypes
import inspect
import os
import re
import warnings

import numpy as np
import pytest
import scipy.sparse as sp

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

    sig = inspect.signature(pkg.laplace_learning_trials)
    assert list(sig.parameters) == ["features", "train_idx", "label_matrix", "k", "epsilon", "tau", "tol", "targets"]
    d = {p.name: p.default for p in sig.parameters.values()}
    assert d["k"] == 50 and d["epsilon"] == "auto" and d["tau"] == 0.0 and d["tol"] == 1e-10 and d["targets"] is None
    assert "laplace_learning_trials" in pkg.__all__
    raw = ctypes.CDLL(libmod.LIB_PATH)
    for nm in ("gll_laplace_eval_trials_workspace_bytes", "gll_laplace_eval_trials"):
        assert hasattr(raw, nm) and nm in libmod.EXPORTS
    assert "laplace_trials_setup" in libmod.kernel_names()
    text = open(os.path.join(ROOT, "include", "gll_b200.h")).read()
    assert int(re.search(r"#define\s+GLL_STATUS_BAD_INDEX\s+(\d+)", text).group(1)) == libmod.STATUS_BAD_INDEX == 16


def test_c_argument_checks(libmod):
    lib = libmod.lib
    buf = ctypes.c_void_p(16)  # never dereferenced: the checks fail first

    def call(X=buf, n=300, d=8, k=50, idx=buf, Y=buf, T=4, k_lab=30, l=3, tol=1e-10, maxit=100, pred=buf, labels=buf, info=buf, ws=buf):
        return lib.gll_laplace_eval_trials(X, n, d, k, idx, 1, Y, T, k_lab, l, 1, 0.0, 0.0, tol, maxit, pred, labels, None, None, None,
                                           info, ws, 1 << 30, None)

    bad = (dict(X=None), dict(idx=None), dict(Y=None), dict(pred=None), dict(labels=None), dict(info=None), dict(ws=None),
           dict(T=0), dict(n=1 << 20, T=1 << 10, l=3),                              # T >= 1, n T lpad < 2^31
           dict(k=1), dict(k=65), dict(n=40, k=41, k_lab=10), dict(n=255, k=34),   # 2 <= k <= 64, k <= n, n >= 256 when k > 33
           dict(k_lab=0), dict(k_lab=300), dict(l=0), dict(d=0),                    # 1 <= k_lab < n, l >= 1, d >= 1
           dict(tol=0.0), dict(tol=-1.0), dict(maxit=0),                            # tol > 0, cg_max_iter >= 1
           dict(T=1 << 19, l=4), dict(n=40, k=20, k_lab=10, T=1 << 16, l=33))      # T l <= 65535 * 32 (refinement grid)
    for kw in bad:
        assert call(**kw) == ERR_ARG, kw
    wsb = lib.gll_laplace_eval_trials_workspace_bytes  # (n, d, k, l, T, k_lab)
    for args in ((300, 8, 50, 3, 0, 30), (1 << 20, 8, 25, 3, 1 << 10, 30), (300, 8, 1, 3, 4, 30), (300, 8, 65, 3, 4, 30),
                 (40, 8, 41, 3, 4, 10), (255, 8, 34, 3, 4, 10), (300, 8, 50, 3, 4, 0), (300, 8, 50, 3, 4, 300),
                 (300, 8, 50, 0, 4, 30), (300, 0, 50, 3, 4, 30), (300, 8, 50, 4, 1 << 19, 30), (40, 8, 20, 33, 1 << 16, 10)):
        assert wsb(*args) == 0, args
    assert wsb(300, 8, 50, 3, 4, 30) > 0 and wsb(2000, 64, 50, 37, 4, 74) > 0
    assert wsb(40, 8, 20, 32, 65535, 10) > 0 and wsb(40, 8, 20, 1, 65535 * 32, 10) > 0  # T l = 65535 * 32 is accepted


@pytest.mark.parametrize("kwargs, exc, match", [
    (dict(), RuntimeError, "no CPU path"),
    (dict(X=torch.zeros(2, 300, 8)), ValueError, "features"), (dict(I=torch.zeros(30, dtype=torch.long)), ValueError, "train_idx"),
    (dict(I=torch.zeros(2, 30)), ValueError, "int64 or int32"), (dict(Y=torch.zeros(30, 3)), ValueError, "label_matrix"),
    (dict(Y=torch.zeros(3, 30, 3)), ValueError, "label_matrix"), (dict(Y=torch.zeros(2, 29, 3)), ValueError, "label_matrix"),
    (dict(I=torch.zeros(0, 30, dtype=torch.long), Y=torch.zeros(0, 30, 3)), ValueError, "T >= 1"),
    (dict(k=1), ValueError, "k must be"), (dict(k=65), ValueError, "k must be"),
    (dict(X=torch.zeros(200, 8), k=34), ValueError, "n >= 256"),
    (dict(I=torch.zeros(2, 0, dtype=torch.long), Y=torch.zeros(2, 0, 3)), ValueError, "k_lab"),
    (dict(I=torch.zeros(2, 300, dtype=torch.long), Y=torch.zeros(2, 300, 3)), ValueError, "k_lab"),
    (dict(Y=torch.zeros(2, 30, 0)), ValueError, "class column"), (dict(epsilon="knn"), ValueError, "epsilon"),
    (dict(tol=0.0), ValueError, "tol"), (dict(targets=torch.zeros(270, dtype=torch.long)), ValueError, "targets"),
    (dict(targets=torch.zeros(2, 300, dtype=torch.long)), ValueError, "targets"),
    (dict(I=torch.zeros(1, 30, dtype=torch.long).expand(1 << 19, 30), Y=torch.zeros(1, 30, 4).expand(1 << 19, 30, 4)), ValueError,
     "T l must be")])
def test_python_validation_before_any_device_call(libmod, kwargs, exc, match):
    import graphlearninglayer_b200 as pkg

    X = kwargs.pop("X", torch.zeros(300, 8))  # CPU tensors: every argument check must come first
    idx = kwargs.pop("I", torch.zeros(2, 30, dtype=torch.long))
    Y = kwargs.pop("Y", torch.zeros(2, 30, 3))
    with pytest.raises(exc, match=match):
        pkg.laplace_learning_trials(X, idx, Y, **kwargs)


# ---------------------------------------------------------------------------------------------------- model of the masked solve
def schedule():
    text = open(os.path.join(ROOT, "include", "gll_b200.h")).read()

    def val(name):
        return float(re.search(r"#define\s+%s\s+(\S+)" % name, text).group(1))

    return int(val("GLL_LAPLACE_ROUNDS")), val("GLL_LAPLACE_CG_RTOL0"), val("GLL_LAPLACE_CG_RTOL")


def masked_system(W, idx, Ys, tau):
    """The trials' full-graph system in the device's column layout: dg = row-sum degree + tau, b (n, T lpad) = W_ul Y per trial,
    clamp (n, T lpad) = row labeled in the column's trial.  Padding columns are zero and never clamped."""
    W = sp.csr_matrix(W).astype(np.float32).astype(np.float64)
    n = W.shape[0]
    T, k_lab = idx.shape
    l = Ys.shape[2]
    lpad = (l + 3) // 4 * 4
    dg = np.asarray(W.sum(axis=1)).ravel() + tau
    b = np.zeros((n, T * lpad))
    clamp = np.zeros((n, T * lpad), dtype=bool)
    for t in range(T):
        b[:, t * lpad:t * lpad + l] = W[:, idx[t]] @ Ys[t].astype(np.float64)
        clamp[idx[t], t * lpad:(t + 1) * lpad] = True
    b[clamp] = 0.0
    return W, dg, b, clamp, lpad


def masked_pcg(W, diag, b, clamp, rel=None, iters=None, f32=True, chunk=128):
    """The streaming kernel's masked Jacobi-PCG: per-column step lengths and freeze, A p zeroed on clamped entries, fp64 dots;
    chunks of `chunk` columns, each with its own relative tolerance rel * (largest column norm of the chunk's b).  iters: a fixed
    number of iterations instead.  Returns (x, iterations per chunk)."""
    ft = np.float32 if f32 else np.float64
    Wf, dgf = W.astype(ft), diag.astype(ft)
    x = np.zeros(b.shape, dtype=ft)
    its = []
    for c0 in range(0, b.shape[1], chunk):
        cs = slice(c0, c0 + chunk)
        mask = clamp[:, cs]
        r = b[:, cs].astype(ft)
        dinv = (ft(1) / dgf)[:, None]
        z = r * dinv
        p = z.copy()
        xc = np.zeros_like(r)

        def dot(a, c):
            return np.einsum("ij,ij->j", a.astype(np.float64), c.astype(np.float64))

        rz, rr = dot(r, z), dot(r, r)
        tol2 = 0.0 if rel is None else rel * rel * rr.max()
        it = 0
        while (rr.max() > tol2 and it < 5000) if iters is None else it < iters:
            it += 1
            ap = (dgf[:, None] * p - (Wf @ p).astype(ft)).astype(ft)
            ap[mask] = 0
            pap = dot(p, ap)
            live = rr > tol2
            al = np.where(live, rz / np.where(pap != 0, pap, 1), 0).astype(ft)
            xc = xc + al * p
            r = r - al * ap
            z = r * dinv
            rzn, rrn = dot(r, z), dot(r, r)
            be = np.where((rrn > tol2) & (rz != 0), rzn / np.where(rz != 0, rz, 1), 0).astype(ft)
            p = z + be * p
            rz, rr = rzn, rrn
        x[:, cs] = xc
        its.append(it)
    return x, its


def refine_model_trials(W, idx, Ys, tau, rounds, rtol0, rtol, tol=1e-10):
    """gll_laplace_eval_trials on the host: fp64 residual r = b - A x on the unclamped entries, the scaled column norms of every
    round (T, l), correction solves while any column of any trial is above tol.  Returns (norms per round, iterations, final x)."""
    W, dg, b, clamp, lpad = masked_system(W, idx, Ys, tau)
    T, l = idx.shape[0], Ys.shape[2]
    x = masked_pcg(W, dg, b, clamp, rtol0)[0].astype(np.float64)
    e = np.zeros_like(x)
    norms, iters = [], []
    for _ in range(rounds):
        x = x + e
        r = b - (dg[:, None] * x - W @ x)
        r[clamp] = 0.0
        cn = np.sqrt((r * r / (dg[:, None] + 1e-10)).sum(axis=0)).reshape(T, lpad)[:, :l]
        norms.append(cn)
        if not cn.max() <= tol:
            e, its = masked_pcg(W, dg, r, clamp, rtol)
            e = e.astype(np.float64)
            iters.append(max(its))
        else:
            e = np.zeros_like(x)
            iters.append(0)
    return norms, iters, x + e


def model_data(seed, n=600, l=5, far=8):
    """l Gaussian classes plus a small far cluster that reaches the rest only through a few weak edges."""
    X, _, yb, yq = O.synth_inputs(seed, l, n - l - far, 16, l, 1.5)
    rng = np.random.default_rng(seed)
    X = np.concatenate([X, (X.mean(axis=0) + 3.0 + 0.05 * rng.standard_normal((far, X.shape[1]))).astype(np.float32)])
    y = np.concatenate([yb, yq, np.zeros(far, dtype=np.int64)])
    return X, y


def draw_trials(seed, y, l, T, per_class, skip_class=None):
    """T labeled sets; trial t takes per_class(t) rows of every class (of every class but skip_class in trial 0)."""
    rng = np.random.default_rng(seed)
    per = [per_class(t) for t in range(T)]
    k_lab = max(per) * l
    idx = np.zeros((T, k_lab), dtype=np.int64)
    Ys = np.zeros((T, k_lab, l), dtype=np.float32)
    for t in range(T):
        classes = [c for c in range(l) if not (t == 0 and c == skip_class)]
        rows = np.concatenate([rng.choice(np.flatnonzero(y == c), per[t], replace=False) for c in classes])
        pool = np.setdiff1d(np.flatnonzero(np.isin(y, classes)), rows)
        extra = rng.choice(pool, k_lab - len(rows), replace=False)  # fills k_lab with rows of the same classes
        rows = np.concatenate([rows, extra])
        idx[t] = rows
        Ys[t, np.arange(k_lab), y[rows]] = 1.0
    return idx, Ys


def test_masked_operator_and_cg_equal_the_compact_system():
    X, y = model_data(3, n=300)
    W = sp.csr_matrix(O.build_graph(X, 20, "auto").W).astype(np.float32).astype(np.float64)
    idx, Ys = draw_trials(4, y, 5, 3, lambda t: 2 + t)
    tau = 0.07
    _, dg, b, clamp, lpad = masked_system(W, idx, Ys, tau)
    n = W.shape[0]
    for t in range(idx.shape[0]):
        lab = idx[t]
        U = np.setdiff1d(np.arange(n), lab)
        perm = np.concatenate([lab, U])
        Wp = W[perm][:, perm]
        Lp = sp.diags(np.asarray(Wp.sum(axis=1)).ravel()) - Wp
        k_lab = len(lab)
        A_c = (Lp[k_lab:, k_lab:] + tau * sp.identity(n - k_lab)).toarray()
        b_c = -(Lp[k_lab:, :k_lab] @ Ys[t].astype(np.float64))
        # the masked operator on vectors supported on U, restricted to U
        E = np.zeros((n, len(U)))
        E[U, np.arange(len(U))] = 1.0
        AE = dg[:, None] * E - W @ E
        AE[lab] = 0.0
        np.testing.assert_allclose(AE[U], A_c, rtol=1e-13, atol=1e-15)
        np.testing.assert_allclose(b[U, t * lpad:t * lpad + 5], b_c, rtol=1e-13, atol=1e-15)
    # fp64 CG iterates: all trials' columns at once (own alpha, beta) against each trial's compact solve
    x_m, _ = masked_pcg(W, dg, b, clamp, iters=25, f32=False)
    assert np.all(x_m[clamp] == 0.0)
    for t in range(idx.shape[0]):
        U = np.setdiff1d(np.arange(n), idx[t])
        cols = slice(t * lpad, t * lpad + 5)
        no_clamp = np.zeros((len(U), 5), dtype=bool)
        off = W[U][:, U]
        x_c, _ = masked_pcg(off, dg[U], b[U, cols], no_clamp, iters=25, f32=False)
        assert O.max_rel(x_m[U, cols], x_c) < 1e-10, t


@pytest.mark.parametrize("T", [1, 16, 64])
@pytest.mark.parametrize("tau", [0.0, 0.07])
def test_trials_refinement_meets_every_column_with_a_round_to_spare(T, tau):
    rounds, rtol0, rtol = schedule()
    X, y = model_data(10 + T)
    W = O.build_graph(X, 20, "auto").W
    idx, Ys = draw_trials(T, y, 5, T, lambda t: 1 + t % 5, skip_class=0 if tau > 0 else None)
    norms, iters, _ = refine_model_trials(W, idx, Ys, tau, rounds, rtol0, rtol)
    first = next((i for i, nv in enumerate(norms) if nv.max() <= 1e-10), None)
    assert first is not None and first <= rounds - 2, (T, tau, [float(nv.max()) for nv in norms])
    assert all(it == 0 for it in iters[first:])
    assert np.all(norms[first] <= 1e-10)  # every column of every trial


# ---------------------------------------------------------------------------------------------------- on the GPU
def _data(seed, n, d, l, sigma=2.0):
    X, _, yb, yq = O.synth_inputs(seed, l, n - l, d, l, sigma)
    return X, np.concatenate([yb, yq]).astype(np.int64)


def _info():
    from graphlearninglayer_b200.laplace_eval import last_eval_info

    return last_eval_info()


def _w_natural(pkg, X, k, eps):
    return sp.csr_matrix(pkg.knn_sym_dist(X, k, eps)[0]).astype(np.float64)


def _labels_match(a, ref_pred, b):
    """labels equal, except rows whose top-two margin in the reference is below 1e-8"""
    top = np.sort(ref_pred, axis=1)
    ok = (a == b) | (top[:, -1] - top[:, -2] < 1e-8)
    return bool(ok.all())


def _scaled_residual(A, b, x):
    r = b - A @ x
    return np.sqrt((r * r / (A.diagonal()[:, None] + 1e-10)).sum(axis=0))


def _check_trials(pkg, X, idx, Ys, y, k, eps, tau, res, trials=None, W=None):
    """every trial against laplace_learning on X[perm_t] and the stop rule on the natural graph's system restricted to it"""
    n = X.shape[0]
    pred, labels = res.pred.cpu().numpy(), res.labels.cpu().numpy()
    correct = None if res.correct is None else res.correct.cpu().numpy()
    W = _w_natural(pkg, X, k, eps) if W is None else W
    L = (sp.diags(np.asarray(W.sum(axis=1)).ravel()) - W).tocsr()
    tau32 = float(np.float32(tau))  # the C ABI takes tau as fp32
    resid = _info()["resid_per_trial"]
    for t in (range(idx.shape[0]) if trials is None else trials):
        lab = idx[t]
        U = np.setdiff1d(np.arange(n), lab)
        A = (L[U][:, U] + tau32 * sp.identity(len(U))).tocsr()
        b = -(L[U][:, lab] @ Ys[t].astype(np.float64))
        assert np.all(_scaled_residual(A, b, pred[t, U]) <= 1e-10 * (1 + 1e-6)), t
        assert resid[t] <= 1e-10, (t, resid[t])
        np.testing.assert_array_equal(pred[t, lab], Ys[t])
        np.testing.assert_array_equal(labels[t, lab], Ys[t].argmax(axis=1))
        perm = np.concatenate([lab, U])
        one = pkg.laplace_learning(torch.as_tensor(X[perm]).cuda(), torch.as_tensor(Ys[t]).cuda(), k=k, epsilon=eps, tau=tau,
                                   targets=torch.as_tensor(y[U]).cuda())
        ref = one.pred.cpu().numpy()
        assert O.max_rel(pred[t, U], ref) < 1e-6, t
        assert _labels_match(labels[t, U], ref, one.labels.cpu().numpy()), t
        if correct is not None:
            flips = int((labels[t, U] != one.labels.cpu().numpy()).sum())
            assert abs(int(correct[t]) - int(one.correct)) <= flips, t  # equal unless a near-tie flipped


def _run(pkg, X, idx, Ys, y=None, **kw):
    return pkg.laplace_learning_trials(torch.as_tensor(X).cuda(), torch.as_tensor(idx).cuda(), torch.as_tensor(Ys).cuda(),
                                       targets=None if y is None else torch.as_tensor(y).cuda(), **kw)


def _random_trials(seed, y, l, T, k_lab):
    rng = np.random.default_rng(seed)
    idx = np.stack([rng.choice(len(y), k_lab, replace=False) for _ in range(T)]).astype(np.int64)
    return idx, np.eye(l, dtype=np.float32)[y[idx]]


# (n, k_lab, d, l, T)
SHAPES = [((3000, 500, 64, 10, 8), ("auto", 0.0)), ((3000, 500, 64, 10, 8), (1.0, 0.07))] + \
         [((2000, 30, 64, 10, 64), et) for et in (("auto", 0.0), (1.0, 0.0), ("auto", 0.07), (1.0, 0.07))] + \
         [((1500, 74, 32, 37, 4), ("auto", 0.0))]


@pytest.mark.gpu
@pytest.mark.parametrize("shape, et", SHAPES, ids=["3000x8-auto-0", "3000x8-1-0.07", "2000x64-auto-0", "2000x64-1-0",
                                                   "2000x64-auto-0.07", "2000x64-1-0.07", "1500x4-l37-chunked"])
def test_trials_match_laplace_learning_on_permuted_features(gpu, shape, et):
    n, k_lab, d, l, T = shape
    eps, tau = et
    X, y = _data(n + T, n, d, l)
    idx, Ys = _random_trials(T, y, l, T, k_lab)
    res = _run(gpu, X, idx, Ys, y, epsilon=eps, tau=tau)
    torch.cuda.synchronize()
    assert res.pred.shape == (T, n, l) and res.pred.dtype == torch.float64
    assert res.labels.shape == (T, n) and res.correct.shape == (T,) and res.correct.dtype == torch.int64
    info = _info()
    assert info["status"] & ~8 == 0 and info["resid"] <= 1e-10 and len(info["resid_per_trial"]) == T
    _check_trials(gpu, X, idx, Ys, y, 50, eps, tau, res)


@pytest.mark.gpu
def test_one_trial_equals_laplace_learning(gpu):
    X, y = _data(7, 2000, 64, 10)
    k_lab = 100
    Y = np.eye(10, dtype=np.float32)[y[:k_lab]]
    a = gpu.laplace_learning(torch.as_tensor(X).cuda(), torch.as_tensor(Y).cuda(), targets=torch.as_tensor(y[k_lab:]).cuda())
    b = _run(gpu, X, np.arange(k_lab)[None], Y[None], y, tau=0.0)
    torch.cuda.synchronize()
    assert O.max_rel(b.pred[0, k_lab:].cpu().numpy(), a.pred.cpu().numpy()) < 1e-6
    assert _labels_match(b.labels[0, k_lab:].cpu().numpy(), a.pred.cpu().numpy(), a.labels.cpu().numpy())
    assert int(b.correct[0]) == int(a.correct)


@pytest.mark.gpu
def test_overlapping_and_repeated_labeled_sets(gpu):
    X, y = _data(8, 1200, 32, 5)
    idx, Ys = _random_trials(9, y, 5, 4, 40)
    r = np.setdiff1d(np.arange(1200), idx[:3])[0]
    idx[0, 5] = idx[1, 0] = r  # labeled in trials 0 and 1, unlabeled in trial 2
    Ys[0, 5] = Ys[1, 0] = np.eye(5, dtype=np.float32)[y[r]]
    idx[3] = idx[2]  # same index set, different labels
    Ys[3] = np.roll(Ys[2], 1, axis=1)
    res = _run(gpu, X, idx, Ys, y)
    torch.cuda.synchronize()
    _check_trials(gpu, X, idx, Ys, y, 50, "auto", 0.0, res)
    assert not torch.equal(res.pred[2], res.pred[3])


@pytest.mark.gpu
def test_invalid_trials_leave_the_valid_ones_unaffected(gpu, monkeypatch):
    n, l = 1500, 5
    X, y = _data(9, n, 32, l)
    idx, Ys = _random_trials(10, y, l, 6, 30)
    valid = [0, 2, 4]
    idx[1, 7] = idx[1, 3]  # a repeat
    idx[3, 0] = -1
    idx[5, 29] = n
    monkeypatch.setenv("GLL_B200_CHECK", "1")
    with warnings.catch_warnings(record=True) as rec:
        warnings.simplefilter("always")
        res = _run(gpu, X, idx, Ys, y)
        torch.cuda.synchronize()
    assert any("labeled-row indices" in str(w.message) for w in rec)
    info = _info()
    assert info["status"] & 16 and info["status"] & 1 == 0
    pred, labels, correct = res.pred.cpu().numpy(), res.labels.cpu().numpy(), res.correct.cpu().numpy()
    for t in (1, 3, 5):
        assert np.all(np.isnan(pred[t])) and np.all(labels[t] == -1) and correct[t] == -1
        assert np.isnan(info["resid_per_trial"][t])
    _check_trials(gpu, X, idx, Ys, y, 50, "auto", 0.0, res, trials=valid)
    alone = _run(gpu, X, idx[valid], Ys[valid], y)  # the valid trials on their own
    torch.cuda.synchronize()
    assert O.max_rel(pred[valid], alone.pred.cpu().numpy()) < 1e-6
    assert np.array_equal(correct[valid], alone.correct.cpu().numpy())
    # int32 indices: the same call
    res32 = _run(gpu, X, idx.astype(np.int32), Ys, y)
    torch.cuda.synchronize()
    assert torch.equal(res32.pred.nan_to_num(7.0), res.pred.nan_to_num(7.0)) and torch.equal(res32.correct, res.correct)


@pytest.mark.gpu
def test_deterministic_and_graph_capturable(gpu):
    n, l = 2000, 10
    X, y = _data(11, n, 64, l)
    X2, _ = _data(12, n, 64, l)
    idx, Ys = _random_trials(13, y, l, 16, 50)  # T lpad = 192: the chunked solve
    Xt, It, Yt, tt = (torch.as_tensor(v).cuda() for v in (X, idx, Ys, y))
    a = gpu.laplace_learning_trials(Xt, It, Yt, targets=tt)
    b = gpu.laplace_learning_trials(Xt, It, Yt, targets=tt)
    ref = gpu.laplace_learning_trials(torch.as_tensor(X2).cuda(), It, Yt, targets=tt)
    torch.cuda.synchronize()
    assert torch.equal(a.pred, b.pred) and torch.equal(a.labels, b.labels) and torch.equal(a.correct, b.correct)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        gpu.laplace_learning_trials(Xt, It, Yt, targets=tt)
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        c = gpu.laplace_learning_trials(Xt, It, Yt, targets=tt)
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(c.pred, a.pred) and torch.equal(c.labels, a.labels) and torch.equal(c.correct, a.correct)
    Xt.copy_(torch.as_tensor(X2).cuda())  # replay on new inputs
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(c.pred, ref.pred) and torch.equal(c.labels, ref.labels) and torch.equal(c.correct, ref.correct)


@pytest.mark.gpu
def test_more_trials_than_a_grid_dimension(gpu):
    """T = 65 536 trials, one more than a grid's y extent: the last trial against a T = 1 call on its labeled set"""
    n, l, k_lab, T = 200, 3, 12, 1 << 16
    X, y = _data(16, n, 16, l)
    rng = np.random.default_rng(17)
    idx = np.argsort(rng.random((T, n)), axis=1)[:, :k_lab].astype(np.int64)
    Ys = np.eye(l, dtype=np.float32)[y[idx]]
    res = _run(gpu, X, idx, Ys, y, k=20)
    torch.cuda.synchronize()
    assert res.pred.shape == (T, n, l) and res.correct.shape == (T,)
    info = _info()
    assert info["status"] & ~8 == 0 and len(info["resid_per_trial"]) == T
    assert np.all(np.asarray(info["resid_per_trial"]) <= 1e-10)  # NaN fails
    one = _run(gpu, X, idx[-1:], Ys[-1:], y, k=20)
    torch.cuda.synchronize()
    a, b = res.pred[-1].cpu().numpy(), one.pred[0].cpu().numpy()
    assert O.max_rel(a, b) < 1e-6
    assert _labels_match(res.labels[-1].cpu().numpy(), b, one.labels[0].cpu().numpy())
    flips = int((res.labels[-1] != one.labels[0]).sum())
    assert abs(int(res.correct[-1]) - int(one.correct[0])) <= flips


@pytest.mark.gpu
def test_max_iter_warning(gpu, monkeypatch):
    X, y = _data(14, 1000, 64, 10)
    idx, Ys = _random_trials(15, y, 10, 4, 40)
    monkeypatch.setenv("GLL_B200_CG_MAXIT", "2")
    monkeypatch.setenv("GLL_B200_CHECK", "1")
    with warnings.catch_warnings(record=True) as rec:
        warnings.simplefilter("always")
        _run(gpu, X, idx, Ys)
        torch.cuda.synchronize()
    assert any("max iter reached" in str(w.message) for w in rec)
    info = _info()
    assert info["status"] & 1 and max(info["resid_per_trial"]) > 1e-10
