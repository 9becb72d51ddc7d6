"""CPU checks of laplace_learning (graphlearninglayer_b200/laplace_eval.py, gll_laplace_eval): the Python contract, and a numpy
model of the device refinement that justifies its schedule (GLL_LAPLACE_ROUNDS / GLL_LAPLACE_CG_RTOL0 / GLL_LAPLACE_CG_RTOL in
include/gll_b200.h): an fp32 Jacobi-PCG with the chosen relative tolerances inside fp64 residual rounds reaches the reference's
stop rule ||M r_c||_2 <= 1e-10 on every column with at least one round to spare, and a round after convergence changes nothing."""
import inspect
import os
import re

import numpy as np
import pytest
import scipy.sparse as sp

from oracle import gll_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def schedule():
    text = open(os.path.join(ROOT, "include", "gll_b200.h")).read()

    def val(name):
        return float(re.search(r"#define\s+%s\s+(\S+)" % name, text).group(1))

    return int(val("GLL_LAPLACE_ROUNDS")), val("GLL_LAPLACE_CG_RTOL0"), val("GLL_LAPLACE_CG_RTOL")


@pytest.fixture(scope="module")
def pkg():
    from graphlearninglayer_b200 import build

    build.build()
    import graphlearninglayer_b200

    return graphlearninglayer_b200


def test_signature_and_exports(pkg):
    sig = inspect.signature(pkg.laplace_learning)
    assert list(sig.parameters) == ["features", "label_matrix", "k", "epsilon", "tau", "tol", "targets"]
    d = {p.name: p.default for p in sig.parameters.values()}
    assert d["k"] == 50 and d["epsilon"] == "auto" and d["tau"] == 0.0 and d["tol"] == 1e-10 and d["targets"] is None
    assert pkg.LaplaceResult._fields == ("pred", "labels", "correct")
    assert "laplace_learning" in pkg.__all__


def test_cpu_tensors_refused(pkg):
    import torch

    X = torch.randn(300, 8)
    Y = torch.eye(4)[torch.arange(40) % 4]
    with pytest.raises(RuntimeError, match="no CPU path"):
        pkg.laplace_learning(X, Y)


@pytest.mark.parametrize("kwargs, match", [
    (dict(k=1), "k must be"), (dict(k=65), "k must be"), (dict(n=200, k=40), "n >= 256"), (dict(k_lab=0), "k_lab"),
    (dict(k_lab=300), "k_lab"), (dict(one_d=True), "label_matrix"), (dict(epsilon="knn"), "epsilon"), (dict(tol=0.0), "tol"),
    (dict(targets=5), "targets")])
def test_bad_arguments_rejected_before_any_device_call(pkg, kwargs, match):
    import torch

    n, k_lab = kwargs.pop("n", 300), kwargs.pop("k_lab", 40)
    X = torch.randn(n, 8)  # a CPU tensor: the argument check must come first
    Y = torch.eye(4)[torch.arange(k_lab) % 4]
    if kwargs.pop("one_d", False):
        Y = Y[:, 0]
    if "targets" in kwargs:
        kwargs["targets"] = torch.zeros(kwargs["targets"], dtype=torch.long)
    with pytest.raises(ValueError, match=match):
        pkg.laplace_learning(X, Y, **kwargs)


# ---------------------------------------------------------------------------------------------------- model of the device path
def pcg32(off, diag, b, rel, max_iter=5000):
    """fp32 Jacobi-PCG on diag - off, x0 = 0, all columns together with the per-column freeze of the device kernels; stops when
    every column has ||r_c||_2 <= rel * max_c ||b_c||_2 (a negative tolerance of gll_cg_solve).  Dots in fp64 like the kernels."""
    off = off.astype(np.float32)
    diag = diag.astype(np.float32)
    b = b.astype(np.float32)
    dinv = (np.float32(1) / diag)[:, None]

    def dot(a, c):
        return np.einsum("ij,ij->j", a.astype(np.float64), c.astype(np.float64))

    x = np.zeros_like(b)
    r = b.copy()
    z = r * dinv
    p = z.copy()
    rz, rr = dot(r, z), dot(r, r)
    tol2 = rel * rel * rr.max()
    it = 0
    while rr.max() > tol2 and it < max_iter:
        it += 1
        ap = diag[:, None] * p - (off @ p).astype(np.float32)
        pap = dot(p, ap)
        live = rr > tol2
        al = np.where(live, rz / np.where(pap != 0, pap, 1), 0).astype(np.float32)
        x = x + al * p
        r = r - al * ap
        z = r * dinv
        rzn, rrn = dot(r, z), dot(r, r)
        be = np.where((rrn > tol2) & (rz != 0), rzn / np.where(rz != 0, rz, 1), 0).astype(np.float32)
        p = z + be * p
        rz, rr = rzn, rrn
    return x, it


def refine_model(W, Y, tau, rounds, rtol0, rtol, tol=1e-10):
    """gll_laplace_eval on the host: returns (scaled residual measured by every round, correction iterations of every round,
    the solution after every round, final solution)."""
    W = sp.csr_matrix(W).astype(np.float32).astype(np.float64)  # the stored fp32 weights, evaluated in fp64
    k_lab = Y.shape[0]
    deg = np.asarray(W.sum(axis=1)).ravel()  # row sums (the kernel's degree)
    Wuu, Wul = W[k_lab:, k_lab:].tocsr(), W[k_lab:, :k_lab]
    dg = deg[k_lab:] + tau
    b = Wul @ np.asarray(Y, dtype=np.float64)
    diag32 = (np.asarray(W.astype(np.float32).sum(axis=1)).ravel()[k_lab:].astype(np.float32) + np.float32(tau))
    x = pcg32(Wuu, diag32, b, rtol0)[0].astype(np.float64)
    e = np.zeros_like(x)
    norms, iters, xs = [], [], []
    for _ in range(rounds):
        x = x + e
        xs.append(x.copy())
        r = b - (dg[:, None] * x - Wuu @ x)
        nrm = np.sqrt((r * r / (dg[:, None] + 1e-10)).sum(axis=0))
        norms.append(nrm)
        if not nrm.max() <= tol:
            e, it = pcg32(Wuu, diag32, r, rtol)
            e = e.astype(np.float64)
        else:
            e, it = np.zeros_like(x), 0  # right-hand-side scale 0: the CG stops at iteration 0 with x = 0
        iters.append(it)
    return norms, iters, xs, x + e


def model_systems():
    z = np.load(os.path.join(ROOT, "tests", "golden", "eval_k50.npz"))
    seed, k_lab, m, d, l, knn = (int(v) for v in z["params"])
    _, Y, _, _ = O.synth_inputs(seed, k_lab, m, d, l, float(z["sigma"]))
    W1 = sp.csr_matrix((z["w_data"], z["w_indices"], z["w_indptr"]), shape=(k_lab + m,) * 2)
    X2, Y2, _, _ = O.synth_inputs(7, 1000, 4000, 64, 10, 3.0)
    W2 = O.build_graph(X2, 50, "auto").W
    return [("eval_k50", W1, Y, float(z["tau"])), ("synthetic n=5000 k=50 tau=0", W2, Y2, 0.0)]


@pytest.mark.parametrize("case", [0, 1])
def test_refinement_schedule_reaches_reference_tolerance_with_a_round_to_spare(case):
    name, W, Y, tau = model_systems()[case]
    rounds, rtol0, rtol = schedule()
    norms, iters, xs, final = refine_model(W, Y, tau, rounds, rtol0, rtol)
    first = next((i for i, nv in enumerate(norms) if nv.max() <= 1e-10), None)
    assert first is not None and first <= rounds - 2, (name, [float(nv.max()) for nv in norms])
    for i in range(first, rounds):  # rounds after convergence: no iterations, identical residual, identical solution
        assert iters[i] == 0
        assert np.array_equal(norms[i], norms[first]) and np.array_equal(xs[i], xs[first])
    assert np.array_equal(final, xs[first])
    assert np.all(norms[first] <= 1e-10)
    assert all(0 < it < 200 for it in iters[:first])  # the inner tolerances are reachable in fp32
