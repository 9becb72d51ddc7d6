"""GPU checks of laplace_learning (gll_laplace_eval): the reference's utils.laplace (utils.py:570-593) on device features --
against the reference fixture, against the numpy/scipy wrapper path, the stop rule recomputed on the host in fp64, labels and
hit count, determinism and CUDA-graph capture, and the full CIFAR-10-sized evaluation (n = 70 000, k = 50)."""
import os
import warnings

import numpy as np
import pytest
import scipy.sparse as sparse
import scipy.sparse.linalg as sla

from oracle import gll_oracle as O

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope="module")
def pkg():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import graphlearninglayer_b200

    return graphlearninglayer_b200


def eval_info():
    from graphlearninglayer_b200.laplace_eval import last_eval_info

    return last_eval_info()


def run(pkg, X, Y, **kw):
    t = kw.pop("targets", None)
    res = pkg.laplace_learning(torch.as_tensor(X).cuda(), torch.as_tensor(Y).cuda(),
                               targets=None if t is None else torch.as_tensor(t).cuda(), **kw)
    torch.cuda.synchronize()
    return res


def system(pkg, X, k_lab, Y, k, eps, tau):
    """L_uu + tau I and b = -L_ul Y in fp64 from knn_sym_dist's W, with the row-sum degree gll_laplace_eval uses."""
    W = sparse.csr_matrix(pkg.knn_sym_dist(X, k, eps)[0])
    L = (sparse.diags(np.asarray(W.sum(axis=1)).ravel()) - W).tocsr()
    A = (L[k_lab:, k_lab:] + tau * sparse.identity(X.shape[0] - k_lab)).tocsr()
    b = -(L[k_lab:, :k_lab] @ np.asarray(Y, dtype=np.float64))
    return A, b


def scaled_residual(A, b, x):
    """||M (b - A x)||_2 per column, M = diag(A + 1e-10)^(-1/2): the reference's stop quantity (make_golden_eval.py:41-45)."""
    r = b - A @ x
    return np.sqrt((r * r / (A.diagonal()[:, None] + 1e-10)).sum(axis=0))


def wrapper_laplace(pkg, X, Y, k_lab, eps, tau):
    """utils.py:570-593 on the numpy/scipy wrappers (as test_eval_path_like_utils_laplace restates it)."""
    W = pkg.knn_sym_dist(X, 50, eps)[0]
    L = (sparse.diags(np.asarray(W.sum(axis=0)).ravel()) - W).tocsr()
    Luu = (L[k_lab:, k_lab:] + tau * sparse.identity(X.shape[0] - k_lab)).tocsr()
    Lul = L[k_lab:, :k_lab]
    M = sparse.diags(1.0 / np.sqrt(Luu.diagonal() + 1e-10))
    return M @ pkg.stable_conjgrad(M @ Luu @ M, -(M @ (Lul @ Y.astype(np.float64))))


def test_matches_reference_fixture(pkg):
    g = np.load(os.path.join(HERE, "golden", "eval_k50.npz"))
    seed, k_lab, m, d, l, knn = (int(v) for v in g["params"])
    X, Y, _, _ = O.synth_inputs(seed, k_lab, m, d, l, float(g["sigma"]))
    res = run(pkg, X, Y, k=knn, epsilon="auto", tau=float(g["tau"]))
    pred = res.pred.cpu().numpy()
    assert res.pred.dtype == torch.float64 and pred.shape == (m, l)
    assert O.max_rel(pred, g["pred"]) < 1e-5
    assert np.array_equal(pred.argmax(axis=1), g["pred"].argmax(axis=1))


@pytest.mark.parametrize("eps", ["auto", 1.0])
@pytest.mark.parametrize("tau", [0.0, 0.07])
def test_matches_wrapper_path(pkg, eps, tau):
    X, Y, _, _ = O.synth_inputs(23, 500, 2500, 64, 10, 2.0)
    ours = run(pkg, X, Y, k=50, epsilon=eps, tau=tau).pred.cpu().numpy()
    ref = wrapper_laplace(pkg, X, Y, 500, eps, tau)
    assert O.max_rel(ours, ref) < 1e-6
    assert np.array_equal(ours.argmax(axis=1), ref.argmax(axis=1))


@pytest.mark.parametrize("tol", [1e-10, 1e-6])
def test_stop_rule_on_host(pkg, tol):
    X, Y, _, _ = O.synth_inputs(5, 400, 2000, 64, 10, 2.5)
    res = run(pkg, X, Y, k=50, tol=tol)
    A, b = system(pkg, X, 400, Y, 50, "auto", 0.0)
    nrm = scaled_residual(A, b, res.pred.cpu().numpy())
    assert np.all(nrm <= tol * (1 + 1e-6)), nrm
    info = eval_info()
    assert info["status"] & 1 == 0 and info["resid"] <= tol


def test_loose_tolerance_needs_no_correction(pkg):
    X, Y, _, _ = O.synth_inputs(5, 400, 2000, 64, 10, 2.5)
    run(pkg, X, Y, k=50, tol=1e-3)
    info = eval_info()
    assert info["rounds"] == 0 and info["cg_iters_correction"] == 0 and info["round_iters"] == [0, 0, 0, 0], info
    assert info["cg_iters_first"] > 0 and info["resid"] <= 1e-3


def test_labels_and_correct_count(pkg):
    X, Y, _, yq = O.synth_inputs(11, 300, 1700, 64, 10, 3.0)
    t = yq.astype(np.int64).copy()
    t[::7] = -1  # rows that are not scored
    res = run(pkg, X, Y, k=40, targets=t)
    assert res.labels.dtype == torch.int64 and res.correct.dtype == torch.int64 and res.correct.dim() == 0
    assert torch.equal(res.labels, res.pred.argmax(dim=1))
    tt = torch.as_tensor(t).cuda()
    assert int(res.correct) == int(((tt >= 0) & (res.labels == tt)).sum())
    assert run(pkg, X, Y, k=40).correct is None


def test_disconnected_cluster_gives_zero_rows(pkg):
    X, Y, _, yq = O.synth_inputs(3, 300, 1200, 32, 5, 2.0)
    rng = np.random.default_rng(0)
    far = (50.0 + 0.1 * rng.standard_normal((64, 32))).astype(np.float32)
    Xa = np.concatenate([X, far])
    t = np.concatenate([yq, np.zeros(64, dtype=np.int64)])
    t[-3:] = 2
    res = run(pkg, Xa, Y, k=50, epsilon=1.0, tau=0.05, targets=t)
    pred = res.pred.cpu().numpy()
    assert np.all(pred[-64:] == 0.0) and np.all(res.labels.cpu().numpy()[-64:] == 0)
    tt = torch.as_tensor(t).cuda()
    assert int(res.correct) == int(((tt >= 0) & (res.labels == tt)).sum())


def test_many_classes_chunked_solver(pkg):
    X, Y, _, _ = O.synth_inputs(4, 1500, 1500, 64, 150, 1.0)
    res = run(pkg, X, Y, k=30, tau=0.01)
    A, b = system(pkg, X, 1500, Y, 30, "auto", 0.01)
    ref = sla.splu(A.tocsc()).solve(b)
    pred = res.pred.cpu().numpy()
    assert pred.shape == (1500, 150)
    assert O.max_rel(pred, ref) < 1e-6
    info = eval_info()
    assert info["status"] & 1 == 0 and info["resid"] <= 1e-10 and info["rounds"] >= 1


def test_deterministic_and_graph_capturable(pkg):
    X, Y, _, yq = O.synth_inputs(9, 500, 2500, 64, 10, 2.0)
    Xt, Yt, tt = torch.as_tensor(X).cuda(), torch.as_tensor(Y).cuda(), torch.as_tensor(yq).cuda()
    a = pkg.laplace_learning(Xt, Yt, targets=tt)
    b = pkg.laplace_learning(Xt, Yt, targets=tt)
    torch.cuda.synchronize()
    assert torch.equal(a.pred, b.pred) and torch.equal(a.labels, b.labels) and torch.equal(a.correct, b.correct)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        pkg.laplace_learning(Xt, Yt, targets=tt)
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        c = pkg.laplace_learning(Xt, Yt, targets=tt)
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(c.pred, a.pred) and torch.equal(c.labels, a.labels) and torch.equal(c.correct, a.correct)


def test_max_iter_warning(pkg, monkeypatch):
    X, Y, _, _ = O.synth_inputs(5, 400, 2000, 64, 10, 2.5)
    monkeypatch.setenv("GLL_B200_CG_MAXIT", "2")
    monkeypatch.setenv("GLL_B200_CHECK", "1")
    with warnings.catch_warnings(record=True) as rec:
        warnings.simplefilter("always")
        run(pkg, X, Y, k=50)
    assert any("max iter reached" in str(w.message) for w in rec)
    assert eval_info()["status"] & 1


def test_full_size_evaluation(pkg):
    """SURVEY 3.4: CIFAR-10-sized evaluation graph, 10 000 labeled + 60 000 unlabeled rows, k = 50."""
    X, Y, _, yq = O.synth_inputs(0, 10000, 60000, 128, 10, 3.0)
    res = run(pkg, X, Y, k=50, targets=yq.astype(np.int64))
    A, b = system(pkg, X, 10000, Y, 50, "auto", 0.0)
    pred = res.pred.cpu().numpy()
    assert np.all(scaled_residual(A, b, pred) <= 1e-10 * (1 + 1e-6))
    assert int(res.correct) == int((pred.argmax(axis=1) == yq).sum())
