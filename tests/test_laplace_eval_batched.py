"""laplace_learning_batched (gll_laplace_eval_batched): the Laplace-learning evaluation over B independent graphs in one call,
and the segmented kNN search for 33 < k <= 64 it runs on.

Without a GPU: the C argument checks (they return before any CUDA call), the Python validation, and a numpy model of the
batched refinement -- B block-diagonal graphs solved together with shared CG step lengths under the GLL_LAPLACE_* schedule, the
stop rule tested per graph.  On a GPU: the segmented lists for k in {34, 50, 64} bit for bit against gll_knn per segment, B = 1
bit for bit against laplace_learning, B > 1 against per-graph solutions and the reference's stop rule recomputed on the host,
a disconnected cluster in one graph, determinism and CUDA-graph replay, and the max-iteration warning.
"""
import ctypes
import inspect
import os
import re
import warnings

import numpy as np
import pytest
import scipy.sparse as sp
import scipy.sparse.linalg as sla

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

    sig = inspect.signature(pkg.laplace_learning_batched)
    assert list(sig.parameters) == ["features", "label_matrix", "k", "epsilon", "tau", "tol", "targets"]
    d = {p.name: p.default for p in sig.parameters.values()}
    assert d["k"] == 50 and d["epsilon"] == "auto" and d["tau"] == 0.0 and d["tol"] == 1e-10 and d["targets"] is None
    assert "laplace_learning_batched" in pkg.__all__
    raw = ctypes.CDLL(libmod.LIB_PATH)
    for nm in ("gll_laplace_eval_batched_workspace_bytes", "gll_laplace_eval_batched"):
        assert hasattr(raw, nm) and nm in libmod.EXPORTS


def test_c_argument_checks(libmod):
    lib, seg = libmod.lib, libmod.seg_ptr_array
    buf = ctypes.c_void_p(16)  # never dereferenced: the checks fail first

    def call(X=buf, Y=buf, B=4, n=300, d=8, k=50, l=3, k_lab=30, tol=1e-10, maxit=100, pred=buf, labels=buf, info=buf, ws=buf):
        return lib.gll_laplace_eval_batched(X, Y, B, n, d, k, l, k_lab, 1, 0.0, 0.0, tol, maxit, pred, labels, None, None, None, info,
                                            ws, 1 << 30, None)

    for kw in (dict(X=None), dict(Y=None), dict(pred=None), dict(labels=None), dict(info=None), dict(ws=None),  # null pointers
               dict(B=0), dict(B=1 << 16, n=1 << 15),                                 # B >= 1, B n < 2^31
               dict(k=1), dict(k=65), dict(n=40, k=41, k_lab=10),                       # 2 <= k <= 64, k <= n
               dict(B=2, n=100, k=34), dict(B=1, n=255, k=50),                          # B n >= 256 when k > 33
               dict(k_lab=0), dict(k_lab=300), dict(l=0), dict(d=0),                    # 1 <= k_lab < n, l >= 1, d >= 1
               dict(tol=0.0), dict(tol=-1.0), dict(maxit=0)):                           # tol > 0, cg_max_iter >= 1
        assert call(**kw) == ERR_ARG, kw
    wsb = lib.gll_laplace_eval_batched_workspace_bytes
    for args in ((0, 300, 8, 50, 3, 30), (1 << 16, 1 << 15, 8, 50, 3, 30), (4, 300, 8, 1, 3, 30), (4, 300, 8, 65, 3, 30),
                 (4, 40, 8, 41, 3, 10), (2, 100, 8, 34, 3, 10), (4, 300, 8, 50, 3, 0), (4, 300, 8, 50, 3, 300),
                 (4, 300, 8, 50, 0, 30), (4, 300, 0, 50, 3, 30)):
        assert wsb(*args) == 0, args
    # the segmented search itself: k = 50 needs every segment >= k rows and n >= 256
    knn = lib.gll_knn_segments
    assert knn(buf, 300, 8, 50, seg([0, 260, 300]), 2, buf, buf, None, buf, 1 << 30, None) == ERR_ARG  # a segment of 40 < k
    assert knn(buf, 200, 8, 50, seg([0, 100, 200]), 2, buf, buf, None, buf, 1 << 30, None) == ERR_ARG  # n < 256
    assert knn(buf, 300, 8, 65, seg([0, 150, 300]), 2, buf, buf, None, buf, 1 << 30, None) == ERR_ARG  # k > 64
    assert lib.gll_knn_segments_workspace_bytes(300, 8, 50, seg([0, 260, 300]), 2) == 0
    assert lib.gll_knn_segments_workspace_bytes(200, 8, 50, seg([0, 100, 200]), 2) == 0


@pytest.mark.parametrize("kwargs, exc, match", [
    (dict(), RuntimeError, "no CPU path"),
    (dict(X=torch.zeros(300, 8)), ValueError, "features"), (dict(Y=torch.zeros(30, 3)), ValueError, "label_matrix"),
    (dict(Y=torch.zeros(3, 30, 3)), ValueError, "label_matrix"), (dict(X=torch.zeros(0, 300, 8), Y=torch.zeros(0, 30, 3)), ValueError, "B"),
    (dict(k=1), ValueError, "k must be"), (dict(k=65), ValueError, "k must be"),
    (dict(X=torch.zeros(2, 100, 8), Y=torch.zeros(2, 30, 3), k=34), ValueError, "B n >= 256"),
    (dict(Y=torch.zeros(2, 0, 3)), ValueError, "k_lab"), (dict(Y=torch.zeros(2, 300, 3)), ValueError, "k_lab"),
    (dict(Y=torch.zeros(2, 30, 0)), ValueError, "class column"), (dict(epsilon="knn"), ValueError, "epsilon"),
    (dict(tol=0.0), ValueError, "tol"), (dict(targets=torch.zeros(2, 30, dtype=torch.long)), ValueError, "targets"),
    (dict(targets=torch.zeros(540, dtype=torch.long)), ValueError, "targets")])
def test_python_validation_before_any_device_call(libmod, kwargs, exc, match):
    import graphlearninglayer_b200 as pkg

    X = kwargs.pop("X", torch.zeros(2, 300, 8))  # CPU tensors: every argument check must come first
    Y = kwargs.pop("Y", torch.zeros(2, 30, 3))
    with pytest.raises(exc, match=match):
        pkg.laplace_learning_batched(X, Y, **kwargs)


# ---------------------------------------------------------------------------------------------------- model of the batched refinement
def schedule():
    text = open(os.path.join(ROOT, "include", "gll_b200.h")).read()

    def val(name):
        return float(re.search(r"#define\s+%s\s+(\S+)" % name, text).group(1))

    return int(val("GLL_LAPLACE_ROUNDS")), val("GLL_LAPLACE_CG_RTOL0"), val("GLL_LAPLACE_CG_RTOL")


def refine_model_batched(graphs, tau, rounds, rtol0, rtol, tol=1e-10):
    """gll_laplace_eval_batched on the host: the graphs' unlabeled systems as one block-diagonal system, every fp32 PCG shared
    by all graphs (pcg32 of test_laplace_eval_cpu.py: one step length per class column over all rows), the stop rule per graph.
    Returns (per round: [B, l] scaled residual norms), correction iterations per round, the solution after every round, final."""
    from test_laplace_eval_cpu import pcg32

    blocks, dgs, bs, d32s = [], [], [], []
    for W, Y in graphs:
        W = sp.csr_matrix(W).astype(np.float32).astype(np.float64)
        k_lab = Y.shape[0]
        deg = np.asarray(W.sum(axis=1)).ravel()
        blocks.append(W[k_lab:, k_lab:])
        dgs.append(deg[k_lab:] + tau)
        bs.append(W[k_lab:, :k_lab] @ np.asarray(Y, dtype=np.float64))
        d32s.append(np.asarray(W.astype(np.float32).sum(axis=1)).ravel()[k_lab:].astype(np.float32) + np.float32(tau))
    Wuu, dg, b, diag32 = sp.block_diag(blocks).tocsr(), np.concatenate(dgs), np.vstack(bs), np.concatenate(d32s)
    cuts = np.cumsum([0] + [blk.shape[0] for blk in blocks])
    x = pcg32(Wuu, diag32, b, rtol0)[0].astype(np.float64)
    e = np.zeros_like(x)
    norms, iters, xs = [], [], []
    for _ in range(rounds):
        x = x + e
        xs.append(x.copy())
        r = b - (dg[:, None] * x - Wuu @ x)
        q = r * r / (dg[:, None] + 1e-10)
        nrm = np.stack([np.sqrt(q[cuts[g]:cuts[g + 1]].sum(axis=0)) for g in range(len(blocks))])
        norms.append(nrm)
        if not nrm.max() <= tol:  # one graph above tol: every graph gets a correction
            e, it = pcg32(Wuu, diag32, r, rtol)
            e = e.astype(np.float64)
        else:
            e, it = np.zeros_like(x), 0
        iters.append(it)
    return norms, iters, xs, x + e


def model_graphs(B):
    """B graphs of different conditioning: cluster spreads from 1 to 4, and every fourth graph has a small far cluster that
    only reaches the rest through a few weak edges (its kNN lists must leave the cluster)."""
    out = []
    for g in range(B):
        k_lab, m = (25, 75) if B > 8 else (100, 400)
        X, Y, _, _ = O.synth_inputs(1000 + g, k_lab, m, 16, 5, 1.0 + 3.0 * (g % 7) / 6.0)
        if g % 4 == 0:
            rng = np.random.default_rng(g)
            far = (X[k_lab:].mean(axis=0) + 3.0 + 0.05 * rng.standard_normal((8, X.shape[1]))).astype(np.float32)
            X = np.concatenate([X, far])
        out.append((O.build_graph(X, 20, "auto").W, Y))
    return out


@pytest.mark.parametrize("B", [1, 8, 64])
def test_batched_refinement_meets_every_graphs_stop_rule_with_a_round_to_spare(B):
    rounds, rtol0, rtol = schedule()
    norms, iters, xs, final = refine_model_batched(model_graphs(B), 0.0, rounds, rtol0, rtol)
    first = next((i for i, nv in enumerate(norms) if nv.max() <= 1e-10), None)
    assert first is not None and first <= rounds - 2, (B, [float(nv.max()) for nv in norms])
    for i in range(first, rounds):  # rounds after convergence: no iterations, identical residuals, identical solution
        assert iters[i] == 0
        assert np.array_equal(norms[i], norms[first]) and np.array_equal(xs[i], xs[first])
    assert np.array_equal(final, xs[first])
    assert np.all(norms[first] <= 1e-10)  # every column of every graph


# ---------------------------------------------------------------------------------------------------- segmented kNN, k > 33
def _feats(seed, n, d):
    g = np.random.default_rng(seed)
    c = g.standard_normal((8, d))
    X = c[g.integers(0, 8, n)] + 0.6 * g.standard_normal((n, d))
    X /= np.linalg.norm(X, axis=1, keepdims=True)
    return torch.as_tensor(X.astype(np.float32)).cuda()


class _env:
    def __init__(self, env):
        self.env = env

    def __enter__(self):
        self.old = {k: os.environ.get(k) for k in self.env}
        os.environ.update(self.env)

    def __exit__(self, *a):
        for k, v in self.old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def _knn(libmod, X, k):
    n, d = X.shape
    with _env({"GLL_B200_KNN_PATH": "tc"} if n < 256 else {}):  # k > 33 runs on the tensor-core path only
        idx = torch.empty((n, k), dtype=torch.int32, device=X.device)
        dist = torch.empty((n, k), dtype=torch.float32, device=X.device)
        wsb = libmod.lib.gll_knn_workspace_bytes(n, d, k)
        ws = torch.empty(wsb, dtype=torch.uint8, device=X.device)
        libmod.check(libmod.lib.gll_knn(X.data_ptr(), n, d, k, idx.data_ptr(), dist.data_ptr(), None, ws.data_ptr(), wsb,
                                        torch.cuda.current_stream().cuda_stream), "gll_knn")
        torch.cuda.synchronize()
    return idx, dist


def _check_segments(libmod, X, k, seg, env):
    n, d = X.shape
    sp_ = libmod.seg_ptr_array(seg)
    idx = torch.empty((n, k), dtype=torch.int32, device=X.device)
    dist = torch.empty((n, k), dtype=torch.float32, device=X.device)
    info = torch.zeros(libmod.INFO_WORDS, dtype=torch.int32, device=X.device)
    with _env(env):
        wsb = libmod.lib.gll_knn_segments_workspace_bytes(n, d, k, sp_, len(seg) - 1)
        assert wsb > 0
        ws = torch.empty(wsb, dtype=torch.uint8, device=X.device)
        libmod.check(libmod.lib.gll_knn_segments(X.data_ptr(), n, d, k, sp_, len(seg) - 1, idx.data_ptr(), dist.data_ptr(),
                                                 info.data_ptr(), ws.data_ptr(), wsb, torch.cuda.current_stream().cuda_stream),
                     "gll_knn_segments")
        torch.cuda.synchronize()
    for s in range(len(seg) - 1):
        a, b = seg[s], seg[s + 1]
        ri, rd = _knn(libmod, X[a:b].contiguous(), k)
        assert torch.equal(idx[a:b], ri + a), (env, s, b - a)
        assert torch.equal(dist[a:b], rd), (env, s, b - a)
    return idx, info


SIZES = [64, 100, 255, 256, 257, 300, 2000]
ENVS = [{}, {"GLL_B200_KNN_PAIR": "1"}, {"GLL_B200_KNN_SPLIT": "f16x2"}, {"GLL_B200_KNN_FORCE_FALLBACK": "300"}]


@pytest.mark.gpu
@pytest.mark.parametrize("k", [34, 50, 64])
@pytest.mark.parametrize("d", [64, 200, 512])
@pytest.mark.parametrize("env", ENVS, ids=["default", "pair", "f16x2", "fallback"])
def test_segments_k_above_33_bit_identical_to_per_segment(libmod, gpu, k, d, env):
    sizes = SIZES[::-1] if d == 200 else SIZES  # segment edges land at different tile offsets
    seg = np.concatenate([[0], np.cumsum(sizes)]).tolist()
    _, info = _check_segments(libmod, _feats(d + k, seg[-1], d), k, seg, env)
    if "GLL_B200_KNN_FORCE_FALLBACK" in env:
        assert int(info[libmod.INFO_KNN_FALLBACK_ROWS]) >= 300


@pytest.mark.gpu
def test_segments_k50_large_aligned(libmod, gpu):
    seg = [10512 * b for b in range(9)]  # > 4 x 148 row tiles: every CTA owns whole row tiles
    _check_segments(libmod, _feats(3, seg[-1], 128), 50, seg, {})


@pytest.mark.gpu
def test_segments_k50_duplicate_graphs_never_cross(libmod, gpu):
    A = _feats(11, 300, 64)
    X = torch.cat((A, A, _feats(12, 260, 64))).contiguous()
    seg = [0, 300, 600, 860]
    idx, _ = _check_segments(libmod, X, 50, seg, {})
    lo = torch.as_tensor(np.repeat(seg[:-1], np.diff(seg)), device=X.device)[:, None]
    hi = torch.as_tensor(np.repeat(seg[1:], np.diff(seg)), device=X.device)[:, None]
    assert bool(((idx >= lo) & (idx < hi)).all())


# ---------------------------------------------------------------------------------------------------- the evaluation
def _batch(seed, B, k_lab, m, d, l, sigma=2.0):
    Xs, Ys, ys = [], [], []
    for b in range(B):
        X, Y, _, yq = O.synth_inputs(seed + b, k_lab, m, d, l, sigma)
        Xs.append(X)
        Ys.append(Y)
        ys.append(yq.astype(np.int64))
    return np.stack(Xs), np.stack(Ys), np.stack(ys)


def _cuda(*a):
    return [torch.as_tensor(v).cuda() for v in a]


def _info():
    from graphlearninglayer_b200.laplace_eval import last_eval_info

    return last_eval_info()


def _system(pkg, X, k_lab, Y, k, eps, tau):
    """L_uu + tau I and b = -L_ul Y in fp64 from knn_sym_dist's W, with the row-sum degree the evaluation uses."""
    with _env({"GLL_B200_KNN_PATH": "tc"} if X.shape[0] < 256 else {}):
        W = sp.csr_matrix(pkg.knn_sym_dist(X, k, eps)[0])
    L = (sp.diags(np.asarray(W.sum(axis=1)).ravel()) - W).tocsr()
    tau = float(np.float32(tau))  # the C ABI takes tau as fp32: the device solves with that value
    A = (L[k_lab:, k_lab:] + tau * sp.identity(X.shape[0] - k_lab)).tocsr()
    b = -(L[k_lab:, :k_lab] @ np.asarray(Y, dtype=np.float64))
    return A, b


def _scaled_residual(A, b, x):
    r = b - A @ x
    return np.sqrt((r * r / (A.diagonal()[:, None] + 1e-10)).sum(axis=0))


def _labels_match(a, ref_pred, b):
    """labels equal, except rows whose top-two margin in the reference is below 1e-8"""
    top = np.sort(ref_pred, axis=1)
    ok = (a == b) | (top[:, -1] - top[:, -2] < 1e-8)
    return bool(ok.all())


def _check_against_per_graph(pkg, X, Y, yq, k, eps, tau, res, graphs=None):
    B, n, _ = X.shape
    k_lab = Y.shape[1]
    pred, labels, correct = (v.cpu().numpy() for v in res)
    resid = _info()["resid_per_graph"]
    assert len(resid) == B
    for b in (range(B) if graphs is None else graphs):
        A, rhs = _system(pkg, X[b], k_lab, Y[b], k, eps, tau)
        assert np.all(_scaled_residual(A, rhs, pred[b]) <= 1e-10 * (1 + 1e-6)), b
        assert resid[b] <= 1e-10, (b, resid[b])
        if n >= 256 or k <= 33:  # the per-graph call (k > 33 needs n >= 256 on one graph)
            one = pkg.laplace_learning(*_cuda(X[b], Y[b]), k=k, epsilon=eps, tau=tau, targets=torch.as_tensor(yq[b]).cuda())
            ref, ref_correct = one.pred.cpu().numpy(), int(one.correct)
        else:  # otherwise the system solved directly
            ref = sla.splu(A.tocsc()).solve(rhs)
            ref_correct = int((ref.argmax(axis=1) == yq[b]).sum())
        assert O.max_rel(pred[b], ref) < 1e-6, b
        ref_labels = ref.argmax(axis=1)
        assert _labels_match(labels[b], ref, ref_labels), b
        assert abs(int(correct[b]) - ref_correct) <= int((labels[b] != ref_labels).sum()), b  # equal unless a near-tie flipped


@pytest.mark.gpu
@pytest.mark.parametrize("eps,tau", [("auto", 0.0), (1.0, 0.0), ("auto", 0.07), (1.0, 0.07)])
def test_batch_of_one_bit_identical(gpu, eps, tau):
    from graphlearninglayer_b200 import laplace_eval

    X, Y, yq = _batch(31, 1, 500, 2500, 64, 10)
    Xt, Yt, tt = _cuda(X, Y, yq)
    a = gpu.laplace_learning(Xt[0], Yt[0], epsilon=eps, tau=tau, targets=tt[0])
    ia = laplace_eval._last_info.clone()
    b = gpu.laplace_learning_batched(Xt, Yt, epsilon=eps, tau=tau, targets=tt)
    ib = laplace_eval._last_info.clone()
    torch.cuda.synchronize()
    assert b.pred.shape == (1, 2500, 10) and b.labels.shape == (1, 2500) and b.correct.shape == (1,)
    assert torch.equal(a.pred, b.pred[0]) and torch.equal(a.labels, b.labels[0]) and torch.equal(a.correct, b.correct[0])
    assert torch.equal(ia, ib)
    info = _info()
    assert len(info["resid_per_graph"]) == 1 and np.float32(info["resid_per_graph"][0]) == np.float32(info["resid"])


SHAPES = [(4, 500, 2500, 64, 10), (64, 25, 75, 64, 5)]


@pytest.mark.gpu
@pytest.mark.parametrize("shape", SHAPES, ids=["500+2500x4", "25+75x64"])
@pytest.mark.parametrize("eps,tau", [("auto", 0.0), (1.0, 0.0), ("auto", 0.07), (1.0, 0.07)])
def test_batched_matches_per_graph_calls(gpu, shape, eps, tau):
    B, k_lab, m, d, l = shape
    X, Y, yq = _batch(200 + B, B, k_lab, m, d, l)
    res = gpu.laplace_learning_batched(*_cuda(X, Y), k=50, epsilon=eps, tau=tau, targets=torch.as_tensor(yq).cuda())
    torch.cuda.synchronize()
    assert res.pred.shape == (B, m, l) and res.pred.dtype == torch.float64
    assert res.labels.shape == (B, m) and res.correct.shape == (B,) and res.correct.dtype == torch.int64
    info = _info()
    assert info["status"] & 1 == 0 and info["resid"] <= 1e-10
    _check_against_per_graph(gpu, X, Y, yq, 50, eps, tau, res)


@pytest.mark.gpu
def test_disconnected_cluster_leaves_other_graphs_unaffected(gpu):
    B, k_lab, m, d, l = 4, 300, 1264, 32, 5
    X, Y, yq = _batch(300, B, k_lab, m - 64, d, l)
    rng = np.random.default_rng(0)
    far = (50.0 + 0.1 * rng.standard_normal((64, d))).astype(np.float32)
    X = np.stack([np.concatenate([X[b], far if b == 1 else X[b][-64:] + 0.01]) for b in range(B)])
    yq = np.stack([np.concatenate([yq[b], np.zeros(64, dtype=np.int64) if b == 1 else yq[b][-64:]]) for b in range(B)])
    res = gpu.laplace_learning_batched(*_cuda(X, Y), k=50, epsilon=1.0, tau=0.0, targets=torch.as_tensor(yq).cuda())
    torch.cuda.synchronize()
    pred = res.pred.cpu().numpy()
    assert np.all(pred[1, -64:] == 0.0) and np.all(res.labels.cpu().numpy()[1, -64:] == 0)
    _check_against_per_graph(gpu, X, Y, yq, 50, 1.0, 0.0, res, graphs=[0, 2, 3])


@pytest.mark.gpu
def test_deterministic_and_graph_capturable(gpu):
    B, k_lab, m, d, l = 8, 100, 400, 64, 10
    X, Y, yq = _batch(400, B, k_lab, m, d, l)
    X2, _, _ = _batch(500, B, k_lab, m, d, l)
    Xt, Yt, tt = _cuda(X, Y, yq)
    a = gpu.laplace_learning_batched(Xt, Yt, targets=tt)
    b = gpu.laplace_learning_batched(Xt, Yt, targets=tt)
    ref = gpu.laplace_learning_batched(torch.as_tensor(X2).cuda(), Yt, targets=tt)
    torch.cuda.synchronize()
    assert torch.equal(a.pred, b.pred) and torch.equal(a.labels, b.labels) and torch.equal(a.correct, b.correct)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        gpu.laplace_learning_batched(Xt, Yt, targets=tt)
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        c = gpu.laplace_learning_batched(Xt, Yt, targets=tt)
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(c.pred, a.pred) and torch.equal(c.labels, a.labels) and torch.equal(c.correct, a.correct)
    Xt.copy_(torch.as_tensor(X2).cuda())  # replay on new inputs
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(c.pred, ref.pred) and torch.equal(c.labels, ref.labels) and torch.equal(c.correct, ref.correct)


@pytest.mark.gpu
def test_max_iter_warning(gpu, monkeypatch):
    X, Y, _ = _batch(600, 4, 100, 400, 64, 10)
    monkeypatch.setenv("GLL_B200_CG_MAXIT", "2")
    monkeypatch.setenv("GLL_B200_CHECK", "1")
    with warnings.catch_warnings(record=True) as rec:
        warnings.simplefilter("always")
        gpu.laplace_learning_batched(*_cuda(X, Y))
        torch.cuda.synchronize()
    assert any("max iter reached" in str(w.message) for w in rec)
    info = _info()
    assert info["status"] & 1 and max(info["resid_per_graph"]) > 1e-10
