"""Batched independent graphs: the segmented kNN search (gll_knn_segments) and LaplaceLearningSparseHardBatched.

GPU tests check the segmented lists bit for bit against gll_knn on each segment alone, and the batched layer against
per-graph layer calls and the fp64 oracle.  The tests without the gpu marker need no device: argument checks of the C
entry points (which return before any CUDA call), the Python validation and the row reorder helpers.
"""
import ctypes
import os

import numpy as np
import pytest

from oracle import gll_oracle as O

torch = pytest.importorskip("torch")

K = 25


@pytest.fixture(scope="module")
def libmod():
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
def test_reorder_round_trip(libmod):
    from graphlearninglayer_b200.GLL import labeled_first, natural_order

    X = torch.arange(5 * 9 * 3, dtype=torch.float32).reshape(5, 9, 3)
    Xg = labeled_first(X, 4)
    assert Xg.shape == (45, 3)
    assert torch.equal(Xg[:20].reshape(5, 4, 3), X[:, :4]) and torch.equal(Xg[20:].reshape(5, 5, 3), X[:, 4:])
    assert torch.equal(natural_order(Xg, 5, 4), X)


def test_new_entry_points_exported(libmod):
    raw = ctypes.CDLL(libmod.LIB_PATH)
    for nm in ("gll_knn_segments_workspace_bytes", "gll_knn_segments", "gll_knn_segments_units", "gll_batched_workspace_bytes",
               "gll_forward_batched"):
        assert hasattr(raw, nm) and nm in libmod.EXPORTS
    import graphlearninglayer_b200 as pkg

    assert "LaplaceLearningSparseHardBatched" in pkg.__all__


def test_segment_argument_checks(libmod):
    lib, seg = libmod.lib, libmod.seg_ptr_array
    ERR_ARG = -1
    buf = ctypes.c_void_p(16)  # never dereferenced: the checks fail first

    def call(X, n, k, sp, nseg, idx=buf):
        return lib.gll_knn_segments(X, n, 8, k, sp, nseg, idx, buf, None, buf, 1 << 30, None)

    good = seg([0, 30, 60])
    assert call(None, 60, K, good, 2) == ERR_ARG  # null X
    assert call(buf, 60, K, good, 2, idx=None) == ERR_ARG  # null output
    assert call(buf, 60, K, None, 2) == ERR_ARG  # null seg_ptr
    assert call(buf, 60, K, seg([1, 30, 60]), 2) == ERR_ARG  # does not start at 0
    assert call(buf, 60, K, seg([0, 30, 59]), 2) == ERR_ARG  # does not end at n
    assert call(buf, 60, K, seg([0, 40, 30, 60]), 3) == ERR_ARG  # not increasing
    assert call(buf, 60, K, seg([0, 36, 60]), 2) == ERR_ARG  # a segment of 24 < k rows
    assert call(buf, 80, 34, seg([0, 40, 80]), 2) == ERR_ARG  # k > 33
    assert call(buf, 80, 1, seg([0, 40, 80]), 2) == ERR_ARG  # k < 2
    assert call(buf, 60, K, good, 0) == ERR_ARG  # no segment
    assert lib.gll_knn_segments_workspace_bytes(60, 8, K, seg([0, 36, 60]), 2) == 0
    assert lib.gll_knn_segments_workspace_bytes(60, 8, K, good, 2) > 0
    fb = lib.gll_forward_batched
    assert fb(None, buf, 2, 50, 8, K, 3, 10, 1, 0.0, 0.0, 1e-7, 100, buf, buf, 1, buf, 1 << 30, None) == ERR_ARG
    assert fb(buf, buf, 2, 20, 8, K, 3, 10, 1, 0.0, 0.0, 1e-7, 100, buf, buf, 1, buf, 1 << 30, None) == ERR_ARG  # n < k
    assert fb(buf, buf, 2, 50, 8, K, 3, 50, 1, 0.0, 0.0, 1e-7, 100, buf, buf, 1, buf, 1 << 30, None) == ERR_ARG  # k_lab = n
    assert fb(buf, buf, 0, 50, 8, K, 3, 10, 1, 0.0, 0.0, 1e-7, 100, buf, buf, 1, buf, 1 << 30, None) == ERR_ARG  # B = 0
    assert fb(buf, buf, 2, 50, 8, 34, 3, 10, 1, 0.0, 0.0, 1e-7, 100, buf, buf, 1, buf, 1 << 30, None) == ERR_ARG  # k > 33
    assert lib.gll_batched_workspace_bytes(2, 20, 8, K, 3, 10) == 0
    assert lib.gll_batched_workspace_bytes(2, 50, 8, 34, 3, 10) == 0


def test_python_validation(libmod):
    from graphlearninglayer_b200 import LaplaceLearningSparseHardBatched as L

    X = torch.zeros(2, 40, 8)
    Y = torch.zeros(2, 10, 3)
    with pytest.raises(RuntimeError):
        L.apply(X, Y)  # CPU tensors
    with pytest.raises(ValueError):
        L.apply(X[0], Y)  # 2-D features
    with pytest.raises(ValueError):
        L.apply(X, Y[:1])  # batch sizes differ
    with pytest.raises(ValueError):
        L.apply(X, Y[:, :0])  # k_lab = 0
    with pytest.raises(ValueError):
        L.apply(X, torch.zeros(2, 40, 3))  # m = 0
    with pytest.raises(ValueError):
        L.apply(torch.zeros(2, 24, 8), Y)  # n < 25
    with pytest.raises(ValueError):
        L.apply(X, Y, 0.0, "nope")


# ---------------------------------------------------------------------------------------------------- segmented kNN
def _feats(seed, n, d):
    g = np.random.default_rng(seed)
    c = g.standard_normal((8, d))
    X = c[g.integers(0, 8, n)] + 0.6 * g.standard_normal((n, d))
    X /= np.linalg.norm(X, axis=1, keepdims=True)
    return torch.as_tensor(X.astype(np.float32)).cuda()


def _knn(libmod, X, k):
    n, d = X.shape
    idx = torch.empty((n, k), dtype=torch.int32, device=X.device)
    dist = torch.empty((n, k), dtype=torch.float32, device=X.device)
    wsb = libmod.lib.gll_knn_workspace_bytes(n, d, k)
    ws = torch.empty(wsb, dtype=torch.uint8, device=X.device)
    libmod.check(libmod.lib.gll_knn(X.data_ptr(), n, d, k, idx.data_ptr(), dist.data_ptr(), None, ws.data_ptr(), wsb,
                                    torch.cuda.current_stream().cuda_stream), "gll_knn")
    return idx, dist


def _knn_segments(libmod, X, k, seg):
    n, d = X.shape
    sp = libmod.seg_ptr_array(seg)
    idx = torch.empty((n, k), dtype=torch.int32, device=X.device)
    dist = torch.empty((n, k), dtype=torch.float32, device=X.device)
    info = torch.zeros(libmod.INFO_WORDS, dtype=torch.int32, device=X.device)
    wsb = libmod.lib.gll_knn_segments_workspace_bytes(n, d, k, sp, len(seg) - 1)
    assert wsb > 0
    ws = torch.empty(wsb, dtype=torch.uint8, device=X.device)
    libmod.check(libmod.lib.gll_knn_segments(X.data_ptr(), n, d, k, sp, len(seg) - 1, idx.data_ptr(), dist.data_ptr(), info.data_ptr(),
                                             ws.data_ptr(), wsb, torch.cuda.current_stream().cuda_stream), "gll_knn_segments")
    return idx, dist, info


def _check_segments(libmod, X, k, seg, env):
    old = {kk: os.environ.get(kk) for kk in env}
    os.environ.update(env)
    try:
        idx, dist, info = _knn_segments(libmod, X, k, seg)
    finally:
        for kk, v in old.items():
            if v is None:
                os.environ.pop(kk, None)
            else:
                os.environ[kk] = v
    torch.cuda.synchronize()
    for s in range(len(seg) - 1):
        a, b = seg[s], seg[s + 1]
        ri, rd = _knn(libmod, X[a:b].contiguous(), k)
        assert torch.equal(idx[a:b], ri + a), (env, s, b - a)
        assert torch.equal(dist[a:b], rd), (env, s, b - a)
    return info


SIZES = [25, 31, 33, 100, 127, 128, 129, 300, 2000]
ENVS = [{}, {"GLL_B200_KNN_PATH": "simt"}, {"GLL_B200_KNN_PATH": "tc"}, {"GLL_B200_KNN_PATH": "tc", "GLL_B200_KNN_PAIR": "1"},
        {"GLL_B200_KNN_FORCE_FALLBACK": "300"}, {"GLL_B200_KNN_PATH": "simt", "GLL_B200_KNN_FORCE_FALLBACK": "300"}]


@pytest.mark.gpu
@pytest.mark.parametrize("d", [64, 200, 512])
@pytest.mark.parametrize("env", ENVS, ids=["default", "simt", "tc", "tc_pair", "fallback", "simt_fallback"])
def test_segments_bit_identical_to_per_segment(libmod, gpu, d, env):
    sizes = SIZES[::-1] if d == 200 else SIZES  # segment edges land at different column-tile offsets
    seg = np.concatenate([[0], np.cumsum(sizes)]).tolist()
    X = _feats(d, seg[-1], d)
    info = _check_segments(libmod, X, K, seg, env)
    if "GLL_B200_KNN_FORCE_FALLBACK" in env:
        assert int(info[libmod.INFO_KNN_FALLBACK_ROWS]) >= 300


@pytest.mark.gpu
@pytest.mark.parametrize("k", [2, 33])
def test_segments_k_range(libmod, gpu, k):
    seg = [0, 33, 90, 400, 433]
    _check_segments(libmod, _feats(7, seg[-1], 64), k, seg, {})


@pytest.mark.gpu
def test_segments_large_aligned(libmod, gpu):
    # 8 x 10512 rows: > 4 x 148 row tiles, every CTA owns whole row tiles (CTA pairs and the resident A operand by default)
    seg = [10512 * b for b in range(9)]
    X = _feats(3, seg[-1], 128)
    su, uu = ctypes.c_longlong(), ctypes.c_longlong()
    libmod.lib.gll_knn_segments_units(seg[-1], 128, libmod.seg_ptr_array(seg), 8, ctypes.byref(su), ctypes.byref(uu))
    assert 0 < su.value < uu.value / 6
    _check_segments(libmod, X, K, seg, {})


@pytest.mark.gpu
@pytest.mark.parametrize("env", [{}, {"GLL_B200_KNN_PATH": "simt"}], ids=["default", "simt"])
def test_duplicate_graphs_never_cross(libmod, gpu, env):
    A = _feats(11, 300, 64)
    X = torch.cat((A, A, _feats(12, 200, 64))).contiguous()
    seg = [0, 300, 600, 800]
    _check_segments(libmod, X, K, seg, env)
    idx, _, _ = _knn_segments(libmod, X, K, seg)
    rows = torch.arange(800, device=X.device)[:, None]
    lo = torch.as_tensor(np.repeat(seg[:-1], np.diff(seg)), device=X.device)[:, None]
    hi = torch.as_tensor(np.repeat(seg[1:], np.diff(seg)), device=X.device)[:, None]
    assert bool(((idx >= lo) & (idx < hi)).all()) and torch.equal(idx[:, 0:1], rows.int())


# ---------------------------------------------------------------------------------------------------- the layer
def _batch(seed, B, k_lab, m, d, l, sigma=2.0):
    Xs, Ys, ys = [], [], []
    for b in range(B):
        X, Y, _, yq = O.synth_inputs(seed + b, k_lab, m, d, l, sigma)
        Xs.append(X)
        Ys.append(Y)
        ys.append(yq)
    return np.stack(Xs), np.stack(Ys), np.stack(ys)


def _loss(pred, tgt):
    # sum over graphs of the reference's custom_ce_loss (mean over each graph's rows): graph b's gradient is its own loss's
    m = pred.shape[-2]
    oh = torch.nn.functional.one_hot(tgt, pred.shape[-1]).to(pred.dtype)
    return -torch.sum(oh * torch.log(pred + 1e-8)) / m


def _run_batched(pkg, X, Y, yq, tau, eps):
    Xt = torch.as_tensor(X).cuda().requires_grad_(True)
    pred = pkg.LaplaceLearningSparseHardBatched.apply(Xt, Y, tau, eps)
    _loss(pred, torch.as_tensor(yq).cuda()).backward()
    torch.cuda.synchronize()
    return pred.detach(), Xt.grad


def _run_single(pkg, X, Y, yq, tau, eps):
    Xt = torch.as_tensor(X).cuda().requires_grad_(True)
    pred = pkg.LaplaceLearningSparseHard.apply(Xt, Y, tau, eps)
    _loss(pred, torch.as_tensor(yq).cuda()).backward()
    torch.cuda.synchronize()
    return pred.detach(), Xt.grad


@pytest.mark.gpu
@pytest.mark.parametrize("tau,eps", [(0.0, "auto"), (0.07, 1.0)])
def test_batch_of_one_bit_identical(gpu, tau, eps):
    X, Y, yq = _batch(21, 1, 1000, 1000, 128, 10)
    pb, gb = _run_batched(gpu, X, torch.as_tensor(Y).cuda(), yq, tau, eps)
    ps, gs = _run_single(gpu, X[0], torch.as_tensor(Y[0]).cuda(), yq[0], tau, eps)
    assert torch.equal(pb[0], ps) and torch.equal(gb[0], gs)


# (B, k_lab, m, d, l, cluster spread): at d = 512 a spread of 2 makes the predictions one-hot to the last bit (the oracle's dX
# is ~1e-18), so that shape takes the spread bench.py uses for it
CASES = [(4, 1000, 1000, 128, 10, 2.0), (4, 4096, 512, 512, 10, 4.5), (64, 25, 75, 64, 5, 2.0)]


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=["c1x4", "4096+512x4", "25+75x64"])
@pytest.mark.parametrize("setting", ["auto", "fixed_tau", "int64"])
def test_batched_matches_per_graph_and_oracle(gpu, case, setting):
    B, k_lab, m, d, l, sigma = case
    tau, eps = (0.07, 1.0) if setting == "fixed_tau" else (0.0, "auto")
    X, Y, yq = _batch(100 + B, B, k_lab, m, d, l, sigma)
    Yt = torch.as_tensor(Y).cuda()
    if setting == "int64":
        Yt = Yt.long()
    pb, gb = _run_batched(gpu, X, Yt, yq, tau, eps)
    assert pb.shape == (B, m, l) and gb.shape == (B, k_lab + m, d)
    for b in range(B):
        ps, gs = _run_single(gpu, X[b], Yt[b], yq[b], tau, eps)
        assert O.max_rel(pb[b].cpu().numpy(), ps.cpu().numpy()) < 1e-5, b
        assert O.max_rel(gb[b].cpu().numpy(), gs.cpu().numpy()) < 1e-5, b
    for b in sorted({0, B - 1}):
        f, _, _, bw = O.fwd_bwd(X[b].astype(np.float64), Y[b], yq[b], tau, eps, solver="lu")
        assert O.max_rel(pb[b].cpu().numpy(), f.pred) < 1e-5, b
        assert O.max_rel(gb[b].cpu().numpy(), bw.dX) < 1e-5, b


@pytest.mark.gpu
def test_per_graph_state_bit_identical(gpu):
    from graphlearninglayer_b200.GLL import _batched_forward_impl, _forward_impl

    B, k_lab, m, d, l = 3, 200, 500, 64, 6
    n = k_lab + m
    X, Y, _ = _batch(55, B, k_lab, m, d, l)
    Xt, Yt = torch.as_tensor(X).cuda(), torch.as_tensor(Y).cuda()
    _, st, _ = _batched_forward_impl(Xt, Yt, 0.0, "auto")
    N, k = B * n, st.k
    pos = np.concatenate([np.concatenate([b * k_lab + np.arange(k_lab), B * k_lab + b * m + np.arange(m)]) for b in range(B)])
    E = int(st.view("row_ptr", torch.int32, N + 1)[-1])
    rp = st.view("row_ptr", torch.int32, N + 1).cpu().numpy()
    col = st.view("col", torch.int32, E).cpu().numpy()
    arrs = {nm: st.view(nm, torch.float32, E).cpu().numpy() for nm in ("dist", "w")}
    eps = st.view("eps", torch.float32, N).cpu().numpy()
    deg = st.view("deg", torch.float32, N).cpu().numpy()
    kappa = st.view("kappa", torch.int32, N).cpu().numpy()
    kidx = st.view("knn_idx", torch.int32, N * k).cpu().numpy().reshape(N, k)
    for b in range(B):
        _, s1, _ = _forward_impl(Xt[b], Yt[b], 0.0, "auto")
        torch.cuda.synchronize()
        E1 = int(s1.view("row_ptr", torch.int32, n + 1)[-1])
        rp1 = s1.view("row_ptr", torch.int32, n + 1).cpu().numpy()
        col1 = s1.view("col", torch.int32, E1).cpu().numpy()
        p = pos[b * n:(b + 1) * n]
        inv = np.full(N, -1)
        inv[p] = np.arange(n)
        assert np.array_equal(kidx[p], pos[b * n + s1.view("knn_idx", torch.int32, n * k).cpu().numpy().reshape(n, k)])
        for t in range(n):
            e0, e1 = rp[p[t]], rp[p[t] + 1]
            assert np.array_equal(inv[col[e0:e1]], col1[rp1[t]:rp1[t + 1]]), (b, t)
            for nm, a in arrs.items():
                assert np.array_equal(a[e0:e1], s1.view(nm, torch.float32, E1).cpu().numpy()[rp1[t]:rp1[t + 1]]), (nm, b, t)
        assert np.array_equal(eps[p], s1.view("eps", torch.float32, n).cpu().numpy())
        assert np.array_equal(deg[p], s1.view("deg", torch.float32, n).cpu().numpy())
        assert np.array_equal(inv[kappa[p]], s1.view("kappa", torch.int32, n).cpu().numpy())


@pytest.mark.gpu
def test_deterministic_and_graph_capturable(gpu):
    B, k_lab, m, d, l = 8, 250, 1250, 128, 10
    X, Y, yq = _batch(77, B, k_lab, m, d, l)
    X2, _, _ = _batch(88, B, k_lab, m, d, l)
    Yt, tt = torch.as_tensor(Y).cuda(), torch.as_tensor(yq).cuda()
    p1, g1 = _run_batched(gpu, X, Yt, yq, 0.0, "auto")
    p2, g2 = _run_batched(gpu, X, Yt, yq, 0.0, "auto")
    assert torch.equal(p1, p2) and torch.equal(g1, g2)
    ref_p, ref_g = _run_batched(gpu, X2, Yt, yq, 0.0, "auto")

    Xs = torch.as_tensor(X).cuda().requires_grad_(True)

    def step():
        Xs.grad = None
        pred = gpu.LaplaceLearningSparseHardBatched.apply(Xs, Yt, 0.0, "auto")
        _loss(pred, tt).backward()
        return pred.detach(), Xs.grad

    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        step()
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        pc, gc = step()
    with torch.no_grad():
        Xs.copy_(torch.as_tensor(X2).cuda())
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(pc, ref_p) and torch.equal(gc, ref_g)
