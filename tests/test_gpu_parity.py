"""GPU parity tests (run on the B200 box: ``pytest -m gpu``).  Every check goes through the C ABI of
libgll_b200.so -- stage entry points directly, or gll_forward/gll_backward via the autograd Function -- and compares
with the fp64 oracle (oracle/gll_oracle.py) and with the fixtures produced by the unmodified reference GLL.py.

Tolerances (BASELINE.json north_star): kNN index sets bit-exact modulo documented distance ties; pred and dX within
1e-5 relative (max|delta| / max|ref|) in fp32.
"""
import ctypes as C
import os
import warnings

import numpy as np
import pytest
import scipy.sparse as sp

from conftest import golden_names, load_golden
from oracle import gll_oracle as O

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

TOL = 1e-5  # north_star: pred and dL/dfeatures within 1e-5 relative in fp32


@pytest.fixture(scope="module")
def gll():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import graphlearninglayer_b200 as pkg
    from graphlearninglayer_b200 import _lib

    return pkg, _lib


def dev_t(a, dtype):
    return torch.as_tensor(np.ascontiguousarray(a)).to("cuda", dtype).contiguous()


def run_knn(_lib, X, k=25):
    n, d = X.shape
    Xc = dev_t(X, torch.float32)
    idx = torch.empty((n, k), dtype=torch.int32, device="cuda")
    dist = torch.empty((n, k), dtype=torch.float32, device="cuda")
    info = torch.zeros(_lib.INFO_WORDS, dtype=torch.int32, device="cuda")
    wsb = _lib.lib.gll_knn_workspace_bytes(n, d, k)
    ws = torch.empty(wsb, dtype=torch.uint8, device="cuda")
    _lib.check(_lib.lib.gll_knn(Xc.data_ptr(), n, d, k, idx.data_ptr(), dist.data_ptr(), info.data_ptr(), ws.data_ptr(), wsb,
                                torch.cuda.current_stream().cuda_stream), "gll_knn")
    torch.cuda.synchronize()
    return idx, dist, info


def run_graph(_lib, idx, dist):
    n, k = idx.shape
    emax = _lib.lib.gll_max_edges(n, k)
    row_ptr = torch.empty(n + 1, dtype=torch.int32, device="cuda")
    col = torch.empty(emax, dtype=torch.int32, device="cuda")
    dd = torch.empty(emax, dtype=torch.float32, device="cuda")
    info = torch.zeros(_lib.INFO_WORDS, dtype=torch.int32, device="cuda")
    wsb = _lib.lib.gll_graph_workspace_bytes(n, k)
    ws = torch.empty(wsb, dtype=torch.uint8, device="cuda")
    _lib.check(_lib.lib.gll_graph_build(idx.data_ptr(), dist.data_ptr(), n, k, row_ptr.data_ptr(), col.data_ptr(), dd.data_ptr(),
                                        info.data_ptr(), ws.data_ptr(), wsb, torch.cuda.current_stream().cuda_stream),
               "gll_graph_build")
    torch.cuda.synchronize()
    E = int(row_ptr[-1].item())
    assert int(info[_lib.INFO_NNZ].item()) == E
    return row_ptr, col, dd, E


def run_weights(_lib, idx, dist, row_ptr, col, dd, Y, eps, tau):
    n, k = idx.shape
    k_lab, l = Y.shape
    m = n - k_lab
    lp = _lib.lib.gll_padded_classes(l)
    emax = _lib.lib.gll_max_edges(n, k)
    f32, i32 = torch.float32, torch.int32
    Yc = dev_t(Y, f32)
    o = dict(eps=torch.empty(n, dtype=f32, device="cuda"), kappa=torch.empty(n, dtype=i32, device="cuda"),
             w=torch.empty(emax, dtype=f32, device="cuda"), deg=torch.empty(n, dtype=f32, device="cuda"),
             uu_ptr=torch.empty(m + 1, dtype=i32, device="cuda"), uu_col=torch.empty(emax, dtype=i32, device="cuda"),
             uu_val=torch.empty(emax, dtype=f32, device="cuda"), diag=torch.empty(m, dtype=f32, device="cuda"),
             rhs=torch.empty((m, lp), dtype=f32, device="cuda"), ut=torch.zeros((n, lp), dtype=f32, device="cuda"),
             info=torch.zeros(_lib.INFO_WORDS, dtype=i32, device="cuda"))
    wsb = _lib.lib.gll_weights_workspace_bytes(n, k)
    ws = torch.empty(wsb, dtype=torch.uint8, device="cuda")
    auto = isinstance(eps, str)
    _lib.check(_lib.lib.gll_edge_weights(idx.data_ptr(), dist.data_ptr(), row_ptr.data_ptr(), col.data_ptr(), dd.data_ptr(),
                                         Yc.data_ptr(), n, k, l, k_lab, int(auto), 0.0 if auto else float(eps), float(tau),
                                         o["eps"].data_ptr(), o["kappa"].data_ptr(), o["w"].data_ptr(), o["deg"].data_ptr(),
                                         o["uu_ptr"].data_ptr(), o["uu_col"].data_ptr(), o["uu_val"].data_ptr(),
                                         o["diag"].data_ptr(), o["rhs"].data_ptr(), o["ut"].data_ptr(), o["info"].data_ptr(),
                                         ws.data_ptr(), wsb, torch.cuda.current_stream().cuda_stream), "gll_edge_weights")
    torch.cuda.synchronize()
    return o


def run_cg(_lib, Luu: sp.csr_matrix, B: np.ndarray, tol=1e-7, max_iter=5000):
    """Feeds an oracle-built system to gll_cg_solve: diag + negated off-diagonal."""
    m, l = B.shape
    lp = _lib.lib.gll_padded_classes(l)
    dg = Luu.diagonal()
    off = (Luu - sp.diags(dg)).tocsr()
    off.eliminate_zeros()
    off.sort_indices()
    ptr = dev_t(off.indptr, torch.int32)
    col = dev_t(off.indices, torch.int32)
    val = dev_t(-off.data, torch.float32)
    diag = dev_t(dg, torch.float32)
    rhs = torch.zeros((m, lp), dtype=torch.float32, device="cuda")
    rhs[:, :l] = dev_t(B, torch.float32)
    x = torch.empty((m, lp), dtype=torch.float32, device="cuda")
    stat = torch.zeros(4, dtype=torch.int32, device="cuda")
    wsb = _lib.lib.gll_cg_workspace_bytes(m, l)
    ws = torch.empty(wsb, dtype=torch.uint8, device="cuda")
    _lib.check(_lib.lib.gll_cg_solve(ptr.data_ptr(), col.data_ptr(), val.data_ptr(), diag.data_ptr(), rhs.data_ptr(), m, l, tol,
                                     max_iter, x.data_ptr(), stat.data_ptr(), stat[1:].data_ptr(), stat[2:].data_ptr(),
                                     ws.data_ptr(), wsb, torch.cuda.current_stream().cuda_stream), "gll_cg_solve")
    torch.cuda.synchronize()
    s = stat.cpu().numpy()
    return x[:, :l].double().cpu().numpy(), int(s[0]), float(s[1:2].view(np.float32)[0]), int(s[2])


# ----------------------------------------------------------------------------------------------------------------
# K1: kNN
# ----------------------------------------------------------------------------------------------------------------
# d = 13000: the brute-force fallback's row copy (4 d bytes) is past the 48 KB that needs no dynamic shared memory opt-in
KNN_SHAPES = [(0, 300, 500, 64, 10, 2.0), (3, 37, 91, 19, 3, 1.0), (1, 1000, 1000, 128, 10, 3.0),
              (4, 2048, 1024, 512, 10, 4.5), (6, 10, 20, 7, 2, 0.5), (8, 500, 700, 130, 5, 2.0), (9, 30, 270, 13000, 5, 2.0)]


def _set_knn_path(monkeypatch, path):
    """simt: fp32 SIMT Gram; tc: tcgen05 Gram on the scaled fp16 rows, hi.hi (one MMA pass, the default); tc-f16x2: the same
    with the A side split, (hi + lo).hi (two passes)."""
    monkeypatch.setenv("GLL_B200_KNN_PATH", "tc" if path.startswith("tc") else path)
    monkeypatch.setenv("GLL_B200_KNN_SPLIT", "f16x2" if path == "tc-f16x2" else "f16x1")


@pytest.mark.parametrize("path", ["simt", "tc", "tc-f16x2"])  # every Gram path must give the exact lists
@pytest.mark.parametrize("seed,k_lab,m,d,l,sigma", KNN_SHAPES)
def test_knn_bit_exact_vs_oracle(gll, monkeypatch, path, seed, k_lab, m, d, l, sigma):
    _, _lib = gll
    _set_knn_path(monkeypatch, path)
    X, *_ = O.synth_inputs(seed, k_lab, m, d, l, sigma)
    ref_ind, ref_dist = O.exact_knn(X, 25)
    idx, dist, info = run_knn(_lib, X)
    ind = idx.cpu().numpy().astype(np.int64)
    exact, tie, bad = O.knn_sets_match(ind, ref_ind, ref_dist)
    assert bad == 0, (exact, tie, bad)
    assert np.array_equal(ind[:, 0], np.arange(X.shape[0]))  # self first (GLL.py:183 contract)
    same = np.all(ind == ref_ind, axis=1)
    assert same.mean() > 0.999  # order (distance, index); only exact-distance ties computed differently may differ
    d_gpu = dist.cpu().numpy()
    assert np.array_equal(d_gpu[same], ref_dist[same].astype(np.float32))  # fp64 direct differences rounded to fp32


@pytest.mark.parametrize("path", ["simt", "tc", "tc-f16x2"])
def test_knn_duplicates_and_tiny_n(gll, monkeypatch, path):
    _, _lib = gll
    _set_knn_path(monkeypatch, path)
    rng = np.random.default_rng(0)
    X = rng.standard_normal((60, 16)).astype(np.float32)
    X[10:40] = X[10]  # 30 identical points: zero distances, ties broken by index
    idx, dist, _ = run_knn(_lib, X)
    ind, dd = idx.cpu().numpy(), dist.cpu().numpy()
    ref_ind, ref_dist = O.exact_knn(X, 25)
    assert np.array_equal(np.sort(dd, axis=1), np.sort(ref_dist.astype(np.float32), axis=1))
    assert (dd[10:40, :25] == 0).all()
    # n == k edge: every row lists every node
    X2 = rng.standard_normal((25, 8)).astype(np.float32)
    idx2, _, _ = run_knn(_lib, X2)
    assert np.array_equal(np.sort(idx2.cpu().numpy(), axis=1), np.tile(np.arange(25), (25, 1)))


@pytest.mark.parametrize("path", ["tc", "tc-f16x2"])
@pytest.mark.parametrize("scale", [1.0, 3.0e4, 2.0e-6, "ragged"])
def test_knn_f16_split_any_feature_scale(gll, monkeypatch, scale, path):
    """The fp16 split scales X by a power of two derived from max |x_i|^2, so features far outside fp16's range (or rows of very
    different norms) must give the same exact lists as the SIMT path, with (almost) no rows sent to the brute-force fallback."""
    _, _lib = gll
    X, *_ = O.synth_inputs(5, 1500, 1100, 192, 10, 3.0)
    if scale == "ragged":
        X = X * np.logspace(-3, 3, X.shape[0], dtype=np.float32)[np.random.default_rng(0).permutation(X.shape[0]), None]
    else:
        X = (X * np.float32(scale)).astype(np.float32)
    _set_knn_path(monkeypatch, "simt")
    i_s, d_s, _ = run_knn(_lib, X)
    _set_knn_path(monkeypatch, path)
    i_h, d_h, info = run_knn(_lib, X)
    assert torch.equal(i_s, i_h) and torch.equal(d_s, d_h)
    if scale != "ragged":  # rows 1e6 apart in norm: small rows are legitimately unprovable against the largest row's error
        assert int(info[_lib.INFO_KNN_FALLBACK_ROWS].item()) < 0.02 * X.shape[0]


def test_knn_one_pass_full_size_matches_two_pass(gll, monkeypatch):
    """C2 size: one MMA pass (hi.hi, the default) and two ((hi + lo).hi) select the same exact lists, neither needs the
    fallback."""
    _, _lib = gll
    X, *_ = O.synth_inputs(1, 10000, 512, 512, 10, 4.5)
    _set_knn_path(monkeypatch, "tc")
    i0, d0, info0 = run_knn(_lib, X)
    _set_knn_path(monkeypatch, "tc-f16x2")
    i1, d1, info1 = run_knn(_lib, X)
    assert torch.equal(i0, i1) and torch.equal(d0, d1)
    # one pass carries a bound of ~1.3e-3 on d^2 against ~8e-4 for two: a handful of rows out of 10512 may need the fallback
    assert int(info0[_lib.INFO_KNN_FALLBACK_ROWS].item()) <= 4 and int(info1[_lib.INFO_KNN_FALLBACK_ROWS].item()) == 0


@pytest.mark.parametrize("forced", [1, 3, 700, 5000])
def test_knn_fallback_rows_dealt_over_all_ctas(gll, monkeypatch, forced):
    """Rows whose completeness proof fails are redone by exact brute force; few rows are split into column chunks over all
    CTAs and merged (1, 3: chunked; 700, 5000: one or more rows per CTA).  Forced here for the first rows: same lists."""
    _, _lib = gll
    X, *_ = O.synth_inputs(12, 3000, 1777, 200, 10, 3.5)
    i0, d0, info0 = run_knn(_lib, X)
    monkeypatch.setenv("GLL_B200_KNN_FORCE_FALLBACK", str(forced))
    i1, d1, info1 = run_knn(_lib, X)
    assert int(info1[_lib.INFO_KNN_FALLBACK_ROWS].item()) >= min(forced, X.shape[0])
    assert torch.equal(i0, i1) and torch.equal(d0, d1)


@pytest.mark.parametrize("passes", [1, 2])
@pytest.mark.parametrize("d", [512, 200])
def test_tensor_core_accumulator_matches_split_model(gll, monkeypatch, passes, d):
    """What the tensor core accumulates for one (row tile, column tile) unit against the numpy model of the fp16 operands
    (oracle/split_model.py), within the fp32-accumulation budget of knn_tc_err_coef -- one pass (hi.hi) and two
    ((hi + lo).hi; fp16 SUBNORMAL `lo` operands must take part there)."""
    from oracle import split_model as S

    _, _lib = gll
    _set_knn_path(monkeypatch, "tc-f16x2" if passes == 2 else "tc")
    X, *_ = O.synth_inputs(13, 600, 680, d, 10, 4.5)
    n = X.shape[0]
    rt, ct = 3, 2
    Xt = dev_t(X, torch.float32)
    acc = torch.empty((128, 256), dtype=torch.float32, device="cuda")
    rscale = torch.empty(n, dtype=torch.float32, device="cuda")
    wsb = _lib.lib.gll_knn_workspace_bytes(n, d, 25)
    ws = torch.empty(wsb, dtype=torch.uint8, device="cuda")
    _lib.check(_lib.lib.gll_debug_gram_tile(Xt.data_ptr(), n, d, rt, ct, acc.data_ptr(), rscale.data_ptr(), ws.data_ptr(), wsb,
                                            torch.cuda.current_stream().cuda_stream), "gll_debug_gram_tile")
    torch.cuda.synchronize()
    rows, cols = np.arange(rt * 128, rt * 128 + 128), np.arange(ct * 256, ct * 256 + 256)
    hi, lo, E, sq, rho = S.split_f16(X)
    assert np.array_equal(rscale.cpu().numpy(), np.ldexp(np.float32(1), E).astype(np.float32))
    a = (hi.astype(np.float64) + (lo.astype(np.float64) if passes == 2 else 0.0))[rows]
    b = hi.astype(np.float64)[cols]
    want = a @ b.T
    got = acc.cpu().numpy().astype(np.float64)
    steps = passes * int(np.ceil(d / 16)) + 8
    budget = steps * 2.0 ** -22 * ((a ** 2).sum(axis=1)[:, None] + (b ** 2).sum(axis=1)[None, :])  # un-margined share of the coefficient
    err = np.abs(got - want)
    assert float((err / budget).max()) <= 1.0, float((err / budget).max())


def test_knn_paths_agree_and_tc_is_used(gll, monkeypatch):
    """Default dispatch takes the tensor-core kernel at this size; its lists are identical to the SIMT kernel's."""
    _, _lib = gll
    X, *_ = O.synth_inputs(12, 3000, 1777, 200, 10, 3.5)  # n, d not multiples of the tile sizes
    names = _lib.kernel_names()
    tc_id, simt_id = names.index("knn_gram_topk_tcgen05"), names.index("knn_gram_topk_simt")
    monkeypatch.delenv("GLL_B200_KNN_PATH", raising=False)
    before = _lib.launch_count(tc_id)
    i_tc, d_tc, info = run_knn(_lib, X)
    assert _lib.launch_count(tc_id) == before + 1
    monkeypatch.setenv("GLL_B200_KNN_PATH", "simt")
    before = _lib.launch_count(simt_id)
    i_s, d_s, _ = run_knn(_lib, X)
    assert _lib.launch_count(simt_id) == before + 1
    assert torch.equal(i_tc, i_s) and torch.equal(d_tc, d_s)
    assert int(info[_lib.INFO_KNN_FALLBACK_ROWS].item()) < 0.02 * X.shape[0]


def test_knn_cta_pair_variant(gll, monkeypatch):
    """Cluster-of-2 variant of the tensor-core kernel (tcgen05.mma.cta_group::2, M = 256: each CTA stages its 128 rows of A and
    half of the B tile): identical lists."""
    _, _lib = gll
    X, *_ = O.synth_inputs(12, 3000, 1777, 200, 10, 3.5)
    monkeypatch.setenv("GLL_B200_KNN_PATH", "tc")
    monkeypatch.setenv("GLL_B200_KNN_PAIR", "0")
    i0, d0, _ = run_knn(_lib, X)
    monkeypatch.setenv("GLL_B200_KNN_PAIR", "1")
    i1, d1, _ = run_knn(_lib, X)
    assert torch.equal(i0, i1) and torch.equal(d0, d1)


@pytest.mark.parametrize("pair", ["0", "1"])
@pytest.mark.parametrize("split", ["", "f16x2"])
@pytest.mark.parametrize("d", [64, 200])
def test_knn_resident_a_operand(gll, monkeypatch, pair, split, d):
    """Resident-A mode of the tensor-core kernel (the K blocks of a row tile's A operand stay in shared memory while the CTA
    sweeps column tiles; default on large graphs only): forced on a graph whose CTAs change row tiles several times, with
    and without CTA pairs, one and two MMA passes -- identical lists."""
    _, _lib = gll
    X, *_ = O.synth_inputs(13, 3000, 2900, d, 10, 3.5)
    monkeypatch.setenv("GLL_B200_KNN_PATH", "tc")
    monkeypatch.setenv("GLL_B200_KNN_PAIR", pair)
    if split:
        monkeypatch.setenv("GLL_B200_KNN_SPLIT", split)
    monkeypatch.setenv("GLL_B200_KNN_ARES", "0")
    i0, d0, _ = run_knn(_lib, X)
    monkeypatch.setenv("GLL_B200_KNN_ARES", "1")
    i1, d1, _ = run_knn(_lib, X)
    assert torch.equal(i0, i1) and torch.equal(d0, d1)
    ref_idx, _ = O.exact_knn_rows(X, np.arange(0, X.shape[0], 53), 25)
    assert np.array_equal(i1.cpu().numpy()[::53], ref_idx)


def test_knn_full_size_properties(gll):
    """C4 size (n=16384, d=512): properties that need no oracle: self first, sorted distances, symmetric distances on
    mutual pairs, distances equal to a torch fp64 recomputation on the chosen pairs, and k-th distance <= any
    non-neighbour distance on sampled rows."""
    _, _lib = gll
    X, *_ = O.synth_inputs(2, 2048, 14336, 512, 10, 4.5)
    idx, dist, info = run_knn(_lib, X)
    ind = idx.long()
    n = X.shape[0]
    assert torch.equal(ind[:, 0].cpu(), torch.arange(n))
    assert bool((dist[:, 1:] >= dist[:, :-1]).all())
    Xd = torch.as_tensor(X).cuda().double()
    rows = torch.arange(0, n, 97, device="cuda")
    ref = torch.cdist(Xd[rows], Xd, compute_mode="donot_use_mm_for_euclid_dist")
    ref[torch.arange(len(rows)), rows] = -1.0
    kth = torch.sort(ref, dim=1).values[:, :25]
    kth[:, 0] = 0
    assert torch.equal(kth.float(), dist[rows])
    got = torch.gather(ref, 1, ind[rows])
    got[:, 0] = 0
    assert torch.equal(got.float(), dist[rows])


# ----------------------------------------------------------------------------------------------------------------
# K2 + K3: graph and weights
# ----------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("eps,tau", [("auto", 0.0), (1.0, 0.07)])
@pytest.mark.parametrize("seed,k_lab,m,d,l,sigma", [(0, 300, 500, 64, 10, 2.0), (3, 37, 91, 19, 3, 1.0)])
def test_graph_and_weights_vs_oracle(gll, seed, k_lab, m, d, l, sigma, eps, tau):
    _, _lib = gll
    X, Y, *_ = O.synth_inputs(seed, k_lab, m, d, l, sigma)
    f = O.forward(X, Y, tau, eps, solver="lu")
    g = f.graph
    idx = dev_t(g.knn_ind, torch.int32)
    dist = dev_t(g.knn_dist, torch.float32)
    row_ptr, col, dd, E = run_graph(_lib, idx, dist)
    assert np.array_equal(row_ptr.cpu().numpy(), g.dist.indptr)          # bit-exact integer work
    assert np.array_equal(col[:E].cpu().numpy(), g.dist.indices)
    assert np.array_equal(dd[:E].cpu().numpy(), g.dist.data.astype(np.float32))
    o = run_weights(_lib, idx, dist, row_ptr, col, dd, Y, eps, tau)
    assert np.array_equal(o["eps"].cpu().numpy(), g.eps.astype(np.float32))
    if eps == "auto":
        assert np.array_equal(o["kappa"].cpu().numpy(), g.kappa)
    assert O.max_rel(o["w"][:E].cpu().numpy(), g.W.data) < 1e-6
    assert O.max_rel(o["deg"].cpu().numpy(), f.deg) < 1e-6
    assert O.max_rel(o["diag"].cpu().numpy(), f.Luu.diagonal()) < 1e-6
    assert O.max_rel(o["rhs"][:, :l].cpu().numpy(), f.B) < 1e-6
    off = (f.Luu - sp.diags(f.Luu.diagonal())).tocsr()
    off.eliminate_zeros()
    off.sort_indices()
    nuu = int(o["uu_ptr"][-1].item())
    assert np.array_equal(o["uu_ptr"].cpu().numpy(), off.indptr)
    assert np.array_equal(o["uu_col"][:nuu].cpu().numpy(), off.indices)
    assert O.max_rel(o["uu_val"][:nuu].cpu().numpy(), -off.data) < 1e-6
    assert np.array_equal(o["ut"][:k_lab, :l].cpu().numpy(), Y)


def test_graph_drops_zero_distance_edges(gll):
    """sparse.find at GLL.py:198 drops exact zeros: duplicate points are not edges."""
    _, _lib = gll
    rng = np.random.default_rng(1)
    X = rng.standard_normal((80, 12)).astype(np.float32)
    X[5] = X[6]
    ind, dist = O.exact_knn(X, 25)
    g = O.build_graph(X, 25, 1.0, knn=(ind, dist))
    row_ptr, col, dd, E = run_graph(_lib, dev_t(ind, torch.int32), dev_t(dist, torch.float32))
    assert np.array_equal(row_ptr.cpu().numpy(), g.dist.indptr)
    assert np.array_equal(col[:E].cpu().numpy(), g.dist.indices)
    assert 6 not in col[row_ptr[5]:row_ptr[6]].cpu().numpy()


# ----------------------------------------------------------------------------------------------------------------
# K4: CG
# ----------------------------------------------------------------------------------------------------------------
# "": the dispatch by size (here the multi-CTA on-chip kernel: the stage entry point passes no sparsity hint); "cluster": the
# eight-CTA cluster kernel where its item budget allows (up to 12 class columns here), the multi-CTA kernel beyond;
# "resident": the multi-CTA on-chip kernel for every l; "streaming": the global-memory kernel that only ~1M-row systems reach on
# their own, forced so that it is covered at a size the CPU checker can solve
@pytest.mark.parametrize("path", ["", "streaming", "resident", "cluster"])
@pytest.mark.parametrize("l", [1, 3, 10, 37, 100, 150])  # 150 > 128 class columns: solved in column chunks
def test_cg_vs_direct_solve(gll, monkeypatch, l, path):
    _, _lib = gll
    if path:
        monkeypatch.setenv("GLL_B200_CG_PATH", path)
    X, Y, *_ = O.synth_inputs(3, 160, 1500, 24, l, 1.5)
    f = O.forward(X, Y, 0.02, 1.0, solver="lu")
    x, iters, resid, status = run_cg(_lib, f.Luu, f.B, tol=1e-7)
    assert status == 0 and 0 < iters < 2000 and resid <= 1e-7
    assert O.max_rel(x, f.pred) < TOL
    true_res = np.sqrt(((f.Luu @ x - f.B) ** 2).sum(axis=0)).max()
    assert true_res < 5e-5  # fp32 storage of A and x bounds the true residual


@pytest.mark.parametrize("m,l", [(64, 1), (65, 13), (511, 10), (2048, 3), (2048, 16), (700, 40), (700, 100)])
def test_cg_cluster_kernel_edge_sizes(gll, monkeypatch, m, l):
    """The eight-CTA cluster kernel (GLL_CG_KERNEL_CLUSTER = 3) at the edges of its range (64 and 2048 rows, a last CTA with one
    row or none, one class, up to four items per thread; 40 classes at 700 rows are 3 items per thread).  100 classes at 700 rows
    are 8 items per thread, beyond its budget: that system falls through to the multi-CTA kernel (GLL_CG_KERNEL_RESIDENT = 1).
    Forced: the stage entry point passes no sparsity hint and would pick the other kernels."""
    _, _lib = gll
    monkeypatch.setenv("GLL_B200_CG_PATH", "cluster")
    assert _lib.lib.gll_cg_kernel(m, l, 0.0) == (1 if (m, l) == (700, 100) else 3)
    X, Y, *_ = O.synth_inputs(31 + m + l, 120, m, 20, l, 1.5)
    f = O.forward(X, Y, 0.03, 1.0, solver="lu")
    x, iters, resid, status = run_cg(_lib, f.Luu, f.B, tol=1e-7)
    assert status == 0 and 0 < iters < 500 and resid <= 1e-7
    assert O.max_rel(x, f.pred) < TOL


def test_knn_cta_pairs_by_default_with_an_odd_number_of_row_tiles(gll):
    """From 8192 rows the search runs on CTA pairs by default; 8300 rows = 65 row tiles: the last pair has one real row tile."""
    _, _lib = gll
    X, *_ = O.synth_inputs(41, 4000, 4300, 32, 10, 3.0)
    idx, dist, info = run_knn(_lib, X)
    rows = np.arange(0, X.shape[0], 37)
    rows = np.concatenate([rows, np.arange(X.shape[0] - 140, X.shape[0])])   # all of the last (ragged) row tiles
    ref_idx, ref_dist = O.exact_knn_rows(X, rows, 25)
    assert np.array_equal(idx.cpu().numpy()[rows], ref_idx)
    assert np.array_equal(dist.cpu().numpy()[rows], ref_dist.astype(np.float32))


@pytest.mark.parametrize("path", ["", "streaming", "small", "cluster"])
def test_cg_zero_rhs_column_and_maxiter(gll, monkeypatch, path):
    _, _lib = gll
    if path:
        monkeypatch.setenv("GLL_B200_CG_PATH", path)  # "small": the one-CTA kernel (<= 512 rows)
    X, Y, *_ = O.synth_inputs(5, 100, 400 if path == "small" else 900, 16, 4, 1.5)
    f = O.forward(X, Y, 0.05, 1.0, solver="lu")
    B = f.B.copy()
    B[:, 2] = 0.0  # a frozen column from the start (the per-column mask of GLL.py:262-263 must not divide 0/0)
    x, iters, resid, status = run_cg(_lib, f.Luu, B, tol=1e-7)
    assert status == 0 and np.all(x[:, 2] == 0) and np.isfinite(x).all()
    ref = O.solve(f.Luu, B, "lu")
    assert O.max_rel(x, ref) < TOL
    x2, it2, _, status2 = run_cg(_lib, f.Luu, f.B, tol=1e-12, max_iter=3)
    assert it2 == 3 and status2 & 1  # GLL_STATUS_CG_NOT_CONVERGED <-> 'max iter reached' (GLL.py:273-274)


def test_cg_relative_tolerance(gll):
    _, _lib = gll
    X, Y, *_ = O.synth_inputs(5, 100, 900, 16, 4, 1.5)
    f = O.forward(X, Y, 0.05, 1.0, solver="lu")
    B = f.B * 1e4
    x, iters, resid, status = run_cg(_lib, f.Luu, B, tol=-1e-7)
    assert status == 0
    assert O.max_rel(x, f.pred * 1e4) < TOL


# ----------------------------------------------------------------------------------------------------------------
# end to end through the autograd Function (gll_forward / gll_backward)
# ----------------------------------------------------------------------------------------------------------------
def layer_fwd_bwd(pkg, X, Y, yq, tau, eps):
    Xt = torch.as_tensor(X).cuda().requires_grad_(True)
    Yt = torch.as_tensor(Y).cuda()
    pred = pkg.LaplaceLearningSparseHard.apply(Xt, Yt, tau, eps)
    tgt = torch.nn.functional.one_hot(torch.as_tensor(yq).cuda(), pred.shape[1]).to(pred.dtype)
    loss = -torch.sum(tgt * torch.log(pred + 1e-8)) / pred.shape[0]  # custom_ce_loss, losses.py:128-136
    loss.backward()
    torch.cuda.synchronize()
    return pred.detach(), loss.detach(), Xt.grad


@pytest.mark.parametrize("name", golden_names())
def test_layer_matches_reference_fixture(gll, name):
    """Fixtures were produced by the UNMODIFIED /root/reference/GLL.py (oracle/make_golden.py)."""
    pkg, _lib = gll
    g, X, Y, yq = load_golden(name)
    pred, loss, dX = layer_fwd_bwd(pkg, X, Y, yq, g["tau_arg"], g["eps_arg"])
    assert pred.dtype == torch.float64 and dX.dtype == torch.float32  # GLL.py:66,154
    assert O.max_rel(pred.cpu().numpy(), g["pred"]) < TOL
    assert abs(loss.item() - float(g["loss"])) < 1e-5 * max(1.0, abs(float(g["loss"])))
    s = int(g["dX_stride"])
    dXn = dX.cpu().numpy()
    assert np.abs(dXn[::s] - g["dX"]).max() <= TOL * float(g["dX_absmax"])
    assert abs(np.linalg.norm(dXn.astype(np.float64)) / float(g["dX_fro"]) - 1) < TOL
    assert np.abs(dXn.astype(np.float64).sum(axis=0) - g["dX_colsum"]).max() <= 10 * TOL * float(g["dX_absmax"])
    info = pkg.last_info()
    assert info["status"] & ~_lib.STATUS_KNN_FALLBACK == 0, info


@pytest.mark.parametrize("eps,tau", [("auto", 0.0), (1.0, 0.07), ("auto", 0.07)])
def test_layer_vs_oracle_mid_size(gll, eps, tau):
    """n = 6144 (above the LU fixtures, oracle solves by fp64 CG to 1e-13)."""
    pkg, _ = gll
    X, Y, _, yq = O.synth_inputs(21, 1024, 5120, 256, 10, 3.0)
    f, loss_ref, gout, bw = O.fwd_bwd(X, Y, yq, tau, eps, solver="cg")
    pred, loss, dX = layer_fwd_bwd(pkg, X, Y, yq, tau, eps)
    assert O.max_rel(pred.cpu().numpy(), f.pred) < TOL
    assert O.max_rel(dX.cpu().numpy(), bw.dX) < TOL


@pytest.mark.parametrize("eps,tau", [("auto", 0.0), (1.0, 0.07)])
def test_layer_vs_oracle_c4_full_size(gll, eps, tau):
    """BASELINE.json configs[3] at its own size: 2048 labeled + 14336 unlabeled nodes, d = 512, 10 classes, both bandwidth
    modes (the north star's parity target: pred and dL/dfeatures within 1e-5 relative of the reference path,
    GLL.py:53,93,146-159; the oracle solves by fp64 CG to 1e-13 because SuperLU needs minutes at this size)."""
    pkg, _lib = gll
    X, Y, _, yq = O.synth_inputs(2000, 2048, 14336, 512, 10, 4.5)
    f, loss_ref, gout, bw = O.fwd_bwd(X, Y, yq, tau, eps, solver="cg")
    pred, loss, dX = layer_fwd_bwd(pkg, X, Y, yq, tau, eps)
    info = pkg.last_info()
    assert info["status"] & ~_lib.STATUS_KNN_FALLBACK == 0 and info["knn_fallback_rows"] <= 8, info  # rows redone exactly
    assert info["nnz"] == f.graph.W.nnz                      # same union graph as the oracle's exact search
    assert O.max_rel(pred.cpu().numpy(), f.pred) < TOL
    assert abs(loss.item() - loss_ref) < 1e-5 * max(1.0, abs(loss_ref))
    assert O.max_rel(dX.cpu().numpy(), bw.dX) < TOL


def test_layer_more_than_128_classes(gll):
    """The reference layer has no class limit (GLL.py:53 solves all columns of label_matrix); the CG kernels take 128 class
    columns per launch, gll_forward / gll_backward chunk the rest."""
    pkg, _lib = gll
    X, Y, _, yq = O.synth_inputs(5, 300, 700, 32, 130, 1.5)
    f, loss_ref, gout, bw = O.fwd_bwd(X, Y, yq, 0.05, "auto", solver="lu")
    pred, loss, dX = layer_fwd_bwd(pkg, X, Y, yq, 0.05, "auto")
    assert pkg.last_info()["status"] == 0
    assert O.max_rel(pred.cpu().numpy(), f.pred) < TOL
    assert O.max_rel(dX.cpu().numpy(), bw.dX) < TOL


def test_graphed_step_replays_the_layer(gll):
    """forward + loss + backward captured into CUDA graphs once and replayed on NEW inputs of the same shape: bit-equal to
    the eager call (the library's launches carry no host-side data dependence; SURVEY.md section 7 step 5)."""
    pkg, _lib = gll
    from graphlearninglayer_b200.graphed import GraphedStep
    from graphlearninglayer_b200.losses import custom_ce_loss

    k_lab, m, d, l = 700, 500, 64, 10
    step = GraphedStep(k_lab + m, d, k_lab, l, "cuda", tau=0.0, epsilon="auto")
    head = GraphedStep(k_lab + m, d, k_lab, l, "cuda", tau=0.0, epsilon="auto", loss_head=True)  # layer + loss in one node
    for seed in (3, 4):
        X, Y, _, yq = O.synth_inputs(seed, k_lab, m, d, l, 2.0)
        Xt = torch.as_tensor(X).cuda().requires_grad_(True)
        Yt, yt = torch.as_tensor(Y).cuda(), torch.as_tensor(yq).cuda()
        pred = pkg.LaplaceLearningSparseHard.apply(Xt, Yt, 0.0, "auto")
        loss = custom_ce_loss(pred, yt)
        loss.backward()
        before = _lib.launch_count()
        loss_g = step(torch.as_tensor(X).cuda(), Yt, yt)
        assert _lib.launch_count() == before          # nothing was launched through the API: the graphs replayed
        assert torch.equal(step.pred, pred.detach()) and torch.equal(step.dX, Xt.grad)
        assert loss_g.item() == loss.item()
        loss_h = head(torch.as_tensor(X).cuda(), Yt, yt)
        assert loss_h.item() == loss.item() and torch.equal(head.pred, pred.detach()) and torch.equal(head.dX, Xt.grad)
    f, loss_ref, gout, bw = O.fwd_bwd(X, Y, yq, 0.0, "auto", solver="lu")
    assert O.max_rel(step.pred.cpu().numpy(), f.pred) < TOL and O.max_rel(step.dX.cpu().numpy(), bw.dX) < TOL


@pytest.mark.parametrize("eps,tau", [("auto", 0.0), (1.0, 0.07)])
def test_base_set_evaluator_equals_full_search(gll, eps, tau):
    """utils.py:596-621 (test_network): the same base rows in every call, only the batch changes.  The evaluator searches the
    base set among itself ONCE; per batch its predictions and kNN lists must be bit-identical to the layer / gll_knn on the
    concatenated matrix (n_base = 1500 is not a multiple of the 128-row tile; batches of different sizes)."""
    pkg, _lib = gll
    from graphlearninglayer_b200.evalcache import BaseSetEvaluator

    Xall, Y, _, _ = O.synth_inputs(17, 1500, 1100, 96, 10, 2.5)
    base = torch.as_tensor(Xall[:1500]).cuda()
    Yt = torch.as_tensor(Y).cuda()
    ev = BaseSetEvaluator(base, Yt, tau=tau, epsilon=eps)
    for lo, hi in ((1500, 1800), (1800, 2311), (2311, 2600)):
        batch = torch.as_tensor(Xall[lo:hi]).cuda()
        pred = ev(batch)
        full = torch.cat((base, batch), 0)
        with torch.no_grad():
            ref = pkg.LaplaceLearningSparseHard.apply(full, Yt, tau, eps)
        i_ref, d_ref, _ = run_knn(_lib, full.cpu().numpy())
        assert torch.equal(ev.knn_idx, i_ref) and torch.equal(ev.knn_dist, d_ref)
        assert pred.dtype == ref.dtype and torch.equal(pred, ref)
        assert int(ev.info[_lib.INFO_STATUS].item()) & ~_lib.STATUS_KNN_FALLBACK == 0
    f = O.forward(np.concatenate([Xall[:1500], Xall[2311:2600]]), Y, tau, eps, solver="lu")
    assert O.max_rel(pred.cpu().numpy(), f.pred) < TOL


def test_layer_full_size_properties(gll):
    """C4 size (2048 + 14336, d=512): invariants of SURVEY 4 that need no oracle."""
    pkg, _lib = gll
    X, Y, _, yq = O.synth_inputs(2, 2048, 14336, 512, 10, 4.5)
    pred, loss, dX = layer_fwd_bwd(pkg, X, Y, yq, 0.0, "auto")
    p = pred.cpu().numpy()
    assert np.abs(p.sum(axis=1) - 1.0).max() < 2e-5      # tau = 0: harmonic extension of one-hot rows sums to 1
    assert p.min() > -1e-5 and p.max() < 1 + 1e-5        # discrete maximum principle
    g = dX.cpu().numpy().astype(np.float64)
    assert np.isfinite(g).all()
    assert np.abs(g.sum(axis=0)).max() <= 1e-4 * np.abs(g).sum(axis=0).max()  # sum_i dX_i = 0: loss is translation invariant
    assert np.linalg.norm(g[:2048]) > 0.01 * np.linalg.norm(g)               # base rows get gradient too
    info = pkg.last_info()
    assert info["status"] & ~_lib.STATUS_KNN_FALLBACK == 0 and info["cg_iters_fwd"] > 0 and info["cg_iters_bwd"] > 0
    # linearity of the backward in grad_output: bwd(2 g) = 2 bwd(g)
    Xt = torch.as_tensor(X).cuda().requires_grad_(True)
    pr = pkg.LaplaceLearningSparseHard.apply(Xt, torch.as_tensor(Y).cuda(), 0.0, "auto")
    gsel = torch.randn(pr.shape, dtype=pr.dtype, device="cuda", generator=torch.Generator("cuda").manual_seed(0))
    (g1,) = torch.autograd.grad((pr * gsel).sum(), Xt, retain_graph=True)
    (g2,) = torch.autograd.grad((pr * (2 * gsel)).sum(), Xt)
    assert torch.allclose(g2, 2 * g1, rtol=0, atol=2e-5 * g1.abs().max().item())


def test_layer_api_contract(gll):
    pkg, _ = gll
    X, Y, _, yq = O.synth_inputs(9, 100, 200, 32, 5, 1.5)
    Xt = torch.as_tensor(X).cuda()
    # two-argument call: tau = 0, epsilon = 'auto', int64 labels (train_and_adversarial.py:545,552)
    p2 = pkg.LaplaceLearningSparseHard.apply(Xt, torch.as_tensor(Y).long().cuda())
    p4 = pkg.LaplaceLearningSparseHard.apply(Xt, torch.as_tensor(Y).cuda(), 0, "auto")
    assert torch.equal(p2, p4) and p2.shape == (200, 5) and p2.dtype == torch.float64 and p2.is_cuda
    with torch.no_grad():  # train_and_adversarial.py:579-595
        p3 = pkg.LaplaceLearningSparseHard.apply(Xt, torch.as_tensor(Y).cuda())
    assert torch.equal(p3, p2)
    # callers mutate the output in place (adversarial.py:691) and then still backpropagate
    Xg = Xt.clone().requires_grad_(True)
    out = pkg.LaplaceLearningSparseHard.apply(Xg, torch.as_tensor(Y).cuda(), 0.07, 1.0)
    ref = O.forward(X, Y, 0.07, 1.0)
    out2 = out.clone()
    out2[0, 0] = -1000000
    out2.sum().backward()
    assert Xg.grad is not None and Xg.grad.shape == Xg.shape and torch.isfinite(Xg.grad).all()
    assert O.max_rel(out.detach().cpu().numpy(), ref.pred) < TOL
    with pytest.raises(RuntimeError):  # no CPU path by design
        pkg.LaplaceLearningSparseHard.apply(torch.as_tensor(X), torch.as_tensor(Y))
    with pytest.raises(ValueError):
        pkg.LaplaceLearningSparseHard.apply(Xt, torch.as_tensor(Y).cuda(), 0, "banana")


def test_layer_is_deterministic(gll):
    pkg, _ = gll
    X, Y, _, yq = O.synth_inputs(1, 1000, 1000, 128, 10, 3.0)
    a = layer_fwd_bwd(pkg, X, Y, yq, 0.0, "auto")
    b = layer_fwd_bwd(pkg, X, Y, yq, 0.0, "auto")
    assert torch.equal(a[0], b[0]) and torch.equal(a[2], b[2])  # no floating-point atomics anywhere


def test_eps_tiny_warns(gll, monkeypatch):
    pkg, _ = gll
    monkeypatch.setenv("GLL_B200_CHECK", "1")
    rng = np.random.default_rng(0)
    X = rng.standard_normal((80, 8)).astype(np.float32)
    X[30:60] = X[30]  # >= 24 duplicates: epsilon_i = 0 (GLL.py:240-241 warns)
    Y = np.eye(4, dtype=np.float32)[np.arange(20) % 4]
    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter("always")
        pkg.LaplaceLearningSparseHard.apply(torch.as_tensor(X).cuda(), torch.as_tensor(Y).cuda())
        torch.cuda.synchronize()
    assert any("Epsilon in KNN" in str(x.message) for x in w)
    # default mode: no host sync inside the call; the status word is copied behind it and the warning comes with a later call
    monkeypatch.delenv("GLL_B200_CHECK")
    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter("always")
        pkg.LaplaceLearningSparseHard.apply(torch.as_tensor(X).cuda(), torch.as_tensor(Y).cuda())
        torch.cuda.synchronize()
        first = [x for x in w if "Epsilon in KNN" in str(x.message)]
        pkg.LaplaceLearningSparseHard.apply(torch.as_tensor(X).cuda(), torch.as_tensor(Y).cuda())
        torch.cuda.synchronize()
        pkg.LaplaceLearningSparseHard.apply(torch.as_tensor(X).cuda(), torch.as_tensor(Y).cuda())
    assert any("Epsilon in KNN" in str(x.message) for x in w) and len(first) <= 1


# ----------------------------------------------------------------------------------------------------------------
# numpy / scipy wrappers (utils.py:570-593 call sites)
# ----------------------------------------------------------------------------------------------------------------
def test_knn_sym_dist_wrapper(gll):
    pkg, _ = gll
    X, *_ = O.synth_inputs(0, 300, 500, 64, 10, 2.0)
    g = O.build_graph(X, 25, "auto")
    W, V, mod_V, Cm, knn_ind = pkg.knn_sym_dist(X, 25, "auto")
    assert sp.issparse(W) and W.shape == (800, 800)
    assert np.array_equal(W.indptr, g.W.indptr) and np.array_equal(W.indices, g.W.indices)
    assert O.max_rel(W.data, g.W.data) < 1e-6 and O.max_rel(V.data, g.V.data) < 1e-6
    assert O.max_rel(mod_V.data, g.modV.data) < 1e-6
    assert np.array_equal(np.asarray(Cm.argmax(axis=0)).ravel(), g.kappa)
    assert np.array_equal(knn_ind, g.knn_ind)
    W50, V50, mv, cc, ki = pkg.knn_sym_dist(X, 30, 1.0)  # a different k (utils.py:651 uses 50 at eval; kernel max is 33)
    assert isinstance(mv, int) and mv == 0 and isinstance(cc, int) and cc == 0 and ki.shape == (800, 30)  # GLL.py:229-230
    g30 = O.build_graph(X, 30, 1.0)
    assert np.array_equal(W50.indices, g30.W.indices) and O.max_rel(W50.data, g30.W.data) < 1e-6


def test_stable_conjgrad_wrapper(gll, capsys):
    pkg, _ = gll
    X, Y, *_ = O.synth_inputs(3, 150, 1450, 16, 6, 1.0)
    f = O.forward(X, Y, 0.05, 1.0, solver="lu")
    # the live call site (utils.py:586-591): Jacobi-scaled system, default tol = 1e-10
    Mh = sp.diags(1.0 / np.sqrt(f.Luu.diagonal() + 1e-10))
    A = (Mh @ f.Luu @ Mh).tocsr()
    b = Mh @ f.B
    y = pkg.stable_conjgrad(A, b)
    assert np.sqrt(((A @ y - b) ** 2).sum(axis=0)).max() <= 1e-10
    assert O.max_rel(Mh @ y, f.pred) < 1e-8
    y1 = pkg.stable_conjgrad(A, b[:, 0], tol=1e-8)  # 1-D right-hand side
    assert y1.shape == (1450,) and np.abs(A @ y1 - b[:, 0]).max() < 1e-8
    pkg.stable_conjgrad(A, b, max_iter=2, tol=1e-12)
    assert "max iter reached" in capsys.readouterr().out


# ----------------------------------------------------------------------------------------------------------------
# one graph over several ranks (sharded.py), executed as virtual ranks on this single GPU
# ----------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("world", [2, 3])
@pytest.mark.parametrize("eps,tau", [("auto", 0.0), (1.0, 0.07)])
def test_sharded_layer_matches_single_gpu_layer(gll, world, eps, tau):
    pkg, _ = gll
    from graphlearninglayer_b200.sharded import ShardedLaplaceLearning, last_info

    X, Y, _, yq = O.synth_inputs(31, 700, 2300, 96, 13, 2.5)  # l = 13: uneven column blocks; n = 3000: ragged row blocks
    ref_pred, ref_loss, ref_dX = layer_fwd_bwd(pkg, X, Y, yq, tau, eps)
    Xt = torch.as_tensor(X).cuda().requires_grad_(True)
    pred = ShardedLaplaceLearning.apply(Xt, torch.as_tensor(Y).cuda(), tau, eps, None, world)
    tgt = torch.nn.functional.one_hot(torch.as_tensor(yq).cuda(), pred.shape[1]).to(pred.dtype)
    loss = -torch.sum(tgt * torch.log(pred + 1e-8)) / pred.shape[0]
    loss.backward()
    torch.cuda.synchronize()
    assert pred.dtype == torch.float64 and Xt.grad.dtype == torch.float32
    # column blocks are solved independently of each other (GLL.py:262-269): same answer as the unsharded solve
    assert O.max_rel(pred.detach().cpu().numpy(), ref_pred.cpu().numpy()) < 2e-6
    assert O.max_rel(Xt.grad.cpu().numpy(), ref_dX.cpu().numpy()) < 2e-6
    info = last_info()
    assert info["status"] & ~8 == 0 and info["cg_iters_fwd"] > 0 and info["cg_iters_bwd"] > 0


def test_sharded_layer_vs_oracle(gll):
    pkg, _ = gll
    from graphlearninglayer_b200.sharded import ShardedLaplaceLearning

    X, Y, _, yq = O.synth_inputs(21, 1024, 5120, 256, 10, 3.0)
    f, loss_ref, gout, bw = O.fwd_bwd(X, Y, yq, 0.0, "auto", solver="cg")
    Xt = torch.as_tensor(X).cuda().requires_grad_(True)
    pred = ShardedLaplaceLearning.apply(Xt, torch.as_tensor(Y).cuda(), 0.0, "auto", None, 4)
    tgt = torch.nn.functional.one_hot(torch.as_tensor(yq).cuda(), pred.shape[1]).to(pred.dtype)
    (-torch.sum(tgt * torch.log(pred + 1e-8)) / pred.shape[0]).backward()
    assert O.max_rel(pred.detach().cpu().numpy(), f.pred) < TOL
    assert O.max_rel(Xt.grad.cpu().numpy(), bw.dX) < TOL


def _stagewise_fp64_check(X, Y, yq, g, pred, dX, n_sample=16, seed=0):
    """Full-size checker for graphs the oracle cannot rebuild in seconds (n >= 131072): every stage of the path is
    re-evaluated in fp64 on the host FROM THE PREVIOUS STAGE'S DEVICE OUTPUT, on all rows where that is cheap and on a
    sample of rows where it is not.  Returns a dict of error measures.
      kNN        sampled rows: fp64 brute force over all n points (O.exact_knn_rows), set equality          GLL.py:181-189
      eps, W     sampled rows and their neighbours: eps = 25th distance, W = exp(-4 d^2 / eps_i eps_j)      GLL.py:205,216
      forward    ||L_uu pred - B||_2 / ||B||_2 per class column, L from the device's W in fp64              GLL.py:29-53
      adjoint    the same for the adjoint solve                                                             GLL.py:93
      dX         sampled rows: sum_j t_ij (x_i - x_j) from the device's U, w, W, eps, kappa in fp64         GLL.py:104-159
    """
    n, d = X.shape
    k_lab, l = Y.shape
    out = {}
    rng = np.random.default_rng(seed)
    rows_s = np.sort(rng.choice(n, size=n_sample, replace=False))
    row_ptr = g.row_ptr.cpu().numpy().astype(np.int64)
    E = int(row_ptr[-1])
    col = g.col[:E].cpu().numpy().astype(np.int64)
    dist = g.dist[:E].cpu().numpy().astype(np.float64)
    w = g.w[:E].cpu().numpy().astype(np.float64)
    eps = g.eps.cpu().numpy().astype(np.float64)
    kappa = g.kappa.cpu().numpy().astype(np.int64)
    knn_idx = g.knn_idx[:n].cpu().numpy().astype(np.int64)
    # -- kNN on the sample and on the sample's neighbours (needed for eps_j)
    nb = np.unique(np.concatenate([col[row_ptr[i]:row_ptr[i + 1]] for i in rows_s] + [rows_s]))
    ref_idx, ref_dist = O.exact_knn_rows(X, nb, 25)
    pos = {int(r): t for t, r in enumerate(nb)}
    exact, tie, bad = O.knn_sets_match(knn_idx[nb], ref_idx, ref_dist)
    out["knn_bad_rows"], out["knn_rows_checked"] = bad, len(nb)
    eps_ref = ref_dist[:, -1]
    out["eps_err"] = float(np.max(np.abs(eps[nb] - eps_ref) / eps_ref))
    werr = 0.0
    for i in rows_s:
        e0, e1 = row_ptr[i], row_ptr[i + 1]
        j = col[e0:e1]
        dij = np.sqrt(((X[i].astype(np.float64) - X[j].astype(np.float64)) ** 2).sum(axis=1))
        wref = np.exp(-4.0 * dij * dij / eps_ref[pos[int(i)]] / np.array([eps_ref[pos[int(t)]] for t in j]))
        werr = max(werr, float(np.max(np.abs(w[e0:e1] - wref) / np.maximum(wref, 1e-30))))
    out["w_err"] = werr
    # -- both solves against the device's own weights, fp64
    W = sp.csr_matrix((w, col, row_ptr), shape=(n, n))
    Luu, B, _ = O.laplace_system(W, Y, 0.0)
    P = pred.cpu().numpy()
    out["fwd_residual"] = float(np.max(np.linalg.norm(Luu @ P - B, axis=0) / np.linalg.norm(B, axis=0)))
    _, gout = O.ce_loss_and_grad(P, yq)
    wt = g.wt[:, :l].double().cpu().numpy()
    ut = g.ut[:, :l].double().cpu().numpy()
    assert np.abs(ut[k_lab:] - P).max() <= 1e-6 * np.abs(P).max() and np.array_equal(ut[:k_lab], Y.astype(np.float64))
    gn = np.linalg.norm(gout, axis=0)
    out["adj_residual"] = float(np.max(np.linalg.norm(Luu @ wt[k_lab:] - gout, axis=0)[gn > 0] / gn.max()))
    # -- per-edge G, V, modV, b (all rows, chunked) and dX on the sample
    rows_all = np.repeat(np.arange(n), np.diff(row_ptr))
    V = -8.0 * w / eps[rows_all] / eps[col]
    Gv = np.empty(E)
    for s0 in range(0, E, 1 << 19):
        s1 = min(E, s0 + (1 << 19))
        r_, c_ = rows_all[s0:s1], col[s0:s1]
        Gv[s0:s1] = -np.einsum("ij,ij->i", wt[r_] - wt[c_], ut[r_] - ut[c_])
    b = np.bincount(rows_all, weights=Gv * (dist * dist * V / (eps[rows_all] ** 2) / 2.0), minlength=n)
    dXn = dX.cpu().numpy().astype(np.float64)
    scale = np.abs(dXn).max()
    derr = 0.0
    for i in rows_s:
        e0, e1 = row_ptr[i], row_ptr[i + 1]
        j = col[e0:e1]
        t = Gv[e0:e1] * V[e0:e1] - (j == kappa[i]) * b[i] - (kappa[j] == i) * b[j]
        ref = (t[:, None] * (X[i].astype(np.float64)[None, :] - X[j].astype(np.float64))).sum(axis=0)
        derr = max(derr, float(np.abs(dXn[i] - ref).max() / scale))
    out["dx_err"] = derr
    return out


@pytest.mark.parametrize("partition", ["columns", "rows"])
def test_sharded_c5s_size_stagewise(gll, partition):
    """BASELINE.json configs[4] at 1/8 of its size (n = 131072 nodes, 8192 labeled, d = 256, 100 classes, eps = 'auto') --
    the size ONE of eight ranks holds of the 1M-node graph -- sharded over virtual ranks, both CG partitions; the kNN
    search runs in its large-graph (aligned, whole row tiles per CTA) mode at d = 256."""
    pkg, _lib = gll
    from graphlearninglayer_b200 import sharded as sh

    X, Y, _, yq = O.synth_inputs(1000, 8192, 122880, 256, 100, 3.0)
    Xt = torch.as_tensor(X).cuda().requires_grad_(True)
    pred = sh.ShardedLaplaceLearning.apply(Xt, torch.as_tensor(Y).cuda(), 0.0, "auto", None, 2, partition)
    tgt = torch.nn.functional.one_hot(torch.as_tensor(yq).cuda(), pred.shape[1]).to(pred.dtype)
    (-torch.sum(tgt * torch.log(pred + 1e-8)) / pred.shape[0]).backward()
    torch.cuda.synchronize()
    info = sh.last_info()
    assert info["status"] & ~_lib.STATUS_KNN_FALLBACK == 0 and info["knn_fallback_rows"] <= 16, info
    p = pred.detach().cpu().numpy()
    assert np.abs(p.sum(axis=1) - 1.0).max() < 5e-5 and p.min() > -1e-5   # tau = 0: rows of the harmonic extension sum to 1
    r = _stagewise_fp64_check(X, Y, yq, sh._last_graph, pred.detach(), Xt.grad)
    assert r["knn_bad_rows"] == 0 and r["knn_rows_checked"] > 300, r
    assert r["eps_err"] < 1e-6 and r["w_err"] < 1e-5, r
    assert r["fwd_residual"] < 1e-5 and r["adj_residual"] < 1e-5, r
    assert r["dx_err"] < TOL, r


@pytest.mark.parametrize("world", [1, 2, 5])
@pytest.mark.parametrize("eps,tau", [("auto", 0.0), (1.0, 0.07)])
def test_sharded_layer_row_partitioned_cg(gll, world, eps, tau):
    """The north star's partition of the solve: rows of x, r, p, s split over the ranks, iterate all-gathered and dot
    products all-reduced every iteration (csrc/cg_rows.cu), here with virtual ranks on one GPU."""
    pkg, _ = gll
    from graphlearninglayer_b200.sharded import ShardedLaplaceLearning, last_info

    X, Y, _, yq = O.synth_inputs(33, 700, 2300, 96, 13, 2.5)  # m = 2300: ragged row blocks (last one short)
    f, loss_ref, gout, bw = O.fwd_bwd(X, Y, yq, tau, eps, solver="lu")
    Xt = torch.as_tensor(X).cuda().requires_grad_(True)
    pred = ShardedLaplaceLearning.apply(Xt, torch.as_tensor(Y).cuda(), tau, eps, None, world, "rows")
    tgt = torch.nn.functional.one_hot(torch.as_tensor(yq).cuda(), pred.shape[1]).to(pred.dtype)
    (-torch.sum(tgt * torch.log(pred + 1e-8)) / pred.shape[0]).backward()
    torch.cuda.synchronize()
    assert pred.dtype == torch.float64 and Xt.grad.dtype == torch.float32
    assert O.max_rel(pred.detach().cpu().numpy(), f.pred) < TOL
    assert O.max_rel(Xt.grad.cpu().numpy(), bw.dX) < TOL
    info = last_info()
    assert info["status"] & ~8 == 0 and 0 < info["cg_iters_fwd"] < 200 and 0 < info["cg_iters_bwd"] < 200


def test_cg_rows_stages_solve_to_tolerance(gll):
    """gll_cg_rows_* through the C ABI on a hand-built SPD system, 3 virtual ranks, 100 class columns; fp64 direct solve
    as the checker; zero right-hand-side columns are frozen from the start (GLL.py:262-263)."""
    import scipy.sparse as sparse
    import scipy.sparse.linalg as spla

    _, _lib = gll
    lib = _lib.lib
    rng = np.random.default_rng(3)
    m, l = 1500, 100
    A = sparse.random(m, m, density=0.01, random_state=7, format="csr")
    A = (A + A.T).tocsr()
    A.setdiag(0)
    A.eliminate_zeros()
    A.sort_indices()
    diag = np.asarray(A.sum(axis=1)).ravel() + 0.05 + rng.random(m)
    B = rng.standard_normal((m, l))
    B[:, 17] = 0.0
    lp = lib.gll_padded_classes(l)
    rhs = np.zeros((m, lp), np.float32)
    rhs[:, :l] = B
    ref = spla.spsolve((sparse.diags(diag) - A).tocsc(), rhs.astype(np.float64))
    ptr, col, val = dev_t(A.indptr, torch.int32), dev_t(A.indices, torch.int32), dev_t(A.data, torch.float32)
    dg, b = dev_t(diag, torch.float32), dev_t(rhs, torch.float32)
    world, per = 3, 512
    s = torch.cuda.current_stream().cuda_stream
    x = torch.zeros((world * per, lp), dtype=torch.float32, device="cuda")
    u = torch.zeros_like(x)
    st = []
    for r in range(world):
        lo, hi = min(m, r * per), min(m, (r + 1) * per)
        wsb = lib.gll_cg_rows_workspace_bytes(hi - lo, l)
        st.append((lo, hi, torch.empty(wsb, dtype=torch.uint8, device="cuda"), wsb, torch.zeros(3 * lp, dtype=torch.float64, device="cuda"),
                   torch.zeros(4, dtype=torch.int32, device="cuda")))
        _lib.check(lib.gll_cg_rows_init(dg.data_ptr(), b.data_ptr(), m, l, lo, hi, x.data_ptr(), u.data_ptr(), st[r][2].data_ptr(),
                                        wsb, s), "init")
    for it in range(400):
        for lo, hi, ws, wsb, sums, ctrl in st:
            _lib.check(lib.gll_cg_rows_spmv(ptr.data_ptr(), col.data_ptr(), val.data_ptr(), dg.data_ptr(), m, l, lo, hi, u.data_ptr(),
                                            sums.data_ptr(), ws.data_ptr(), wsb, s), "spmv")
        tot = st[0][4] + st[1][4] + st[2][4]
        for lo, hi, ws, wsb, sums, ctrl in st:
            sums.copy_(tot)
            _lib.check(lib.gll_cg_rows_update(dg.data_ptr(), m, l, lo, hi, sums.data_ptr(), it, 400, 1e-6, x.data_ptr(), u.data_ptr(),
                                              ctrl.data_ptr(), 0, ws.data_ptr(), wsb, s), "update")
        if st[0][5][0].item():
            break
    ctrls = torch.stack([c for *_, c in st]).cpu().numpy()
    assert (ctrls[:, 0] == 1).all() and (ctrls[:, 1] == ctrls[0, 1]).all() and (ctrls[:, 2] == 0).all() and 0 < ctrls[0, 1] < 400
    got = x[:m].cpu().numpy().astype(np.float64)
    assert np.all(got[:, 17] == 0.0)
    assert O.max_rel(got, ref) < 1e-5
    resid = (sparse.diags(diag) - A) @ got - rhs
    assert np.sqrt((resid ** 2).sum(axis=0)).max() < 1e-6 * np.sqrt((rhs.astype(np.float64) ** 2).sum(axis=0)).max()  # fp32 floor


def test_knn_row_blocks_equal_full_search(gll):
    _, _lib = gll
    X, *_ = O.synth_inputs(12, 3000, 1777, 200, 10, 3.5)
    n, d = X.shape
    full_i, full_d, _ = run_knn(_lib, X)
    Xc = dev_t(X, torch.float32)
    idx = torch.full((n, 25), -1, dtype=torch.int32, device="cuda")
    dd = torch.zeros((n, 25), dtype=torch.float32, device="cuda")
    info = torch.zeros(_lib.INFO_WORDS, dtype=torch.int32, device="cuda")
    for lo, hi in [(0, 1664), (1664, 3328), (3328, n)]:  # blocks start on multiples of 128
        wsb = _lib.lib.gll_knn_rows_workspace_bytes(n, d, 25, lo, hi)
        ws = torch.empty(wsb, dtype=torch.uint8, device="cuda")
        _lib.check(_lib.lib.gll_knn_rows(Xc.data_ptr(), n, d, 25, lo, hi, idx.data_ptr(), dd.data_ptr(), info.data_ptr(),
                                         ws.data_ptr(), wsb, torch.cuda.current_stream().cuda_stream), "gll_knn_rows")
    torch.cuda.synchronize()
    assert torch.equal(idx, full_i) and torch.equal(dd, full_d)


# ----------------------------------------------------------------------------------------------------------------
# evaluation path (SURVEY 8f-1): utils.laplace uses k = 50 neighbours and the Jacobi-scaled stable_conjgrad
# ----------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [34, 50, 64])
def test_knn_large_k_two_round_search(gll, k):
    _, _lib = gll
    X, *_ = O.synth_inputs(17, 900, 2100, 128, 10, 3.0)
    ref_ind, ref_dist = O.exact_knn(X, k)
    idx, dist, info = run_knn(_lib, X, k)
    ind = idx.cpu().numpy().astype(np.int64)
    exact, tie, bad = O.knn_sets_match(ind, ref_ind, ref_dist)
    assert bad == 0, (exact, tie, bad)
    same = np.all(ind == ref_ind, axis=1)
    assert same.mean() > 0.999
    assert np.array_equal(dist.cpu().numpy()[same], ref_dist[same].astype(np.float32))


def test_knn_large_k_with_duplicates(gll):
    _, _lib = gll
    rng = np.random.default_rng(5)
    X = rng.standard_normal((400, 24)).astype(np.float32)
    X[50:120] = X[50]  # 70 identical points: more zero-distance ties than one round of 32 can hold
    ref_ind, ref_dist = O.exact_knn(X, 50, slack=40)
    idx, dist, _ = run_knn(_lib, X, 50)
    assert np.array_equal(np.sort(dist.cpu().numpy(), axis=1), np.sort(ref_dist.astype(np.float32), axis=1))
    assert np.array_equal(idx.cpu().numpy()[50:120, :50], ref_ind[50:120])  # ties resolved by index in both


@pytest.mark.parametrize("k", [25, 50])
def test_knn_lattice_points_massive_ties(gll, monkeypatch, k):
    """Features on a small integer lattice: squared distances take a handful of values, so nearly every candidate decision is a
    value tie (within one row's set, between the sets of a row, between the two rounds of a k > 33 search).  The lists must be
    the oracle's -- ties by index -- whatever the packed, truncated keys of the tensor-core epilogue do with equal values."""
    _, _lib = gll
    monkeypatch.setenv("GLL_B200_KNN_PATH", "tc")
    rng = np.random.default_rng(11)
    X = rng.integers(0, 3, size=(3000, 10)).astype(np.float32)
    ref_ind, ref_dist = O.exact_knn(X, k, slack=600)
    idx, dist, info = run_knn(_lib, X, k)
    assert np.array_equal(dist.cpu().numpy(), ref_dist.astype(np.float32))
    assert np.array_equal(idx.cpu().numpy(), ref_ind)


def test_eval_path_like_utils_laplace(gll):
    """The reference's evaluation routine (utils.py:570-593) run on our drop-in wrappers: k = 50 graph, Jacobi-scaled
    system, stable_conjgrad to 1e-10, argmax accuracy -- against the same steps on the fp64 oracle."""
    import scipy.sparse as sparse

    pkg, _ = gll
    X, Y, y_base, yq = O.synth_inputs(23, 500, 2500, 64, 10, 2.0)
    k_lab, tau, eps = 500, 1e-8, "auto"

    def laplace(knn_sym_dist, stable_conjgrad):          # utils.py:570-593, condensed
        W = knn_sym_dist(X, 50, eps)[0]
        L = (sparse.diags(np.asarray(W.sum(axis=0)).ravel()) - W).tocsr()
        Luu = (L[k_lab:, k_lab:] + tau * sparse.identity(X.shape[0] - k_lab)).tocsr()
        Lul = L[k_lab:, :k_lab]
        M = sparse.diags(1.0 / np.sqrt(Luu.diagonal() + 1e-10))
        Pred = stable_conjgrad(M @ Luu @ M, -(M @ (Lul @ Y.astype(np.float64))))
        return M @ Pred

    def oracle_knn_sym_dist(data, k, epsilon):
        g = O.build_graph(data, k, epsilon)
        return g.W, g.V, g.modV, None, g.knn_ind

    def oracle_cg(A, b):
        return O.textbook_cg(sparse.csr_matrix(A), b, tol=1e-12)[0]

    ours = laplace(pkg.knn_sym_dist, pkg.stable_conjgrad)
    ref = laplace(oracle_knn_sym_dist, oracle_cg)
    assert O.max_rel(ours, ref) < 1e-6
    assert np.array_equal(ours.argmax(axis=1), ref.argmax(axis=1))


def test_host_pipeline_matches_plain_calls(gll):
    """HostPipeline (H2D / kernels / D2H of neighbouring calls overlapped on three streams) returns, for every call, exactly
    what the plain layer call returns on the same inputs -- several different graphs in flight, slots reused."""
    pkg, _ = gll
    from graphlearninglayer_b200.hostpipe import HostPipeline

    k_lab, m, d, l = 300, 200, 64, 7
    batches = []
    for seed in range(5):
        X, Y, _, yq = O.synth_inputs(40 + seed, k_lab, m, d, l, 2.0)
        batches.append((torch.as_tensor(X).pin_memory(), torch.as_tensor(Y).pin_memory(), yq))
    tgts = [torch.nn.functional.one_hot(torch.as_tensor(yq), l).to(torch.float64).cuda() for *_, yq in batches]
    order = []
    pipe = HostPipeline(k_lab + m, d, k_lab, l, "cuda", tau=0.0, epsilon="auto",
                        loss_fn=lambda pred, slot: -torch.sum(tgts[order[-1]] * torch.log(pred + 1e-8)) / m)
    got = []
    for i, (Xh, Yh, _) in enumerate(batches):
        if pipe.outstanding == pipe.depth:
            p, g = pipe.collect()
            got.append((p.clone(), g.clone()))
        order.append(i)
        pipe.submit(Xh, Yh)
    got += [(p.clone(), g.clone()) for p, g in pipe.drain()]
    assert len(got) == len(batches)
    for i, (Xh, Yh, yq) in enumerate(batches):
        ref_pred, _, ref_dX = layer_fwd_bwd(pkg, Xh.numpy(), Yh.numpy(), yq, 0.0, "auto")
        assert torch.equal(got[i][0], ref_pred.cpu()) and torch.equal(got[i][1], ref_dX.cpu())


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
def test_fused_ce_loss_matches_reference_formula(gll, dtype):
    """graphlearninglayer_b200.losses.custom_ce_loss vs the reference function body (losses.py:128-136), value and gradient."""
    from graphlearninglayer_b200.losses import custom_ce_loss

    g = torch.Generator().manual_seed(3)
    m, l = 777, 10
    p = torch.softmax(torch.randn(m, l, generator=g, dtype=torch.float64), dim=1).to(dtype).cuda()
    p[5] = 0.0                                   # exact zeros are what the 1e-8 is for
    t = torch.randint(0, l, (m,), generator=g).cuda()
    a = p.clone().requires_grad_(True)
    one_hot = torch.nn.functional.one_hot(t, num_classes=l).to(a.dtype)
    ref = -torch.sum(one_hot * torch.log(a + 1e-8)) / m
    (3.0 * ref).backward()
    b = p.clone().requires_grad_(True)
    ours = custom_ce_loss(b, t)
    (3.0 * ours).backward()
    tol = 1e-12 if dtype == torch.float64 else 2e-6
    assert ours.dtype == dtype and ours.shape == ref.shape
    assert abs(ours.item() - ref.item()) <= tol * abs(ref.item())
    assert torch.allclose(b.grad, a.grad, rtol=tol, atol=0.0)


@pytest.mark.parametrize("upstream", [1.0, 0.37])
def test_layer_with_loss_head_equals_two_calls(gll, upstream):
    """LaplaceLearningCELoss (layer + custom_ce_loss in one autograd node; the adjoint solve reads d loss / d pred and the upstream
    scalar itself) against the two separate calls: the same loss bits, the same prediction bits, dX within fp32 rounding of the
    one extra multiplication."""
    pkg, _ = gll
    from graphlearninglayer_b200.losses import custom_ce_loss, laplace_ce_loss
    X, Y, _, yq = O.synth_inputs(21, 600, 300, 48, 7, 3.0)
    Yt, tq = torch.as_tensor(Y).cuda(), torch.as_tensor(yq).cuda()
    Xa = torch.as_tensor(X).cuda().requires_grad_(True)
    pred_a = pkg.LaplaceLearningSparseHard.apply(Xa, Yt, 0.01, "auto")
    loss_a = custom_ce_loss(pred_a, tq)
    (loss_a * upstream).backward()
    Xb = torch.as_tensor(X).cuda().requires_grad_(True)
    loss_b, pred_b = laplace_ce_loss(Xb, Yt, tq, 0.01, "auto")
    (loss_b * upstream).backward()
    assert torch.equal(pred_a.detach(), pred_b) and torch.equal(loss_a.detach(), loss_b.detach())
    assert not pred_b.requires_grad
    assert O.max_rel(Xb.grad.cpu().numpy(), Xa.grad.cpu().numpy()) < 2e-6


def test_fused_ce_loss_many_rows(gll):
    """More than 4096 rows: several CTAs, partial sums added by a second tiny launch (sharded 1M-node graph path)."""
    from graphlearninglayer_b200.losses import custom_ce_loss

    g = torch.Generator().manual_seed(4)
    m, l = 50001, 100
    p = torch.softmax(torch.randn(m, l, generator=g, dtype=torch.float64), dim=1).cuda()
    t = torch.randint(0, l, (m,), generator=g).cuda()
    a = p.clone().requires_grad_(True)
    ref = -torch.sum(torch.nn.functional.one_hot(t, num_classes=l).to(a.dtype) * torch.log(a + 1e-8)) / m
    ref.backward()
    b = p.clone().requires_grad_(True)
    ours = custom_ce_loss(b, t)
    ours.backward()
    assert abs(ours.item() - ref.item()) <= 1e-12 * abs(ref.item())
    assert torch.allclose(b.grad, a.grad, rtol=1e-12, atol=0.0)


def test_knn_large_graph_mode_against_brute_force(gll):
    """n = 80000: the tensor-core kernel runs in its large-graph mode (whole row tiles per CTA, all CTAs sweeping the column tiles).
    512 random rows are checked against a float64 brute-force search (the CPU oracle would take minutes at this size)."""
    _, _lib = gll
    g = torch.Generator().manual_seed(11)
    n, d, k = 80000, 32, 25
    X = torch.nn.functional.normalize(torch.randn(n, d, generator=g), dim=1).numpy()
    idx, dist, info = run_knn(_lib, X, k)
    assert int(info[_lib.INFO_KNN_FALLBACK_ROWS]) < n // 100
    Xd = torch.as_tensor(X).cuda().double()
    rows = torch.randperm(n, generator=g)[:512].cuda()
    D = torch.cdist(Xd[rows], Xd)                       # 512 x n, float64
    D[torch.arange(512, device="cuda"), rows] = -1.0    # self first
    ref_d, ref_i = torch.topk(D, k, dim=1, largest=False)
    got_i = idx[rows].long()
    same = (got_i == ref_i).all(dim=1)
    # float64 cdist and the kernel's exact distances can order two neighbours at ~1e-16 relative distance differently
    assert same.float().mean().item() > 0.99
    assert torch.equal(torch.sort(got_i, dim=1).values[same], torch.sort(ref_i, dim=1).values[same])
    assert torch.allclose(dist[rows][:, 1:].double(), ref_d[:, 1:], rtol=1e-6, atol=0.0)


def test_normalized_variant_matches_torch_normalize_plus_layer(gll):
    """LaplaceLearningSparseHardNormalized(feat) == LaplaceLearningSparseHard(F.normalize(feat, dim=1)) with PyTorch's own
    autograd through the normalisation (networks/BuildNet.py:101), value and gradient with respect to the raw features."""
    pkg, _ = gll
    X, Y, _, yq = O.synth_inputs(51, 400, 600, 64, 10, 2.0)
    g = torch.Generator().manual_seed(2)
    raw = (torch.as_tensor(X) * (0.5 + 3.0 * torch.rand(X.shape[0], 1, generator=g))).cuda()   # rows of different lengths
    Yt = torch.as_tensor(Y).cuda()
    tgt = torch.nn.functional.one_hot(torch.as_tensor(yq).cuda(), 10).double()
    a = raw.clone().requires_grad_(True)
    pa = pkg.LaplaceLearningSparseHard.apply(torch.nn.functional.normalize(a, dim=1), Yt, 0.0, "auto")
    (-torch.sum(tgt * torch.log(pa + 1e-8)) / 600).backward()
    b = raw.clone().requires_grad_(True)
    pb = pkg.LaplaceLearningSparseHardNormalized.apply(b, Yt, 0.0, "auto")
    (-torch.sum(tgt * torch.log(pb + 1e-8)) / 600).backward()
    assert O.max_rel(pb.detach().cpu().numpy(), pa.detach().cpu().numpy()) < 2e-6
    assert O.max_rel(b.grad.cpu().numpy(), a.grad.cpu().numpy()) < 1e-5


def test_eval_path_matches_reference_fixture(gll):
    """utils.laplace (utils.py:570-593) as the reference runs it -- UNMODIFIED knn_sym_dist (k = 50) and stable_conjgrad of
    GLL.py, fixture tests/golden/eval_k50.npz -- against the same steps on our drop-in wrappers."""
    import hashlib
    import os

    import scipy.sparse as sparse

    pkg, _ = gll
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "eval_k50.npz"))
    seed, k_lab, m, d, l, knn = (int(v) for v in g["params"])
    X, Y, _, yq = O.synth_inputs(seed, k_lab, m, d, l, float(g["sigma"]))
    assert hashlib.sha256(X.tobytes()).hexdigest() == str(g["x_sha256"])
    W_ref = sparse.csr_matrix((g["w_data"], g["w_indices"], g["w_indptr"]), shape=(k_lab + m, k_lab + m))
    W = sparse.csr_matrix(pkg.knn_sym_dist(X, knn, "auto")[0])
    W.sort_indices()
    assert np.array_equal(W.indptr, W_ref.indptr) and np.array_equal(W.indices, W_ref.indices)   # same graph
    assert np.max(np.abs(W.data - W_ref.data)) < 2e-6                                            # fp32 weights
    L = (sparse.diags(np.asarray(W.sum(axis=0)).ravel()) - W).tocsr()
    Luu = (L[k_lab:, k_lab:] + float(g["tau"]) * sparse.identity(m)).tocsr()
    M = sparse.diags(1.0 / np.sqrt(Luu.diagonal() + 1e-10))
    Pred = M @ pkg.stable_conjgrad(M @ Luu @ M, -(M @ (L[k_lab:, :k_lab] @ Y.astype(np.float64))))
    assert O.max_rel(Pred, g["pred"]) < 1e-5
    assert np.array_equal(Pred.argmax(axis=1), g["pred"].argmax(axis=1))
