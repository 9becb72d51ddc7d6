"""CPU checks of the drop-in boundary: the shared library loads, exports every symbol include/gll_b200.h declares,
and its host-only queries work without a GPU (no compute calls here)."""
import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def libmod():
    from graphlearninglayer_b200 import build

    build.build()
    from graphlearninglayer_b200 import _lib

    return _lib


def declared_symbols():
    text = open(os.path.join(ROOT, "include", "gll_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(gll_[a-z0-9_]+)\s*\(", text)))


def test_every_declared_symbol_is_exported(libmod):
    names = declared_symbols()
    assert len(names) >= 20
    raw = ctypes.CDLL(libmod.LIB_PATH)
    for nm in names:
        assert hasattr(raw, nm), f"{nm} declared in include/gll_b200.h but not exported"
    assert sorted(libmod.EXPORTS) == names  # the ctypes binding covers the whole header


def test_host_queries(libmod):
    lib = libmod.lib
    assert lib.gll_version() >= 100
    assert lib.gll_padded_classes(10) == 12 and lib.gll_padded_classes(100) == 100 and lib.gll_padded_classes(1) == 4
    assert lib.gll_max_edges(1000, 25) == 2 * 1000 * 24
    L = libmod.state_layout(2000, 25, 10, 1000)
    offs = [getattr(L, n) for n in libmod.Layout._names]
    assert all(o % 256 == 0 for o in offs) and offs == sorted(offs) and L.total >= offs[-2]
    assert lib.gll_workspace_bytes(2000, 128, 25, 10, 1000) >= lib.gll_knn_workspace_bytes(2000, 128, 25)
    assert lib.gll_kernel_count() == len(libmod.kernel_names()) and "cg_persistent" in libmod.kernel_names()
    with pytest.raises(libmod.GllError):
        libmod.state_layout(10, 25, 3, 10)  # k_lab must be < n
    assert b"k_lab" in lib.gll_last_error()


def test_layer_refuses_cpu_tensors(libmod):
    import torch

    import graphlearninglayer_b200 as pkg

    X = torch.randn(64, 8)
    Y = torch.eye(4)[torch.arange(16) % 4]
    with pytest.raises(RuntimeError, match="no CPU path"):
        pkg.LaplaceLearningSparseHard.apply(X, Y)


def test_dropin_module_exports_reference_names(libmod):
    """utils.py:25 does `from GLL import LaplaceLearningSparseHard, knn_sym_dist, stable_conjgrad`."""
    import importlib.util

    spec = importlib.util.spec_from_file_location("GLL", os.path.join(ROOT, "graphlearninglayer_b200", "dropin", "GLL.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    for nm in ("LaplaceLearningSparseHard", "knn_sym_dist", "stable_conjgrad"):
        assert hasattr(mod, nm)
    import inspect

    sig = inspect.signature(mod.LaplaceLearningSparseHard.forward)
    assert list(sig.parameters) == ["ctx", "X", "label_matrix", "tau", "epsilon"]  # GLL.py:14
    assert sig.parameters["tau"].default == 0 and sig.parameters["epsilon"].default == "auto"
    assert list(inspect.signature(mod.stable_conjgrad).parameters) == ["A", "b", "x0", "max_iter", "tol"]  # GLL.py:247
    assert list(inspect.signature(mod.knn_sym_dist).parameters) == ["data", "k", "epsilon"]  # GLL.py:180


def test_side_modules_refuse_cpu_tensors_and_mirror_reference_signatures(libmod):
    """No CPU path anywhere: the fused loss, the normalised variant and the host pipeline all raise on CPU inputs; the loss
    keeps the reference signature custom_ce_loss(softmax_logits, targets) (losses.py:128)."""
    import inspect

    import torch

    import graphlearninglayer_b200 as pkg
    from graphlearninglayer_b200 import hostpipe, losses

    assert list(inspect.signature(losses.custom_ce_loss).parameters) == ["softmax_logits", "targets"]
    with pytest.raises(RuntimeError, match="no CPU path"):
        losses.custom_ce_loss(torch.full((4, 3), 1 / 3), torch.zeros(4, dtype=torch.long))
    with pytest.raises(RuntimeError, match="no CPU path"):
        pkg.LaplaceLearningSparseHardNormalized.apply(torch.randn(64, 8), torch.eye(4)[torch.arange(16) % 4])
    with pytest.raises(RuntimeError, match="no CPU path"):
        hostpipe.HostPipeline(64, 8, 16, 4, "cpu", loss_fn=lambda p, s: p.sum())
    sig = inspect.signature(pkg.LaplaceLearningSparseHardNormalized.forward)
    assert list(sig.parameters) == ["ctx", "feat", "label_matrix", "tau", "epsilon"]


def test_peer_table_matches_the_header(libmod):
    """ctypes mirror of struct gll_peers: 3 x 8 pointers + world + rank, and the host-side size queries of the peer-memory CG."""
    P = libmod.Peers
    assert ctypes.sizeof(P) == 3 * 8 * ctypes.sizeof(ctypes.c_void_p) + 2 * ctypes.sizeof(ctypes.c_int)
    assert [f[0] for f in P._fields_] == ["u", "mail", "flags", "world", "rank"]
    lib = libmod.lib
    assert lib.gll_cg_rows_peer_flag_bytes() == 2 * 8 * 4           # [2 flag kinds][8 ranks] unsigned
    assert lib.gll_cg_rows_peer_mail_bytes() == 2 * 8 * 3 * 128 * 8  # [2 parities][8 ranks][3 dots x 128 columns] doubles
    assert lib.gll_ce_loss_workspace_bytes(512) == 0 and lib.gll_ce_loss_workspace_bytes(100000) > 0
    assert lib.gll_cg_rows_workspace_bytes(1000, 10) > 4 * 1000 * 12 * 4


STREAMING, RESIDENT, SMALL, CLUSTER = 0, 1, 2, 3  # GLL_CG_KERNEL_*


@pytest.mark.parametrize("path,cases", [
    # (m, l, hint) -> kernel.  Unset or empty: cluster for 0 < hint <= 5 where it fits, else small where it fits, else resident
    # where it fits, else streaming.
    ("", [((63, 10, 1.4), SMALL), ((64, 10, 1.4), CLUSTER), ((2048, 10, 1.4), CLUSTER), ((2049, 10, 1.4), RESIDENT),
          ((300, 10, 0.0), SMALL), ((300, 10, 5.0), CLUSTER), ((300, 10, 5.01), SMALL),
          ((2048, 20, 1.4), CLUSTER), ((2048, 21, 1.4), RESIDENT),
          ((512, 10, 0.0), SMALL), ((513, 10, 0.0), RESIDENT), ((512, 16, 0.0), SMALL), ((512, 17, 0.0), RESIDENT),
          ((700, 40, 0.0), RESIDENT), ((3000, 10, 0.0), RESIDENT), ((1_000_000, 10, 0.0), STREAMING)]),
    ("small", [((300, 10, 1.4), SMALL), ((512, 16, 1.4), SMALL), ((700, 10, 1.4), RESIDENT), ((1_000_000, 10, 0.0), STREAMING)]),
    ("cluster", [((300, 10, 0.0), CLUSTER), ((63, 10, 0.0), SMALL), ((700, 40, 0.0), CLUSTER), ((700, 100, 0.0), RESIDENT),
                 ((2049, 10, 0.0), RESIDENT), ((1_000_000, 10, 0.0), STREAMING)]),
    ("resident", [((300, 10, 1.4), RESIDENT), ((64, 1, 0.0), RESIDENT), ((1_000_000, 10, 0.0), STREAMING)]),
    ("streaming", [((300, 10, 1.4), STREAMING), ((3000, 10, 0.0), STREAMING)]),
    ("other", [((300, 10, 1.4), RESIDENT), ((1_000_000, 10, 0.0), STREAMING)]),
])
def test_cg_kernel_table(libmod, monkeypatch, path, cases):
    """gll_cg_kernel: which CG kernel a solve of m rows and l classes takes, under GLL_B200_CG_PATH, at the edges of each kernel.
    lp = 4 ceil(l / 4) padded columns, Q = lp / 4 class quads.  The expected values follow from the size rules of the kernels:
      cluster  64 <= m <= 2048; R = 32 ceil(ceil(m / 8) / 32) rows per CTA; Q R items over 320 threads, at most 4 per thread;
               shared memory within 208 KB.  (2048, 20): R = 256, Q = 5, 1280 items = 4 per thread; (2048, 21): Q = 6, 5 per
               thread.  (700, 40): R = 96, Q = 10, 3 per thread and 118 KB: it fits; (700, 100): Q = 25, 8 per thread.
      small    m <= 512; rows padded to a power of two P >= 32; Q P items over 512 threads, at most 4 per thread; shared memory
               within 160 KB.  (512, 16): Q = 4, 4 per thread and 134 KB; (512, 17): Q = 5, 5 per thread.
      resident fits unless a CTA's rows (m over up to 148 SMs) overflow 200 KB of shared memory: 10^6 rows do.
    "small" / "cluster" put that kernel first and ignore the hint; any other non-empty value skips both minibatch kernels."""
    monkeypatch.setenv("GLL_B200_CG_PATH", path)
    lib = libmod.lib
    got = [lib.gll_cg_kernel(m, l, h) for (m, l, h), _ in cases]
    assert got == [k for _, k in cases]
    assert lib.gll_cg_kernel(100, 0, 0.0) == -1 and lib.gll_cg_kernel(100, 129, 0.0) == -1 and lib.gll_cg_kernel(0, 10, 0.0) == -1
