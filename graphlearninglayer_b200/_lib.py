"""ctypes binding of libgll_b200.so (C ABI declared in include/gll_b200.h).

The library is the product: there is NO CPU fallback.  If the shared object is missing this module raises
at import time with the build command; nothing else in the package will work without it.
"""
from __future__ import annotations

import ctypes as C
import os

PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(PKG, "libgll_b200.so")

GLL_OK = 0
STATUS_CG_NOT_CONVERGED = 1
STATUS_EPS_TINY = 2
STATUS_NONFINITE = 4
STATUS_KNN_FALLBACK = 8
STATUS_BAD_INDEX = 16

INFO_STATUS, INFO_NNZ, INFO_NNZ_UU, INFO_CG_ITERS_FWD, INFO_CG_ITERS_BWD = 0, 1, 2, 3, 4
INFO_KNN_FALLBACK_ROWS, INFO_CG_RESID_FWD, INFO_CG_RESID_BWD = 5, 6, 7
INFO_LAPLACE_ROUNDS, INFO_LAPLACE_CG_ITERS, INFO_LAPLACE_RESID, INFO_LAPLACE_RESID0, INFO_LAPLACE_ROUND_ITERS = 8, 9, 10, 11, 14
INFO_CG_BARRIER = 12  # two words: the on-chip CG's grid barrier
INFO_WORDS = 16


class GllError(RuntimeError):
    pass


class Peers(C.Structure):
    """gll_peers (include/gll_b200.h): every rank's u array, mailbox and flag block as mapped in this process."""
    _fields_ = [("u", C.c_void_p * 8), ("mail", C.c_void_p * 8), ("flags", C.c_void_p * 8), ("world", C.c_int), ("rank", C.c_int)]


class Layout(C.Structure):
    """Mirror of ``gll_layout`` (include/gll_b200.h): byte offsets into the state buffer."""
    _names = ["knn_idx", "knn_dist", "row_ptr", "col", "dist", "w", "gv", "eps", "kappa", "deg", "bvec", "uu_ptr",
              "uu_col", "uu_val", "diag", "rhs", "ut", "wt", "info", "total"]
    _fields_ = [(n, C.c_size_t) for n in _names]


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -m graphlearninglayer_b200.build` "
            "(nvcc, sm_100a).  graphlearninglayer_b200 has no CPU or PyTorch fallback.")
    lib = C.CDLL(LIB_PATH)
    vp, sz, i32, f32 = C.c_void_p, C.c_size_t, C.c_int, C.c_float

    def sig(name, res, args):
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
        return fn

    sig("gll_last_error", C.c_char_p, [])
    sig("gll_version", i32, [])
    sig("gll_device_sm_count", i32, [])
    sig("gll_kernel_count", i32, [])
    sig("gll_kernel_name", C.c_char_p, [i32])
    sig("gll_launch_count", C.c_longlong, [i32])
    sig("gll_profile_enable", None, [i32])
    sig("gll_debug_cg_trace", None, [vp])
    sig("gll_debug_knn_trace", None, [vp])
    sig("gll_profile_collect", i32, [C.POINTER(C.c_double), C.POINTER(C.c_longlong)])
    sig("gll_padded_classes", i32, [i32])
    sig("gll_max_edges", sz, [i32, i32])
    sig("gll_state_layout", i32, [i32, i32, i32, i32, C.POINTER(Layout)])
    sig("gll_workspace_bytes", sz, [i32, i32, i32, i32, i32])
    sig("gll_knn_workspace_bytes", sz, [i32, i32, i32])
    sig("gll_graph_workspace_bytes", sz, [i32, i32])
    sig("gll_weights_workspace_bytes", sz, [i32, i32])
    sig("gll_cg_workspace_bytes", sz, [i32, i32])
    sig("gll_knn", i32, [vp, i32, i32, i32, vp, vp, vp, vp, sz, vp])
    sig("gll_graph_build", i32, [vp, vp, i32, i32, vp, vp, vp, vp, vp, sz, vp])
    sig("gll_edge_weights", i32, [vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, f32, f32,
                                  vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, sz, vp])
    sig("gll_cg_solve", i32, [vp, vp, vp, vp, vp, i32, i32, f32, i32, vp, vp, vp, vp, vp, sz, vp])
    sig("gll_cg_solve_hint", i32, [vp, vp, vp, vp, vp, i32, i32, f32, i32, vp, vp, vp, vp, vp, sz, vp, f32])
    sig("gll_cg_kernel", i32, [i32, i32, f32])
    sig("gll_backward_edges", i32, [vp, i32, i32, i32, i32, i32, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp])
    sig("gll_debug_gram_tile", i32, [vp, i32, i32, i32, i32, vp, vp, vp, sz, vp])
    sig("gll_base_cache_bytes", sz, [i32])
    sig("gll_base_cache_workspace_bytes", sz, [i32, i32])
    sig("gll_base_cache_build", i32, [vp, i32, i32, vp, vp, sz, vp])
    sig("gll_knn_cached_workspace_bytes", sz, [i32, i32, i32, i32])
    sig("gll_knn_cached", i32, [vp, i32, i32, i32, i32, vp, vp, vp, vp, vp, sz, vp])
    sig("gll_knn_rows_workspace_bytes", sz, [i32, i32, i32, i32, i32])
    sig("gll_knn_rows", i32, [vp, i32, i32, i32, i32, i32, vp, vp, vp, vp, sz, vp])
    sig("gll_backward_edges_rows", i32, [vp, i32, i32, i32, i32, i32, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, vp])
    sig("gll_cg_rows_workspace_bytes", sz, [i32, i32])
    sig("gll_cg_rows_init", i32, [vp, vp, i32, i32, i32, i32, vp, vp, vp, sz, vp])
    sig("gll_cg_rows_spmv", i32, [vp, vp, vp, vp, i32, i32, i32, i32, vp, vp, vp, sz, vp])
    sig("gll_cg_rows_update", i32, [vp, i32, i32, i32, i32, vp, i32, i32, f32, vp, vp, vp, vp, vp, sz, vp])
    sig("gll_cg_rows_peer_mail_bytes", sz, [])
    sig("gll_cg_rows_peer_flag_bytes", sz, [])
    u32, pp = C.c_uint, C.POINTER(Peers)
    sig("gll_cg_rows_init_p2p", i32, [vp, vp, i32, i32, i32, i32, vp, pp, u32, vp, sz, vp])
    sig("gll_cg_rows_spmv_p2p", i32, [vp, vp, vp, vp, i32, i32, i32, i32, pp, u32, vp, vp, sz, vp])
    sig("gll_cg_rows_update_p2p", i32, [vp, i32, i32, i32, i32, i32, i32, f32, vp, pp, u32, vp, vp, vp, sz, vp])
    sig("gll_normalize_rows", i32, [vp, i32, i32, f32, vp, vp, vp])
    sig("gll_normalize_rows_backward", i32, [vp, vp, vp, i32, i32, vp, vp])
    sig("gll_csr_residual_f64", i32, [vp, vp, vp, vp, vp, i32, i32, vp, vp])
    sig("gll_ce_loss_workspace_bytes", sz, [i32])
    sig("gll_ce_loss", i32, [vp, i32, vp, i32, i32, vp, vp, vp, vp, sz, vp])
    sig("gll_pack_columns", i32, [vp, i32, i32, i32, i32, vp, i32, vp])
    sig("gll_unpack_columns", i32, [vp, i32, i32, i32, i32, vp, i32, vp])
    sig("gll_unpack_pred", i32, [vp, i32, i32, vp, i32, vp])
    sig("gll_pack_grad", i32, [vp, i32, i32, i32, vp, vp])
    sig("gll_forward", i32, [vp, vp, i32, i32, i32, i32, i32, i32, f32, f32, f32, i32, vp, vp, i32, vp, sz, vp])
    sig("gll_backward", i32, [vp, vp, i32, i32, i32, i32, i32, i32, i32, f32, i32, vp, vp, vp, sz, vp])
    sig("gll_backward_scaled", i32, [vp, vp, i32, vp, i32, i32, i32, i32, i32, i32, i32, f32, i32, vp, vp, vp, sz, vp])
    ip, llp = C.POINTER(C.c_int), C.POINTER(C.c_longlong)
    sig("gll_knn_segments_workspace_bytes", sz, [i32, i32, i32, ip, i32])
    sig("gll_knn_segments", i32, [vp, i32, i32, i32, ip, i32, vp, vp, vp, vp, sz, vp])
    sig("gll_knn_segments_units", None, [i32, i32, ip, i32, llp, llp])
    sig("gll_batched_workspace_bytes", sz, [i32, i32, i32, i32, i32, i32])
    sig("gll_forward_batched", i32, [vp, vp, i32, i32, i32, i32, i32, i32, i32, f32, f32, f32, i32, vp, vp, i32, vp, sz, vp])
    sig("gll_laplace_eval_workspace_bytes", sz, [i32, i32, i32, i32, i32])
    sig("gll_laplace_eval", i32, [vp, vp, i32, i32, i32, i32, i32, i32, f32, f32, C.c_double, i32, vp, vp, vp, vp, vp, vp, sz, vp])
    sig("gll_laplace_eval_batched_workspace_bytes", sz, [i32, i32, i32, i32, i32, i32])
    sig("gll_laplace_eval_batched", i32, [vp, vp, i32, i32, i32, i32, i32, i32, i32, f32, f32, C.c_double, i32, vp, vp, vp, vp, vp,
                                          vp, vp, sz, vp])
    sig("gll_laplace_eval_trials_workspace_bytes", sz, [i32, i32, i32, i32, i32, i32])
    sig("gll_laplace_eval_trials", i32, [vp, i32, i32, i32, vp, i32, vp, i32, i32, i32, i32, f32, f32, C.c_double, i32, vp, vp, vp,
                                         vp, vp, vp, vp, sz, vp])
    return lib


lib = _load()

#: every symbol include/gll_b200.h declares (tests check the .so exports all of them)
EXPORTS = ["gll_last_error", "gll_version", "gll_device_sm_count", "gll_kernel_count", "gll_kernel_name",
           "gll_launch_count", "gll_profile_enable", "gll_profile_collect", "gll_debug_cg_trace", "gll_debug_knn_trace", "gll_padded_classes", "gll_max_edges",
           "gll_state_layout", "gll_workspace_bytes", "gll_knn_workspace_bytes", "gll_graph_workspace_bytes",
           "gll_weights_workspace_bytes", "gll_cg_workspace_bytes", "gll_knn", "gll_graph_build", "gll_edge_weights",
           "gll_cg_solve", "gll_cg_solve_hint", "gll_cg_kernel", "gll_backward_edges", "gll_forward", "gll_backward", "gll_backward_scaled", "gll_knn_rows_workspace_bytes", "gll_knn_rows",
           "gll_backward_edges_rows", "gll_pack_columns", "gll_unpack_columns", "gll_unpack_pred", "gll_pack_grad",
           "gll_cg_rows_workspace_bytes", "gll_cg_rows_init", "gll_cg_rows_spmv", "gll_cg_rows_update", "gll_ce_loss", "gll_ce_loss_workspace_bytes",
           "gll_cg_rows_peer_mail_bytes", "gll_cg_rows_peer_flag_bytes", "gll_cg_rows_init_p2p", "gll_cg_rows_spmv_p2p",
           "gll_cg_rows_update_p2p", "gll_csr_residual_f64", "gll_normalize_rows",
           "gll_normalize_rows_backward", "gll_debug_gram_tile", "gll_base_cache_bytes", "gll_base_cache_workspace_bytes",
           "gll_base_cache_build", "gll_knn_cached_workspace_bytes", "gll_knn_cached", "gll_laplace_eval_workspace_bytes",
           "gll_laplace_eval", "gll_knn_segments_workspace_bytes", "gll_knn_segments", "gll_knn_segments_units",
           "gll_batched_workspace_bytes", "gll_forward_batched", "gll_laplace_eval_batched_workspace_bytes", "gll_laplace_eval_batched",
           "gll_laplace_eval_trials_workspace_bytes", "gll_laplace_eval_trials"]


def check(rc: int, what: str) -> None:
    if rc != GLL_OK:
        msg = lib.gll_last_error().decode("utf-8", "replace")
        raise GllError(f"{what} failed (code {rc}): {msg}")


def state_layout(n: int, k: int, l: int, k_lab: int) -> Layout:
    L = Layout()
    check(lib.gll_state_layout(n, k, l, k_lab, C.byref(L)), "gll_state_layout")
    return L


def seg_ptr_array(seg_ptr) -> "C.Array":
    """Host int32 array of segment offsets for gll_knn_segments* (seg_ptr_host)."""
    v = [int(x) for x in seg_ptr]
    return (C.c_int * len(v))(*v)


def launch_count(kernel_id: int = -1) -> int:
    """Kernel launches issued by the library so far (all kernels when kernel_id < 0)."""
    return int(lib.gll_launch_count(kernel_id))


def kernel_names() -> list:
    return [lib.gll_kernel_name(i).decode() for i in range(lib.gll_kernel_count())]


def profile_collect() -> dict:
    """{kernel name: (summed ms, launches)} of the launches recorded since the last call (synchronises)."""
    nk = lib.gll_kernel_count()
    ms = (C.c_double * nk)()
    cnt = (C.c_longlong * nk)()
    check(lib.gll_profile_collect(ms, cnt), "gll_profile_collect")
    return {lib.gll_kernel_name(i).decode(): (float(ms[i]), int(cnt[i])) for i in range(nk) if cnt[i]}
