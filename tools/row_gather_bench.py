"""Phase 2 of the backward edge pass (K6 `row_gather_kernel`, csrc/backward.cu) on its own, at C2 size, for one or more builds
of the library side by side.  Run on the GPU box:

    python tools/row_gather_bench.py [--lib PATH ...] [--launches 200] [--runs 3] [--out FILE.json]

Graph, gv and b: one forward + backward of the layer on C2's inputs (synth_inputs(0, 10000, 512, 512, 10, 4.5): 10 512 rows,
k = 25, eps = 'auto').  Features: seeded N(0, I/d) rows of each width d.  Shapes: d = 19, 99, 130, 515, 2051 (float chunks), 512
with X and dX one float off 16-byte alignment (float chunks), 128, 512, 2048 (float4 chunks).

Every --lib (default: the package's library) runs gll_backward_edges_rows(..., phases=2) on the same device arrays.  A run
times `launches` back-to-back launches with CUDA events; the libraries alternate within each run, and the median of `runs`
runs is reported.  X is below the 126 MB L2 at every width, so the neighbour rows are read from L2, as in the layer's backward
right after the forward.  The dX of every library is compared byte for byte with the first one's.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from graphlearninglayer_b200 import GLL, _lib  # noqa: E402
from graphlearninglayer_b200.synth import synth_inputs  # noqa: E402

K_LAB, M, D_GRAPH, L, SIGMA = 10000, 512, 512, 10, 4.5
SHAPES = [(19, False), (99, False), (130, False), (515, False), (2051, False), (512, True), (128, False), (512, False), (2048, False)]


def gpu_identity():
    out = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30)
        out["power_limit_and_max_sm_clock"] = q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unavailable"
    except (OSError, subprocess.SubprocessError):
        out["power_limit_and_max_sm_clock"] = "unavailable"
    return out


def load(path):
    lib = C.CDLL(os.path.abspath(path))
    vp, i32 = C.c_void_p, C.c_int
    fn = lib.gll_backward_edges_rows
    fn.restype = i32
    fn.argtypes = [vp, i32, i32, i32, i32, i32, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, vp]
    lib.gll_last_error.restype = C.c_char_p
    return lib


def c2_graph():
    """The layer's state after one forward + backward on C2's inputs: CSR, eps, kappa, ut, wt, gv and b on the device."""
    X, Y, *_ = synth_inputs(0, K_LAB, M, D_GRAPH, L, SIGMA)
    pred, st, Xc = GLL._forward_impl(torch.as_tensor(X).cuda(), torch.as_tensor(Y).cuda(), 0.0, "auto")
    g = torch.as_tensor(np.random.default_rng(1).standard_normal((M, L))).cuda()
    GLL._backward_impl(st, Xc, g)
    torch.cuda.synchronize()
    return st


def gather_args(st, X, dX, d):
    n, lp = st.n, (st.l + 3) // 4 * 4
    E = int(st.view("row_ptr", torch.int32, n + 1)[-1].item())
    ptr = {name: st.view(name, dt, cnt).data_ptr() for name, dt, cnt in (
        ("row_ptr", torch.int32, n + 1), ("col", torch.int32, E), ("dist", torch.float32, E), ("w", torch.float32, E),
        ("eps", torch.float32, n), ("kappa", torch.int32, n), ("ut", torch.float32, n * lp), ("wt", torch.float32, n * lp),
        ("gv", torch.float32, E), ("bvec", torch.float32, n))}
    return (X.data_ptr(), n, d, st.l, st.k_lab, int(st.eps_auto), ptr["row_ptr"], ptr["col"], ptr["dist"], ptr["w"], ptr["eps"],
            ptr["kappa"], ptr["ut"], ptr["wt"], ptr["gv"], ptr["bvec"], dX.data_ptr(), 0, n, 2,
            torch.cuda.current_stream().cuda_stream), E


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib", action="append", default=None, help="library to time (repeatable; default: the package's)")
    ap.add_argument("--launches", type=int, default=200)
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("row_gather_bench.py needs a CUDA device")
    paths = a.lib or [_lib.LIB_PATH]
    libs = [load(p) for p in paths]
    st = c2_graph()
    out = dict(gpu=gpu_identity(), libs=paths, launches=a.launches, runs=a.runs,
               workload=f"C2 graph (synth_inputs(0, {K_LAB}, {M}, {D_GRAPH}, {L}, {SIGMA}), k=25, eps='auto'), phase 2 only",
               cases=[])
    for d, misaligned in SHAPES:
        n, off = st.n, int(misaligned)
        xbuf = torch.empty(n * d + off, dtype=torch.float32, device="cuda")
        xbuf[off:].copy_(torch.as_tensor(np.random.default_rng(d).standard_normal(n * d) / np.sqrt(d)).float())
        dbuf = torch.empty(n * d + off, dtype=torch.float32, device="cuda")
        X, dX = xbuf[off:], dbuf[off:]
        args, E = gather_args(st, X, dX, d)
        results, ref = [], None
        for lib in libs:  # warm-up, and each library's dX
            dbuf.fill_(float("nan"))
            rc = lib.gll_backward_edges_rows(*args)
            if rc != _lib.GLL_OK:
                raise RuntimeError(f"gll_backward_edges_rows failed: {lib.gll_last_error().decode()}")
            torch.cuda.synchronize()
            host = dX.cpu().numpy().tobytes()
            ref = host if ref is None else ref
            results.append(dict(identical_to_first=host == ref, us=[]))
        for _ in range(a.runs):
            for lib, r in zip(libs, results):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(a.launches):
                    lib.gll_backward_edges_rows(*args)
                e1.record()
                torch.cuda.synchronize()
                r["us"].append(e0.elapsed_time(e1) * 1e3 / a.launches)
        for r in results:
            r["median_us"] = float(np.median(r["us"]))
        out["cases"].append(dict(d=d, misaligned=misaligned, n=n, edges=E, per_lib=results))
        print(json.dumps(out["cases"][-1]), flush=True)
    text = json.dumps(out, indent=1)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
