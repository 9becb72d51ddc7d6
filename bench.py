#!/usr/bin/env python
"""bench.py -- GLL hot-path benchmark (BASELINE.json metric: GLL fwd+bwd calls/s, CG iterations/s vs HBM roofline).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c1|c2|c3|c4|c5|c5s] [--impl b200|reference]
                    [--dump-outputs DIR]

One "step" = one call of the hot path on one synthetic graph:
    pred = LaplaceLearningSparseHard.apply(X, Y, tau, eps); loss = custom_ce_loss(pred, y); loss.backward()
Workloads (BASELINE.json configs, SURVEY.md 8d): c1 = 1000 + 1000, d=128, eps=1 (the reference's CPU-runnable case);
c2 = 10000 base + 512 batch, d=512, eps='auto' (default: the config the metric is quoted on for one GPU); c3 = 4096 + 512;
c4 = 2048 + 14336 (CG roofline study); c5 / c5s = ONE graph of 2^20 / 2^17 nodes sharded over the ranks.
N > 1: every rank runs its own independent graph of the same shape (different seed) -- the layer has no
parameters, so there is no data-path collective (weak scaling, SURVEY.md 8e row 1).

value  : calls/s with X, Y resident in HBM, timed per step with CUDA events on the launch stream, L2 flushed
         between steps, max over ranks.
e2e    : the same call through the public autograd API starting from pinned HOST buffers: H2D of X and Y, the call,
         D2H of pred and dX, all inside the timed region, ONE CALL AT A TIME (what a training loop sees); the
         double-buffered HostPipeline figure for independent calls is reported beside it (e2e.pipelined_value).
roofline / kernels : a second pass of the same K steps with the library's per-kernel CUDA-event brackets on
         (gll_profile_enable), so the timed `value` pass carries no instrumentation.  roofline.cg_c4_* (N = 1): the
         north star's own figure -- CG iterations/s and algorithmic GB/s of the on-chip CG at n = 16384.
config.c5_* / config.c5s_* : the sharded 1M-node graph (BASELINE.json configs[4]) timed at this N (strong scaling: the same
         graph at every N) and, at N > 1, the parity of the sharded path against the unsharded layer on real ranks.
cpu_baseline : the fp64 numpy/scipy oracle (a port of the reference's GLL.py, see oracle/gll_oracle.py) on this
         box's host cores, rank 0 at N=1 only, bounded sample; plus the reference's own stable_conjgrad semantics
         (GLL.py:247-276, alias included) timed on the C4 system: cpu_baseline.cg_iters_per_sec.
--impl reference : only the oracle port, all host threads, same JSON line with "impl": "reference".
--dump-outputs DIR : pred, loss and dX of the last step of the pass `value` is timed on, as DIR/<name>.npy (rank 0;
         a tensor over 30 MB as a seeded sample of its rows).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

# name: (k_lab, m, d, l, sigma, tau, eps)
WORKLOADS = {
    "c1": (1000, 1000, 128, 10, 3.0, 0.0, 1.0),          # BASELINE.json configs[0]: the reference's CPU-runnable case
    "c2": (10000, 512, 512, 10, 4.5, 0.0, "auto"),
    "c3": (4096, 512, 512, 10, 4.5, 0.0, "auto"),
    "c4": (2048, 14336, 512, 10, 4.5, 0.0, "auto"),
    "c5": (65536, 983040, 256, 100, 3.0, 0.0, "auto"),   # ONE graph sharded over the ranks (strong scaling)
    "c5s": (8192, 122880, 256, 100, 3.0, 0.0, "auto"),   # 1/8-size version of c5 for quick runs
}
SHARDED = ("c5", "c5s")
WORKLOAD_DESC = {
    "c1": "LaplaceLearningSparseHard fwd+bwd, 1000 base + 1000 batch, d=128, l=10, eps=1, tau=0, k=25",
    "c2": "GLL classifier head, 10000 base + 512 batch, d=512, l=10, eps='auto', tau=0, k=25",
    "c3": "data-parallel GLL step, 4096 base + 512 batch per rank, d=512, l=10, eps='auto', tau=0, k=25",
    "c4": "large single graph, 2048 base + 14336 unlabeled, d=512, l=10, eps='auto', tau=0, k=25, CG tol 1e-7",
    "c5": "sharded Laplace learning, ONE graph of n=2^20 nodes (65536 labeled), d=256, l=100, eps='auto', tau=0, k=25; "
          "kNN/backward row-sharded, CG column-sharded, NCCL all-gathers",
    "c5s": "sharded Laplace learning, ONE graph of n=131072 nodes (8192 labeled), d=256, l=100, eps='auto', tau=0, k=25; "
           "kNN/backward row-sharded, CG column-sharded, NCCL all-gathers",
}
METRIC = "gll_fwd_bwd_calls_per_sec"
UNIT = "calls/s"


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        z = json.load(open(p))
        return dict(hbm_gbs=float(z["hbm_gbs"]), tflops=float(z["bf16_tflops"]), source="measured (MEASURED_PEAKS.json, burst)",
                    tflops_sustained=float(z.get("bf16_tflops_sustained", z["bf16_tflops"])))
    return dict(hbm_gbs=6650.0, tflops=1590.0, source="fallback (B200_PROFILING.md)")


class ClockSampler:
    """nvidia-smi sampled every 100 ms during the timed region (B200_PROFILING.md clocks line)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
                pw.append(float(r[2]))
                for nm, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            except (ValueError, IndexError):
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


# ----------------------------------------------------------------------------------------------------------------
# CPU arm: the oracle port of the reference path (checker code; never on the GPU product path)
# ----------------------------------------------------------------------------------------------------------------
def pin_host_threads():
    """All host cores for the CPU arm, the same at every N (torchrun exports OMP_NUM_THREADS=1 to its children)."""
    n = os.cpu_count() or 1
    try:
        import torch

        torch.set_num_threads(n)
    except Exception:
        pass
    try:
        from threadpoolctl import threadpool_limits

        threadpool_limits(limits=n)
    except Exception:
        pass
    return host_threads()


def cpu_calls(workload, seed, n_calls, budget_s):
    from oracle import gll_oracle as O

    k_lab, m, d, l, sigma, tau, eps = WORKLOADS[workload]
    X, Y, _, yq = O.synth_inputs(seed, k_lab, m, d, l, sigma)
    times = []
    t_all = time.perf_counter()
    for _ in range(n_calls):
        t0 = time.perf_counter()
        O.fwd_bwd(X, Y, yq, tau, eps)  # exact kNN + scipy graph + LU/CG solves + per-edge backward, fp64
        times.append(time.perf_counter() - t0)
        if time.perf_counter() - t_all > budget_s:
            break
    return times


def cpu_cg_iters_per_sec(budget_s=20.0):
    """The reference's own CG (stable_conjgrad, GLL.py:247-276, with its `p = r` alias) on the C4 system L_uu u = B:
    matvecs per second on the host (SURVEY 8d last row).  Returns (iters/s, matvecs, seconds) or None."""
    from oracle import gll_oracle as O

    k_lab, m, d, l, sigma, tau, eps = WORKLOADS["c4"]
    X, Y, _, _ = O.synth_inputs(2000, k_lab, m, d, l, sigma)
    g = O.build_graph(X, 25, eps)
    Luu, B, _ = O.laplace_system(g.W, Y, tau)
    t0 = time.perf_counter()
    _, its = O.reference_semantics_cg(Luu, B, tol=1e-6, max_iter=2000)  # BASELINE configs[3]: CG to 1e-6 residual
    dt = time.perf_counter() - t0
    return its / dt, its, dt


def host_threads():
    try:
        from threadpoolctl import threadpool_info

        return max([p.get("num_threads", 1) for p in threadpool_info()] + [1])
    except Exception:
        return os.cpu_count() or 1


CONFIG_KEYS = ("workload", "l2", "parallelism", "cg_tol", "loss", "what", "execution", "eager_calls_per_sec", "loss_head_calls_per_sec", "c4_calls_per_sec", "c4_ms_per_call",
               "c5_ms_per_call", "c5_nodes", "c5_cg_partition", "c5_knn_ms", "c5_cg_solve_ms_fwd", "c5_cg_solve_ms_bwd",
               "c5s_ms_per_call_columns", "c5s_ms_per_call_rows_p2p", "c5s_parity_pred_vs_unsharded",
               "c5s_parity_dx_vs_unsharded", "c5s_parity_rows_p2p_pred", "c5s_parity_rows_p2p_dx")


def make_config(**kw):
    """Both arms print the same key set (flat scalars: the driver keeps those)."""
    cfg = {k: None for k in CONFIG_KEYS}
    cfg.update(kw)
    return cfg


def run_reference(args, rank, world):
    if rank != 0:
        return
    cores = pin_host_threads()
    warm = cpu_calls(args.workload, 1000, args.warmup, 120.0)  # honours --warmup (bounded to two minutes)
    times = cpu_calls(args.workload, 1000, args.steps, 1e9)
    total = float(np.sum(times))
    val = len(times) / total
    cb = {"value": val, "unit": UNIT, "cores": cores, "kind": "port",
          "sample": f"{len(times)} full fwd+bwd calls of the workload"}
    if args.workload == "c4" or args.cpu_cg:
        r = cpu_cg_iters_per_sec()
        cb.update({"cg_iters_per_sec": r[0], "cg_matvecs": r[1], "cg_seconds": r[2],
                   "cg_what": "stable_conjgrad semantics (GLL.py:247-276, p = r alias included) on the C4 L_uu, tol 1e-6"})
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": len(times),
        "warmup": len(warm), "ms_per_step": 1e3 * total / len(times), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic gaussian clusters (graphlearninglayer_b200.synth), L2-normalised",
        "config": make_config(workload=args.workload + ": " + WORKLOAD_DESC[args.workload],
                              l2="n/a (host arm)", parallelism="one process, all host threads", cg_tol=1e-13,
                              loss="custom_ce_loss formula in numpy (losses.py:128-136)",
                              what="oracle port of /root/reference GLL.py (exact kNN instead of annoy, scipy sparse, SuperLU/CG), "
                                   "one process on the host cores; the Python reference itself cannot travel to the GPU box"),
        "cpu_baseline": cb,
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------------------------------------------
def algorithmic_work(name, shp, info):
    """(bound, work per launch, unit) for the kernels with a roofline entry (DESIGN.md, SURVEY.md 8d)."""
    n, d, l, m, k = shp["n"], shp["d"], shp["l"], shp["m"], 25
    E, Euu = info["nnz"], info["nnz_uu"]
    if name.startswith("knn_gram_topk"):
        return "tensor", 2.0 * n * n * d, "flop"
    if name == "cg_persistent":
        # B_iter = 8 E_uu + 4 (m+1) + 11 * 4 m l per iteration; one launch = one solve; fwd and bwd solves averaged
        iters = 0.5 * (info["cg_iters_fwd"] + info["cg_iters_bwd"])
        return "hbm", iters * (8.0 * Euu + 4.0 * (m + 1) + 44.0 * m * l), "B"
    if name == "row_gather":
        return "hbm", 8.0 * E + 8.0 * n * d + 12.0 * n, "B"
    if name == "edge_grad":
        return "hbm", 16.0 * E + 8.0 * n * l + 8.0 * n, "B"
    if name == "knn_rerank":
        return "hbm", 4.0 * n * d + 8.0 * n * 32 + 8.0 * n * k, "B"
    if name == "edge_weights":
        return "hbm", 8.0 * n * k + 12.0 * E + 4.0 * (n + 1) + 4.0 * m * l, "B"
    return "hbm", None, "B"


DUMP_BYTES_PER_ARRAY = 30_000_000  # pred and dX: a dump stays under 64 MB


def dump_outputs(out_dir, arrays):
    """--dump-outputs: writes each tensor as out_dir/<name>.npy (float32 / float64, as computed), so that two builds can be
    compared output for output.  A tensor above DUMP_BYTES_PER_ARRAY is cut to a sample of its rows drawn with a fixed
    seed (sorted; the same rows in every run of the same workload)."""
    import torch

    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        t = t.detach()
        if t.dtype not in (torch.float32, torch.float64):
            raise TypeError(f"bench.py: output {name} is {t.dtype}, not float32/float64")
        if t.numel() * t.element_size() > DUMP_BYTES_PER_ARRAY:
            keep = DUMP_BYTES_PER_ARRAY // (t[0].numel() * t.element_size())
            rows = np.sort(np.random.default_rng(0).choice(t.shape[0], size=keep, replace=False))
            print(f"bench.py: {name} dumped as a seeded sample of {keep} of its {t.shape[0]} rows", file=sys.stderr)
            t = t[torch.as_tensor(rows, device=t.device)]
        np.save(os.path.join(out_dir, name + ".npy"), t.cpu().numpy())


def run_b200(args, rank, world, local_rank):
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the B200 arm has no CPU fallback (use --impl reference for the CPU arm)")
    import graphlearninglayer_b200 as pkg
    from graphlearninglayer_b200 import _lib, ranks
    from graphlearninglayer_b200.synth import synth_inputs  # numpy input generator (the oracle is not imported by this arm)

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=dev)

    def step_fn(shape_name, seed):
        k_lab, m, d, l, sigma, tau, eps = WORKLOADS[shape_name]
        if shape_name in SHARDED:
            from graphlearninglayer_b200.sharded import ShardedLaplaceLearning

            layer = ShardedLaplaceLearning.apply  # every rank passes the same graph, collectives inside
        else:
            layer = pkg.LaplaceLearningSparseHard.apply
        X, Y, _, yq = synth_inputs(seed, k_lab, m, d, l, sigma)
        Xh = torch.as_tensor(X).pin_memory()
        Yh = torch.as_tensor(Y).pin_memory()
        Xd = Xh.to(dev).requires_grad_(True)
        Yd = Yh.to(dev)
        yq_d = torch.as_tensor(yq).to(dev)
        if args.loss == "torch":   # the reference function body, op by op (losses.py:128-136)
            tgt = torch.nn.functional.one_hot(yq_d, l).to(torch.float64)

            def ce(pred):
                return -torch.sum(tgt * torch.log(pred + 1e-8)) / m
        else:                      # the same function as one kernel (graphlearninglayer_b200/losses.py, SURVEY 8f-3)
            from graphlearninglayer_b200.losses import custom_ce_loss

            def ce(pred):
                return custom_ce_loss(pred, yq_d)
        predh = torch.empty((m, l), dtype=torch.float64).pin_memory()
        dXh = torch.empty((k_lab + m, d), dtype=torch.float32).pin_memory()
        Xe = torch.empty_like(Xd).requires_grad_(True)
        Ye = torch.empty_like(Yd)

        # "ev": set to a list to have resident() record (start, after forward+loss, end) events;
        # "out": (pred, loss, dX) of the latest resident() call, what a caller of the layer receives
        split = {"ev": None, "out": None}

        def resident():
            Xd.grad = None
            ev = None
            if split["ev"] is not None:
                ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
                ev[0].record()
            pred = layer(Xd, Yd, tau, eps)
            loss = ce(pred)  # custom_ce_loss, losses.py:128-136
            if ev is not None:
                ev[1].record()
            loss.backward()
            if ev is not None:
                ev[2].record()
                split["ev"].append(ev)
            split["out"] = (pred.detach(), loss.detach(), Xd.grad)  # detached: the layer's state is freed with its graph
            return loss

        def e2e():
            Xe.grad = None
            with torch.no_grad():
                Xe.copy_(Xh, non_blocking=True)
                Ye.copy_(Yh, non_blocking=True)
            pred = layer(Xe, Ye, tau, eps)
            loss = ce(pred)
            loss.backward()
            predh.copy_(pred.detach(), non_blocking=True)
            dXh.copy_(Xe.grad, non_blocking=True)
            return loss

        def e2e_pipelined(steps, warmup):
            """Same host-buffer calls, double buffered (graphlearninglayer_b200.hostpipe): H2D of step i+1 and D2H of
            step i-1 overlap the kernels of step i.  Returns the device-timed ms for `steps` calls, all copies inside."""
            from graphlearninglayer_b200.hostpipe import HostPipeline

            pipe = HostPipeline(k_lab + m, d, k_lab, l, dev, tau=tau, epsilon=eps, layer=layer, depth=3,
                                loss_fn=lambda pred, slot: ce(pred))
            for _ in range(warmup):
                if pipe.outstanding == pipe.depth:
                    pipe.collect()
                pipe.submit(Xh, Yh)
            pipe.drain()
            torch.cuda.synchronize()
            if dist is not None:
                dist.barrier()
            torch.cuda.synchronize()
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ev0.record()
            for _ in range(steps):
                if pipe.outstanding == pipe.depth:
                    pipe.collect()
                pipe.submit(Xh, Yh)
            pipe.drain()
            ev1.record()
            torch.cuda.synchronize()
            if dist is not None:
                dist.barrier()
            ms = ev0.elapsed_time(ev1)
            _, ms, _ = ranks.aggregate_throughput(steps, ms, device=str(dev))
            return ms, pipe.h2d_bytes, pipe.d2h_bytes

        shp = dict(n=k_lab + m, d=d, l=l, m=m, k_lab=k_lab)
        h2d = Xh.numel() * 4 + Yh.numel() * 4
        d2h = predh.numel() * 8 + dXh.numel() * 4
        split["tensors"] = dict(Xd=Xd, Yd=Yd, yq=yq_d, tau=tau, eps=eps)
        return resident, e2e, shp, h2d, d2h, e2e_pipelined, split

    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # 256 MiB > 126 MB L2

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        for a, b in ev:
            flush.zero_()          # L2 flush between timed iterations (outside the event pair)
            a.record()
            fn()
            b.record()
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()
        tot_ms = sum(a.elapsed_time(b) for a, b in ev)
        # whole-job time = max over ranks (graphlearninglayer_b200.ranks: all_reduce MAX; no data-path collective)
        _, tot_ms, _ = ranks.aggregate_throughput(steps, tot_ms, device=str(dev))
        return tot_ms

    sharded = args.workload in SHARDED
    # weak scaling measures the machine, not the data: every rank runs the SAME synthetic graph (seed 1000), each on its own
    # GPU with its own buffers.  (Different seeds change a rank's step by up to 8 %: a seed whose graph has rows that need the
    # exact brute-force fallback pays ~0.02 ms per such row, and the job waits for its slowest rank.)
    seed = 1000 if (sharded or not args.rank_seeds) else ranks.rank_seed(1000, rank)
    resident, e2e, shp, h2d, d2h, e2e_pipelined, split = step_fn(args.workload, seed)
    jobs = 1 if sharded else world  # graphs finished per step by the whole job
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    l0 = _lib.launch_count()
    eager_ms = timed(resident, args.steps, args.warmup)
    launches = (_lib.launch_count() - l0) * args.steps // (args.steps + args.warmup)
    # the same step replayed from CUDA graphs (graphlearninglayer_b200.graphed: forward + loss and backward captured once,
    # two graph launches per step, the same kernels): this is `value`; the eager figure is kept beside it
    tot_ms, execution = eager_ms, "eager launches through LaplaceLearningSparseHard.apply"
    outputs = split["out"]  # (pred, loss, dX) of the last step of the path `value` is timed on
    extra_cfg = {}
    if not sharded and not args.no_cuda_graph and args.loss == "fused":
        try:
            from graphlearninglayer_b200.graphed import GraphedStep

            tn = split["tensors"]
            gs = GraphedStep(shp["n"], shp["d"], shp["k_lab"], shp["l"], dev, tau=tn["tau"], epsilon=tn["eps"],
                             warmup_inputs=(tn["Xd"].detach(), tn["Yd"], tn["yq"]))
            replayed = {}

            def replay():
                loss = gs(tn["Xd"], tn["Yd"], tn["yq"])
                replayed["out"] = (gs.pred, loss, gs.dX)  # static tensors of gs, untouched by the other passes

            tot_ms = timed(replay, args.steps, args.warmup)
            execution = "CUDA graph replay (GraphedStep: 2 graph launches per step, same kernels)"
            outputs = replayed["out"]
        except Exception as e:  # capture not available: say so, keep the eager number
            execution += f" (graph capture failed: {type(e).__name__}: {e})"[:300]
        try:  # extra, NOT the headline: the same step with the loss fused behind the layer in one autograd node (8f-3)
            gh = GraphedStep(shp["n"], shp["d"], shp["k_lab"], shp["l"], dev, tau=tn["tau"], epsilon=tn["eps"],
                             warmup_inputs=(tn["Xd"].detach(), tn["Yd"], tn["yq"]), loss_head=True)
            head_ms = timed(lambda: gh(tn["Xd"], tn["Yd"], tn["yq"]), args.steps, args.warmup)
            extra_cfg["loss_head_calls_per_sec"] = jobs * 1e3 / (head_ms / args.steps)
        except Exception as e:
            print(f"bench.py: loss-head variant not measured: {type(e).__name__}: {e}", file=sys.stderr)
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, dict(zip(("pred", "loss", "dX"), outputs)))
    e2e_ms = timed(e2e, args.steps, args.warmup)
    pipe_ms = None
    if not sharded:
        pipe_ms, _, _ = e2e_pipelined(args.steps, args.warmup)
    if sharded:
        from graphlearninglayer_b200 import sharded as sharded_mod

        info = sharded_mod.last_info()
    else:
        info = pkg.last_info()

    # forward / backward split (SURVEY 8d), its own pass: two extra events per step
    split["ev"] = []
    for _ in range(args.steps):
        flush.zero_()
        resident()
    torch.cuda.synchronize()
    fwd_ms = sum(e[0].elapsed_time(e[1]) for e in split["ev"]) / args.steps
    bwd_ms = sum(e[1].elapsed_time(e[2]) for e in split["ev"]) / args.steps
    split["ev"] = None

    # per-kernel pass (instrumented; not the pass `value` comes from)
    _lib.lib.gll_profile_enable(1)
    _lib.profile_collect()
    for _ in range(args.steps):
        flush.zero_()
        resident()
    torch.cuda.synchronize()
    prof = _lib.profile_collect()
    _lib.lib.gll_profile_enable(0)

    extra = {}
    c4 = None
    if rank == 0 and world == 1 and args.workload not in ("c4",) + SHARDED and not args.no_large_graph:
        # the CG roofline study (BASELINE.json configs[3]); reported beside the headline, not instead of it
        r4, _, shp4, _, _, _, _ = step_fn("c4", 2000)
        ms4 = timed(r4, 5, 3)
        info4 = pkg.last_info()
        _lib.lib.gll_profile_enable(1)
        _lib.profile_collect()
        for _ in range(5):
            flush.zero_()
            r4()
        torch.cuda.synchronize()
        prof4 = _lib.profile_collect()
        _lib.lib.gll_profile_enable(0)
        c4 = large_graph_report(prof4, shp4, info4, ms4 / 5)
        extra["large_graph_c4"] = c4
        del r4
        torch.cuda.empty_cache()

    # ---- the sharded 1M-node graph (BASELINE.json configs[4]) at this N: strong scaling, plus parity on real ranks ----
    shard_cfg = {}
    if not sharded and not args.no_sharded:
        shard_cfg = sharded_lines(args, rank, world, dev, dist)

    if rank == 0:
        peaks = load_peaks()
        per_step = tot_ms / args.steps
        kern = {}
        step_kernel_ms = sum(v[0] for v in prof.values()) / args.steps
        for nm, (ms, cnt) in sorted(prof.items(), key=lambda kv: -kv[1][0]):
            kern[nm] = {"ms_per_launch": ms / cnt, "launches_per_step": cnt / args.steps,
                        "share_of_kernel_time": (ms / args.steps) / step_kernel_ms}
        top = max(prof.items(), key=lambda kv: kv[1][0])[0]
        if sharded:
            top = "knn_gram_topk_tcgen05" if "knn_gram_topk_tcgen05" in prof else top
            shp = dict(shp, n_rows_this_rank=-(-shp["n"] // world))
        bound, work, unit = algorithmic_work(top, shp, info)
        if sharded and bound == "tensor":
            work = work / world  # each rank searches n/world rows against all n columns
        t_s = prof[top][0] / prof[top][1] * 1e-3
        peak_source = peaks["source"]
        if bound == "tensor":
            ach, peak, u = work / t_s / 1e12, peaks["tflops"], "TFLOP/s"
            if t_s > 0.05 and "tflops_sustained" in peaks:  # a launch of tens of ms runs under the power cap: sustained cuBLAS figure
                peak, peak_source = peaks["tflops_sustained"], "measured (MEASURED_PEAKS.json, sustained: the launch lasts > 50 ms)"
        else:
            ach, peak, u = (work / t_s / 1e9 if work else None), peaks["hbm_gbs"], "GB/s"
        traffic = None  # DRAM bytes per launch of that kernel from the committed ncu --set full capture (same workload)
        tpath = os.path.join(ROOT, "profiles", "ncu_traffic.json")
        if os.path.exists(tpath):
            traffic = json.load(open(tpath)).get(args.workload, {}).get(top)
        roofline = {"kernel": top, "bound": bound, "achieved": ach, "peak": peak, "unit": u,
                    "frac": (ach / peak if ach else None), "traffic": traffic, "peak_source": peak_source,
                    "algorithmic_work_per_launch": work, "work_unit": unit, "launch_ms": t_s * 1e3,
                    "share_of_step": (prof[top][0] / args.steps) / step_kernel_ms}
        if bound == "tensor" and top == "knn_gram_topk_tcgen05":
            # one fp16 MMA pass (hi.hi) by default, two ((hi + lo).hi) with GLL_B200_KNN_SPLIT=f16x2; `achieved` counts 2 n^2 d once
            passes = 2 if os.environ.get("GLL_B200_KNN_SPLIT") == "f16x2" else 1
            roofline.update({"mma_passes": passes, "issued": ach * passes, "issued_frac": ach * passes / peak})
        if c4 is not None and "cg" in c4:
            # the north star's own figure, flat so that the driver's record keeps it: the on-chip CG at n = 16384
            cg = c4["cg"]
            roofline.update({"cg_c4_us_per_iter": cg["us_per_iter"], "cg_c4_iters_per_sec": cg["iters_per_sec"],
                             "cg_c4_bytes_per_iter": cg["bytes_per_iter"], "cg_c4_achieved_gbs": cg["achieved_gbs"],
                             "cg_c4_frac_of_hbm_peak": cg["frac"], "cg_c4_ms_per_solve": cg["ms_per_solve"],
                             "cg_c4_iters_fwd": c4["graph"]["cg_iters_fwd"], "cg_c4_iters_bwd": c4["graph"]["cg_iters_bwd"],
                             "cg_c4_note": "working set (4 MB CSR + vectors) is on chip: an iteration is two grid barriers + one "
                                           "L1TEX-bound gather, not HBM traffic; see profiles/r02_cg_trace.md"})
        cpu = None
        if world == 1 and not args.no_cpu_baseline and not sharded:
            cores = pin_host_threads()
            times = cpu_calls(args.workload, 1000, 4, 25.0)
            cpu = {"value": len(times) / float(np.sum(times)), "unit": UNIT, "cores": cores, "kind": "port",
                   "sample": f"{len(times)} full fwd+bwd calls of the same workload through oracle/gll_oracle.py (fp64)"}
            r = cpu_cg_iters_per_sec()
            cpu.update({"cg_iters_per_sec": r[0], "cg_matvecs": r[1], "cg_seconds": r[2],
                        "cg_what": "stable_conjgrad semantics (GLL.py:247-276, p = r alias included) on the C4 L_uu, tol 1e-6"})
        cfg = make_config(
            workload=args.workload + ": " + WORKLOAD_DESC[args.workload],
            l2="flushed between timed steps (256 MiB memset outside the event pairs)",
            parallelism=(f"one graph over {world} rank(s): rows (kNN, backward) + "
                         + ("class columns (CG, no per-iteration collective)" if args.cg_partition == "columns" else
                            "rows (CG: NCCL all-gather of the iterate + all-reduce of the dot products per iteration)"
                            if args.cg_partition == "rows" else
                            "rows (CG: iterate and dot products exchanged INSIDE the kernels over NVLink peer memory)")
                         if sharded else f"independent graphs x{world}"),
            cg_tol=1e-7,
            loss=("custom_ce_loss as one kernel (graphlearninglayer_b200.losses; formula of losses.py:128-136)"
                  if args.loss == "fused" else "custom_ce_loss with the reference's PyTorch ops (losses.py:128-136)"),
            what="libgll_b200.so (sm_100a kernels) through LaplaceLearningSparseHard.apply",
            execution=execution, eager_calls_per_sec=jobs * 1e3 / (eager_ms / args.steps),
            **shard_cfg, **extra_cfg)
        if c4 is not None:
            cfg.update(c4_calls_per_sec=c4["calls_per_sec"], c4_ms_per_call=c4["ms_per_call"])
        line = {
            "metric": METRIC, "value": jobs * 1e3 / per_step, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": per_step, "higher_is_better": True,
            "scaling": "strong" if sharded else "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic gaussian clusters (graphlearninglayer_b200.synth), L2-normalised, one graph per rank "
                                    + ("(a different seed per rank)" if args.rank_seeds else "(the same seed on every rank)"),
            "config": cfg,
            # e2e: host buffers in, host buffers out, every copy inside the timed region, ONE CALL AT A TIME on one stream
            # (a training loop's calls depend on each other).  pipelined_value: independent calls through HostPipeline
            # (depth 3: H2D(i+1) | kernels(i) | D2H(i-1) on three streams).
            "e2e": {"value": jobs * 1e3 / (e2e_ms / args.steps), "unit": UNIT, "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "ms_per_step": e2e_ms / args.steps,
                    "mode": "serial: one call at a time on one stream (H2D, kernels, D2H back to back), L2 flushed between steps",
                    **({"pipelined_value": jobs * 1e3 / (pipe_ms / args.steps), "pipelined_ms_per_step": pipe_ms / args.steps,
                        "pipelined_mode": "HostPipeline depth 3, independent calls; bound by the PCIe copies in both directions"}
                       if pipe_ms is not None else {})},
            "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline,
            "fwd_bwd_split_ms": {"forward_and_loss": fwd_ms, "backward": bwd_ms},
            "graph": {"nnz": info["nnz"], "nnz_uu": info["nnz_uu"], "cg_iters_fwd": info["cg_iters_fwd"],
                      "cg_iters_bwd": info["cg_iters_bwd"], "knn_fallback_rows": info["knn_fallback_rows"], "status": info["status"],
                      **({"cg_solve_ms_fwd_bwd": info.get("cg_solve_ms")} if sharded else {})},
            "kernels": kern,
            "cpu_baseline": cpu,
        }
        line.update(extra)
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()


def sharded_lines(args, rank, world, dev, dist):
    """ONE graph over all ranks (graphlearninglayer_b200.sharded): the 1M-node graph of BASELINE.json configs[4] timed at
    this N with the current kernels (strong scaling: the same graph at every N; N = 1 is the reference point), and at
    N > 1 the 131072-node graph run sharded on the REAL ranks -- class-column CG and the row-partitioned CG over NVLink peer
    memory -- against the unsharded layer on rank 0.  Returns flat config entries (identical on every rank)."""
    import torch

    from graphlearninglayer_b200 import LaplaceLearningSparseHard, sharded as sh
    from graphlearninglayer_b200.losses import custom_ce_loss
    from graphlearninglayer_b200.synth import synth_inputs

    out = {}

    def run(shape, partition, calls, seed=1000):
        k_lab, m, d, l, sigma, tau, eps = WORKLOADS[shape]
        X, Y, _, yq = synth_inputs(seed, k_lab, m, d, l, sigma)  # the same graph on every rank
        Xd = torch.as_tensor(X).to(dev).requires_grad_(True)
        Yd = torch.as_tensor(Y).to(dev)
        yq_d = torch.as_tensor(yq).to(dev)
        del X

        def call(layer):
            Xd.grad = None
            pred = layer(Xd, Yd, tau, eps)
            custom_ce_loss(pred, yq_d).backward()
            return pred.detach()

        def sharded_layer(a, b, c, e):
            return sh.ShardedLaplaceLearning.apply(a, b, c, e, None, 0, partition)

        for _ in range(2):  # warm-up (allocator, symmetric memory rendezvous, NCCL channels and their lazily grown buffers)
            pred = call(sharded_layer)
        per_call = []
        for _ in range(calls):  # one event pair per call, barrier in front; the MEDIAN call is reported (a first call after an
            torch.cuda.synchronize()  # allocator trim or an NCCL buffer growth takes 3-5x the steady time)
            if dist is not None:
                dist.barrier()
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ev0.record()
            pred = call(sharded_layer)
            ev1.record()
            torch.cuda.synchronize()
            per_call.append(ev0.elapsed_time(ev1))
        ms = sorted(per_call)[len(per_call) // 2]
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        info = sh.last_info()
        return float(t.item()), pred, Xd.grad.detach().clone(), info, (lambda: call(LaplaceLearningSparseHard.apply), Xd)

    def rel(a, b):
        return float((a - b).abs().max().item() / max(b.abs().max().item(), 1e-300))

    if world > 1:
        ms_c, pred_c, dx_c, _, (unsharded, Xd) = run("c5s", "columns", 3)
        out["c5s_ms_per_call_columns"] = ms_c
        errs = torch.zeros(4, dtype=torch.float64, device=dev)
        if rank == 0:  # the unsharded layer on one GPU is the yardstick (itself checked against the oracle in tests/)
            pred_u = unsharded()
            dx_u = Xd.grad.detach().clone()
            errs[0], errs[1] = rel(pred_c, pred_u), rel(dx_c, dx_u)
        del unsharded, Xd
        try:
            ms_p, pred_p, dx_p, _, keep = run("c5s", "rows-p2p", 3)
            del keep
            out["c5s_ms_per_call_rows_p2p"] = ms_p
            if rank == 0:
                errs[2], errs[3] = rel(pred_p, pred_u), rel(dx_p, dx_u)
        except Exception as e:  # symmetric memory unavailable on this box: say so instead of dying
            out["c5s_ms_per_call_rows_p2p"] = None
            if rank == 0:
                print(f"bench.py: rows-p2p not run: {e}", file=sys.stderr)
            errs[2] = errs[3] = float("nan")
        dist.broadcast(errs, 0)
        e = errs.cpu().tolist()
        out.update(c5s_parity_pred_vs_unsharded=e[0], c5s_parity_dx_vs_unsharded=e[1], c5s_parity_rows_p2p_pred=e[2],
                   c5s_parity_rows_p2p_dx=e[3])
        torch.cuda.empty_cache()
    if not args.no_c5:
        ms5, _, _, info5, keep = run("c5", "columns", 3)
        del keep
        solve = info5.get("cg_solve_ms") or [None, None]
        out.update(c5_ms_per_call=ms5, c5_nodes=WORKLOADS["c5"][0] + WORKLOADS["c5"][1], c5_cg_partition="columns",
                   c5_cg_solve_ms_fwd=solve[-2] if len(solve) >= 2 else None, c5_cg_solve_ms_bwd=solve[-1] if solve else None)
        torch.cuda.empty_cache()
    return out


def large_graph_report(prof, shp, info, ms_per_call):
    peaks = load_peaks()
    out = {"workload": "c4: " + WORKLOAD_DESC["c4"], "calls_per_sec": 1e3 / ms_per_call, "ms_per_call": ms_per_call,
           "graph": {k: info[k] for k in ("nnz", "nnz_uu", "cg_iters_fwd", "cg_iters_bwd", "cg_resid_fwd", "cg_resid_bwd",
                                          "knn_fallback_rows", "status")}}
    if "cg_persistent" in prof:
        ms, cnt = prof["cg_persistent"]
        iters = info["cg_iters_fwd"] + info["cg_iters_bwd"]
        solves_ms = ms / (cnt / 2)  # one fwd + one adjoint solve per call
        m, l, Euu = shp["m"], shp["l"], info["nnz_uu"]
        b_iter = 8.0 * Euu + 4.0 * (m + 1) + 44.0 * m * l
        gbs = b_iter * iters / (solves_ms * 1e-3) / 1e9
        out["cg"] = {"iters_per_sec": iters / (solves_ms * 1e-3), "us_per_iter": 1e3 * solves_ms / iters, "ms_per_solve": solves_ms / 2,
                     "bytes_per_iter": b_iter, "achieved_gbs": gbs, "peak_gbs": peaks["hbm_gbs"],
                     "frac": gbs / peaks["hbm_gbs"], "note": "working set is L2-resident at this size (SURVEY 8d)"}
    tot = sum(v[0] for v in prof.values())
    out["kernels"] = {nm: {"ms_per_launch": ms / cnt, "share_of_kernel_time": ms / tot}
                      for nm, (ms, cnt) in sorted(prof.items(), key=lambda kv: -kv[1][0])}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workload", choices=sorted(WORKLOADS), default="c2")
    ap.add_argument("--impl", choices=["b200", "reference"], default="b200")
    ap.add_argument("--loss", choices=["fused", "torch"], default="fused",
                    help="custom_ce_loss of the step: graphlearninglayer_b200.losses (one kernel) or the reference's PyTorch ops")
    ap.add_argument("--cg-partition", choices=["columns", "rows", "rows-p2p"], default="columns",
                    help="sharded workloads: split the CG solves by class columns (no per-iteration collective) or by rows "
                         "(all-gather + all-reduce per iteration)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-large-graph", action="store_true")
    ap.add_argument("--rank-seeds", action="store_true", help="N > 1: a different synthetic graph per rank (default: the same graph)")
    ap.add_argument("--no-cuda-graph", action="store_true", help="`value` from eager launches instead of CUDA graph replay")
    ap.add_argument("--no-sharded", action="store_true", help="skip the sharded c5 / c5s lines")
    ap.add_argument("--no-c5", action="store_true", help="skip the 1M-node graph (keeps the c5s parity lines at N > 1)")
    ap.add_argument("--cpu-cg", action="store_true", help="reference arm: also time the reference's CG on the C4 system")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the timed path's last step returned (pred, loss, dX) as "
                         "DIR/<name>.npy; inputs are seeded, so two builds can be compared output for output")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs dumps the B200 arm's outputs; it does not apply to --impl reference")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    os.environ["GLL_B200_SHARD_CG"] = args.cg_partition
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_b200(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
