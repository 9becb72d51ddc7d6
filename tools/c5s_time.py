import os, sys, time, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from graphlearninglayer_b200 import LaplaceLearningSparseHard, sharded as sh, last_info, _lib
from graphlearninglayer_b200.losses import custom_ce_loss
from graphlearninglayer_b200.synth import synth_inputs
k_lab, m, d, l = 8192, 122880, 256, 100
X, Y, _, yq = synth_inputs(1000, k_lab, m, d, l, 3.0)
Xd = torch.as_tensor(X).cuda().requires_grad_(True); Yd = torch.as_tensor(Y).cuda(); yq_d = torch.as_tensor(yq).cuda()
def call(layer):
    Xd.grad = None
    pred = layer(Xd, Yd, 0.0, "auto")
    custom_ce_loss(pred, yq_d).backward()
for part in ("columns", "rows"):
    lay = lambda a, b, c, e: sh.ShardedLaplaceLearning.apply(a, b, c, e, None, 2, part)
    call(lay); torch.cuda.synchronize()
    _lib.lib.gll_profile_enable(1); _lib.profile_collect()
    for i in range(3):
        t0 = time.perf_counter(); call(lay); torch.cuda.synchronize(); print(part, i, round((time.perf_counter() - t0) * 1e3, 2), "ms")
    p = _lib.profile_collect(); _lib.lib.gll_profile_enable(0)
    print({k: (round(v[0], 2), v[1]) for k, v in p.items()})
    print(sh.last_info())
call(LaplaceLearningSparseHard.apply); torch.cuda.synchronize()
t0 = time.perf_counter(); call(LaplaceLearningSparseHard.apply); torch.cuda.synchronize(); print("unsharded", round((time.perf_counter() - t0) * 1e3, 2), "ms", last_info())
_lib.lib.gll_profile_enable(1); _lib.profile_collect()
call(LaplaceLearningSparseHard.apply); torch.cuda.synchronize()
p = _lib.profile_collect(); _lib.lib.gll_profile_enable(0)
print("unsharded kernels", {k: (round(v[0], 2), v[1]) for k, v in p.items()})
ts = []
for i in range(6):
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter(); e0.record(); call(LaplaceLearningSparseHard.apply); e1.record(); t1 = time.perf_counter()
    torch.cuda.synchronize()
    ts.append((round(e0.elapsed_time(e1), 2), round((t1 - t0) * 1e3, 2)))
print("unsharded (device ms, host enqueue ms):", ts)
