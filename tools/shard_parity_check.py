import os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from graphlearninglayer_b200 import LaplaceLearningSparseHard, sharded as sh, last_info
from graphlearninglayer_b200.losses import custom_ce_loss
from graphlearninglayer_b200.synth import synth_inputs
k_lab, m, d, l = 8192, 122880, 256, 100
X, Y, _, yq = synth_inputs(1000, k_lab, m, d, l, 3.0)
Xd = torch.as_tensor(X).cuda().requires_grad_(True); Yd = torch.as_tensor(Y).cuda(); yq_d = torch.as_tensor(yq).cuda()
def call(layer):
    Xd.grad = None
    pred = layer(Xd, Yd, 0.0, "auto")
    custom_ce_loss(pred, yq_d).backward()
    return pred.detach().clone(), Xd.grad.detach().clone()
pu, du = call(LaplaceLearningSparseHard.apply); print("unsharded", last_info())
for part in ("columns", "rows"):
    for em in (2, 8):
        pc, dc = call(lambda a, b, c, e: sh.ShardedLaplaceLearning.apply(a, b, c, e, None, em, part))
        print(part, em, "pred diff", float((pc - pu).abs().max() / pu.abs().max()), "dx diff", float((dc - du).abs().max() / du.abs().max()), sh.last_info()["knn_fallback_rows"], "alias", pc.data_ptr() == pu.data_ptr())
