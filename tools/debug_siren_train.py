"""SirenNeRF fused training path bring-up: forward-train raw vs inference kernel; gradients vs the fp32 layer-wise path."""
import sys
import torch
from msra_practice_project_b200 import models, ops

n, s = (int(sys.argv[1]), int(sys.argv[2])) if len(sys.argv) > 2 else (700, 64)
g = torch.Generator().manual_seed(1)
torch.manual_seed(0)
net = models.SirenNeRF().cuda()
o = torch.tensor([0.0, 0.0, 1.2]).expand(n, 3)
d = torch.nn.functional.normalize(torch.randn(n, 3, generator=g) * 0.25 + torch.tensor([0.0, 0.0, -1.0]), dim=-1)
rays = torch.stack([o, d], 1).cuda()
z = (torch.sort(torch.rand(n, s, generator=g), -1).values * 1.0 + 0.5).cuda()
up = torch.randn(n * s, 4, generator=g).cuda()
kind = models.KIND_SIREN
flat = models.flat_params(net).detach()
with torch.no_grad():
    raw_inf = ops.mlp(net, rays=rays, z=z, precision="bf16")
raw_tr, saved = ops.tc_train_forward(ops.pack_tc(flat, kind), kind, rays, z)
torch.cuda.synchronize()
print("train-forward vs inference raw: max abs diff", (raw_tr - raw_inf).abs().max().item(), "saved bytes", saved.numel())
if len(sys.argv) > 3:
    res = {}
    for mode in ("fp32", "bf16"):
        ops.set_grad_precision(mode)
        net.zero_grad(set_to_none=True)
        raw = ops.mlp(net, rays=rays, z=z)
        (raw * up).sum().backward()
        torch.cuda.synchronize()
        res[mode] = {k: p.grad.detach().clone() for k, p in net.named_parameters()}
    for k in res["fp32"]:
        ga, gb = res["fp32"][k].reshape(-1), res["bf16"][k].reshape(-1)
        cos = torch.dot(ga, gb) / (ga.norm() * gb.norm() + 1e-30)
        print("%-28s |fp32| %.4e |bf16| %.4e rel %.4g cos %.4f" % (k, ga.norm(), gb.norm(), (ga - gb).norm() / max(ga.norm().item(), 1e-20), cos))
