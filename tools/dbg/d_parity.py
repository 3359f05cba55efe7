"""Relative errors of the full-size Discriminator (bf16) against the fp32 CPU oracle: default engine and the opt-in
pooled-once shortcut (IEA_DBLOCK_POOL_ONCE=1)."""
import os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import iea_gan_b200 as P
from iea_gan_b200.default_config import shipped_config
from oracle import iea_oracle as O

def rel(a, b):
    a, b = a.detach().float().cpu(), b.detach().float().cpu()
    return float((a - b).norm() / (b.norm() + 1e-30))

cfg = shipped_config(H_base=1, device="cuda")
torch.manual_seed(0)
D0 = P.Discriminator(**cfg)
with torch.no_grad():
    D0.blocks[2][2].gamma.fill_(0.5)
sd = {k: v.detach().clone() for k, v in D0.state_dict().items()}
torch.manual_seed(21)
x = torch.rand(40, 1, 256, 256) * 2 - 1
y = torch.arange(40)
go, ge = torch.randn(40), torch.randn(40, cfg["hypersphere_dim"])
names = [n for n, p in D0.named_parameters() if p.dim() >= 2][:60]
for n in names:
    sd[n].requires_grad_(True)
xr = x.clone().requires_grad_(True)
pr, er, orr = O.discriminator_forward(sd, dict(cfg, device="cpu"), xr, y, training=True)
((orr * go).sum() + (er * ge).sum()).backward()
res = {}
for tag, env in (("once", {"IEA_DBLOCK_POOL_ONCE": "1"}), ("old", {})):
    os.environ.update(env)
    torch.manual_seed(0)
    D = P.Discriminator(**cfg)
    D.load_state_dict({k: v.detach() for k, v in sd.items()})
    D = D.cuda().train()
    xg = x.cuda().requires_grad_(True)
    p, e, o = D(xg, y.cuda())
    ((o * go.cuda()).sum() + (e * ge.cuda()).sum()).backward()
    torch.cuda.synchronize()
    for k in env:
        os.environ.pop(k)
    got = dict(D.named_parameters())
    res[tag] = {"e": rel(e, er), "o": rel(o, orr), "dx": rel(xg.grad, xr.grad)}
    res[tag].update({n: rel(got[n].grad, sd[n].grad) for n in names})
print("%-34s %10s %10s" % ("", "pool_once", "default"))
for k in res["once"]:
    print("%-34s %10.4f %10.4f" % (k, res["once"][k], res["old"][k]))
