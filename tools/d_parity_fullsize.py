import os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
def rel(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return float((a - b).norm() / (b.norm() + 1e-30))
import iea_gan_b200 as P
from iea_gan_b200.default_config import shipped_config
from oracle import iea_oracle as O
cfg = shipped_config(H_base=1, device="cuda")
torch.manual_seed(0)
D0 = P.Discriminator(**cfg)
with torch.no_grad():
    D0.blocks[2][2].gamma.fill_(0.5)
sd0 = {k: v.detach().clone() for k, v in D0.state_dict().items()}
torch.manual_seed(21)
x = torch.rand(40, 1, 256, 256) * 2 - 1
y = torch.arange(40)
go, ge = torch.randn(40), torch.randn(40, cfg["hypersphere_dim"])
names = ["input_conv.weight", "linear0.weight", "linear1.weight", "blocks.0.0.conv2.weight", "blocks.2.2.theta.weight", "blocks.3.1.conv3.weight", "blocks.5.0.conv1.weight"]
sd = {k: v.clone() for k, v in sd0.items()}
for n in names: sd[n].requires_grad_(True)
xr = x.clone().requires_grad_(True)
pr, er, orr = O.discriminator_forward(sd, dict(cfg, device="cpu"), xr, y, training=True)
((orr * go).sum() + (er * ge).sum()).backward()
for mode in ("bf16", "fp32"):
    os.environ["IEA_ACT_DTYPE"] = mode
    D = P.Discriminator(**cfg)
    D.load_state_dict(sd0)
    D = D.cuda().train()
    xg = x.cuda().requires_grad_(True)
    p, e, o = D(xg, y.cuda())
    ((o * go.cuda()).sum() + (e * ge.cuda()).sum()).backward()
    print(mode, "embed %.3g out %.3g dx %.3g" % (rel(e, er), rel(o, orr), rel(xg.grad, xr.grad)), " ".join("%s %.3g" % (n.split(".weight")[0], rel(dict(D.named_parameters())[n].grad, sd[n].grad)) for n in names))
