"""debug: stand-alone GBlock per-parameter errors vs the reference-run vectors; loss trajectories fp32 vs bf16."""
import functools, json, os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests")); sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
import torch
os.environ["IEA_ACT_DTYPE"] = "fp32"
import iea_gan_b200.sn_layers as SL
from iea_gan_b200 import nets
import iea_gan_b200 as P
SN = dict(num_svs=1, num_itrs=1, eps=1e-6)
from golden_io import load_golden
gold = load_golden(os.path.join(ROOT, "tests/golden/modules"))
def rel(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return float((a - b).norm() / (b.norm() + 1e-30))
conv = functools.partial(SL.SNConv2d, kernel_size=3, padding=1, **SN)
lin = functools.partial(SL.SNLinear, bias=False, **SN)
bn = functools.partial(SL.ccbn, which_linear=lin, input_size=32, eps=1e-5)
relu = torch.nn.ReLU(inplace=False)
up = functools.partial(torch.nn.functional.interpolate, scale_factor=2)
for name, m in (("GBlock_up", nets.GBlock(64, 32, which_conv=conv, which_bn=bn, activation=relu, upsample=up)),
                ("GBlock_same", nets.GBlock(64, 64, which_conv=conv, which_bn=bn, activation=relu, upsample=None))):
    rec = gold[name]
    m.load_state_dict(rec["state"]); m = m.cuda().train()
    ins = [t.cuda().requires_grad_(True) for t in rec["inputs"]]
    out = m(*ins)
    g = torch.Generator().manual_seed(rec["cot_seed"])
    w = torch.randn(rec["outputs"][0].shape, generator=g)
    print(name, "out", rel(out, rec["outputs"][0]))
    (out * w.cuda()).sum().backward()
    print("  dx", rel(ins[0].grad, rec["input_grads"][0]), "dy", rel(ins[1].grad, rec["input_grads"][1]))
    ps = dict(m.named_parameters())
    for k, r in rec["param_grads"].items():
        print("  %-22s rel %.3g  |mine| %.3g |ref| %.3g" % (k, rel(ps[k].grad, r), float(ps[k].grad.norm()), float(r.norm())))
# trajectories
from iea_gan_b200.train_step import make_train_step, NormalNoise
cfg = json.load(open(os.path.join(ROOT, "tests/golden/small_cfg.json"))); cfg["device"] = "cuda"
for adt in ("fp32", "bf16", "fp32"):
    os.environ["IEA_ACT_DTYPE"] = adt
    torch.manual_seed(0)
    G, D = P.Generator(**cfg).cuda().train(), P.Discriminator(**cfg).cuda().train()
    torch.manual_seed(77); torch.cuda.manual_seed(77)
    train = make_train_step(G, D, P.G_D(G, D), NormalNoise(40, cfg["dim_z"], "cuda"), cfg)
    y = torch.arange(40, device="cuda")
    for i in range(20):
        x = torch.rand(40, 1, 64, 64, device="cuda") * 2 - 1
        o = train(x, y)
        print(adt, i, " ".join("%s %.4f" % (k[:6], v) for k, v in o.items()))
