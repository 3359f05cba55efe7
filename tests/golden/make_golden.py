"""Generate the golden vectors that pin oracle/iea_oracle.py to the real reference.

Run in the BUILD container only (it imports the unmodified reference from
/root/reference, which does not exist on the GPU box):

    python tests/golden/make_golden.py

It writes small fixtures next to this file:
  small_cfg.json        the reduced configuration (resolution 64, G_ch 16, D_ch 32)
  state_checksums.json  per-tensor (sum, abs-sum) of the reference's freshly
                        constructed G and D state dicts for seed 0 (ctor / RNG parity)
  small_fwd/            seeded inputs and the reference's G / D / DiffAugment / loss outputs
  small_step/           one unmodified train_fns.train step: the 5 returned floats,
                        per-parameter gradient norms, a few full gradients, u0/sv0 and
                        BN running statistics after the step
  full_checksums.json   ctor checksums of the shipped-size nets (H_base 1 and 3)
small_fwd/ and small_step/ are golden sets in the layout of golden_io.py.
"""
import json
import os
import sys
import types

import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from golden_io import save_golden  # noqa: E402

REF = "/root/reference"
HERE = os.path.dirname(os.path.abspath(__file__))


def import_reference():
    for name in ["boost_histogram", "matplotlib", "matplotlib.pyplot", "seaborn", "cleanfid",
                 "cleanfid.downloads_helper", "cleanfid.inception_pytorch", "cleanfid.resize",
                 "cleanfid.utils", "cleanfid.features", "cleanfid.inception_torchscript"]:
        m = types.ModuleType(name)
        m.__path__ = []
        sys.modules.setdefault(name, m)
    sys.modules["cleanfid.inception_pytorch"].InceptionV3 = object
    sys.modules["matplotlib"].pyplot = sys.modules["matplotlib.pyplot"]
    sys.path.insert(0, REF)
    import model, layers, RRM, diff_aug, loss  # noqa
    return model, layers, RRM, diff_aug, loss


def base_config():
    with open(os.path.join(REF, "config.json")) as f:
        cfg = json.load(f)
    cfg["device"] = "cpu"
    return cfg


def small_config():
    cfg = base_config()
    cfg.update(resolution=64, G_ch=16, D_ch=32, H_base=1, D_attn="16", clip_norm=1e9,
               num_workers=0, ema=False)
    return cfg


def checksums(sd):
    return {k: [float(v.double().sum()), float(v.double().abs().sum()), list(v.shape)] for k, v in sd.items()}


def main():
    model, layers, RRM, diff_aug, loss = import_reference()
    torch.set_num_threads(8)
    cfg = small_config()
    with open(os.path.join(HERE, "small_cfg.json"), "w") as f:
        json.dump(cfg, f, indent=1)

    # ---------------- ctor parity ----------------
    torch.manual_seed(0)
    G = model.Generator(**cfg)
    D = model.Discriminator(**cfg)
    sums = {"G": checksums(G.state_dict()), "D": checksums(D.state_dict())}
    with open(os.path.join(HERE, "state_checksums.json"), "w") as f:
        json.dump(sums, f)

    # ---------------- forward vectors ----------------
    y = torch.arange(40)
    out = {}
    torch.manual_seed(101)
    z = torch.randn(40, cfg["dim_z"])
    G.train()
    with torch.no_grad():
        img = G(z, y)  # draws rdof = randn(40,4) from the same stream
    out["g_train_img"] = img.clone()
    out["g_u0_linear_after"] = G.linear.u0.clone()
    out["g_sv0_linear_after"] = G.linear.sv0.clone()
    out["g_bn_mean_after"] = G.blocks[0][0].bn1.stored_mean.clone()
    out["g_bn_var_after"] = G.blocks[0][0].bn1.stored_var.clone()
    torch.manual_seed(102)
    G.eval()
    with torch.no_grad():
        out["g_eval_img"] = G(z, y).clone()
    G.train()
    torch.manual_seed(103)
    x_real = torch.rand(40, 1, 64, 64) * 2 - 1
    D.train()
    with torch.no_grad():
        p, e, o = D(x_real, y)
    out["x_real"], out["d_proxy"], out["d_embed"], out["d_out"] = x_real, p.clone(), e.clone(), o.clone()
    # attention with a non-zero gamma (gamma is initialised to 0, layers.py:281)
    with torch.no_grad():
        D.blocks[1][2].gamma.fill_(0.7)
        p2, e2, o2 = D(x_real, y)
        D.blocks[1][2].gamma.fill_(0.0)
    out["d_embed_gamma07"], out["d_out_gamma07"] = e2.clone(), o2.clone()
    torch.manual_seed(104)
    xa = diff_aug.DiffAugment(x_real, policy="color,translation,cutout")
    out["diffaug_out"] = xa.clone()
    # non-square DiffAugment (H_base = 3 geometry)
    torch.manual_seed(105)
    x_ns = torch.rand(8, 1, 32, 96) * 2 - 1
    out["x_ns"] = x_ns
    torch.manual_seed(106)
    out["diffaug_ns_out"] = diff_aug.DiffAugment(x_ns, policy="color,translation,cutout").clone()
    # losses on the D outputs
    crit = loss.Conditional_Contrastive_loss("cpu", 40, False)
    torch.manual_seed(107)
    ef = torch.nn.functional.normalize(torch.randn(40, 1024), dim=1)
    out["embed_fake_rand"] = ef
    out["loss_contra"] = crit(e, p, None, y, 1.0, 0).clone()
    out["loss_unif"] = loss.unif_loss(e).clone()
    out["loss_iea"] = loss.IEA_loss(ef, e).clone()
    lr_, lf_ = loss.loss_hinge_dis(o * 3 - 0.5, o * 2 + 0.3)
    out["loss_hinge"] = torch.stack([lr_, lf_, loss.loss_hinge_gen(o)])
    # H_base = 3 generator forward (non-square), checksummed only
    cfg3 = dict(cfg, H_base=3)
    torch.manual_seed(0)
    G3 = model.Generator(**cfg3)
    torch.manual_seed(108)
    z3 = torch.randn(40, cfg["dim_z"])
    with torch.no_grad():
        img3 = G3(z3, y)
    out["g3_img_sub"] = img3[:, :, ::4, ::4].clone()
    out["g3_mean_std"] = torch.stack([img3.mean(dim=[1, 2, 3]), img3.std(dim=[1, 2, 3])])
    save_golden(os.path.join(HERE, "small_fwd"), out)

    # ---------------- one unmodified train step ----------------
    import train_fns
    import utils
    torch.manual_seed(0)
    G = model.Generator(**cfg)
    D = model.Discriminator(**cfg)
    GD = model.G_D(G, D)
    z_, y_ = utils.prepare_z_y(40, cfg["dim_z"], cfg["n_classes"], device="cpu", z_var=cfg["z_var"])
    state = {"itr": 0}
    train = train_fns.GAN_training_function(G, D, GD, z_, y_, None, state, cfg, "cpu")
    G.train(); D.train()
    torch.manual_seed(201)
    x = torch.rand(40, 1, 64, 64) * 2 - 1
    torch.manual_seed(202)
    losses = train(x, y)
    step = {"x": x, "losses": losses}
    step["g_grad_norm"] = {k: float(p.grad.norm()) for k, p in G.named_parameters()}
    step["d_grad_norm"] = {k: float(p.grad.norm()) for k, p in D.named_parameters()}
    keep_g = ["blocks.0.0.conv2.weight", "blocks.7.0.conv3.weight", "linear_f.weight", "shared.weight",
              "blocks.3.0.bn2.gain.weight", "output_layer.2.weight", "RR_G.layers.0.self_attn.qkv_proj.weight",
              "output_layer.0.gain"]
    keep_d = ["input_conv.weight", "blocks.1.2.theta.weight", "blocks.1.2.gamma", "blocks.3.1.conv3.weight",
              "embed.weight", "linear1.weight", "RR_D.layers.0.self_attn.qkv_proj.weight", "norm.weight",
              "blocks.0.0.conv_sc.weight", "linear0.weight"]
    gp, dp = dict(G.named_parameters()), dict(D.named_parameters())
    # full gradients for small tensors, the first 65536 elements (flattened) for large ones
    step["g_grads"] = {k: gp[k].grad.reshape(-1)[:65536].clone() for k in keep_g}
    step["d_grads"] = {k: dp[k].grad.reshape(-1)[:65536].clone() for k in keep_d}
    gs, ds = G.state_dict(), D.state_dict()
    step["g_buffers"] = {k: gs[k].clone() for k in ["linear.u0", "linear.sv0", "blocks.5.0.conv2.u0",
                                                    "blocks.5.0.bn3.stored_mean", "blocks.5.0.bn3.stored_var",
                                                    "output_layer.0.stored_var"]}
    step["d_buffers"] = {k: ds[k].clone() for k in ["input_conv.u0", "input_conv.sv0", "embed.u0", "linear1.sv0"]}
    save_golden(os.path.join(HERE, "small_step"), step)

    # ---------------- shipped-size ctor checksums ----------------
    full = {}
    for hb in (1, 3):
        c = dict(base_config(), H_base=hb)
        torch.manual_seed(0)
        Gf = model.Generator(**c)
        Df = model.Discriminator(**c)
        full["H%d" % hb] = {"G": checksums(Gf.state_dict()), "D": checksums(Df.state_dict()),
                            "G_params": sum(p.numel() for p in Gf.parameters()),
                            "D_params": sum(p.numel() for p in Df.parameters())}
    with open(os.path.join(HERE, "full_checksums.json"), "w") as f:
        json.dump(full, f)
    print("golden vectors written to", HERE)


if __name__ == "__main__":
    main()
