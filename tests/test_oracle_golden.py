"""The oracle (oracle/iea_oracle.py) against the golden vectors produced by the REAL
reference (tests/golden/make_golden.py).  CPU only.  Tolerances: the oracle and the
reference run the same fp32 torch kernels in a slightly different association order,
so outputs agree to ~1e-5 relative; gradients to 1e-4 relative L2."""
import json
import os

import pytest
import torch

import iea_gan_b200 as P
from oracle import iea_oracle as O

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")


def rel(a, b):
    return float((a.double() - b.double()).norm() / (b.double().norm() + 1e-30))


def fresh(cfg, seed=0):
    torch.manual_seed(seed)
    G = P.Generator(**cfg)
    D = P.Discriminator(**cfg)
    sg = {k: v.detach().clone() for k, v in G.state_dict().items()}
    sd = {k: v.detach().clone() for k, v in D.state_dict().items()}
    return sg, sd


def checksum_close(got, want, abs_sum):
    """Constructor checksums.  Initialisers that go through the host's BLAS / LAPACK (the QR of the orthogonal init)
    round differently with the CPU's vector unit and thread count: a tensor's sum moves by up to ~4e-8 of its
    abs-sum between hosts.  A different draw order or initialiser moves it by ~abs-sum / sqrt(numel) or more."""
    return abs(got - want) < 1e-9 + 1e-6 * abs_sum


def test_ctor_matches_reference_checksums(small_cfg):
    with open(os.path.join(GOLDEN, "state_checksums.json")) as f:
        ref = json.load(f)
    sg, sd = fresh(small_cfg)
    for name, s in (("G", sg), ("D", sd)):
        assert list(s.keys()) == list(ref[name].keys())
        for k, v in s.items():
            assert list(v.shape) == ref[name][k][2], k
            assert checksum_close(float(v.double().sum()), ref[name][k][0], ref[name][k][1]), k
            assert checksum_close(float(v.double().abs().sum()), ref[name][k][1], ref[name][k][1]), k


@pytest.mark.parametrize("hb", [1, 3])
def test_full_size_ctor_checksums(hb):
    with open(os.path.join(GOLDEN, "full_checksums.json")) as f:
        ref = json.load(f)["H%d" % hb]
    with open(os.path.join(GOLDEN, "small_cfg.json")) as f:
        cfg = json.load(f)
    cfg.update(resolution=256, G_ch=32, D_ch=32, H_base=hb, D_attn="32")
    torch.manual_seed(0)
    G = P.Generator(**cfg)
    D = P.Discriminator(**cfg)
    assert sum(p.numel() for p in G.parameters()) == ref["G_params"]
    assert sum(p.numel() for p in D.parameters()) == ref["D_params"]
    for name, net in (("G", G), ("D", D)):
        s = net.state_dict()
        assert list(s.keys()) == list(ref[name].keys())
        for k, v in s.items():
            assert checksum_close(float(v.double().sum()), ref[name][k][0], ref[name][k][1]), k


def test_generator_forward(small_cfg, golden_fwd):
    sg, _ = fresh(small_cfg)
    y = torch.arange(40)
    torch.manual_seed(101)
    z = torch.randn(40, small_cfg["dim_z"])
    rdof = torch.randn(40, small_cfg["rdof_dim"])
    with torch.no_grad():
        img = O.generator_forward(sg, small_cfg, z, y, rdof, training=True)
    assert rel(img, golden_fwd["g_train_img"]) < 2e-5
    assert rel(sg["linear.u0"], golden_fwd["g_u0_linear_after"]) < 1e-6
    assert rel(sg["linear.sv0"], golden_fwd["g_sv0_linear_after"]) < 1e-6
    assert rel(sg["blocks.0.0.bn1.stored_mean"], golden_fwd["g_bn_mean_after"]) < 1e-5
    assert rel(sg["blocks.0.0.bn1.stored_var"], golden_fwd["g_bn_var_after"]) < 1e-5
    torch.manual_seed(102)
    rdof = torch.randn(40, small_cfg["rdof_dim"])
    before = {k: v.clone() for k, v in sg.items()}
    with torch.no_grad():
        img = O.generator_forward(sg, small_cfg, z, y, rdof, training=False)
    assert rel(img, golden_fwd["g_eval_img"]) < 2e-5
    assert all(torch.equal(before[k], sg[k]) for k in sg), "eval mode must not write buffers"


def test_generator_forward_hbase3(small_cfg, golden_fwd):
    cfg = dict(small_cfg, H_base=3)
    sg, _ = fresh(cfg)
    torch.manual_seed(108)
    z = torch.randn(40, cfg["dim_z"])
    rdof = torch.randn(40, cfg["rdof_dim"])
    with torch.no_grad():
        img = O.generator_forward(sg, cfg, z, torch.arange(40), rdof, training=True)
    assert img.shape == (40, 1, 64, 192)
    assert rel(img[:, :, ::4, ::4], golden_fwd["g3_img_sub"]) < 2e-5


def test_discriminator_forward(small_cfg, golden_fwd):
    _, sd = fresh(small_cfg)
    y = torch.arange(40)
    with torch.no_grad():
        p, e, o = O.discriminator_forward(sd, small_cfg, golden_fwd["x_real"], y, training=True)
        assert rel(p, golden_fwd["d_proxy"]) < 1e-5
        assert rel(e, golden_fwd["d_embed"]) < 1e-4
        assert rel(o, golden_fwd["d_out"]) < 1e-4
        sd["blocks.1.2.gamma"].fill_(0.7)
        p, e, o = O.discriminator_forward(sd, small_cfg, golden_fwd["x_real"], y, training=True)
        assert rel(e, golden_fwd["d_embed_gamma07"]) < 1e-4
        assert rel(o, golden_fwd["d_out_gamma07"]) < 1e-4


def test_diffaugment(golden_fwd):
    torch.manual_seed(104)
    d = O.diffaug_draws(40, 64, 64)
    assert rel(O.diffaugment(golden_fwd["x_real"], d), golden_fwd["diffaug_out"]) < 1e-6
    torch.manual_seed(106)
    d = O.diffaug_draws(8, 32, 96)
    assert rel(O.diffaugment(golden_fwd["x_ns"], d), golden_fwd["diffaug_ns_out"]) < 1e-6


def test_losses(golden_fwd):
    e, p, o, ef = (golden_fwd[k] for k in ("d_embed", "d_proxy", "d_out", "embed_fake_rand"))
    assert abs(float(O.contrastive(e, p)) - float(golden_fwd["loss_contra"])) < 1e-5
    assert abs(float(O.uniformity(e)) - float(golden_fwd["loss_unif"])) < 1e-5
    assert abs(float(O.iea(ef, e)) - float(golden_fwd["loss_iea"])) < 1e-6
    lr_, lf_ = O.hinge_dis(o * 3 - 0.5, o * 2 + 0.3)
    got = torch.stack([lr_, lf_, O.hinge_gen(o)])
    assert torch.allclose(got, golden_fwd["loss_hinge"], atol=1e-6)


def test_train_step_matches_unmodified_train_fns(small_cfg, golden_step):
    """One D step + one G step: the 5 floats train_fns.train returns, every parameter's
    gradient norm, selected full gradients and the buffers after the step."""
    cfg = small_cfg
    sg, sd = fresh(cfg)
    y = torch.arange(40)
    torch.manual_seed(0)  # consume what prepare_z_y consumed in the reference run: nothing seeded after
    torch.manual_seed(202)
    noise = {}
    for ph in ("d", "g"):
        noise["z_" + ph] = torch.empty(40, cfg["dim_z"]).normal_(0, 1)
        noise["rdof_" + ph] = torch.randn(40, cfg["rdof_dim"])
        noise["aug_" + ph] = O.diffaug_draws(40, 64, 64)
    mk = lambda s, lr, b1, b2: torch.optim.Adam([s[k] for k in O.param_names(s)], lr=lr, betas=(b1, b2),
                                                weight_decay=0, eps=cfg["adam_eps"])
    opt_g, opt_d = mk(sg, cfg["G_lr"], cfg["G_B1"], cfg["G_B2"]), mk(sd, cfg["D_lr"], cfg["D_B1"], cfg["D_B2"])
    losses = O.train_step(sg, sd, cfg, golden_step["x"], y, noise, opt_g, opt_d)
    for k, v in golden_step["losses"].items():
        assert abs(losses[k] - v) < 2e-4 * max(1.0, abs(v)), (k, losses[k], v)
    for tag, s, norms, grads in (("G", sg, golden_step["g_grad_norm"], golden_step["g_grads"]),
                                 ("D", sd, golden_step["d_grad_norm"], golden_step["d_grads"])):
        for k, v in norms.items():
            got = float(s[k].grad.norm())
            assert abs(got - v) < 2e-3 * max(v, 1e-6) + 1e-7, (tag, k, got, v)
        for k, v in grads.items():
            assert rel(s[k].grad.reshape(-1)[:65536], v) < 1e-3, (tag, k)
    for k, v in golden_step["g_buffers"].items():
        assert rel(sg[k], v) < 1e-4, k
    for k, v in golden_step["d_buffers"].items():
        assert rel(sd[k], v) < 1e-4, k


def test_input_pipeline_matches_reference_transforms(golden_modules):
    """oracle.preprocess_events against the reference's own transform chain (utils/dataloader.py:69-77) run on
    synthetic decoded images by tests/golden/make_golden_modules.py."""
    d = golden_modules["pipeline"]
    got = O.preprocess_events(d["u8"], d["draws"])
    assert got.shape == d["out"].shape == (6, 1, 256, 48)
    assert float((got - d["out"]).abs().max()) < 1e-6
