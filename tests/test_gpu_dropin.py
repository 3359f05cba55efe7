"""The drop-in claim, executed: the reference's UNMODIFIED train_fns.GAN_training_function (staged byte for
byte under baseline/_ref by tools/fetch_ref.py) drives the B200 modules of iea_gan_b200/dropin -- with the
reference's own utils.prepare_z_y Distribution tensors, utils.toggle_grad, utils.make_mask, utils.ortho,
torch's clip_grad_norm_, G.optim / D.optim and utils.apply_ema -- and must reproduce the reference's own CPU run
of the same step (the tests/golden/small_step/ golden set) or, for two events, the CPU oracle.

Nothing of the caller is patched: the only hooks are the z_ tensor's sample_() (replaced on the INSTANCE so
the step sees the golden run's CPU draws) and iea_gan_b200.noise.replay for the in-forward draws.
"""
import os
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))


def rel(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return float((a - b).norm() / (b.norm() + 1e-30))


@pytest.fixture(scope="module")
def ref_modules():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import fetch_ref
    if not fetch_ref.present():
        pytest.skip("the reference's unmodified train_fns.py / utils/ are not part of this repository: "
                    "stage them under baseline/_ref with python tools/fetch_ref.py --src <reference checkout>")
    saved_path, saved_mods = list(sys.path), dict(sys.modules)
    fetch_ref.activate(dropin=True)
    import model, train_fns, utils, loss  # noqa: E401
    assert model.__file__.startswith(os.path.join(ROOT, "iea_gan_b200", "dropin"))
    assert loss.__file__.startswith(os.path.join(ROOT, "iea_gan_b200", "dropin"))
    assert train_fns.__file__.startswith(os.path.join(ROOT, "baseline", "_ref"))
    assert utils.__file__.startswith(os.path.join(ROOT, "baseline", "_ref"))
    yield model, train_fns, utils
    sys.path[:] = saved_path
    for k in list(sys.modules):
        if k not in saved_mods:
            del sys.modules[k]


def cpu_draws(cfg, seed, rows, hh, ww):
    """The golden run's CPU random stream of one step, in order: per phase z.normal_, randn rdof, 7 DiffAugment draws."""
    from oracle import iea_oracle as O
    torch.manual_seed(seed)
    phases = []
    for _ in range(2):
        z = torch.empty(rows, cfg["dim_z"]).normal_(0, 1)
        rd = torch.randn(rows, cfg["rdof_dim"])
        d = O.diffaug_draws(rows, hh, ww)
        phases.append((z, rd, d))
    return phases


def replay_list(phases):
    out = []
    for _, rd, d in phases:
        out.append(("randn", rd))
        out += [("rand", d["brightness"]), ("rand", d["saturation"]), ("rand", d["contrast"])]
        out += [("randint", d[k]) for k in ("tx", "ty", "ox", "oy")]
    return out


def build(model, utils, train_fns, cfg, rows, phases, ema=False):
    torch.manual_seed(0)
    G = model.Generator(**cfg).cuda()
    D = model.Discriminator(**cfg).cuda()
    GD = model.G_D(G, D)
    z_, y_ = utils.prepare_z_y(rows, cfg["dim_z"], cfg["n_classes"], device="cuda", z_var=cfg["z_var"])
    it = iter(phases)
    z_.sample_ = lambda: z_.copy_(next(it)[0].cuda())  # the golden run's z draws instead of the CUDA generator's
    e = None
    if ema:
        G_ema = model.Generator(**dict(cfg, skip_init=True, no_optim=True)).cuda()
        e = utils.apply_ema(G, G_ema, cfg["ema_decay"], cfg["ema_start"])
    train = train_fns.GAN_training_function(G, D, GD, z_, y_, e, {"itr": 0}, dict(cfg, ema=ema), "cuda")
    G.train(); D.train()
    return G, D, train


@pytest.mark.parametrize("adt", ["fp32", "bf16"])
def test_unmodified_train_fns_one_event_vs_reference_run(ref_modules, small_cfg, golden_step, adt):
    """Tolerances as tests/test_gpu_discriminator.py::test_train_step_vs_unmodified_train_fns: fp32 activations
    1e-3 on the five floats / 1e-2 on gradient norms; bf16 3e-2 / 0.15."""
    from iea_gan_b200 import noise
    model, train_fns, utils = ref_modules
    os.environ["IEA_ACT_DTYPE"] = adt
    try:
        cfg = dict(small_cfg, device="cuda")
        phases = cpu_draws(cfg, 202, 40, 64, 64)
        G, D, train = build(model, utils, train_fns, cfg, 40, phases, ema=True)
        with noise.replay(replay_list(phases)):
            losses = train(golden_step["x"].cuda(), torch.arange(40, device="cuda"))
        ltol, gtol, ftol = (1e-3, 1e-2, 2e-2) if adt == "fp32" else (3e-2, 0.15, 0.2)
        for k, v in golden_step["losses"].items():
            assert abs(losses[k] - v) < ltol * max(1.0, abs(v)), (k, losses[k], v)
        atol = 1e-6 if adt == "fp32" else 2e-3
        bad = []
        for tag, net, norms in (("G", G, golden_step["g_grad_norm"]), ("D", D, golden_step["d_grad_norm"])):
            for k, p in net.named_parameters():
                got = float(p.grad.norm())
                if abs(got - norms[k]) > gtol * max(norms[k], 1e-6) + atol:
                    bad.append((tag, k, got, norms[k]))
        assert not bad, bad[:10]
        for net, grads in ((G, golden_step["g_grads"]), (D, golden_step["d_grads"])):
            ps = dict(net.named_parameters())
            for k, v in grads.items():
                assert rel(ps[k].grad.reshape(-1)[:65536], v) < ftol, k
        for net, bufs in ((G, golden_step["g_buffers"]), (D, golden_step["d_buffers"])):
            for k, v in bufs.items():
                assert rel(net.state_dict()[k], v) < (1e-4 if adt == "fp32" else 3e-2), k
    finally:
        os.environ.pop("IEA_ACT_DTYPE", None)


def test_unmodified_train_fns_two_events_vs_oracle(ref_modules, small_cfg):
    """batch_size = 80 = two events through the unchanged caller (SURVEY 8(d) multi-event extension): losses,
    gradients and the parameters AFTER both optimizer steps against the CPU oracle's step (fp32 activations)."""
    from iea_gan_b200 import noise
    from oracle import iea_oracle as O
    import iea_gan_b200 as P
    model, train_fns, utils = ref_modules
    os.environ["IEA_ACT_DTYPE"] = "fp32"
    try:
        rows = 80
        cfg = dict(small_cfg, device="cuda", batch_size=rows)
        phases = cpu_draws(cfg, 303, rows, 64, 64)
        G, D, train = build(model, utils, train_fns, cfg, rows, phases)
        torch.manual_seed(0)
        ccfg = dict(cfg, device="cpu")
        sd_g = {k: v.detach().clone() for k, v in P.Generator(**ccfg).state_dict().items()}
        sd_d = {k: v.detach().clone() for k, v in P.Discriminator(**ccfg).state_dict().items()}
        torch.manual_seed(304)
        x = torch.rand(rows, 1, 64, 64) * 2 - 1
        y = torch.arange(40).repeat(2)
        with noise.replay(replay_list(phases)):
            got = train(x.cuda(), y.cuda())
        nz = dict(z_d=phases[0][0], rdof_d=phases[0][1], aug_d=phases[0][2], z_g=phases[1][0], rdof_g=phases[1][1],
                  aug_g=phases[1][2])
        pg, pd = O.param_names(sd_g), O.param_names(sd_d)
        adam = lambda sd, names, lr, b1: torch.optim.Adam([sd[k] for k in names], lr=lr, betas=(b1, cfg["G_B2"]),
                                                          weight_decay=0, eps=cfg["adam_eps"])
        want = O.train_step(sd_g, sd_d, ccfg, x, y, nz, opt_g=adam(sd_g, pg, cfg["G_lr"], cfg["G_B1"]),
                            opt_d=adam(sd_d, pd, cfg["D_lr"], cfg["D_B1"]))
        for k, v in want.items():
            assert abs(got[k] - v) < 1e-3 * max(1.0, abs(v)), (k, got[k], v)
        bad = []
        for tag, net, sd in (("G", G, sd_g), ("D", D, sd_d)):
            for k, p in net.named_parameters():
                r = rel(p.grad, sd[k].grad)
                if r > 2e-2 and float(sd[k].grad.norm()) > 1e-5:
                    bad.append((tag, "grad", k, r))
        assert not bad, bad[:10]
        # both optimizers stepped (FusedAdam here, torch.optim.Adam in the oracle): the UPDATE of the whole net must
        # agree -- Adam moves every weight by ~lr*sign(grad), so elements whose gradient is rounding noise may differ
        torch.manual_seed(0)
        p0g = [p.detach().clone() for p in P.Generator(**ccfg).parameters()]
        p0d = [p.detach().clone() for p in P.Discriminator(**ccfg).parameters()]
        for tag, net, sd, p0 in (("G", G, sd_g, p0g), ("D", D, sd_d, p0d)):
            got_u = torch.cat([(p.detach().cpu() - q).reshape(-1) for p, q in zip(net.parameters(), p0)])
            ref_u = torch.cat([(sd[k].detach() - q).reshape(-1) for (k, _), q in zip(net.named_parameters(), p0)])
            assert float(ref_u.norm()) > 0 and rel(got_u, ref_u) < 5e-2, (tag, rel(got_u, ref_u))
    finally:
        os.environ.pop("IEA_ACT_DTYPE", None)
