"""Every module of the drop-in surface, called STAND-ALONE on the B200, against vectors produced by the real
reference (tests/golden/make_golden_modules.py -> tests/golden/modules/): outputs, input gradients, parameter gradients
and the buffers the call leaves behind (u0 / sv0 / running statistics).

Tolerances: fp32 activations (IEA_ACT_DTYPE=fp32, same arithmetic as the reference in another summation
order) 2e-4 relative L2 on outputs, 2e-3 on gradients; bf16 activations 4e-2 / 1.5e-1 (small tensors, a
handful of ReLU-mask flips are not averaged away).  Buffers 1e-4.
"""
import functools
import os

import pytest
import torch

pytestmark = pytest.mark.gpu
SN = dict(num_svs=1, num_itrs=1, eps=1e-6)


def rel(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return float((a - b).norm() / (b.norm() + 1e-30))


@pytest.fixture(scope="module")
def gold(golden_modules):
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return golden_modules


@pytest.fixture(params=["fp32", "bf16"])
def adt(request):
    os.environ["IEA_ACT_DTYPE"] = request.param
    yield request.param
    os.environ.pop("IEA_ACT_DTYPE", None)


def tols(adt, feature_only=False):
    """(output, gradient) tolerance; feature_only: modules whose arithmetic is fp32 in both modes."""
    return (2e-4, 2e-3) if (adt == "fp32" or feature_only) else (4e-2, 1.5e-1)


def check(m, rec, adt, feature_only=False, n_out=1):
    t_out, t_g = tols(adt, feature_only)
    m.load_state_dict(rec["state"])
    m = m.cuda()
    ins = [t.cuda().requires_grad_(t.is_floating_point()) for t in rec["inputs"]]
    out = m(*ins)
    outs = list(out) if isinstance(out, (tuple, list)) else [out]
    g = torch.Generator().manual_seed(rec["cot_seed"])
    ws = [torch.randn(o.shape, generator=g) for o in rec["outputs"][:n_out]]
    for o, r in zip(outs, rec["outputs"]):
        assert o.shape == r.shape
        assert rel(o, r) < t_out, ("output", rel(o, r))
    sum((o * w.cuda()).sum() for o, w in zip(outs, ws)).backward()
    for t, r in zip(ins, rec["input_grads"]):
        if r is not None:
            assert rel(t.grad, r) < t_g, ("input grad", rel(t.grad, r))
    ps = dict(m.named_parameters())
    scale = max(float(r.norm()) for r in rec["param_grads"].values())
    for k, r in rec["param_grads"].items():
        assert ps[k].grad is not None, k
        if float(r.norm()) < 1e-6 * scale:
            # exactly-zero gradient (a conv bias in front of a batch-norm; the reference's value is rounding noise
            # too): ours must be noise on the scale of the module's gradients
            assert float(ps[k].grad.norm()) < (1e-6 if adt == "fp32" else 1e-3) * scale, (k, float(ps[k].grad.norm()), scale)
            continue
        assert rel(ps[k].grad, r) < t_g, (k, rel(ps[k].grad, r))
    bufs = dict(m.named_buffers())
    for k, r in rec["after"].items():
        assert rel(bufs[k].float(), r.float()) < (1e-4 if (adt == "fp32" or feature_only) else 3e-2), (k, rel(bufs[k], r))
    return m


def test_snconv2d(gold, adt):
    import iea_gan_b200.sn_layers as SL
    check(SL.SNConv2d(16, 32, 3, padding=1, **SN).train(), gold["SNConv2d_3x3"], adt)
    check(SL.SNConv2d(32, 16, 1, padding=0, **SN).eval(), gold["SNConv2d_1x1_eval"], adt)


def test_snlinear_snembedding_w_power_iteration(gold):
    import iea_gan_b200.sn_layers as SL
    check(SL.SNLinear(48, 24, **SN).train(), gold["SNLinear"], "fp32")
    check(SL.SNEmbedding(40, 64, **SN).train(), gold["SNEmbedding"], "fp32")
    rec = gold["SN_W_"]
    m = SL.SNLinear(20, 12, **SN).train()
    m.load_state_dict(rec["state"])
    m = m.cuda()
    w = m.W_()
    assert rel(w, rec["outputs"][0]) < 1e-5
    (w * rec["cot"][0].cuda()).sum().backward()
    assert rel(m.weight.grad, rec["param_grads"]["weight"]) < 1e-4
    assert rel(m.u0, rec["after"]["u0"]) < 1e-5 and rel(m.sv0, rec["after"]["sv0"]) < 1e-5
    p = gold["power_iteration"]
    u = p["u_in"].clone().cuda()
    svs, us, vs = SL.power_iteration(p["W"].cuda(), [u], update=True, eps=1e-6)
    assert rel(svs[0], p["sv"]) < 1e-5 and rel(us[0], p["u"]) < 1e-5 and rel(vs[0], p["v"]) < 1e-5
    assert rel(u, p["u_after"]) < 1e-5


def _ccbn(SL, **kw):
    lin = functools.partial(SL.SNLinear, bias=False, **SN)
    return SL.ccbn(16, which_linear=lin, input_size=32, eps=1e-5, **kw)


def test_ccbn_bn(gold, adt):
    import iea_gan_b200.sn_layers as SL
    check(_ccbn(SL).train(), gold["ccbn_train"], adt)
    check(_ccbn(SL).eval(), gold["ccbn_eval"], adt)
    check(SL.bn(16).train(), gold["bn_train"], adt)


def test_mybn_family(gold, adt):
    """mybn=True (layers.py:547-599): biased running variance, standing statistics, eval division; and the
    functional forms manual_bn / fused_bn."""
    import iea_gan_b200.sn_layers as SL
    t_out, _ = tols(adt)
    check(_ccbn(SL, mybn=True).train(), gold["ccbn_mybn_train"], adt)
    r1, r2, r3 = gold["bn_mybn_standing"]
    m = SL.bn(16, mybn=True).train()
    m.bn.accumulate_standing = True
    m = check(m, r1, adt)
    # second training call accumulates on top of the first; then eval divides by the counter
    for rec, train in ((r2, True), (r3, False)):
        m.train(train)
        x = rec["inputs"][0].cuda()
        with torch.no_grad():
            y = m(x)
        assert rel(y, rec["outputs"][0]) < t_out
        for k, r in rec["after"].items():
            assert rel(dict(m.named_buffers())[k], r) < (1e-4 if adt == "fp32" else 3e-2), k
    r = gold["manual_bn"]
    y, mu, var = SL.manual_bn(r["x"].cuda(), r["gain"].cuda(), r["bias"].cuda(), return_mean_var=True, eps=1e-5)
    assert rel(y, r["y"]) < t_out and rel(mu, r["mean"]) < 1e-3 + t_out and rel(var, r["var"]) < 1e-3 + t_out
    r = gold["fused_bn"]
    y = SL.fused_bn(r["x"].cuda(), r["mean"].cuda(), r["var"].cuda(), r["gain"].cuda(), r["bias"].cuda(), 1e-5)
    assert rel(y, r["y"]) < t_out


def test_attention(gold, adt):
    import iea_gan_b200.sn_layers as SL
    check(SL.Attention(64, functools.partial(SL.SNConv2d, **SN)).train(), gold["Attention"], adt)


def test_dblock(gold, adt):
    import iea_gan_b200.sn_layers as SL
    from iea_gan_b200 import nets
    conv = functools.partial(SL.SNConv2d, kernel_size=3, padding=1, **SN)
    relu = torch.nn.ReLU(inplace=False)
    check(nets.DBlock(32, 64, which_conv=conv, wide=True, activation=relu, preactivation=True,
                      downsample=torch.nn.AvgPool2d(2)).train(), gold["DBlock_down"], adt)
    check(nets.DBlock(64, 64, which_conv=conv, wide=True, activation=relu, preactivation=True,
                      downsample=None).train(), gold["DBlock_same"], adt)


def test_gblock(gold, adt):
    import iea_gan_b200.sn_layers as SL
    from iea_gan_b200 import nets
    conv = functools.partial(SL.SNConv2d, kernel_size=3, padding=1, **SN)
    lin = functools.partial(SL.SNLinear, bias=False, **SN)
    bn = functools.partial(SL.ccbn, which_linear=lin, input_size=32, eps=1e-5)
    relu = torch.nn.ReLU(inplace=False)
    up = functools.partial(torch.nn.functional.interpolate, scale_factor=2)
    check(nets.GBlock(64, 32, which_conv=conv, which_bn=bn, activation=relu, upsample=up).train(), gold["GBlock_up"], adt)
    check(nets.GBlock(64, 64, which_conv=conv, which_bn=bn, activation=relu, upsample=None).train(),
          gold["GBlock_same"], adt)


def test_rrm_mha_sdp(gold):
    import iea_gan_b200.relational as RR
    import iea_gan_b200.sn_layers as SL
    lin = functools.partial(SL.SNLinear, **SN)
    check(RR.RelationalReasoning(num_layers=1, input_dim=128, dim_feedforward=128, which_linear=torch.nn.Linear,
                                 num_heads=2, dropout=0.0, hidden_dim=128).train(), gold["RRM_G"], "fp32", True)
    check(RR.RelationalReasoning(num_layers=1, input_dim=64, dim_feedforward=96, which_linear=lin, num_heads=4,
                                 dropout=0.0, hidden_dim=64).train(), gold["RRM_SN"], "fp32", True)
    m = check(RR.MultiheadAttention(64, 64, 4, lin).train(), gold["MHA"], "fp32", True)
    r = gold["MHA_attention"]
    m.load_state_dict(r["state"])
    with torch.no_grad():
        _, att = m(r["x"].cuda(), return_attention=True)
    assert rel(att, r["att"]) < 2e-4
    r = gold["sdp"]
    q, k, v = [r[n].cuda().requires_grad_(True) for n in "qkv"]
    vals, att = RR.scaled_dot_product(q, k, v)
    assert rel(vals, r["values"]) < 1e-5 and rel(att, r["att"]) < 1e-5
    (vals * r["cot"].cuda()).sum().backward()
    assert rel(q.grad, r["dq"]) < 1e-4 and rel(k.grad, r["dk"]) < 1e-4 and rel(v.grad, r["dv"]) < 1e-4


def test_l2_loss(gold):
    from iea_gan_b200 import losses
    r = gold["l2_loss"]
    a, b = r["a"].cuda().requires_grad_(True), r["b"].cuda().requires_grad_(True)
    l = losses.l2_loss(a, b)
    assert abs(float(l) - float(r["loss"])) < 1e-6
    l.backward()
    assert rel(a.grad, r["da"]) < 1e-6 and rel(b.grad, r["db"]) < 1e-6


def test_module_on_non_current_device(gold):
    """A module living on cuda:1 while cuda:0 is current launches on cuda:1 (needs two GPUs)."""
    if torch.cuda.device_count() < 2:
        pytest.skip("one GPU")
    import iea_gan_b200.sn_layers as SL
    rec = gold["SNLinear"]
    m = SL.SNLinear(48, 24, **SN).train()
    m.load_state_dict(rec["state"])
    m = m.to("cuda:1")
    assert torch.cuda.current_device() == 0
    y = m(rec["inputs"][0].to("cuda:1"))
    assert y.device.index == 1 and rel(y, rec["outputs"][0]) < 2e-4


def test_input_pipeline(gold):
    """iea_event_preprocess (pad + log-norm + dequantisation noise + normalise on the GPU) against the reference's
    transform chain; then the prefetcher end to end (shapes, value range, every batch delivered)."""
    from iea_gan_b200 import pipeline
    d = gold["pipeline"]
    got = pipeline.preprocess_events(d["u8"].cuda(), draws=d["draws"].cuda())
    assert got.shape == d["out"].shape and rel(got, d["out"]) < 1e-6
    clean = pipeline.preprocess_events(d["u8"].cuda(), scale=0)
    assert float((clean[:, :, :3] + 1).abs().max()) == 0.0 and float(clean.max()) <= 1.0
    batches = [((torch.rand(40, 250, 64) ** 8 * 255).to(torch.uint8), torch.arange(40)) for _ in range(3)]
    seen = 0
    for x, y in pipeline.EventPrefetcher(batches, "cuda"):
        assert x.shape == (40, 1, 256, 64) and x.is_cuda and float(x.min()) >= -1.0 and float(x.max()) <= 1.0 + 8e-3
        assert torch.equal(y.cpu(), torch.arange(40))
        seen += 1
    assert seen == 3


def test_rrm_large_batch_tcgen05_linears():
    """64 events (2560 rows >= engine.TC_LINEAR_MIN_ROWS): the RRM's 512-wide linears run as tcgen05 GEMMs (bf16
    operands, fp32 accumulation) -- against the fp32 CPU oracle: output 2e-2, input / weight gradients 5e-2; and the
    same module on 4 events (fp32 CUDA-core path) must agree with the oracle to 2e-4 (the switch is by row count)."""
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import iea_gan_b200.relational as RR
    import iea_gan_b200.sn_layers as SL
    from iea_gan_b200 import engine as E
    from oracle import iea_oracle as O
    lin = functools.partial(SL.SNLinear, **SN)
    torch.manual_seed(3)
    m = RR.RelationalReasoning(num_layers=1, input_dim=512, dim_feedforward=512, which_linear=lin, num_heads=4,
                               dropout=0.0, hidden_dim=512).train()
    for b, t_out, t_g in ((64, 2e-2, 5e-2), (4, 2e-4, 2e-3)):
        assert (40 * b >= E.TC_LINEAR_MIN_ROWS) == (b == 64)
        sd = {"RR." + k: v.detach().clone() for k, v in m.state_dict().items()}
        x = torch.randn(b, 40, 512, generator=torch.Generator().manual_seed(b))
        cot = torch.randn(b, 40, 512, generator=torch.Generator().manual_seed(b + 1))
        names = ["RR.layers.0.self_attn.qkv_proj.weight", "RR.layers.0.linear_net.3.weight", "RR.layers.0.norm1.weight"]
        for k in names:
            sd[k].requires_grad_(True)
        xr = x.clone().requires_grad_(True)
        ref = O.rrm_forward(sd, O._Weights(sd, True, 1e-6), "RR", xr, 4)
        (ref * cot).sum().backward()
        mg = RR.RelationalReasoning(num_layers=1, input_dim=512, dim_feedforward=512, which_linear=lin, num_heads=4,
                                    dropout=0.0, hidden_dim=512).train()
        mg.load_state_dict(m.state_dict())
        mg = mg.cuda()
        xg = x.cuda().requires_grad_(True)
        out = mg(xg)
        assert rel(out, ref) < t_out, (b, rel(out, ref))
        (out * cot.cuda()).sum().backward()
        assert rel(xg.grad, xr.grad) < t_g, (b, rel(xg.grad, xr.grad))
        ps = dict(mg.named_parameters())
        for k in names:
            assert rel(ps[k[3:]].grad, sd[k].grad) < t_g, (b, k, rel(ps[k[3:]].grad, sd[k].grad))
