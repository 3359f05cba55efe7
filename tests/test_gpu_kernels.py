"""GPU parity tests of the individual kernels against plain torch fp32 (through the C ABI).
Tolerances: fp32 kernels 1e-4 relative L2 (different summation order); bf16 storage 1.5e-2."""
import ctypes as C
import math
import os

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu


def rel(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return float((a - b).norm() / (b.norm() + 1e-30))


@pytest.fixture(scope="module")
def eng():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from iea_gan_b200 import engine, _lib
    _lib.lib()
    torch.backends.cudnn.allow_tf32 = False   # the torch reference must be real fp32
    torch.backends.cuda.matmul.allow_tf32 = False
    return engine


class _Mod(torch.nn.Module):
    pass


def make_sn_conv(cin, cout, k, dev, bias=True):
    from iea_gan_b200 import sn_layers as SL
    m = SL.SNConv2d(cin, cout, k, padding=k // 2, bias=bias, eps=1e-6).to(dev)
    return m


@pytest.mark.parametrize("cin,cout,k", [(16, 32, 3), (64, 16, 1), (1, 32, 3), (32, 1, 3), (12, 20, 3)])
def test_sn_power_iter_and_pack(eng, cin, cout, k):
    dev = "cuda"
    torch.manual_seed(1)
    m = make_sn_conv(cin, cout, k, dev)
    grp = eng.SNGroup()
    l = grp.add(m, torch.float32)
    W = m.weight.detach().reshape(cout, -1).clone()
    u0 = m.u0.clone()
    v = F.normalize(u0 @ W, eps=1e-6)
    un = F.normalize(v @ W.t(), eps=1e-6)
    sig = float(((v @ W.t()) @ un.t()).squeeze())
    m.train()
    grp.run(True, True)
    torch.cuda.synchronize()
    assert rel(l.v(), v.view(-1)) < 1e-5
    assert rel(m.u0, un) < 1e-5
    assert abs(float(m.sv0) - sig) < 1e-4 * abs(sig)
    assert abs(float(l.inv_sigma()) - 1 / sig) < 1e-4 / abs(sig)
    wp = m.weight.detach().permute(0, 2, 3, 1).reshape(cout, k * k, cin)
    assert torch.equal(l.wp, wp)
    wd = m.weight.detach().flip(2, 3).permute(1, 2, 3, 0).reshape(cin, k * k, cout)
    assert torch.equal(l.wd, wd)
    # eval mode: nothing is written
    m.eval()
    ub, sb = m.u0.clone(), m.sv0.clone()
    grp.run(False, False)
    torch.cuda.synchronize()
    assert torch.equal(ub, m.u0) and torch.equal(sb, m.sv0)


def _ref_T(x, scale, shift, relu, mode):
    if scale is not None:
        x = x * scale[:, :, None, None] + shift[:, :, None, None]
    if relu:
        x = F.relu(x)
    if mode == 1:
        x = F.interpolate(x, scale_factor=2)
    elif mode == 2:
        x = F.avg_pool2d(x, 2)
    return x


@pytest.mark.parametrize("adt", ["fp32", "bf16"])
@pytest.mark.parametrize("cin,cout,k,mode,relu,aff,resm", [
    (16, 32, 3, 0, True, True, None), (64, 16, 1, 1, True, True, 1), (32, 48, 3, 2, True, False, 2),
    (1, 32, 3, 0, False, False, None), (32, 1, 3, 0, True, True, None), (20, 12, 1, 0, False, False, 0)])
def test_conv_fprop_and_backward(eng, adt, cin, cout, k, mode, relu, aff, resm):
    """Fused conv forward + every backward product against torch autograd."""
    from iea_gan_b200 import _lib as L
    os.environ["IEA_ACT_DTYPE"] = adt
    os.environ["IEA_CONV_IMPL"] = "generic"
    try:
        dev = "cuda"
        at = eng.act_dtype()
        torch.manual_seed(2)
        n, h, w = 40, 8, 12
        hs, ws = (h // 2, w // 2) if mode == 1 else ((2 * h, 2 * w) if mode == 2 else (h, w))
        m = make_sn_conv(cin, cout, k, dev)
        m.train()
        x = torch.randn(n, cin, hs, ws, device=dev)
        xq = x.to(at).float()  # what the kernel sees
        scale = (torch.rand(n, cin, device=dev) + 0.5) if aff else None
        shift = torch.randn(n, cin, device=dev) * 0.3 if aff else None
        rc = None
        if resm is not None:
            rc = cout if resm != 2 else cout
            rh, rw = (h // 2, w // 2) if resm == 1 else ((2 * h, 2 * w) if resm == 2 else (h, w))
            r = torch.randn(n, cout + 4, rh, rw, device=dev)
            rq = r.to(at).float()
        # --- torch reference with autograd
        Wt = m.weight.detach().clone().requires_grad_(True)
        bt = m.bias.detach().clone().requires_grad_(True)
        W2 = Wt.reshape(cout, -1)
        u0 = m.u0.clone()
        with torch.no_grad():
            v = F.normalize(u0 @ W2, eps=1e-6)
            un = F.normalize(v @ W2.t(), eps=1e-6)
        sig = ((v @ W2.t()) @ un.t()).squeeze()
        xr = xq.clone().requires_grad_(True)
        sr = scale.clone().requires_grad_(True) if aff else None
        hr = shift.clone().requires_grad_(True) if aff else None
        a = _ref_T(xr, sr, hr, relu, mode)
        Wq = Wt.detach().to(at).float()  # value the kernel multiplies with; gradient flows to Wt
        yref = F.conv2d(a, (Wq + (Wt - Wt.detach())) / sig, bt, padding=k // 2)
        if resm is not None:
            rr = rq.clone().requires_grad_(True)
            yref = yref + _ref_T(rr[:, :cout], None, None, False, resm)
        # --- kernel
        grp = eng.SNGroup()
        l = grp.add(m, at)
        grp.run(True, True)
        tape = eng.Tape(True)
        xv = eng.Var(x.permute(0, 2, 3, 1).contiguous().to(at))
        ss = eng.ScaleShift(scale.contiguous(), shift.contiguous()) if aff else None
        resv = None
        if resm is not None:
            resv = eng.Var(r.permute(0, 2, 3, 1).contiguous().to(at))
        yv = eng.conv(tape, xv, l, n, h, w, k, bias=m.bias, in_mode=mode, in_relu=relu, ss=ss, res=resv,
                      res_mode=resm or 0, res_c=cout if resm is not None else 0, stats=True, out_dtype=torch.float32)
        y = yv.t.permute(0, 3, 1, 2)
        tol = 2e-5 if adt == "fp32" else 1.5e-2
        assert rel(y, yref) < tol
        # epilogue statistics
        st = yv.t.reshape(-1, cout)
        part = yv.bn
        # backward
        gy = torch.randn_like(yref)
        yref.backward(gy)
        yv.g = gy.permute(0, 2, 3, 1).contiguous()
        tape.backward()
        torch.cuda.synchronize()
        btol = 1e-4 if adt == "fp32" else 2.5e-2
        assert rel(xv.g.float().permute(0, 3, 1, 2), xr.grad) < btol
        assert rel(tape.pgrads[id(m.weight)], Wt.grad) < btol
        assert rel(tape.pgrads[id(m.bias)], bt.grad) < btol
        if aff:
            assert rel(ss.dscale, sr.grad) < btol
            assert rel(ss.dshift, hr.grad) < btol
        if resm is not None:
            assert rel(resv.g.float().permute(0, 3, 1, 2), rr.grad) < btol
    finally:
        os.environ.pop("IEA_ACT_DTYPE", None)
        os.environ.pop("IEA_CONV_IMPL", None)


def test_conv_epilogue_stats(eng):
    os.environ["IEA_ACT_DTYPE"] = "fp32"
    try:
        dev = "cuda"
        torch.manual_seed(3)
        n, h, w, cin, cout = 80, 8, 8, 16, 24
        m = make_sn_conv(cin, cout, 3, dev)
        grp = eng.SNGroup()
        l = grp.add(m, torch.float32)
        grp.run(True, False)
        x = torch.randn(n, h, w, cin, device=dev)
        yv = eng.conv(eng.Tape(False), eng.Var(x), l, n, h, w, 3, bias=m.bias, stats=True, out_dtype=torch.float32)
        part, tiles, count = yv.bn
        assert count == 40 * h * w and tiles == count // 128
        y = yv.t.reshape(2, -1, cout)
        s = part.reshape(2, tiles, cout, 2).sum(1)
        assert rel(s[..., 0], y.sum(1)) < 1e-5
        assert rel(s[..., 1], (y * y).sum(1)) < 1e-5
    finally:
        os.environ.pop("IEA_ACT_DTYPE", None)


def test_layernorm_mha_l2norm(eng):
    dev = "cuda"
    torch.manual_seed(4)
    ln = torch.nn.LayerNorm(128).to(dev)
    with torch.no_grad():
        ln.weight.uniform_(0.5, 1.5)
        ln.bias.normal_()
    x = torch.randn(80, 128, device=dev)
    xr = x.clone().requires_grad_(True)
    yr = ln(xr)
    tape = eng.Tape(True)
    xv = eng.Var(x)
    yv = eng.layernorm(tape, xv, ln)
    assert rel(yv.t, yr) < 1e-5
    g = torch.randn_like(yr)
    yr.backward(g)
    yv.g = g
    tape.backward()
    assert rel(xv.g, xr.grad) < 1e-4
    assert rel(tape.pgrads[id(ln.weight)], ln.weight.grad) < 1e-4
    assert rel(tape.pgrads[id(ln.bias)], ln.bias.grad) < 1e-4
    # per-head interleaved attention (RRM.py:49-53)
    for heads, d in ((2, 64), (4, 128)):
        E = 2
        qkv = torch.randn(E * 40, heads * 3 * d, device=dev)
        qr = qkv.clone().requires_grad_(True)
        t = qr.reshape(E, 40, heads, 3 * d).permute(0, 2, 1, 3)
        q, k, v = t.chunk(3, dim=-1)
        att = F.softmax(q @ k.transpose(-2, -1) / math.sqrt(d), dim=-1)
        val = (att @ v).permute(0, 2, 1, 3).reshape(E * 40, heads * d)
        tape = eng.Tape(True)
        qv = eng.Var(qkv)
        vv, att_k = eng.mha_core(tape, qv, E, 40, heads, d)
        assert rel(vv.t, val) < 1e-5
        assert rel(att_k, att) < 1e-5
        g = torch.randn_like(val)
        val.backward(g)
        vv.g = g
        tape.backward()
        assert rel(qv.g, qr.grad) < 1e-4


@pytest.mark.parametrize("cin,cout,k,mode,relu,aff,resm,hw", [
    (16, 16, 3, 0, True, True, None, (16, 16)), (16, 32, 1, 0, True, True, 0, (16, 16)),
    (32, 32, 3, 1, True, True, 1, (16, 16)), (64, 16, 1, 0, True, True, None, (8, 8)),
    (64, 64, 3, 2, True, False, 2, (8, 8)), (128, 128, 3, 0, True, True, None, (4, 4)),
    (512, 128, 1, 0, True, True, None, (4, 4)), (128, 512, 1, 0, False, False, 0, (4, 4)),
    (32, 64, 1, 0, False, False, None, (12, 20)), (256, 32, 1, 0, True, False, None, (8, 8)),
    (16, 16, 3, 1, True, True, None, (32, 24)), (64, 64, 3, 0, True, True, 0, (16, 8)),
    (32, 32, 3, 0, False, False, None, (48, 16)), (64, 256, 1, 2, True, False, 2, (8, 16)),
    (128, 32, 1, 0, True, True, None, (16, 16)), (16, 64, 1, 0, True, True, 1, (16, 16))])
@pytest.mark.parametrize("variant", ["resident", "stream"])
def test_conv_tcgen05_matches_generic(eng, variant, cin, cout, k, mode, relu, aff, resm, hw):
    _tc_vs_generic(eng, variant, cin, cout, k, mode, relu, aff, resm, hw, 40)


@pytest.mark.parametrize("cin,cout,k,mode,relu,aff,resm,hw,n", [
    (16, 16, 3, 0, True, True, None, (32, 64), 80),   # 4-wide macro tiles, interior + border patches, 2 events
    (16, 16, 3, 1, True, True, 1, (32, 32), 80),      # nearest-up2 input folded into the chunk offsets
    (16, 32, 1, 0, True, True, 1, (32, 32), 80),      # 1x1, up2 residual (GBlock conv4 + shortcut)
    (16, 32, 1, 0, False, False, 2, (16, 16), 40),    # pooled residual
    (32, 16, 3, 0, True, False, None, (16, 32), 40),  # 2-wide macro tiles
    (32, 32, 3, 0, True, True, 0, (32, 16), 80),
    (64, 32, 3, 0, True, True, None, (16, 16), 40),   # single-tile patches, 8 planes
    (64, 16, 1, 0, True, True, None, (16, 24), 40),   # 1x1 whose images are 3 tiles (macro width falls to 1)
    (32, 32, 1, 0, False, False, None, (12, 20), 40)])  # ragged tail: 9600 pixels = 37.5 macro tiles
@pytest.mark.parametrize("producer", ["tma", "cp.async"])
def test_conv_thin_macro_tiles(eng, producer, cin, cout, k, mode, relu, aff, resm, hw, n):
    """conv_thin.cu (macro-tile tcgen05 kernel for Cin <= 64, Cout 16/32) against the CUDA-core kernel, with
    the TMA box-load producer (same-resolution inputs, Cout 16) and with the cp.async slot-table producer."""
    os.environ["IEA_THIN_TMA"] = "1" if producer == "tma" else "0"
    try:
        _tc_vs_generic(eng, "resident", cin, cout, k, mode, relu, aff, resm, hw, n)
    finally:
        os.environ.pop("IEA_THIN_TMA", None)


def _tc_vs_generic(eng, variant, cin, cout, k, mode, relu, aff, resm, hw, n):
    """The tcgen05/TMEM implicit-GEMM path against the CUDA-core path on the same descriptor: same
    bf16 inputs and weights, fp32 accumulation in both, so they agree to bf16 output rounding
    (<= 1 ulp of bf16 = 2^-8 relative per element; 6e-3 relative L2 bound) -- forward, statistics
    and every backward product that runs through the kernel (data gradient)."""
    os.environ["IEA_ACT_DTYPE"] = "bf16"
    tc_impl = "stream" if variant == "stream" else "tcgen05"  # stream: conv_tc_kernel wherever it takes the shape
    try:
        dev = "cuda"
        torch.manual_seed(5)
        h, w = hw
        hs, ws = (h // 2, w // 2) if mode == 1 else ((2 * h, 2 * w) if mode == 2 else (h, w))
        m = make_sn_conv(cin, cout, k, dev)
        m.train()
        grp = eng.SNGroup()
        l = grp.add(m, torch.bfloat16)
        grp.run(True, True)
        assert l.wp_tc is not None
        x = torch.randn(n, hs, ws, cin, device=dev).bfloat16()
        scale = (torch.rand(n, cin, device=dev) + 0.5) if aff else None
        shift = (torch.randn(n, cin, device=dev) * 0.3) if aff else None
        res = None
        if resm is not None:
            rh, rw = (h // 2, w // 2) if resm == 1 else ((2 * h, 2 * w) if resm == 2 else (h, w))
            res = torch.randn(n, rh, rw, cout + 16, device=dev).bfloat16()
        outs = {}
        for impl in ("generic", tc_impl):
            os.environ["IEA_CONV_IMPL"] = impl
            tape = eng.Tape(True)
            xv = eng.Var(x)
            ss = eng.ScaleShift(scale, shift) if aff else None
            rv = eng.Var(res) if res is not None else None
            yv = eng.conv(tape, xv, l, n, h, w, k, bias=m.bias, in_mode=mode, in_relu=relu, ss=ss, res=rv,
                          res_mode=resm or 0, res_c=cout if resm is not None else 0, stats=True)
            torch.manual_seed(6)
            yv.g = torch.randn(n, h, w, cout, device=dev).bfloat16()
            m.bias.requires_grad_(False)
            tape.backward()
            torch.cuda.synchronize()
            # statistics: compare per-event totals (the two kernels tile the image differently)
            st = yv.bn[0].reshape(n // 40, yv.bn[1], cout, 2).sum(1) if yv.bn else None
            outs[impl] = (yv.t.float(), st, xv.g.float(), tape.pgrads[id(m.weight)].clone())
        a, b = outs["generic"], outs[tc_impl]
        assert rel(b[0], a[0]) < 6e-3
        if a[1] is not None:
            assert rel(b[1], a[1]) < 6e-3
        assert rel(b[2], a[2]) < 1e-2
        assert rel(b[3], a[3]) < 1e-2  # weight gradient: mma.sync split-K kernel vs CUDA-core kernel
    finally:
        os.environ.pop("IEA_ACT_DTYPE", None)
        os.environ.pop("IEA_CONV_IMPL", None)


@pytest.mark.parametrize("cin,cout,k,hw,gdt", [(1, 32, 3, (32, 32), "bf16"), (32, 1, 3, (32, 32), "fp32"),
                                              (128, 32, 1, (16, 16), "bf16"), (64, 128, 1, (16, 16), "bf16"),
                                              (128, 128, 3, (16, 16), "bf16"), (512, 128, 1, (8, 8), "bf16"),
                                              (128, 512, 1, (8, 8), "bf16"), (256, 64, 1, (16, 16), "bf16"),
                                              (128, 128, 3, (8, 8), "bf16"), (128, 128, 3, (4, 4), "bf16"),
                                              (32, 16, 3, (12, 20), "bf16"),
                                              # macro-tile kernel (Cin, Cout in {16, 32}; 4- and 2-wide macro tiles)
                                              (16, 16, 3, (32, 64), "bf16"), (32, 32, 3, (16, 32), "bf16"),
                                              (16, 32, 3, (32, 16), "bf16"), (32, 16, 3, (16, 16), "bf16"),
                                              # ... and its 1x1 form (pixel runs of 128*mt inside an image)
                                              (32, 16, 1, (32, 32), "bf16"), (64, 32, 1, (16, 16), "bf16"),
                                              (16, 64, 1, (16, 32), "bf16"), (16, 16, 1, (32, 32), "bf16")])
def test_wgrad_mma_thin_and_wide(eng, cin, cout, k, hw, gdt):
    """The 1-channel stem / output convs (zero-extended operands) and the many-block 1x1 shapes of the
    tensor-core weight-gradient kernel against the CUDA-core kernel."""
    from iea_gan_b200 import _lib as L
    import ctypes as C
    dev = "cuda"
    torch.manual_seed(9)
    n, (h, w) = 40, hw
    x = torch.randn(n, h, w, cin, device=dev)
    x = x if cin == 1 else x.bfloat16()
    g = torch.randn(n, h, w, cout, device=dev)
    g = g if gdt == "fp32" else g.bfloat16()
    wp = torch.zeros(cout, k * k, cin, device=dev)
    y = torch.empty(n, h, w, cout, device=dev, dtype=torch.bfloat16)
    d = eng._desc(n, h, w, cin, cout, k, x, x.data_ptr(), cin, 0, False, None, None, wp, None, 0, None, None, 0, 0,
                  -1, y, y.data_ptr(), cout, 0, None)
    slices = L.call("iea_conv_wgrad_mma_slices", C.byref(d), L.dt(g), cout)
    assert slices > 0
    gp = torch.empty(slices, cout, k * k * cin, device=dev)
    db = torch.full((cout,), float("nan"), device=dev)
    fused = L.call("iea_conv_wgrad_mma", C.byref(d), g.data_ptr(), L.dt(g), cout, gp.data_ptr(), db.data_ptr(), L.stream())
    ref = torch.empty(8, cout, k * k * cin, device=dev)
    L.call("iea_conv_wgrad", C.byref(d), g.data_ptr(), L.dt(g), cout, ref.data_ptr(), 8, L.stream())
    torch.cuda.synchronize()
    assert rel(gp[0], ref.sum(0)) < 5e-3  # slice 0 = fixed-order sum of the per-CTA partials
    if fused:  # bias gradient from the same pass (ones-column MMA on the g fragments)
        assert rel(db, g.float().reshape(-1, cout).sum(0)) < 2e-3


@pytest.mark.parametrize("n,hw,hwk", [(40, 1024, 256), (6, 3072, 768), (3, 128, 128)])
def test_attention_tcgen05_vs_torch(eng, n, hw, hwk):
    """BigGAN attention core (layers.py:289-299) on the tcgen05 kernels (attn_tc.cu) at the shipped
    channel counts (ck 32, cv 128): forward, lse and the three input gradients against torch fp32 on the
    same bf16 inputs, and against the CUDA-core kernels.  Tolerance: P and dS are rounded to bf16
    before their second GEMM (2^-9 relative per element) and the outputs are bf16."""
    dev = "cuda"
    ck, cv = 32, 128
    torch.manual_seed(11)
    th = (torch.randn(n, hw, ck, device=dev) * 0.7).bfloat16()
    ph = (torch.randn(n, hwk, ck, device=dev) * 0.7).bfloat16()
    gv = torch.randn(n, hwk, cv, device=dev).bfloat16()
    go = torch.randn(n, hw, cv, device=dev).bfloat16()
    tr, pr, gr = (t.float().requires_grad_(True) for t in (th, ph, gv))
    beta = F.softmax(tr @ pr.transpose(1, 2), dim=-1)
    o_ref = beta @ gr
    o_ref.backward(go.float())
    lse_ref = torch.logsumexp(tr.detach() @ pr.detach().transpose(1, 2), dim=-1)
    outs = {}
    try:
        for impl in ("tcgen05", "generic"):
            os.environ["IEA_ATTN_IMPL"] = impl
            tape = eng.Tape(True)
            tv, pv, gvv = eng.Var(th), eng.Var(ph), eng.Var(gv)
            ov = eng.attn_core(tape, tv, pv, gvv, n, hw, hwk, ck, cv)
            ov.g = go
            tape.backward()
            torch.cuda.synchronize()
            outs[impl] = (ov.t.float(), tv.g.float(), pv.g.float(), gvv.g.float())
    finally:
        os.environ.pop("IEA_ATTN_IMPL", None)
    refs = (o_ref, tr.grad, pr.grad, gr.grad)
    for name, got, ref, gen in zip(("o", "dtheta", "dphi", "dg"), outs["tcgen05"], refs, outs["generic"]):
        assert rel(got, ref) < 1.5e-2, name
        assert rel(got, gen) < 1.5e-2, name


@pytest.mark.parametrize("rows,cin,cout,xdt,aff,relu,res", [
    (320, 12096, 256, "fp32", True, False, False),   # grouped ccbn data gradient: cluster of 8 over K
    (80, 256, 8192, "fp32", False, False, False),    # G.linear forward: one K slice, many column tiles
    (120, 1536, 512, "bf16", False, True, True),     # ragged rows, bf16 input, fused ReLU + residual
    (40, 516, 260, "fp32", True, True, False)])      # K and N tails
def test_skinny_linear_cluster_splitk(eng, rows, cin, cout, xdt, aff, relu, res):
    """linear_skinny.cu (64x64 tiles, split-K over a thread-block cluster reduced through distributed
    shared memory) against torch fp32: y = relu?(x*s+t) W^T / sigma + b (+ residual)."""
    from iea_gan_b200 import _lib as L
    dev = "cuda"
    torch.manual_seed(13)
    x = torch.randn(rows, cin, device=dev)
    x = x.bfloat16() if xdt == "bf16" else x
    w = torch.randn(cout, cin, device=dev) * 0.05
    b = torch.randn(cout, device=dev)
    osc = torch.tensor([0.7], device=dev)
    sc = torch.rand(cin, device=dev) + 0.5 if aff else None
    sh = torch.randn(cin, device=dev) if aff else None
    r = torch.randn(rows, cout, device=dev) if res else None
    y = torch.empty(rows, cout, device=dev)
    d = eng._desc(rows, 1, 1, cin, cout, 1, x, x.data_ptr(), cin, 0, relu, sc, sh, w, osc, 0, b,
                  eng.Var(r) if res else None, 0, cout if res else 0, -1, y, y.data_ptr(), cout, 0, None, in_bcast=1 if aff else 0)
    L.call("iea_conv_fprop", C.byref(d), L.stream())
    t = x.float()
    if aff:
        t = t * sc + sh
    if relu:
        t = t.relu()
    ref = (t.double() @ w.double().t()).float() * 0.7 + b
    if res:
        ref = ref + r
    torch.cuda.synchronize()
    assert rel(y, ref) < 2e-5


@pytest.mark.parametrize("cin,cout,hw,relu,aff,ds,resm,beta", [
    (64, 16, (64, 64), True, True, True, None, 0), (16, 64, (64, 64), True, True, True, 0, 0),
    (32, 32, (32, 64), True, False, False, None, 1), (128, 32, (32, 32), True, True, True, None, 0),
    (32, 128, (64, 32), False, False, False, None, 0), (64, 64, (32, 32), True, True, False, None, 1),
    (16, 16, (128, 64), True, True, True, None, 0),
    # one shared slot (two producer groups on it), in-place ReLU with the statistics adjoint, affine without ReLU
    (128, 64, (32, 32), True, True, True, None, 0), (64, 32, (32, 64), True, False, True, None, 0),
    (16, 32, (64, 64), False, True, True, None, 1)])
def test_fused_1x1_backward_vs_torch(eng, cin, cout, hw, relu, aff, ds, resm, beta):
    """iea_conv_bwd1x1 (statistics adjoint + weight / bias gradient + data gradient + prologue adjoint of a 1x1 layer
    in one tcgen05 kernel) against torch autograd, through engine.conv's backward: dx (also accumulated onto an
    existing gradient), dW (through the spectral-norm backward), db, dscale / dshift, the residual gradient.
    Tolerance 2.5e-2 relative L2 (bf16 operands, fp32 accumulation), as the unfused bf16 path."""
    os.environ["IEA_ACT_DTYPE"] = "bf16"
    try:
        dev = "cuda"
        at = torch.bfloat16
        torch.manual_seed(3)
        n, (h, w) = 40, hw
        m = make_sn_conv(cin, cout, 1, dev)
        m.train()
        x = torch.randn(n, cin, h, w, device=dev)
        xq = x.to(at).float()
        scale = (torch.rand(n, cin, device=dev) + 0.5) if aff else None
        shift = torch.randn(n, cin, device=dev) * 0.3 if aff else None
        Wt = m.weight.detach().clone().requires_grad_(True)
        bt = m.bias.detach().clone().requires_grad_(True)
        W2 = Wt.reshape(cout, -1)
        with torch.no_grad():
            v = F.normalize(m.u0.clone() @ W2, eps=1e-6)
            un = F.normalize(v @ W2.t(), eps=1e-6)
        sig = ((v @ W2.t()) @ un.t()).squeeze()
        xr = xq.clone().requires_grad_(True)
        sr = scale.clone().requires_grad_(True) if aff else None
        hr = shift.clone().requires_grad_(True) if aff else None
        a = _ref_T(xr, sr, hr, relu, 0)
        Wq = Wt.detach().to(at).float()
        yref = F.conv2d(a, (Wq + (Wt - Wt.detach())) / sig, bt)
        if resm is not None:
            r = torch.randn(n, cout + 8, h, w, device=dev)
            rr = r.to(at).float().clone().requires_grad_(True)
            yref = yref + rr[:, :cout]
        grp = eng.SNGroup()
        l = grp.add(m, at)
        grp.run(True, True)
        tape = eng.Tape(True)
        xv = eng.Var(x.permute(0, 2, 3, 1).contiguous().to(at))
        ss = eng.ScaleShift(scale.contiguous(), shift.contiguous()) if aff else None
        resv = eng.Var(r.permute(0, 2, 3, 1).contiguous().to(at)) if resm is not None else None
        yv = eng.conv(tape, xv, l, n, h, w, 1, bias=m.bias, in_relu=relu, ss=ss, res=resv, res_mode=0,
                      res_c=cout if resm is not None else 0, stats=True)
        yq = yv.t.float().permute(0, 3, 1, 2)
        assert rel(yq, yref) < 1.5e-2
        # loss = sum(y * gy) + a function of the per-event batch statistics of y (what a following batch-norm adds):
        # sum_c (a1[c] * sum_px y + a2[c] * sum_px y^2)  ->  dL/dy = gy + a1 + 2 y a2 = exactly the (ds1, ds2) adjoint
        gy = torch.randn_like(yref)
        loss = (yref * gy).sum()
        if ds:
            a1, a2 = torch.randn(1, cout, device=dev) * 0.1, torch.randn(1, cout, device=dev) * 0.05
            yd = yq.detach()  # the kernel uses the stored (bf16) y in the 2*y*ds2 term
            loss = loss + (yref * (a1.view(1, cout, 1, 1) + 2 * yd * a2.view(1, cout, 1, 1))).sum()
        loss.backward()
        yv.g = gy.permute(0, 2, 3, 1).contiguous().to(at)
        if ds:
            yv.ds = (a1.contiguous(), a2.contiguous(), n * h * w)
        g0 = None
        if beta:
            g0 = torch.randn(n, h, w, cin, device=dev).to(at)
            xv.g = g0.clone()
        tape.backward()
        torch.cuda.synchronize()
        want_dx = xr.grad + (g0.float().permute(0, 3, 1, 2) if beta else 0)
        assert rel(xv.g.float().permute(0, 3, 1, 2), want_dx) < 2.5e-2
        assert rel(tape.pgrads[id(m.weight)], Wt.grad) < 2.5e-2
        assert rel(tape.pgrads[id(m.bias)], bt.grad) < 2.5e-2
        if aff:
            assert rel(ss.dscale, sr.grad) < 2.5e-2
            assert rel(ss.dshift, hr.grad) < 2.5e-2
        if resm is not None:
            assert rel(resv.g.float().permute(0, 3, 1, 2)[:, :cout], rr.grad[:, :cout]) < 2.5e-2
        # and the kernel really was the fused one
        import ctypes as C
        dq = eng._desc(n, h, w, cin, cout, 1, xv.t, xv.off(), xv.ld, 0, relu, scale, shift, l.wp, None, 0, None, None, 0, 0,
                       -1, yv.t, yv.off(), yv.ld, 0, None)
        from iea_gan_b200 import _lib as L
        assert L.call("iea_conv_bwd1x1_grid", C.byref(dq)) > 0
    finally:
        os.environ.pop("IEA_ACT_DTYPE", None)


@pytest.mark.parametrize("dtype,c,ld_in,ld_out", [(torch.bfloat16, 32, 32, 64), (torch.float32, 16, 24, 16), (torch.bfloat16, 64, 64, 64)])
def test_avgpool2_channel_windows_vs_torch(eng, dtype, c, ld_in, ld_out):
    """iea_avgpool2_fwd (nn.AvgPool2d(2) of an NHWC channel window into a channel window, model.py:541-557) against
    torch: fp32 average of the four pixels, one rounding to the storage dtype; untouched channels stay untouched."""
    from iea_gan_b200 import _lib as L
    torch.manual_seed(4)
    n, h, w = 3, 12, 20
    x = torch.randn(n, h, w, ld_in, device="cuda").to(dtype)
    y = torch.full((n, h // 2, w // 2, ld_out), 7.0, device="cuda").to(dtype)
    L.call("iea_avgpool2_fwd", x.data_ptr(), L.dt(x), n, h, w, c, ld_in, y.data_ptr(), ld_out, L.stream())
    ref = torch.nn.functional.avg_pool2d(x[..., :c].float().permute(0, 3, 1, 2), 2).permute(0, 2, 3, 1).to(dtype)
    torch.cuda.synchronize()
    if dtype == torch.bfloat16:
        assert torch.equal(y[..., :c], ref)  # sums of four bf16 values are exact in fp32
    else:
        assert torch.allclose(y[..., :c], ref, rtol=1e-6, atol=1e-7)
    assert bool((y[..., c:] == 7.0).all())
