"""The TMA-fed tcgen05 kernel of the wide-output 1x1 layers (wide::conv_wide_kernel in conv_wide.cu) against the
resident-weight kernel it replaces there (conv_tc2_kernel, IEA_CONV_IMPL=tc2) on the same descriptor.  Both run the
same MMA instruction shape over the channels in the same order, the same fp32 epilogue and bf16 rounding, and take
the batch-norm partial sums of each 128-pixel tile from the rounded outputs in the same order into the same slot, so
the layer output and its statistics must be bitwise equal.  Shapes outside the new kernel's envelope must run as
before; the profiler's kernel names show which kernel ran."""
import os

import pytest
import torch

from test_gpu_kernels import _tc_vs_generic, make_sn_conv

pytestmark = pytest.mark.gpu

NEW, OLD = "wide::conv_wide_kernel", "conv_tc2_kernel"
TC2 = {"IEA_CONV_IMPL": "tc2"}  # automatic routing, with conv_tc2 wherever conv_wide would run


@pytest.fixture(scope="module")
def eng():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from iea_gan_b200 import engine, _lib
    _lib.lib()
    return engine


def _run(eng, variant, cin, cout, hw, resm, aff, relu, n, xwin=False, acc=False, stats=True):
    """Forward and statistics of one 1x1 layer with the given kernel selection; returns the outputs and the names of
    the kernels that ran.  resm: None, 0 (same resolution), 1 (nearest-up2) or 2 (2x2 pooled); the residual tensor
    carries 16 channels more than the layer reads.  xwin: the input is a channel window of a wider tensor."""
    os.environ["IEA_ACT_DTYPE"] = "bf16"
    os.environ.update(variant)
    try:
        dev = "cuda"
        torch.manual_seed(5)
        h, w = hw
        m = make_sn_conv(cin, cout, 1, dev)
        m.train()
        grp = eng.SNGroup()
        l = grp.add(m, torch.bfloat16)
        grp.run(True, True)
        x = torch.randn(n, h, w, cin + (16 if xwin else 0), device=dev).bfloat16()
        scale = (torch.rand(n, cin, device=dev) + 0.5) if aff else None
        shift = (torch.randn(n, cin, device=dev) * 0.3) if aff else None
        res = None
        if resm is not None:
            rh, rw = {0: (h, w), 1: (h // 2, w // 2), 2: (2 * h, 2 * w)}[resm]
            res = torch.randn(n, rh, rw, cout + 16, device=dev).bfloat16()
        y0 = torch.randn(n, h, w, cout, device=dev).bfloat16() if acc else None

        def once():
            xv = eng.Var(x, c0=8, c=cin) if xwin else eng.Var(x)
            ss = eng.ScaleShift(scale, shift) if aff else None
            rv = eng.Var(res) if res is not None else None
            out = eng.Var(y0.clone()) if acc else None
            return eng.conv(eng.Tape(False), xv, l, n, h, w, 1, bias=m.bias, in_relu=relu, ss=ss, res=rv,
                            res_mode=resm or 0, res_c=cout if resm is not None else 0, acc_c0=cout // 2 if acc else -1,
                            out=out, stats=stats)

        # The layer runs four times, identically, inside the profiled region and the outputs are the last pass's: late
        # in a long test process the profiler drops the first three kernel records of each session, and without
        # statistics a pass is one launch.
        torch.cuda.synchronize()
        with torch.no_grad(), torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            for _ in range(3):
                once()
            yv = once()
            torch.cuda.synchronize()
        names = " ".join(e.key for e in prof.key_averages())
        st = yv.bn[0].clone() if (stats and yv.bn) else None
        return (yv.t.clone(), st), names
    finally:
        for k in ("IEA_ACT_DTYPE", "IEA_CONV_IMPL"):
            os.environ.pop(k, None)


def _same(a, b):
    return a.shape == b.shape and torch.equal(a.view(torch.int16) if a.dtype == torch.bfloat16 else a.view(torch.int32),
                                              b.view(torch.int16) if b.dtype == torch.bfloat16 else b.view(torch.int32))


def _check(new, old):
    for what, a, b in zip(("y", "statistics"), new, old):
        if b is None:
            assert a is None
            continue
        assert _same(a, b), "%s differs from conv_tc2: max |diff| %g" % (what, float((a.float() - b.float()).abs().max()))


# (cin, cout, (h, w), residual mode, affine, relu, n): the wide-output 1x1 layers of a Generator sampling pass
# (GBlock conv4 with its shortcut residual, the 256 -> 64 conv1 layers) at 16 events
SAMPLING = [
    (32, 64, (128, 128), 1, True, True, 640),
    (16, 64, (128, 128), 0, True, True, 640),
    (64, 128, (64, 64), 1, True, True, 640),
    (32, 128, (64, 64), 0, True, True, 640),
    (256, 64, (32, 32), None, True, True, 640),
    (64, 256, (32, 32), 0, True, True, 640),
    (64, 256, (32, 32), 1, True, True, 640),
    (256, 64, (16, 16), None, True, True, 640),
    (128, 256, (16, 16), 1, True, True, 640),
    (64, 256, (16, 16), 0, True, True, 640),
]
# the same layers at one event with the prologue off / ReLU only / affine only, and other geometries: an H_base = 3
# width, up2 runs at w = 128 and w = 256, Cin 128 -> Cout 64 / 128
ONE_EVENT = [(ci, co, hw, r, False, False, 40) for ci, co, hw, r, _, _, _ in SAMPLING] + [
    (32, 64, (128, 128), 1, False, True, 40),
    (64, 128, (64, 64), None, True, False, 40),
    (32, 128, (32, 96), 0, True, True, 40),
    (64, 64, (32, 96), None, True, True, 40),
    (16, 64, (256, 256), 1, True, True, 40),
    (128, 64, (16, 16), 0, True, True, 40),
    (128, 128, (32, 32), 1, False, True, 40),
]


@pytest.mark.parametrize("cin,cout,hw,resm,aff,relu,n", SAMPLING + ONE_EVENT)
def test_wide_matches_tc2_bitwise(eng, cin, cout, hw, resm, aff, relu, n):
    new, kn = _run(eng, {}, cin, cout, hw, resm, aff, relu, n)
    old, ko = _run(eng, TC2, cin, cout, hw, resm, aff, relu, n)
    assert NEW in kn, "conv_wide did not run: " + kn
    assert NEW not in ko and OLD in ko
    _check(new, old)


@pytest.mark.parametrize("cin,cout,hw,resm", [(64, 128, (32, 32), 0), (32, 64, (64, 64), 1), (256, 64, (16, 16), None)])
def test_wide_channel_window_no_stats(eng, cin, cout, hw, resm):
    """The input is a channel window of a wider tensor (x_ld > cin), with and without statistics."""
    for stats in (True, False):
        new, kn = _run(eng, {}, cin, cout, hw, resm, True, True, 40, xwin=True, stats=stats)
        old, ko = _run(eng, TC2, cin, cout, hw, resm, True, True, 40, xwin=True, stats=stats)
        assert NEW in kn and NEW not in ko
        _check(new, old)


# shapes the new kernel does not take: images of 8x8 and 8x24 pixels (not whole 128-pixel tiles), a pooled residual,
# the accumulate epilogue, Cout 32 and Cout 512
@pytest.mark.parametrize("cin,cout,hw,resm,acc", [(64, 128, (8, 8), 0, False), (128, 256, (8, 24), None, False),
                                                  (64, 128, (16, 16), 2, False), (64, 128, (16, 16), None, True),
                                                  (128, 32, (32, 32), 0, False), (128, 512, (16, 16), None, False)])
def test_wide_fallback_shapes(eng, cin, cout, hw, resm, acc):
    new, kn = _run(eng, {}, cin, cout, hw, resm, True, True, 40, acc=acc)
    old, ko = _run(eng, TC2, cin, cout, hw, resm, True, True, 40, acc=acc)
    assert NEW not in kn and NEW not in ko
    _check(new, old)


@pytest.mark.parametrize("cin,cout,resm,hw,n", [(32, 128, 0, (32, 32), 40), (64, 256, 1, (16, 16), 80)])
def test_wide_vs_generic(eng, cin, cout, resm, hw, n):
    """Forward, statistics and data gradient of the new path against the CUDA-core kernel (bf16 tolerances)."""
    _tc_vs_generic(eng, "resident", cin, cout, 1, 0, True, True, resm, hw, n)
