"""The staged-patch tcgen05 kernel of the wide low-resolution 3x3 layers (conv_lr_kernel in conv_tc.cu) against the
streaming kernel (conv_tc_kernel, IEA_CONV_IMPL=stream) on the same descriptor.  Both accumulate every output
element over the same products in the same order (tap, k block, 16-channel step) and tile the pixels alike, so
the layer output, its batch-norm partial sums and the data gradient must be bitwise equal.  Shapes the new kernel
does not take must fall back to the streaming kernel; the profiler's kernel names show which one ran."""
import os

import pytest
import torch

from test_gpu_kernels import _tc_vs_generic, make_sn_conv

pytestmark = pytest.mark.gpu

NEW, OLD = "conv_lr_kernel", "conv_tc_kernel"
STREAM = {"IEA_CONV_IMPL": "stream"}  # the streaming kernel wherever it takes the shape


@pytest.fixture(scope="module")
def eng():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from iea_gan_b200 import engine, _lib
    _lib.lib()
    return engine


def _run(eng, variant, cin, cout, mode, relu, aff, resm, hw, n, stats):
    """Forward (+ statistics) and data gradient of one 3x3 layer with the given kernel selection; returns the
    outputs and the names of the kernels that ran."""
    os.environ["IEA_ACT_DTYPE"] = "bf16"
    os.environ.update(variant)
    try:
        dev = "cuda"
        torch.manual_seed(5)
        h, w = hw
        hs, ws = (h // 2, w // 2) if mode == 1 else (h, w)
        m = make_sn_conv(cin, cout, 3, dev)
        m.train()
        grp = eng.SNGroup()
        l = grp.add(m, torch.bfloat16)
        grp.run(True, True)
        x = torch.randn(n, hs, ws, cin, device=dev).bfloat16()
        scale = (torch.rand(n, cin, device=dev) + 0.5) if aff else None
        shift = (torch.randn(n, cin, device=dev) * 0.3) if aff else None
        res = None
        if resm is not None:
            rh, rw = (h // 2, w // 2) if resm == 1 else (h, w)
            res = torch.randn(n, rh, rw, cout + 16, device=dev).bfloat16()
        g = torch.randn(n, h, w, cout, device=dev).bfloat16()
        torch.cuda.synchronize()
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            tape = eng.Tape(True)
            xv = eng.Var(x)
            ss = eng.ScaleShift(scale, shift) if aff else None
            rv = eng.Var(res) if res is not None else None
            yv = eng.conv(tape, xv, l, n, h, w, 3, bias=m.bias, in_mode=mode, in_relu=relu, ss=ss, res=rv,
                          res_mode=resm or 0, res_c=cout if resm is not None else 0, stats=stats)
            yv.g = g
            m.bias.requires_grad_(False)
            tape.backward()
            torch.cuda.synchronize()
        names = " ".join(e.key for e in prof.key_averages())
        st = yv.bn[0].clone() if (stats and yv.bn) else None
        return (yv.t.clone(), st, xv.g.clone()), names
    finally:
        for k in ("IEA_ACT_DTYPE", "IEA_CONV_IMPL"):
            os.environ.pop(k, None)


def _same(a, b):
    return a.shape == b.shape and torch.equal(a.view(torch.int16) if a.dtype == torch.bfloat16 else a.view(torch.int32),
                                              b.view(torch.int16) if b.dtype == torch.bfloat16 else b.view(torch.int32))


# (cin, cout, in_mode, in_relu, affine, residual mode, (h, w), n): every 3x3 layer of G and D at 8x8 and 16x16
# (H_base 1) with direct / nearest-up2 inputs, the prologue on and off, direct / up2 residuals, 1 and 16 events;
# plus other row-tile geometries (one image per tile, 4 rows of 32)
CASES = [
    (128, 128, 1, True, True, None, (16, 16), 640),   # GBlock conv1, 8x8 -> 16x16
    (128, 128, 0, True, True, 1, (16, 16), 640),      # GBlock conv2 + up2 shortcut
    (128, 128, 1, True, True, None, (8, 8), 640),
    (128, 128, 0, True, True, 0, (8, 8), 640),
    (128, 128, 0, True, True, None, (16, 16), 40),
    (128, 128, 1, True, False, 1, (8, 8), 40),
    (128, 128, 0, False, False, None, (8, 8), 40),
    (128, 128, 0, False, True, 0, (16, 16), 40),
    (64, 128, 0, True, True, None, (16, 16), 40),
    (128, 64, 1, True, True, None, (8, 8), 40),
    (64, 64, 0, True, True, 0, (8, 8), 40),
    (128, 128, 0, True, True, None, (8, 16), 40),
    (128, 128, 1, True, True, 1, (32, 32), 40),
]


@pytest.mark.parametrize("cin,cout,mode,relu,aff,resm,hw,n", CASES)
def test_lowres_matches_stream_impl_bitwise(eng, cin, cout, mode, relu, aff, resm, hw, n):
    new, kn = _run(eng, {}, cin, cout, mode, relu, aff, resm, hw, n, True)
    old, ko = _run(eng, STREAM, cin, cout, mode, relu, aff, resm, hw, n, True)
    assert NEW in kn, "the staged-patch kernel did not run: " + kn
    assert NEW not in ko and OLD in ko
    for what, a, b in zip(("y", "statistics", "dx"), new, old):
        if b is None:
            assert a is None
            continue
        assert _same(a, b), "%s differs from the streaming kernel: max |diff| %g" % (
            what, float((a.float() - b.float()).abs().max()))


@pytest.mark.parametrize("hw,n", [((8, 8), 41), ((8, 8), 1)])
def test_lowres_partial_last_tile(eng, hw, n):
    """An odd image count at 8x8, where a 128-pixel tile holds two images: the last tile's second image does not
    exist and its rows must read as zero padding (no statistics: they need whole events)."""
    new, kn = _run(eng, {}, 128, 128, 0, True, True, None, hw, n, False)
    old, _ = _run(eng, STREAM, 128, 128, 0, True, True, None, hw, n, False)
    assert NEW in kn
    assert _same(new[0], old[0]) and _same(new[2], old[2])


# the H_base = 3 widths (4x12, 8x24, 16x48) and 4x4 stay on the streaming kernel
@pytest.mark.parametrize("hw,mode", [((4, 12), 0), ((8, 24), 1), ((16, 48), 1), ((16, 48), 0), ((4, 4), 0),
                                     ((4, 4), 1)])
def test_lowres_fallback_shapes(eng, hw, mode):
    new, kn = _run(eng, {}, 128, 128, mode, True, True, 0, hw, 40, True)
    old, _ = _run(eng, STREAM, 128, 128, mode, True, True, 0, hw, 40, True)
    assert NEW not in kn and OLD in kn
    for a, b in zip(new, old):
        assert _same(a, b)


@pytest.mark.parametrize("cin,cout,mode,relu,aff,resm,hw,n", [
    (128, 128, 1, True, True, None, (16, 16), 40), (128, 128, 0, True, True, 1, (16, 16), 80),
    (128, 128, 0, True, False, 0, (8, 8), 40), (64, 128, 1, False, True, None, (8, 8), 40)])
def test_lowres_vs_generic(eng, cin, cout, mode, relu, aff, resm, hw, n):
    """Forward, statistics and data gradient of the new path against the CUDA-core kernel (bf16 tolerances)."""
    _tc_vs_generic(eng, "resident", cin, cout, 3, mode, relu, aff, resm, hw, n)
