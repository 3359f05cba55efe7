"""Per-launch timing of the wide-output 1x1 convolutions of one Generator sampling pass (H_base 1): conv_tc2 (the
descriptor's impl set to IMPL_TC2) against the default choice, conv_wide where it takes the shape, in the same
process.

The descriptors are captured from a real sampling pass of `events` x 40 images; each one is then launched on its
own, old and new alternating, with CUDA events around every launch.  Printed per launch: median ms of each kernel,
algorithmic GB/s (input + output + weights, each read or written once) and real GB/s (the same plus the residual,
which these layers also read).
usage: python tools/bench_wide.py [events=16] [reps=40]"""
import ctypes as C
import os
import statistics
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import iea_gan_b200 as P  # noqa: E402
from iea_gan_b200 import _lib as L  # noqa: E402
from iea_gan_b200 import engine as E_  # noqa: E402
from iea_gan_b200.default_config import shipped_config  # noqa: E402
from bench_lowres import gpu_info  # noqa: E402


def wide_1x1(d):
    """The launches conv_wide would take: 1x1, direct input, 64..256 output channels, whole 128-pixel tiles per image,
    no pooled residual or accumulate (the kernel's own envelope check decides the rest)."""
    return (d.ksize == 1 and d.in_mode == L.IN_DIRECT and d.cout in (64, 128, 256) and (d.h * d.w) % 128 == 0
            and d.acc_c0 < 0 and not (d.res and d.res_mode == L.IN_POOL2))


def main():
    if not torch.cuda.is_available():
        raise SystemExit("bench_wide.py needs a CUDA device")
    events = int(sys.argv[1]) if len(sys.argv) > 1 else 16
    reps = int(sys.argv[2]) if len(sys.argv) > 2 else 40
    cfg = shipped_config(H_base=1, device="cuda")
    torch.manual_seed(0)
    G = P.Generator(**cfg).cuda()
    G.train()
    n = 40 * events
    z = torch.randn(n, cfg["dim_z"], device="cuda")
    y = torch.arange(40, device="cuda").repeat(events)
    with torch.no_grad():
        G(z, y)
    # capture the convolution descriptors of one pass; the buffers they point at stay in torch's caching allocator
    descs = []
    k0 = E_.K

    def k_capture(name, *args, **kw):
        if name == "iea_conv_fprop":
            d = L.ConvDesc.from_buffer_copy(args[0]._obj)
            if wide_1x1(d):
                descs.append(d)
        return k0(name, *args, **kw)
    E_.K = k_capture
    try:
        with torch.no_grad():
            G(z, y)
    finally:
        E_.K = k0
    torch.cuda.synchronize()
    stream = L.stream()

    def tc2(d):
        d = L.ConvDesc.from_buffer_copy(d)
        d.impl = L.IMPL_TC2
        return d
    arms = [(tc2(d), d) for d in descs]  # (old: conv_tc2, new: as captured)

    times = [([], []) for _ in descs]
    ev = [[(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(2)]
          for _ in descs]
    for rep in range(reps + 5):  # 5 warm-up rounds
        pending = []
        for i, arm in enumerate(arms):
            for on in (0, 1) if rep % 2 == 0 else (1, 0):
                a, b = ev[i][on]
                a.record()
                E_.call("iea_conv_fprop", C.byref(arm[on]), stream)
                b.record()
                pending.append((i, on, a, b))
        torch.cuda.synchronize()
        if rep >= 5:
            for i, on, a, b in pending:
                times[i][on].append(a.elapsed_time(b))

    print("# %s" % gpu_info())
    print("# Generator sampling, H_base 1, %d events (%d images): %d wide-output 1x1 launches, median of %d "
          "alternating launches each" % (events, n, len(descs), reps))
    print("%-40s %8s %8s %6s %9s %9s %9s %9s" % ("layer", "tc2 ms", "wide ms", "x", "tc2 algGB", "wide algGB",
                                                 "tc2 realGB", "wide realGB"))
    tot = [0.0, 0.0]
    for d, (t0, t1) in zip(descs, times):
        m0, m1 = statistics.median(t0), statistics.median(t1)
        tot[0] += m0
        tot[1] += m1
        M = d.n * d.h * d.w
        alg = 2.0 * (M * d.cin + M * d.cout + d.cout * d.cin)
        real = alg
        if d.res:
            real += 2.0 * (M // 4 if d.res_mode == L.IN_UP2 else M) * d.res_c
        tag = "%dx%d %d->%d%s%s" % (d.h, d.w, d.cin, d.cout, {None: "", 0: " res", 1: " up2res"}[
            d.res_mode if d.res else None], " st" if d.stats else "")
        print("%-40s %8.4f %8.4f %6.2f %9.0f %9.0f %9.0f %9.0f" % (tag, m0, m1, m0 / m1, alg / m0 * 1e-6,
                                                                 alg / m1 * 1e-6, real / m0 * 1e-6, real / m1 * 1e-6))
    print("%-40s %8.4f %8.4f %6.2f" % ("total", tot[0], tot[1], tot[0] / tot[1]))


if __name__ == "__main__":
    main()
