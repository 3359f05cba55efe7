"""Per-launch timing of the wide low-resolution convolutions of one Generator sampling pass (H_base 1), streaming
kernel (the descriptor's impl set to IMPL_TC_STREAM) against the default choice, the staged-patch kernel where it
takes the shape, in the same process.

The descriptors are captured from a real sampling pass of `events` x 40 images; each one is then launched on its
own, old and new alternating, with CUDA events around every launch.  A layer's inputs (<= 42 MB) stay in the
126 MB L2 between repetitions, as they mostly do in the step, where the previous layer has just written them.
Printed per launch: median ms of each kernel, achieved TFLOP/s (2*M*Cin*Cout*taps) and algorithmic GB/s
(input + output + weights + residual, each read or written once).
usage: python tools/bench_lowres.py [events=16] [reps=40]"""
import ctypes as C
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import iea_gan_b200 as P  # noqa: E402
from iea_gan_b200 import _lib as L  # noqa: E402
from iea_gan_b200 import engine as E_  # noqa: E402
from iea_gan_b200.default_config import shipped_config  # noqa: E402


def gpu_info():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=clocks.sm,clocks.max.sm,power.limit", "--format=csv,noheader",
                            "-i", "0"], capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "not available"
    return "%s; SM clock, max SM clock, power limit: %s" % (name, q)


def wide_lowres(d):
    """The layers whose weights do not fit next to a staged patch: >= 128-channel 3x3 at 4x4..16x16 and 512-channel
    1x1 at 4x4 and 8x8 (not the head linears, which run as 1x1 convolutions on 1x1 images)."""
    if d.ksize == 3:
        return d.cin >= 128 and d.cout >= 128 and d.h <= 16 and d.in_mode != L.IN_POOL2
    return max(d.cin, d.cout) >= 512 and 4 <= d.h <= 8


def main():
    if not torch.cuda.is_available():
        raise SystemExit("bench_lowres.py needs a CUDA device")
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
            if wide_lowres(d):
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

    def streaming(d):
        d = L.ConvDesc.from_buffer_copy(d)
        d.impl = L.IMPL_TC_STREAM
        return d
    arms = [(streaming(d), d) for d in descs]  # (old: streaming kernel, new: as captured)

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
    print("# Generator sampling, H_base 1, %d events (%d images): %d wide low-resolution launches, median of %d "
          "alternating launches each, L2 warm" % (events, n, len(descs), reps))
    print("%-44s %8s %8s %6s %8s %8s %8s %8s" % ("layer", "old ms", "new ms", "x", "old TF/s", "new TF/s", "old GB/s",
                                                  "new GB/s"))
    tot = [0.0, 0.0]
    for d, (t0, t1) in zip(descs, times):
        m0, m1 = statistics.median(t0), statistics.median(t1)
        tot[0] += m0
        tot[1] += m1
        M = d.n * d.h * d.w
        taps = d.ksize * d.ksize
        flop = 2.0 * M * d.cin * d.cout * taps
        hs, ws = (d.h // 2, d.w // 2) if d.in_mode == L.IN_UP2 else (d.h, d.w)
        byts = 2.0 * (d.n * hs * ws * d.cin + M * d.cout + d.cout * d.cin * taps)
        if d.res:
            rh, rw = (d.h // 2, d.w // 2) if d.res_mode == L.IN_UP2 else (d.h, d.w)
            byts += 2.0 * d.n * rh * rw * d.res_c
        tag = "%dx%d %d->%d k%d%s%s%s" % (d.h, d.w, d.cin, d.cout, d.ksize, " up2" if d.in_mode == L.IN_UP2 else "",
                                          " res" if d.res else "", " st" if d.stats else "")
        print("%-44s %8.4f %8.4f %6.2f %8.1f %8.1f %8.0f %8.0f" % (tag, m0, m1, m0 / m1, flop / m0 * 1e-9,
                                                                   flop / m1 * 1e-9, byts / m0 * 1e-6, byts / m1 * 1e-6))
    print("%-44s %8.4f %8.4f %6.2f" % ("total", tot[0], tot[1], tot[0] / tot[1]))


if __name__ == "__main__":
    main()
