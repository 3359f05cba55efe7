#!/usr/bin/env python
"""bench.py -- IEA-GAN hot-path throughput on B200 (one process per GPU).

    python bench.py --gpus N --steps K --warmup W [--workload sample|train|attn-sweep] [--impl reference]

Workloads (BASELINE.json configs):
  sample      (default, configs[1]) Generator sampling, 16 events per GPU (640 images of 256x256, H_base=1), bf16
              activations, train-mode batch statistics exactly as model.generate runs it (model.py:1130-1139),
              random-init weights, synthetic z.  A "step" is one Generator forward over that batch;
              value = events/s over all ranks with z already in HBM; e2e = the same through the public API with
              pinned-host z in and the ADU-post-processed images (model.py:1139-1147) copied back to pinned host
              memory every step.  The default run also carries the train step (configs[2]) as "train_step", the
              shipped 256x768 geometry as "hbase3", and on rank 0 at N=1 the CPU baselines and the roofline.
  train       (configs[2], configs[3] under torchrun) the full G+D step, 8 events per GPU: D step + G step with
              DiffAugment, contrastive / IEA / uniformity losses, ortho-reg, clip + Adam, EMA.
  attn-sweep  (configs[4]) RelationalReasoning.forward on (B,40,128) h=2 and (B,40,512) h=4 and layers.Attention
              on (40B,256,32,32) for B = 1..256 events, forward and forward+backward.

`--impl reference` times the reference's OWN CPU implementation (the unmodified sources staged under
baseline/_ref by tools/fetch_ref.py; the CPU oracle port when they are absent) on all host cores: sampling
through model.generate and the G+D step through train_fns.GAN_training_function, one event per step.

`--dump-outputs DIR` (sample / train workloads) writes what the timed paths returned in their last step as
DIR/<name>.npy: the images of the sampling step, as many as DUMP_BYTES holds, picked with a fixed seed (device
output and the post-processed host copy of the end-to-end path), and the five floats of the train step.  Inputs and weights
come from fixed seeds, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

# SURVEY.md section 8(d): algorithmic bytes / flops per event at H_base=1 (bf16, layer granular)
G_FWD_BYTES_PER_EVENT = 2.03e9
G_FWD_FLOP_PER_EVENT = 0.134e12
TRAIN_BYTES_PER_EVENT = 31.2e9
TRAIN_FLOP_PER_EVENT = 1.73e12
DUMP_BYTES = 32 << 20  # float32 bytes of the dumped images (both sampling arrays): 64 images at 256x256


def dump_pick(n, image_bytes):
    """The fixed, seeded choice of images of a batch of n that --dump-outputs writes."""
    g = torch.Generator().manual_seed(0)
    return torch.randperm(n, generator=g)[:max(1, DUMP_BYTES // image_bytes)].sort().values


def write_dump(path, arrays):
    import numpy as np
    os.makedirs(path, exist_ok=True)
    for name, v in arrays.items():
        a = v.detach().cpu().double().numpy() if v.dtype == torch.float64 else v.detach().cpu().float().numpy()
        np.save(os.path.join(path, name + ".npy"), a)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return d["hbm_gbs"], d.get("bf16_tflops_sustained", d["bf16_tflops"]), d["bf16_tflops"], "measured"
    return 6650.0, 1590.0, 1590.0, "fallback"


class ClockSampler(threading.Thread):
    """SM clock / throttle-reason samples during the timed region: NVML at 10 Hz (nvidia-smi, 5 Hz,
    when NVML is not importable)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.sm, self.mx, self.reasons, self.stop_flag = index, [], [], set(), False
        self.nv = None
        try:
            import pynvml
            pynvml.nvmlInit()
            # NVML enumerates physical devices: map the (possibly CUDA_VISIBLE_DEVICES-remapped) ordinal by PCI bus id
            props = torch.cuda.get_device_properties(index)
            bus = props.pci_bus_id if hasattr(props, "pci_bus_id") else None
            h = None
            if bus is not None:
                for i in range(pynvml.nvmlDeviceGetCount()):
                    hi = pynvml.nvmlDeviceGetHandleByIndex(i)
                    if pynvml.nvmlDeviceGetPciInfo(hi).bus == bus:
                        h = hi
            self.nv, self.h = pynvml, h if h is not None else pynvml.nvmlDeviceGetHandleByIndex(index)
        except Exception:
            self.nv = None

    def _nvml(self):
        nv, h = self.nv, self.h
        self.sm.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
        self.mx.append(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
        r = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
        for name, bit in (("hw_slowdown", nv.nvmlClocksEventReasonHwSlowdown),
                          ("hw_thermal_slowdown", nv.nvmlClocksEventReasonHwThermalSlowdown),
                          ("sw_thermal_slowdown", nv.nvmlClocksEventReasonSwThermalSlowdown),
                          ("sw_power_cap", nv.nvmlClocksEventReasonSwPowerCap)):
            if r & bit:
                self.reasons.add(name)

    def _smi(self):
        out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                              "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
        for line in out.strip().splitlines():
            r = [t.strip() for t in line.split(",")]
            if r[1].isdigit():
                self.sm.append(int(r[1]))
            if r[2].isdigit():
                self.mx.append(int(r[2]))
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                if v.lower().startswith("active"):
                    self.reasons.add(name)

    def run(self):
        while not self.stop_flag:
            try:
                if self.nv is not None:
                    self._nvml()
                else:
                    self._smi()
            except Exception:
                if self.nv is not None:
                    self.nv = None  # fall back to nvidia-smi
            time.sleep(0.1 if self.nv is not None else 0.2)

    def summary(self):
        self.stop_flag = True
        sm = sorted(self.sm)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(self.mx) if self.mx else None,
                "reasons": sorted(self.reasons), "samples": len(sm),
                "source": "nvml" if self.nv is not None else "nvidia-smi"}


def timed(fn, steps, warmup, dist_on, finish=None, per_step=False):
    """W untimed + K timed calls bracketed by barrier + synchronize; CUDA-event time per step (ms), max over ranks.
    finish() runs before the closing event (joins side streams into the timed stream).  per_step: also the
    individual step times of this rank (an event after every step)."""
    import torch.distributed as dist
    for _ in range(warmup):
        fn()
    if finish is not None:
        finish()
    torch.cuda.synchronize()
    if dist_on:
        dist.barrier()
    torch.cuda.synchronize()
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1 if per_step else 2)]
    evs[0].record()
    for i in range(steps):
        fn()
        if per_step and i + 1 < steps:
            evs[i + 1].record()
    if finish is not None:
        finish()
    evs[-1].record()
    torch.cuda.synchronize()
    if dist_on:
        dist.barrier()
    ms = evs[0].elapsed_time(evs[-1]) / steps
    if dist_on:
        t = torch.tensor([ms], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t)
    if per_step:
        each = sorted(evs[i].elapsed_time(evs[i + 1]) for i in range(steps))
        return ms, {"median": round(each[len(each) // 2], 3), "min": round(each[0], 3), "max": round(each[-1], 3),
                    "p10": round(each[len(each) // 10], 3), "p90": round(each[(len(each) * 9) // 10], 3)}
    return ms


def build_nets(cfg, device, with_d):
    import iea_gan_b200 as P
    torch.manual_seed(0)
    G = P.Generator(**cfg).to(device)
    D = P.Discriminator(**cfg).to(device) if with_d else None
    return G, D


# ---------------------------------------------------------------------------------------- rooflines
def _time_call(fn, reps=5, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


# The four heaviest launches of a 16-event sampling pass (profiles/layers_r02_sample16.txt), 640 images each:
#   tag: (h, w, cin, cout, k, residual channels [nearest-up2 from a tensor with twice as many], statistics, label)
ROOFLINE_LAYERS = {
    "l32_64": (128, 128, 32, 64, 1, 64, True,
               "iea_conv_fprop 32->64 1x1 @128x128 + ccbn/ReLU prologue + up2 residual + stats epilogue (tc2::conv_tc2_kernel)"),
    "l32_1": (256, 256, 32, 1, 3, 0, False,
              "iea_conv_fprop 32->1 3x3 @256x256 + bn/ReLU prologue, the output conv (thin::conv_thin_kernel)"),
    "l16_32": (256, 256, 16, 32, 1, 32, True,
               "iea_conv_fprop 16->32 1x1 @256x256 + ccbn/ReLU prologue + up2 residual + stats epilogue "
               "(thin::conv_thin_kernel, TMA-store flavour)"),
    "l16_16": (256, 256, 16, 16, 3, 0, True,
               "iea_conv_fprop 16->16 3x3 @256x256 + ccbn/ReLU prologue + stats epilogue (thin::conv_thin_kernel)"),
}


def roofline_layer(E_, tag, n=640):
    """One of ROOFLINE_LAYERS as a callable that launches exactly that layer (also used by tools/prof_kernel.py under
    ncu).  Returns (call, algorithmic bytes per launch, bytes of the fused residual read, label)."""
    import iea_gan_b200.sn_layers as SL
    from iea_gan_b200 import _lib as L
    h, w, cin, cout, k, res_c, stats, label = ROOFLINE_LAYERS[tag]
    adt = E_.act_dtype()
    esz = 2 if adt == torch.bfloat16 else 4
    tape = E_.Tape(False)
    m = SL.SNConv2d(cin, cout, k, padding=k // 2, eps=1e-6).cuda()
    grp = E_.SNGroup()
    l = grp.add(m, adt)
    grp.run(True, False)
    x = torch.randn(n, h, w, cin, device="cuda").to(adt)
    ss = E_.ScaleShift(torch.rand(n, cin, device="cuda") + 0.5, torch.randn(n, cin, device="cuda"))
    kw = dict(bias=m.bias, in_relu=True, ss=ss, stats=stats)
    extra = 0
    if res_c:
        r = E_.Var(torch.randn(n, h // 2, w // 2, 2 * res_c, device="cuda").to(adt), need=False)
        kw.update(res=r, res_mode=L.IN_UP2, res_c=res_c)
        extra = n * (h // 2) * (w // 2) * res_c * esz
    xv = E_.Var(x, need=False)
    bytes_ = n * h * w * (cin + cout) * esz + k * k * cin * cout * esz
    return (lambda: E_.conv(tape, xv, l, n, h, w, k, **kw)), bytes_, extra, label


def kernel_rooflines(E_, hbm_peak, which):
    """`dominant`: the launch of the sampling step that takes the most time -- chosen LIVE among the four heaviest
    layers of the pass, each timed alone at the batch's 640 images with CUDA events on the launching stream;
    `r1_dominant`: the layer that was dominant in round 1 (16 -> 32 1x1 @256^2 + up2 residual, 0.30 then);
    `best`: the 16 -> 16 3x3 @256^2 layer.  Algorithmic bytes = layer input + output (bf16) + weights, SURVEY
    section 8(d); the fused residual read is reported separately as fused_extra_bytes and NOT counted.  `traffic` =
    DRAM bytes of the same launch from the committed ncu capture (profiles/top_kernel_traffic.json)."""
    traffic = {}
    tp = os.path.join(ROOT, "profiles", "top_kernel_traffic.json")
    if os.path.exists(tp):
        with open(tp) as f:
            traffic = json.load(f)
    res = {}
    for tag in ROOFLINE_LAYERS:
        call, bytes_, extra, label = roofline_layer(E_, tag)
        ms = _time_call(call)
        ach = bytes_ / (ms * 1e-3) / 1e9
        t = traffic.get(tag, {})
        res[tag] = {"bound": "hbm", "tag": tag, "kernel": label, "achieved": round(ach, 1), "peak": hbm_peak, "peak_source": which,
                    "unit": "GB/s", "frac": round(ach / hbm_peak, 4), "traffic": t.get("dram_bytes_per_launch"),
                    "traffic_source": t.get("source"), "ms_per_launch": round(ms, 4),
                    "algorithmic_bytes_per_launch": bytes_, "fused_extra_bytes": extra, "images": 640}
        del call
        torch.cuda.empty_cache()
    dom = max(res, key=lambda k_: res[k_]["ms_per_launch"])
    res[dom]["kernel"] += " -- the longest launch of the sampling pass"
    return {"dominant": res[dom], "r1_dominant": res["l16_32"], "best": res["l16_16"],
            "all_ms": {k_: v["ms_per_launch"] for k_, v in res.items()}}


# ---------------------------------------------------------------------------------------- CPU arms
def _ref_staged():
    try:
        import fetch_ref
        return fetch_ref.present()
    except Exception:
        return False


def cpu_reference(cfg, sample_reps, train_reps, train_warm=1):
    """The reference's own implementation on the host cores.  kind 'reference': the unmodified sources under
    baseline/_ref (model.generate; train_fns.GAN_training_function with utils.prepare_z_y / apply_ema), else kind
    'port': the CPU oracle.  Returns dict(sample_s, train_s, cores, kind, sample_desc, train_desc)."""
    torch.set_num_threads(os.cpu_count() or 1)
    c = dict(cfg, device="cpu")
    res = {"cores": torch.get_num_threads()}
    if _ref_staged():
        import fetch_ref
        keep = list(sys.path)
        fetch_ref.activate(dropin=False)
        try:
            import model as rmodel
            import train_fns as rtrain
            import utils as rutils
            torch.manual_seed(0)
            G = rmodel.Generator(**c)
            res["kind"] = "reference"
            ts = []
            for _ in range(sample_reps + 1):
                t0 = time.perf_counter()
                rmodel.generate(G)  # randn z, forward in train mode, ADU post-process (model.py:1130-1148)
                ts.append(time.perf_counter() - t0)
            ts = sorted(ts[1:])
            res["sample_s"] = ts[len(ts) // 2]
            res["sample_desc"] = ("unmodified reference model.generate (baseline/_ref), fp32, 1 event per call, "
                                  "median of %d after 1 warm-up" % sample_reps)
            if train_reps > 0:
                D = rmodel.Discriminator(**c)
                GD = rmodel.G_D(G, D)
                G_ema = rmodel.Generator(**dict(c, skip_init=True, no_optim=True))
                ema = rutils.apply_ema(G, G_ema, c["ema_decay"], c["ema_start"])
                z_, y_ = rutils.prepare_z_y(40, c["dim_z"], c["n_classes"], device="cpu", z_var=c["z_var"])
                state = {"itr": 0}
                train = rtrain.GAN_training_function(G, D, GD, z_, y_, ema, state, dict(c, batch_size=40, ema=True), "cpu")
                G.train(); D.train()
                x, y = torch.rand(40, 1, 256, 256 * c["H_base"]) * 2 - 1, torch.arange(40)
                ts = []
                for i in range(train_warm + train_reps):
                    t0 = time.perf_counter()
                    train(x, y)
                    ts.append(time.perf_counter() - t0)
                ts = sorted(ts[train_warm:])
                res["train_s"] = ts[len(ts) // 2]
                res["train_desc"] = ("unmodified reference train_fns.GAN_training_function step (D step + G step + "
                                     "ortho + Adam + EMA), fp32, 1 event, median of %d after %d warm-up"
                                     % (train_reps, train_warm))
        finally:
            sys.path[:] = keep
        return res
    from oracle import iea_oracle as O
    import iea_gan_b200 as P
    torch.manual_seed(0)
    G = P.Generator(**c)
    sd = {k: v.detach().clone() for k, v in G.state_dict().items()}
    y = torch.arange(40)
    res["kind"] = "port"
    ts = []
    for _ in range(sample_reps + 1):
        z, rd = torch.randn(40, c["dim_z"]), torch.randn(40, c["rdof_dim"])
        t0 = time.perf_counter()
        with torch.no_grad():
            O.generate_postprocess(O.generator_forward(sd, c, z, y, rd, training=True))
        ts.append(time.perf_counter() - t0)
    ts = sorted(ts[1:])
    res["sample_s"] = ts[len(ts) // 2]
    res["sample_desc"] = "CPU oracle port (oracle/iea_oracle.py) generator forward + post-process, 1 event, median of %d" % sample_reps
    if train_reps > 0:
        D = P.Discriminator(**c)
        sdd = {k: v.detach().clone() for k, v in D.state_dict().items()}
        x = torch.rand(40, 1, 256, 256 * c["H_base"]) * 2 - 1
        ts = []
        for i in range(train_warm + train_reps):
            nz = {}
            for ph in ("d", "g"):
                nz["z_" + ph], nz["rdof_" + ph] = torch.randn(40, c["dim_z"]), torch.randn(40, c["rdof_dim"])
                nz["aug_" + ph] = O.diffaug_draws(40, 256, 256 * c["H_base"])
            t0 = time.perf_counter()
            O.train_step(sd, sdd, c, x, y, nz)
            ts.append(time.perf_counter() - t0)
        ts = sorted(ts[train_warm:])
        res["train_s"] = ts[len(ts) // 2]
        res["train_desc"] = "CPU oracle port train step (no optimizer update), 1 event, median of %d" % train_reps
    return res


def run_reference(args, cfg):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    t0 = time.perf_counter()
    train = args.workload == "train"
    # --steps sets both samples: ~3 s per sampling call, ~25-30 s per train step on a 16-thread host
    k_s = k_t = max(1, args.steps)
    r = cpu_reference(cfg, k_s, k_t, train_warm=1)
    vs, vt = 1.0 / r["sample_s"], 1.0 / r["train_s"]
    cb_s = {"value": round(vs, 4), "unit": "events/s", "cores": r["cores"], "kind": r["kind"], "sample": r["sample_desc"]}
    cb_t = {"value": round(vt, 5), "unit": "events/s", "cores": r["cores"], "kind": r["kind"], "sample": r["train_desc"]}
    tr = {"metric": "G+D train-step events/s (40 PXD imgs/event)", "value": round(vt, 5), "unit": "events/s",
          "ms_per_step": round(r["train_s"] * 1e3, 1), "events_per_step": 1, "steps": k_t, "warmup": 1, "cpu_baseline": cb_t,
          "e2e": {"value": round(vt, 5), "unit": "events/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    if train:
        line = dict(tr, impl="reference", n_gpus=args.gpus, higher_is_better=True, scaling="weak", vs_baseline=None,
                    dtype="f32", data="synthetic",
                    config={"workload": "full G+D train step, H_base=%d, 1 event per step on CPU" % args.hbase,
                            "events_per_step": 1})
    else:
        line = {"impl": "reference", "metric": "G-sample events/s (40 PXD imgs/event)", "value": round(vs, 4),
                "unit": "events/s", "n_gpus": args.gpus, "steps": k_s, "warmup": 1,
                "ms_per_step": round(r["sample_s"] * 1e3, 2), "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": "Generator sampling, H_base=%d (256x%d), train-mode BN, 1 event per step on CPU"
                                       % (args.hbase, 256 * args.hbase), "events_per_step": 1},
                "cpu_baseline": cb_s,
                "e2e": {"value": round(vs, 4), "unit": "events/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "train_step": tr}
    line["wall_s"] = round(time.perf_counter() - t0, 1)
    print(json.dumps(line))


def stock_torch_gpu(cfg, dev):
    """The same unmodified reference modules on this B200 through stock PyTorch (cuDNN / cuBLAS), fp32 with TF32
    as torch defaults, 1 event per call (the reference cannot batch events: model.py:466): the existing-kernel
    bar on the same hardware, next to this repo's numbers at the same 1-event batch."""
    if not _ref_staged():
        return None
    import fetch_ref
    keep = list(sys.path)
    fetch_ref.activate(dropin=False)
    try:
        import model as rmodel
        import train_fns as rtrain
        import utils as rutils
        c = dict(cfg, device="cuda")
        torch.manual_seed(0)
        G = rmodel.Generator(**c).to(dev)
        D = rmodel.Discriminator(**c).to(dev)
        G.train(); D.train()
        z = torch.randn(40, c["dim_z"], device=dev)
        y = torch.arange(40, device=dev)

        def samp():
            with torch.no_grad():
                return G(z, y)
        ms_s = _time_call(samp, reps=10, warm=3)
        GD = rmodel.G_D(G, D)
        G_ema = rmodel.Generator(**dict(c, skip_init=True, no_optim=True)).to(dev)
        ema = rutils.apply_ema(G, G_ema, c["ema_decay"], c["ema_start"])
        z_, y_ = rutils.prepare_z_y(40, c["dim_z"], c["n_classes"], device="cuda", z_var=c["z_var"])
        train = rtrain.GAN_training_function(G, D, GD, z_, y_, ema, {"itr": 0}, dict(c, batch_size=40, ema=True), "cuda")
        x = torch.rand(40, 1, 256, 256 * c["H_base"], device=dev) * 2 - 1
        ms_t = _time_call(lambda: train(x, y), reps=5, warm=3)
        return {"what": "unmodified reference modules (baseline/_ref) through stock torch %s on this GPU, fp32, "
                        "1 event per call" % torch.__version__,
                "sample_ms_per_event": round(ms_s, 3), "sample_events_per_s": round(1e3 / ms_s, 2),
                "train_ms_per_event": round(ms_t, 2), "train_events_per_s": round(1e3 / ms_t, 3)}
    finally:
        sys.path[:] = keep
        for m in ("model", "layers", "RRM", "diff_aug", "loss", "train_fns", "utils", "cr_diff_aug", "mycleanfid"):
            for k in [k for k in sys.modules if k == m or k.startswith(m + ".")]:
                del sys.modules[k]


# ---------------------------------------------------------------------------------------- GPU workloads
def bench_sample(args, cfg, dev, world, dist_on, ev, K_, W, hbm_peak, dump=None):
    """dump: dict that receives the images of the last timed step (device path and end-to-end path)."""
    from iea_gan_b200 import engine as E_
    res_w = 256 * cfg["H_base"]
    G, _ = build_nets(cfg, dev, False)
    G.train()  # model.generate never calls eval(): batch statistics (SURVEY 3.4)
    n = 40 * ev
    z = torch.randn(n, cfg["dim_z"], device=dev)
    y = torch.arange(40, device=dev).repeat(ev)

    last = {}

    def step():
        with torch.no_grad():
            img = G(z, y)
        if dump is not None:
            last["img"] = img
        return img
    step()
    torch.cuda.synchronize()
    l0 = E_.LAUNCHES[0]
    ms, spread = timed(step, K_, W, dist_on, per_step=True)
    launches = (E_.LAUNCHES[0] - l0) // (K_ + W)
    value = ev * world / (ms * 1e-3)
    # end to end through the public API: pinned host z -> device, forward, ADU post-process, D2H
    zh = torch.randn(n, cfg["dim_z"]).pin_memory()
    yh = torch.arange(40).repeat(ev).pin_memory()
    # two pinned result buffers and a copy stream: the device->host read of step i overlaps the forward of
    # step i+1 (every step still uploads its z, y and downloads its full result; the closing event waits
    # for the last download)
    outh = [torch.empty((n, 250, res_w), dtype=torch.float32).pin_memory() for _ in range(2)]
    copy_stream = torch.cuda.Stream(device=dev)
    turn = [0]

    def step_e2e():
        with torch.no_grad():
            img = G(zh.to(dev, non_blocking=True), yh.to(dev, non_blocking=True))
            post = E_.adu_postprocess(img)
        copy_stream.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(copy_stream):
            outh[turn[0] & 1].copy_(post, non_blocking=True)
        post.record_stream(copy_stream)
        turn[0] += 1
    ms_e = timed(step_e2e, K_, W, dist_on, finish=lambda: torch.cuda.current_stream().wait_stream(copy_stream))
    if dump is not None:
        pick = dump_pick(n, (256 + 250) * res_w * 4)
        dump["sample_images"] = last.pop("img")[pick.to(dev)]
        dump["sample_e2e_images"] = outh[(turn[0] - 1) & 1][pick]
    hb = cfg["H_base"]
    gb = G_FWD_BYTES_PER_EVENT * ev * hb
    out = {"metric": "G-sample events/s (40 PXD imgs/event)", "value": round(value, 2), "unit": "events/s",
           "steps": K_, "warmup": W, "ms_per_step": round(ms, 3), "ms_spread": spread, "events_per_gpu": ev,
           "gpu_launches": launches,
           "e2e": {"value": round(ev * world / (ms_e * 1e-3), 2), "unit": "events/s",
                   "h2d_bytes_per_step": zh.numel() * 4 + yh.numel() * 8,
                   "d2h_bytes_per_step": outh[0].numel() * 4, "ms_per_step": round(ms_e, 3),
                   "overlap": "D2H of step i on a copy stream under the forward of step i+1"},
           "step_roofline": {"algorithmic_GB_per_step": round(gb / 1e9, 2),
                             "achieved_GBs": round(gb / (ms * 1e-3) / 1e9, 1),
                             "frac_of_hbm_peak": round(gb / (ms * 1e-3) / 1e9 / hbm_peak, 4)}}
    del G, z, outh
    torch.cuda.empty_cache()
    return out


def bench_train(args, cfg, dev, world, dist_on, ev, K_, W, hbm_peak, graph, dump=None, prefix="train"):
    """dump: dict that receives the five floats of the last timed step of the device-resident path."""
    import iea_gan_b200 as P
    from iea_gan_b200 import engine as E_
    from iea_gan_b200 import dp
    from iea_gan_b200.train_step import make_train_step, NormalNoise, EMA
    res_w = 256 * cfg["H_base"]
    G, D = build_nets(cfg, dev, True)
    G.train(); D.train()
    GD = P.G_D(G, D)
    if dist_on:
        dp.broadcast_state(G)
        dp.broadcast_state(D)
        dp.attach(G)  # end-of-backward all-reduce of the flat gradient buffers: nothing in the step knows about ranks
        dp.attach(D)
    n = 40 * ev
    tcfg = dict(cfg, batch_size=n, micro_events=8 if ev > 8 else 0)
    z_ = NormalNoise(n, cfg["dim_z"], dev)
    G_ema = P.Generator(**dict(cfg, skip_init=True, no_optim=True)).to(dev)
    ema = EMA(G, G_ema, cfg["ema_decay"], cfg["ema_start"])
    train = make_train_step(G, D, GD, z_, tcfg, ema=ema, **({"cuda_graph": True} if graph else {}))
    x = torch.rand(n, 1, 256, res_w, device=dev) * 2 - 1
    y = torch.arange(40, device=dev).repeat(ev)
    xh = (torch.rand(n, 1, 256, res_w) * 2 - 1).pin_memory()
    yh = torch.arange(40).repeat(ev).pin_memory()
    # (the caching allocator needs ~10 full G+D steps to stop growing: warm up that long before timing)
    wt = max(W, 10)
    l0 = E_.LAUNCHES[0]
    last = {}

    def step():
        last["losses"] = train(x, y)
    ms_t, spread = timed(step, K_, wt, dist_on, per_step=True)
    if dump is not None:
        for k, v in last["losses"].items():
            dump["%s_%s" % (prefix, k)] = torch.tensor(v, dtype=torch.float64)
    launches_t = getattr(train, "launches_per_step", None) or (E_.LAUNCHES[0] - l0) // (K_ + wt)
    ms_te = timed(lambda: train(xh.to(dev, non_blocking=True), yh.to(dev, non_blocking=True)), K_, 3, dist_on)
    hb = cfg["H_base"]
    tr = {"metric": "G+D train-step events/s (40 PXD imgs/event)", "value": round(ev * world / (ms_t * 1e-3), 3),
          "unit": "events/s", "ms_per_step": round(ms_t, 2), "ms_spread": spread, "events_per_gpu": ev, "steps": K_,
          "warmup": wt, "gpu_launches": launches_t, "cuda_graph": bool(graph),
          "e2e": {"value": round(ev * world / (ms_te * 1e-3), 3), "unit": "events/s",
                  "h2d_bytes_per_step": xh.numel() * 4 + yh.numel() * 8, "d2h_bytes_per_step": 5 * 4,
                  "ms_per_step": round(ms_te, 2)},
          "step_roofline": {"achieved_GBs": round(TRAIN_BYTES_PER_EVENT * ev * hb / (ms_t * 1e-3) / 1e9, 1),
                            "frac_of_hbm_peak": round(TRAIN_BYTES_PER_EVENT * ev * hb / (ms_t * 1e-3) / 1e9 / hbm_peak, 4),
                            "achieved_TFLOPs": round(TRAIN_FLOP_PER_EVENT * ev * hb / (ms_t * 1e-3) / 1e12, 1)}}
    del G, D, GD, train, x, G_ema, ema
    torch.cuda.empty_cache()
    return tr


def bench_attn_sweep(args, cfg, dev, hbm_peak, tf_peak):
    """BASELINE configs[4]: the two RRMs and the BigGAN self-attention block over B events, fwd and fwd+bwd.
    FLOP per event: RRM = 2*(6*S*E^2 + 2*S^2*E) (SURVEY Appendix A: 4.34 / 64.6 MMAC for E = 128 / 512);
    Attention block = 2 * 40 * 125.8 MMAC (1x1 convs + QK^T + PV at 32x32, C = 256); backward = 2x forward.
    Algorithmic bytes: RRM in + out (fp32) + weights once; Attention x in + out (bf16)."""
    import functools
    import iea_gan_b200.relational as RR
    import iea_gan_b200.sn_layers as SL
    sn = dict(num_svs=1, num_itrs=1, eps=cfg["SN_eps"])
    lin = functools.partial(SL.SNLinear, **sn)
    torch.manual_seed(0)
    mods = {
        "rrm_g_e128_h2": (RR.RelationalReasoning(num_layers=1, input_dim=128, dim_feedforward=128, which_linear=torch.nn.Linear,
                                                 num_heads=2, dropout=0.0, hidden_dim=128).to(dev).train(), 128),
        "rrm_d_e512_h4": (RR.RelationalReasoning(num_layers=1, input_dim=512, dim_feedforward=512, which_linear=lin,
                                                 num_heads=4, dropout=0.0, hidden_dim=512).to(dev).train(), 512),
    }
    att = SL.Attention(256, functools.partial(SL.SNConv2d, **sn)).to(dev).train()
    with torch.no_grad():
        att.gamma.fill_(0.5)
    rows = []
    events = [int(e) for e in args.sweep.split(",")]
    for name, (m, e) in mods.items():
        flop = 2 * (6 * 40 * e * e + 2 * 40 * 40 * e)
        wbytes = sum(p.numel() for p in m.parameters()) * 4
        for b in events:
            x = torch.randn(b, 40, e, device=dev)
            with torch.no_grad():
                ms_f = _time_call(lambda: m(x), reps=10)
            xg = x.clone().requires_grad_(True)

            def fb():
                for p in m.parameters():
                    p.grad = None
                xg.grad = None
                m(xg).sum().backward()
            ms_b = _time_call(fb, reps=5)
            byt = 2 * x.numel() * 4 + wbytes
            rows.append({"op": name, "events": b, "fwd_ms": round(ms_f, 4), "fwd_bwd_ms": round(ms_b, 4),
                         "fwd_events_per_s": round(b / ms_f * 1e3, 1),
                         "fwd_TFLOPs": round(flop * b / ms_f / 1e9, 3), "fwd_bwd_TFLOPs": round(3 * flop * b / ms_b / 1e9, 3),
                         "fwd_frac_tensor_peak": round(flop * b / ms_f / 1e9 / tf_peak, 5),
                         "fwd_GBs": round(byt / ms_f / 1e6, 1), "fwd_frac_hbm_peak": round(byt / ms_f / 1e6 / hbm_peak, 5)})
            del x, xg
    flop = 2 * 40 * 125.8e6
    # the block as the Discriminator runs it: NHWC bf16 in HBM, no layout conversion (engine-level call)
    from iea_gan_b200 import engine as E_
    amods = [att.theta, att.phi, att.g, att.o]
    grp, hs = E_._mod_plan(att, amods, [E_.act_dtype()] * 4)
    for b in events:
        n = 40 * b
        xn = torch.randn(n, 32, 32 * cfg["H_base"], 256, device=dev).to(E_.act_dtype())

        def fwd_native():
            grp.run(True, False)
            return E_._attention(E_.Tape(False), att, E_.Var(xn, need=False), n, 32, 32 * cfg["H_base"], hs)

        def fb_native():
            tape = E_.Tape(True)
            grp.run(True, True)
            xv = E_.Var(xn, need=True)
            o = E_._attention(tape, att, xv, n, 32, 32 * cfg["H_base"], hs)
            o.g = xn  # any gradient of the right shape
            tape.backward()
        ms_f = _time_call(fwd_native, reps=5 if b < 64 else 3, warm=2)
        try:
            ms_b = _time_call(fb_native, reps=3 if b < 64 else 2, warm=1)
        except torch.OutOfMemoryError:
            ms_b = float("nan")
            torch.cuda.empty_cache()
        byt = 2 * xn.numel() * xn.element_size()
        rows.append({"op": "attention_c256_32x32_native", "events": b, "fwd_ms": round(ms_f, 4), "fwd_bwd_ms": round(ms_b, 4),
                     "fwd_events_per_s": round(b / ms_f * 1e3, 1),
                     "fwd_TFLOPs": round(flop * b / ms_f / 1e9, 3), "fwd_bwd_TFLOPs": round(3 * flop * b / ms_b / 1e9, 3),
                     "fwd_frac_tensor_peak": round(flop * b / ms_f / 1e9 / tf_peak, 5),
                     "fwd_GBs": round(byt / ms_f / 1e6, 1), "fwd_frac_hbm_peak": round(byt / ms_f / 1e6 / hbm_peak, 5),
                     "note": "as inside the Discriminator: NHWC bf16 activations, theta/phi/g/o 1x1 convs + max-pools + "
                             "tcgen05 attention core + gamma residual"})
        del xn
        torch.cuda.empty_cache()
    for b in events:
        n = 40 * b
        x = torch.randn(n, 256, 32, 32 * cfg["H_base"], device=dev)
        x = x.to(memory_format=torch.contiguous_format)
        with torch.no_grad():
            ms_f = _time_call(lambda: att(x), reps=5 if b < 64 else 2, warm=2)
        xg = x.requires_grad_(True)

        def fb():
            for p in att.parameters():
                p.grad = None
            xg.grad = None
            att(xg).sum().backward()
        try:
            ms_b = _time_call(fb, reps=3 if b < 64 else 2, warm=1)
        except torch.OutOfMemoryError:  # (256 events through the fp32 NCHW module API: > 170 GB of saved tensors)
            ms_b = float("nan")
            torch.cuda.empty_cache()
        byt = 2 * x.numel() * 2
        rows.append({"op": "attention_c256_32x32", "events": b, "fwd_ms": round(ms_f, 4), "fwd_bwd_ms": round(ms_b, 4),
                     "fwd_events_per_s": round(b / ms_f * 1e3, 1),
                     "fwd_TFLOPs": round(flop * b / ms_f / 1e9, 3), "fwd_bwd_TFLOPs": round(3 * flop * b / ms_b / 1e9, 3),
                     "fwd_frac_tensor_peak": round(flop * b / ms_f / 1e9 / tf_peak, 5),
                     "fwd_GBs": round(byt / ms_f / 1e6, 1), "fwd_frac_hbm_peak": round(byt / ms_f / 1e6 / hbm_peak, 5),
                     "note": "module API: NCHW fp32 in/out, includes the layout conversions"})
        del x, xg
        torch.cuda.empty_cache()
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="sample", choices=["sample", "train", "attn-sweep"])
    ap.add_argument("--events", type=int, default=0, help="events per GPU (default 16 sampling / 8 training)")
    ap.add_argument("--global-events", type=int, default=0,
                    help="train: TOTAL events per step over all ranks (strong scaling, BASELINE configs[3]: 64); "
                         "per-GPU events above 8 are processed as 8-event micro-batches with accumulated gradients")
    ap.add_argument("--hbase", type=int, default=1)
    ap.add_argument("--sweep", default="1,4,16,64,256", help="event counts of --workload attn-sweep")
    ap.add_argument("--no-graph", action="store_true", help="train step launched kernel by kernel instead of as a CUDA graph")
    ap.add_argument("--no-extras", action="store_true", help="skip the cpu baselines / rooflines / extra workloads")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step of the sample / train paths to DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "b200" or args.workload == "attn-sweep"):
        raise SystemExit("--dump-outputs covers the b200 sample and train workloads")
    from iea_gan_b200.default_config import shipped_config
    cfg = shipped_config(H_base=args.hbase, clip_norm=1e9)  # clip_norm: otherwise G never steps (train_fns.py:190)
    if args.impl == "reference":
        return run_reference(args, cfg)

    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dist_on = world > 1
    if dist_on:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    cfg["device"] = "cuda"
    from iea_gan_b200 import engine as E_
    from iea_gan_b200 import train_step as TS
    hbm_peak, tf_peak, tf_burst, which = peaks()
    W = max(args.warmup, 3)
    K_ = max(args.steps, 1)
    res_w = 256 * args.hbase
    dtype = "bf16" if E_.act_dtype() == torch.bfloat16 else "f32"
    graph = (not args.no_graph) and hasattr(TS, "GRAPH_SUPPORTED")
    common = {"n_gpus": world, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": dtype,
              "data": "synthetic"}
    sampler = ClockSampler(local)
    sampler.start()
    extras = rank == 0 and world == 1 and not args.no_extras
    dump = {} if args.dump_outputs and rank == 0 else None

    if args.workload == "attn-sweep":
        rows = bench_attn_sweep(args, cfg, dev, hbm_peak, tf_burst)
        big = [r for r in rows if r["op"] == "rrm_d_e512_h4"][-1]
        line = dict(common, metric="RRM (E=512, h=4) forward events/s over %d-event sets" % big["events"],
                    value=big["fwd_events_per_s"], unit="events/s", steps=10, warmup=3, ms_per_step=big["fwd_ms"],
                    config={"workload": "RRM + self-attention microbench over 40-image event sets (BASELINE configs[4])",
                            "events": args.sweep, "H_base": args.hbase,
                            "l2": "weights (<= 6.3 MB) are L2-resident by design; activations of >= 64 events exceed L2"},
                    sweep=rows, clocks=sampler.summary(), gpu_launches=E_.LAUNCHES[0],
                    peaks={"hbm_GBs": hbm_peak, "bf16_TFLOPs_burst": tf_burst, "source": which})
        if rank == 0:
            print(json.dumps(line), flush=True)
        return

    if args.workload == "sample":
        s = bench_sample(args, cfg, dev, world, dist_on, args.events or 16, K_, W, hbm_peak, dump=dump)
        line = dict(common, **s)
        line["config"] = {"workload": "Generator sampling (RRM + ccbn + SNConv2d), %d events/GPU, 256x%d, train-mode BN, "
                                      "random-init weights" % (s["events_per_gpu"], res_w),
                          "events_per_gpu": s["events_per_gpu"], "H_base": args.hbase, "parallelism": "dp%d" % world,
                          "l2": "per-step working set (>1 GB of activations) far exceeds the 126 MB L2"}
        line["clocks"] = sampler.summary()
        if not args.no_extras:
            line["train_step"] = bench_train(args, cfg, dev, world, dist_on, 8, K_, W, hbm_peak, graph, dump=dump,
                                             prefix="train_step")
    else:
        ev_t = args.events or 8
        if args.global_events:
            if args.global_events % world:
                raise SystemExit("--global-events %d does not split over %d ranks" % (args.global_events, world))
            ev_t = args.global_events // world
            common["scaling"] = "strong"
        t = bench_train(args, cfg, dev, world, dist_on, ev_t, K_, W, hbm_peak, graph, dump=dump)
        line = dict(common, **t)
        if args.global_events:
            line["global_events"] = args.global_events
            line["micro_events"] = 8 if ev_t > 8 else ev_t
        line["config"] = {"workload": "full G+D hinge/contrastive train step with DiffAugment, ortho-reg, clip + Adam, "
                                      "EMA, %d events/GPU, 256x%d" % (t["events_per_gpu"], res_w),
                          "events_per_gpu": t["events_per_gpu"], "H_base": args.hbase, "parallelism": "dp%d" % world,
                          "clip_norm": 1e9, "l2": "per-step working set (tens of GB) far exceeds the 126 MB L2"}
        line["clocks"] = sampler.summary()
    if extras:
        try:
            if args.hbase == 1 and args.workload == "sample":
                c3 = dict(cfg, H_base=3)
                h3 = bench_sample(args, c3, dev, world, False, 8, K_, W, hbm_peak)
                line["hbase3"] = {k: h3[k] for k in ("value", "unit", "ms_per_step", "events_per_gpu", "e2e", "step_roofline")}
                line["hbase3"]["workload"] = "Generator sampling at the shipped geometry 256x768 (H_base=3), 8 events"
        except Exception as e:
            line["hbase3"] = {"error": repr(e)}
        try:
            rl = kernel_rooflines(E_, hbm_peak, which)
            line["roofline"] = rl["dominant"]
            line["roofline_r1_dominant"] = rl["r1_dominant"]
            line["roofline_best_kernel"] = rl["best"]
            line["roofline_candidates_ms"] = rl["all_ms"]
        except Exception as e:  # never lose the headline because an extra failed
            line["roofline"] = {"error": repr(e)}
        try:
            st = stock_torch_gpu(cfg, dev)
            if st is not None:
                line["stock_torch_gpu"] = st
        except Exception as e:
            line["stock_torch_gpu"] = {"error": repr(e)}
        torch.cuda.empty_cache()
        try:
            want_train = args.workload == "train" or "train_step" in line
            r = cpu_reference(dict(cfg, device="cpu"), 2 if args.workload == "sample" else 1, 1 if want_train else 0,
                              train_warm=0)
            cb_s = {"value": round(1.0 / r["sample_s"], 4), "unit": "events/s", "cores": r["cores"], "kind": r["kind"],
                    "sample": r["sample_desc"]}
            if want_train:
                cb_t = {"value": round(1.0 / r["train_s"], 5), "unit": "events/s", "cores": r["cores"], "kind": r["kind"],
                        "sample": r["train_desc"].replace("median of 1 after 0 warm-up", "one step, no warm-up")}
            if args.workload == "train":
                line["cpu_baseline"] = cb_t
            else:
                line["cpu_baseline"] = cb_s
                if want_train:
                    line["train_step"]["cpu_baseline"] = cb_t
        except Exception as e:
            line["cpu_baseline"] = {"error": repr(e)}
    if dump is not None:
        write_dump(args.dump_outputs, dump)
    if rank == 0:
        print(json.dumps(line), flush=True)
    if dist_on:
        # leave without tearing NCCL down: a captured CUDA graph still holds NCCL kernels of this communicator, and
        # destroying the process group under it aborted rank 0 (SIGABRT) after the line had been printed
        import gc
        gc.collect()
        torch.cuda.synchronize()
        dist.barrier()
        torch.cuda.synchronize()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


if __name__ == "__main__":
    main()
