"""Execution engine: schedules the fused sm_100a kernels of libiea_sm100.so for the
Generator / Discriminator forward and backward passes.

Design (B200-first, not a port of the reference's layer-by-layer autograd graph):
  * activations live in HBM as NHWC bf16 (fp32 when IEA_ACT_DTYPE=fp32 for tight
    parity runs); parameters stay fp32 in the reference's layout;
  * one grouped launch runs the spectral-norm power iteration of every layer of a
    net and repacks the weights for the conv kernels (`SNGroup`); W/sigma is never
    materialised, 1/sigma is an epilogue scale;
  * batch-norm statistics come out of the producer conv's epilogue and the
    normalise + gain/bias + ReLU (+ nearest-upsample / avg-pool) is the consumer
    conv's prologue, so every activation is written once and read once;
  * all 96 ccbn gain/bias linears of G are ONE grouped GEMM on the shared
    conditioning vector;
  * backward is a small explicit tape (`Tape`) per net call, bridged to torch
    autograd by one `autograd.Function` per net, so parameter gradients honour
    `requires_grad` toggling and `no_grad`.
"""
import ctypes as C
import os

import numpy as np
import torch

from . import _lib as L
from . import noise
from ._lib import call, ptr, dt

IMGS = 40  # images per event (model.py:466)


_ENV = os.environ._data if hasattr(os.environ, "_data") else None  # raw bytes mapping: no encode/decode per lookup


def _env(name_b, name, default):
    if _ENV is not None:
        v = _ENV.get(name_b)
        return default if v is None else v.decode()
    return os.environ.get(name, default)


def act_dtype():
    return torch.float32 if _env(b"IEA_ACT_DTYPE", "IEA_ACT_DTYPE", "bf16") == "fp32" else torch.bfloat16


def conv_impl():
    return {"auto": L.IMPL_AUTO, "generic": L.IMPL_GENERIC, "tcgen05": L.IMPL_TCGEN05, "stream": L.IMPL_TC_STREAM,
            "tc2": L.IMPL_TC2}[
        _env(b"IEA_CONV_IMPL", "IEA_CONV_IMPL", "auto")]


LAUNCHES = [0]  # kernels launched through the C ABI (bench.py reports it)


GRAPH_KEEP = None  # while a CUDA graph is being captured: list that keeps pinned host tables alive for its replays
TRACE = None    # debugging aid: a list that receives (shape tag, output tensor) of every conv() call
PROFILE = None  # tools/prof_layers.py sets this to a list: (name, tag, start event, end event) per C-ABI call


def _tag(name, args):
    """Shape tag of a call for the per-layer profile (convolution descriptors carry their geometry)."""
    a0 = getattr(args[0], "_obj", None) if args else None
    if isinstance(a0, L.ConvDesc):
        return "n%d %dx%d %d->%d k%d in%d%s%s%s%s" % (a0.n, a0.h, a0.w, a0.cin, a0.cout, a0.ksize, a0.in_mode,
                                                    " aff" if a0.in_scale else "", " relu" if a0.in_relu else "",
                                                    " res%d" % a0.res_mode if a0.res else "", " st" if a0.stats else "")
    return " ".join(str(a) for a in args if isinstance(a, int) and 0 <= a < (1 << 31))[:48]


def K(name, *args, launches=1):
    LAUNCHES[0] += launches
    if PROFILE is None:
        return call(name, *args)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    rc = call(name, *args)
    b.record()
    PROFILE.append((name, _tag(name, args), a, b))
    return rc


def cdiv(a, b):
    return (a + b - 1) // b


def on_tensor_device(fn):
    """Run an entry point with the CUDA device of its first tensor / module argument current: the C ABI launches
    on the current device's stream, so a net living on cuda:1 while cuda:0 is current must switch first."""
    import functools

    @functools.wraps(fn)
    def wrapped(*args, **kw):
        dev = None
        for a in args:
            if isinstance(a, torch.Tensor):
                dev = a.device
            elif isinstance(a, torch.nn.Module):
                dev = next((t.device for t in a.parameters()), None)
            elif isinstance(a, (list, tuple)) and a and isinstance(a[0], torch.nn.Module):
                dev = next((t.device for t in a[0].parameters()), None)
            if dev is not None:
                break
        if dev is None or dev.type != "cuda" or dev.index is None or dev.index == torch._C._cuda_getDevice():
            return fn(*args, **kw)
        with torch.cuda.device(dev):
            return fn(*args, **kw)
    return wrapped


# ------------------------------------------------------------------ tape
class Var:
    """A tensor flowing through a net with an optional gradient slot.  The kernels see it as a
    matrix of rows x ld with a channel window [c0, c0+c)."""
    __slots__ = ("t", "c0", "c", "ld", "g", "ds", "bn", "need", "sc_var")

    def __init__(self, t, need=True, c0=0, c=None):
        self.t = t
        self.ld = t.shape[-1]
        self.c0 = c0
        self.c = self.ld if c is None else c
        self.g = None
        self.ds = None      # (ds1, ds2, rows_per_event): batch-norm statistics gradient
        self.bn = None      # (partials, tiles_per_event, count_per_event)
        self.need = need
        self.sc_var = None  # Var of a shortcut conv that wrote a channel window of this tensor

    def off(self, t=None):
        t = self.t if t is None else t
        return t.data_ptr() + self.c0 * t.element_size()


class Tape:
    def __init__(self, record, flat=None):
        self.record = record
        self.nodes = []
        self.pgrads = {}
        self.sn_jobs = []  # deferred W/sigma backward of the layers of this pass: one grouped launch
        self.flat = flat   # optim.FlatGrads of the owning net: parameter gradients are written in place
        self.direct = set()
        self.sn_targets = set()  # gradient tensors the queued (not yet launched) spectral-norm jobs will write

    def add(self, fn):
        if self.record:
            self.nodes.append(fn)

    def backward(self):
        for fn in reversed(self.nodes):
            fn()
        self.nodes = []
        self.flush_sn()

    def sn_weight_bwd(self, gp, nsplit, layer, saved, dw, beta=0.0):
        """Queue dW = beta*dW + G/sigma - (<G,W>/sigma^2) u v^T for one layer (iea_sn_weight_bwd_grouped)."""
        isg, u_, v_ = saved
        self.sn_jobs.append((gp, nsplit, layer.weight, u_, v_, isg, layer.spectral, dw, layer.rows, layer.cin, layer.taps,
                             beta))
        self.sn_targets.add(dw.data_ptr())

    def flush_sn(self):
        jobs, self.sn_jobs = self.sn_jobs, []
        self.sn_targets = set()
        if not jobs:
            return
        items = (L.SnBwdItem * len(jobs))()
        b0 = 0
        for it, (gp, nsplit, w, u_, v_, isg, spectral, dw, rows, cin, taps, beta) in zip(items, jobs):
            nb = max(1, min(256, (rows * cin * taps + 1023) // 1024))
            it.gpart, it.w, it.u, it.v, it.inv_sigma, it.dw = ptr(gp), ptr(w), ptr(u_), ptr(v_), ptr(isg), ptr(dw)
            it.nsplit, it.spectral, it.rows, it.cin, it.taps, it.beta = nsplit, spectral, rows, cin, taps, beta
            it.block0, it.nblocks = b0, nb
            b0 += nb
        dev = jobs[0][7].device
        host = torch.frombuffer(bytearray(bytes(items)), dtype=torch.uint8).pin_memory()
        table = host.to(dev, non_blocking=True)
        K("iea_sn_weight_bwd_grouped", ptr(table), len(jobs), b0, ptr(_f32(b0, dev)), L.stream(), launches=2)
        if GRAPH_KEEP is not None:
            GRAPH_KEEP.append(host)  # the captured host->device copy re-reads this buffer at every replay
        self._sn_keep = (host, table)  # (stream-ordered allocators make dropping the job tensors safe once enqueued)

    def galloc(self, param, accumulate_ok=False):
        """Where a kernel should write the gradient of `param`: (tensor, beta).
        With a flat gradient buffer (optim.FlatGrads) the tensor is the parameter's view of it: attached as
        `param.grad` and overwritten (beta 0) when `param.grad` is None -- the first backward after
        zero_grad() -- or accumulated into (beta 1, for kernels that can: accumulate_ok) when `param.grad`
        already is that view (second Discriminator call of a pass, gradient accumulation).  Otherwise a fresh
        tensor that pgrad() adds into the view / hands to autograd."""
        fl = self.flat
        if fl is not None:
            k = id(param)
            v = fl.views.get(k)
            if v is not None:
                g = param.grad
                if g is None:
                    param.grad = v
                    self.direct.add(k)
                    return v, 0.0
                if g.data_ptr() == fl.ptrs[k]:
                    self.direct.add(k)
                    if accumulate_ok:
                        if fl.ptrs[k] in self.sn_targets:
                            self.flush_sn()  # (two queued jobs of one grouped launch must not write the same tensor)
                        return v, 1.0
        return torch.empty_like(param), 0.0

    def pgrad(self, param, g):
        """Record gradient contribution g (the tensor a kernel wrote) of `param`."""
        k = id(param)
        acc = self.pgrads.get(k)
        if acc is None and k in self.direct:
            acc = self.flat.views[k]
            self.pgrads[k] = acc
            if g.data_ptr() == acc.data_ptr():
                return
        elif acc is None:
            fl = self.flat
            if fl is not None and k in fl.views:
                # a gradient produced outside galloc (small tensors: LayerNorm, bn gain / bias, gamma, embeddings):
                # move it into the flat buffer so that EVERY gradient of the net lives there
                tgt, beta = self.galloc(param, accumulate_ok=True)
                if k in self.direct:
                    K("iea_axpby", ptr(g), L.F32, 1.0, ptr(tgt), L.F32, beta, ptr(tgt), L.F32, g.numel(), L.stream())
                    self.pgrads[k] = tgt
                    return
            self.pgrads[k] = g
            return
        if g.data_ptr() == acc.data_ptr():
            return  # written in place with beta = 1
        if acc.data_ptr() in self.sn_targets:
            self.flush_sn()  # (the accumulation reads a gradient a queued job has not written yet)
        K("iea_axpby", ptr(g), L.F32, 1.0, ptr(acc), L.F32, 1.0, ptr(acc), L.F32, g.numel(), L.stream())


def _accum_target(v):
    """(gradient buffer of v, beta): beta = 1 when a previous consumer already wrote it."""
    if v.g is None:
        v.g = torch.empty_like(v.t)
        return v.g, 0.0
    return v.g, 1.0


def add_grad(v, g):
    if v.g is None:
        v.g = g
    else:
        K("iea_axpby", ptr(g), dt(g), 1.0, ptr(v.g), dt(v.g), 1.0, ptr(v.g), dt(v.g), g.numel(), L.stream())


def _scalar(device):
    """0-d fp32 result tensor of a loss kernel (NOT a view of a 1-element buffer: callers accumulate losses in
    place -- `G_loss += ...`, train_fns.py:168 -- which autograd forbids on a view made inside a custom Function)."""
    return torch.empty((), dtype=torch.float32, device=device)


def _f32(n, device):
    return torch.empty(max(int(n), 1), dtype=torch.float32, device=device)


# ------------------------------------------------------------------ spectral norm group
class SNLayer:
    """One (optionally spectrally-normalised) weight inside an SNGroup."""
    __slots__ = ("mod", "weight", "rows", "cin", "taps", "spectral", "pack_dtype", "wp", "wd", "index",
                 "colscale", "group", "wd_ld", "shared", "wp_tc", "wd_tc", "want_tc")

    def inv_sigma(self):
        return self.group.cur[0][self.index:self.index + 1]

    def u(self):
        o = self.group.u_off[self.index]
        return self.group.cur[1][o:o + self.rows]

    def v(self):
        o = self.group.v_off[self.index]
        return self.group.cur[2][o:o + self.cin * self.taps]

    def saved(self):
        """(inv_sigma, u', v) of the CURRENT forward call, to be captured by backward closures."""
        return self.inv_sigma(), self.u(), self.v()


class SNGroup:
    """All weights of a net that go through the grouped power-iteration / repack kernel
    (layers.py:89-165).  Built once per net; `run()` is called at the top of each forward."""

    def __init__(self):
        self.layers = []
        self.key = None
        self.shared_packs = []
        self.tables = {}
        self.cur = None

    def add(self, mod, pack_dtype, tc=False):
        """tc: also keep the bf16 tensor-core packs for a layer whose regular packs are fp32 (the head / RRM linears:
        with >= TC_LINEAR_MIN_ROWS rows they run as tcgen05 GEMMs, see linear())."""
        w = mod.weight
        l = SNLayer()
        l.mod, l.weight = mod, w
        l.rows = w.shape[0]
        l.cin, l.taps = (w.shape[1], w.shape[2] * w.shape[3]) if w.dim() == 4 else (w.shape[1], 1)
        l.spectral = 1 if hasattr(mod, "u0") else 0
        l.pack_dtype = pack_dtype
        l.index = len(self.layers)
        l.group = self
        l.colscale = None
        l.wp = l.wd = l.wp_tc = l.wd_tc = None
        l.wd_ld = l.rows
        l.shared = False
        l.want_tc = bool(tc)
        self.layers.append(l)
        return l

    def add_shared(self, mods, pack_dtype):
        """Several linears on the same input packed into one [sum rows][cin] matrix with a
        per-output-column 1/sigma vector (the grouped ccbn GEMM)."""
        ls = [self.add(m, pack_dtype) for m in mods]
        for l in ls:
            l.shared = True
        self.shared_packs.append(ls)
        return ls

    def _signature(self):
        ls = self.layers
        return (ls[0].weight.data_ptr(), ls[-1].weight.data_ptr(), ls[0].weight.device, len(ls))

    def _build(self, device):
        ls = self.layers
        total = {torch.float32: 0, torch.bfloat16: 0}
        al = lambda n: (n + 63) // 64 * 64
        offs = []
        for l in ls:
            if l.shared:
                offs.append(None)
                continue
            offs.append(total[l.pack_dtype])
            total[l.pack_dtype] += 2 * al(l.rows * l.cin * l.taps)
        shared_info = []
        for grp in self.shared_packs:
            rows, cin = sum(l.rows for l in grp), grp[0].cin
            shared_info.append((total[grp[0].pack_dtype], rows, cin))
            total[grp[0].pack_dtype] += 2 * al(rows * cin)
        self.packs = {d: torch.zeros(max(n, 1), dtype=d, device=device) for d, n in total.items()}
        self.colscales = []
        for (o, rows, cin), grp in zip(shared_info, self.shared_packs):
            buf = self.packs[grp[0].pack_dtype]
            n = rows * cin
            wp = buf[o:o + n].view(rows, cin)
            wd = buf[o + al(n):o + al(n) + n].view(cin, rows)
            cs = torch.ones(rows, dtype=torch.float32, device=device)
            self.colscales.append((wp, wd, cs))
            r0 = 0
            for l in grp:
                l.wp, l.wd, l.wd_ld, l.colscale = wp[r0:r0 + l.rows], wd[:, r0:r0 + l.rows], rows, cs[r0:r0 + l.rows]
                r0 += l.rows
        for l, o in zip(ls, offs):
            if o is None:
                continue
            buf = self.packs[l.pack_dtype]
            n = l.rows * l.cin * l.taps
            l.wp = buf[o:o + n].view(l.rows, l.taps, l.cin)
            l.wd = buf[o + al(n):o + al(n) + n].view(l.cin, l.taps, l.rows)
        # bf16 copies in the tcgen05 kernel's order for the tensor-core-eligible layers
        tc_ok = lambda c: c in (16, 32) or (c >= 64 and c % 64 == 0)
        tc_total, tc_offs = 0, []
        pad16 = lambda c: (c + 15) // 16 * 16
        for l in ls:
            # output channels may be padded to 16 (the 32->1 output conv of G, the 32->1 dgrad of D's stem)
            f = (not l.shared) and (l.pack_dtype == torch.bfloat16 or l.want_tc) and tc_ok(pad16(l.cin))
            b = (not l.shared) and (l.pack_dtype == torch.bfloat16 or l.want_tc) and tc_ok(l.rows)
            nf, nb = al(pad16(l.rows) * pad16(l.cin) * l.taps), al(l.rows * pad16(l.cin) * l.taps)
            tc_offs.append((tc_total if f else None, tc_total + nf if b else None))
            tc_total += (nf + nb) if (f or b) else 0
        self.tc_pack = torch.zeros(max(tc_total, 1), dtype=torch.bfloat16, device=device)
        for l, (fo, bo) in zip(ls, tc_offs):
            nf, nb = pad16(l.rows) * pad16(l.cin) * l.taps, l.rows * pad16(l.cin) * l.taps
            l.wp_tc = self.tc_pack[fo:fo + nf] if fo is not None else None
            l.wd_tc = self.tc_pack[bo:bo + nb] if bo is not None else None
        chunks, metas, scratch, uo, vo = [], [], 0, 0, 0
        self.u_off, self.v_off = [], []
        for i, l in enumerate(ls):
            cols = l.cin * l.taps
            rows_per = max(1, 32768 // cols)
            c0 = len(chunks)
            for r in range(0, l.rows, rows_per):
                chunks.append((i, r, min(l.rows, r + rows_per)))
            metas.append((c0, len(chunks) - c0, scratch))
            scratch += (len(chunks) - c0) * cols + l.rows
            self.u_off.append(uo)
            self.v_off.append(vo)
            uo += l.rows
            vo += cols
        self.metas = metas
        self.chunks = torch.tensor(np.array(chunks, dtype=np.int32).reshape(-1), dtype=torch.int32, device=device)
        self.n_chunks = len(chunks)
        self.scratch = torch.empty(scratch, dtype=torch.float32, device=device)
        self.max_cols = max(l.cin * l.taps for l in ls)
        self.inv_sigma = torch.ones(len(ls), dtype=torch.float32, device=device)
        self.u_new = torch.zeros(uo, dtype=torch.float32, device=device)
        self.v_new = torch.zeros(vo, dtype=torch.float32, device=device)
        self.sig_scratch = torch.zeros(len(ls), dtype=torch.float32, device=device)
        self.tables = {}
        self.u_dst = [l.mod.u0.view(-1) for l in ls if l.spectral]
        self.u_src = [self.u_new[self.u_off[l.index]:self.u_off[l.index] + l.rows] for l in ls if l.spectral]

    def _table(self, training, need_bwd):
        key = (bool(training), bool(need_bwd))
        if key not in self.tables:
            ls = self.layers
            arr = (L.SnLayer * len(ls))()
            for i, l in enumerate(ls):
                a = arr[i]
                c0, nch, so = self.metas[i]
                a.w = l.weight.data_ptr()
                if l.spectral:
                    a.u_in = l.mod.u0.data_ptr()
                    a.sigma_out = l.mod.sv0.data_ptr() if training else self.sig_scratch.data_ptr() + 4 * i
                a.u_out = self.u_new.data_ptr() + 4 * self.u_off[i]
                a.v_out = self.v_new.data_ptr() + 4 * self.v_off[i]
                a.inv_sigma_out = self.inv_sigma.data_ptr() + 4 * i
                if l.colscale is not None:
                    a.colscale_out, a.colscale_n = l.colscale.data_ptr(), l.rows
                a.pack_fprop = l.wp.data_ptr()
                a.pack_dgrad = l.wd.data_ptr() if need_bwd else None
                a.pack_tc_fprop = ptr(l.wp_tc)
                a.pack_tc_dgrad = ptr(l.wd_tc) if need_bwd else None
                a.pack_tc_rows, a.pack_tc_cin = (l.rows + 15) // 16 * 16, (l.cin + 15) // 16 * 16
                a.rows, a.cin, a.taps, a.pack_dgrad_ld = l.rows, l.cin, l.taps, l.wd_ld
                a.pack_dtype = L.F32 if l.pack_dtype == torch.float32 else L.BF16
                a.spectral = l.spectral
                a.eps = float(l.mod.eps) if l.spectral else 0.0
                a.chunk0, a.nchunks, a.scratch_off = c0, nch, so
            host = torch.frombuffer(bytearray(bytes(arr)), dtype=torch.uint8)
            self.tables[key] = host.to(self.inv_sigma.device)
        return self.tables[key]

    def run(self, training, need_bwd):
        """One grouped power iteration + repack (4 launches for the whole net).  After it the layer
        handles expose wp / wd and, through saved(), THIS call's (1/sigma, u', v): when a backward
        will follow they are snapshots, so two forwards before one backward keep their own values."""
        ls = self.layers
        L.require_device(ls[0].weight)
        sig = self._signature()
        if sig != self.key:
            self._build(ls[0].weight.device)
            self.key = sig
        K("iea_sn_power_iter", ptr(self._table(training, need_bwd)), len(ls), ptr(self.chunks), self.n_chunks,
          ptr(self.scratch), self.max_cols, L.stream(), launches=4)
        if training and self.u_dst:  # u0 <- u' (layers.py:106-107); sv0 was written by the kernel
            torch._foreach_copy_(self.u_dst, self.u_src)
        if need_bwd:
            self.cur = (self.inv_sigma.clone(), self.u_new.clone(), self.v_new.clone())
        else:
            self.cur = (self.inv_sigma, self.u_new, self.v_new)


# ------------------------------------------------------------------ fused conv op
def _desc(n, h, w, cin, cout, k, x_t, x_ptr, x_ld, in_mode, in_relu, scale, shift, wp, out_scale,
          out_scale_stride, bias, res, res_mode, res_c, acc_c0, y_t, y_ptr, y_ld, act, stats, in_bcast=0, wtc=None):
    d = L.ConvDesc()
    d.n, d.h, d.w, d.cin, d.cout, d.ksize = n, h, w, cin, cout, k
    d.x, d.x_dtype, d.x_ld, d.in_mode, d.in_relu = x_ptr, dt(x_t), x_ld, in_mode, int(in_relu)
    d.in_scale, d.in_shift, d.in_bcast = ptr(scale), ptr(shift), in_bcast
    d.wpack, d.w_dtype = wp.data_ptr(), dt(wp)
    d.wpack_tc = ptr(wtc)
    d.cout_tc = (cout + 15) // 16 * 16
    d.out_scale, d.out_scale_stride = ptr(out_scale), out_scale_stride
    d.bias = ptr(bias)
    if res is not None:
        d.res, d.res_dtype, d.res_ld, d.res_mode, d.res_c = res.off(), dt(res.t), res.ld, res_mode, res_c
    d.acc_c0 = acc_c0
    d.y, d.y_dtype, d.y_ld, d.act = y_ptr, dt(y_t), y_ld, act
    d.stats = ptr(stats)
    d.impl = conv_impl()
    return d


class ScaleShift:
    """Per-(image, channel) affine of a batch-norm, consumed by a conv prologue."""
    __slots__ = ("scale", "shift", "dscale", "dshift", "mean", "rstd")

    def __init__(self, scale, shift, mean=None, rstd=None):
        self.scale, self.shift, self.dscale, self.dshift, self.mean, self.rstd = scale, shift, None, None, mean, rstd


def conv(tape, xv, layer, n, h, w, k, *, bias=None, in_mode=L.IN_DIRECT, in_relu=False, ss=None, res=None,
         res_mode=L.IN_DIRECT, res_c=0, acc_c0=-1, out=None, act=L.ACT_NONE, stats=False, out_dtype=None,
         out_shape=None, grouped=None):
    """y = act(conv_k(T(x)) * (1/sigma) + bias + residual); see iea_conv_desc in include/iea_b200.h.
    `layer` is an SNLayer.  grouped = (wp, wd, colscale, cout, layers) runs several layers that share
    the input as one GEMM with a per-output-column 1/sigma (the ccbn gain/bias linears)."""
    cin = xv.c
    dev = xv.t.device
    if grouped is not None:
        wp_t, wd_t, colscale, cout, wls = grouped
        osc, oss = colscale, 1
        wp_tc = wd_tc = None
    else:
        wp_t, wd_t, colscale, cout, wls = layer.wp, layer.wd, None, layer.rows, [layer]
        osc, oss = layer.inv_sigma(), 0
        wp_tc, wd_tc = layer.wp_tc, layer.wd_tc
    if out is None:
        od = out_dtype or act_dtype()
        yv = Var(torch.empty(out_shape or (n, h, w, cout), dtype=od, device=dev))
    else:
        yv = out
    y = yv.t
    M = n * h * w
    scale = ss.scale if ss is not None else None
    shift = ss.shift if ss is not None else None
    d = _desc(n, h, w, cin, cout, k, xv.t, xv.off(), xv.ld, in_mode, in_relu, scale, shift, wp_t, osc, oss,
              bias, res, res_mode, res_c, acc_c0, y, yv.off(), yv.ld, act, None, wtc=wp_tc)
    st, slots = None, 0
    if stats:  # the kernel chosen for this shape decides how many partial-sum slots per event it writes
        d.stats = 1
        slots = call("iea_conv_stats_slots", C.byref(d))
        st = torch.zeros((max(n // IMGS, 1) * slots, cout, 2), dtype=torch.float32, device=dev) if slots > 0 else None
        d.stats = ptr(st)
    K("iea_conv_fprop", C.byref(d), L.stream())
    if TRACE is not None:
        TRACE.append((_tag("iea_conv_fprop", (C.byref(d),)), yv.t, st))
    if stats:
        yv.bn = (st, slots, IMGS * h * w) if slots > 0 else None
    if not tape.record:
        return yv
    saved = [l.saved() for l in wls]

    def fwd_desc():  # the forward geometry / prologue, for wgrad and the prologue backward
        return _desc(n, h, w, cin, cout, k, xv.t, xv.off(), xv.ld, in_mode, in_relu, scale, shift, wp_t,
                     None, 0, None, None, 0, 0, -1, y, yv.off(), yv.ld, 0, None)

    def dgrad_into(g_t, g_ptr, g_ld, dst, dst_ptr, accumulate):
        if colscale is not None:  # per-input-column 1/sigma of the grouped GEMM
            dd = _desc(n, h, w, cout, cin, k, g_t, g_ptr, g_ld, 0, 0, colscale, torch.zeros_like(colscale), wd_t,
                       None, 0, None, None, 0, 0, 0 if accumulate else -1, dst, dst_ptr, cin, 0, None, in_bcast=1)
        else:
            dd = _desc(n, h, w, cout, cin, k, g_t, g_ptr, g_ld, 0, 0, None, None, wd_t, saved[0][0], 0,
                       None, None, 0, 0, 0 if accumulate else -1, dst, dst_ptr, cin, 0, None, wtc=wd_tc)
        K("iea_conv_fprop", C.byref(dd), L.stream())

    def bw_fused_1x1(grid):
        """The whole backward of a same-resolution 1x1 layer in ONE kernel (iea_conv_bwd1x1): statistics adjoint, weight
        and bias gradient, data gradient and prologue adjoint -- g, y and x are read once, dx is written once."""
        g_t = yv.g
        g_ptr, g_ld = yv.off(g_t), yv.ld
        a = L.Bwd1x1Args()
        if yv.ds is not None and res is None:
            ds1, ds2, rpe_ = yv.ds
            a.y, a.y_ld, a.ds1, a.ds2, a.rows_per_event = yv.off(), yv.ld, ptr(ds1), ptr(ds2), rpe_
        elif yv.ds is not None:  # the residual branch needs the statistics-adjusted gradient as a tensor
            ds1, ds2, rpe_ = yv.ds
            geff = torch.empty((M, cout), dtype=g_t.dtype, device=dev)
            K("iea_conv_out_bwd", g_ptr, dt(g_t), g_ld, yv.off(), dt(y), yv.ld, act, ptr(ds1), ptr(ds2), M, rpe_,
              cout, ptr(geff), dt(geff), L.stream())
            g_t, g_ptr, g_ld = geff, geff.data_ptr(), cout
        if a.rows_per_event == 0:
            a.rows_per_event = 1
        if res is not None and res.need:
            rg, beta = _accum_target(res)
            K("iea_residual_bwd", g_ptr, dt(g_t), g_ld, n, h, w, res_c, res_mode, res.off(rg), dt(rg), res.ld,
              res.c, beta, L.stream())
        if yv.sc_var is not None:
            yv.sc_var.g = g_t
        l = wls[0]
        isg, u_, v_ = saved[0]
        need_w = l.weight.requires_grad
        need_db = bias is not None and bias.requires_grad and need_w
        kdim = cin
        keep = [g_t]
        a.g, a.g_ld, a.wd_tc, a.inv_sigma = g_ptr, g_ld, ptr(wd_tc), ptr(isg)
        if need_w:
            wpart = torch.empty((grid + 1) * cout * kdim + grid * cout, dtype=torch.float32, device=dev)
            a.wpart = ptr(wpart)
            keep.append(wpart)
            if need_db:
                db = tape.galloc(bias)[0]
                a.dbias = ptr(db)
        if xv.need:
            xg, beta = _accum_target(xv)
            a.dx, a.dx_ld, a.beta = xv.off(xg), xv.ld, beta
        if ss is not None:
            dsc, dsh = torch.empty_like(ss.scale), torch.empty_like(ss.shift)
            ss.dscale, ss.dshift = dsc, dsh
            dfw0 = fwd_desc()
            scr = _f32(call("iea_conv_bwd1x1_scratch_floats", C.byref(dfw0)), dev)
            a.dscale, a.dshift, a.scratch = ptr(dsc), ptr(dsh), ptr(scr)
        dfw = fwd_desc()
        K("iea_conv_bwd1x1", C.byref(dfw), C.byref(a), L.stream(), launches=1 + (2 if need_db else 1 if need_w else 0) + (1 if ss is not None else 0))
        if need_w:
            dw, beta_w = tape.galloc(l.weight, accumulate_ok=True)
            tape.sn_weight_bwd(wpart[:cout * kdim].view(1, cout, kdim), 1, l, (isg, u_, v_), dw, beta_w)
            tape.pgrad(l.weight, dw)
            if need_db:
                tape.pgrad(bias, db)
        elif bias is not None and bias.requires_grad:
            db = tape.galloc(bias)[0]
            K("iea_colsum", g_ptr, dt(g_t), g_ld, M, cout, ptr(db), 0.0, ptr(_f32(300 * cout, dev)), L.stream(), launches=2)
            tape.pgrad(bias, db)

    def bw():
        if yv.g is None:
            return
        if (k == 1 and in_mode == L.IN_DIRECT and grouped is None and act == L.ACT_NONE and wd_tc is not None
                and yv.g.dtype == torch.bfloat16 and xv.t.dtype == torch.bfloat16 and y.dtype == torch.bfloat16
                and conv_impl() != L.IMPL_GENERIC and (xv.need or ss is not None or wls[0].weight.requires_grad)
                and (res is None or dt(res.t) == L.BF16)):
            dfq = fwd_desc()
            grid = call("iea_conv_bwd1x1_grid", C.byref(dfq))
            if grid > 0:
                return bw_fused_1x1(grid)
        g_t = yv.g
        g_ptr, g_ld = yv.off(g_t), yv.ld
        if yv.ds is not None or act == L.ACT_TANH:
            ds1, ds2, rpe_ = yv.ds if yv.ds is not None else (None, None, 1)
            geff = torch.empty((M, cout), dtype=g_t.dtype, device=dev)
            K("iea_conv_out_bwd", g_ptr, dt(g_t), g_ld, yv.off(), dt(y), yv.ld, act, ptr(ds1), ptr(ds2), M, rpe_,
              cout, ptr(geff), dt(geff), L.stream())
            g_t, g_ptr, g_ld = geff, geff.data_ptr(), cout
        need_db = bias is not None and bias.requires_grad
        db = tape.galloc(bias)[0] if need_db else None
        db_done = False
        if res is not None and res.need:
            rg, beta = _accum_target(res)
            K("iea_residual_bwd", g_ptr, dt(g_t), g_ld, n, h, w, res_c, res_mode, res.off(rg), dt(rg), res.ld,
              res.c, beta, L.stream())
        if yv.sc_var is not None:
            yv.sc_var.g = g_t  # the shortcut conv wrote channels >= acc_c0 of y: same gradient tensor
        if any(l.weight.requires_grad for l in wls):
            kdim = cin * k * k
            dfw = fwd_desc()
            nsplit = call("iea_conv_wgrad_mma_slices", C.byref(dfw), dt(g_t), g_ld) if conv_impl() != L.IMPL_GENERIC else 0
            if nsplit > 0:  # tensor-core split-K over pixel tiles, one partial per (CTA, k-step group)
                gpart = torch.empty((nsplit, cout, kdim), dtype=torch.float32, device=dev)
                # (the same pass also sums g over the pixels: the bias gradient, when asked for)
                db_done = K("iea_conv_wgrad_mma", C.byref(dfw), g_ptr, dt(g_t), g_ld, ptr(gpart), ptr(db), L.stream(),
                            launches=3 if need_db else 2) == 1
                gpart, nsplit = gpart[:1], 1  # slice 0 now holds the sum of the per-CTA partials
            else:
                nsplit = max(1, min(64, M // 4096))
                gpart = torch.empty((nsplit, cout, kdim), dtype=torch.float32, device=dev)
                K("iea_conv_wgrad", C.byref(dfw), g_ptr, dt(g_t), g_ld, ptr(gpart), nsplit, L.stream())
            r0 = 0
            for l, (isg, u_, v_) in zip(wls, saved):
                if l.weight.requires_grad:
                    dw, beta = tape.galloc(l.weight, accumulate_ok=True)
                    gp = gpart if len(wls) == 1 else gpart[:, r0:r0 + l.rows].contiguous()
                    tape.sn_weight_bwd(gp, nsplit, l, (isg, u_, v_), dw, beta)
                    tape.pgrad(l.weight, dw)
                r0 += l.rows
        if need_db:
            if not db_done:
                K("iea_colsum", g_ptr, dt(g_t), g_ld, M, cout, ptr(db), 0.0, ptr(_f32(300 * cout, dev)), L.stream(),
                  launches=2)
            tape.pgrad(bias, db)
        plain = in_mode == L.IN_DIRECT and not in_relu and ss is None and xv.c == xv.ld
        if xv.need and plain:
            xg, beta = _accum_target(xv)
            dgrad_into(g_t, g_ptr, g_ld, xg, xg.data_ptr(), beta != 0.0)
        elif xv.need or ss is not None:
            da = torch.empty((M, cin), dtype=act_dtype(), device=dev)
            dgrad_into(g_t, g_ptr, g_ld, da, da.data_ptr(), False)
            xg, beta, xg_ptr = None, 0.0, None
            if xv.need:
                xg, beta = _accum_target(xv)
                xg_ptr = xv.off(xg)
            dsc = dsh = None
            if ss is not None:
                dsc, dsh = torch.empty_like(ss.scale), torch.empty_like(ss.shift)
                ss.dscale, ss.dshift = dsc, dsh
            dfw = fwd_desc()
            K("iea_conv_input_bwd", C.byref(dfw), ptr(da), dt(da), xg_ptr, dt(xg) if xg is not None else 0, xv.ld,
              beta, ptr(dsc), ptr(dsh), ptr(_f32(n * 64 * cin * 2, dev)), L.stream(), launches=2)
    tape.add(bw)
    return yv


# ------------------------------------------------------------------ batch norm glue
def ensure_stats(xv, n, h, w):
    """Batch-norm partial sums of xv: from the producer's epilogue when present, else one
    stand-alone pass."""
    if xv.bn is None:
        rpe = IMGS * h * w
        tiles = max(1, min(64, rpe // 512))
        part = torch.empty((n // IMGS, tiles, xv.c, 2), dtype=torch.float32, device=xv.t.device)
        K("iea_bn_stats", xv.off(), dt(xv.t), xv.ld, n * h * w, rpe, xv.c, tiles, ptr(part), L.stream())
        xv.bn = (part, tiles, rpe)
    return xv.bn


def _ticket(owner, c, dev):
    """Per-layer self-resetting counters of the one-launch finalize (caller-owned: include/iea_b200.h)."""
    t = owner.__dict__.get("_iea_ticket") if owner is not None else None
    if t is None or t.device != dev or t.numel() < cdiv(c, 8):
        t = torch.zeros(cdiv(c, 8), dtype=torch.int32, device=dev)
        if owner is not None:
            owner.__dict__["_iea_ticket"] = t
    return t


def bn_affine(tape, xv, n, h, w, *, gain, gain_ld, gain_add, bias, bias_ld, stored_mean, stored_var, training,
              eps, momentum=0.1, dgain=None, dbias=None, dgb_ld=0, gain_param=None, bias_param=None, owner=None,
              mode=None):
    """Finalize the batch statistics of xv into a per-(n,c) ScaleShift (layers.py:656-689, 728-742).
    ccbn: gain/bias are raw device addresses of column windows of the grouped-GEMM output (row
    stride gain_ld) and dgain/dbias the matching windows of its gradient buffer; plain bn:
    gain_param/bias_param are the (C,) parameters."""
    c, dev, events = xv.c, xv.t.device, n // IMGS
    part, tiles, count = ensure_stats(xv, n, h, w) if training else (None, 0, IMGS * h * w)
    scale = torch.empty((n, c), dtype=torch.float32, device=dev)
    shift = torch.empty((n, c), dtype=torch.float32, device=dev)
    mean = torch.empty((events, c), dtype=torch.float32, device=dev)
    rstd = torch.empty((events, c), dtype=torch.float32, device=dev)
    K("iea_bn_finalize", ptr(part), events, tiles, count, IMGS, c, gain, gain_ld, gain_add, bias, bias_ld,
      ptr(stored_mean), ptr(stored_var), int(training) if mode is None else mode, momentum, eps, ptr(mean), ptr(rstd),
      ptr(scale), ptr(shift), ptr(_ticket(owner, c, dev)) if training else None, L.stream())
    ss = ScaleShift(scale, shift, mean, rstd)
    if tape.record:
        def bw():
            if ss.dscale is None:
                return
            ds1 = torch.empty((events, c), dtype=torch.float32, device=dev)
            ds2 = torch.empty((events, c), dtype=torch.float32, device=dev)
            if gain_param is not None:
                dg = torch.empty(c, dtype=torch.float32, device=dev)
                db = torch.empty(c, dtype=torch.float32, device=dev)
                K("iea_bn_finalize_bwd", ptr(ss.dscale), ptr(ss.dshift), ptr(scale), ptr(mean), ptr(rstd), events,
                  IMGS, count, c, gain, gain_ld, gain_add, ptr(dg), 0, ptr(db), 0, 1, int(training), ptr(ds1),
                  ptr(ds2), L.stream())
                if gain_param.requires_grad:
                    tape.pgrad(gain_param, dg)
                if bias_param.requires_grad:
                    tape.pgrad(bias_param, db)
            else:
                K("iea_bn_finalize_bwd", ptr(ss.dscale), ptr(ss.dshift), ptr(scale), ptr(mean), ptr(rstd), events,
                  IMGS, count, c, gain, gain_ld, gain_add, dgain, dgb_ld, dbias, dgb_ld, 0, int(training),
                  ptr(ds1), ptr(ds2), L.stream())
            if training and xv.need:
                xv.ds = (ds1, ds2, count)
        tape.add(bw)
    return ss


# ------------------------------------------------------------------ small ops with tape
def layernorm(tape, xv, ln):
    x = xv.t
    rows, dim = x.shape[0], x.shape[-1]
    y = torch.empty_like(x)
    mean, rstd = _f32(rows, x.device), _f32(rows, x.device)
    K("iea_layernorm_fwd", ptr(x), ptr(ln.weight), ptr(ln.bias), rows, dim, ln.eps, ptr(y), ptr(mean), ptr(rstd),
      L.stream())
    yv = Var(y)
    if tape.record:
        def bw():
            if yv.g is None:
                return
            need_p = ln.weight.requires_grad
            dx = torch.empty_like(x)
            dg = _f32(dim, x.device) if need_p else None
            db = _f32(dim, x.device) if need_p else None
            K("iea_layernorm_bwd", ptr(yv.g), ptr(x), ptr(ln.weight), ptr(mean), ptr(rstd), rows, dim, ptr(dx),
              ptr(dg), ptr(db), 1, L.stream(), launches=2)
            if need_p:
                tape.pgrad(ln.weight, dg)
                tape.pgrad(ln.bias, db)
            if xv.need:
                add_grad(xv, dx)
        tape.add(bw)
    return yv


def mha_core(tape, qkvv, events, seq, heads, d):
    qkv = qkvv.t
    val = torch.empty((events * seq, heads * d), dtype=torch.float32, device=qkv.device)
    att = torch.empty((events, heads, seq, seq), dtype=torch.float32, device=qkv.device)
    K("iea_mha_fwd", ptr(qkv), events, seq, heads, d, ptr(val), ptr(att), L.stream())
    vv = Var(val)
    if tape.record:
        def bw():
            if vv.g is None:
                return
            dq = torch.empty_like(qkv)
            K("iea_mha_bwd", ptr(vv.g), ptr(qkv), ptr(att), events, seq, heads, d, ptr(dq), L.stream())
            add_grad(qkvv, dq)
        tape.add(bw)
    return vv, att


TC_LINEAR_MIN_ROWS = 2048  # feature matrices with at least this many rows go to the tcgen05 GEMM


def _cast(tape, xv, dtype, add=None):
    """y = dtype(x) [+ add] as one pass (iea_axpby); backward casts the gradient back (and feeds `add`)."""
    x = xv.t
    y = torch.empty(x.shape, dtype=dtype, device=x.device)
    b = add.t if add is not None else x
    K("iea_axpby", ptr(x), dt(x), 1.0, ptr(b), dt(b), 1.0 if add is not None else 0.0, ptr(y), dt(y), x.numel(), L.stream())
    yv = Var(y)
    if tape.record:
        def bw():
            if yv.g is None:
                return
            if xv.need:
                g = torch.empty(x.shape, dtype=x.dtype, device=x.device)
                K("iea_axpby", ptr(yv.g), dt(yv.g), 1.0, ptr(yv.g), dt(yv.g), 0.0, ptr(g), dt(g), g.numel(), L.stream())
                add_grad(xv, g)
            if add is not None and add.need:
                add_grad(add, yv.g if add.g is not None else yv.g.clone())
        tape.add(bw)
    return yv


def _linear_tc_ok(xv, layer, out_dtype):
    n = xv.t.shape[0]
    cout, cin = layer.rows, layer.cin
    return (n >= TC_LINEAR_MIN_ROWS and layer.wp_tc is not None and act_dtype() == torch.bfloat16
            and conv_impl() != L.IMPL_GENERIC and xv.t.dtype == torch.float32 and out_dtype == torch.float32
            and xv.c == xv.ld and cin % 64 == 0 and ((cout <= 256 and cout % 16 == 0) or cout % 256 == 0))


def linear(tape, xv, layer, *, bias=None, in_relu=False, res=None, out_dtype=torch.float32):
    """F.linear(x, W/sigma, b) [+ residual] on a (rows, K) feature matrix: the 1x1 conv with h=w=1.
    Few rows (one to a few dozen events): fp32 CUDA-core kernels (weight-read bound, cluster split-K).  From
    TC_LINEAR_MIN_ROWS rows on (the 256-event RRM sweep: 10240 x 512 x 1536) the product is a real GEMM and runs
    on the tcgen05 kernel: bf16 operands, fp32 accumulation in TMEM, fp32 features in and out."""
    n = xv.t.shape[0]
    if _linear_tc_ok(xv, layer, out_dtype):
        yb = conv(tape, _cast(tape, xv, torch.bfloat16), layer, n, 1, 1, 1, bias=bias, in_relu=in_relu,
                  out_dtype=torch.bfloat16, out_shape=(n, layer.rows))
        return _cast(tape, yb, torch.float32, add=res)
    return conv(tape, xv, layer, n, 1, 1, 1, bias=bias, in_relu=in_relu, res=res,
                res_c=layer.rows if res is not None else 0, out_dtype=out_dtype, out_shape=(n, layer.rows))


def rrm(tape, xv, blocks, final_norm, sn):
    """RelationalReasoning.forward on rows grouped by event: x (40E, dim) fp32 (RRM.py:98-125)."""
    events = xv.t.shape[0] // IMGS
    for blk in blocks:
        at = blk.self_attn
        h1 = layernorm(tape, xv, blk.norm1)
        qkv = linear(tape, h1, sn[at.qkv_proj], bias=at.qkv_proj.bias)
        val, _ = mha_core(tape, qkv, events, IMGS, at.num_heads, at.head_dim)
        x1 = linear(tape, val, sn[at.o_proj], bias=at.o_proj.bias, res=xv)
        h2 = layernorm(tape, x1, blk.norm2)
        l0, l3 = blk.linear_net[0], blk.linear_net[3]
        f = linear(tape, h2, sn[l0], bias=l0.bias)
        xv = linear(tape, f, sn[l3], bias=l3.bias, in_relu=True, res=x1)  # ReLU fused as the prologue
    if final_norm is not None:
        xv = layernorm(tape, xv, final_norm)
    return xv


def cat_cols(tape, a, b):
    """torch.cat([a, b], 1) on small fp32 feature matrices (host-side plumbing)."""
    v = Var(torch.cat([a.t, b.t], 1))
    if tape.record:
        ca = a.t.shape[1]

        def bw():
            if v.g is None:
                return
            if a.need:
                add_grad(a, v.g[:, :ca].contiguous())
            if b.need:
                add_grad(b, v.g[:, ca:].contiguous())
        tape.add(bw)
    return v


def embedding(tape, idx, weight, sn_layer=None):
    """F.embedding(idx, W [/sigma]) (model.py:462; layers.py:259 for the SN variant)."""
    n, dim = idx.shape[0], weight.shape[1]
    scale = sn_layer.inv_sigma() if sn_layer is not None else None
    out = torch.empty((n, dim), dtype=torch.float32, device=weight.device)
    K("iea_embedding_fwd", ptr(idx), ptr(weight), ptr(scale), n, dim, ptr(out), L.stream())
    v = Var(out)
    if tape.record and weight.requires_grad:
        saved = sn_layer.saved() if sn_layer is not None else None

        def bw():
            if v.g is None:
                return
            G = torch.empty_like(weight)  # gradient w.r.t. the normalised table
            K("iea_embedding_bwd", ptr(idx), ptr(v.g), None, n, dim, weight.shape[0], ptr(G), L.stream())
            if saved is not None:
                dw = torch.empty_like(weight)
                K("iea_sn_weight_bwd", ptr(G), 1, ptr(weight), ptr(saved[1]), ptr(saved[2]), ptr(saved[0]), 1,
                  ptr(dw), 0.0, weight.shape[0], dim, 1, ptr(_f32(520, weight.device)), L.stream(), launches=2)
                G = dw
            tape.pgrad(weight, G)
        tape.add(bw)
    return v


def nchw_to_nhwc(tape, xv, n, c, hh, ww):
    """(n, c*hh*ww) features viewed NCHW by the reference (model.py:477-479) -> NHWC activation."""
    src = xv.t
    out = torch.empty((n, hh, ww, c), dtype=act_dtype(), device=src.device)
    K("iea_nchw_to_nhwc", ptr(src), dt(src), ptr(out), dt(out), n, c, hh * ww, L.stream())
    ov = Var(out)
    if tape.record:
        def bw():
            if ov.g is None:
                return
            g = ov.g
            if ov.ds is not None:
                ds1, ds2, rpe = ov.ds
                ge = torch.empty_like(g)
                K("iea_conv_out_bwd", ptr(g), dt(g), c, ptr(out), dt(out), c, 0, ptr(ds1), ptr(ds2), n * hh * ww,
                  rpe, c, ptr(ge), dt(ge), L.stream())
                g = ge
            dx = torch.empty((n, c * hh * ww), dtype=torch.float32, device=src.device)
            K("iea_nhwc_to_nchw", ptr(g), dt(g), ptr(dx), L.F32, n, c, hh * ww, L.stream())
            add_grad(xv, dx)
        tape.add(bw)
    return ov


# ------------------------------------------------------------------ Generator
class GPlan:
    """Static per-Generator schedule: the SN group and the grouped ccbn GEMM layout."""

    def __init__(self, G):
        from . import sn_layers as SL
        self.sn = SNGroup()
        self.h = {}
        big = act_dtype()
        self.h[G.linear_f] = self.sn.add(G.linear_f, torch.float32)
        for blk in G.RR_G.layers:
            for m in (blk.self_attn.qkv_proj, blk.self_attn.o_proj, blk.linear_net[0], blk.linear_net[3]):
                self.h[m] = self.sn.add(m, torch.float32)
        self.h[G.linear] = self.sn.add(G.linear, big)
        self.ccbn = []
        for bl in G.blocks:
            for m in bl:
                if isinstance(m, SL.Attention):
                    raise NotImplementedError("G_attn: the shipped config has no attention in G (config.json:27)")
                for cv in (m.conv1, m.conv2, m.conv3, m.conv4):
                    self.h[cv] = self.sn.add(cv, big)
                self.ccbn += [m.bn1, m.bn2, m.bn3, m.bn4]
        oc = G.output_layer[2]
        self.h[oc] = self.sn.add(oc, big)
        mods, off, self.gb_off = [], 0, {}
        for b in self.ccbn:
            self.gb_off[b] = (off, off + b.output_size)
            off += 2 * b.output_size
            mods += [b.gain, b.bias]
        self.gb_cols = off
        self.gb_layers = self.sn.add_shared(mods, torch.float32)
        for m, l in zip(mods, self.gb_layers):
            self.h[m] = l


def _plan(net, cls):
    p = net.__dict__.get("_iea_plan")
    if p is None or p[0] != act_dtype():
        p = (act_dtype(), cls(net))
        net.__dict__["_iea_plan"] = p
    return p[1]


def bn_state(bnm):
    """(stored_mean, stored_var, mode, owner) of a ccbn / bn module: F.batch_norm running statistics
    (layers.py:664-673, 733-742) or, with mybn=True, the myBN child's (layers.py:547-599: biased variance,
    optional standing-statistics accumulation; eval divides standing sums by the counter)."""
    if not getattr(bnm, "mybn", False):
        return bnm.stored_mean, bnm.stored_var, int(bnm.training), bnm
    b = bnm.bn
    if bnm.training:
        if b.accumulate_standing:
            b.accumulation_counter += 1.0
        return b.stored_mean, b.stored_var, (1 | 4) if b.accumulate_standing else (1 | 2), b
    if b.accumulate_standing:
        return b.stored_mean / b.accumulation_counter, b.stored_var / b.accumulation_counter, 0, b
    return b.stored_mean, b.stored_var, 0, b


def _gblock(tape, blk, x, n, hh, ww, plan, gb, dgb, training):
    """One bottleneck GBlock as 4 fused convs (model.py:54-71): every ccbn+ReLU(+upsample) is the
    prologue of the conv that consumes it, every conv's epilogue emits the next BN's statistics, and
    the channel-dropped (upsampled) skip is the epilogue residual of conv4."""
    h_ = plan.h
    up = blk.upsample is not None
    gld = plan.gb_cols

    def aff(bnm, xv, h, w):
        g0, b0 = plan.gb_off[bnm]
        sm, sv, mode, owner = bn_state(bnm)
        return bn_affine(tape, xv, n, h, w, gain=gb.data_ptr() + 4 * g0, gain_ld=gld, gain_add=1.0,
                         bias=gb.data_ptr() + 4 * b0, bias_ld=gld, stored_mean=sm,
                         stored_var=sv, training=training, eps=bnm.eps, owner=owner, mode=mode,
                         momentum=bnm.momentum if getattr(bnm, "mybn", False) else 0.1,  # layers.py:671 hard-codes 0.1
                         dgain=(dgb.data_ptr() + 4 * g0) if dgb is not None else None,
                         dbias=(dgb.data_ptr() + 4 * b0) if dgb is not None else None, dgb_ld=gld)
    h1 = conv(tape, x, h_[blk.conv1], n, hh, ww, 1, bias=blk.conv1.bias, in_relu=True,
              ss=aff(blk.bn1, x, hh, ww), stats=True)
    ho, wo = (hh * 2, ww * 2) if up else (hh, ww)
    h2 = conv(tape, h1, h_[blk.conv2], n, ho, wo, 3, bias=blk.conv2.bias, in_relu=True,
              ss=aff(blk.bn2, h1, hh, ww), in_mode=L.IN_UP2 if up else L.IN_DIRECT, stats=True)
    h3 = conv(tape, h2, h_[blk.conv3], n, ho, wo, 3, bias=blk.conv3.bias, in_relu=True,
              ss=aff(blk.bn3, h2, ho, wo), stats=True)
    out = conv(tape, h3, h_[blk.conv4], n, ho, wo, 1, bias=blk.conv4.bias, in_relu=True,
               ss=aff(blk.bn4, h3, ho, wo), res=x, res_mode=L.IN_UP2 if up else L.IN_DIRECT,
               res_c=blk.out_channels, stats=True)
    return out, ho, wo


def _g_body(G, tape, z, y, rdof):
    plan = _plan(G, GPlan)
    sn, h_ = plan.sn, plan.h
    training = G.training
    n = z.t.shape[0]
    if n % IMGS:
        raise ValueError("a batch of %d rows is not a whole number of 40-image events" % n)
    sn.run(training, tape.record)
    emb = embedding(tape, y, G.shared.weight)
    c = cat_cols(tape, emb, Var(rdof, need=False))
    c = linear(tape, c, h_[G.linear_f], bias=G.linear_f.bias)
    c = rrm(tape, c, G.RR_G.layers, G.RR_G.norm, h_)
    cond = cat_cols(tape, c, z)  # hier: the same 256-vector conditions every ccbn (model.py:471-473)
    # all ccbn gain/bias linears as ONE GEMM: (40E x 256) . (256 x sum 2C), per-column 1/sigma
    wp, wd, cs = sn.colscales[0]
    gbv = conv(tape, cond, None, n, 1, 1, 1, out_dtype=torch.float32, out_shape=(n, plan.gb_cols),
               grouped=(wp, wd, cs, plan.gb_cols, plan.gb_layers))
    gb, dgb = gbv.t, None
    if tape.record:
        dgb = torch.zeros_like(gb)  # the bn backward kernels write their (dgain, dbias) windows into it
        gbv.g = dgb
    bwid, hb = G.bottom_width, G.H_base
    hh, ww = bwid, bwid * hb
    lin = linear(tape, cond, h_[G.linear], bias=G.linear.bias)
    h = nchw_to_nhwc(tape, lin, n, G.arch["in_channels"][0], hh, ww)
    for bl in G.blocks:
        for blk in bl:
            h, hh, ww = _gblock(tape, blk, h, n, hh, ww, plan, gb, dgb, training)
    obn, oconv = G.output_layer[0], G.output_layer[2]
    sm, sv, mode, owner = bn_state(obn)
    ss = bn_affine(tape, h, n, hh, ww, gain=ptr(obn.gain), gain_ld=0, gain_add=0.0, bias=ptr(obn.bias), bias_ld=0,
                   stored_mean=sm, stored_var=sv, training=training, eps=obn.eps,
                   momentum=obn.momentum, gain_param=obn.gain, bias_param=obn.bias, owner=owner, mode=mode)
    img = conv(tape, h, h_[oconv], n, hh, ww, 3, bias=oconv.bias, in_relu=True, ss=ss, act=L.ACT_TANH,
               out_dtype=torch.float32)
    return img, hh, ww


# ------------------------------------------------------------------ autograd bridge
class _NetFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, body, n_in, owner, *args):
        flat = None
        if owner is not None and len(args) > n_in:
            from .optim import FlatGrads
            flat = FlatGrads.of(owner)
        tape = Tape(True, flat)
        in_vars = [Var(a, need=bool(a.requires_grad)) for a in args[:n_in]]
        outs = body(tape, *in_vars)
        ctx.tape, ctx.in_vars, ctx.outs, ctx.params, ctx.n_in, ctx.owner = tape, in_vars, outs, args[n_in:], n_in, owner
        res = tuple(o.t for o in outs)
        return res if len(res) > 1 else res[0]

    @staticmethod
    def backward(ctx, *gouts):
        tape = ctx.tape
        if tape is None:
            raise RuntimeError("iea_gan_b200: a net call can be back-propagated only once")
        for o, g in zip(ctx.outs, gouts):
            if g is not None:
                o.g = g.contiguous().to(o.t.dtype).view(o.t.shape)
        tape.backward()
        gin = [v.g.view(v.t.shape) if (v.need and v.g is not None and ctx.needs_input_grad[3 + i]) else None
               for i, v in enumerate(ctx.in_vars)]
        # gradients written in place into the net's flat buffer (param.grad is already that view) are not handed to
        # autograd a second time
        gp = [tape.pgrads.get(id(p)) if (ctx.needs_input_grad[3 + ctx.n_in + j] and id(p) not in tape.direct) else None
              for j, p in enumerate(ctx.params)]
        ctx.tape = None
        owner = ctx.owner
        if owner is not None and tape.direct:
            sync = owner.__dict__.get("_iea_grad_sync")
            if sync is not None:
                sync.after_backward(owner)  # data-parallel: all-reduce the flat buffer at the end of this backward pass
        return (None, None, None) + tuple(gin) + tuple(gp)


def run_net(body, inputs, params, owner=None):
    """Execute body(tape, *in_vars) -> [Var] with a tape (under autograd) or without one.
    owner: the Generator / Discriminator whose parameters these are -- its gradients then live in one flat
    buffer (optim.FlatGrads) that the kernels write in place."""
    record = torch.is_grad_enabled() and (any(a.requires_grad for a in inputs) or any(p.requires_grad for p in params))
    if record:
        return _NetFn.apply(body, len(inputs), owner, *inputs, *params)
    with torch.no_grad():
        outs = body(Tape(False), *[Var(a, need=False) for a in inputs])
    res = tuple(o.t for o in outs)
    return res if len(res) > 1 else res[0]


def _params(net):
    """Cached parameter list of a whole net (the module-tree walk costs ~1 ms per call)."""
    ps = net.__dict__.get("_iea_params")
    if ps is None:
        ps = net.__dict__["_iea_params"] = list(net.parameters())
    return ps


def _plain(t, dtype=torch.float32):
    if type(t) is not torch.Tensor:
        t = t.as_subclass(torch.Tensor)  # utils.Distribution instances flow in from train_fns.py
    return t.contiguous() if t.dtype == dtype else t.to(dtype).contiguous()


@on_tensor_device
def generator_forward(G, z, y):
    z = _plain(z)
    L.require_device(z)
    n = z.shape[0]
    # same draw as model.py:466: torch.randn on the device generator before anything else (40E rows)
    rdof = noise.randn(n, G.rdof_dim, z.device)
    y = _plain(y, torch.int64)
    geo = {}

    def body(tape, zv):
        img, hh, ww = _g_body(G, tape, zv, y, rdof)
        geo["hw"] = (hh, ww)
        return [img]
    out = run_net(body, [z], _params(G), owner=G)
    return out.view(n, 1, *geo["hw"])  # one channel: NHWC and NCHW coincide


@on_tensor_device
def adu_postprocess(img):
    n, _, h, w = img.shape
    img = img.contiguous()
    out = torch.empty((n, h - 6, w), dtype=torch.float32, device=img.device)
    K("iea_adu_postprocess", ptr(img), n, h, w, ptr(out), L.stream())
    return out


# ------------------------------------------------------------------ Discriminator ops
def avgpool2_into(tape, xv, out, n, hh, ww):
    """nn.AvgPool2d(2) of xv (n x hh x ww) written into the channel window `out` of a (n x hh/2 x ww/2) tensor.
    Backward: the un-pooling adjoint of out's gradient, accumulated onto xv's (iea_residual_bwd, POOL2 mode)."""
    c = xv.c
    K("iea_avgpool2_fwd", xv.off(), dt(xv.t), n, hh, ww, c, xv.ld, out.off(), out.ld, L.stream())
    if tape.record and xv.need:
        def bw():
            if out.g is None:
                return
            rg, beta = _accum_target(xv)
            K("iea_residual_bwd", out.off(out.g), dt(out.g), out.ld, n, hh // 2, ww // 2, c, L.IN_POOL2, xv.off(rg), dt(rg),
              xv.ld, xv.c, beta, L.stream())
        tape.add(bw)
    return out


def maxpool2(tape, xv, n, hh, ww):
    c = xv.c
    y = torch.empty((n, hh // 2, ww // 2, c), dtype=xv.t.dtype, device=xv.t.device)
    idx = torch.empty((n, hh // 2, ww // 2, c), dtype=torch.uint8, device=xv.t.device)
    K("iea_maxpool2_fwd", ptr(xv.t), dt(xv.t), n, hh, ww, c, ptr(y), ptr(idx), L.stream())
    yv = Var(y)
    if tape.record:
        def bw():
            if yv.g is None:
                return
            dx = torch.empty_like(xv.t)
            K("iea_maxpool2_bwd", ptr(yv.g), dt(yv.g), ptr(idx), n, hh, ww, c, ptr(dx), L.stream())
            add_grad(xv, dx)
        tape.add(bw)
    return yv


def attn_core(tape, th, ph, gv, n, hw, hwk, ck, cv):
    o = torch.empty((n, hw, cv), dtype=th.t.dtype, device=th.t.device)
    lse = _f32(n * hw, th.t.device)
    K("iea_attn_fwd", ptr(th.t), ptr(ph.t), ptr(gv.t), dt(th.t), n, hw, hwk, ck, cv, ptr(o), ptr(lse), L.stream())
    ov = Var(o)
    if tape.record:
        def bw():
            if ov.g is None:
                return
            dth, dph, dg = torch.empty_like(th.t), torch.empty_like(ph.t), torch.empty_like(gv.t)
            K("iea_attn_bwd", ptr(ov.g), ptr(th.t), ptr(ph.t), ptr(gv.t), ptr(o), ptr(lse), dt(o), n, hw, hwk, ck,
              cv, ptr(dth), ptr(dph), ptr(dg), ptr(_f32(n * hw, o.device)), L.stream(), launches=2)
            add_grad(th, dth)
            add_grad(ph, dph)
            add_grad(gv, dg)
        tape.add(bw)
    return ov


def gamma_residual(tape, ov, xv, gamma):
    y = torch.empty_like(xv.t)
    K("iea_gamma_residual", ptr(ov.t), ptr(xv.t), dt(xv.t), ptr(gamma), ptr(y), y.numel(), L.stream())
    yv = Var(y)
    if tape.record:
        def bw():
            if yv.g is None:
                return
            do = torch.empty_like(ov.t)
            dgm = _f32(1, y.device)
            K("iea_gamma_residual_bwd", ptr(yv.g), ptr(ov.t), dt(y), ptr(gamma), ptr(do), ptr(dgm),
              ptr(_f32(600, y.device)), y.numel(), L.stream(), launches=2)
            if gamma.requires_grad:
                tape.pgrad(gamma, dgm.view(gamma.shape))
            add_grad(ov, do)
            if xv.need:
                add_grad(xv, yv.g if xv.g is not None else yv.g.clone())
        tape.add(bw)
    return yv


def relu_sumpool(tape, xv, n, hw):
    c = xv.c
    out = torch.empty((n, c), dtype=torch.float32, device=xv.t.device)
    K("iea_relu_sumpool_fwd", ptr(xv.t), dt(xv.t), n, hw, c, ptr(out), L.stream())
    ov = Var(out)
    if tape.record:
        def bw():
            if ov.g is None or not xv.need:
                return
            dx = torch.empty_like(xv.t)
            K("iea_relu_sumpool_bwd", ptr(xv.t), dt(xv.t), ptr(ov.g), n, hw, c, ptr(dx), dt(dx), L.stream())
            add_grad(xv, dx)
        tape.add(bw)
    return ov


def l2norm(tape, xv, eps=1e-12):
    x = xv.t
    rows, dim = x.shape
    y, nrm = torch.empty_like(x), _f32(rows, x.device)
    K("iea_l2norm_fwd", ptr(x), rows, dim, eps, ptr(y), ptr(nrm), L.stream())
    yv = Var(y)
    if tape.record:
        def bw():
            if yv.g is None or not xv.need:
                return
            dx = torch.empty_like(x)
            K("iea_l2norm_bwd", ptr(yv.g), ptr(y), ptr(nrm), rows, dim, eps, ptr(dx), L.stream())
            add_grad(xv, dx)
        tape.add(bw)
    return yv


class DPlan:
    def __init__(self, D):
        from . import sn_layers as SL
        self.sn = SNGroup()
        self.h = {}
        big = act_dtype()
        add = lambda m, d: self.h.__setitem__(m, self.sn.add(m, d))
        add(D.input_conv, big)
        for stage in D.blocks:
            for m in stage:
                if isinstance(m, SL.Attention):
                    for cv in (m.theta, m.phi, m.g, m.o):
                        add(cv, big)
                else:
                    for cv in (m.conv1, m.conv2, m.conv3, m.conv4):
                        add(cv, big)
                    if m.learnable_sc:
                        add(m.conv_sc, big)
        add(D.linear0, torch.float32)
        for blk in D.RR_D.layers:
            for m in (blk.self_attn.qkv_proj, blk.self_attn.o_proj, blk.linear_net[0], blk.linear_net[3]):
                self.h[m] = self.sn.add(m, torch.float32, tc=True)
        self.h[D.linear1] = self.sn.add(D.linear1, torch.float32, tc=True)
        add(D.embed, torch.float32)


def _dblock(tape, blk, x, n, hh, ww, h_):
    """Bottleneck DBlock as fused convs (model.py:541-557): the pre-activation ReLUs and the
    AvgPool2d are conv prologues, the concat shortcut is written straight into the channel window
    [Cin, Cout) of the output by conv_sc and the pooled identity half is conv4's epilogue residual."""
    down = blk.downsample is not None
    cin, cout = blk.in_channels, blk.out_channels
    h1 = conv(tape, x, h_[blk.conv1], n, hh, ww, 1, bias=blk.conv1.bias, in_relu=blk.preactivation)
    h2 = conv(tape, h1, h_[blk.conv2], n, hh, ww, 3, bias=blk.conv2.bias, in_relu=True)
    h3 = conv(tape, h2, h_[blk.conv3], n, hh, ww, 3, bias=blk.conv3.bias, in_relu=True)
    ho, wo = (hh // 2, ww // 2) if down else (hh, ww)
    mode = L.IN_POOL2 if down else L.IN_DIRECT
    if down and blk.learnable_sc and _env(b"IEA_DBLOCK_POOL_ONCE", "IEA_DBLOCK_POOL_ONCE", "0") == "1":
        # OPT-IN (IEA_DBLOCK_POOL_ONCE=1): the shortcut torch.cat([pool(x), conv_sc(pool(x))], 1) as ONE tensor R.  x is
        # pooled once into R[..., :cin] (by default it is gathered 2x2 twice, by conv_sc's prologue and by conv4's residual
        # read), conv_sc reads that window at the low resolution and writes R[..., cin:], conv4 takes R as a plain
        # same-resolution residual (its fast epilogue), and the backward un-pools once.  148.0 -> 142.8 ms per 8-event
        # train step and exact with fp32 activations (tests/test_gpu_discriminator.py) -- but with bf16 activations the
        # identity half is rounded BEFORE the add, and the attention theta / phi gradients of the full-size net (the most
        # rounding-sensitive tensors of D at random init) move from 12-15 % to 39-42 % off the fp32 CPU restatement, everything
        # else unchanged (tools/dbg/d_parity.py).  Not the default for that reason.
        R = Var(torch.empty((n, ho, wo, cout), dtype=act_dtype(), device=x.t.device))
        xp, scv = Var(R.t, c0=0, c=cin), Var(R.t, c0=cin, c=cout - cin)
        avgpool2_into(tape, x, xp, n, hh, ww)
        conv(tape, xp, h_[blk.conv_sc], n, ho, wo, 1, bias=blk.conv_sc.bias, out=scv)
        if tape.record:
            def link():  # conv4's backward has produced R's gradient: both windows read / extend it
                xp.g = R.g
                scv.g = R.g
            tape.add(link)
        y = conv(tape, h3, h_[blk.conv4], n, ho, wo, 1, bias=blk.conv4.bias, in_relu=True, in_mode=mode, res=R,
                 res_mode=L.IN_DIRECT, res_c=cout)
        return y, ho, wo
    y = Var(torch.empty((n, ho, wo, cout), dtype=act_dtype(), device=x.t.device))
    if blk.learnable_sc:
        scv = Var(y.t, c0=cin, c=cout - cin)
        conv(tape, x, h_[blk.conv_sc], n, ho, wo, 1, bias=blk.conv_sc.bias, in_mode=mode, out=scv)
        y.sc_var = scv
    conv(tape, h3, h_[blk.conv4], n, ho, wo, 1, bias=blk.conv4.bias, in_relu=True, in_mode=mode, res=x,
         res_mode=mode, res_c=cin, acc_c0=cin if blk.learnable_sc else -1, out=y)
    return y, ho, wo


def _attention(tape, m, x, n, hh, ww, h_):
    """layers.py:283-300 with the attention map kept on chip (iea_attn_fwd / iea_attn_bwd)."""
    ck, cv = m.ch // 8, m.ch // 2
    th = conv(tape, x, h_[m.theta], n, hh, ww, 1)
    ph = maxpool2(tape, conv(tape, x, h_[m.phi], n, hh, ww, 1), n, hh, ww)
    gv = maxpool2(tape, conv(tape, x, h_[m.g], n, hh, ww, 1), n, hh, ww)
    oc = attn_core(tape, th, ph, gv, n, hh * ww, hh * ww // 4, ck, cv)
    o = conv(tape, oc, h_[m.o], n, hh, ww, 1)
    return gamma_residual(tape, o, x, m.gamma)


def _d_body(D, tape, xv, y, hh, ww):
    from . import sn_layers as SL
    plan = _plan(D, DPlan)
    sn, h_ = plan.sn, plan.h
    n = xv.t.shape[0]
    if n % IMGS:
        raise ValueError("a batch of %d rows is not a whole number of 40-image events" % n)
    sn.run(D.training, tape.record)
    h = conv(tape, xv, h_[D.input_conv], n, hh, ww, 3, bias=D.input_conv.bias)
    for stage in D.blocks:
        for m in stage:
            if isinstance(m, SL.Attention):
                h = _attention(tape, m, h, n, hh, ww, h_)
            else:
                h, hh, ww = _dblock(tape, m, h, n, hh, ww, h_)
    f = relu_sumpool(tape, h, n, hh * ww)                         # torch.sum(relu(h), [2,3])  model.py:912
    out = linear(tape, f, h_[D.linear0], bias=D.linear0.bias)      # uses the pre-RRM features  model.py:915
    proxy = l2norm(tape, embedding(tape, y, D.embed.weight, sn_layer=h_[D.embed]))
    r = rrm(tape, f, D.RR_D.layers, D.RR_D.norm, h_)
    e = linear(tape, r, h_[D.linear1], bias=D.linear1.bias)
    e = l2norm(tape, layernorm(tape, e, D.norm))
    return [proxy, e, out]


@on_tensor_device
def discriminator_forward(D, x, y):
    x = _plain(x)
    L.require_device(x)
    n, c, hh, ww = x.shape
    if c != 1:
        raise ValueError("the PXD discriminator takes single-channel images (model.py:730)")
    y = _plain(y, torch.int64)
    x4 = x.view(n, hh, ww, 1)  # one channel: NCHW == NHWC

    def body(tape, xv):
        return _d_body(D, tape, xv, y, hh, ww)
    proxy, embed, out = run_net(body, [x4], _params(D), owner=D)
    return proxy, embed, out.view(n)


# ------------------------------------------------------------------ DiffAugment
class _AugFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, draws):
        n, _, h, w = x.shape
        d = L.AugDraws()
        keep = []

        def col(t, dtype):
            t = t.reshape(-1).to(dtype).contiguous()
            keep.append(t)
            return t.data_ptr()
        if "brightness" in draws:
            d.brightness = col(draws["brightness"], torch.float32)
        if "contrast" in draws:
            d.contrast = col(draws["contrast"], torch.float32)
        if "tx" in draws:
            d.tx, d.ty = col(draws["tx"], torch.int64), col(draws["ty"], torch.int64)
        if "ox" in draws:
            d.ox, d.oy = col(draws["ox"], torch.int64), col(draws["oy"], torch.int64)
            d.cut_h, d.cut_w = int(draws["cut_h"]), int(draws["cut_w"])
        y = torch.empty_like(x)
        K("iea_diffaug_fwd", ptr(x), C.byref(d), n, h, w, ptr(y), ptr(_f32(n, x.device)), L.stream(), launches=2)
        ctx.d, ctx.keep, ctx.geo = d, keep, (n, h, w)
        return y

    @staticmethod
    def backward(ctx, gy):
        n, h, w = ctx.geo
        gy = gy.contiguous()
        dx = torch.empty_like(gy)
        K("iea_diffaug_bwd", ptr(gy), C.byref(ctx.d), n, h, w, ptr(dx), ptr(_f32(n, gy.device)), L.stream(),
          launches=2)
        return dx, None


@on_tensor_device
def diffaug_apply(x, draws):
    """One fused pass over the image for whichever of brightness / contrast / translation / cutout
    `draws` holds (saturation is the identity for one channel; its draw is only consumed)."""
    x = _plain(x)
    L.require_device(x)
    if x.shape[1] != 1:
        raise NotImplementedError("DiffAugment is built for the single-channel PXD images")
    return _AugFn.apply(x, draws)


# ------------------------------------------------------------------ losses
class _LossFn(torch.autograd.Function):
    """Generic wrapper: fwd(inputs...) -> (loss tensor(s), saved); bwd(saved, grad) -> input grads."""

    @staticmethod
    def forward(ctx, fwd, bwd, *xs):
        out, saved = fwd(*xs)
        ctx.bwd, ctx.saved, ctx.xs = bwd, saved, xs
        return out

    @staticmethod
    def backward(ctx, *g):
        grads = ctx.bwd(ctx.saved, ctx.xs, [t.contiguous() if t is not None else None for t in g], ctx.needs_input_grad[2:])
        return (None, None) + tuple(grads)


def _loss_scratch(events, dim, device):
    """Partial-Gram scratch of the Gram-based losses (iea_loss_scratch_floats in include/iea_b200.h)."""
    key = (events, dim)
    n = _LOSS_SCRATCH.get(key)
    if n is None:
        n = _LOSS_SCRATCH[key] = call("iea_loss_scratch_floats", events, IMGS, dim)
    return _f32(n, device)


_LOSS_SCRATCH = {}


def _events(x):
    n = x.shape[0]
    if n % IMGS:
        raise ValueError("loss input of %d rows is not a whole number of 40-image events" % n)
    return n // IMGS


@on_tensor_device
def loss_hinge_dis(dis_fake, dis_real):
    f, r = _plain(dis_fake).view(-1), _plain(dis_real).view(-1)
    L.require_device(f)
    n = f.numel()

    def fwd(f, r):
        out = _f32(2, f.device)
        K("iea_loss_hinge_dis", ptr(f), ptr(r), n, ptr(out), L.stream())
        return (out[0].clone(), out[1].clone()), None

    def bwd(saved, xs, g, need):
        dout = torch.stack([g[0] if g[0] is not None else torch.zeros_like(xs[0][0]),
                            g[1] if g[1] is not None else torch.zeros_like(xs[0][0])]).contiguous()
        df, dr = torch.empty_like(xs[0]), torch.empty_like(xs[1])
        K("iea_loss_hinge_dis_bwd", ptr(xs[0]), ptr(xs[1]), ptr(dout), n, ptr(df), ptr(dr), L.stream())
        return df, dr
    loss_real, loss_fake = _LossFn.apply(fwd, bwd, f, r)
    return loss_real, loss_fake


@on_tensor_device
def _mean_loss(x, scale):
    x = _plain(x).view(-1)
    L.require_device(x)
    n = x.numel()

    def fwd(x):
        out = _scalar(x.device)
        K("iea_loss_mean", ptr(x), n, scale, ptr(out), L.stream())
        return out, None

    def bwd(saved, xs, g, need):
        dx = torch.empty_like(xs[0])
        K("iea_loss_mean_bwd", ptr(g[0]), n, scale, ptr(dx), L.stream())
        return (dx,)
    return _LossFn.apply(fwd, bwd, x)


def loss_hinge_gen(dis_fake):
    return _mean_loss(dis_fake, -1.0)


@on_tensor_device
def loss_l2(a, b):
    """loss.l2_loss = MSELoss (loss.py:41-44; the consistency-regularisation term of train_fns.py:75-77)."""
    a, b = _plain(a).reshape(-1), _plain(b).reshape(-1)
    L.require_device(a)
    n = a.numel()
    if b.numel() != n:
        raise ValueError("l2_loss: operands of %d and %d elements" % (n, b.numel()))

    def fwd(a, b):
        out = _scalar(a.device)
        K("iea_loss_l2", ptr(a), ptr(b), n, ptr(out), L.stream())
        return out, None

    def bwd(saved, xs, g, need):
        da, db = torch.empty_like(xs[0]), torch.empty_like(xs[1])
        K("iea_loss_l2_bwd", ptr(xs[0]), ptr(xs[1]), ptr(g[0]), n, ptr(da), ptr(db), L.stream())
        return da, db
    return _LossFn.apply(fwd, bwd, a, b)


@on_tensor_device
def loss_contrastive(embed, proxy, temperature, margin):
    e, p = _plain(embed), _plain(proxy)
    L.require_device(e)
    ev, dim = _events(e), e.shape[1]

    def fwd(e, p):
        out = _scalar(e.device)
        saved = _f32(ev * (2 * IMGS * IMGS + 4 * IMGS + 1), e.device)
        K("iea_loss_contrastive_fwd", ptr(e), ptr(p), ev, IMGS, dim, temperature, margin, ptr(out), ptr(saved),
          ptr(_loss_scratch(ev, dim, e.device)), L.stream(), launches=3)
        return out, saved

    def bwd(saved, xs, g, need):
        de, dp = torch.empty_like(xs[0]), torch.empty_like(xs[1])
        K("iea_loss_contrastive_bwd", ptr(xs[0]), ptr(xs[1]), ptr(saved), ptr(g[0]), ev, IMGS, dim, temperature,
          ptr(de), ptr(dp), L.stream())
        return de, dp
    return _LossFn.apply(fwd, bwd, e, p)


@on_tensor_device
def loss_iea(k_f, k_r):
    f, r = _plain(k_f), _plain(k_r).detach()
    L.require_device(f)
    ev, dim = _events(f), f.shape[1]

    def fwd(f, r):
        out = _scalar(f.device)
        saved = _f32(ev * (IMGS * IMGS + 1), f.device)
        K("iea_loss_iea_fwd", ptr(f), ptr(r), ev, IMGS, dim, ptr(out), ptr(saved),
          ptr(_loss_scratch(ev, dim, f.device)), L.stream(), launches=4)
        return out, saved

    def bwd(saved, xs, g, need):
        df = torch.empty_like(xs[0])
        K("iea_loss_iea_bwd", ptr(xs[0]), ptr(saved), ptr(g[0]), ev, IMGS, dim, ptr(df), L.stream())
        return df, None
    return _LossFn.apply(fwd, bwd, f, r)


@on_tensor_device
def loss_uniformity(x, t):
    x = _plain(x)
    L.require_device(x)
    ev, dim = _events(x), x.shape[1]

    def fwd(x):
        out = _scalar(x.device)
        saved = _f32(ev * (IMGS * IMGS + 2), x.device)
        K("iea_loss_unif_fwd", ptr(x), ev, IMGS, dim, t, ptr(out), ptr(saved),
          ptr(_loss_scratch(ev, dim, x.device)), L.stream(), launches=3)
        return out, saved

    def bwd(saved, xs, g, need):
        dx = torch.empty_like(xs[0])
        K("iea_loss_unif_bwd", ptr(xs[0]), ptr(saved), ptr(g[0]), ev, IMGS, dim, t, ptr(dx), L.stream())
        return (dx,)
    return _LossFn.apply(fwd, bwd, x)


# ------------------------------------------------------------------ module-level API (stand-alone layers)
def _mod_plan(mod, mods, dtypes):
    key = "_iea_modplan"
    p = mod.__dict__.get(key)
    if p is None or p[0] != act_dtype():
        grp = SNGroup()
        hs = {m: grp.add(m, d, tc=(d == torch.float32 and m.weight.dim() == 2)) for m, d in zip(mods, dtypes)}
        p = (act_dtype(), grp, hs)
        mod.__dict__[key] = p
    return p[1], p[2]


def _to_nhwc(tape, x4):
    """NCHW torch tensor -> NHWC activation Var (with the inverse as its backward)."""
    n, c, hh, ww = x4.t.shape
    out = torch.empty((n, hh, ww, c), dtype=act_dtype(), device=x4.t.device)
    K("iea_nchw_to_nhwc", ptr(x4.t), dt(x4.t), ptr(out), dt(out), n, c, hh * ww, L.stream())
    ov = Var(out)
    if tape.record:
        def bw():
            if ov.g is None or not x4.need:
                return
            g = ov.g
            if ov.ds is not None:  # gradient through the batch statistics of a batch-norm that consumed `out`
                ds1, ds2, rpe = ov.ds
                ge = torch.empty_like(g)
                K("iea_conv_out_bwd", ptr(g), dt(g), c, ptr(out), dt(out), c, 0, ptr(ds1), ptr(ds2), n * hh * ww,
                  rpe, c, ptr(ge), dt(ge), L.stream())
                g = ge
            dx = torch.empty_like(x4.t)
            K("iea_nhwc_to_nchw", ptr(g), dt(g), ptr(dx), dt(dx), n, c, hh * ww, L.stream())
            add_grad(x4, dx)
        tape.add(bw)
    return ov


def _to_nchw(tape, xv, n, hh, ww, dtype=torch.float32):
    c = xv.c
    out = torch.empty((n, c, hh, ww), dtype=dtype, device=xv.t.device)
    K("iea_nhwc_to_nchw", ptr(xv.t), dt(xv.t), ptr(out), dt(out), n, c, hh * ww, L.stream())
    ov = Var(out)
    if tape.record:
        def bw():
            if ov.g is None:
                return
            g = torch.empty_like(xv.t)
            K("iea_nchw_to_nhwc", ptr(ov.g), dt(ov.g), ptr(g), dt(g), n, c, hh * ww, L.stream())
            add_grad(xv, g)
        tape.add(bw)
    return ov


@on_tensor_device
def module_conv(m, x):
    x = _plain(x)
    L.require_device(x)
    grp, hs = _mod_plan(m, [m], [act_dtype()])
    n, _, hh, ww = x.shape

    def body(tape, xv):
        grp.run(m.training, tape.record)
        y = conv(tape, _to_nhwc(tape, xv), hs[m], n, hh, ww, m.kernel_size[0], bias=m.bias)
        return [_to_nchw(tape, y, n, hh, ww)]
    return run_net(body, [x], list(m.parameters()))


@on_tensor_device
def module_linear(m, x):
    x = _plain(x)
    L.require_device(x)
    grp, hs = _mod_plan(m, [m], [torch.float32])
    lead = x.shape[:-1]
    x2 = x.reshape(-1, x.shape[-1])

    def body(tape, xv):
        grp.run(m.training, tape.record)
        return [linear(tape, xv, hs[m], bias=m.bias)]
    return run_net(body, [x2], list(m.parameters())).view(*lead, -1)


@on_tensor_device
def module_embedding(m, idx):
    L.require_device(m.weight)
    grp, hs = _mod_plan(m, [m], [torch.float32])
    idx = _plain(idx, torch.int64)

    def body(tape):
        grp.run(m.training, tape.record)
        return [embedding(tape, idx.view(-1), m.weight, sn_layer=hs[m])]
    return run_net(body, [], list(m.parameters())).view(*idx.shape, -1)


@on_tensor_device
def sn_weight_standalone(m):
    """SN.W_(): weight / sigma, differentiable w.r.t. weight (layers.py:151-165)."""
    L.require_device(m.weight)
    grp, hs = _mod_plan(m, [m], [torch.float32])
    rows = m.weight.shape[0]
    idx = torch.arange(rows, device=m.weight.device)

    def body(tape):
        grp.run(m.training, tape.record)
        l = hs[m]
        w2 = m.weight.view(rows, -1)
        out = torch.empty_like(w2)
        K("iea_embedding_fwd", ptr(idx), ptr(w2), ptr(l.inv_sigma()), rows, w2.shape[1], ptr(out), L.stream())
        v = Var(out)
        if tape.record:
            saved = l.saved()

            def bw():
                if v.g is None:
                    return
                # v.g is d(W/sigma) in the master layout [rows][cin][taps]; the kernel wants [rows][taps][cin]
                G = v.g.view(rows, l.cin, l.taps).transpose(1, 2).contiguous()
                dw = torch.empty_like(m.weight)
                K("iea_sn_weight_bwd", ptr(G), 1, ptr(m.weight), ptr(saved[1]), ptr(saved[2]), ptr(saved[0]), 1,
                  ptr(dw), 0.0, rows, l.cin, l.taps, ptr(_f32(520, dw.device)), L.stream(), launches=2)
                tape.pgrad(m.weight, dw)
            tape.add(bw)
        return [v]
    return run_net(body, [], [m.weight]).view_as(m.weight)


@on_tensor_device
def power_iteration_single(W, u, update, eps):
    """layers.power_iteration for one singular vector, on the grouped kernel."""
    L.require_device(W)

    class _M:  # minimal layer record
        pass
    m = _M()
    m.weight, m.u0, m.sv0, m.eps = W.detach().contiguous(), u.view(1, -1).contiguous().clone(), _f32(1, W.device), eps
    grp = SNGroup()
    l = grp.add(m, torch.float32)
    grp.run(True, False)
    if update:
        u.view(-1).copy_(m.u0.view(-1))
    return m.sv0[0].clone(), m.u0.clone(), l.v().view(1, -1).clone()


@on_tensor_device
def module_bn(m, x):
    """layers.bn.forward as stats + affine kernels (stand-alone use; inside G it is fused)."""
    x = _plain(x)
    L.require_device(x)
    n, c, hh, ww = x.shape

    def body(tape, xv):
        xn = _to_nhwc(tape, xv)
        sm, sv, mode, owner = bn_state(m)
        ss = bn_affine(tape, xn, n, hh, ww, gain=ptr(m.gain), gain_ld=0, gain_add=0.0, bias=ptr(m.bias), bias_ld=0,
                       stored_mean=sm, stored_var=sv, training=m.training, eps=m.eps,
                       momentum=m.momentum, gain_param=m.gain, bias_param=m.bias, owner=owner, mode=mode)
        return [_to_nchw(tape, affine(tape, xn, ss, n, hh * ww, False), n, hh, ww)]
    return run_net(body, [x], list(m.parameters()))


@on_tensor_device
def bn_functional(x, gain, bias, *, stored_mean, stored_var, training, mode, eps, momentum, owner=None,
                  want_stats=False):
    """Batch-norm with caller-supplied per-sample (N,C) or per-channel (1,C) gain / bias TENSORS (autograd
    flows into them): the arithmetic of myBN.forward / manual_bn / fused_bn (layers.py:505-599).
    training: batch statistics per event (running statistics per `mode`, see iea_bn_finalize);
    otherwise the given stored statistics."""
    x = _plain(x)
    L.require_device(x)
    n, c, hh, ww = x.shape
    dev = x.device

    def rows(t, fill):
        if t is None:
            return torch.full((n, c), fill, dtype=torch.float32, device=dev)
        return _plain(t).reshape(-1, c).expand(n, c).contiguous()
    g2, b2 = rows(gain, 1.0), rows(bias, 0.0)
    keep = {}

    def body(tape, xv, gv, bv):
        xn = _to_nhwc(tape, xv)
        dgb = torch.zeros((n, 2 * c), dtype=torch.float32, device=dev) if tape.record else None
        if tape.record:
            def bw():  # (added first: runs after the finalize backward has filled dgb)
                gv.g, bv.g = dgb[:, :c].contiguous(), dgb[:, c:].contiguous()
            tape.add(bw)
        ss = bn_affine(tape, xn, n, hh, ww, gain=gv.t.data_ptr(), gain_ld=c, gain_add=0.0, bias=bv.t.data_ptr(),
                       bias_ld=c, stored_mean=stored_mean, stored_var=stored_var, training=training, eps=eps,
                       momentum=momentum, dgain=dgb.data_ptr() if dgb is not None else None,
                       dbias=(dgb.data_ptr() + 4 * c) if dgb is not None else None, dgb_ld=2 * c, owner=owner,
                       mode=mode)
        keep["ss"] = ss
        return [_to_nchw(tape, affine(tape, xn, ss, n, hh * ww, False), n, hh, ww)]
    out = run_net(body, [x, g2, b2], [])
    if want_stats:
        ss = keep["ss"]
        return out, ss.mean, (ss.rstd.double().pow(-2) - eps).float()
    return out


def module_mybn(m, x, gain, bias):
    """myBN.forward(x, gain, bias) (layers.py:570-599)."""
    if m.training:
        if m.accumulate_standing:
            m.accumulation_counter += 1.0
        mode = (1 | 4) if m.accumulate_standing else (1 | 2)
        sm, sv = m.stored_mean, m.stored_var
    else:
        mode = 0
        sm, sv = m.stored_mean, m.stored_var
        if m.accumulate_standing:
            sm, sv = sm / m.accumulation_counter, sv / m.accumulation_counter
    return bn_functional(x, gain, bias, stored_mean=sm, stored_var=sv, training=m.training, mode=mode, eps=m.eps,
                         momentum=m.momentum, owner=m)


def affine(tape, xv, ss, n, hw, relu):
    """y = [relu](x*scale + shift): the stand-alone form of the conv prologue."""
    c = xv.c
    y = torch.empty_like(xv.t)
    K("iea_affine_act", ptr(xv.t), dt(xv.t), ptr(ss.scale), ptr(ss.shift), n, hw, c, int(relu), ptr(y), dt(y), L.stream())
    yv = Var(y)
    if tape.record:
        def bw():
            if yv.g is None:
                return
            # reuse the prologue-backward kernel with an identity 1x1 geometry
            d = _desc(n, 1, hw, c, c, 1, xv.t, xv.off(), xv.ld, 0, relu, ss.scale, ss.shift, xv.t, None, 0, None,
                      None, 0, 0, -1, y, y.data_ptr(), c, 0, None)
            xg, beta = _accum_target(xv)
            dsc, dsh = torch.empty_like(ss.scale), torch.empty_like(ss.shift)
            K("iea_conv_input_bwd", C.byref(d), ptr(yv.g), dt(yv.g), ptr(xg), dt(xg), xv.ld, beta, ptr(dsc),
              ptr(dsh), ptr(_f32(n * 64 * c * 2, y.device)), L.stream(), launches=2)
            ss.dscale, ss.dshift = dsc, dsh
        tape.add(bw)
    return yv


@on_tensor_device
def module_ccbn(m, x, y):
    """layers.ccbn.forward stand-alone: the two SNLinears as one grouped GEMM, stats, affine."""
    x, y = _plain(x), _plain(y)
    L.require_device(x)
    n, c, hh, ww = x.shape
    key = "_iea_modplan"
    p = m.__dict__.get(key)
    if p is None:
        grp = SNGroup()
        ls = grp.add_shared([m.gain, m.bias], torch.float32)
        p = (grp, ls)
        m.__dict__[key] = p
    grp, ls = p

    def body(tape, xv, yv):
        grp.run(m.training, tape.record)
        wp, wd, cs = grp.colscales[0]
        gbv = conv(tape, yv, None, n, 1, 1, 1, out_dtype=torch.float32, out_shape=(n, 2 * c),
                   grouped=(wp, wd, cs, 2 * c, ls))
        gb, dgb = gbv.t, None
        if tape.record:
            dgb = torch.zeros_like(gb)
            gbv.g = dgb
        xn = _to_nhwc(tape, xv)
        sm, sv, mode, owner = bn_state(m)
        ss = bn_affine(tape, xn, n, hh, ww, gain=gb.data_ptr(), gain_ld=2 * c, gain_add=1.0,
                       bias=gb.data_ptr() + 4 * c, bias_ld=2 * c, stored_mean=sm,
                       stored_var=sv, training=m.training, eps=m.eps, momentum=m.momentum if m.mybn else 0.1, owner=owner,
                       mode=mode,
                       dgain=dgb.data_ptr() if dgb is not None else None,
                       dbias=(dgb.data_ptr() + 4 * c) if dgb is not None else None, dgb_ld=2 * c)
        return [_to_nchw(tape, affine(tape, xn, ss, n, hh * ww, False), n, hh, ww)]
    return run_net(body, [x, y], list(m.parameters()))


class _BlockPlan:
    """SN group of one stand-alone GBlock: its four convs + the eight ccbn linears as one grouped GEMM."""

    def __init__(self, blk):
        self.sn = SNGroup()
        self.h = {cv: self.sn.add(cv, act_dtype()) for cv in (blk.conv1, blk.conv2, blk.conv3, blk.conv4)}
        mods, off, self.gb_off = [], 0, {}
        for b in (blk.bn1, blk.bn2, blk.bn3, blk.bn4):
            self.gb_off[b] = (off, off + b.output_size)
            off += 2 * b.output_size
            mods += [b.gain, b.bias]
        self.gb_cols = off
        self.gb_layers = self.sn.add_shared(mods, torch.float32)


@on_tensor_device
def module_gblock(blk, x, y):
    """GBlock.forward(x, y) stand-alone (model.py:54-71): the same four fused convs as inside the Generator,
    with this block's eight ccbn gain / bias linears as one grouped GEMM on y."""
    x, y = _plain(x), _plain(y)
    L.require_device(x)
    for b in (blk.bn1, blk.bn2, blk.bn3, blk.bn4):
        if not hasattr(b, "gain") or not hasattr(b.gain, "weight"):
            raise NotImplementedError("stand-alone GBlock is built for which_bn=ccbn (the Generator's)")
    plan = _plan(blk, _BlockPlan)
    n, _, hh, ww = x.shape
    geo = {}

    def body(tape, xv, yv):
        plan.sn.run(blk.training, tape.record)
        wp, wd, cs = plan.sn.colscales[0]
        gbv = conv(tape, yv, None, n, 1, 1, 1, out_dtype=torch.float32, out_shape=(n, plan.gb_cols),
                   grouped=(wp, wd, cs, plan.gb_cols, plan.gb_layers))
        dgb = None
        if tape.record:
            dgb = torch.zeros_like(gbv.t)
            gbv.g = dgb
        out, ho, wo = _gblock(tape, blk, _to_nhwc(tape, xv), n, hh, ww, plan, gbv.t, dgb, blk.training)
        geo["hw"] = (ho, wo)
        return [_to_nchw(tape, out, n, ho, wo)]
    return run_net(body, [x, y], list(blk.parameters()))


@on_tensor_device
def module_dblock(blk, x):
    x = _plain(x)
    L.require_device(x)
    mods = [blk.conv1, blk.conv2, blk.conv3, blk.conv4] + ([blk.conv_sc] if blk.learnable_sc else [])
    grp, hs = _mod_plan(blk, mods, [act_dtype()] * len(mods))
    n, _, hh, ww = x.shape

    def body(tape, xv):
        grp.run(blk.training, tape.record)
        y, ho, wo = _dblock(tape, blk, _to_nhwc(tape, xv), n, hh, ww, hs)
        return [_to_nchw(tape, y, n, ho, wo)]
    return run_net(body, [x], list(blk.parameters()))


@on_tensor_device
def module_attention(m, x):
    x = _plain(x)
    L.require_device(x)
    mods = [m.theta, m.phi, m.g, m.o]
    grp, hs = _mod_plan(m, mods, [act_dtype()] * 4)
    n, _, hh, ww = x.shape

    def body(tape, xv):
        grp.run(m.training, tape.record)
        return [_to_nchw(tape, _attention(tape, m, _to_nhwc(tape, xv), n, hh, ww, hs), n, hh, ww)]
    return run_net(body, [x], list(m.parameters()))


@on_tensor_device
def module_rrm(blocks, final_norm, x):
    x = _plain(x)
    L.require_device(x)
    owner = blocks[0]
    mods = []
    for b in blocks:
        mods += [b.self_attn.qkv_proj, b.self_attn.o_proj, b.linear_net[0], b.linear_net[3]]
    grp, hs = _mod_plan(owner, mods, [torch.float32] * len(mods))
    b_, s, e = x.shape
    if s != IMGS:
        raise NotImplementedError("the RRM kernels attend over the 40 sensors of an event (seq = 40)")
    params = [p for b in blocks for p in b.parameters()] + (list(final_norm.parameters()) if final_norm is not None else [])

    def body(tape, xv):
        grp.run(owner.training, tape.record)
        return [rrm(tape, xv, blocks, final_norm, hs)]
    return run_net(body, [x.reshape(b_ * s, e)], params).view(b_, s, e)


@on_tensor_device
def module_mha(m, x, return_attention=False):
    x = _plain(x)
    L.require_device(x)
    grp, hs = _mod_plan(m, [m.qkv_proj, m.o_proj], [torch.float32] * 2)
    b_, s, e = x.shape
    if s != IMGS:
        raise NotImplementedError("the RRM kernels attend over the 40 sensors of an event (seq = 40)")
    keep = {}

    def body(tape, xv):
        grp.run(m.training, tape.record)
        qkv = linear(tape, xv, hs[m.qkv_proj], bias=m.qkv_proj.bias)
        val, att = mha_core(tape, qkv, b_, s, m.num_heads, m.head_dim)
        keep["att"] = att
        return [linear(tape, val, hs[m.o_proj], bias=m.o_proj.bias)]
    o = run_net(body, [x.reshape(b_ * s, e)], list(m.parameters())).view(b_, s, e)
    return (o, keep["att"]) if return_attention else o


@on_tensor_device
def module_sdp(q, k, v):
    """RRM.scaled_dot_product on (B, h, 40, d) tensors: (values, attention map), differentiable w.r.t.
    q, k, v through the values (RRM.py:10-16; the map is returned for inspection, as get_attention_maps
    uses it, and carries no gradient)."""
    q, k, v = _plain(q), _plain(k), _plain(v)
    L.require_device(q)
    b_, hds, s, d = q.shape
    if s != IMGS or k.shape != q.shape or v.shape != q.shape:
        raise NotImplementedError("the RRM kernels attend over the 40 sensors of an event with equal q/k/v widths")
    keep = {}

    def body(tape, qv, kv, vv):
        # the kernel reads the module's own layout: rows (B*S), columns [head][q | k | v]
        qkv = torch.cat([qv.t, kv.t, vv.t], -1).permute(0, 2, 1, 3).reshape(b_ * s, hds * 3 * d).contiguous()
        pk = Var(qkv)
        val, att = mha_core(tape, pk, b_, s, hds, d)
        keep["att"] = att
        out = Var(val.t.view(b_, s, hds, d).permute(0, 2, 1, 3).contiguous())
        if tape.record:
            def bw_in():  # (runs last) split d(qkv) back into the three inputs
                if pk.g is None:
                    return
                g = pk.g.view(b_, s, hds, 3 * d).permute(0, 2, 1, 3)
                qv.g, kv.g, vv.g = (g[..., :d].contiguous(), g[..., d:2 * d].contiguous(), g[..., 2 * d:].contiguous())

            def bw_out():  # (runs first) gradient of the returned (B,h,S,d) values -> kernel layout
                if out.g is not None:
                    val.g = out.g.permute(0, 2, 1, 3).reshape(b_ * s, hds * d).contiguous()
            tape.nodes.insert(0, bw_in)
            tape.add(bw_out)
        return [out]
    vals = run_net(body, [q, k, v], [])
    return vals, keep["att"]
