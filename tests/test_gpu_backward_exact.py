"""Exact tests of the convolution backward kernels at the batch the train step runs (8 events = 320 images) and at
one event (40 images).

Which weight-gradient or fused 1x1-backward kernel runs, its grid and how many tiles each CTA accumulates depend on
M = n*h*w, so a kernel exercised at 40 images is not the one the benchmark runs at 320.  The module first runs one
eager bf16 train step of the full-size nets (8 events) with `engine.K` wrapped and records every backward launch:
iea_conv_wgrad_mma, iea_conv_wgrad, iea_conv_bwd1x1, the data-gradient iea_conv_fprop calls, iea_conv_input_bwd,
iea_conv_out_bwd, iea_residual_bwd and iea_colsum.  Each distinct geometry (sizes, channel windows / pixel strides,
prologue, modes, dtypes) is then replayed through the C ABI on fresh data at the captured batch and at 40 images.

Data on which fp32 is exact (so every result must equal the fp64 reference bit for bit, whatever the summation
order, split or tiling):
  * activations x in {-4, -3.5, ..., 4}; gradients g in {-2..2}; batch-norm scale in {0.5, 1, 1.5, 2} and shift in
    {-2, -1.5, ..., 2}; weights in {-8..8}/8 (integer master weights / 8 packed by SNGroup); 1/sigma 1 or 0.5;
    ds1 in {0, +-1/8}, ds2 in {0, +-1/8}; a tanh output y in {-7..7}/8.  relu(x*scale + shift) and the fused
    geff = g + ds1 + 2 y ds2 are then exact in bf16 as well (the tcgen05 prologues compute in bf16).
  * ties at zero on purpose: where T(x) is thinned, x is set to the largest half-step value with
    x*scale + shift <= 0, which is exactly 0 for many (scale, shift) pairs; relu'(0) = 0 everywhere.
  * magnitude budget: for every output element sum |term| / unit < 2^22 (unit = the value grid of one term), computed
    in fp64 from |g|, |T(x)|, |W| and asserted.  The inputs are thinned (a fraction of g, or of T(x) via the zero-tie
    values, is non-zero) with a density chosen from M, and thinned further until the budget holds.
  * the fp64 reference multiplies explicitly (shifted-tap matmuls), so its sums of grid values are exact too.
  * fp32 outputs compare as int32 bit patterns, bf16 outputs as int16 against torch's round-to-nearest-even of the
    exact value (zeros compared without their sign).  Values outside the channel windows are a bf16-exact sentinel,
    and output channels outside the window must keep it.

The profiler records the CUDA kernels of every replay: the route-coverage test asserts that every backward kernel
was reached and lists the geometries whose weight-gradient / fused 1x1 kernel differs between 40 and 320 images.
"""
import ctypes as C
import traceback

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

DEV = "cuda"
F64 = torch.float64
TD = {0: torch.float32, 1: torch.bfloat16}
LIMIT = 2.0 ** 22   # budget: sum |term| / unit stays below this (2 bits of headroom under fp32's 24)
SENT = 1000.0       # filler outside channel windows (exact in bf16 and fp32)
SMALL_N = 40        # one event
PTR = ("x", "in_scale", "in_shift", "wpack", "wpack_tc", "out_scale", "bias", "res", "y", "stats")

ROUTES = {}    # (family, geometry label) -> {n: set of kernel names}
SEEN = set()   # every kernel name any replay ran


@pytest.fixture(scope="module")
def eng():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from iea_gan_b200 import engine, _lib
    _lib.lib()
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    return engine


# ------------------------------------------------------------------ geometry capture
def _al(p):
    return p is not None and int(p) % 16 == 0


def _desc_rec(d):
    r = {f: getattr(d, f) for f, _ in d._fields_ if f not in PTR}
    r.update(aff=bool(d.in_scale), tc=bool(d.wpack_tc), osc=bool(d.out_scale), bias_=bool(d.bias), res_=bool(d.res),
             x_al=_al(d.x), y_al=_al(d.y))
    r.pop("impl")
    return r


def _record(name, args):
    """Geometry of one backward launch: descriptor fields (pointers reduced to present / 16-byte aligned) and the
    scalar arguments of the call."""
    a = list(args)
    if name == "iea_conv_wgrad_mma":
        return dict(d=_desc_rec(a[0]._obj), g_dt=a[2], g_ld=a[3], g_al=_al(a[1]), db=bool(a[5]))
    if name == "iea_conv_wgrad":
        return dict(d=_desc_rec(a[0]._obj), g_dt=a[2], g_ld=a[3], g_al=_al(a[1]))
    if name == "iea_conv_fprop":
        return dict(d=_desc_rec(a[0]._obj))
    if name == "iea_conv_bwd1x1":
        b = a[1]._obj
        return dict(d=_desc_rec(a[0]._obj), ds=bool(b.ds1), dx=bool(b.dx), w=bool(b.wpart), db=bool(b.dbias),
                    ss=bool(b.dscale), g_ld=b.g_ld, y_ld=b.y_ld, dx_ld=b.dx_ld, beta=b.beta, rpe=b.rows_per_event)
    if name == "iea_conv_input_bwd":
        return dict(d=_desc_rec(a[0]._obj), da_dt=a[2], dx=bool(a[3]), dx_dt=a[4], dx_ld=a[5], beta=a[6],
                    ss=bool(a[7]), scratch=bool(a[9]), da_al=_al(a[1]), dx_al=_al(a[3]) if a[3] else True)
    if name == "iea_conv_out_bwd":
        return dict(dy_dt=a[1], dy_ld=a[2], y_dt=a[4], y_ld=a[5], act=a[6], ds=bool(a[7]), rows=a[9], rpe=a[10], c=a[11],
                    g_dt=a[13], al=_al(a[0]) and _al(a[3]) and _al(a[12]))
    if name == "iea_colsum":
        return dict(g_dt=a[1], g_ld=a[2], rows=a[3], c=a[4], beta=a[6], al=_al(a[0]))
    if name == "iea_residual_bwd":
        return dict(g_dt=a[1], g_ld=a[2], n=a[3], h=a[4], w=a[5], res_c=a[6], res_mode=a[7], dres_dt=a[9], dres_ld=a[10],
                    dres_c=a[11], beta=a[12], al=_al(a[0]) and _al(a[8]))
    return None


def _key(rec):
    return repr(sorted((k, sorted(v.items()) if isinstance(v, dict) else v) for k, v in rec.items()))


@pytest.fixture(scope="module")
def captured(eng):
    """One eager bf16 train step of the full-size nets at 8 events (what bench.py times), with engine.K wrapped:
    {ABI name: [distinct geometries]} of every backward launch, and the step's batch."""
    from iea_gan_b200.default_config import shipped_config
    from test_gpu_fullsize import draws_for, fresh_nets, gpu_step
    cfg = shipped_config(H_base=1, device="cuda", clip_norm=1e9)
    rows = 320
    phases = draws_for(cfg, 601, rows, 256, 256)
    torch.manual_seed(602)
    x = torch.rand(rows, 1, 256, 256) * 2 - 1
    y = torch.arange(40).repeat(rows // 40)
    names = {"iea_conv_wgrad_mma", "iea_conv_wgrad", "iea_conv_bwd1x1", "iea_conv_fprop", "iea_conv_input_bwd",
             "iea_conv_out_bwd", "iea_residual_bwd", "iea_colsum"}
    seen, depth = {}, [0]
    orig_k, orig_bwd = eng.K, eng.Tape.backward

    def k_rec(name, *args, launches=1):
        if name in names and (name != "iea_conv_fprop" or depth[0] > 0):
            rec = _record(name, args)
            seen.setdefault(name, {}).setdefault(_key(rec), rec)
        return orig_k(name, *args, launches=launches)

    def bwd_rec(self):
        depth[0] += 1
        try:
            return orig_bwd(self)
        finally:
            depth[0] -= 1

    eng.K, eng.Tape.backward = k_rec, bwd_rec
    try:
        nets = fresh_nets(cfg)
        gpu_step(cfg, phases, x, y, "bf16", nets=nets)
    finally:
        eng.K, eng.Tape.backward = orig_k, orig_bwd
    del nets
    torch.cuda.empty_cache()
    out = {k: list(v.values()) for k, v in seen.items()}
    print("\ncaptured backward geometries: " + ", ".join("%s %d" % (k, len(v)) for k, v in sorted(out.items())))
    return out, rows


# ------------------------------------------------------------------ exact data
class Data:
    def __init__(self, seed):
        self.g = torch.Generator(device=DEV).manual_seed(seed)

    def grid(self, shape, lo, hi, den, p=1.0):
        """values {lo..hi}/den, each kept with probability p (else 0)"""
        v = torch.randint(lo, hi + 1, shape, generator=self.g, device=DEV).to(F64) / den
        if p < 1.0:
            v = v * (torch.rand(shape, generator=self.g, device=DEV) < p)
        return v

    def affine(self, rows, c):
        return self.grid((rows, c), 1, 4, 2), self.grid((rows, c), -4, 4, 2)

    def x(self, shape, s, t, relu, p):
        """x [n, hs, ws, c] in {-4..4}/1 step 1/2; a fraction 1-p of the entries is set where T(x) = 0 (the largest
        half-step x with x*s + t <= 0: ties at exactly 0 wherever -t/s is on the grid), when the prologue allows it."""
        x = self.grid(shape, -8, 8, 2)
        if p >= 1.0:
            return x
        off = torch.rand(shape, generator=self.g, device=DEV) >= p
        if s is not None and relu:
            z = (torch.floor(-2 * t / s) / 2).clamp(-4, 4)[:, None, None, :].expand(shape)
        elif s is None:
            z = torch.zeros_like(x) if not relu else -x.abs()
        else:
            return x  # an affine without ReLU is never 0 by construction: g carries the thinning
        return torch.where(off, z, x)


def src_res(h, w, mode):
    return (h // 2, w // 2) if mode == 1 else ((2 * h, 2 * w) if mode == 2 else (h, w))


def ref_T(x, s, t, relu, mode):
    """the conv prologue on fp64 values: [n, hs, ws, c] -> [n, h, w, c]"""
    if s is not None:
        x = x * s[:, None, None, :] + t[:, None, None, :]
    if relu:
        x = torch.relu(x)
    if mode == 1:
        x = x.repeat_interleave(2, 1).repeat_interleave(2, 2)
    elif mode == 2:
        x = (x[:, 0::2, 0::2] + x[:, 1::2, 0::2] + x[:, 0::2, 1::2] + x[:, 1::2, 1::2]) * 0.25
    return x


def _taps(T, k, i0, i1):
    n_, h, w, c = T[i0:i1].shape
    if k == 1:
        yield 0, T[i0:i1].reshape(-1, c)
        return
    Tp = F.pad(T[i0:i1], (0, 0, 1, 1, 1, 1))
    for tap in range(9):
        ky, kx = divmod(tap, 3)
        yield tap, Tp[:, ky:ky + h, kx:kx + w].reshape(-1, c)


def ref_wgrad(g, T, k):
    """dW[co][tap][ci] = sum_px g[px][co] T[px + tap offset][ci] (zero padding), fp64 explicit products"""
    n, co, ci = g.shape[0], g.shape[-1], T.shape[-1]
    out = torch.zeros(co, k * k, ci, dtype=F64, device=DEV)
    for i in range(0, n, 40):
        gg = g[i:i + 40].reshape(-1, co).t()
        for tap, sh in _taps(T, k, i, i + 40):
            out[:, tap] += gg @ sh
    return out


def ref_fprop(x, wp, k):
    """y[px][co] = sum_tap sum_ci x[px + tap offset][ci] wp[co][tap][ci]"""
    n, h, w, _ = x.shape
    out = torch.empty(n, h, w, wp.shape[0], dtype=F64, device=DEV)
    for i in range(0, n, 40):
        acc = 0
        for tap, sh in _taps(x, k, i, i + 40):
            acc = acc + sh @ wp[:, tap].t()
        out[i:i + 40] = acc.view(-1, h, w, wp.shape[0])
    return out


def budget(absval, unit, what):
    worst = float(absval.max()) / unit if absval.numel() else 0.0
    assert worst < LIMIT, "%s: magnitude budget %.3g units >= 2^22: the data is not exact" % (what, worst)
    return worst


def fits(absval, unit):
    return absval.numel() == 0 or float(absval.max()) / unit < LIMIT / 2


def rne_exact(ref, dtype):
    """the exact fp64 value in the output dtype: exact in fp32 (asserted), then one round-to-nearest-even"""
    f = ref.float()
    assert torch.equal(f.double(), ref), "reference value not exact in fp32"
    return f.to(dtype)


def mismatch(got, ref):
    """'' when the bit patterns agree (zeros without their sign), else a description of the first difference"""
    want = rne_exact(ref, got.dtype)
    iv = torch.int16 if got.dtype == torch.bfloat16 else torch.int32
    a, b = (got + 0.0).contiguous(), (want + 0.0).contiguous()
    eq = a.view(iv) == b.view(iv)
    if bool(eq.all()):
        return ""
    bad = (~eq).nonzero()
    i = tuple(bad[0].tolist())
    return "%d of %d differ, first at %s: got %r want %r" % (bad.shape[0], eq.numel(), i, float(got[i]), float(want[i]))


class Buf:
    """rows x ld activation buffer (sentinel-filled) with a channel window [c0, c0 + c)"""

    def __init__(self, rows, ld, c, dtype, aligned=True, vals=None):
        es = torch.tensor([], dtype=dtype).element_size()
        c0 = ld - c if (ld > c and (((ld - c) * es) % 16 == 0) == aligned) else 0
        self.t = torch.full((rows, ld), SENT, dtype=dtype, device=DEV)
        self.c0, self.c, self.ld, self.dtype = c0, c, ld, dtype
        if vals is not None:
            self.win().copy_(vals.reshape(rows, c))

    def win(self):
        return self.t[:, self.c0:self.c0 + self.c]

    def ptr(self):
        return self.t.data_ptr() + self.c0 * self.t.element_size()

    def outside_ok(self):
        o = torch.cat([self.t[:, :self.c0], self.t[:, self.c0 + self.c:]], 1)
        return bool((o.float() == SENT).all())


def profiled(fn):
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        rc = fn()
        torch.cuda.synchronize()
    names = {e.key for e in prof.key_averages()}
    SEEN.update(names)
    return rc, names


def kernel_of(names):
    for k in ("c1_wgrad_kernel", "wgrad_tc_kernel", "wgrad3_kernel", "wgrad_mma_kernel<9", "wgrad_mma_kernel<1",
              "bwd1x1_kernel", "conv_wgrad_generic"):
        if any(k in s for s in names):
            return k
    return "?"


def make_desc(r, n, x, wp=None, y=None, scale=None, shift=None, osc=None, wtc=None):
    from iea_gan_b200 import _lib as L
    d = L.ConvDesc()
    for f, v in r.items():
        if hasattr(d, f) and f != "n":
            setattr(d, f, v)
    d.n = n
    d.x = x.ptr()
    d.in_scale, d.in_shift = (scale.data_ptr(), shift.data_ptr()) if scale is not None else (None, None)
    d.wpack = wp.data_ptr() if wp is not None else None
    d.wpack_tc = wtc.data_ptr() if wtc is not None else None
    d.out_scale = osc.data_ptr() if osc is not None else None
    d.y = y.ptr() if y is not None else None
    d.bias = d.res = d.stats = None
    d.res_c = 0 if not r.get("res_") else r["res_c"]
    d.impl = 0
    return d


def sn_layer(eng, rows, cin, k, dtype, data, tc=False):
    """an SNConv2d with weights {-8..8}/8 and its packs (fprop / dgrad, plain and tcgen05 order) from SNGroup"""
    from iea_gan_b200 import sn_layers as SL
    m = SL.SNConv2d(cin, rows, k, padding=k // 2, bias=False, eps=1e-6).to(DEV)
    with torch.no_grad():
        m.weight.copy_(data.grid(m.weight.shape, -8, 8, 8).float())
    grp = eng.SNGroup()
    l = grp.add(m, dtype, tc=tc)
    grp.run(True, True)
    torch.cuda.synchronize()
    return m, l, grp


def prologue(data, r, n):
    """inputs of a conv prologue for geometry r: x values [n, hs, ws, cin], scale / shift or None, and T(x)"""
    hs, ws = src_res(r["h"], r["w"], r["in_mode"])
    s = t = None
    if r["aff"]:
        s, t = data.affine(1 if r["in_bcast"] else n, r["cin"])
    return hs, ws, s, t


def t_unit(r):
    u = 0.25 if r["aff"] else 0.5
    return u / 4 if r["in_mode"] == 2 else u


def _label(r, extra=""):
    d = r["d"] if "d" in r else r
    return "%dx%d %d->%d k%d in%d%s%s%s xld%d%s" % (d["h"], d["w"], d["cin"], d["cout"], d["ksize"], d["in_mode"],
                                                  " aff" if d["aff"] else "", " bc" if d.get("in_bcast") else "",
                                                  " relu" if d["in_relu"] else "", d["x_ld"], extra)


# ------------------------------------------------------------------ replays
def replay_wgrad(eng, rec, n, seed, mma=True):
    """iea_conv_wgrad_mma (slice 0 of gpart, dbias and the 0/1 return per plan) or iea_conv_wgrad (sum of its
    slices) against the fp64 weight gradient."""
    from iea_gan_b200 import _lib as L
    r = rec["d"]
    h, w, cin, cout, k = r["h"], r["w"], r["cin"], r["cout"], r["ksize"]
    data = Data(seed)
    hs, ws, s, t = prologue(data, r, n)
    M = n * h * w
    xdt, gdt = TD[r["x_dtype"]], TD[rec["g_dt"]]
    unit = t_unit(r)
    p_g, p_x = min(0.5, 2.0 ** 18 / M), 1.0
    for _ in range(12):
        xv = data.x((n, hs, ws, cin), s, t, r["in_relu"], p_x)
        T = ref_T(xv, s, t, r["in_relu"], r["in_mode"])
        g = data.grid((n, h, w, cout), -2, 2, 1, p_g)
        bound = ref_wgrad(g.abs(), T.abs(), k)
        if fits(bound, unit) and fits(g.abs().reshape(-1, cout).sum(0), 1.0):
            break
        p_g, p_x = p_g / 4, max(p_x / 2, 1 / 64)
    budget(bound, unit, "dW")
    ref = ref_wgrad(g, T, k)
    x = Buf(n * hs * ws, r["x_ld"], cin, xdt, r["x_al"], xv)
    gb = Buf(M, rec["g_ld"], cout, gdt, rec["g_al"], g)
    sc = s.float().contiguous() if s is not None else None
    sh = t.float().contiguous() if t is not None else None
    d = make_desc(r, n, x, scale=sc, shift=sh)
    out = []
    if mma:
        slices = L.call("iea_conv_wgrad_mma_slices", C.byref(d), rec["g_dt"], rec["g_ld"])
        if slices <= 0:
            return ["iea_conv_wgrad_mma_slices returned %d" % slices], set()
        gp = torch.full((slices, cout * k * k * cin), float("nan"), device=DEV)
        db = torch.full((cout,), float("nan"), device=DEV)
        rc, names = profiled(lambda: L.call("iea_conv_wgrad_mma", C.byref(d), gb.ptr(), rec["g_dt"], rec["g_ld"],
                                            gp.data_ptr(), db.data_ptr(), L.stream()))
        kern = kernel_of(names)
        want_rc = 0 if kern in ("c1_wgrad_kernel", "wgrad_tc_kernel") else 1
        if rc != want_rc:
            out.append("%s returned %d, want %d" % (kern, rc, want_rc))
        e = mismatch(gp[0].view(cout, k * k, cin), ref)
        if e:
            out.append("dW (%s): %s" % (kern, e))
        if rc == 1:
            e = mismatch(db, g.reshape(-1, cout).sum(0))
            if e:
                out.append("dbias (%s): %s" % (kern, e))
    else:
        nsplit = max(1, min(64, M // 4096))
        gp = torch.full((nsplit, cout, k * k * cin), float("nan"), device=DEV)
        _, names = profiled(lambda: L.call("iea_conv_wgrad", C.byref(d), gb.ptr(), rec["g_dt"], rec["g_ld"],
                                           gp.data_ptr(), nsplit, L.stream()))
        tot = gp.double().sum(0)  # each slice is exact, so is their fp64 sum
        e = mismatch(tot.float().view(cout, k * k, cin), ref)
        if e:
            out.append("dW (conv_wgrad_generic, %d splits): %s" % (nsplit, e))
    return out, names


def replay_dgrad(eng, rec, n, seed, acc_variants=True):
    """a data-gradient iea_conv_fprop (dgrad pack of an integer-weight layer, 1/sigma 0.5) -> da, also with
    acc_c0 = 0 (da += the product)"""
    from iea_gan_b200 import _lib as L
    r = rec["d"]
    h, w, cin, cout, k = r["h"], r["w"], r["cin"], r["cout"], r["ksize"]
    data = Data(seed)
    M = n * h * w
    wdt = TD[r["w_dtype"]]
    m, l, grp = sn_layer(eng, cin, cout, k, wdt, data, tc=r["tc"] and wdt == torch.float32)
    wd = l.wd.double().reshape(cout, k * k, cin)
    wtc = l.wd_tc if r["tc"] else None
    if r["tc"] and wtc is None:
        return ["no tcgen05 dgrad pack for this shape"], set()
    hs, ws, s, t = prologue(data, r, n)
    isg = 0.5 if r["osc"] else 1.0
    unit = (0.5 if r["aff"] else 1.0) * 0.125 * isg
    p = 1.0
    for _ in range(8):
        g = data.grid((n, hs, ws, cin), -2, 2, 1, p)
        Tg = ref_T(g, s, t, r["in_relu"], r["in_mode"])
        bound = ref_fprop(Tg.abs(), wd.abs(), k) * isg
        if fits(bound + 4.0, unit):
            break
        p /= 4
    budget(bound + 4.0, unit, "da")
    prod = ref_fprop(Tg, wd, k) * isg
    xb = Buf(n * hs * ws, r["x_ld"], cin, TD[r["x_dtype"]], r["x_al"], g)
    sc = s.float().contiguous() if s is not None else None
    sh = t.float().contiguous() if t is not None else None
    osc = torch.tensor([isg], device=DEV) if r["osc"] else None
    out, names = [], set()
    for acc in ([r["acc_c0"]] + ([0 if r["acc_c0"] < 0 else -1] if acc_variants else [])):
        old = data.grid((M, cout), -4, 4, 2)
        yb = Buf(M, r["y_ld"], cout, TD[r["y_dtype"]], r["y_al"], old)
        d = make_desc(dict(r, acc_c0=acc), n, xb, wp=l.wd, y=yb, scale=sc, shift=sh, osc=osc, wtc=wtc)
        _, nm = profiled(lambda: L.call("iea_conv_fprop", C.byref(d), L.stream()))
        names |= nm
        want = prod.reshape(M, cout) + (old if acc == 0 else 0)
        e = mismatch(yb.win(), want)
        if e:
            out.append("da (acc_c0 %d): %s" % (acc, e))
        if not yb.outside_ok():
            out.append("da (acc_c0 %d): wrote outside its channel window" % acc)
    return out, names


def ref_input_bwd(da, xv, s, t, relu, mode):
    """(gm at x's resolution, mask) of the prologue adjoint"""
    if mode == 1:
        gs = da[:, 0::2, 0::2] + da[:, 1::2, 0::2] + da[:, 0::2, 1::2] + da[:, 1::2, 1::2]
    elif mode == 2:
        gs = da.repeat_interleave(2, 1).repeat_interleave(2, 2) * 0.25
    else:
        gs = da
    pre = xv * s[:, None, None, :] + t[:, None, None, :] if s is not None else xv
    return torch.where(pre > 0, gs, torch.zeros_like(gs)) if relu else gs


def replay_input_bwd(eng, rec, n, seed, betas=None):
    """iea_conv_input_bwd: dx (beta 0 / 1) and dscale / dshift"""
    from iea_gan_b200 import _lib as L
    r = rec["d"]
    h, w, cin = r["h"], r["w"], r["cin"]
    data = Data(seed)
    hs, ws, s, t = prologue(data, r, n)
    unit_da = 0.25 if r["in_mode"] == 2 else 1.0
    p = min(1.0, 2.0 ** 16 / (hs * ws))
    for _ in range(8):
        xv = data.x((n, hs, ws, cin), s, t, r["in_relu"], 1.0)
        da = data.grid((n, h, w, cin), -2, 2, 1, p)
        gm = ref_input_bwd(da, xv, s, t, r["in_relu"], r["in_mode"])
        bsc = (gm.abs() * xv.abs()).sum((1, 2))
        if fits(bsc, unit_da * 0.5) and fits(gm.abs().sum((1, 2)), unit_da):
            break
        p /= 4
    budget(bsc, unit_da * 0.5, "dscale")
    xdt = TD[r["x_dtype"]]
    x = Buf(n * hs * ws, r["x_ld"], cin, xdt, r["x_al"], xv)
    dab = torch.empty(n * h * w, cin, dtype=TD[rec["da_dt"]], device=DEV)
    dab.copy_(da.reshape(-1, cin))
    sc = s.float().contiguous() if s is not None else None
    sh = t.float().contiguous() if t is not None else None
    d = make_desc(r, n, x, scale=sc, shift=sh)
    sm = s[:, None, None, :] if s is not None else 1.0
    out, names = [], set()
    for beta in (betas if betas is not None else sorted({rec["beta"], 1.0 - rec["beta"]})):
        dx = None
        if rec["dx"]:
            old = data.grid((n * hs * ws, cin), -4, 4, 2)
            dx = Buf(n * hs * ws, rec["dx_ld"], cin, TD[rec["dx_dt"]], rec["dx_al"], old)
        dsc = torch.full((n, cin), float("nan"), device=DEV) if rec["ss"] else None
        dsh = torch.full((n, cin), float("nan"), device=DEV) if rec["ss"] else None
        scr = torch.empty(n * 64 * cin * 2, device=DEV) if rec["scratch"] else None
        _, nm = profiled(lambda: L.call("iea_conv_input_bwd", C.byref(d), dab.data_ptr(), rec["da_dt"],
                                        dx.ptr() if dx is not None else None, rec["dx_dt"], rec["dx_ld"], beta,
                                        dsc.data_ptr() if dsc is not None else None,
                                        dsh.data_ptr() if dsh is not None else None,
                                        scr.data_ptr() if scr is not None else None, L.stream()))
        names |= nm
        if dx is not None:
            want = (gm * sm).reshape(-1, cin) + (beta * old if beta else 0)
            e = mismatch(dx.win(), want)
            if e:
                out.append("dx (beta %g): %s" % (beta, e))
            if not dx.outside_ok():
                out.append("dx (beta %g): wrote outside its channel window" % beta)
        if dsc is not None:
            for nm_, got, want in (("dscale", dsc, (gm * xv).sum((1, 2))), ("dshift", dsh, gm.sum((1, 2)))):
                e = mismatch(got, want)
                if e:
                    out.append("%s (beta %g): %s" % (nm_, beta, e))
    return out, names


def ds_vectors(data, events, c):
    """ds1[e][c] in {0, +-1/8}, non-zero for one event per channel (its sum over an event's rows stays in budget);
    ds2[e][c] in {0, +-1/8}"""
    e_of_c = torch.arange(c, device=DEV) % events
    ds1 = data.grid((events, c), -1, 1, 8) * (torch.arange(events, device=DEV)[:, None] == e_of_c[None, :])
    ds2 = data.grid((events, c), -1, 1, 8)
    return ds1, ds2


def replay_out_bwd(eng, rec, rows, seed):
    """iea_conv_out_bwd: g = dy [* (1 - y^2)] + ds1[e] + 2 y ds2[e], with per-event values so a wrong event shows"""
    from iea_gan_b200 import _lib as L
    c, rpe = rec["c"], rec["rpe"]
    events = (rows + rpe - 1) // rpe
    data = Data(seed)
    dy = data.grid((rows, c), -2, 2, 1)
    tanh = rec["act"] == 2
    y = data.grid((rows, c), -7, 7, 8) if tanh else data.grid((rows, c), -8, 8, 2)
    ds1, ds2 = ds_vectors(data, events, c) if rec["ds"] else (None, None)
    want = dy * (1 - y * y) if tanh else dy.clone()
    unit = 1 / 64 if tanh else 0.125
    if ds1 is not None:
        e = torch.arange(rows, device=DEV) // rpe
        want = want + ds1[e] + 2 * y * ds2[e]
    if TD[rec["g_dt"]] == torch.bfloat16:
        budget(want.abs() * 2 ** 14, unit, "g (exact in bf16)")  # |g| / unit < 2^8
    dyb = Buf(rows, rec["dy_ld"], c, TD[rec["dy_dt"]], rec["al"], dy)
    yb = Buf(rows, rec["y_ld"], c, TD[rec["y_dt"]], rec["al"], y)
    g = torch.full((rows, c), float("nan"), dtype=TD[rec["g_dt"]], device=DEV)
    d1 = ds1.float().contiguous() if ds1 is not None else None
    d2 = ds2.float().contiguous() if ds2 is not None else None
    _, names = profiled(lambda: L.call("iea_conv_out_bwd", dyb.ptr(), rec["dy_dt"], rec["dy_ld"], yb.ptr(), rec["y_dt"],
                                       rec["y_ld"], rec["act"], d1.data_ptr() if d1 is not None else None,
                                       d2.data_ptr() if d2 is not None else None, rows, rpe, c, g.data_ptr(),
                                       rec["g_dt"], L.stream()))
    e = mismatch(g, want)
    return (["g: " + e] if e else []), names


def replay_residual(eng, rec, n, seed):
    """iea_residual_bwd: dres (+)= the adjoint of the epilogue's residual read (direct, up2 sum, pool2 quarter)"""
    from iea_gan_b200 import _lib as L
    h, w, mode, res_c, dres_c = rec["h"], rec["w"], rec["res_mode"], rec["res_c"], rec["dres_c"]
    hs, ws = src_res(h, w, mode)
    data = Data(seed)
    g = data.grid((n, h, w, res_c), -2, 2, 1)
    if mode == 1:
        adj = g[:, 0::2, 0::2] + g[:, 1::2, 0::2] + g[:, 0::2, 1::2] + g[:, 1::2, 1::2]
    elif mode == 2:
        adj = g.repeat_interleave(2, 1).repeat_interleave(2, 2) * 0.25
    else:
        adj = g
    adj = torch.cat([adj, torch.zeros(n, hs, ws, dres_c - res_c, dtype=F64, device=DEV)], 3).reshape(-1, dres_c)
    gfull = torch.cat([g, data.grid((n, h, w, rec["g_ld"] - res_c), -2, 2, 1)], 3) if rec["g_ld"] > res_c else g
    gt = gfull.reshape(-1, rec["g_ld"]).to(TD[rec["g_dt"]])
    out, names = [], set()
    for beta in sorted({rec["beta"], 1.0 - rec["beta"]}):
        old = data.grid((n * hs * ws, dres_c), -4, 4, 2)
        db = Buf(n * hs * ws, rec["dres_ld"], dres_c, TD[rec["dres_dt"]], rec["al"], old)
        _, nm = profiled(lambda: L.call("iea_residual_bwd", gt.data_ptr(), rec["g_dt"], rec["g_ld"], n, h, w, res_c, mode,
                                        db.ptr(), rec["dres_dt"], rec["dres_ld"], dres_c, beta, L.stream()))
        names |= nm
        e = mismatch(db.win(), adj + (beta * old if beta else 0))
        if e:
            out.append("dres (beta %g): %s" % (beta, e))
        if not db.outside_ok():
            out.append("dres (beta %g): wrote outside its channel window" % beta)
    return out, names


def replay_colsum(eng, rec, rows, seed):
    """iea_colsum: out[c] (+)= sum over rows of g[row][c]"""
    from iea_gan_b200 import _lib as L
    c = rec["c"]
    data = Data(seed)
    g = data.grid((rows, c), -2, 2, 1, min(1.0, 2.0 ** 19 / rows))
    budget(g.abs().sum(0), 1.0, "colsum")
    gb = Buf(rows, rec["g_ld"], c, TD[rec["g_dt"]], rec["al"], g)
    out, names = [], set()
    for beta in sorted({rec["beta"], 1.0 - rec["beta"]}):
        old = data.grid((c,), -4, 4, 2)
        o = old.float().clone()
        scr = torch.empty(300 * c, device=DEV)
        _, nm = profiled(lambda: L.call("iea_colsum", gb.ptr(), rec["g_dt"], rec["g_ld"], rows, c, o.data_ptr(), beta,
                                        scr.data_ptr(), L.stream()))
        names |= nm
        e = mismatch(o, g.sum(0) + (beta * old if beta else 0))
        if e:
            out.append("colsum (beta %g): %s" % (beta, e))
    return out, names


def replay_bwd1x1(eng, rec, n, seed, beta, with_ds):
    """iea_conv_bwd1x1: dW (slice 0 of wpart), db, dx (beta), dscale / dshift, with geff = g + ds1 + 2 y ds2"""
    from iea_gan_b200 import _lib as L
    r = rec["d"]
    h, w, cin, cout = r["h"], r["w"], r["cin"], r["cout"]
    M, hw = n * h * w, h * w
    rpe = 40 * hw
    events = max(1, n // 40)
    data = Data(seed)
    m, l, grp = sn_layer(eng, cout, cin, 1, torch.bfloat16, data)
    W = m.weight.detach().double().reshape(cout, cin)
    s = t = None
    if r["aff"]:
        s, t = data.affine(1 if r["in_bcast"] else n, cin)
    isg = 0.5
    unit_g, unit_T = 0.125, t_unit(r)
    unit_da = unit_g * 0.125 * isg
    p_g, p_x = min(0.5, 2.0 ** 17 / M), min(1.0, 2.0 ** 15 / rpe)
    for _ in range(12):
        xv = data.x((n, h, w, cin), s, t, r["in_relu"], p_x)
        T = ref_T(xv, s, t, r["in_relu"], 0).reshape(M, cin)
        g = data.grid((M, cout), -2, 2, 1, p_g)
        y = data.grid((M, cout), -8, 8, 2, p_g)
        geff = g
        if with_ds:
            ds1, ds2 = ds_vectors(data, events, cout)
            e = torch.arange(M, device=DEV) // rpe
            geff = g + ds1[e] + 2 * y * ds2[e]
        gm_abs = geff.abs() @ W.abs() * isg
        pre = (xv * s[:, None, None, :] + t[:, None, None, :]) if s is not None else xv
        if r["in_relu"]:
            gm_abs = gm_abs * (pre > 0).reshape(M, cin)
        xa = xv.abs().reshape(n, hw, cin)
        ok = (fits(geff.abs().t() @ T.abs(), unit_g * unit_T) and fits(geff.abs().sum(0), unit_g)
              and fits(gm_abs, unit_da) and fits((gm_abs.view(n, hw, cin) * xa).sum(1), unit_da * 0.5)
              and fits(gm_abs.view(n, hw, cin).sum(1), unit_da))
        if ok:
            break
        p_g, p_x = p_g / 4, p_x / 2
    budget(geff.abs().t() @ T.abs(), unit_g * unit_T, "dW")
    budget(gm_abs.view(n, hw, cin).sum(1), unit_da, "dshift")
    budget((gm_abs.view(n, hw, cin) * xa).sum(1), unit_da * 0.5, "dscale")
    budget(geff.abs() * 2 ** 14, unit_g, "geff (exact in bf16)")
    da = geff @ W * isg
    gm = torch.where(pre.reshape(M, cin) > 0, da, torch.zeros_like(da)) if r["in_relu"] else da
    sm = s.repeat_interleave(hw, 0) if (s is not None and not r["in_bcast"]) else (s if s is not None else 1.0)
    gmq = gm.float().bfloat16().double()  # the dscale / dshift sums take the bf16 gm (as the unfused path's bf16 da)
    x = Buf(M, r["x_ld"], cin, torch.bfloat16, r["x_al"], xv)
    gb = Buf(M, rec["g_ld"], cout, torch.bfloat16, True, g)
    yb = Buf(M, max(rec["y_ld"], cout), cout, torch.bfloat16, True, y)
    old = data.grid((M, cin), -4, 4, 2)
    dx = Buf(M, max(rec["dx_ld"], cin), cin, torch.bfloat16, True, old)
    sc = s.float().contiguous() if s is not None else None
    sh = t.float().contiguous() if t is not None else None
    d = make_desc(r, n, x, wp=l.wp, scale=sc, shift=sh)
    grid = L.call("iea_conv_bwd1x1_grid", C.byref(d))
    if grid <= 0:
        return ["iea_conv_bwd1x1_grid returned %d" % grid], set()
    a = L.Bwd1x1Args()
    a.g, a.g_ld, a.wd_tc = gb.ptr(), gb.ld, l.wd_tc.data_ptr()
    isg_t = torch.tensor([isg], device=DEV)
    a.inv_sigma = isg_t.data_ptr()
    d1 = d2 = None
    if with_ds:
        d1, d2 = ds1.float().contiguous(), ds2.float().contiguous()
        a.y, a.y_ld, a.ds1, a.ds2 = yb.ptr(), yb.ld, d1.data_ptr(), d2.data_ptr()
    a.rows_per_event = rpe
    wpart = torch.full(((grid + 1) * cout * cin + grid * cout,), float("nan"), device=DEV)
    db = torch.full((cout,), float("nan"), device=DEV)
    a.wpart, a.dbias = wpart.data_ptr(), db.data_ptr()
    a.dx, a.dx_ld, a.beta = dx.ptr(), dx.ld, beta
    dsc = dsh = scr = None
    if s is not None:
        dsc = torch.full((n, cin), float("nan"), device=DEV)
        dsh = torch.full((n, cin), float("nan"), device=DEV)
        scr = torch.empty(max(1, L.call("iea_conv_bwd1x1_scratch_floats", C.byref(d))), device=DEV)
        a.dscale, a.dshift, a.scratch = dsc.data_ptr(), dsh.data_ptr(), scr.data_ptr()
    _, names = profiled(lambda: L.call("iea_conv_bwd1x1", C.byref(d), C.byref(a), L.stream()))
    out = []
    checks = [("dW", wpart[:cout * cin].view(cout, cin), geff.t() @ T), ("db", db, geff.sum(0)),
              ("dx", dx.win(), gm * sm + (beta * old if beta else 0))]
    if dsc is not None:
        checks += [("dscale", dsc, (gmq.view(n, hw, cin) * xv.reshape(n, hw, cin)).sum(1)),
                   ("dshift", dsh, gmq.view(n, hw, cin).sum(1))]
    for nm_, got, want in checks:
        e = mismatch(got, want)
        if e:
            out.append("%s (beta %g, ds %d): %s" % (nm_, beta, with_ds, e))
    if not dx.outside_ok():
        out.append("dx: wrote outside its channel window")
    return out, names


# ------------------------------------------------------------------ running the table
def _run(family, label, n, fn):
    try:
        errs, names = fn()
    except Exception:  # an ABI error is a finding of this geometry, not of the whole table
        errs, names = ["raised:\n" + traceback.format_exc(limit=4)], set()
    ROUTES.setdefault((family, label), {})[n] = names
    return ["%s [%s] n=%d: %s" % (family, label, n, e) for e in errs]


def _sizes(n_cap):
    return sorted({n_cap, SMALL_N}, reverse=True)


def _report(fails):
    assert not fails, "%d exact mismatches:\n  " % len(fails) + "\n  ".join(fails[:40])


def test_wgrad_exact(eng, captured):
    """every captured iea_conv_wgrad_mma / iea_conv_wgrad geometry at the step's batch and at 40 images"""
    cap, n_cap = captured
    fails, count = [], 0
    for name, mma in (("iea_conv_wgrad_mma", True), ("iea_conv_wgrad", False)):
        for i, rec in enumerate(cap.get(name, [])):
            for n in _sizes(rec["d"]["n"]):
                fails += _run(name, _label(rec, " gld%d" % rec["g_ld"]), n,
                              lambda: replay_wgrad(eng, rec, n, 1000 + i, mma))
                count += 1
    print("\nwgrad replays: %d" % count)
    assert cap.get("iea_conv_wgrad_mma"), "the train step ran no iea_conv_wgrad_mma"
    _report(fails)


def test_bwd1x1_exact(eng, captured):
    """every captured fused 1x1 backward: dW, db, dx (beta 0 and 1), dscale / dshift, with and without ds1 / ds2;
    at 40 images only when the fused kernel takes the shape there (else the unfused sequence runs)"""
    from iea_gan_b200 import _lib as L
    cap, n_cap = captured
    fails = []
    for i, rec in enumerate(cap.get("iea_conv_bwd1x1", [])):
        for n in _sizes(rec["d"]["n"]):
            if n != rec["d"]["n"] and n * rec["d"]["h"] * rec["d"]["w"] < 148 * 128:
                continue
            for beta, ds in ((0.0, rec["ds"]), (1.0, True)):
                fails += _run("iea_conv_bwd1x1", _label(rec, " ds%d b%g" % (ds, beta)), n,
                              lambda: replay_bwd1x1(eng, rec, n, 2000 + i, beta, ds))
    assert cap.get("iea_conv_bwd1x1"), "the train step ran no iea_conv_bwd1x1"
    _report(fails)


def test_dgrad_exact(eng, captured):
    """every captured data-gradient convolution: da, overwritten and accumulated (acc_c0 = 0)"""
    cap, _ = captured
    fails = []
    for i, rec in enumerate(cap.get("iea_conv_fprop", [])):
        for n in _sizes(rec["d"]["n"]):
            fails += _run("dgrad", _label(rec, " acc%d" % rec["d"]["acc_c0"]), n,
                          lambda: replay_dgrad(eng, rec, n, 3000 + i))
    _report(fails)


def test_input_bwd_exact(eng, captured):
    """every captured iea_conv_input_bwd (direct, up2, pool2; vec, plain and generic kernels): dx with beta 0 and 1,
    dscale / dshift"""
    cap, _ = captured
    fails = []
    for i, rec in enumerate(cap.get("iea_conv_input_bwd", [])):
        for n in _sizes(rec["d"]["n"]):
            fails += _run("input_bwd", _label(rec, " dx%d ss%d" % (rec["dx"], rec["ss"])), n,
                          lambda: replay_input_bwd(eng, rec, n, 4000 + i))
    _report(fails)


def test_out_residual_colsum_exact(eng, captured):
    """every captured iea_conv_out_bwd (8 events of ds1 / ds2), iea_residual_bwd (beta 0 and 1) and iea_colsum"""
    cap, n_cap = captured
    fails = []
    for i, rec in enumerate(cap.get("iea_conv_out_bwd", [])):
        for rows in sorted({rec["rows"], rec["rows"] * SMALL_N // n_cap}, reverse=True):
            fails += _run("out_bwd", "c%d act%d ds%d rows%d" % (rec["c"], rec["act"], rec["ds"], rec["rows"]), rows,
                          lambda: replay_out_bwd(eng, rec, rows, 5000 + i))
    for i, rec in enumerate(cap.get("iea_residual_bwd", [])):
        for n in _sizes(rec["n"]):
            fails += _run("residual_bwd", "%dx%d c%d/%d mode%d" % (rec["h"], rec["w"], rec["res_c"], rec["dres_c"],
                                                                   rec["res_mode"]), n,
                          lambda: replay_residual(eng, rec, n, 6000 + i))
    for i, rec in enumerate(cap.get("iea_colsum", [])):
        for rows in sorted({rec["rows"], max(1, rec["rows"] * SMALL_N // n_cap)}, reverse=True):
            fails += _run("colsum", "c%d rows%d" % (rec["c"], rec["rows"]), rows,
                          lambda: replay_colsum(eng, rec, rows, 7000 + i))
    _report(fails)


# ------------------------------------------------------------------ hand cases
def conv_rec(h, w, cin, cout, k, *, n=320, mode=0, relu=True, aff=True, x_ld=None, x_dtype=1):
    return dict(n=n, h=h, w=w, cin=cin, cout=cout, ksize=k, x_dtype=x_dtype, x_ld=x_ld or cin, in_mode=mode,
                in_relu=int(relu), in_bcast=0, w_dtype=1, cout_tc=(cout + 15) // 16 * 16, out_scale_stride=0,
                res_dtype=0, res_ld=0, res_mode=0, res_c=0, acc_c0=-1, y_dtype=1, y_ld=cout, act=0, aff=aff, tc=False,
                osc=False, bias_=False, res_=False, x_al=True, y_al=True)


HAND = [  # (what, forward geometry, g_dtype, g_ld)
    ("1x1 on 12x20 images: tiles straddle images, per-pixel affine", conv_rec(12, 20, 32, 32, 1), 1, 32),
    ("1x1 on 12x20 images, 64 -> 128", conv_rec(12, 20, 64, 128, 1), 1, 128),
    ("3x3 at 8x8: one masked edge tile per image", conv_rec(8, 8, 32, 32, 3), 1, 32),
    ("3x3 at 4x4: one masked edge tile per image", conv_rec(4, 4, 32, 16, 3), 1, 16),
    ("H_base 3 width 4x12", conv_rec(4, 12, 128, 128, 3), 1, 128),
    ("H_base 3 width 8x24", conv_rec(8, 24, 32, 32, 3), 1, 32),
    ("H_base 3 width 16x48", conv_rec(16, 48, 16, 16, 3), 1, 16),
    ("channel windows x_ld > cin, g_ld > cout", conv_rec(16, 16, 32, 16, 3, x_ld=48), 1, 32),
    ("channel windows, 1x1", conv_rec(32, 32, 16, 32, 1, x_ld=64), 1, 48),
    ("up2 input 3x3", conv_rec(32, 32, 16, 16, 3, mode=1), 1, 16),
    ("pool2 input 1x1", conv_rec(16, 16, 64, 32, 1, mode=2, aff=False), 1, 32),
    ("D stem: 1 -> 32 3x3, fp32 image", conv_rec(64, 64, 1, 32, 3, relu=False, aff=False, x_dtype=0), 1, 32),
    ("G output conv: 32 -> 1 3x3", conv_rec(64, 64, 32, 1, 3), 0, 1),
]


@pytest.mark.parametrize("case", range(len(HAND)), ids=[h[0] for h in HAND])
def test_hand_cases_exact(eng, case):
    """shapes the train step does not produce but the ABI accepts, through iea_conv_wgrad_mma and iea_conv_wgrad,
    at 320 and 40 images"""
    what, r, gdt, gld = HAND[case]
    rec = dict(d=r, g_dt=gdt, g_ld=gld, g_al=True, db=True)
    fails = []
    for n in (320, SMALL_N):
        fails += _run("hand wgrad_mma", what, n, lambda: replay_wgrad(eng, rec, n, 8000 + case, True))
        fails += _run("hand wgrad", what, n, lambda: replay_wgrad(eng, rec, n, 8100 + case, False))
    _report(fails)


def test_hand_tanh_output_conv_exact(eng):
    """G's 32 -> 1 output conv: the ACT_TANH conv_out_bwd dy (1 - y^2) with y in {-7..7}/8, bf16 and fp32, then the
    1-channel weight gradient of its result"""
    fails = []
    for n in (320, SMALL_N):
        rows = n * 64 * 64
        for gdt in (0, 1):
            rec = dict(dy_dt=gdt, dy_ld=1, y_dt=gdt, y_ld=1, act=2, ds=False, rows=rows, rpe=40 * 64 * 64, c=1, g_dt=gdt,
                       al=True)
            fails += _run("hand out_bwd", "tanh c1 dt%d" % gdt, rows, lambda: replay_out_bwd(eng, rec, rows, 8200 + gdt))
        rec = dict(dy_dt=1, dy_ld=16, y_dt=1, y_ld=16, act=0, ds=True, rows=n * 4096, rpe=40 * 4096, c=16, g_dt=1,
                   al=True)
        fails += _run("hand out_bwd", "ds c16 ld16", n, lambda: replay_out_bwd(eng, rec, n * 4096, 8210))
    _report(fails)


# ------------------------------------------------------------------ route coverage
WANT_KERNELS = ["c1_wgrad_kernel", "wgrad_tc_kernel", "wgrad3_kernel", "wgrad_mma_kernel<9", "wgrad_mma_kernel<1",
                "conv_wgrad_generic", "bwd1x1_kernel", "conv_input_bwd_plain", "conv_input_bwd_vec", "conv_out_bwd_vec"]


def test_route_coverage(eng, captured):
    """the replays above reached every backward kernel, and some geometry runs a different weight-gradient or fused
    1x1 kernel at the step's batch than at 40 images (those shapes were not reached by a 40-image test before)"""
    assert ROUTES, "run the whole module: the replays record the kernels"
    missing = [k for k in WANT_KERNELS if not any(k in s for s in SEEN)]
    print("\nkernels seen: " + ", ".join(sorted(k for k in WANT_KERNELS if k not in missing)))
    differ = []
    for (family, label), by_n in sorted(ROUTES.items()):
        if family not in ("iea_conv_wgrad_mma", "iea_conv_bwd1x1", "hand wgrad_mma") or len(by_n) < 2:
            continue
        ks = {n: kernel_of(v) for n, v in by_n.items()}
        if len(set(ks.values())) > 1:
            differ.append("%s [%s]: %s" % (family, label, ", ".join("n=%d %s" % kv for kv in sorted(ks.items()))))
    print("geometries whose kernel differs between batches:\n  " + "\n  ".join(differ))
    assert not missing, "kernels no replay reached: %s" % missing
    assert differ, "no geometry changes kernel between 40 images and the step's batch"
