"""ctypes binding of libiea_sm100.so (C ABI in include/iea_b200.h).

The shared library is built in-tree by `make -C iea_gan_b200/csrc` (or
__graft_entry__.build()).  There is no fallback: if the library is missing or
the device is not sm_100, every call raises.
"""
import ctypes as C
import os
import subprocess

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libiea_sm100.so")

F32, BF16 = 0, 1
IN_DIRECT, IN_UP2, IN_POOL2 = 0, 1, 2
ACT_NONE, ACT_RELU, ACT_TANH = 0, 1, 2
IMPL_AUTO, IMPL_GENERIC, IMPL_TCGEN05, IMPL_TC_STREAM = 0, 1, 2, 3

vp, i32, i64, f32 = C.c_void_p, C.c_int32, C.c_int64, C.c_float


class SnLayer(C.Structure):
    _fields_ = [("w", vp), ("u_in", vp), ("u_out", vp), ("v_out", vp), ("sigma_out", vp),
                ("inv_sigma_out", vp), ("colscale_out", vp), ("pack_fprop", vp), ("pack_dgrad", vp),
                ("rows", i32), ("cin", i32), ("taps", i32), ("colscale_n", i32), ("pack_dgrad_ld", i32),
                ("pack_tc_fprop", vp), ("pack_tc_dgrad", vp), ("pack_tc_rows", i32), ("pack_tc_cin", i32),
                ("pack_dtype", i32), ("spectral", i32), ("eps", f32), ("chunk0", i32), ("nchunks", i32),
                ("scratch_off", i64)]


class SnBwdItem(C.Structure):
    _fields_ = [("gpart", vp), ("w", vp), ("u", vp), ("v", vp), ("inv_sigma", vp), ("dw", vp),
                ("nsplit", i32), ("spectral", i32), ("rows", i32), ("cin", i32), ("taps", i32), ("beta", f32),
                ("block0", i32), ("nblocks", i32)]


class ConvDesc(C.Structure):
    _fields_ = [("n", i64), ("h", i32), ("w", i32), ("cin", i32), ("cout", i32), ("ksize", i32),
                ("x", vp), ("x_dtype", i32), ("x_ld", i32), ("in_mode", i32), ("in_relu", i32),
                ("in_scale", vp), ("in_shift", vp), ("in_bcast", i32),
                ("wpack", vp), ("w_dtype", i32), ("wpack_tc", vp), ("cout_tc", i32),
                ("out_scale", vp), ("out_scale_stride", i32), ("bias", vp),
                ("res", vp), ("res_dtype", i32), ("res_ld", i32), ("res_mode", i32), ("res_c", i32),
                ("acc_c0", i32), ("y", vp), ("y_dtype", i32), ("y_ld", i32), ("act", i32),
                ("stats", vp), ("impl", i32)]


class MtChunk(C.Structure):
    _fields_ = [("p", vp), ("g", vp), ("m", vp), ("v", vp), ("ema", vp), ("n", i32), ("tensor", i32)]


class Bwd1x1Args(C.Structure):
    _fields_ = [("g", vp), ("y", vp), ("ds1", vp), ("ds2", vp), ("wd_tc", vp), ("inv_sigma", vp), ("dx", vp), ("wpart", vp),
                ("dbias", vp), ("dscale", vp), ("dshift", vp), ("scratch", vp), ("rows_per_event", i64), ("g_ld", i32),
                ("y_ld", i32), ("dx_ld", i32), ("beta", f32)]


class OrthoItem(C.Structure):
    _fields_ = [("w", vp), ("grad", vp), ("gram", vp), ("rownorm", vp), ("gram_part", vp), ("rows", i32), ("cols", i32),
                ("tall", i32), ("strength", f32), ("ksplits", i32), ("pad_", i32)]


class AugDraws(C.Structure):
    _fields_ = [("brightness", vp), ("contrast", vp), ("tx", vp), ("ty", vp), ("ox", vp), ("oy", vp),
                ("cut_h", i32), ("cut_w", i32)]


_SIG = {
    "iea_version": [],
    "iea_require_sm100": [i32],
    "iea_sm_count": [i32],
    "iea_sn_power_iter": [vp, i32, vp, i32, vp, i32, vp],
    "iea_sn_weight_bwd": [vp, i32, vp, vp, vp, vp, i32, vp, f32, i32, i32, i32, vp, vp],
    "iea_sn_weight_bwd_grouped": [vp, i32, i32, vp, vp],
    "iea_conv_fprop": [vp, vp],
    "iea_conv_tc_supported": [vp],
    "iea_conv_stats_slots": [vp],
    "iea_conv_wgrad": [vp, vp, i32, i32, vp, i32, vp],
    "iea_conv_wgrad_mma_slices": [vp, i32, i32],
    "iea_conv_wgrad_mma": [vp, vp, i32, i32, vp, vp, vp],
    "iea_conv_input_bwd": [vp, vp, i32, vp, i32, i32, f32, vp, vp, vp, vp],
    "iea_conv_out_bwd": [vp, i32, i32, vp, i32, i32, i32, vp, vp, i64, i32, i32, vp, i32, vp],
    "iea_colsum": [vp, i32, i32, i64, i32, vp, f32, vp, vp],
    "iea_residual_bwd": [vp, i32, i32, i64, i32, i32, i32, i32, vp, i32, i32, i32, f32, vp],
    "iea_bn_stats": [vp, i32, i32, i64, i32, i32, i32, vp, vp],
    "iea_bn_finalize": [vp, i32, i32, i64, i32, i32, vp, i64, f32, vp, i64, vp, vp, i32, f32, f32, vp, vp, vp, vp, vp, vp],
    "iea_bn_finalize_bwd": [vp, vp, vp, vp, vp, i32, i32, i64, i32, vp, i64, f32, vp, i64, vp, i64, i32, i32, vp, vp, vp],
    "iea_affine_act": [vp, i32, vp, vp, i64, i64, i32, i32, vp, i32, vp],
    "iea_nchw_to_nhwc": [vp, i32, vp, i32, i64, i32, i64, vp],
    "iea_nhwc_to_nchw": [vp, i32, vp, i32, i64, i32, i64, vp],
    "iea_axpby": [vp, i32, f32, vp, i32, f32, vp, i32, i64, vp],
    "iea_gamma_residual": [vp, vp, i32, vp, vp, i64, vp],
    "iea_gamma_residual_bwd": [vp, vp, i32, vp, vp, vp, vp, i64, vp],
    "iea_embedding_fwd": [vp, vp, vp, i64, i32, vp, vp],
    "iea_embedding_bwd": [vp, vp, vp, i64, i32, i32, vp, vp],
    "iea_relu_sumpool_fwd": [vp, i32, i64, i64, i32, vp, vp],
    "iea_relu_sumpool_bwd": [vp, i32, vp, i64, i64, i32, vp, i32, vp],
    "iea_avgpool2_fwd": [vp, i32, i64, i32, i32, i32, i32, vp, i32, vp],
    "iea_maxpool2_fwd": [vp, i32, i64, i32, i32, i32, vp, vp, vp],
    "iea_maxpool2_bwd": [vp, i32, vp, i64, i32, i32, i32, vp, vp],
    "iea_layernorm_fwd": [vp, vp, vp, i64, i32, f32, vp, vp, vp, vp],
    "iea_layernorm_bwd": [vp, vp, vp, vp, vp, i64, i32, vp, vp, vp, i32, vp],
    "iea_l2norm_fwd": [vp, i64, i32, f32, vp, vp, vp],
    "iea_l2norm_bwd": [vp, vp, vp, i64, i32, f32, vp, vp],
    "iea_mha_fwd": [vp, i32, i32, i32, i32, vp, vp, vp],
    "iea_mha_bwd": [vp, vp, vp, i32, i32, i32, i32, vp, vp],
    "iea_attn_fwd": [vp, vp, vp, i32, i64, i32, i32, i32, i32, vp, vp, vp],
    "iea_attn_bwd": [vp, vp, vp, vp, vp, vp, i32, i64, i32, i32, i32, i32, vp, vp, vp, vp, vp],
    "iea_diffaug_fwd": [vp, vp, i64, i32, i32, vp, vp, vp],
    "iea_diffaug_bwd": [vp, vp, i64, i32, i32, vp, vp, vp],
    "iea_loss_hinge_dis": [vp, vp, i64, vp, vp],
    "iea_loss_hinge_dis_bwd": [vp, vp, vp, i64, vp, vp, vp],
    "iea_loss_mean": [vp, i64, f32, vp, vp],
    "iea_loss_mean_bwd": [vp, i64, f32, vp, vp],
    "iea_loss_scratch_floats": [i32, i32, i32],
    "iea_loss_l2": [vp, vp, i64, vp, vp],
    "iea_loss_l2_bwd": [vp, vp, vp, i64, vp, vp, vp],
    "iea_loss_contrastive_fwd": [vp, vp, i32, i32, i32, f32, f32, vp, vp, vp, vp],
    "iea_loss_contrastive_bwd": [vp, vp, vp, vp, i32, i32, i32, f32, vp, vp, vp],
    "iea_loss_iea_fwd": [vp, vp, i32, i32, i32, vp, vp, vp, vp],
    "iea_loss_iea_bwd": [vp, vp, vp, i32, i32, i32, vp, vp],
    "iea_loss_unif_fwd": [vp, i32, i32, i32, f32, vp, vp, vp, vp],
    "iea_loss_unif_bwd": [vp, vp, vp, i32, i32, i32, f32, vp, vp],
    "iea_adu_postprocess": [vp, i64, i32, i32, vp, vp],
    "iea_event_preprocess": [vp, i64, i32, i32, i32, vp, f32, vp, vp],
    "iea_conv_bwd1x1_grid": [vp],
    "iea_conv_bwd1x1_scratch_floats": [vp],
    "iea_conv_bwd1x1": [vp, vp, vp],
    "iea_mt_sqnorm": [vp, i32, vp, vp],
    "iea_mt_adam": [vp, i32, vp, f32, f32, f32, f32, vp, vp, vp],
    "iea_mt_lerp": [vp, i32, vp, vp],
    "iea_ortho_grouped": [vp, vp, i32, vp, i32, vp, i32, vp, i32, vp],
}

_RET64 = {"iea_loss_scratch_floats", "iea_conv_bwd1x1_scratch_floats"}  # sizes come back as int64_t; everything else is an int status
_lib = None
_checked_devices = set()


def build(force=False):
    """Compile libiea_sm100.so in-tree with nvcc for sm_100a (needs no GPU)."""
    src = os.path.join(_HERE, "csrc")
    if force:
        subprocess.check_call(["make", "-C", src, "clean"], stdout=subprocess.DEVNULL)
    subprocess.check_call(["make", "-C", src, "-j8"], stdout=subprocess.DEVNULL)
    return LIB_PATH


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError("libiea_sm100.so is not built (%s): run `make -C iea_gan_b200/csrc` or "
                              "__graft_entry__.build(); there is no fallback path" % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        L.iea_last_error.restype = C.c_char_p
        L.iea_last_error.argtypes = []
        for name, sig in _SIG.items():
            fn = getattr(L, name)  # raises AttributeError if the symbol is not exported
            fn.restype = C.c_int64 if name in _RET64 else C.c_int
            fn.argtypes = sig
        _lib = L
    return _lib


def exported_symbols():
    return list(_SIG.keys()) + ["iea_last_error"]


_FN = {}


def call(name, *args):
    fn = _FN.get(name)
    if fn is None:
        fn = _FN[name] = getattr(lib(), name)
    rc = fn(*args)
    if rc < 0:
        raise RuntimeError("%s failed (%d): %s" % (name, rc, lib().iea_last_error().decode()))
    return rc


def require_device(t):
    """No CPU path: every tensor handed to a kernel must live on an sm_100 CUDA device."""
    if not t.is_cuda:
        raise RuntimeError("iea_gan_b200 kernels need CUDA tensors on a B200 (sm_100a); got a %s tensor and "
                           "there is no CPU fallback" % t.device)
    idx = t.device.index if t.device.index is not None else torch.cuda.current_device()
    if idx not in _checked_devices:
        call("iea_require_sm100", idx)
        _checked_devices.add(idx)
    return idx


def ptr(t):
    return None if t is None else t.data_ptr()


def dt(t):
    if t.dtype == torch.float32:
        return F32
    if t.dtype == torch.bfloat16:
        return BF16
    raise TypeError("unsupported dtype %s (kernels take float32 / bfloat16)" % t.dtype)


def stream():
    """Raw handle of torch's current CUDA stream (the C-level getter: torch.cuda.current_stream() builds a
    Stream object and re-resolves the device on every call, ~15 us x 1300 calls per train step)."""
    try:
        return torch._C._cuda_getCurrentRawStream(torch._C._cuda_getDevice())
    except AttributeError:  # private API moved: the public path
        return torch.cuda.current_stream().cuda_stream
