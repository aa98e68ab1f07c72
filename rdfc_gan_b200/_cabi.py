"""ctypes binding of librdfc_b200.so (include/rdfc_b200.h).  There is no fallback: if the library is missing the
import fails, and every call raises RuntimeError with rdfc_last_error() on a non-zero status -- the same exception
type the reference's AT_ASSERTM / AT_ERROR surface in Python (deformconv/src/modulated_deform_conv.h:43)."""
import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "librdfc_b200.so")

F32, F64, BF16, F16 = 0, 1, 2, 3          # F16: the split [hi | lo] tensors of the fp32_tc training mode
ACT_NONE, ACT_RELU, ACT_LEAKY02, ACT_TANH, ACT_SIGMOID = range(5)
PATH_SIMT_F32, PATH_UMMA_BF16, PATH_UMMA_F32X3 = 0, 1, 2
AFFINITY = {"AS": 0, "ASS": 1, "TC": 2, "TGASS": 3}
DETERMINISTIC = 1                         # flags of the *_ex backward entry points
PAD_REFLECT, PAD_REPLICATE = 0, 1
_DT = {torch.float32: F32, torch.float64: F64, torch.bfloat16: BF16, torch.float16: F16}

c_int, c_void_p, c_float = ctypes.c_int, ctypes.c_void_p, ctypes.c_float


class FuseOut(ctypes.Structure):
    _fields_ = [("d1", c_void_p), ("c1", c_void_p), ("c2", c_void_p), ("pred", c_void_p)]


class DcnShape(ctypes.Structure):
    _fields_ = [(n, c_int) for n in ("B", "Cin", "H", "W", "Cout", "kh", "kw", "sh", "sw", "ph", "pw", "dh", "dw",
                                     "group", "deformable_group", "im2col_step")]


class View(ctypes.Structure):
    _fields_ = [("ptr", c_void_p), ("dtype", c_int), ("C", c_int), ("pix_stride", c_int), ("nchw", c_int)]


class ConvDesc(ctypes.Structure):
    _fields_ = [("B", c_int), ("Hi", c_int), ("Wi", c_int), ("Ho", c_int), ("Wo", c_int), ("kh", c_int), ("kw", c_int),
                ("stride", c_int), ("pad", c_int), ("transposed", c_int), ("act", c_int), ("path", c_int),
                ("inp", View), ("in2", View), ("out", View), ("residual", View), ("weight", c_void_p),
                ("scale", c_void_p), ("shift", c_void_p), ("workspace", c_void_p), ("workspace_bytes", ctypes.c_size_t)]


class HeadsDesc(ctypes.Structure):
    _fields_ = [("B", c_int), ("H", c_int), ("W", c_int), ("inp", View), ("weight", c_void_p), ("shift", c_void_p),
                ("ncols", c_int), ("act", c_int * 16), ("out", c_void_p * 16), ("out_bstride", ctypes.c_longlong * 16),
                ("workspace", c_void_p), ("workspace_bytes", ctypes.c_size_t)]


class StemDesc(ctypes.Structure):
    _fields_ = [("B", c_int), ("H", c_int), ("W", c_int), ("in0", c_void_p), ("C0", c_int), ("in1", c_void_p),
                ("out", View), ("out2", View), ("weight", c_void_p), ("scale", c_void_p), ("shift", c_void_p), ("act", c_int)]


class WadainConvDesc(ctypes.Structure):
    _fields_ = [("B", c_int), ("H", c_int), ("W", c_int), ("style", View), ("x", View), ("out", View), ("weight", c_void_p),
                ("bias", c_void_p), ("mean", c_void_p), ("rstd", c_void_p), ("gwbw", View)]


class WgradDesc(ctypes.Structure):
    _fields_ = [("B", c_int), ("Hg", c_int), ("Wg", c_int), ("Hi", c_int), ("Wi", c_int), ("k", c_int), ("stride", c_int),
                ("pad", c_int), ("grad_out", View), ("input", View)]


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -m rdfc_gan_b200.build` (nvcc, sm_100a). "
            "rdfc_gan_b200 has no CPU or PyTorch fallback.")
    lib = ctypes.CDLL(LIB_PATH)
    lib.rdfc_last_error.restype = ctypes.c_char_p
    lib.rdfc_launch_count.restype = ctypes.c_uint64
    lib.rdfc_fuse_depth_forward.argtypes = [c_void_p] * 6 + [ctypes.c_size_t, c_void_p]
    lib.rdfc_dcn_forward.argtypes = [c_void_p] * 6 + [ctypes.POINTER(DcnShape), c_int, c_void_p]
    lib.rdfc_dcn_backward.argtypes = [c_void_p] * 10 + [ctypes.POINTER(DcnShape), c_int, c_void_p]
    lib.rdfc_dcn_out_size.argtypes = [ctypes.POINTER(DcnShape), ctypes.POINTER(c_int), ctypes.POINTER(c_int)]
    lib.rdfc_nlspn_affinity_forward.argtypes = [c_void_p] * 5 + [c_int, c_int, c_void_p, c_void_p, c_int, c_int, c_int,
                                                                c_void_p]
    lib.rdfc_nlspn_propagate_forward.argtypes = [c_void_p] * 4 + [c_int] + [c_void_p] * 3 + [c_int] * 5 + [ctypes.POINTER(FuseOut), c_void_p]
    lib.rdfc_nlspn_packed_bytes.argtypes = [c_int] * 3
    lib.rdfc_nlspn_packed_bytes.restype = ctypes.c_size_t
    lib.rdfc_nlspn_affinity_forward_packed.argtypes = [c_void_p] * 5 + [c_int, c_int, c_void_p, c_int, c_int, c_int, c_void_p]
    lib.rdfc_nlspn_propagate_forward_packed.argtypes = [c_void_p] * 3 + [c_int] + [c_void_p] * 2 + [c_int] * 5 + [ctypes.POINTER(FuseOut), c_void_p]
    lib.rdfc_dev_set_knob.argtypes = [ctypes.c_char_p, ctypes.c_longlong]
    VP = ctypes.POINTER(View)
    lib.rdfc_bn_workspace_floats.argtypes = [ctypes.c_longlong, c_int]
    lib.rdfc_bn_stats.argtypes = [VP, ctypes.c_longlong, c_void_p, c_void_p, c_void_p, c_void_p]
    lib.rdfc_affine_act_forward.argtypes = [VP, c_void_p, c_void_p, VP, c_int, VP, ctypes.c_longlong, c_void_p]
    lib.rdfc_bn_act_backward.argtypes = [VP, VP, VP, c_void_p, c_void_p, c_void_p, c_int, VP, VP, c_void_p, c_void_p, c_void_p,
                                         ctypes.c_longlong, c_void_p]
    lib.rdfc_bn_frozen_backward.argtypes = [VP, VP, c_int, VP, c_void_p, c_void_p, ctypes.c_longlong, c_void_p]
    lib.rdfc_conv_wgrad_workspace_floats.argtypes = [ctypes.POINTER(WgradDesc)]
    lib.rdfc_conv_wgrad_workspace_floats.restype = ctypes.c_longlong
    lib.rdfc_conv_wgrad.argtypes = [ctypes.POINTER(WgradDesc), c_void_p, c_void_p, c_void_p]
    lib.rdfc_split_scaled.argtypes = [VP, ctypes.c_longlong, VP, c_void_p, c_void_p]
    lib.rdfc_conv_forward_split.argtypes = [ctypes.POINTER(ConvDesc), c_void_p]
    lib.rdfc_conv_wgrad_split_workspace_floats.argtypes = [ctypes.POINTER(WgradDesc)]
    lib.rdfc_conv_wgrad_split_workspace_floats.restype = ctypes.c_longlong
    lib.rdfc_conv_wgrad_split.argtypes = [ctypes.POINTER(WgradDesc), c_void_p, c_void_p, c_void_p, c_void_p]
    lib.rdfc_pad_nhwc_forward.argtypes = [VP] + [c_int] * 5 + [VP, c_void_p]
    lib.rdfc_pad_nhwc_backward.argtypes = [VP] + [c_int] * 5 + [VP, c_void_p]
    lib.rdfc_first_conv_forward.argtypes = [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_int, VP, c_void_p]
    lib.rdfc_maxpool3x3s2_forward.argtypes = [VP, VP, c_int, c_int, c_int, c_void_p]
    lib.rdfc_se_weights.argtypes = [c_void_p] * 6 + [c_int, c_int, c_int, c_void_p]
    lib.rdfc_adaptive_avgpool_forward.argtypes = [VP, VP, c_int, c_int, c_int, c_int, c_void_p]
    lib.rdfc_upsample_nearest_forward.argtypes = [VP, VP, c_int, c_int, c_int, c_int, c_int, c_void_p]
    lib.rdfc_upsample_dw_forward.argtypes = [VP, c_void_p, c_void_p, VP, VP, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p]
    lib.rdfc_depth_metric_nchunk.argtypes = [ctypes.c_longlong]
    lib.rdfc_depth_metric_sums.argtypes = [c_void_p] * 3 + [ctypes.c_float] * 3 + [c_void_p] * 2 + [c_int, ctypes.c_longlong, c_void_p]
    lib.rdfc_nlspn_affinity_backward.argtypes = [c_void_p] * 5 + [c_int] * 2 + [c_void_p] * 6 + [c_int] * 3 + [c_void_p]
    lib.rdfc_nlspn_propagate_backward.argtypes = [c_void_p] * 7 + [c_int] + [c_void_p] * 4 + [c_int] * 4 + [c_void_p]
    for name in ("rdfc_dcn_backward", "rdfc_nlspn_affinity_backward", "rdfc_nlspn_propagate_backward"):
        getattr(lib, name + "_ex").argtypes = getattr(lib, name).argtypes + [c_int]
    lib.rdfc_conv_forward.argtypes = [ctypes.POINTER(ConvDesc), c_void_p]
    lib.rdfc_heads_forward.argtypes = [ctypes.POINTER(HeadsDesc), c_void_p]
    lib.rdfc_stem_forward.argtypes = [ctypes.POINTER(StemDesc), c_void_p]
    lib.rdfc_pack_stem_input.argtypes = [c_void_p, c_int, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p]
    lib.rdfc_wadain_conv_forward.argtypes = [ctypes.POINTER(WadainConvDesc), c_void_p]
    lib.rdfc_wadain_tile.argtypes = [c_int]
    lib.rdfc_instnorm_stats.argtypes = [ctypes.POINTER(View), c_int, c_int, c_int, c_float, c_int, c_int, c_void_p,
                                        c_void_p, c_void_p, c_void_p]
    lib.rdfc_wadain_apply.argtypes = [ctypes.POINTER(View)] * 4 + [c_void_p, c_void_p, ctypes.POINTER(View), c_int,
                                                                  c_int, c_int, c_void_p]
    lib.rdfc_adain_apply.argtypes = [ctypes.POINTER(View)] + [c_void_p] * 4 + [ctypes.POINTER(View), c_int, c_int,
                                                                              c_int, c_void_p]
    lib.rdfc_norm_apply.argtypes = [ctypes.POINTER(View), c_void_p, c_void_p, ctypes.POINTER(View), c_int, c_int,
                                    c_int, c_void_p]
    lib.rdfc_instnorm_nchunk.argtypes = [c_int]
    return lib


lib = _load()

EXPORTS = ["rdfc_abi_version", "rdfc_last_error", "rdfc_launch_count", "rdfc_dcn_out_size", "rdfc_dcn_forward",
           "rdfc_dcn_backward", "rdfc_nlspn_affinity_forward", "rdfc_nlspn_propagate_forward", "rdfc_nlspn_propagate_backward", "rdfc_nlspn_affinity_backward",
           "rdfc_nlspn_packed_bytes", "rdfc_nlspn_affinity_forward_packed", "rdfc_nlspn_propagate_forward_packed",
           "rdfc_fuse_depth_forward", "rdfc_conv_forward", "rdfc_heads_forward", "rdfc_instnorm_nchunk", "rdfc_instnorm_stats",
           "rdfc_wadain_apply", "rdfc_adain_apply", "rdfc_norm_apply", "rdfc_depth_metric_nchunk", "rdfc_depth_metric_sums", "rdfc_stem_forward", "rdfc_pack_stem_input",
           "rdfc_wadain_tile", "rdfc_wadain_conv_forward", "rdfc_dev_set_knob", "rdfc_dev_umma_timers",
           "rdfc_bn_workspace_floats", "rdfc_bn_stats", "rdfc_affine_act_forward", "rdfc_bn_act_backward",
           "rdfc_conv_wgrad_workspace_floats", "rdfc_conv_wgrad", "rdfc_first_conv_forward", "rdfc_maxpool3x3s2_forward", "rdfc_se_weights",
           "rdfc_adaptive_avgpool_forward", "rdfc_upsample_nearest_forward", "rdfc_upsample_dw_forward",
           "rdfc_split_scaled", "rdfc_conv_forward_split", "rdfc_conv_wgrad_split_workspace_floats", "rdfc_conv_wgrad_split",
           "rdfc_dcn_backward_ex", "rdfc_nlspn_affinity_backward_ex", "rdfc_nlspn_propagate_backward_ex",
           "rdfc_pad_nhwc_forward", "rdfc_pad_nhwc_backward", "rdfc_bn_frozen_backward"]


KNOB_UNSET = -(1 << 63)


def set_knob(name, value=None):
    """Development knobs (the RDFC_* environment variables, cached by the library on first use): override one at run time;
    value None restores the default."""
    check(lib.rdfc_dev_set_knob(name.encode(), KNOB_UNSET if value is None else int(value)))


def backward_call(name, *args):
    """Call the backward entry point `name`; under torch.use_deterministic_algorithms (read at call time, warn_only included) its
    _ex variant with DETERMINISTIC, whose scatters accumulate in 64-bit fixed point and are bit-reproducible."""
    if torch.are_deterministic_algorithms_enabled():
        check(getattr(lib, name + "_ex")(*args, DETERMINISTIC))
    else:
        check(getattr(lib, name)(*args))


def check(rc):
    if rc != 0:
        raise RuntimeError(lib.rdfc_last_error().decode("utf-8", "replace"))


def launch_count():
    return int(lib.rdfc_launch_count())


def stream_ptr(device=None):
    return c_void_p(torch.cuda.current_stream(device).cuda_stream)


def ptr(t):
    return None if t is None else c_void_p(t.data_ptr())


def dtype_code(t):
    try:
        return _DT[t.dtype]
    except KeyError:
        raise RuntimeError(f"rdfc_gan_b200: unsupported dtype {t.dtype}") from None


def require_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            # deformconv/src/modulated_deform_conv.h:43
            raise RuntimeError("Not implemented on the CPU")


def view(t, C=None, c0=0, nchw=False):
    """View over an NHWC tensor (B,H,W,Ctot) selecting channels [c0, c0+C); or over a contiguous NCHW tensor."""
    if t is None:
        return View(None, 0, 0, 0, 0)
    if nchw:
        assert t.is_contiguous()
        return View(t.data_ptr(), dtype_code(t), t.shape[1], 0, 1)
    assert t.dim() == 4 and nhwc_viewable(t), "NHWC tensor (or a channel slice of one) expected"
    ctot = t.shape[3]
    C = ctot - c0 if C is None else C
    assert 0 <= c0 and c0 + C <= ctot
    return View(t.data_ptr() + c0 * t.element_size(), dtype_code(t), C, ctot if t.is_contiguous() else t.stride(2), 0)


def nhwc_viewable(t):
    """True if ``t`` (B,H,W,C) is a dense NHWC tensor or a CHANNEL SLICE of one (what autograd hands back for the inputs of a
    torch.cat along the channels): channels contiguous, one pixel pitch S >= C for the three outer dimensions.  Such tensors go to
    the kernels as (pointer, C, pixel stride) views -- no .contiguous() copy."""
    if t.dim() != 4:
        return False
    if t.is_contiguous():
        return True
    B, H, W, Cc = t.shape
    sb, sh, sw, sc = t.stride()
    return (sc == 1 and sw >= Cc and sw % 8 == 0 and (H == 1 or sh == W * sw) and (B == 1 or sb == H * W * sw) and W > 1
            and t.data_ptr() % 16 == 0)
