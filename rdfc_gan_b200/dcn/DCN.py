"""Drop-in for the reference's compiled pybind module ``DCN`` (nlspn/deformconv/src/vision.cpp:7-12).

Same six names, same positional signatures, same return conventions (fresh contiguous NCHW tensors; backward returns
a list), same RuntimeError conditions -- but the work is done by librdfc_b200.so through its C ABI
(include/rdfc_b200.h: rdfc_dcn_forward / rdfc_dcn_backward; under torch.use_deterministic_algorithms the backward calls
rdfc_dcn_backward_ex with RDFC_DETERMINISTIC, whose grad_input scatter is bit-reproducible).  ``install()`` registers this module as
``sys.modules['DCN']`` so the reference's unmodified ``modulated_deform_conv_func.py`` / ``nlspn_model.py`` import it.
"""
import sys

import torch

from .. import _cabi as C


def _shape(input, weight, kh, kw, sh, sw, ph, pw, dh, dw, group, deformable_group, im2col_step):
    # deformconv/src/cuda/modulated_deform_conv_cuda.cu:39-73
    if not input.is_contiguous():
        raise RuntimeError("input tensor has to be contiguous")
    if not weight.is_contiguous():
        raise RuntimeError("weight tensor has to be contiguous")
    if input.dim() != 4 or weight.dim() != 4:
        raise RuntimeError("input and weight must be 4-D")
    B, Cin, H, W = input.shape
    if weight.shape[2] != kh or weight.shape[3] != kw:
        raise RuntimeError("Input shape and kernel shape wont match: (%d x %d vs %d x %d)." %
                           (weight.shape[2], weight.shape[3], kh, kw))
    if Cin != weight.shape[1] * group:
        raise RuntimeError("Input shape and kernel channels wont match: (%d vs %d)." % (Cin, weight.shape[1] * group))
    return C.DcnShape(B, Cin, H, W, weight.shape[0], kh, kw, sh, sw, ph, pw, dh, dw, group, deformable_group,
                      im2col_step)


def _out_hw(s):
    ho, wo = C.c_int(), C.c_int()
    C.check(C.lib.rdfc_dcn_out_size(s, ho, wo))
    return ho.value, wo.value


def _check_aux(s, offset, mask, Ho, Wo):
    K = s.kh * s.kw
    if tuple(offset.shape) != (s.B, s.deformable_group * 2 * K, Ho, Wo):
        raise RuntimeError("offset shape %s does not match (%d, %d, %d, %d)" %
                           (tuple(offset.shape), s.B, s.deformable_group * 2 * K, Ho, Wo))
    if mask is not None and tuple(mask.shape) != (s.B, s.deformable_group * K, Ho, Wo):
        raise RuntimeError("mask shape %s does not match (%d, %d, %d, %d)" %
                           (tuple(mask.shape), s.B, s.deformable_group * K, Ho, Wo))


def _forward(input, weight, bias, offset, mask, *geo):
    C.require_cuda(input, weight, bias, offset, mask)
    s = _shape(input, weight, *geo)
    Ho, Wo = _out_hw(s)
    # the reference indexes offset/mask as if contiguous (SURVEY.md 8a quirk 5); make that true instead of mis-reading
    offset = offset.contiguous()
    mask = None if mask is None else mask.contiguous()
    _check_aux(s, offset, mask, Ho, Wo)
    dt = C.dtype_code(input)
    for t in (weight, bias, offset, mask):
        if t is not None and t.dtype != input.dtype:
            raise RuntimeError("all tensors must share the input's dtype")
    out = torch.empty((s.B, s.Cout, Ho, Wo), dtype=input.dtype, device=input.device)
    with torch.cuda.device(input.device):
        C.check(C.lib.rdfc_dcn_forward(C.ptr(input), C.ptr(weight), C.ptr(bias.contiguous()), C.ptr(offset), C.ptr(mask),
                                       C.ptr(out), s, dt, C.stream_ptr(input.device)))
    return out


def _backward(input, weight, bias, offset, mask, grad_output, *geo):
    C.require_cuda(input, weight, bias, offset, mask, grad_output)
    s = _shape(input, weight, *geo)
    Ho, Wo = _out_hw(s)
    offset = offset.contiguous()
    mask = None if mask is None else mask.contiguous()
    _check_aux(s, offset, mask, Ho, Wo)
    grad_output = grad_output.contiguous()
    if tuple(grad_output.shape) != (s.B, s.Cout, Ho, Wo):   # modulated_deform_conv_cuda.cu:183-190
        raise RuntimeError("grad_output shape %s does not match the output" % (tuple(grad_output.shape),))
    grad_input = torch.empty_like(input)
    grad_offset = torch.empty_like(offset)
    grad_mask = None if mask is None else torch.empty_like(mask)
    grad_weight = torch.empty_like(weight)
    grad_bias = torch.empty_like(bias)
    with torch.cuda.device(input.device):
        C.backward_call("rdfc_dcn_backward", C.ptr(input), C.ptr(weight), C.ptr(offset), C.ptr(mask), C.ptr(grad_output),
                        C.ptr(grad_input), C.ptr(grad_offset), C.ptr(grad_mask), C.ptr(grad_weight),
                        C.ptr(grad_bias), s, C.dtype_code(input), C.stream_ptr(input.device))
    return grad_input, grad_offset, grad_mask, grad_weight, grad_bias


def modulated_deform_conv_forward(input, weight, bias, offset, mask, kernel_h, kernel_w, stride_h, stride_w, pad_h,
                                  pad_w, dilation_h, dilation_w, group, deformable_group, im2col_step):
    """deformconv/src/modulated_deform_conv.h:10-44"""
    return _forward(input, weight, bias, offset, mask, kernel_h, kernel_w, stride_h, stride_w, pad_h, pad_w,
                    dilation_h, dilation_w, group, deformable_group, im2col_step)


def modulated_deform_conv_backward(input, weight, bias, offset, mask, grad_output, kernel_h, kernel_w, stride_h,
                                   stride_w, pad_h, pad_w, dilation_h, dilation_w, group, deformable_group,
                                   im2col_step):
    """deformconv/src/modulated_deform_conv.h:46-86 -> [grad_input, grad_offset, grad_mask, grad_weight, grad_bias]"""
    return list(_backward(input, weight, bias, offset, mask, grad_output, kernel_h, kernel_w, stride_h, stride_w,
                          pad_h, pad_w, dilation_h, dilation_w, group, deformable_group, im2col_step))


def deform_conv_forward(input, weight, bias, offset, kernel_h, kernel_w, stride_h, stride_w, pad_h, pad_w,
                        dilation_h, dilation_w, group, deformable_group, im2col_step):
    """deformconv/src/deform_conv.h (DCN v1 = modulated with mask == 1)"""
    return _forward(input, weight, bias, offset, None, kernel_h, kernel_w, stride_h, stride_w, pad_h, pad_w,
                    dilation_h, dilation_w, group, deformable_group, im2col_step)


def deform_conv_backward(input, weight, bias, offset, grad_output, kernel_h, kernel_w, stride_h, stride_w, pad_h,
                         pad_w, dilation_h, dilation_w, group, deformable_group, im2col_step):
    """-> [grad_input, grad_offset, grad_weight, grad_bias]"""
    gi, go, _, gw, gb = _backward(input, weight, bias, offset, None, grad_output, kernel_h, kernel_w, stride_h,
                                  stride_w, pad_h, pad_w, dilation_h, dilation_w, group, deformable_group, im2col_step)
    return [gi, go, gw, gb]


def deform_psroi_pooling_forward(*args, **kwargs):
    """Out of scope (SURVEY.md 2.1 row 1: never called by any generator); present so the module surface matches."""
    raise RuntimeError("deform_psroi_pooling_forward is not part of the generator hot path and is not implemented")


def deform_psroi_pooling_backward(*args, **kwargs):
    raise RuntimeError("deform_psroi_pooling_backward is not part of the generator hot path and is not implemented")


def install():
    """Make ``import DCN`` resolve to this module (what nlspn/modulated_deform_conv_func.py:13 does)."""
    sys.modules["DCN"] = sys.modules[__name__]
    return sys.modules[__name__]
