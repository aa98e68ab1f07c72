"""Input gradients of the generator's conv layers on the tcgen05 conv kernel (SURVEY 8f rank 1, first conv piece).

No new kernel: the data gradient of a conv is itself one of the three forms `rdfc_conv_forward` runs,

* 3x3 stride-1 pad-1 conv        -> 3x3 stride-1 conv of grad_out with the filter flipped and (Cout, Cin) swapped,
* 3x3 stride-2 pad-1 conv        -> the k3 s2 p1 transposed conv of grad_out with the SAME filter, cropped to the input size
                                    (an odd input size is the output_padding = 0 case),
* k3 s2 p1 op1 transposed conv   -> the 3x3 stride-2 pad-1 conv of grad_out with the SAME filter,

so dgrad runs at the forward kernel's speed.  bf16 NHWC activations, fp32 accumulation.  The filter gradient (an MN-major
GEMM with K = pixels) is not built yet.  Replaces what autograd does for `nn.Conv2d` / `nn.ConvTranspose2d` inside
`ResNetEncoderDecoder` (encoder_decoder/resnet_encoder_decoder.py) -- cuDNN's dgrad in the reference.
"""
import ctypes

import torch

from . import _cabi as C
from .engine import pack_weight


def pack_filter(w_oihw):
    """(Cout, Cin, kh, kw) -> the UMMA filter layout [tap][Cin/8][CoutP][8] bf16 (engine.pack_weight's layout)."""
    Cin = w_oihw.shape[1]
    if Cin % 32:
        raise RuntimeError(f"tensor-core conv needs Cin % 32 == 0, got {Cin}")
    return pack_weight(w_oihw.detach().float(), umma=True)


def _run(x, packed, Cout, stride, transposed, out_hw):
    C.require_cuda(x)
    B, H, W, Cin = x.shape
    x = x.contiguous()
    out = torch.empty((B, out_hw[0], out_hw[1], Cout), dtype=torch.bfloat16, device=x.device)
    scale = torch.ones(Cout, device=x.device)
    shift = torch.zeros(Cout, device=x.device)
    d = C.ConvDesc()
    d.B, d.Hi, d.Wi, d.Ho, d.Wo = B, H, W, out_hw[0], out_hw[1]
    d.kh = d.kw = 3
    d.stride, d.pad, d.transposed, d.act = stride, 1, int(transposed), C.ACT_NONE
    d.path = C.PATH_UMMA_BF16
    d.inp, d.in2, d.out, d.residual = C.view(x), C.view(None), C.view(out), C.view(None)
    d.weight, d.scale, d.shift = packed.data_ptr(), scale.data_ptr(), shift.data_ptr()
    with torch.cuda.device(x.device):
        C.check(C.lib.rdfc_conv_forward(ctypes.byref(d), C.stream_ptr(x.device)))
    return out


def conv2d_input_grad(grad_out, weight, stride, in_hw):
    """dL/dx of y = conv2d(x, weight (Cout, Cin, 3, 3), stride in {1, 2}, padding 1).
    grad_out (B, Ho, Wo, Cout) bf16 NHWC -> (B, Hi, Wi, Cin) bf16 NHWC."""
    Cout, Cin = weight.shape[:2]
    if tuple(weight.shape[2:]) != (3, 3) or stride not in (1, 2):
        raise RuntimeError("conv2d_input_grad covers the generator's 3x3 stride-1 / stride-2 convs")
    if grad_out.dtype != torch.bfloat16 or grad_out.shape[-1] != Cout:
        raise RuntimeError("grad_out must be bf16 NHWC with Cout channels")
    if stride == 1:
        w = weight.detach().flip(2, 3).permute(1, 0, 2, 3)            # (Cin, Cout, 3, 3): a conv from Cout to Cin channels
        return _run(grad_out, pack_filter(w), Cin, 1, False, tuple(in_hw))
    # stride 2: scatter form = the transposed conv; engine._pack hands ConvT filters (in, out, kh, kw) over as (out, in, kh, kw)
    return _run(grad_out, pack_filter(weight.detach().permute(1, 0, 2, 3)), Cin, 2, True, tuple(in_hw))


def conv_transpose2d_input_grad(grad_out, weight):
    """dL/dx of y = conv_transpose2d(x, weight (Cin, Cout, 3, 3), stride 2, padding 1, output_padding 1)[..., :Ho, :Wo].
    grad_out (B, Ho, Wo, Cout) bf16 NHWC (zero-extended by the caller if it was cropped) -> (B, ceil(Ho/2), ceil(Wo/2), Cin)."""
    Cin, Cout = weight.shape[:2]
    B, Ho, Wo, _ = grad_out.shape
    return _run(grad_out, pack_filter(weight.detach()), Cin, 2, False, ((Ho + 1) // 2, (Wo + 1) // 2))
