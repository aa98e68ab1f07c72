"""Differentiable building blocks of the TRAINING step on the sm_100a kernels (SURVEY 8f rank 1).

What the reference gets from autograd + cuDNN inside ``conv_bn_relu`` / ``convt_bn_relu`` / torchvision ``BasicBlock`` in
train() mode (encoder_decoder/common.py:29-61, encoder_decoder/encoder_decoder.py:39-59) becomes two autograd Functions over
bf16 NHWC tensors:

* ``conv2d_nhwc``   forward = ``rdfc_conv_forward`` (tcgen05 implicit GEMM); data gradient = the same kernel in one of the conv
                    forms, with a transformed filter (_Conv2dNHWC.backward); filter gradient = ``rdfc_conv_wgrad``.
* ``bn_act``        BatchNorm2d with BATCH statistics (+ running-stat update) fused with the residual add and the
                    (Leaky)ReLU: ``rdfc_bn_stats`` + ``rdfc_affine_act_forward``; backward = ``rdfc_bn_act_backward``.

Both dispatch on the activation dtype.  bf16 is the default training mode.  fp32 tensors select the ``fp32_tc`` mode: the same
conv forms, every contraction (forward, data gradient, filter gradient) on the tensor cores with split fp16 operands
x = x_hi + x_lo (``x_hi W_hi + x_hi W_lo + x_lo W_hi``), each operand first scaled by a power of two taken from its own largest
magnitude (``rdfc_split_scaled``; the factors stay on the device) and the exact inverse multiplied back in the epilogue / the
filter gradient's reduction; the BatchNorm kernels read and write fp32.

Everything else of the training forward (the 3 / 1-channel stems, the <= 8-channel ``*_dec0`` heads, the W-AdaIN modulation,
losses) is plain differentiable PyTorch on the same tensors -- < 1 % of the FLOPs (DESIGN.md section 7 lists what is not on
the repo's kernels yet).
"""
import ctypes

import torch

from . import _cabi as C
from .engine import pack_weight


def _dense(t):
    """The tensor itself when the kernels can read it as a (pointer, channels, pixel stride) view -- dense NHWC or a channel slice of a
    dense NHWC tensor, which is what autograd returns for the operands of a channel concatenation -- else a contiguous copy."""
    return t if C.nhwc_viewable(t) else t.contiguous()


def _pow2_factor(t):
    """The power of two s with max|t| * s in [1024, 2048) (1 for an all-zero or non-finite tensor), as rdfc_split_scaled chooses
    it, computed on the device: a 1-element fp32 tensor."""
    amax = t.detach().abs().amax().float().reshape(1)
    _, e = torch.frexp(amax)
    s = torch.exp2((11 - e).clamp(-100, 100).float())
    return torch.where((amax > 0) & torch.isfinite(amax), s, torch.ones_like(s))


def _split(t):
    """fp32 NHWC tensor (or channel slice) -> (fp16 (B, H, W, 2C) = [hi | lo] of s * t, s as a 1-element device tensor)."""
    B, H, W, Cc = t.shape
    xs = torch.empty((B, H, W, 2 * Cc), dtype=torch.float16, device=t.device)
    s = torch.empty(1, dtype=torch.float32, device=t.device)
    vx, vo = C.view(t), C.view(xs)
    with torch.cuda.device(t.device):
        C.check(C.lib.rdfc_split_scaled(ctypes.byref(vx), B * H * W, ctypes.byref(vo), C.ptr(s), C.stream_ptr(t.device)))
    return xs, s


def _operand(t):
    """An activation as the contractions read it: (t, None) for bf16; for fp32 (the fp32_tc mode) its split and factor, _split(t)."""
    return _split(t) if t.dtype == torch.float32 else (t, None)


def _conv(x, sx, w_oihw, k, stride, transposed, out_hw):
    """(x, sx) = _operand(input); w_oihw (O, I, k, k) float -> (B, Ho, Wo, O) = conv(input, w), no bias / activation: bf16 from a bf16
    input, fp32 from a split one (x_hi W_hi + x_hi W_lo + x_lo W_hi of the scaled operands, the inverse scales in the epilogue)."""
    B, H, W, Cx = x.shape
    Cin, O = (Cx if sx is None else Cx // 2), w_oihw.shape[0]
    if Cin % 32 or O % 8 or w_oihw.shape[1] != Cin:
        raise RuntimeError(f"tensor-core conv needs Cin % 32 == 0 and Cout % 8 == 0, got {Cin} -> {O}")
    w = w_oihw.detach().float()
    d = C.ConvDesc()
    d.B, d.Hi, d.Wi, d.Ho, d.Wo = B, H, W, out_hw[0], out_hw[1]
    d.kh = d.kw = k
    d.stride, d.pad, d.transposed, d.act = stride, (k - 1) // 2, int(transposed), C.ACT_NONE
    if sx is None:
        packed, inv = pack_weight(w, umma=True), None
        d.path, fn, dtype = C.PATH_UMMA_BF16, C.lib.rdfc_conv_forward, torch.bfloat16
    else:
        sw = _pow2_factor(w)
        packed = pack_weight(w * sw, umma=True, x3=True)                   # [W_hi ; W_lo ; W_hi] of the scaled filter
        inv = (1.0 / (sx * sw)).expand((O + 15) // 16 * 16).contiguous()   # exact: powers of two
        d.path, fn, dtype = C.PATH_UMMA_F32X3, C.lib.rdfc_conv_forward_split, torch.float32
    out = torch.empty((B, out_hw[0], out_hw[1], O), dtype=dtype, device=x.device)
    d.inp, d.in2, d.out, d.residual = C.view(x), C.view(None), C.view(out), C.view(None)
    d.weight, d.scale, d.shift = packed.data_ptr(), None if inv is None else inv.data_ptr(), None
    with torch.cuda.device(x.device):
        C.check(fn(ctypes.byref(d), C.stream_ptr(x.device)))
    return out


def _wgrad(grad_out, inp, k, stride, sg=None, sx=None):
    """sum_p grad_out[p, o] * inp[stride * p - pad + tap, i] -> (O, I, k, k) fp32.  bf16 operands, or split ones with their factors
    ((grad_out, sg), (inp, sx) from _split: the three products reduced once, the inverse scales applied there)."""
    B, Hg, Wg, O = grad_out.shape
    _, Hi, Wi, I = inp.shape
    if sx is not None:
        O, I = O // 2, I // 2
    d = C.WgradDesc()
    d.B, d.Hg, d.Wg, d.Hi, d.Wi, d.k, d.stride, d.pad = B, Hg, Wg, Hi, Wi, k, stride, (k - 1) // 2
    d.grad_out, d.input = C.view(grad_out), C.view(inp)
    n = (C.lib.rdfc_conv_wgrad_workspace_floats if sx is None else C.lib.rdfc_conv_wgrad_split_workspace_floats)(ctypes.byref(d))
    if n < 0:
        raise RuntimeError(C.lib.rdfc_last_error().decode("utf-8", "replace"))
    ws = torch.empty(n, dtype=torch.float32, device=inp.device)
    gw = torch.empty((O, I, k, k), dtype=torch.float32, device=inp.device)
    with torch.cuda.device(inp.device):
        if sx is None:
            C.check(C.lib.rdfc_conv_wgrad(ctypes.byref(d), C.ptr(gw), C.ptr(ws), C.stream_ptr(inp.device)))
        else:
            inv = 1.0 / (sg * sx)
            C.check(C.lib.rdfc_conv_wgrad_split(ctypes.byref(d), C.ptr(inv), C.ptr(gw), C.ptr(ws), C.stream_ptr(inp.device)))
    return gw


class _Conv2dNHWC(torch.autograd.Function):
    """The conv forms and their data-gradient transforms; the arithmetic follows the input's dtype (_operand).  In the fp32_tc mode the
    split input (as many bytes as the fp32 input) is kept for the filter gradient instead of the input itself."""
    @staticmethod
    def forward(ctx, x, weight, k, stride, transposed):
        C.require_cuda(x, weight)
        x = _dense(x)
        B, H, W, _ = x.shape
        if transposed:                      # ConvTranspose2d(k3, s2, p1, op1): weight (Cin, Cout, 3, 3), output exactly 2x
            out_hw = (2 * H, 2 * W)
            w_oihw = weight.detach().permute(1, 0, 2, 3)
        else:
            p = (k - 1) // 2
            out_hw = ((H + 2 * p - k) // stride + 1, (W + 2 * p - k) // stride + 1)
            w_oihw = weight.detach()
        x, sx = _operand(x)
        ctx.save_for_backward(x, sx, weight)
        ctx.cfg = (k, stride, transposed)
        return _conv(x, sx, w_oihw, k, stride, transposed, out_hw)

    @staticmethod
    def backward(ctx, gy):
        x, sx, weight = ctx.saved_tensors
        k, stride, transposed = ctx.cfg
        g, sg = _operand(_dense(gy))
        B, H, W = x.shape[:3]
        w = weight.detach()
        gx = gw = None
        if ctx.needs_input_grad[0]:
            if transposed:                  # dgrad of the transposed conv = the stride-2 conv with the SAME filter (O = Cin, I = Cout)
                gx = _conv(g, sg, w, 3, 2, False, (H, W))
            elif k == 3 and stride == 1:    # flipped filter, (Cout, Cin) swapped
                gx = _conv(g, sg, w.flip(2, 3).permute(1, 0, 2, 3), 3, 1, False, (H, W))
            elif k == 3:                    # stride 2: the transposed conv with the same filter, cropped to the input size
                gx = _conv(g, sg, w.permute(1, 0, 2, 3), 3, 2, True, (H, W))
            else:                           # 1x1: W^T per pixel; stride 2 scatters onto the even grid
                t = _conv(g, sg, w.permute(1, 0, 2, 3), 1, 1, False, tuple(gy.shape[1:3]))
                if stride == 1:
                    gx = t
                else:
                    gx = t.new_zeros((B, H, W, t.shape[3]))
                    gx[:, ::2, ::2] = t
        if ctx.needs_input_grad[1]:
            if transposed:                  # roles exchanged: "gradient" = the layer's input, "input" = d(output), stride-2 form
                gw = _wgrad(x, g, 3, 2, sx, sg)                # (Cin, Cout, 3, 3) = ConvTranspose2d's weight layout
            else:
                gw = _wgrad(g, x, k, stride, sg, sx)           # (Cout, Cin, k, k)
            gw = gw.to(weight.dtype)
        return gx, gw, None, None, None


def conv2d_nhwc(x, weight, k=3, stride=1, transposed=False):
    """NHWC convolution (3x3 / 1x1, stride 1 / 2, padding (k-1)/2) or ConvTranspose2d(k3, s2, p1, op1) without bias.
    bf16 ``x``: bf16 operands and result; fp32 ``x``: the fp32_tc split-operand arithmetic, fp32 result."""
    return _Conv2dNHWC.apply(x, weight, k, stride, transposed)


class _BNAct(torch.autograd.Function):
    @staticmethod
    def forward(ctx, y, gamma, beta, residual, act, eps, bn):
        y = _dense(y)
        B, H, W, Cc = y.shape
        npix = B * H * W
        dev = y.device
        ws = torch.empty(C.lib.rdfc_bn_workspace_floats(npix, Cc), dtype=torch.float32, device=dev)
        mean, var = torch.empty(Cc, device=dev), torch.empty(Cc, device=dev)
        vy = C.view(y)
        with torch.cuda.device(dev):
            C.check(C.lib.rdfc_bn_stats(ctypes.byref(vy), npix, C.ptr(ws), C.ptr(mean), C.ptr(var), C.stream_ptr(dev)))
        rstd = torch.rsqrt(var + eps)
        scale = (gamma.detach().float() * rstd).contiguous()
        shift = (beta.detach().float() - mean * scale).contiguous()
        out = torch.empty(y.shape, dtype=y.dtype, device=y.device)
        res = _dense(residual) if residual is not None else None
        vo, vr = C.view(out), C.view(res)
        with torch.cuda.device(dev):
            C.check(C.lib.rdfc_affine_act_forward(ctypes.byref(vy), C.ptr(scale), C.ptr(shift), ctypes.byref(vr) if res is not None else None,
                                                  act, ctypes.byref(vo), npix, C.stream_ptr(dev)))
        if bn is not None and bn.track_running_stats and bn.running_mean is not None:
            with torch.no_grad():               # nn.BatchNorm2d: momentum 0.1, UNBIASED variance in the running estimate
                m = bn.momentum if bn.momentum is not None else 0.1
                bn.running_mean.mul_(1 - m).add_(mean, alpha=m)
                bn.running_var.mul_(1 - m).add_(var * (npix / max(npix - 1, 1)), alpha=m)
                bn.num_batches_tracked += 1
        ctx.save_for_backward(y, out, mean, rstd, gamma)
        ctx.cfg = (act, residual is not None)
        return out

    @staticmethod
    def backward(ctx, gout):
        y, out, mean, rstd, gamma = ctx.saved_tensors
        act, has_res = ctx.cfg
        gout = _dense(gout)
        B, H, W, Cc = y.shape
        npix = B * H * W
        dev = y.device
        dy = torch.empty(y.shape, dtype=y.dtype, device=y.device)
        dres = torch.empty(y.shape, dtype=y.dtype, device=y.device) if (has_res and ctx.needs_input_grad[3]) else None
        ws = torch.empty(C.lib.rdfc_bn_workspace_floats(npix, Cc), dtype=torch.float32, device=dev)
        s_dz, s_dzx = torch.empty(Cc, device=dev), torch.empty(Cc, device=dev)
        g32 = gamma.detach().float().contiguous()
        vg, vo, vy, vdy, vdr = C.view(gout), C.view(out), C.view(y), C.view(dy), C.view(dres)
        with torch.cuda.device(dev):
            C.check(C.lib.rdfc_bn_act_backward(ctypes.byref(vg), ctypes.byref(vo), ctypes.byref(vy), C.ptr(mean), C.ptr(rstd), C.ptr(g32), act,
                                               ctypes.byref(vdy), ctypes.byref(vdr) if dres is not None else None, C.ptr(ws), C.ptr(s_dz),
                                               C.ptr(s_dzx), npix, C.stream_ptr(dev)))
        return dy, s_dzx.to(gamma.dtype), s_dz.to(gamma.dtype), dres, None, None, None


def bn_act(y, bn, residual=None, act=C.ACT_NONE):
    """act(BatchNorm2d_train(y) + residual) over a bf16 or fp32 NHWC tensor (residual of the same dtype); ``bn`` is the nn.BatchNorm2d holding weight / bias and the
    running statistics (updated in place, as nn.BatchNorm2d.forward does in train mode)."""
    return _BNAct.apply(y, bn.weight, bn.bias, residual, act, bn.eps, bn)
