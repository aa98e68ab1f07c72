"""Differentiable building blocks of the TRAINING step on the sm_100a kernels (SURVEY 8f rank 1).

What the reference gets from autograd + cuDNN inside ``conv_bn_relu`` / ``convt_bn_relu`` / torchvision ``BasicBlock`` in
train() mode (encoder_decoder/common.py:29-61, encoder_decoder/encoder_decoder.py:39-59) becomes autograd Functions over
bf16 NHWC tensors (plus the reflection / replication padding of ResnetGenerator, ``pad_nhwc``):

* ``conv2d_nhwc``   forward = ``rdfc_conv_forward`` (tcgen05 implicit GEMM); data gradient = the same kernel in one of the conv
                    forms, with a transformed filter (_Conv2dNHWC.backward); filter gradient = ``rdfc_conv_wgrad``.
* ``bn_act``        BatchNorm2d with BATCH statistics (+ running-stat update) fused with the residual add and the
                    (Leaky)ReLU: ``rdfc_bn_stats`` + ``rdfc_affine_act_forward``; backward = ``rdfc_bn_act_backward``.  For a
                    BatchNorm in train() mode; nn.BatchNorm2d decides per module (``bn_frozen``).
* ``conv_bn_act_frozen``  conv + a FROZEN BatchNorm2d (eval() mode: running statistics, no update) + residual + activation in
                    one tcgen05 launch (the BatchNorm folded into the epilogue's per-channel scale / shift); backward =
                    ``rdfc_bn_frozen_backward`` + the conv's data / filter gradients, without the pre-BatchNorm tensor.

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
import torch.nn.functional as F

from . import _cabi as C
from .engine import GeneratorEngine, pack_weight


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


def _pad32(t):
    """An NHWC tensor with its channels zero-padded to the next multiple of 32; t itself when C % 32 == 0.  The data gradient reads
    d(output) as the conv kernel's input, and that kernel (and the fp32_tc split) takes Cin % 32 == 0 only, while the forward
    accepts any Cout % 8 == 0."""
    n = -t.shape[3] % 32
    return F.pad(t, (0, n)) if n else t


def _conv(x, sx, w_oihw, k, stride, transposed, out_hw, fold=None, residual=None, act=C.ACT_NONE):
    """(x, sx) = _operand(input); w_oihw (O, I, k, k) float -> (B, Ho, Wo, O) = conv(input, w): bf16 from a bf16 input, fp32 from a
    split one (x_hi W_hi + x_hi W_lo + x_lo W_hi of the scaled operands, the inverse scales in the epilogue).  Without ``fold``: no
    bias / activation.  With ``fold`` = (s, t), fp32 (O,) device vectors: act(conv * s + t + residual) in the same launch
    (``residual``: an NHWC tensor of the output's dtype and shape, or None)."""
    B, H, W, Cx = x.shape
    Cin, O = (Cx if sx is None else Cx // 2), w_oihw.shape[0]
    if Cin % 32 or O % 8 or w_oihw.shape[1] != Cin:
        raise RuntimeError(f"tensor-core conv needs Cin % 32 == 0 and Cout % 8 == 0, got {Cin} -> {O}")
    w = w_oihw.detach().float()
    CoutP = (O + 15) // 16 * 16
    d = C.ConvDesc()
    d.B, d.Hi, d.Wi, d.Ho, d.Wo = B, H, W, out_hw[0], out_hw[1]
    d.kh = d.kw = k
    d.stride, d.pad, d.transposed, d.act = stride, (k - 1) // 2, int(transposed), act
    if sx is None:
        packed, scale = pack_weight(w, umma=True), None
        d.path, fn, dtype = C.PATH_UMMA_BF16, C.lib.rdfc_conv_forward, torch.bfloat16
    else:
        sw = _pow2_factor(w)
        packed = pack_weight(w * sw, umma=True, x3=True)                   # [W_hi ; W_lo ; W_hi] of the scaled filter
        scale = (1.0 / (sx * sw)).expand(CoutP).contiguous()               # exact: powers of two
        d.path, fn, dtype = C.PATH_UMMA_F32X3, C.lib.rdfc_conv_forward_split, torch.float32
    shift = None
    if fold is not None:
        s, t = (F.pad(v.float(), (0, CoutP - O)) for v in fold)
        scale = s if scale is None else scale * s
        shift = t.contiguous()
    out = torch.empty((B, out_hw[0], out_hw[1], O), dtype=dtype, device=x.device)
    d.inp, d.in2, d.out, d.residual = C.view(x), C.view(None), C.view(out), C.view(residual)
    d.weight, d.scale, d.shift = packed.data_ptr(), C.ptr(scale), C.ptr(shift)
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


def _conv_form(x, weight, k, stride, transposed):
    """-> (output (Ho, Wo), the filter as (O, I, k, k)) of conv2d_nhwc's conv forms"""
    B, H, W, _ = x.shape
    if transposed:                      # ConvTranspose2d(k3, s2, p1, op1): weight (Cin, Cout, 3, 3), output exactly 2x
        return (2 * H, 2 * W), weight.detach().permute(1, 0, 2, 3)
    p = (k - 1) // 2
    return ((H + 2 * p - k) // stride + 1, (W + 2 * p - k) // stride + 1), weight.detach()


class _Conv2dNHWC(torch.autograd.Function):
    """The conv forms and their data-gradient transforms; the arithmetic follows the input's dtype (_operand).  In the fp32_tc mode the
    split input (as many bytes as the fp32 input) is kept for the filter gradient instead of the input itself."""
    @staticmethod
    def forward(ctx, x, weight, k, stride, transposed):
        C.require_cuda(x, weight)
        x = _dense(x)
        out_hw, w_oihw = _conv_form(x, weight, k, stride, transposed)
        x, sx = _operand(x)
        ctx.save_for_backward(x, sx, weight)
        ctx.cfg = (k, stride, transposed)
        return _conv(x, sx, w_oihw, k, stride, transposed, out_hw)

    @staticmethod
    def backward(ctx, gy):
        x, sx, weight = ctx.saved_tensors
        k, stride, transposed = ctx.cfg
        g, sg = _operand(_pad32(_dense(gy)))
        w = weight.detach()
        gx = gw = None
        if ctx.needs_input_grad[0]:
            gx = _conv_dgrad(g, sg, w, k, stride, transposed, x.shape[:3])
        if ctx.needs_input_grad[1]:
            gw = _conv_wgrad(g, sg, x, sx, k, stride, transposed, gy.shape[3]).to(weight.dtype)
        return gx, gw, None, None, None


def _conv_dgrad(g, sg, w, k, stride, transposed, in_bhw):
    """(g, sg) = _operand(_pad32(d(output))); w: the layer's weight (as conv2d_nhwc takes it) -> d(input) (B, H, W, Cin) of that conv
    form.  The filter's output channels are zero-padded to g's: the padded channels add exact zeros."""
    B, H, W = in_bhw
    n = (g.shape[3] if sg is None else g.shape[3] // 2) - w.shape[1 if transposed else 0]
    if n:
        w = F.pad(w, (0, 0, 0, 0, 0, n) if transposed else (0, 0, 0, 0, 0, 0, 0, n))
    if transposed:                  # dgrad of the transposed conv = the stride-2 conv with the SAME filter (O = Cin, I = Cout)
        return _conv(g, sg, w, 3, 2, False, (H, W))
    if k == 3 and stride == 1:      # flipped filter, (Cout, Cin) swapped
        return _conv(g, sg, w.flip(2, 3).permute(1, 0, 2, 3), 3, 1, False, (H, W))
    if k == 3:                      # stride 2: the transposed conv with the same filter, cropped to the input size
        return _conv(g, sg, w.permute(1, 0, 2, 3), 3, 2, True, (H, W))
    t = _conv(g, sg, w.permute(1, 0, 2, 3), 1, 1, False, tuple(g.shape[1:3]))     # 1x1: W^T per pixel
    if stride == 1:
        return t
    gx = t.new_zeros((B, H, W, t.shape[3]))                                       # stride 2 scatters onto the even grid
    gx[:, ::2, ::2] = t
    return gx


def _conv_wgrad(g, sg, x, sx, k, stride, transposed, cout):
    """The unscaled filter gradient in the layer's weight layout, fp32: (Cout, Cin, k, k), or (Cin, Cout, 3, 3) for the transposed conv
    (the filters of the zero channels _pad32 added to g dropped)."""
    if transposed:                  # roles exchanged: "gradient" = the layer's input, "input" = d(output), stride-2 form
        return _wgrad(x, g, 3, 2, sx, sg)[:, :cout].contiguous()
    return _wgrad(g, x, k, stride, sg, sx)[:cout]


def conv2d_nhwc(x, weight, k=3, stride=1, transposed=False):
    """NHWC convolution (3x3 / 1x1, stride 1 / 2, padding (k-1)/2) or ConvTranspose2d(k3, s2, p1, op1) without bias.
    bf16 ``x``: bf16 operands and result; fp32 ``x``: the fp32_tc split-operand arithmetic, fp32 result.  Cin % 32 == 0 and
    Cout % 8 == 0, in the forward and the backward alike."""
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
    running statistics (updated in place, as nn.BatchNorm2d.forward does in train mode).  Always BATCH statistics, whatever
    ``bn.training`` says: the generators send a frozen BatchNorm (``bn_frozen``) to ``conv_bn_act_frozen`` instead."""
    return _BNAct.apply(y, bn.weight, bn.bias, residual, act, bn.eps, bn)


def bn_frozen(bn):
    """nn.BatchNorm2d's own rule: a BatchNorm in eval() mode that has running statistics normalises with them and updates nothing,
    whatever mode its parent is in (the usual way to freeze BatchNorm while fine-tuning at a small batch)."""
    return not bn.training and bn.running_mean is not None and bn.running_var is not None


class _ConvBNActFrozen(torch.autograd.Function):
    """out = act(s * conv(x, W) + t + residual) with the frozen BatchNorm's s = gamma rsqrt(rv + eps), t = beta - rm s (fp32, on the
    device) in the conv's epilogue.  Saved: the conv's input operand (bf16 input or fp32_tc split), W, s, rstd, rm and -- with an
    activation -- the output; not the pre-BatchNorm tensor.  Backward, with dz = dout act'(out) and G = the unscaled filter gradient
    of dz: d beta = sum dz, d gamma = rstd (<W_c, G_c> - rm_c sum dz_c) (sum_p dz y = <W, G>: y is linear in W), dW = s_c G_c,
    dx = the conv's data gradient of the filter W s applied to dz, d residual = dz."""
    @staticmethod
    def forward(ctx, x, weight, gamma, beta, residual, k, stride, transposed, act, bn):
        C.require_cuda(x, weight, residual)
        x = _dense(x)
        out_hw, w_oihw = _conv_form(x, weight, k, stride, transposed)
        rm = bn.running_mean.detach().float()
        rstd = torch.rsqrt(bn.running_var.detach().float() + bn.eps)
        s, t = GeneratorEngine._bn_fold(bn) if gamma is not None else (rstd, -rm * rstd)
        res = None
        if residual is not None:
            res = _dense(residual)
            want = (x.shape[0], out_hw[0], out_hw[1], w_oihw.shape[0])
            if res.dtype != x.dtype or tuple(res.shape) != want:
                raise RuntimeError(f"conv_bn_act_frozen: residual must be {x.dtype} of shape {want}, got {res.dtype} {tuple(res.shape)}")
        xo, sx = _operand(x)
        out = _conv(xo, sx, w_oihw, k, stride, transposed, out_hw, (s, t), res, act)
        ctx.save_for_backward(xo, sx, weight, out if act != C.ACT_NONE else None, s, rstd, rm)
        ctx.cfg = (k, stride, transposed, act, None if gamma is None else gamma.dtype)
        return out

    @staticmethod
    def backward(ctx, gout):
        xo, sx, weight, out, s, rstd, rm = ctx.saved_tensors
        k, stride, transposed, act, pdt = ctx.cfg
        need_x, need_w, need_g, need_b, need_r = ctx.needs_input_grad[:5]
        gout = _dense(gout)
        B, H, W, Cc = gout.shape
        npix, dev = B * H * W, gout.device
        dz = gout if act == C.ACT_NONE else torch.empty(gout.shape, dtype=gout.dtype, device=dev)
        ws = torch.empty(C.lib.rdfc_bn_workspace_floats(npix, Cc), dtype=torch.float32, device=dev)
        sum_dz = torch.empty(Cc, device=dev)
        vg, vo, vz = C.view(gout), C.view(out), C.view(dz)
        with torch.cuda.device(dev):
            C.check(C.lib.rdfc_bn_frozen_backward(ctypes.byref(vg), ctypes.byref(vo) if out is not None else None, act,
                                                  ctypes.byref(vz) if act != C.ACT_NONE else None, C.ptr(ws), C.ptr(sum_dz), npix,
                                                  C.stream_ptr(dev)))
        w = weight.detach()
        bshape = (1, -1, 1, 1) if transposed else (-1, 1, 1, 1)          # the BatchNorm channel: dim 1 of a ConvTranspose2d weight
        gx = gw = gg = gb = None
        if need_x or need_w or need_g:
            g, sg = _operand(_pad32(dz))
        if need_w or need_g:
            G = _conv_wgrad(g, sg, xo, sx, k, stride, transposed, Cc)
            if need_w:
                gw = (G * s.view(bshape)).to(weight.dtype)
            if need_g:                      # the filter the forward multiplied: bf16-rounded in the bf16 mode
                wq = w.float() if sx is not None else w.to(torch.bfloat16).float()
                gg = (rstd * ((wq * G).sum((0, 2, 3) if transposed else (1, 2, 3)) - rm * sum_dz)).to(pdt)
        if need_x:
            gx = _conv_dgrad(g, sg, w.float() * s.view(bshape), k, stride, transposed, xo.shape[:3])
        if need_b:
            gb = sum_dz.to(pdt)
        return gx, gw, gg, gb, (dz if need_r else None), None, None, None, None, None


def conv_bn_act_frozen(x, weight, bn, k=3, stride=1, transposed=False, residual=None, act=C.ACT_NONE):
    """act(BatchNorm2d_eval(conv(x, weight)) + residual): conv2d_nhwc's conv forms and precision (bf16 ``x``: bf16; fp32 ``x``: the
    fp32_tc split-operand arithmetic) followed by the frozen BatchNorm ``bn`` -- its running statistics, which stay untouched --
    the residual add and none / ReLU / LeakyReLU(0.2), in one tcgen05 launch.  gamma / beta may train (or not, requires_grad=False);
    gradients follow the usual autograd rules for x, weight, gamma, beta and the residual.  Cin % 32 == 0 and Cout % 8 == 0, in the
    forward and the backward alike."""
    if not (bn.running_mean is not None and bn.running_var is not None):
        raise RuntimeError("conv_bn_act_frozen needs a BatchNorm2d with running statistics")
    if act not in (C.ACT_NONE, C.ACT_RELU, C.ACT_LEAKY02):
        raise ValueError(f"conv_bn_act_frozen: activation none / ReLU / LeakyReLU(0.2), got {act}")
    return _ConvBNActFrozen.apply(x, weight, bn.weight, bn.bias, residual, k, stride, transposed, act, bn)


_PAD_MODES = {'reflect': C.PAD_REFLECT, 'replicate': C.PAD_REPLICATE}


class _PadNHWC(torch.autograd.Function):
    """Forward = ``rdfc_pad_nhwc_forward`` (a copy); backward = ``rdfc_pad_nhwc_backward``, a gather in a fixed order (no atomics):
    reproducible under torch.use_deterministic_algorithms, where PyTorch's own CUDA backward of these pads raises."""
    @staticmethod
    def forward(ctx, x, pad, mode):
        C.require_cuda(x)
        x = _dense(x)
        B, H, W, Cc = x.shape
        out = torch.empty((B, H + 2 * pad, W + 2 * pad, Cc), dtype=x.dtype, device=x.device)
        vx, vo = C.view(x), C.view(out)
        with torch.cuda.device(x.device):
            C.check(C.lib.rdfc_pad_nhwc_forward(ctypes.byref(vx), B, H, W, pad, mode, ctypes.byref(vo), C.stream_ptr(x.device)))
        ctx.cfg = (B, H, W, pad, mode)
        return out

    @staticmethod
    def backward(ctx, gy):
        B, H, W, pad, mode = ctx.cfg
        g = _dense(gy)
        gx = torch.empty((B, H, W, g.shape[3]), dtype=g.dtype, device=g.device)
        vg, vx = C.view(g), C.view(gx)
        with torch.cuda.device(g.device):
            C.check(C.lib.rdfc_pad_nhwc_backward(ctypes.byref(vg), B, H, W, pad, mode, ctypes.byref(vx), C.stream_ptr(g.device)))
        return gx, None, None


def pad_nhwc(x, pad, mode):
    """F.pad(x, (p,) * 4, mode) over a bf16 or fp32 NHWC tensor (B, H, W, C) -> (B, H + 2p, W + 2p, C).  ``pad``: p, or the 4-tuple
    (left, right, top, bottom) of nn.ReflectionPad2d / nn.ReplicationPad2d.padding, all four equal; ``mode``: 'reflect' or
    'replicate'.  The forward is a copy (bit for bit F.pad); the backward is a deterministic gather."""
    if mode not in _PAD_MODES:
        raise ValueError(f"pad mode must be 'reflect' or 'replicate', got {mode!r}")
    p = (pad,) * 4 if isinstance(pad, int) else tuple(pad)
    if len(p) != 4 or len(set(p)) != 1:
        raise RuntimeError(f"pad_nhwc pads all four sides alike, got padding {pad}")
    if x.dtype not in (torch.bfloat16, torch.float32):
        raise RuntimeError(f"pad_nhwc takes bf16 or fp32 tensors, not {x.dtype}")
    return _PadNHWC.apply(x, int(p[0]), _PAD_MODES[mode])
