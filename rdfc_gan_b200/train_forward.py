"""Training-mode forward of the generator (autograd), rdf_generator.py:280-414 /
rdf_gan_generator.py:233-361, composed of the differentiable ops of train_ops.py over NHWC tensors: bf16 (the default training
mode) or fp32 (the ``fp32_tc`` mode: split-operand tensor-core arithmetic in the ops, and the PyTorch convs that stay on cuDNN --
stems, ``*_dec0`` heads -- run in true fp32, with TF32 off in their forward and backward).

The convolutions with >= 32 input channels -- every encoder / decoder / ``*_dec1`` layer and the per-pixel EqualLinear of
W-AdaIN, > 99 % of the FLOPs -- run forward, data gradient and filter gradient on this repo's kernels.  Each BatchNorm decides for
itself, as nn.BatchNorm2d does: one in train() mode (+ residual + activation) runs on the fused batch-statistics kernels and
updates its running statistics; a frozen one (eval() mode with running statistics, ``bn_frozen``) is folded with its conv,
residual and activation into one tcgen05 launch (``conv_bn_act_frozen``) and leaves its buffers alone.  The NLSPN runs its fused
forward / backward pair (nlspn.py).  The three
stems (3 / 1 input channels), the ``*_dec0`` heads (<= 8 output channels), the InstanceNorm + modulation of the fusion layers
and the output fusion are differentiable PyTorch expressions on the same tensors.
"""
import contextlib

import torch
import torch.nn.functional as F

from . import _cabi as C
from .model_utils import IN, AdaIN, AdaptiveInstanceNorm
from .train_ops import bn_act, bn_frozen, conv2d_nhwc, conv_bn_act_frozen

BF = torch.bfloat16


def _nhwc(x_nchw):
    return x_nchw.permute(0, 2, 3, 1).contiguous()


@contextlib.contextmanager
def _no_tf32():
    """cuDNN convs in true fp32 (torch lets them use TF32 by default, ~1e-3 relative); the caller's setting comes back after."""
    prev = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        yield
    finally:
        torch.backends.cudnn.allow_tf32 = prev


class _ConvFP32(torch.autograd.Function):
    """F.conv2d(x, w, b, padding) (stride 1) with TF32 off in the forward AND the backward: autograd would run the backward
    under whatever TF32 setting is current when it gets there."""
    @staticmethod
    def forward(ctx, x, w, b, padding):
        with _no_tf32():
            y = F.conv2d(x, w, b, padding=padding)
        ctx.save_for_backward(x, w)
        ctx.cfg = (padding, None if b is None else tuple(b.shape))
        return y

    @staticmethod
    def backward(ctx, gy):
        x, w = ctx.saved_tensors
        padding, bshape = ctx.cfg
        mask = [ctx.needs_input_grad[0], ctx.needs_input_grad[1], bshape is not None and ctx.needs_input_grad[2]]
        with _no_tf32():
            gx, gw, gb = torch.ops.aten.convolution_backward(gy, x, w, list(bshape) if bshape else None, [1, 1], [padding, padding], [1, 1],
                                                             False, [0, 0], 1, mask)
        return gx, gw, gb, None


def _conv(x, w, b, padding, dt):
    """the stems' and heads' cuDNN conv: as is in bf16 mode, true fp32 in fp32_tc mode"""
    if dt == torch.float32:
        return _ConvFP32.apply(x, w, b, padding)
    return F.conv2d(x, w, b, padding=padding)


def _conv_bn(x, weight, bn, k, stride, transposed=False, residual=None, act=C.ACT_NONE):
    """act(bn(conv(x)) + residual): a frozen ``bn`` folded into the conv, else the conv, then the batch-statistics BatchNorm"""
    if bn_frozen(bn):
        return conv_bn_act_frozen(x, weight, bn, k, stride, transposed, residual, act)
    return bn_act(conv2d_nhwc(x, weight, k, stride, transposed), bn, residual, act)


def _conv_bn_act(x, seq, k=3, stride=1, transposed=False, act=C.ACT_LEAKY02, residual=None):
    """conv_bn_relu / convt_bn_relu Sequential (common.py:29-61): [0] conv (no bias with BN), [1] BatchNorm2d, LeakyReLU(0.2)."""
    return _conv_bn(x, seq[0].weight, seq[1], k, stride, transposed, residual, act)


def _basic_block(x, blk):
    """torchvision BasicBlock: relu(bn2(conv2(relu(bn1(conv1(x))))) + identity)"""
    identity = x
    if blk.downsample is not None:
        identity = _conv_bn(x, blk.downsample[0].weight, blk.downsample[1], 1, blk.stride)
    out = _conv_bn(x, blk.conv1.weight, blk.bn1, 3, blk.stride, act=C.ACT_RELU)
    return _conv_bn(out, blk.conv2.weight, blk.bn2, 3, 1, residual=identity, act=C.ACT_RELU)


def _small_conv(x_nhwc, conv, act=None):
    """A conv too thin for the tensor-core kernel (<= 8 output channels): torch, on the NHWC tensor viewed as channels-last NCHW,
    in the activations' dtype.  -> fp32 NCHW"""
    dt = x_nhwc.dtype
    x = x_nhwc.permute(0, 3, 1, 2)                      # channels-last view; channels-last filters keep cuDNN from converting layouts
    w = conv.weight.to(dt).contiguous(memory_format=torch.channels_last)
    y = _conv(x, w, None if conv.bias is None else conv.bias.to(dt), 1, dt).float()
    if act == 'tanh':
        y = torch.tanh(y)
    elif act == 'sigmoid':
        y = torch.sigmoid(y)
    return y.contiguous()


def _instance_norm(x, eps=1e-5, unbiased=False):
    """per (image, channel) over the pixels of an NHWC tensor, fp32 statistics"""
    xf = x.float()
    mean = xf.mean((1, 2), keepdim=True)
    var = xf.var((1, 2), keepdim=True, unbiased=unbiased)
    return xf, mean, var


def _fuse(layer, xr, xd):
    """fuse_layer{n}(rgb feature, depth feature), model_utils.py:53-129, NHWC in / out (the inputs' dtype)"""
    dt = xr.dtype
    if isinstance(layer, AdaptiveInstanceNorm):
        lin = layer.style.linear
        Cx = xr.shape[3]
        w = lin.effective_weight().reshape(lin.out_features, lin.in_features, 1, 1)     # EqualLR: weight_orig * sqrt(2 / fan_in)
        style = conv2d_nhwc(xd, w, 1, 1).float() + lin.bias.float()
        gamma, beta = style[..., :Cx], style[..., Cx:]
        xf, mean, var = _instance_norm(xr)
        out = (xf - mean) * torch.rsqrt(var + 1e-5)
        if layer.weighting:
            gw = conv2d_nhwc(xr, layer.gamma_weight_layer.weight, 1, 1).float() + layer.gamma_weight_layer.bias.float()
            bw = conv2d_nhwc(xr, layer.beta_weight_layer.weight, 1, 1).float() + layer.beta_weight_layer.bias.float()
            out = gw * gamma * out + bw * beta
        else:
            out = gamma * out + beta
        return out.to(dt)
    if isinstance(layer, AdaIN):
        xf, cm, cv = _instance_norm(xr, unbiased=True)
        sf, sm, sv = _instance_norm(xd, unbiased=True)
        return ((xf - cm) / torch.sqrt(cv + 1e-5) * torch.sqrt(sv + 1e-5) + sm).to(dt)
    if isinstance(layer, IN):
        both = torch.cat([xr, xd], 3)
        bf, mean, var = _instance_norm(both)
        normed = ((bf - mean) * torch.rsqrt(var + 1e-5)).to(dt)
        dc = layer.down_channel
        return (conv2d_nhwc(normed, dc.weight, 1, 1).float() + dc.bias.float()).to(dt)
    raise NotImplementedError(type(layer))


def _crop_cat(fd, fe):
    """_concat (rdf_generator.py:243-258): drop the transposed conv's extra row / column, then concatenate channels"""
    return torch.cat([fd[:, :fe.shape[1], :fe.shape[2]], fe], 3)


def generator_forward_train(g, stem_in, depth, dtype=BF):
    """g: RDFGenerator / DCVGANGenerator (train mode; BatchNorms in eval() mode inside it use their running statistics).  stem_in (B, Cs, H, W), depth (B, 1, H, W) fp32 CUDA.  dtype: the activations'
    dtype, torch.bfloat16 (default) or torch.float32 (the fp32_tc training mode).
    -> (depth_map_1, confidence_map_1, depth_map_2, confidence_map_2, pred_depth), fp32 NCHW, attached to the autograd graph."""
    C.require_cuda(stem_in, depth)
    if dtype not in (torch.bfloat16, torch.float32):
        raise ValueError(f"training activations are bf16 or fp32, not {dtype}")
    L = C.ACT_LEAKY02
    # ---- stems (rdf_generator.py:286-292): 3 / 1 input channels, bias, LeakyReLU -- torch
    def stem(x, seq):                                   # fp32 conv (cuDNN's NCHW fp32 kernels), cast BEFORE the layout change (half the bytes)
        return _nhwc(F.leaky_relu(_conv(x, seq[0].weight, seq[0].bias, 1, dtype), 0.2).to(dtype))
    fe1 = {'r': stem(stem_in, g.rgb_branch_en1),
           'd': torch.cat([stem(stem_in, g.depth_branch_en1_rgb), stem(depth, g.depth_branch_en1_depth)], 3)}
    # ---- encoders
    fe = {}
    for x, ed in (('r', g.rgb_branch_encoder_decoder), ('d', g.depth_branch_encoder_decoder)):
        cur = fe1[x]
        for l in (2, 3, 4, 5):
            for blk in getattr(ed, f'en{l}'):
                cur = _basic_block(cur, blk)
            fe[(x, l)] = cur
        fe[(x, 6)] = _conv_bn_act(cur, ed.en6, 3, 2)
    # ---- decoders with RGB <- depth fusion
    xr, xd = fe[('r', 6)], fe[('d', 6)]
    for n, l in enumerate((5, 4, 3, 2), start=1):
        fz = _fuse(getattr(g, f'fuse_layer{n}'), xr, xd)
        r_up = _conv_bn_act(fz, getattr(g.rgb_branch_encoder_decoder, f'de{l}'), 3, 2, transposed=True)
        d_up = _conv_bn_act(xd, getattr(g.depth_branch_encoder_decoder, f'de{l}'), 3, 2, transposed=True)
        xr, xd = _crop_cat(r_up, fe[('r', l)]), _crop_cat(d_up, fe[('d', l)])
    # ---- decode heads
    def head(x, dec1, dec0, skip, act):
        return _small_conv(torch.cat([_conv_bn_act(x, dec1), skip], 3), dec0[0], act)
    d1 = head(xr, g.rgb_pred_dec1, g.rgb_pred_dec0, fe1['r'], 'tanh')
    c1 = head(xr, g.rgb_conf_dec1, g.rgb_conf_dec0, fe1['r'], 'sigmoid')
    pred_init = head(xd, g.id_dec1, g.id_dec0, fe1['d'], 'tanh')
    conf = head(xd, g.cf_dec1, g.cf_dec0, fe1['d'], 'sigmoid')
    if g.use_nlspn_refine:
        guide = head(xd, g.gd_dec1, g.gd_dec0, fe1['d'], None)
        d2, _ = g.nlspn_refine_module(pred_init, guide, conf, depth)
    else:
        d2 = pred_init
    d2 = torch.clamp(d2, min=-1, max=1)
    score = torch.softmax(torch.cat([c1, conf], 1), 1)
    pred = (torch.cat([d1, d2], 1) * score).sum(1, keepdim=True)
    return d1, c1, d2, conf, pred
