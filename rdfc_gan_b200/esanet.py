"""ESANet guidance network -- drop-in for RDF-GAN's ``ESANetOneModality``
(F/lib/models/segmentator/esa_net/esa_net_one_modality.py:11-194, decoder.py, model_utils.py and the ResNet of
F/lib/models/backbone/resnet/resnet.py; F = /root/reference/RDF-GAN): the ``global_guidance_module`` that turns the RGB image
into the 40-channel semantic map RDF-GAN's stems read (rdf_gan_generator.py:235).

Same constructor keywords, same module / parameter names (``state_dict`` loads into and from the reference class with
strict=True).  Inference runs on this repo's kernels through one plan per input shape and precision (buffers + a flat list of
C-ABI calls, captured in a CUDA graph), NHWC activations:

* every GEMM-shaped layer -- the ResNet BasicBlocks, the 1x1 skip / pyramid-pooling convs, the decoder's 3x3 convs, its
  factorised 3x1 / 1x3 convs (as 3x3 filters with zero taps) and conv_out -- on ``rdfc_conv_forward``, BatchNorm folded,
  bias / ReLU / residual fused in the epilogue;
* the 7x7 stride-2 stem, max pooling, squeeze-and-excitation, the pyramid pooling module's average pools / nearest up-sampling
  and the decoder's learned x2 up-sampling (+ skip add) on the small kernels of csrc/esanet.cu.

``set_precision`` selects the arithmetic, with the meanings of the generator's modes (engine.GeneratorEngine):
  'bf16'    (default) bf16 activations, the convs on the tcgen05 tensor cores (RDFC_PATH_UMMA_BF16): the throughput mode;
  'fp32'    fp32 activations, every conv on the CUDA cores in fp32 (RDFC_PATH_SIMT_F32): the parity mode;
  'fp32_tc' fp32 activations, the convs on the tensor cores with split fp16 operands (RDFC_PATH_UMMA_F32X3): each conv's input
            scaled by a power of two of its own before the split (on the device), each filter per output channel
            (engine.pack_weight_x3), so the split keeps fp32's magnitude range.

Covered configuration = the one the reference's scripts use (F/bash/test_nyuv2_Ts2T.sh:7-16): ResNet-18 / 34 BasicBlock encoder,
``weighting_in_encoder='SE-add'``, ``context_module='ppm'``, ``encoder_decoder_fusion='add'``,
``upsampling='learned-3x3-zeropad'``, no pyramid supervision; anything else raises.  eval() only (the reference's RDF-GAN runs the
guidance net frozen); CUDA only.
"""
import ctypes

import torch
import torch.nn as nn

from . import _cabi as C
from .engine import pack_weight, pack_weight_x3

_BLOCKS = {'resnet18': (2, 2, 2, 2), 'resnet34': (3, 4, 6, 3)}
_PRECISIONS = ('bf16', 'fp32', 'fp32_tc')


def _no_forward(self, *a, **k):
    raise RuntimeError(f"{type(self).__name__} is a parameter container; the forward pass runs in rdfc_gan_b200.esanet")


class ConvBNAct(nn.Sequential):
    """model_utils.py:6-18 (names conv / bn / act)"""

    def __init__(self, cin, cout, kernel_size):
        super().__init__()
        self.add_module('conv', nn.Conv2d(cin, cout, kernel_size, padding=kernel_size // 2, bias=False))
        self.add_module('bn', nn.BatchNorm2d(cout))
        self.add_module('act', nn.ReLU(inplace=True))


class BasicBlock(nn.Module):
    forward = _no_forward

    def __init__(self, inplanes, planes, stride=1):
        super().__init__()
        self.conv1 = nn.Conv2d(inplanes, planes, 3, stride, 1, bias=False)
        self.bn1 = nn.BatchNorm2d(planes)
        self.conv2 = nn.Conv2d(planes, planes, 3, 1, 1, bias=False)
        self.bn2 = nn.BatchNorm2d(planes)
        self.downsample = None
        if stride != 1 or inplanes != planes:
            self.downsample = nn.Sequential(nn.Conv2d(inplanes, planes, 1, stride, bias=False), nn.BatchNorm2d(planes))
        self.stride = stride


class NonBottleneck1D(nn.Module):
    """resnet.py:75-143 (ERFNet block): 3x1, 1x3, bn1 (eps 1e-3), 3x1, 1x3, bn2, + input, ReLU"""
    forward = _no_forward

    def __init__(self, planes):
        super().__init__()
        self.conv3x1_1 = nn.Conv2d(planes, planes, (3, 1), padding=(1, 0), bias=True)
        self.conv1x3_1 = nn.Conv2d(planes, planes, (1, 3), padding=(0, 1), bias=True)
        self.bn1 = nn.BatchNorm2d(planes, eps=1e-3)
        self.conv3x1_2 = nn.Conv2d(planes, planes, (3, 1), padding=(1, 0), bias=True)
        self.conv1x3_2 = nn.Conv2d(planes, planes, (1, 3), padding=(0, 1), bias=True)
        self.bn2 = nn.BatchNorm2d(planes, eps=1e-3)


class _ResNet(nn.Module):
    forward = _no_forward

    def __init__(self, layers, input_channels):
        super().__init__()
        self.conv1 = nn.Conv2d(input_channels, 64, kernel_size=7, stride=2, padding=3, bias=False)
        self.bn1 = nn.BatchNorm2d(64)
        inpl = 64
        for i, (planes, n) in enumerate(zip((64, 128, 256, 512), layers), start=1):
            blocks = [BasicBlock(inpl, planes, 1 if i == 1 else 2)] + [BasicBlock(planes, planes) for _ in range(1, n)]
            setattr(self, f'layer{i}', nn.Sequential(*blocks))
            inpl = planes
        self.down_4_channels_out, self.down_8_channels_out, self.down_16_channels_out, self.down_32_channels_out = 64, 128, 256, 512


class SqueezeAndExcitation(nn.Module):
    forward = _no_forward

    def __init__(self, channel, reduction=16):
        super().__init__()
        self.fc = nn.Sequential(nn.Conv2d(channel, channel // reduction, kernel_size=1), nn.ReLU(inplace=True),
                                nn.Conv2d(channel // reduction, channel, kernel_size=1), nn.Sigmoid())


class PyramidPoolingModule(nn.Module):
    forward = _no_forward

    def __init__(self, in_dim, out_dim, bins):
        super().__init__()
        red = in_dim // len(bins)
        self.bins = tuple(bins)
        self.features = nn.ModuleList([nn.Sequential(nn.AdaptiveAvgPool2d(b), ConvBNAct(in_dim, red, 1)) for b in bins])
        self.final_conv = ConvBNAct(in_dim + red * len(bins), out_dim, 1)


class Upsample(nn.Module):
    """decoder.py:137-191, mode 'learned-3x3-zeropad': nearest x2 + depth-wise 3x3 initialised to the bilinear kernel"""
    forward = _no_forward

    def __init__(self, channels):
        super().__init__()
        self.pad = nn.Identity()
        self.conv = nn.Conv2d(channels, channels, groups=channels, kernel_size=3, padding=1)
        w = torch.tensor([[[[0.0625, 0.1250, 0.0625], [0.1250, 0.2500, 0.1250], [0.0625, 0.1250, 0.0625]]]])
        self.conv.weight = nn.Parameter(torch.cat([w] * channels))
        with torch.no_grad():
            self.conv.bias.zero_()


class DecoderModule(nn.Module):
    forward = _no_forward

    def __init__(self, cin, cdec, nblocks):
        super().__init__()
        self.conv3x3 = ConvBNAct(cin, cdec, 3)
        self.decoder_blocks = nn.Sequential(*[NonBottleneck1D(cdec) for _ in range(nblocks)])
        self.upsample = Upsample(cdec)


class Decoder(nn.Module):
    forward = _no_forward

    def __init__(self, cin, cdec, nblocks, num_classes):
        super().__init__()
        self.decoder_module_1 = DecoderModule(cin, cdec[0], nblocks[0])
        self.decoder_module_2 = DecoderModule(cdec[0], cdec[1], nblocks[1])
        self.decoder_module_3 = DecoderModule(cdec[1], cdec[2], nblocks[2])
        self.conv_out = nn.Conv2d(cdec[2], num_classes, kernel_size=3, padding=1)
        self.upsample1 = Upsample(num_classes)
        self.upsample2 = Upsample(num_classes)


class ESANetOneModality(nn.Module):
    def __init__(self, height=480, width=640, num_classes=37, encoder='resnet18', encoder_block='BasicBlock', channels_decoder=None,
                 pretrained_on_imagenet=True, pretrained_dir='./pretrained_model/resnet_on_imagenet', activation='relu', input_channels=3,
                 encoder_decoder_fusion='add', context_module='ppm', nr_decoder_blocks=None, weighting_in_encoder='None',
                 upsampling='bilinear', pyramid_supervision=True):
        super().__init__()
        if pretrained_on_imagenet:
            raise RuntimeError("pretrained_on_imagenet=True downloads torchvision weights in the reference; load a checkpoint with "
                               "load_state_dict instead")
        unsupported = []
        if encoder not in _BLOCKS or encoder_block != 'BasicBlock':
            unsupported.append(f"encoder={encoder}/{encoder_block}")
        if activation.lower() != 'relu':
            unsupported.append(f"activation={activation}")
        if encoder_decoder_fusion != 'add' or weighting_in_encoder != 'SE-add' or upsampling != 'learned-3x3-zeropad':
            unsupported.append(f"fusion={encoder_decoder_fusion}, weighting={weighting_in_encoder}, upsampling={upsampling}")
        if context_module not in ('ppm', 'ppm-1-2-4-8') or pyramid_supervision:
            unsupported.append(f"context_module={context_module}, pyramid_supervision={pyramid_supervision}")
        if num_classes % 8:
            unsupported.append(f"num_classes={num_classes} (a multiple of 8 is needed: 40 in the reference's RDF-GAN setup)")
        if unsupported:
            raise NotImplementedError("rdfc_gan_b200.esanet covers the configuration of F/bash/test_nyuv2_Ts2T.sh:7-16; got " + "; ".join(unsupported))
        channels_decoder = list(channels_decoder or [128, 128, 128])
        nr_decoder_blocks = list(nr_decoder_blocks or [1, 1, 1])
        self.num_classes, self.input_channels = num_classes, input_channels
        self.encoder = _ResNet(_BLOCKS[encoder], input_channels)
        for i, c in enumerate((64, 64, 128, 256, 512)):
            setattr(self, f'se_layer{i}', SqueezeAndExcitation(c))
        for i, (cenc, cdec) in enumerate(zip((64, 128, 256), reversed(channels_decoder)), start=1):
            setattr(self, f'skip_layer{i}', nn.Sequential(*([ConvBNAct(cenc, cdec, 1)] if cenc != cdec else [])))
        bins = (1, 2, 4, 8) if context_module == 'ppm-1-2-4-8' else (1, 5)
        self.context_module = PyramidPoolingModule(512, channels_decoder[0], bins)
        self.decoder = Decoder(channels_decoder[0], channels_decoder, nr_decoder_blocks, num_classes)
        self.precision = 'bf16'
        self._plans = {}
        self._stamp = None

    def set_precision(self, precision):
        """'bf16' (the default: tensor cores, bf16 activations), 'fp32' (CUDA-core fp32, the parity mode) or 'fp32_tc' (fp32
        activations, tensor cores with split fp16 operands).  Returns self.  A generator's ``set_precision`` does not reach the
        guidance module it holds: set both for an fp32 RDF-GAN end to end."""
        if precision not in _PRECISIONS:
            raise ValueError(f"precision must be one of {_PRECISIONS}, got {precision!r}")
        self.precision = precision
        return self

    # ------------------------------------------------------------------------------------------------------------
    def forward(self, image):
        """image (B, input_channels, H, W) fp32 CUDA -> (B, num_classes, 4*ceil(H/4), ...) fp32 logits, as forward_net (:145-172)"""
        if isinstance(image, dict):
            image = image['image']
        C.require_cuda(image)
        if self.training:
            raise RuntimeError("rdfc_gan_b200.esanet runs the frozen guidance network: call .eval()")
        dev = image.device
        if next(self.parameters()).device != dev:
            raise RuntimeError("ESANet parameters and input live on different devices")
        B, Cin, H, W = image.shape
        if Cin != self.input_channels or H < 32 or W < 32:
            raise RuntimeError(f"ESANet expects (B, {self.input_channels}, >=32, >=32) images, got {tuple(image.shape)}")
        stamp = tuple((p.data_ptr(), p._version) for p in list(self.parameters()) + list(self.buffers()))
        with torch.cuda.device(dev), torch.no_grad():
            if stamp != self._stamp:                       # weights changed (or first call): plans bake folded / packed copies
                self._plans.clear()
                self._stamp = stamp
            key = (B, H, W, dev, self.precision)
            plan = self._plans.get(key)
            if plan is None:
                if len(self._plans) >= 4:
                    del self._plans[next(iter(self._plans))]
                plan = self._plans[key] = _build_plan(self, B, H, W, dev, self.precision)
                plan['inp'].copy_(image)
                _capture(plan)
            plan['inp'].copy_(image)
            plan['graph'].replay()
            return plan['out'].clone()


# ----------------------------------------------------------------------------------------------------------------
def _fold(bn):
    scale = bn.weight.detach().float() / torch.sqrt(bn.running_var.detach().float() + bn.eps)
    return scale, bn.bias.detach().float() - bn.running_mean.detach().float() * scale


def _square(w):
    """(O, I, kh, kw) -> (filters, k): the factorised 3x1 / 1x3 kernels embedded in 3x3 filters with zero taps; 1x1 and 3x3 as they are"""
    O, I, kh, kw = w.shape
    if (kh, kw) in ((1, 1), (3, 3)):
        return w, kh
    full = w.new_zeros(O, I, 3, 3)
    full[:, :, (3 - kh) // 2:(3 - kh) // 2 + kh, (3 - kw) // 2:(3 - kw) // 2 + kw] = w
    return full, 3


def _build_plan(net, B, H, W, dev, precision='bf16'):
    keep, steps = [], []
    adt = torch.bfloat16 if precision == 'bf16' else torch.float32
    x3_descs = []            # fp32_tc: descriptors sharing one split-input workspace, sized once every conv is known

    def new(*shape, dtype=None):
        t = torch.empty(shape, dtype=dtype or adt, device=dev)
        keep.append(t)
        return t

    def conv(x, conv_mod, bn, out, act, residual=None, hin=None, stride=1):
        """x / out / residual: (tensor, c0, C) NHWC slices.  Conv2d (+ folded BatchNorm or bias) + activation on the plan's conv path."""
        w, k = _square(conv_mod.weight.detach().float())
        cin = x[2]
        # fp32_tc: the split-operand tensor-core path where its shape rules allow (all ESANet convs), else CUDA-core fp32
        x3 = precision == 'fp32_tc' and cin % 32 == 0 and out[2] >= 16
        umma = precision == 'bf16' or x3
        if bn is not None:
            scale, shift = _fold(bn)
            if conv_mod.bias is not None:            # conv bias in front of a BatchNorm (NonBottleneck1D): bn(conv + b) = scale conv + (scale b + shift)
                shift = shift + scale * conv_mod.bias.detach().float()
        else:
            scale = torch.ones(w.shape[0], device=dev)
            shift = conv_mod.bias.detach().float() if conv_mod.bias is not None else torch.zeros(w.shape[0], device=dev)
        if x3:       # filters scaled per output channel by a power of two, its inverse folded into `scale`
            packed, scale = pack_weight_x3(w, scale)
        else:
            packed = pack_weight(w, umma)
        scale, shift = scale.contiguous(), shift.contiguous()
        Hi, Wi = hin
        Ho, Wo = (Hi - 1) // stride + 1, (Wi - 1) // stride + 1
        d = C.ConvDesc()
        d.B, d.Hi, d.Wi, d.Ho, d.Wo = B, Hi, Wi, Ho, Wo
        d.kh = d.kw = k
        d.stride, d.pad, d.transposed, d.act = stride, (k - 1) // 2, 0, act
        d.path = C.PATH_UMMA_F32X3 if x3 else (C.PATH_UMMA_BF16 if umma else C.PATH_SIMT_F32)
        if x3:
            x3_descs.append((d, B * Hi * Wi * cin * 4 + 16))         # the split input and its scale factor
        d.inp, d.in2 = C.view(x[0], x[2], x[1]), C.view(None)
        d.out = C.view(out[0], out[2], out[1])
        d.residual = C.view(None) if residual is None else C.view(residual[0], residual[2], residual[1])
        d.weight, d.scale, d.shift = packed.data_ptr(), scale.data_ptr(), shift.data_ptr()
        keep.append((d, packed, scale, shift))
        steps.append(lambda s, d=d: C.check(C.lib.rdfc_conv_forward(ctypes.byref(d), s)))
        return (Ho, Wo)

    def se(x, mod, out, hw):
        """x * sigmoid(fc(mean(x))) (model_utils.py:34-49): statistics, the two tiny FCs, one scaling pass"""
        Cc = x[2]
        Hh, Ww = hw
        nchunk = C.lib.rdfc_instnorm_nchunk(Hh * Ww)
        part, mean, rstd, wts = new(B, nchunk, Cc, 2, dtype=torch.float32), new(B, Cc, dtype=torch.float32), new(B, Cc, dtype=torch.float32), \
            new(B, Cc, dtype=torch.float32)
        zeros = torch.zeros(B, Cc, device=dev)
        w1 = mod.fc[0].weight.detach().float().reshape(mod.fc[0].out_channels, Cc).contiguous()
        w2 = mod.fc[2].weight.detach().float().reshape(Cc, mod.fc[0].out_channels).contiguous()
        b1, b2 = mod.fc[0].bias.detach().float().contiguous(), mod.fc[2].bias.detach().float().contiguous()
        vx, vo = C.view(x[0], x[2], x[1]), C.view(out[0], out[2], out[1])
        keep.extend([zeros, w1, w2, b1, b2, vx, vo])
        R = w1.shape[0]
        steps.append(lambda s: C.check(C.lib.rdfc_instnorm_stats(ctypes.byref(vx), B, Hh, Ww, 1e-5, 0, 0, C.ptr(part), C.ptr(mean), C.ptr(rstd), s)))
        steps.append(lambda s: C.check(C.lib.rdfc_se_weights(C.ptr(mean), C.ptr(w1), C.ptr(b1), C.ptr(w2), C.ptr(b2), C.ptr(wts), B, Cc, R, s)))
        steps.append(lambda s: C.check(C.lib.rdfc_norm_apply(ctypes.byref(vx), C.ptr(zeros), C.ptr(wts), ctypes.byref(vo), B, Hh, Ww, s)))

    def res_layer(x, layer, hw):
        cur, hw_cur = x, hw
        for blk in layer:
            planes = blk.conv1.out_channels
            hw_out = ((hw_cur[0] - 1) // blk.stride + 1, (hw_cur[1] - 1) // blk.stride + 1)
            t1, y = new(B, *hw_out, planes), new(B, *hw_out, planes)
            ident = cur
            if blk.downsample is not None:
                ds = new(B, *hw_out, planes)
                conv(cur, blk.downsample[0], blk.downsample[1], (ds, 0, planes), C.ACT_NONE, hin=hw_cur, stride=blk.stride)
                ident = (ds, 0, planes)
            conv(cur, blk.conv1, blk.bn1, (t1, 0, planes), C.ACT_RELU, hin=hw_cur, stride=blk.stride)
            conv((t1, 0, planes), blk.conv2, blk.bn2, (y, 0, planes), C.ACT_RELU, residual=ident, hin=hw_out)
            cur, hw_cur = (y, 0, planes), hw_out
        return cur, hw_cur

    inp = new(B, net.input_channels, H, W, dtype=torch.float32)
    enc = net.encoder
    # ---- stem: conv1 + bn1 + ReLU, SE, max pool (esa_net_one_modality.py:148-150)
    h2 = ((H + 6 - 7) // 2 + 1, (W + 6 - 7) // 2 + 1)
    a0, a0s = new(B, *h2, 64), new(B, *h2, 64)
    sc0, sh0 = (t.contiguous() for t in _fold(enc.bn1))
    w0 = enc.conv1.weight.detach().float().contiguous()
    v_a0 = C.view(a0)
    keep.extend([sc0, sh0, w0, v_a0])
    steps.append(lambda s: C.check(C.lib.rdfc_first_conv_forward(C.ptr(inp), B, net.input_channels, H, W, C.ptr(w0), 7, 2, 3, C.ptr(sc0), C.ptr(sh0), 1,
                                                                 ctypes.byref(v_a0), s)))
    se((a0, 0, 64), net.se_layer0, (a0s, 0, 64), h2)
    h4 = ((h2[0] - 1) // 2 + 1, (h2[1] - 1) // 2 + 1)
    p0 = new(B, *h4, 64)
    v_a0s, v_p0 = C.view(a0s), C.view(p0)
    keep.extend([v_a0s, v_p0])
    steps.append(lambda s: C.check(C.lib.rdfc_maxpool3x3s2_forward(ctypes.byref(v_a0s), ctypes.byref(v_p0), B, h2[0], h2[1], s)))
    # ---- encoder blocks with SE and skips (:152-170)
    cdec = [net.decoder.decoder_module_1.conv3x3.conv.out_channels, net.decoder.decoder_module_2.conv3x3.conv.out_channels,
            net.decoder.decoder_module_3.conv3x3.conv.out_channels]
    cur, hw = (p0, 0, 64), h4
    skips = []
    nbins = len(net.context_module.bins)
    red = 512 // nbins
    for i in (1, 2, 3, 4):
        cur, hw = res_layer(cur, getattr(enc, f'layer{i}'), hw)
        Cc = cur[2]
        if i < 4:
            s_out = new(B, *hw, Cc)
            se(cur, getattr(net, f'se_layer{i}'), (s_out, 0, Cc), hw)
            cur = (s_out, 0, Cc)
            sk = getattr(net, f'skip_layer{i}')
            if len(sk):
                t = new(B, *hw, sk[0].conv.out_channels)
                conv(cur, sk[0].conv, sk[0].bn, (t, 0, t.shape[3]), C.ACT_RELU, hin=hw)
                skips.append(((t, 0, t.shape[3]), hw))
            else:
                skips.append((cur, hw))
        else:
            # the SE output of layer 4 lands in the first slice of the pyramid pooling module's concat buffer
            ppm_cat = new(B, *hw, Cc + red * nbins)
            se(cur, net.se_layer4, (ppm_cat, 0, Cc), hw)
            cur = (ppm_cat, 0, Cc)
    # ---- pyramid pooling (model_utils.py:99-134, nearest up-sampling under 'learned-3x3*')
    for j, (b, feat) in enumerate(zip(net.context_module.bins, net.context_module.features)):
        pooled, red_t = new(B, b, b, 512), new(B, b, b, red)
        v_src, v_pool = C.view(ppm_cat, 512, 0), C.view(pooled)
        keep.extend([v_src, v_pool])
        steps.append(lambda s, v_src=v_src, v_pool=v_pool, b=b, hw=hw: C.check(C.lib.rdfc_adaptive_avgpool_forward(
            ctypes.byref(v_src), ctypes.byref(v_pool), B, hw[0], hw[1], b, s)))
        conv((pooled, 0, 512), feat[1].conv, feat[1].bn, (red_t, 0, red), C.ACT_RELU, hin=(b, b))
        v_red, v_dst = C.view(red_t), C.view(ppm_cat, red, 512 + j * red)
        keep.extend([v_red, v_dst])
        steps.append(lambda s, v_red=v_red, v_dst=v_dst, b=b, hw=hw: C.check(C.lib.rdfc_upsample_nearest_forward(
            ctypes.byref(v_red), ctypes.byref(v_dst), B, b, b, hw[0], hw[1], s)))
    ctx = new(B, *hw, cdec[0])
    conv((ppm_cat, 0, ppm_cat.shape[3]), net.context_module.final_conv.conv, net.context_module.final_conv.bn, (ctx, 0, cdec[0]), C.ACT_RELU, hin=hw)
    cur = (ctx, 0, cdec[0])
    # ---- decoder (decoder.py:64-134)
    for mi, (mod, (skip, skip_hw)) in enumerate(zip((net.decoder.decoder_module_1, net.decoder.decoder_module_2, net.decoder.decoder_module_3),
                                                    reversed(skips))):
        Cd = cdec[mi]
        t = new(B, *hw, Cd)
        conv(cur, mod.conv3x3.conv, mod.conv3x3.bn, (t, 0, Cd), C.ACT_RELU, hin=hw)
        cur = (t, 0, Cd)
        for blk in mod.decoder_blocks:
            u1, u2, u3, u4 = (new(B, *hw, Cd) for _ in range(4))
            conv(cur, blk.conv3x1_1, None, (u1, 0, Cd), C.ACT_RELU, hin=hw)
            conv((u1, 0, Cd), blk.conv1x3_1, blk.bn1, (u2, 0, Cd), C.ACT_RELU, hin=hw)          # conv bias folded below
            conv((u2, 0, Cd), blk.conv3x1_2, None, (u3, 0, Cd), C.ACT_RELU, hin=hw)
            conv((u3, 0, Cd), blk.conv1x3_2, blk.bn2, (u4, 0, Cd), C.ACT_RELU, residual=cur, hin=hw)
            cur = (u4, 0, Cd)
        up = new(B, *skip_hw, Cd)
        wq, bq = mod.upsample.conv.weight.detach().float().contiguous(), mod.upsample.conv.bias.detach().float().contiguous()
        v_in, v_sk, v_up = C.view(cur[0], cur[2], cur[1]), C.view(skip[0], skip[2], skip[1]), C.view(up)
        keep.extend([wq, bq, v_in, v_sk, v_up])
        steps.append(lambda s, v_in=v_in, v_sk=v_sk, v_up=v_up, wq=wq, bq=bq, hw=hw, skip_hw=skip_hw: C.check(C.lib.rdfc_upsample_dw_forward(
            ctypes.byref(v_in), C.ptr(wq), C.ptr(bq), ctypes.byref(v_sk), ctypes.byref(v_up), None, B, hw[0], hw[1], skip_hw[0], skip_hw[1], s)))
        cur, hw = (up, 0, Cd), skip_hw
    nc = net.num_classes
    logits = new(B, *hw, nc)
    conv(cur, net.decoder.conv_out, None, (logits, 0, nc), C.ACT_NONE, hin=hw)
    hw2, hw4 = (2 * hw[0], 2 * hw[1]), (4 * hw[0], 4 * hw[1])
    up1 = new(B, *hw2, nc)
    out = new(B, nc, *hw4, dtype=torch.float32)
    for k_, (src, src_hw, dst_hw, um) in enumerate(((logits, hw, hw2, net.decoder.upsample1), (up1, hw2, hw4, net.decoder.upsample2))):
        wq, bq = um.conv.weight.detach().float().contiguous(), um.conv.bias.detach().float().contiguous()
        v_in = C.view(src)
        keep.extend([wq, bq, v_in])
        if k_ == 0:
            v_o = C.view(up1)
            keep.append(v_o)
            steps.append(lambda s, v_in=v_in, v_o=v_o, wq=wq, bq=bq, a=src_hw, b=dst_hw: C.check(C.lib.rdfc_upsample_dw_forward(
                ctypes.byref(v_in), C.ptr(wq), C.ptr(bq), None, ctypes.byref(v_o), None, B, a[0], a[1], b[0], b[1], s)))
        else:
            steps.append(lambda s, v_in=v_in, wq=wq, bq=bq, a=src_hw, b=dst_hw: C.check(C.lib.rdfc_upsample_dw_forward(
                ctypes.byref(v_in), C.ptr(wq), C.ptr(bq), None, None, C.ptr(out), B, a[0], a[1], b[0], b[1], s)))
    if x3_descs:             # one stream: the convs run one after the other and can share the [hi | lo] copy of their input
        ws = new(max(n for _, n in x3_descs), dtype=torch.uint8)
        for d, _ in x3_descs:
            d.workspace, d.workspace_bytes = ws.data_ptr(), ws.numel()
    return dict(inp=inp, out=out, steps=steps, keep=keep, graph=None)


def _capture(plan):
    cur = torch.cuda.current_stream()
    side = torch.cuda.Stream()
    side.wait_stream(cur)
    with torch.cuda.stream(side):
        for f in plan['steps']:
            f(side.cuda_stream)
    cur.wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        s = torch.cuda.current_stream().cuda_stream
        for f in plan['steps']:
            f(s)
    plan['graph'] = graph
