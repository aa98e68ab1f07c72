"""``ResnetGenerator`` (RDFC-GAN's G_B2A, depth -> RGB of the cycle) -- drop-in for
C/lib/models/generator/resnet_generator.py:6-98 (C = /root/reference/RDFC-GAN): same constructor, the same ``self.model``
Sequential of standard modules (state_dict keys ``model.<i>...`` load into / from the reference class with strict=True).

``forward`` walks that Sequential over NHWC activations: the 3x3 convolutions (stride-2 down-sampling, the 2 x n_blocks
residual-block convs) and the two ConvTranspose2d(k3, s2, p1, op1) layers -- all with >= 64 input channels, > 97 % of the FLOPs --
run on the tcgen05 conv kernel through ``train_ops.conv2d_nhwc`` (forward, data gradient, filter gradient), BatchNorm2d in train()
mode on the fused batch-statistics kernels, the reflection / replication pads on ``train_ops.pad_nhwc`` (a copy forward, a
fixed-order gather backward: reproducible under torch.use_deterministic_algorithms).  Each BatchNorm2d follows its own flag, as in
PyTorch: in a train()-mode generator, a frozen one (eval() mode, running statistics) after a tensor-core conv is folded into that
conv (``train_ops.conv_bn_act_frozen``, no activation; its buffers stay untouched), and one after a 7x7 conv runs as the PyTorch
module.  The two 7x7 convolutions (1 or 3 channels on one side), LeakyReLU(0.01) / PReLU / Tanh and eval-mode / instance
normalisation are differentiable PyTorch ops on the same tensors.

``set_train_precision`` picks the activations' dtype: bf16 (default) or fp32 (``'fp32_tc'``: split-operand tensor-core convs, fp32
BatchNorm, the 7x7 convs in true fp32 with TF32 off).  G_B2A has no separate inference engine, so the setting holds in train() and
eval() alike.  CUDA only: there is no CPU path.
"""
import torch
import torch.nn as nn
import torch.nn.functional as F

from . import _cabi as C
from .generator import _GeneratorBase
from .train_forward import _ConvFP32
from .train_ops import bn_act, bn_frozen, conv2d_nhwc, conv_bn_act_frozen, pad_nhwc


def _nchw(t):
    """NHWC tensor -> the standard-strided NCHW tensor F.pad returns.  cuDNN picks a conv's algorithm by the input's memory format, so
    the 7x7 convs after a pad see the layout they saw when the pads were F.pad: bf16 outputs bit for bit those of that composition."""
    B, H, W, Cc = t.shape
    return t.reshape(B, 1, H, W) if Cc == 1 else t.permute(0, 3, 1, 2).contiguous()


class ResnetBlock(nn.Module):
    """resnet_generator.py:61-98: x + conv_block(x), conv_block = [pad, conv3x3, norm, LeakyReLU(0.01), (dropout), pad, conv3x3, norm]"""

    def __init__(self, dim, padding_type, norm_layer, use_dropout, use_bias):
        super().__init__()
        blocks = []
        for half in range(2):
            p = 0
            if padding_type == 'reflect':
                blocks.append(nn.ReflectionPad2d(1))
            elif padding_type == 'replicate':
                blocks.append(nn.ReplicationPad2d(1))
            elif padding_type == 'zero':
                p = 1
            else:
                raise NotImplementedError('padding [%s] is not implemented' % padding_type)
            blocks += [nn.Conv2d(dim, dim, kernel_size=3, padding=p, bias=use_bias), norm_layer(dim)]
            if half == 0:
                blocks.append(nn.LeakyReLU(negative_slope=0.01, inplace=True))
                if use_dropout:
                    blocks.append(nn.Dropout(0.5))
        self.conv_block = nn.Sequential(*blocks)

    def forward(self, x):
        raise RuntimeError("ResnetBlock is evaluated by ResnetGenerator.forward (NHWC on the sm_100a kernels)")


class ResnetGenerator(nn.Module):
    def __init__(self, input_channels, output_channels, ngf=64, norm_layer='BN2d', use_dropout=False, n_blocks=6, padding_type='reflect'):
        super().__init__()
        assert n_blocks >= 0
        norm_layer = nn.BatchNorm2d if norm_layer.lower() == 'bn2d' else nn.InstanceNorm2d
        use_bias = norm_layer == nn.InstanceNorm2d
        model = [nn.ReflectionPad2d(3), nn.Conv2d(input_channels, ngf, kernel_size=7, padding=0, bias=use_bias), norm_layer(ngf),
                 nn.LeakyReLU(negative_slope=0.01, inplace=True)]
        for i in range(2):
            mult = 2 ** i
            model += [nn.Conv2d(ngf * mult, ngf * mult * 2, kernel_size=3, stride=2, padding=1, bias=use_bias), norm_layer(ngf * mult * 2),
                      nn.PReLU(init=0.25)]
        for _ in range(n_blocks):
            model.append(ResnetBlock(ngf * 4, padding_type=padding_type, norm_layer=norm_layer, use_dropout=use_dropout, use_bias=use_bias))
        for i in range(2):
            mult = 2 ** (2 - i)
            model += [nn.ConvTranspose2d(ngf * mult, ngf * mult // 2, kernel_size=3, stride=2, padding=1, output_padding=1, bias=use_bias),
                      norm_layer(ngf * mult // 2), nn.PReLU(init=0.25)]
        model += [nn.ReflectionPad2d(3), nn.Conv2d(ngf, output_channels, kernel_size=7, padding=0), nn.Tanh()]
        self.model = nn.Sequential(*model)
        self._train_precision = 'bf16'          # set_train_precision; a plain attribute, not part of state_dict

    def set_train_precision(self, precision):
        """'bf16' (bf16 activations, the default) or 'fp32_tc' (fp32 activations and gradients: the 3x3 / transposed convs' forward,
        data and filter gradients on the tensor cores with split fp16 operands, fp32 BatchNorm, the 7x7 convs in true fp32 with
        TF32 off, PReLU / LeakyReLU / Tanh / eval-mode and instance normalisation in fp32) -- the reference's fp32 arithmetic at
        tensor-core speed.  'fp32' (CUDA-core training) is not provided.  G_B2A has no separate inference engine: the setting applies
        to its forward in train() and eval() mode alike.  Not part of ``state_dict``.  Returns self."""
        return _GeneratorBase.set_train_precision(self, precision)

    # ------------------------------------------------------------------------------------------------------------
    @staticmethod
    def _tc_ok(m, x):
        """a layer the tensor-core conv covers: 3x3, >= 32-aligned input channels, stride 1 / 2"""
        Cin = x.shape[3]
        if isinstance(m, nn.ConvTranspose2d):
            return (m.kernel_size == (3, 3) and m.stride == (2, 2) and m.padding == (1, 1) and m.output_padding == (1, 1) and
                    Cin % 32 == 0 and m.out_channels % 8 == 0 and m.groups == 1)
        return (m.kernel_size == (3, 3) and m.stride in ((1, 1), (2, 2)) and m.padding in ((0, 0), (1, 1)) and m.dilation == (1, 1) and
                m.groups == 1 and Cin % 32 == 0 and m.out_channels % 8 == 0)

    def _walk(self, seq, x):
        """x: bf16 or fp32 (fp32_tc) NHWC.  Torch modules see it as a channels-last NCHW view (no copy)."""
        dt = x.dtype
        fp32 = dt == torch.float32
        def via_torch(mod, t):
            return mod(t.permute(0, 3, 1, 2)).permute(0, 2, 3, 1)
        mods = list(seq)
        prev, fused = None, None
        for i, m in enumerate(mods):
            after_pad, prev = isinstance(prev, (nn.ReflectionPad2d, nn.ReplicationPad2d)), m
            if m is fused:                                               # folded into the conv before it
                continue
            if isinstance(m, ResnetBlock):
                x = x + self._walk(m.conv_block, x)
            elif isinstance(m, (nn.ReflectionPad2d, nn.ReplicationPad2d)):
                x = pad_nhwc(x, m.padding, 'reflect' if isinstance(m, nn.ReflectionPad2d) else 'replicate')
            elif isinstance(m, (nn.Conv2d, nn.ConvTranspose2d)) and self._tc_ok(m, x) and (m.padding != (0, 0) or m.stride == (1, 1)):
                nxt = mods[i + 1] if i + 1 < len(mods) else None
                if self.training and m.bias is None and isinstance(nxt, nn.BatchNorm2d) and bn_frozen(nxt):
                    fused = nxt                                          # conv + frozen BatchNorm in one launch
                    conv = lambda t, k, s, tr=False: conv_bn_act_frozen(t, m.weight, nxt, k, s, tr)
                else:
                    conv = lambda t, k, s, tr=False: conv2d_nhwc(t, m.weight, k, s, tr)
                if isinstance(m, nn.ConvTranspose2d):
                    y = conv(x, 3, 2, True)
                elif m.padding == (0, 0):        # the input was padded explicitly (reflection): zero-pad conv, then drop the border
                    y = conv(x, 3, 1)[:, 1:-1, 1:-1]
                else:
                    y = conv(x, 3, m.stride[0])
                x = y if m.bias is None else (y.float() + m.bias).to(dt)
            elif isinstance(m, (nn.Conv2d, nn.ConvTranspose2d)):         # 7x7 / thin convs: fp32 cuDNN (true fp32 in fp32_tc)
                xin = _nchw(x) if after_pad else x.permute(0, 3, 1, 2)
                if not fp32:
                    y = m(xin.float())
                elif (isinstance(m, nn.ConvTranspose2d) or m.kernel_size == (3, 3) or m.stride != (1, 1) or m.dilation != (1, 1)
                      or m.groups != 1 or m.padding[0] != m.padding[1] or m.padding_mode != 'zeros'):
                    raise RuntimeError(f"fp32_tc runs 3x3 and transposed convs on the tensor cores, which need input channels % 32 == 0, "
                                       f"output channels % 8 == 0, stride 1 / 2 and padding 0 / 1 (stride 2: 1): {m} on {x.shape[3]} "
                                       f"channels does not qualify")
                else:
                    y = _ConvFP32.apply(xin, m.weight, m.bias, m.padding[0])
                x = y.permute(0, 2, 3, 1).to(dt)
            elif isinstance(m, nn.BatchNorm2d) and self.training and not bn_frozen(m) and x.shape[3] % 8 == 0:
                x = bn_act(x.contiguous(), m, None, C.ACT_NONE)
            elif isinstance(m, (nn.BatchNorm2d, nn.InstanceNorm2d)):
                x = via_torch(m, x.float()).to(dt)                      # eval-mode / frozen or instance normalisation: fp32 PyTorch
            elif isinstance(m, nn.LeakyReLU):                            # not in place: the producer saved its output for backward
                x = F.leaky_relu(x, m.negative_slope)
            elif isinstance(m, nn.PReLU):                                # fp32 slope parameter: evaluate in fp32
                x = via_torch(m, x.float()).to(dt)
            else:                                                        # Tanh, dropout: element-wise PyTorch
                x = via_torch(m, x)
        return x

    def forward(self, x):
        C.require_cuda(x)
        dt = torch.float32 if self._train_precision == 'fp32_tc' else torch.bfloat16
        y = self._walk(self.model, x.permute(0, 2, 3, 1).to(dt))
        return y.permute(0, 3, 1, 2).float().contiguous()
