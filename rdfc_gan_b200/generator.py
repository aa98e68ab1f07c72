"""Drop-in generators.

``RDFGenerator``     = RDFC-GAN (TPAMI'24)  G/rdf_generator.py:31-414   forward(rgb, depth, normal) -> dict
``DCVGANGenerator``  = RDF-GAN  (CVPR'22)   F/lib/models/generator/rdf_gan_generator/rdf_gan_generator.py:12-361
                                             forward(rgb, depth) -> 5-tuple
(G = /root/reference/RDFC-GAN/lib/models/generator/rdf_generator, F = /root/reference/RDF-GAN.)

Same constructor keywords, same module / parameter names (``state_dict`` loads into and from the reference classes
with strict=True), same outputs.  The forward pass is executed by rdfc_gan_b200.engine on hand-written sm_100a
kernels through the C ABI; tensors must live on a CUDA device (RuntimeError otherwise -- there is no CPU path).
"""
import torch
import torch.nn as nn

from .encoder_decoder import EncoderDecoder, conv_bn_relu
from .engine import GeneratorEngine
from .model_utils import IN, AdaIN, AdaptiveInstanceNorm
from .nlspn import NLSPNRefineModule


class _GeneratorBase(nn.Module):
    def _build(self, encoder_rgb, encoder_depth, pretrained_on_imagenet, semantic_channels_in, fuse_kind, bn,
               rgb_skip_connection_type, depth_skip_connection_type, adain_weighting, rgb_channels_encoder,
               depth_channels_encoder, rgb_channels_decoder, depth_channels_decoder, use_nlspn_refine, nlspn_configs):
        if rgb_skip_connection_type != 'concat' or depth_skip_connection_type != 'concat':
            # the reference's 'add' branch indexes rgb_channels_decoder[4] of a 4-list (rdf_generator.py:120-121)
            raise NotImplementedError("only skip_connection_type='concat' is constructible in the reference")
        if list(rgb_channels_encoder) != [64, 64, 128, 256, 512, 512] or \
                list(depth_channels_encoder) != [64, 64, 128, 256, 512, 512] or \
                list(rgb_channels_decoder) != [256, 128, 64, 64] or list(depth_channels_decoder) != [256, 128, 64, 64]:
            raise NotImplementedError("channel plans other than the reference defaults are not supported "
                                      "(the ResNet layers fix them, encoder_decoder.py:39-46)")
        self.use_nlspn_refine = use_nlspn_refine
        self._train_precision = 'bf16'          # set_train_precision; a plain attribute, not part of state_dict
        self.bn = bn
        self.rgb_skip_connection_type = rgb_skip_connection_type
        self.depth_skip_connection_type = depth_skip_connection_type
        self.fuse_kind = fuse_kind
        self.adain_weighting = bool(adain_weighting)
        self.semantic_channels_in = semantic_channels_in
        self.nlspn_configs = dict(nlspn_configs) if nlspn_configs else None
        ce, cd = rgb_channels_encoder, rgb_channels_decoder
        de, dd = depth_channels_encoder, depth_channels_decoder

        self.rgb_branch_en1 = conv_bn_relu(semantic_channels_in, ce[0], kernel=3, stride=1, padding=1, bn=False)
        self.rgb_branch_encoder_decoder = EncoderDecoder(encoder_rgb, rgb_skip_connection_type, ce[1:], cd,
                                                         pretrained_on_imagenet)
        self.rgb_pred_dec1 = conv_bn_relu(64 + 64, 64, kernel=3, stride=1, padding=1)
        self.rgb_pred_dec0 = conv_bn_relu(64 + 64, 1, kernel=3, stride=1, padding=1, bn=False, relu=False)
        self.rgb_conf_dec1 = conv_bn_relu(64 + 64, 32, kernel=3, stride=1, padding=1)
        self.rgb_conf_dec0 = nn.Sequential(nn.Conv2d(32 + 64, 1, kernel_size=3, stride=1, padding=1), nn.Sigmoid())

        self.depth_branch_en1_rgb = conv_bn_relu(semantic_channels_in, 48, kernel=3, stride=1, padding=1, bn=False)
        self.depth_branch_en1_depth = conv_bn_relu(1, 16, kernel=3, stride=1, padding=1, bn=False)
        self.depth_branch_encoder_decoder = EncoderDecoder(encoder_depth, depth_skip_connection_type, de[1:], dd,
                                                           pretrained_on_imagenet)
        self.id_dec1 = conv_bn_relu(64 + 64, 64, kernel=3, stride=1, padding=1)
        self.id_dec0 = conv_bn_relu(64 + 64, 1, kernel=3, stride=1, padding=1, bn=False, relu=False)
        return ce, cd, de, dd

    def _build_tail(self, ce, cd, de, dd, has_guidance_head, nlspn_configs):
        if has_guidance_head:
            num_neighbors = nlspn_configs['prop_kernel'] * nlspn_configs['prop_kernel'] - 1
            self.gd_dec1 = conv_bn_relu(64 + 64, 64, kernel=3, stride=1, padding=1)
            self.gd_dec0 = conv_bn_relu(64 + 64, num_neighbors, kernel=3, stride=1, padding=1, bn=False, relu=False)
        self.cf_dec1 = conv_bn_relu(64 + 64, 32, kernel=3, stride=1, padding=1)
        self.cf_dec0 = nn.Sequential(nn.Conv2d(32 + 64, 1, kernel_size=3, stride=1, padding=1), nn.Sigmoid())
        if self.use_nlspn_refine:
            self.nlspn_refine_module = NLSPNRefineModule(**nlspn_configs)
        else:
            self.nlspn_refine_module = None     # the reference stores a parameterless NLSPNIdentity object
        for i in range(1, 6):                   # rdf_generator.py:122-146 (concat: identities, no parameters)
            setattr(self, f'rgb_skip_layer{i}', nn.Identity())
            setattr(self, f'depth_skip_layer{i}', nn.Identity())
        # (in_channel, style_dim) of fuse_layer1..5, rdf_generator.py:151-178 (note :163/:169/:175 use the RGB encoder
        # widths for the style dim -- identical numbers with the default plans)
        dims = [(ce[-1], ce[-1]), (cd[0] + ce[-2], dd[0] + de[-2]), (cd[1] + ce[-3], dd[1] + ce[-3]),
                (cd[2] + ce[-4], dd[2] + ce[-4]), (cd[3] + ce[-5], dd[3] + ce[-5])]
        for i, (cin, sdim) in enumerate(dims, start=1):
            if self.fuse_kind == 'WAdaIN':
                layer = AdaptiveInstanceNorm(in_channel=cin, style_dim=sdim, weighting=self.adain_weighting)
            elif self.fuse_kind == 'AdaIN':
                layer = AdaIN()
            elif self.fuse_kind == 'IN':
                layer = IN(in_channel=cin, style_dim=sdim)
            else:
                raise NotImplementedError(self.fuse_kind)
            setattr(self, f'fuse_layer{i}', layer)   # fuse_layer5 is built but never used (rdf_generator.py:371)
        self._engine = None

    # ------------------------------------------------------------------------------------------------------------
    def engine(self, precision=None):
        if self._engine is None:
            object.__setattr__(self, '_engine', GeneratorEngine(self))
        if precision is not None:
            self._engine.precision = precision
        return self._engine

    def set_precision(self, precision):
        """'fp32' (CUDA-core fp32 contraction, the strict <=1e-4 parity mode), 'fp32_tc' (fp32 tensors, contractions on the
        tcgen05 tensor cores with split fp16 operands) or 'bf16' (tcgen05 tensor cores, the throughput mode)."""
        assert precision in ('fp32', 'fp32_tc', 'bf16')
        self.engine(precision)
        return self

    def set_train_precision(self, precision):
        """Arithmetic of the train-mode forward / backward (batch-statistics BatchNorm, autograd): 'bf16' (bf16 activations on the
        tcgen05 tensor cores, the default) or 'fp32_tc' (fp32 activations and gradients; every conv's forward, data gradient and
        filter gradient on the tensor cores with split fp16 operands, each scaled by a power of two from its own largest magnitude;
        fp32 BatchNorm; the cuDNN stems / heads with TF32 off) -- the reference's fp32 training at tensor-core speed.  Strict
        CUDA-core fp32 training is not provided.  Leaves ``set_precision`` (the eval-mode engine) alone, and the reverse; not part of
        ``state_dict``.  Returns self."""
        if precision == 'fp32':
            raise ValueError("train precision 'fp32' (CUDA-core training) is not provided: use 'fp32_tc' for fp32 training on the "
                             "tensor cores, or 'bf16'")
        if precision not in ('bf16', 'fp32_tc'):
            raise ValueError(f"train precision must be 'bf16' or 'fp32_tc', got {precision!r}")
        self._train_precision = precision
        return self

    def _check_inference(self, *tensors):
        for t in tensors:
            if not t.is_cuda:
                raise RuntimeError("rdfc_gan_b200 generators run on CUDA (sm_100a) tensors only; there is no CPU path")
        if torch.is_grad_enabled() and any(t.requires_grad for t in tensors):
            raise RuntimeError("the eval-mode forward is inference-only and returns detached tensors: an input requires grad; "
                               "run under torch.no_grad() or detach the inputs")

    def _run(self, stem_in, depth):
        if self.training:
            # train(): autograd, whatever the grad mode, and each BatchNorm by its own flag (train(): batch statistics, running stats
            # updated; eval(): frozen, running statistics) -- as the reference
            from .train_forward import generator_forward_train
            if self.bn is not True or self.fuse_kind not in ('WAdaIN', 'AdaIN', 'IN'):
                raise NotImplementedError("training-mode forward covers bn=True generators")
            dtype = torch.float32 if getattr(self, '_train_precision', 'bf16') == 'fp32_tc' else torch.bfloat16
            return generator_forward_train(self, stem_in, depth, dtype)
        self._check_inference(stem_in, depth)
        return self.engine().forward(stem_in, depth)

    _OUTPUTS = ('depth_map_1', 'confidence_map_1', 'depth_map_2', 'confidence_map_2', 'pred_depth')

    def _stream(self, pairs, outputs, pre=None):
        """Pipelined inference over HOST (stem input, depth) batches: engine.forward_stream.  ``pre``: a device-side map applied to the
        first tensor of a batch once it is on the GPU (RDF-GAN's guidance network: rgb -> the 40-channel stem input)."""
        want = tuple(self._OUTPUTS.index(k) for k in outputs)
        dev = next(self.parameters()).device
        if dev.type != 'cuda':
            raise RuntimeError("rdfc_gan_b200 generators run on CUDA (sm_100a) devices only; move the module first")
        if self.training:
            raise RuntimeError("stream() is an inference API: call .eval()")
        for res in self.engine().forward_stream(pairs, dev, want, pre=pre):
            yield dict(zip(outputs, res))


class RDFGenerator(_GeneratorBase):
    """rdf_generator.py:31-414.  Eval mode runs the inference engine (``set_precision('bf16' | 'fp32' | 'fp32_tc')``); train mode
    runs batch-statistics BatchNorm with autograd in bf16 or, after ``set_train_precision('fp32_tc')``, in fp32 on split-operand
    tensor-core arithmetic."""

    def __init__(self, encoder_rgb='resnet18', encoder_depth='resnet18', pretrained_on_imagenet=True,
                 semantic_channels_in=3, fuse_depth_in_rgb_decoder='WAdaIN', bn=True,
                 rgb_skip_connection_type='concat', depth_skip_connection_type='concat', adain_weighting=False,
                 rgb_channels_encoder=[64, 64, 128, 256, 512, 512], depth_channels_encoder=[64, 64, 128, 256, 512, 512],
                 rgb_channels_decoder=[256, 128, 64, 64], depth_channels_decoder=[256, 128, 64, 64],
                 use_nlspn_refine=False, nlspn_configs=None, global_guidance_module=None):
        super().__init__()
        ce, cd, de, dd = self._build(encoder_rgb, encoder_depth, pretrained_on_imagenet, semantic_channels_in,
                                     fuse_depth_in_rgb_decoder, bn, rgb_skip_connection_type,
                                     depth_skip_connection_type, adain_weighting, rgb_channels_encoder,
                                     depth_channels_encoder, rgb_channels_decoder, depth_channels_decoder,
                                     use_nlspn_refine, nlspn_configs)
        # rdf_generator.py:58 keeps the guidance module (or an identity lambda); forward never calls it (:283 is commented)
        self.global_guidance_module = global_guidance_module if global_guidance_module is not None else (lambda x: x)
        self._build_tail(ce, cd, de, dd, use_nlspn_refine, nlspn_configs)   # gd_dec* only with NLSPN (:91-95)
        self.use_pretrained_global_guidance_module = False
        self.pretrained_on_imagenet = pretrained_on_imagenet

    def stream(self, batches, outputs=_GeneratorBase._OUTPUTS):
        """Pipelined inference for a stream of HOST batches: ``batches`` yields ``(rgb, depth, normal)`` CPU tensors
        (pinned memory makes the copies asynchronous); yields one dict of pinned CPU tensors per batch, in order, with
        the keys in ``outputs``.  Host->device and device->host copies overlap the forward of the neighbouring batches
        (engine.forward_stream); the arithmetic is exactly ``forward``'s.  A yielded dict is reused two batches later."""
        return self._stream(((normal, depth) for _, depth, normal in batches), outputs)

    def forward(self, rgb, depth, normal):
        """rdf_generator.py:280-414: both stems read ``normal`` (:286,289); ``rgb`` is unused by the reference too."""
        d1, c1, d2, c2, pred = self._run(normal, depth)
        return dict(depth_map_1=d1, confidence_map_1=c1, depth_map_2=d2, confidence_map_2=c2, pred_depth=pred)


class DCVGANGenerator(_GeneratorBase):
    """RDF-GAN generator (rdf_gan_generator.py:12-361).  ``fuse_depth_in_rgb_decoder='AdaIN'`` selects the W-AdaIN
    layer there (:133), and the keyword is spelled ``use_nlpsn_refine`` (:28).  ``global_guidance_module`` is any
    nn.Module mapping rgb -> (B, semantic_channels_in, H, W) (ESANet in the reference's scripts); it is called as is.

    ``set_train_precision('bf16' | 'fp32_tc')`` selects the train-mode arithmetic (see _GeneratorBase.set_train_precision).
    The guidance module keeps its own precision: ``set_precision`` sets the generator's arithmetic only (this repo's ESANet
    stays in its default 'bf16').  RDF-GAN in fp32 end to end is
    ``G.set_precision('fp32'); G.global_guidance_module.set_precision('fp32')``; ``stream`` calls the module as ``forward`` does."""

    def __init__(self, global_guidance_module, encoder_rgb='resnet18', encoder_depth='resnet18',
                 pretrained_on_imagenet=True, semantic_channels_in=40, fuse_depth_in_rgb_decoder='AdaIN', bn=True,
                 rgb_skip_connection_type='concat', depth_skip_connection_type='concat', adain_weighting=False,
                 rgb_channels_encoder=[64, 64, 128, 256, 512, 512], depth_channels_encoder=[64, 64, 128, 256, 512, 512],
                 rgb_channels_decoder=[256, 128, 64, 64], depth_channels_decoder=[256, 128, 64, 64],
                 use_nlpsn_refine=False, nlspn_configs=None):
        super().__init__()
        if fuse_depth_in_rgb_decoder != 'AdaIN':
            raise NotImplementedError("the RDF-GAN generator only defines fuse_depth_in_rgb_decoder='AdaIN' "
                                      "(rdf_gan_generator.py:133)")
        if nlspn_configs is None:
            raise TypeError("nlspn_configs is required (rdf_gan_generator.py:73 indexes it unconditionally)")
        ce, cd, de, dd = self._build(encoder_rgb, encoder_depth, pretrained_on_imagenet, semantic_channels_in,
                                     'WAdaIN', bn, rgb_skip_connection_type, depth_skip_connection_type,
                                     adain_weighting, rgb_channels_encoder, depth_channels_encoder,
                                     rgb_channels_decoder, depth_channels_decoder, use_nlpsn_refine, nlspn_configs)
        self.use_nlpsn_refine = use_nlpsn_refine
        self.global_guidance_module = global_guidance_module
        self._build_tail(ce, cd, de, dd, True, nlspn_configs)               # gd_dec* always exist (:73-76)

    def stream(self, batches, outputs=_GeneratorBase._OUTPUTS):
        """As RDFGenerator.stream for ``(rgb, depth)`` HOST batches.  The guidance network (``global_guidance_module``, e.g. this
        repo's ESANet) runs on the device between the host-to-device copy and the generator, inside the same pipeline."""
        gm = self.global_guidance_module
        pre = None if (gm is None or isinstance(gm, nn.Identity)) else gm
        return self._stream(((rgb, depth) for rgb, depth in batches), outputs, pre=pre)

    def forward(self, rgb, depth):
        """rdf_gan_generator.py:233-361 -> (depth_map_1, confidence_map_1, depth_map_2, confidence_map_2, final)"""
        guidance = rgb if self.global_guidance_module is None else self.global_guidance_module(rgb)
        return self._run(guidance, depth)
