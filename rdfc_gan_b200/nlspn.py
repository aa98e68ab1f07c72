"""NLSPN refinement -- drop-in for nlspn/nlspn_model.py (NLPSN :6-175, NLSPNRefineModule :178-197).

Same constructor arguments, parameter names / shapes (state_dict compatible: ``aff_scale_const``, ``w``, ``b``,
``w_conf``, ``conv_offset_aff.{weight,bias}``), asserts and return tuples.  The forward pass runs two fused sm_100a
kernels through the C ABI (rdfc_nlspn_affinity_forward, rdfc_nlspn_propagate_forward) instead of the reference's
26 DCN calls + ~25 ATen kernels; with gradients enabled the same two stages run as two differentiable ops whose
backwards are fused kernels as well (rdfc_nlspn_affinity_backward, rdfc_nlspn_propagate_backward).  Under
torch.use_deterministic_algorithms the backwards call their _ex variants with RDFC_DETERMINISTIC: fixed-point scatters,
bit-reproducible gradients.  There is no CPU
path and no re-statement of the reference's per-call composition: configurations the fused kernels do not cover
(``prop_kernel != 3``, guidance with other than 8 channels, non-fp32 tensors) raise.
"""
import torch
import torch.nn as nn

from . import _cabi as C


class _PropagateFused(torch.autograd.Function):
    """The T propagation iterations as one differentiable op: forward = rdfc_nlspn_propagate_forward (keeping every
    iteration's result), backward = rdfc_nlspn_propagate_backward (the transposed gather as a scatter per iteration, then ONE
    pass for grad_offset / grad_aff).  Replaces the reference's prop_time ModulatedDeformConvFunction calls and their
    backwards (nlspn_model.py:140-175).  Returns (result, inter) with inter (T,B,1,H,W) = the reference's list_feat stacked;
    gradients arriving through either output are honoured."""

    @staticmethod
    def forward(ctx, feat_init, offset, aff, feat_fix, prop_time, preserve_input):
        B, _, H, W = feat_init.shape
        feat_init, offset, aff = feat_init.contiguous(), offset.contiguous(), aff.contiguous()
        fix = feat_fix.contiguous() if (preserve_input and feat_fix is not None) else None
        out = torch.empty_like(feat_init)
        scratch = torch.empty_like(feat_init)
        inter = torch.empty((prop_time,) + tuple(feat_init.shape), dtype=torch.float32, device=feat_init.device)
        with torch.cuda.device(feat_init.device):
            C.check(C.lib.rdfc_nlspn_propagate_forward(
                C.ptr(feat_init), C.ptr(offset), C.ptr(aff), C.ptr(fix), int(bool(preserve_input)), C.ptr(out),
                C.ptr(scratch), C.ptr(inter) if prop_time > 0 else None, B, H, W, prop_time, 0, None,
                C.stream_ptr(feat_init.device)))
        ctx.save_for_backward(feat_init, offset, aff, fix if fix is not None else feat_init.new_empty(0), inter)
        ctx.cfg = (prop_time, bool(preserve_input), fix is not None)
        return out, inter

    @staticmethod
    def backward(ctx, grad_out, grad_inter):
        feat_init, offset, aff, fix, inter = ctx.saved_tensors
        prop_time, preserve, has_fix = ctx.cfg
        if has_fix and ctx.needs_input_grad[3]:
            raise NotImplementedError("gradient w.r.t. feat_fix (the sparse input depth) is not provided by the fused NLSPN backward")
        B, _, H, W = feat_init.shape
        grad_out = grad_out.contiguous()
        # autograd hands over a dense zero tensor for an unused output; an all-zero grad_inter just adds zeros in the kernel
        g_inter = grad_inter.contiguous() if (grad_inter is not None and prop_time > 0) else None
        g_feat, g_off, g_aff = torch.empty_like(feat_init), torch.empty_like(offset), torch.empty_like(aff)
        scratch = torch.empty((prop_time + 1,) + tuple(feat_init.shape), dtype=torch.float32, device=feat_init.device)
        with torch.cuda.device(feat_init.device):
            C.backward_call(
                "rdfc_nlspn_propagate_backward",
                C.ptr(grad_out), C.ptr(g_inter), C.ptr(feat_init), C.ptr(inter), C.ptr(offset), C.ptr(aff),
                C.ptr(fix) if has_fix else None, int(preserve), C.ptr(g_feat), C.ptr(g_off), C.ptr(g_aff), C.ptr(scratch),
                B, H, W, prop_time, C.stream_ptr(feat_init.device))
        return g_feat, g_off, g_aff, None, None, None


class _AffinityFused(torch.autograd.Function):
    """Offsets + affinities (nlspn_model.py:68-138) as one differentiable op: forward = rdfc_nlspn_affinity_forward, backward =
    rdfc_nlspn_affinity_backward (tanh / scale, confidence product with its transposed 1x1 DCN gathers, abs-sum normalisation,
    aff_ref) followed by the backward of the 8 -> 24 channel conv_offset_aff, which is left to cuDNN (0.24 GFLOP per image)."""

    @staticmethod
    def forward(ctx, guidance, confidence, weight, bias, aff_scale, affinity, conf_prop):
        B, _, H, W = guidance.shape
        guidance, weight, bias = guidance.contiguous(), weight.contiguous(), bias.contiguous()
        conf = confidence.contiguous() if (conf_prop and confidence is not None) else None
        offset = torch.empty((B, 18, H, W), dtype=torch.float32, device=guidance.device)
        aff = torch.empty((B, 9, H, W), dtype=torch.float32, device=guidance.device)
        scale = aff_scale.detach().contiguous()
        with torch.cuda.device(guidance.device):
            C.check(C.lib.rdfc_nlspn_affinity_forward(
                C.ptr(guidance), C.ptr(conf), C.ptr(weight), C.ptr(bias), C.ptr(scale), C.AFFINITY[affinity], int(bool(conf_prop)),
                C.ptr(offset), C.ptr(aff), B, H, W, C.stream_ptr(guidance.device)))
        ctx.save_for_backward(guidance, conf if conf is not None else guidance.new_empty(0), weight, bias, scale, offset)
        ctx.cfg = (affinity, bool(conf_prop), conf is not None)
        return offset, aff

    @staticmethod
    def backward(ctx, g_offset, g_aff):
        guidance, conf, weight, bias, scale, offset = ctx.saved_tensors
        affinity, conf_prop, has_conf = ctx.cfg
        B, _, H, W = guidance.shape
        g_conv = torch.empty((B, 24, H, W), dtype=torch.float32, device=guidance.device)
        g_conf = torch.empty((B, 1, H, W), dtype=torch.float32, device=guidance.device) if has_conf else None
        g_scale = torch.empty((1,), dtype=torch.float32, device=guidance.device) if affinity == 'TGASS' else None
        with torch.cuda.device(guidance.device):
            C.backward_call(
                "rdfc_nlspn_affinity_backward",
                C.ptr(guidance), C.ptr(conf) if has_conf else None, C.ptr(weight), C.ptr(bias), C.ptr(scale), C.AFFINITY[affinity],
                int(conf_prop and has_conf), C.ptr(offset), C.ptr(g_offset.contiguous()), C.ptr(g_aff.contiguous()), C.ptr(g_conv),
                C.ptr(g_conf), C.ptr(g_scale), B, H, W, C.stream_ptr(guidance.device))
        need = ctx.needs_input_grad
        g_guid = torch.nn.grad.conv2d_input(guidance.shape, weight, g_conv, padding=1) if need[0] else None
        g_w = torch.nn.grad.conv2d_weight(guidance, weight.shape, g_conv, padding=1) if need[2] else None
        g_b = g_conv.sum((0, 2, 3)) if need[3] else None
        return (g_guid, g_conf if (has_conf and need[1]) else None, g_w, g_b,
                g_scale if (g_scale is not None and need[4]) else None, None, None)


class NLPSN(nn.Module):
    def __init__(self, channels_g, channels_f, k_g, k_f, prop_time=1, affinity=None, affinity_gamma=0.5,
                 conf_prop=True, preserve_input=False):
        super().__init__()
        self.conf_prop = conf_prop
        self.preserve_input = preserve_input
        assert channels_f == 1, 'only tested with channels_f == 1 but {}'.format(channels_g)
        assert (k_g % 2) == 1, 'only odd kernel is supported but k_g = {}'.format(k_g)
        assert (k_f % 2) == 1, 'only odd kernel is supported but k_g = {}'.format(k_f)
        pad_g = int((k_g - 1) / 2)
        pad_f = int((k_f - 1) / 2)
        self.prop_time = prop_time
        self.affinity = affinity
        self.channels_g = channels_g
        self.channels_f = channels_f
        self.k_g = k_g
        self.k_f = k_f
        self.num = self.k_f * self.k_f - 1          # nlspn_model.py:32
        self.idx_ref = self.num // 2
        if self.affinity in ['AS', 'ASS', 'TC', 'TGASS']:
            self.conv_offset_aff = nn.Conv2d(self.channels_g, 3 * self.num, kernel_size=self.k_g, stride=1,
                                             padding=pad_g, bias=True)
            self.conv_offset_aff.weight.data.zero_()    # :37-38
            self.conv_offset_aff.bias.data.zero_()
            if self.affinity == 'TC':
                self.aff_scale_const = nn.Parameter(self.num * torch.ones(1))
                self.aff_scale_const.requires_grad = False
            elif self.affinity == 'TGASS':
                self.aff_scale_const = nn.Parameter(affinity_gamma * self.num * torch.ones(1))
            else:
                self.aff_scale_const = nn.Parameter(torch.ones(1))
                self.aff_scale_const.requires_grad = False
        else:
            raise NotImplementedError
        # dummy gather parameters, kept for state_dict compatibility (:52-59)
        self.w = nn.Parameter(torch.ones((self.channels_f, 1, self.k_f, self.k_f)))
        self.b = nn.Parameter(torch.zeros(self.channels_f))
        self.w.requires_grad = False
        self.b.requires_grad = False
        self.w_conf = nn.Parameter(torch.ones(1, 1, 1, 1))
        self.w_conf.requires_grad = False
        self.stride = 1
        self.padding = pad_f
        self.dilation = 1
        self.groups = self.channels_f
        self.deformable_groups = 1
        self.im2col_step = 64
        self.return_intermediates = True

    def _require_supported(self, *tensors):
        """The fused kernels hard-code the reference's only setting: a 3x3 propagation kernel fed by 8 guidance channels through
        a 3x3 conv_offset_aff, fp32 tensors on a CUDA device."""
        if self.k_f != 3 or self.k_g != 3 or self.channels_g != 8:
            raise NotImplementedError(
                f"rdfc_gan_b200 NLSPN kernels cover prop_kernel = 3 with 8 guidance channels (the reference's only configuration, "
                f"F/lib/tools/config.py:70); got k_f={self.k_f}, k_g={self.k_g}, channels_g={self.channels_g}")
        C.require_cuda(*tensors, self.conv_offset_aff.weight)
        for t in tensors:
            if t is not None and t.dtype != torch.float32:
                raise RuntimeError(f"rdfc_gan_b200 NLSPN runs on float32 tensors, got {t.dtype}")
            if t is not None and t.device != self.conv_offset_aff.weight.device:
                raise RuntimeError(f"NLSPN parameters are on {self.conv_offset_aff.weight.device}, an input is on {t.device}")

    def _wants_grad(self, *tensors):
        return torch.is_grad_enabled() and (any(t is not None and t.requires_grad for t in tensors) or
                                            any(p.requires_grad for p in self.conv_offset_aff.parameters()) or
                                            self.aff_scale_const.requires_grad)

    def _get_offset_affinity(self, guidance, confidence=None, rgb=None):
        """nlspn_model.py:68-138 -> offset (B,18,H,W), aff (B,9,H,W)"""
        conf = confidence if self.conf_prop else None
        self._require_supported(guidance, conf)
        if self._wants_grad(guidance, conf):
            return _AffinityFused.apply(guidance, conf, self.conv_offset_aff.weight, self.conv_offset_aff.bias,
                                        self.aff_scale_const, self.affinity, self.conf_prop)
        B, _, H, W = guidance.shape
        guidance = guidance.contiguous()
        conf = None if conf is None else conf.contiguous()
        offset = torch.empty((B, 18, H, W), dtype=torch.float32, device=guidance.device)
        aff = torch.empty((B, 9, H, W), dtype=torch.float32, device=guidance.device)
        with torch.cuda.device(guidance.device):
            C.check(C.lib.rdfc_nlspn_affinity_forward(
                C.ptr(guidance), C.ptr(conf), C.ptr(self.conv_offset_aff.weight.detach().contiguous()),
                C.ptr(self.conv_offset_aff.bias.detach().contiguous()), C.ptr(self.aff_scale_const.detach()),
                C.AFFINITY[self.affinity], int(bool(self.conf_prop)), C.ptr(offset), C.ptr(aff), B, H, W,
                C.stream_ptr(guidance.device)))
        return offset, aff

    def forward(self, feat_init, guidance, confidence=None, feat_fix=None, rgb=None):
        """nlspn_model.py:146-175 -> (feat_result, list_feat, offset, aff, aff_scale_const.data)"""
        assert self.channels_g == guidance.shape[1]
        assert self.channels_f == feat_init.shape[1]
        if self.conf_prop:
            assert confidence is not None
        offset, aff = self._get_offset_affinity(guidance, confidence, rgb)
        if self.preserve_input:
            assert feat_init.shape == feat_fix.shape
        fix = feat_fix if self.preserve_input else None
        self._require_supported(feat_init, fix)
        T = self.prop_time
        if self._wants_grad(feat_init, offset, aff):
            feat_result, inter = _PropagateFused.apply(feat_init, offset, aff, fix, T, self.preserve_input)
        else:
            B, _, H, W = feat_init.shape
            feat_init = feat_init.contiguous()
            feat_result, scratch = torch.empty_like(feat_init), torch.empty_like(feat_init)
            inter = (torch.empty((T,) + tuple(feat_init.shape), dtype=torch.float32, device=feat_init.device)
                     if self.return_intermediates and T > 0 else None)
            with torch.cuda.device(feat_init.device):
                C.check(C.lib.rdfc_nlspn_propagate_forward(
                    C.ptr(feat_init), C.ptr(offset.contiguous()), C.ptr(aff.contiguous()), C.ptr(None if fix is None else fix.contiguous()),
                    int(bool(self.preserve_input)), C.ptr(feat_result), C.ptr(scratch), C.ptr(inter), B, H, W, T, 0, None,
                    C.stream_ptr(feat_init.device)))
        list_feat = list(inter.unbind(0)) if (self.return_intermediates and inter is not None and T > 0) else []
        return feat_result, list_feat, offset, aff, self.aff_scale_const.data


class NLSPNRefineModule(nn.Module):
    """nlspn_model.py:178-197"""

    def __init__(self, prop_kernel=3, prop_time=18, affinity='TGASS', affinity_gamma=0.5, conf_prop=True,
                 preserve_input=False):
        super().__init__()
        self.num_neighbors = prop_kernel * prop_kernel - 1
        self.conf_prop = conf_prop
        self.prop_layer = NLPSN(channels_g=self.num_neighbors, channels_f=1, k_g=3, k_f=prop_kernel,
                                prop_time=prop_time, affinity=affinity, affinity_gamma=affinity_gamma,
                                conf_prop=conf_prop, preserve_input=preserve_input)
        self.prop_layer.return_intermediates = False    # the wrapper drops y_inter (:193-197)

    def forward(self, init_pred_depth, guide, confidence, origin_depth, origin_rgb=None):
        y, y_inter, offset, aff, aff_const = self.prop_layer(init_pred_depth, guide, confidence, origin_depth,
                                                             origin_rgb)
        return y, confidence
