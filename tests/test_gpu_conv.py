"""-m gpu: rdfc_conv_forward (CUDA-core fp32 kernel and the tcgen05 bf16 kernel) and the norm/fusion kernels against CPU
torch.nn.functional restatements of the reference layers (encoder_decoder/common.py:29-61, model_utils.py:53-129)."""
import ctypes
import math

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu


def _run_conv(x_nchw, w, scale, shift, *, stride=1, pad=1, act=0, transposed=False, residual=None, bf16=False, crop=None,
              in_pad=0, out_pad=0):
    """x (B,Cin,H,W) fp32 cpu; w conv (Cout,Cin,k,k) or convT (Cin,Cout,k,k).  Returns NCHW fp32 cpu result."""
    from rdfc_gan_b200 import _cabi as C
    B, Cin, H, W = x_nchw.shape
    k = w.shape[-1]
    wg = (w.permute(1, 0, 2, 3) if transposed else w).float()
    Cout = wg.shape[0]
    if transposed:
        Ho, Wo = crop if crop else (2 * H, 2 * W)
    else:
        Ho, Wo = (H + 2 * pad - k) // stride + 1, (W + 2 * pad - k) // stride + 1
    dt = torch.bfloat16 if bf16 else torch.float32
    xin = torch.zeros(B, H, W, Cin + in_pad, dtype=dt, device="cuda")
    xin[..., in_pad:] = x_nchw.permute(0, 2, 3, 1).to(dt).cuda()
    out = torch.full((B, Ho, Wo, Cout + out_pad), 7.0, dtype=dt, device="cuda")
    g = wg.permute(0, 2, 3, 1).reshape(Cout, k * k, Cin)
    if bf16:
        CoutP = (Cout + 15) // 16 * 16
        g = torch.cat([g, g.new_zeros(CoutP - Cout, k * k, Cin)], 0)
        packed = g.reshape(CoutP, k * k, Cin // 8, 8).permute(1, 2, 0, 3).contiguous().to(torch.bfloat16).cuda()
    else:
        packed = g.permute(1, 2, 0).contiguous().cuda()
    d = C.ConvDesc()
    d.B, d.Hi, d.Wi, d.Ho, d.Wo = B, H, W, Ho, Wo
    d.kh = d.kw = k
    d.stride, d.pad, d.transposed, d.act = stride, pad, int(transposed), act
    d.path = C.PATH_UMMA_BF16 if bf16 else C.PATH_SIMT_F32
    d.inp, d.in2, d.out = C.view(xin, Cin, in_pad), C.view(None), C.view(out, Cout, out_pad)
    res_t = None
    if residual is not None:
        res_t = residual.permute(0, 2, 3, 1).to(dt).contiguous().cuda()
        d.residual = C.view(res_t)
    else:
        d.residual = C.view(None)
    sc, sh = scale.float().cuda(), shift.float().cuda()
    d.weight, d.scale, d.shift = packed.data_ptr(), sc.data_ptr(), sh.data_ptr()
    C.check(C.lib.rdfc_conv_forward(ctypes.byref(d), C.stream_ptr()))
    torch.cuda.synchronize()
    if out_pad:
        assert (out[..., :out_pad].float() == 7.0).all(), "wrote outside its channel slice"
    return out[..., out_pad:].float().permute(0, 3, 1, 2).cpu()


def _ref_conv(x, w, scale, shift, *, stride=1, pad=1, act=0, transposed=False, residual=None, crop=None, bf16=False):
    if bf16:    # the kernel sees bf16-rounded inputs / weights / residual and accumulates in fp32
        x, w = x.bfloat16().float(), w.bfloat16().float()
        residual = None if residual is None else residual.bfloat16().float()
    if transposed:
        y = F.conv_transpose2d(x.double(), w.double(), None, stride=2, padding=1, output_padding=1)
        if crop:
            y = y[:, :, :crop[0], :crop[1]]
    else:
        y = F.conv2d(x.double(), w.double(), None, stride, pad)
    y = y * scale.double().view(1, -1, 1, 1) + shift.double().view(1, -1, 1, 1)
    if residual is not None:
        y = y + residual.double()
    y = [lambda v: v, F.relu, lambda v: F.leaky_relu(v, 0.2), torch.tanh, torch.sigmoid][act](y)
    return y.float()


CASES = [
    # B, Cin, Cout, H, W, k, stride, transposed, act, residual, crop
    (2, 64, 64, 20, 27, 3, 1, False, 1, True, None),
    (1, 128, 96, 17, 35, 3, 1, False, 2, False, None),
    (2, 64, 128, 21, 30, 3, 2, False, 1, False, None),
    (2, 64, 128, 21, 30, 1, 2, False, 0, False, None),
    (1, 192, 384, 9, 13, 1, 1, False, 0, False, None),
    (2, 96, 64, 7, 10, 3, 2, True, 2, False, (13, 20)),
    (1, 256, 160, 33, 18, 3, 1, False, 2, False, None),
    (1, 512, 512, 8, 10, 3, 1, False, 1, True, None),
    # large-grid configurations (wide tiles, N = 256, two accumulators, four parity planes): the shapes bench.py runs
    (6, 128, 256, 114, 152, 3, 2, False, 1, False, None),
    (8, 256, 256, 57, 76, 3, 1, False, 1, True, None),
    (4, 64, 64, 228, 304, 3, 1, False, 1, True, None),
    (2, 192, 64, 114, 152, 3, 2, True, 2, False, None),
    # stride 2 through the dense plane (SWIZZLE_128B pixel-pair rows): odd sizes, wide N, 1x1
    (3, 256, 512, 57, 75, 3, 2, False, 1, False, None),
    (2, 128, 256, 29, 38, 1, 2, False, 0, False, None),
    (2, 512, 512, 29, 38, 3, 2, False, 1, False, None),
    # one-accumulator 128 -> 128 tiles; 40 x 40 outputs at stride 1, stride 2 and transposed; 1x1 convs that stage three
    # k-blocks at once (kbs = 3) at stride 1 and 2
    (2, 64, 64, 40, 40, 3, 1, False, 1, False, None),
    (1, 128, 128, 57, 76, 3, 1, False, 1, False, None),
    (2, 64, 128, 40, 40, 3, 2, False, 1, False, None),
    (1, 64, 64, 20, 20, 3, 2, True, 1, False, None),
    (2, 96, 192, 33, 21, 1, 1, False, 1, False, None),
    (2, 96, 192, 33, 21, 1, 2, False, 2, False, None),
]


@pytest.mark.parametrize("case", CASES)
@pytest.mark.parametrize("bf16", [False, True])
def test_conv_paths(case, bf16):
    B, Cin, Cout, H, W, k, stride, transposed, act, use_res, crop = case
    gen = torch.Generator().manual_seed(hash(case) % 1000)
    x = torch.randn(B, Cin, H, W, generator=gen)
    wshape = (Cin, Cout, k, k) if transposed else (Cout, Cin, k, k)
    w = torch.randn(wshape, generator=gen) / math.sqrt(Cin * k * k)
    scale = 0.5 + torch.rand(Cout, generator=gen)
    shift = 0.2 * torch.randn(Cout, generator=gen)
    pad = (k - 1) // 2
    kw = dict(stride=stride, pad=pad, act=act, transposed=transposed, crop=crop)
    ref0 = _ref_conv(x, w, scale, shift, **kw)
    res = torch.randn(ref0.shape, generator=gen) if use_res else None
    ref = _ref_conv(x, w, scale, shift, residual=res, bf16=bf16, **kw)
    got = _run_conv(x, w, scale, shift, residual=res, bf16=bf16, in_pad=32, out_pad=16, **kw)
    assert got.shape == ref.shape
    err = (got - ref).abs().max().item()
    # fp32 path: accumulation order only.  bf16 path: inputs are pre-rounded in the reference, the only extra error
    # is the bf16 rounding of the OUTPUT (rel 2^-9) plus fp32 accumulation order.
    tol = 2e-5 * max(1.0, ref.abs().max().item()) if not bf16 else 2.0 ** -8 * max(1.0, ref.abs().max().item())
    assert err <= tol, (err, tol)


def test_small_cout_and_stem_kernels():
    """Cout <= 8 heads with two concatenated sources and NCHW output; 3-channel NCHW stem (rdf_generator.py:60-102)."""
    from rdfc_gan_b200 import _cabi as C
    gen = torch.Generator().manual_seed(5)
    B, H, W = 2, 19, 23
    a, b2 = torch.randn(B, 64, H, W, generator=gen), torch.randn(B, 64, H, W, generator=gen)
    for Cout, act in ((1, 3), (8, 0), (1, 4)):
        w = torch.randn(Cout, 128, 3, 3, generator=gen) / 30
        bias = torch.randn(Cout, generator=gen)
        ref = [None, None, None, torch.tanh, torch.sigmoid][act](F.conv2d(torch.cat([a, b2], 1).double(), w.double(), bias.double(), 1, 1)) \
            if act else F.conv2d(torch.cat([a, b2], 1).double(), w.double(), bias.double(), 1, 1)
        buf = torch.zeros(B, H, W, 160, device="cuda")
        buf[..., 0:64] = a.permute(0, 2, 3, 1).cuda()
        buf[..., 96:160] = b2.permute(0, 2, 3, 1).cuda()
        out = torch.empty(B, Cout, H, W, device="cuda")
        packed = w.permute(0, 2, 3, 1).reshape(Cout, 9, 128).permute(1, 2, 0).contiguous().cuda()
        d = C.ConvDesc()
        d.B, d.Hi, d.Wi, d.Ho, d.Wo, d.kh, d.kw, d.stride, d.pad, d.act, d.path = B, H, W, H, W, 3, 3, 1, 1, act, 0
        d.inp, d.in2, d.out, d.residual = C.view(buf, 64, 0), C.view(buf, 64, 96), C.view(out, nchw=True), C.view(None)
        bc = bias.cuda()
        d.weight, d.scale, d.shift = packed.data_ptr(), None, bc.data_ptr()
        C.check(C.lib.rdfc_conv_forward(ctypes.byref(d), C.stream_ptr()))
        assert (out.cpu().double() - ref).abs().max() < 2e-5
    x = torch.randn(B, 3, H, W, generator=gen)
    w = torch.randn(48, 3, 3, 3, generator=gen) / 5
    bias = torch.randn(48, generator=gen)
    ref = F.leaky_relu(F.conv2d(x.double(), w.double(), bias.double(), 1, 1), 0.2)
    xc = x.cuda()
    out = torch.zeros(B, H, W, 64, device="cuda")
    packed = w.permute(0, 2, 3, 1).reshape(48, 9, 3).permute(1, 2, 0).contiguous().cuda()
    d = C.ConvDesc()
    d.B, d.Hi, d.Wi, d.Ho, d.Wo, d.kh, d.kw, d.stride, d.pad, d.act, d.path = B, H, W, H, W, 3, 3, 1, 1, 2, 0
    d.inp, d.in2, d.out, d.residual = C.view(xc, nchw=True), C.view(None), C.view(out, 48, 0), C.view(None)
    bc = bias.cuda()
    d.weight, d.scale, d.shift = packed.data_ptr(), None, bc.data_ptr()
    C.check(C.lib.rdfc_conv_forward(ctypes.byref(d), C.stream_ptr()))
    assert (out[..., :48].permute(0, 3, 1, 2).cpu().double() - ref).abs().max() < 2e-5
    assert (out[..., 48:] == 0).all()


def test_instnorm_and_wadain():
    from rdfc_gan_b200 import _cabi as C
    gen = torch.Generator().manual_seed(9)
    B, Cc, H, W = 2, 192, 29, 38
    x = 3 + 2 * torch.randn(B, Cc, H, W, generator=gen)
    gb = torch.randn(B, 2 * Cc, H, W, generator=gen)
    xn = x.permute(0, 2, 3, 1).contiguous().cuda()
    gbn = gb.permute(0, 2, 3, 1).contiguous().cuda()
    nchunk = C.lib.rdfc_instnorm_nchunk(H * W)
    part = torch.empty(B, nchunk, Cc, 2, device="cuda")
    mean, rstd = torch.empty(B, Cc, device="cuda"), torch.empty(B, Cc, device="cuda")
    vx, vgb = C.view(xn), C.view(gbn)
    C.check(C.lib.rdfc_instnorm_stats(ctypes.byref(vx), B, H, W, 1e-5, 0, 0, C.ptr(part), C.ptr(mean), C.ptr(rstd), C.stream_ptr()))
    xd = x.double()
    assert (mean.cpu().double() - xd.mean((2, 3))).abs().max() < 1e-5
    assert (rstd.cpu().double() - 1 / torch.sqrt(xd.var((2, 3), unbiased=False) + 1e-5)).abs().max() < 1e-5
    out = torch.empty_like(xn)
    vo = C.view(out)
    C.check(C.lib.rdfc_wadain_apply(ctypes.byref(vx), ctypes.byref(vgb), None, None, C.ptr(mean), C.ptr(rstd), ctypes.byref(vo),
                                    B, H, W, C.stream_ptr()))
    ref = gb[:, :Cc].double() * F.instance_norm(xd, eps=1e-5) + gb[:, Cc:].double()
    assert (out.permute(0, 3, 1, 2).cpu().double() - ref).abs().max() < 2e-5
    # AdaIN statistics: unbiased variance, std returned
    C.check(C.lib.rdfc_instnorm_stats(ctypes.byref(vx), B, H, W, 1e-5, 1, 1, C.ptr(part), C.ptr(mean), C.ptr(rstd), C.stream_ptr()))
    assert (rstd.cpu().double() - torch.sqrt(xd.var((2, 3), unbiased=True) + 1e-5)).abs().max() < 1e-5


# ---------------------------------------------------------------------------------------------------------------------
# rdfc_stem_forward: the three input stems of rdf_generator.py:286-292 as one tensor-core launch
@pytest.mark.parametrize("B,H,W", [(1, 16, 24), (2, 37, 45), (1, 228, 304)])
def test_fused_stems_match_three_convs(B, H, W):
    from rdfc_gan_b200 import _cabi as C
    g = torch.Generator().manual_seed(H * W + B)
    normal, depth = torch.randn(B, 3, H, W, generator=g), torch.randn(B, 1, H, W, generator=g)
    w_r, w_dr, w_dd = (0.3 * torch.randn(64, 3, 3, 3, generator=g), 0.3 * torch.randn(48, 3, 3, 3, generator=g),
                       0.3 * torch.randn(16, 1, 3, 3, generator=g))
    bias = 0.1 * torch.randn(128, generator=g)
    # reference (conv_bn_relu with bn=False: conv + bias + LeakyReLU(0.2)), on bf16-rounded operands like the kernel
    rb = lambda t: t.bfloat16().float()
    ref_r = F.leaky_relu(F.conv2d(rb(normal), rb(w_r), bias[:64], padding=1), 0.2)
    ref_d = F.leaky_relu(torch.cat([F.conv2d(rb(normal), rb(w_dr), bias[64:112], padding=1),
                                    F.conv2d(rb(depth), rb(w_dd), bias[112:], padding=1)], 1), 0.2)
    # im2col filter bank: rows k = ci*9 + tap for the 3 `normal` channels, then the depth map's nine taps
    Wk = torch.zeros(128, 64)
    Wk[:64, :27], Wk[64:112, :27], Wk[112:, 27:36] = w_r.reshape(64, 27), w_dr.reshape(48, 27), w_dd.reshape(16, 9)
    packed = Wk.reshape(128, 1, 8, 8).permute(1, 2, 0, 3).contiguous().to(torch.bfloat16).cuda()
    out_r = torch.full((B, H, W, 96 + 64), 7.0, dtype=torch.bfloat16, device="cuda")       # destination slices of wider
    out_d = torch.full((B, H, W, 160 + 64), 7.0, dtype=torch.bfloat16, device="cuda")      # buffers, as in the engine
    n_d, d_d = normal.cuda().contiguous(), depth.cuda().contiguous()
    sc, sh = torch.ones(128, device="cuda"), bias.cuda()
    d = C.StemDesc()
    d.B, d.H, d.W = B, H, W
    d.in0, d.C0, d.in1 = n_d.data_ptr(), 3, d_d.data_ptr()
    d.out, d.out2 = C.view(out_r, 64, 96), C.view(out_d, 64, 160)
    d.weight, d.scale, d.shift, d.act = packed.data_ptr(), sc.data_ptr(), sh.data_ptr(), C.ACT_LEAKY02
    C.check(C.lib.rdfc_stem_forward(ctypes.byref(d), C.stream_ptr()))
    torch.cuda.synchronize()
    assert (out_r[..., :96].float() == 7.0).all() and (out_d[..., :160].float() == 7.0).all(), "wrote outside its slice"
    got_r, got_d = out_r[..., 96:].float().permute(0, 3, 1, 2).cpu(), out_d[..., 160:].float().permute(0, 3, 1, 2).cpu()
    for got, ref in ((got_r, ref_r), (got_d, ref_d)):
        tol = 2e-2 * float(ref.abs().max())          # bf16 output rounding (2^-9 relative) + fp32 accumulation order
        assert float((got - ref).abs().max()) <= tol


# ---------------------------------------------------------------------------------------------------------------------
# rdfc_wadain_conv_forward: EqualLinear style projection + W-AdaIN apply (model_utils.py:53-90, weighting=False)
@pytest.mark.parametrize("weighting", [False, True])
@pytest.mark.parametrize("B,H,W,C,Cd", [(2, 15, 19, 512, 512), (1, 29, 38, 768, 768), (2, 20, 28, 192, 192), (1, 9, 11, 64, 32)])
def test_fused_wadain_conv(B, H, W, C, Cd, weighting):
    from rdfc_gan_b200 import _cabi as C_
    g = torch.Generator().manual_seed(C + Cd + H)
    x, style = torch.randn(B, C, H, W, generator=g), torch.randn(B, Cd, H, W, generator=g)
    Wl = torch.randn(2 * C, Cd, generator=g) * math.sqrt(2 / Cd)
    bias = torch.cat([torch.ones(C), torch.zeros(C)]) + 0.1 * torch.randn(2 * C, generator=g)
    rb = lambda t: t.bfloat16().float()
    xb, sb = rb(x), rb(style)
    gb = torch.einsum("bdhw,nd->bnhw", sb, rb(Wl)) + bias.view(1, -1, 1, 1)
    mean = xb.mean((2, 3), keepdim=True)
    rstd = 1.0 / torch.sqrt(xb.var((2, 3), unbiased=False, keepdim=True) + 1e-5)
    ref = gb[:, :C] * (xb - mean) * rstd + gb[:, C:]
    gwbw = rb(1.0 + 0.5 * torch.randn(B, 2 * C, H, W, generator=g))        # gamma/beta_weight_layer(x), model_utils.py:84-88
    if weighting:
        ref = gwbw[:, :C] * gb[:, :C] * (xb - mean) * rstd + gwbw[:, C:] * gb[:, C:]
    tile = C_.lib.rdfc_wadain_tile(C)
    half = tile // 2
    perm = torch.cat([torch.cat([torch.arange(t * half, (t + 1) * half), C + torch.arange(t * half, (t + 1) * half)])
                      for t in range(2 * C // tile)])
    packed = Wl[perm].reshape(2 * C, 1, Cd // 8, 8).permute(1, 2, 0, 3).contiguous().to(torch.bfloat16).cuda()
    x_d = xb.permute(0, 2, 3, 1).contiguous().to(torch.bfloat16).cuda()
    s_d = sb.permute(0, 2, 3, 1).contiguous().to(torch.bfloat16).cuda()
    out = torch.empty(B, H, W, C, dtype=torch.bfloat16, device="cuda")
    b_d, m_d, r_d = bias[perm].cuda(), mean.reshape(B, C).cuda().contiguous(), rstd.reshape(B, C).cuda().contiguous()
    d = C_.WadainConvDesc()
    d.B, d.H, d.W = B, H, W
    d.style, d.x, d.out = C_.view(s_d), C_.view(x_d), C_.view(out)
    d.weight, d.bias, d.mean, d.rstd = packed.data_ptr(), b_d.data_ptr(), m_d.data_ptr(), r_d.data_ptr()
    w_d = gwbw.permute(0, 2, 3, 1).contiguous().to(torch.bfloat16).cuda()
    d.gwbw = C_.view(w_d) if weighting else C_.view(None)
    C_.check(C_.lib.rdfc_wadain_conv_forward(ctypes.byref(d), C_.stream_ptr()))
    torch.cuda.synchronize()
    got = out.float().permute(0, 3, 1, 2).cpu()
    assert float((got - ref).abs().max()) <= 2e-2 * float(ref.abs().max())


@pytest.mark.parametrize("B,H,W,C0,Cpad,with_in1", [(2, 13, 17, 40, 64, True), (1, 228, 304, 40, 64, True), (3, 9, 9, 5, 8, False)])
def test_pack_stem_input(B, H, W, C0, Cpad, with_in1):
    """rdfc_pack_stem_input: [in0 | in1 | zeros] as bf16 NHWC, bit-exact against torch's round-to-nearest-even cast."""
    from rdfc_gan_b200 import _cabi as C
    g = torch.Generator().manual_seed(C0 + H)
    in0 = torch.randn(B, C0, H, W, generator=g).cuda()
    in1 = torch.randn(B, 1, H, W, generator=g).cuda() if with_in1 else None
    out = torch.full((B, H, W, Cpad), 7.0, dtype=torch.bfloat16, device="cuda")
    C.check(C.lib.rdfc_pack_stem_input(C.ptr(in0), C0, C.ptr(in1) if with_in1 else None, C.ptr(out), Cpad, B, H, W, C.stream_ptr()))
    torch.cuda.synchronize()
    ref = torch.zeros(B, H, W, Cpad, device="cuda")
    ref[..., :C0] = in0.permute(0, 2, 3, 1)
    if with_in1:
        ref[..., C0] = in1[:, 0]
    assert torch.equal(out, ref.to(torch.bfloat16))


@pytest.mark.parametrize("shape", [(2, 64, 64, 40, 44, 3, 1, False, True), (3, 128, 128, 29, 38, 3, 1, False, True),
                                   (2, 64, 128, 41, 40, 3, 2, False, False), (1, 128, 160, 30, 52, 3, 1, False, False),
                                   (2, 192, 64, 20, 27, 3, 2, True, False), (2, 96, 192, 33, 21, 1, 2, False, False),
                                   (1, 256, 256, 19, 26, 3, 1, False, True)])
def test_tma_store_epilogue_matches_direct_stores(shape):
    """RDFC_UMMA_TMAOUT: the epilogue that stages 32-channel slabs in shared memory and writes them with cp.async.bulk.tensor
    stores (residual slabs through tensor loads) does the same arithmetic as the per-lane global stores: bit-identical outputs,
    clipped tiles, odd sizes, strided (transposed) store boxes and N = 160 / 256 tiles included; both match the torch reference."""
    from rdfc_gan_b200 import _cabi as C
    B, Cin, Cout, H, W, k, stride, transposed, with_res = shape
    g = torch.Generator().manual_seed(sum(shape[:6]) + 7)
    x = torch.randn(B, Cin, H, W, generator=g)
    w = torch.randn(*((Cin, Cout, k, k) if transposed else (Cout, Cin, k, k)), generator=g) / math.sqrt(Cin * k * k)
    scale, shift = 1 + 0.1 * torch.randn(Cout, generator=g), 0.1 * torch.randn(Cout, generator=g)
    kw = dict(stride=stride, pad=(1 if transposed else k // 2), act=2, transposed=transposed, bf16=True)
    if with_res:
        kw["residual"] = torch.randn(B, Cout, H, W, generator=g)
    outs = []
    for mode in (0, 2, 1):
        C.set_knob("RDFC_UMMA_TMAOUT", mode)
        outs.append(_run_conv(x, w, scale, shift, **kw))
    C.set_knob("RDFC_UMMA_TMAOUT", None)
    assert torch.equal(outs[0], outs[1]) and torch.equal(outs[0], outs[2])
    ref = _ref_conv(x, w, scale, shift, **kw)
    assert float((outs[1] - ref).abs().max()) <= 2e-2 * float(ref.abs().max())
