"""-m gpu: the inference engines' fp32_tc contractions called directly on fp32 data across fp16's range -- rdfc_conv_forward on
RDFC_PATH_UMMA_F32X3 and rdfc_heads_forward on an fp32 buffer -- against fp64 PyTorch on the same fp32 tensors.  Both split their
input into fp16 halves x = x_hi + x_lo, and fp16 keeps 11 significant bits only between 6.1e-5 and 65504: unscaled, inputs of 1e5
overflow and the low half of inputs below ~0.1 loses bits.  The generator / ESANet goldens only see O(1) activations, so the unit
scale appears here only as the baseline row of each sweep."""
import ctypes
import math

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

X_SCALES = [1.0, 1e-3, 1e-7, 1e5]
SENTINEL = 7.0
ACTS = {0: lambda v: v, 1: F.relu, 2: lambda v: F.leaky_relu(v, 0.2), 3: torch.tanh, 4: torch.sigmoid}

# the conv forms the generator engine and ESANet issue on the fp32_tc path:
# name: (B, Cin, Cout, H, W, k, stride, transposed, crop (Ho, Wo) of a transposed conv, residual, act)
FORMS = {
    "k3s1_64_res_relu": (2, 64, 64, 29, 38, 3, 1, False, None, True, 1),
    "k3s2_64_128": (2, 64, 128, 29, 38, 3, 2, False, None, False, 2),
    "k1s2_64_128": (2, 64, 128, 29, 38, 1, 2, False, None, False, 0),
    "k1s1_192_384": (1, 192, 384, 15, 19, 1, 1, False, None, False, 1),
    "convT_512_256_odd": (1, 512, 256, 8, 10, 3, 2, True, (15, 19), False, 2),
    "k3s1_256_160": (1, 256, 160, 15, 19, 3, 1, False, None, False, 1),
    "k3s1_512_512_res": (1, 512, 512, 8, 10, 3, 1, False, None, True, 0),
    "k3s1_128_40": (2, 128, 40, 29, 38, 3, 1, False, None, False, 0),
    "k3s1_64_res_full": (4, 64, 64, 228, 304, 3, 1, False, None, True, 1),
}


def _rel(a, b):
    return float((a.double() - b.double()).norm() / b.double().norm())


def _ws_bytes(npix, C):
    """rdfc_conv_forward / rdfc_heads_forward workspace for an fp32 input: the [hi | lo] split (4 bytes per element) + 16 bytes for
    the split's scale factor"""
    return npix * C * 4 + 16


def _workspace(nbytes):
    return torch.empty(nbytes, dtype=torch.uint8, device="cuda")


def _out_hw(form):
    B, Cin, Cout, H, W, k, s, tr, crop, res, act = form
    if tr:
        return crop
    return (H + 2 * ((k - 1) // 2) - k) // s + 1, (W + 2 * ((k - 1) // 2) - k) // s + 1


def _conv_inputs(form, x_scale, w_scale, gen):
    """x: a channel slice [16, 16 + Cin) of a wider fp32 NHWC tensor; w (Cout, Cin, k, k) (ConvTranspose: (Cin, Cout, k, k)) of
    N(0, 1/K) times w_scale; folded-BatchNorm-like (scale, shift) and a residual at the output's magnitude"""
    B, Cin, Cout, H, W, k, s, tr, crop, res, act = form
    K = Cin * k * k
    xw = torch.randn(B, H, W, Cin + 32, device="cuda", generator=gen) * x_scale
    x = xw[..., 16:16 + Cin]
    w = torch.randn(*((Cin, Cout, k, k) if tr else (Cout, Cin, k, k)), device="cuda", generator=gen) * (w_scale / math.sqrt(K))
    out_mag = x_scale * w_scale
    scale = torch.rand(Cout, device="cuda", generator=gen) + 0.5
    shift = torch.randn(Cout, device="cuda", generator=gen) * (0.1 * out_mag)
    Ho, Wo = _out_hw(form)
    r = torch.randn(B, Ho, Wo, Cout, device="cuda", generator=gen) * out_mag if res else None
    return xw, x, w, scale, shift, r


def _conv_x3(form, xw, w, scale, shift, r, act=None, workspace=None):
    """rdfc_conv_forward on RDFC_PATH_UMMA_F32X3 with the engines' weight packing; output channels [8, 8 + Cout) of a wider fp32 NHWC
    tensor whose other channels hold a sentinel.  -> (B, Ho, Wo, Cout) fp32"""
    from rdfc_gan_b200 import _cabi as C
    from rdfc_gan_b200.engine import pack_weight_x3
    B, Cin, Cout, H, W, k, s, tr, crop, res, act0 = form
    act = act0 if act is None else act
    Ho, Wo = _out_hw(form)
    wg = w.permute(1, 0, 2, 3) if tr else w
    packed, sc = pack_weight_x3(wg, scale)
    out = torch.full((B, Ho, Wo, Cout + 24), SENTINEL, device="cuda")
    ws = _workspace(_ws_bytes(B * H * W, Cin)) if workspace is None else workspace
    d = C.ConvDesc()
    d.B, d.Hi, d.Wi, d.Ho, d.Wo = B, H, W, Ho, Wo
    d.kh = d.kw = k
    d.stride, d.pad, d.transposed, d.act = s, (k - 1) // 2, int(tr), act
    d.path = C.PATH_UMMA_F32X3
    d.inp, d.in2, d.out = C.view(xw, Cin, 16), C.view(None), C.view(out, Cout, 8)
    d.residual = C.view(r)
    d.weight, d.scale, d.shift = packed.data_ptr(), sc.data_ptr(), shift.data_ptr()
    d.workspace, d.workspace_bytes = ws.data_ptr(), ws.numel()
    C.check(C.lib.rdfc_conv_forward(ctypes.byref(d), C.stream_ptr()))
    torch.cuda.synchronize()
    assert (out[..., :8] == SENTINEL).all() and (out[..., 8 + Cout:] == SENTINEL).all(), "wrote outside its channel slice"
    return out[..., 8:8 + Cout]


def _conv_ref(form, x, w, scale, shift, r):
    B, Cin, Cout, H, W, k, s, tr, crop, res, act = form
    xd = x.double().permute(0, 3, 1, 2)
    if tr:
        y = F.conv_transpose2d(xd, w.double(), None, stride=2, padding=1, output_padding=1)[:, :, :crop[0], :crop[1]]
    else:
        y = F.conv2d(xd, w.double(), None, s, (k - 1) // 2)
    y = y * scale.double().view(1, -1, 1, 1) + shift.double().view(1, -1, 1, 1)
    if r is not None:
        y = y + r.double().permute(0, 3, 1, 2)
    return ACTS[act](y).permute(0, 2, 3, 1)


@pytest.mark.parametrize("w_scale", [1.0, 1e-3])
@pytest.mark.parametrize("x_scale", X_SCALES)
@pytest.mark.parametrize("form", list(FORMS))
def test_x3_conv_against_fp64(form, x_scale, w_scale):
    """Every fp32_tc conv form of the engines at input magnitudes 1 .. 1e-7 and 1e5 and filters of N(0, 1/K) and 1e-3 of that:
    finite, and within relative L2 1e-8 * Cin * k^2 of fp64 (test_gpu_train_fp32._conv_bound's rule for this contraction: the
    tensor cores' fp32 accumulation costs ~5e-9 per unit of K, once the split itself keeps 22 bits at every magnitude)."""
    f = FORMS[form]
    gen = torch.Generator(device="cuda").manual_seed(list(FORMS).index(form) * 101 + X_SCALES.index(x_scale) * 7 + int(w_scale == 1.0))
    xw, x, w, scale, shift, r = _conv_inputs(f, x_scale, w_scale, gen)
    y = _conv_x3(f, xw, w, scale, shift, r)
    assert torch.isfinite(y).all(), "non-finite outputs"
    err = _rel(y, _conv_ref(f, x, w, scale, shift, r))
    bound = 1e-8 * f[1] * f[5] ** 2
    assert err <= bound, (err, bound)


@pytest.mark.parametrize("act", [0, 1, 2])
def test_x3_conv_power_of_two_equivariant(act):
    """With no shift, scaling the input and the residual by 2^j scales the output by exactly 2^j: the split is taken of the input
    scaled by a power of two of its own, and the inverse is applied exactly -- bit for bit, from 2^-40 to 2^40."""
    f = FORMS["k3s1_64_res_relu"]
    gen = torch.Generator(device="cuda").manual_seed(77 + act)
    xw, x, w, scale, shift, r = _conv_inputs(f, 1.0, 1.0, gen)
    zero = torch.zeros_like(shift)
    y = _conv_x3(f, xw, w, scale, zero, r, act=act)
    assert torch.isfinite(y).all()
    for j in (-40, -12, 12, 40):
        p = 2.0 ** j
        yj = _conv_x3(f, xw * p, w, scale, zero, r * p, act=act)
        assert torch.equal(yj, y * p), (j, float((yj - y * p).abs().max() / (y * p).abs().max()))


# fused decode heads: (buffer channels, [(output columns, [(conv channel, count, buffer channel)], activation at unit scale)])
# mapped as engine._plan_heads maps the generator's *_dec0 heads onto its head buffers
HEAD_SETS = {
    2: (160, [(1, [(0, 64, 0), (64, 64, 96)], 3), (1, [(0, 32, 64), (32, 64, 96)], 4)]),
    10: (224, [(1, [(0, 64, 0), (64, 64, 160)], 3), (1, [(0, 32, 64), (32, 64, 160)], 4), (8, [(0, 64, 96), (64, 64, 160)], 0)]),
    16: (224, [(1, [(0, 64, 0), (64, 64, 160)], 4), (1, [(0, 32, 64), (32, 64, 160)], 3), (14, [(0, 96, 64), (96, 64, 160)], 0)]),
}


def _heads_case(ncols, H, W, x_scale, gen):
    B = 2
    Ctot, cols = HEAD_SETS[ncols]
    x = torch.randn(B, H, W, Ctot, device="cuda", generator=gen) * x_scale
    convs = []
    for n, segs, act in cols:
        cin = sum(c for _, c, _ in segs)
        w = torch.randn(n, cin, 3, 3, device="cuda", generator=gen) * 0.02        # the init recipe's N(0, 0.02^2)
        b = torch.randn(n, device="cuda", generator=gen) * (0.1 * x_scale)
        convs.append((w, b, segs, act if x_scale == 1.0 else 0))
    return B, Ctot, x, convs


def _heads_x3(B, H, W, Ctot, x, convs, planes, workspace=None):
    """rdfc_heads_forward on the fp32 buffer x with the packing of engine._plan_heads; column q -> planes[:, q] (a (B, nplanes, H, W)
    tensor, so each plane's batch stride is nplanes * H * W)"""
    from rdfc_gan_b200 import _cabi as C
    from rdfc_gan_b200.engine import pack_weight
    nc = sum(w.shape[0] for w, _, _, _ in convs)
    NP = (9 * nc + 15) // 16 * 16
    wq = torch.zeros(nc, Ctot, 3, 3, device="cuda")
    q = 0
    for w, _, segs, _ in convs:
        for s0, n, d0 in segs:
            wq[q:q + w.shape[0], d0:d0 + n] = w[:, s0:s0 + n]
        q += w.shape[0]
    fused = torch.zeros(NP, Ctot, 1, 1, device="cuda")
    fused[:9 * nc, :, 0, 0] = wq.permute(2, 3, 0, 1).reshape(9 * nc, Ctot)
    packed = pack_weight(fused, True, x3=True)
    shift = torch.cat([b for _, b, _, _ in convs] + [torch.zeros(NP - nc, device="cuda")]).contiguous()
    ws = _workspace(_ws_bytes(B * H * W, Ctot)) if workspace is None else workspace
    d = C.HeadsDesc()
    d.B, d.H, d.W = B, H, W
    d.inp = C.view(x)
    d.weight, d.shift = packed.data_ptr(), shift.data_ptr()
    d.workspace, d.workspace_bytes = ws.data_ptr(), ws.numel()
    q = 0
    for w, _, _, act in convs:
        for _ in range(w.shape[0]):
            d.act[q] = act
            d.out[q] = planes.data_ptr() + 4 * q * H * W
            d.out_bstride[q] = planes.shape[1] * H * W
            q += 1
    d.ncols = q
    return C.lib.rdfc_heads_forward(ctypes.byref(d), C.stream_ptr())


@pytest.mark.parametrize("x_scale", X_SCALES)
@pytest.mark.parametrize("hw", [(15, 17), (29, 38), (57, 76)])
@pytest.mark.parametrize("ncols", [2, 10, 16])
def test_x3_heads_against_fp64(ncols, hw, x_scale):
    """The fused *_dec0 heads on an fp32 head buffer (160 / 224 channels, segments as engine._plan_heads maps them), B = 2 into planes
    of a (B, ncols, H, W) tensor, sizes that are not multiples of the 14 x 14 region step: every column within relative L2
    1e-8 * 9 * C of fp64.  Tanh / sigmoid at unit scale; linear columns at the other magnitudes."""
    from rdfc_gan_b200 import _cabi as C
    H, W = hw
    gen = torch.Generator(device="cuda").manual_seed(ncols * 1000 + H + X_SCALES.index(x_scale))
    B, Ctot, x, convs = _heads_case(ncols, H, W, x_scale, gen)
    planes = torch.full((B, ncols, H, W), float("nan"), device="cuda")
    C.check(_heads_x3(B, H, W, Ctot, x, convs, planes))
    torch.cuda.synchronize()
    assert torch.isfinite(planes).all(), "non-finite or unwritten outputs"
    bound = 1e-8 * 9 * Ctot
    xd = x.double().permute(0, 3, 1, 2)
    q = 0
    for w, b, segs, act in convs:
        xin = torch.cat([xd[:, d0:d0 + n] for _, n, d0 in segs], 1)
        want = ACTS[act](F.conv2d(xin, w.double(), b.double(), padding=1))
        for i in range(w.shape[0]):
            err = _rel(planes[:, q], want[:, i])
            assert err <= bound, (q, err, bound)
            q += 1


def test_x3_workspace_rule():
    """The fp32 input's workspace holds the [hi | lo] split and, in a 16-byte tail, the split's scale factor: B*H*W*C*4 + 16 bytes,
    128-byte aligned.  Too small (the split alone), misaligned and NULL workspaces are refused before any launch, naming the size."""
    from rdfc_gan_b200 import _cabi as C
    gen = torch.Generator(device="cuda").manual_seed(3)
    f = FORMS["k3s1_64_res_relu"]
    B, Cin, H, W = f[0], f[1], f[3], f[4]
    xw, x, w, scale, shift, r = _conv_inputs(f, 1.0, 1.0, gen)
    need = _ws_bytes(B * H * W, Cin)
    Bh, Ctot, xh, convs = _heads_case(2, 15, 17, 1.0, gen)
    need_h = _ws_bytes(Bh * 15 * 17, Ctot)
    planes = torch.full((Bh, 2, 15, 17), float("nan"), device="cuda")
    big, big_h = _workspace(need + 256), _workspace(need_h + 256)

    class _At:                       # a workspace tensor stand-in at an offset / of a size / NULL
        def __init__(self, t, off, n):
            self.t, self.off, self.n = t, off, n

        def data_ptr(self):
            return None if self.t is None else self.t.data_ptr() + self.off

        def numel(self):
            return self.n

    for ws in (_At(big, 0, need - 16), _At(big, 64, need), _At(None, 0, need)):
        n0 = C.launch_count()
        with pytest.raises(RuntimeError, match=str(need)):
            _conv_x3(f, xw, w, scale, shift, r, workspace=ws)
        assert C.launch_count() == n0
    for ws in (_At(big_h, 0, need_h - 16), _At(big_h, 64, need_h), _At(None, 0, need_h)):
        n0 = C.launch_count()
        assert _heads_x3(Bh, 15, 17, Ctot, xh, convs, planes, workspace=ws) == -1
        assert str(need_h).encode() in C.lib.rdfc_last_error()
        assert C.launch_count() == n0
    assert torch.isnan(planes).all()
    # exactly the required size, 128-byte aligned, is accepted
    _conv_x3(f, xw, w, scale, shift, r, workspace=_At(big, 128, need))
    C.check(_heads_x3(Bh, 15, 17, Ctot, xh, convs, planes, workspace=_At(big_h, 128, need_h)))
    torch.cuda.synchronize()
    assert torch.isfinite(planes).all()
