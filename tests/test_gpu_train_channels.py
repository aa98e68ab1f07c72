"""-m gpu: the training ops at the channel counts and sizes the per-op tests of test_gpu_train.py / test_gpu_train_fp32.py leave out.

* The element-wise passes of the batch-statistics BatchNorm (csrc/train.cu) have a hoisted form, taken when C / 8 divides the
  256-thread block, and a plain form: both must give the same bits.
* At the training benchmark's size (16 x 228 x 304) a reduction block of the BatchNorm kernels covers ~1 900 pixels (59 per lane)
  instead of the 64 of every smaller shape: bn_act there against fp64, three calls bit-identical (rdfc_bn_frozen_backward:
  test_gpu_frozen_bn.py::test_frozen_backward_kernel).
* Channels that strain the statistics, in one tensor: |mean| = 30 std, a constant channel, 40 channels (a partial 64-channel
  block), a channel-slice input.
* ResnetGenerator with ngf = 48 / 16 in bf16: its thin transposed convs (96 -> 48, 32 -> 16) train on the tensor cores.

Bounds are the per-op tests' own (bf16: one rounding of the output; fp32: BN_BOUND), except where a comment derives one."""
import copy
import json
import os

import numpy as np
import pytest
import torch
import torch.nn as nn

pytestmark = pytest.mark.gpu
BF = torch.bfloat16
DTYPES = pytest.mark.parametrize("dtype", [BF, torch.float32], ids=["bf16", "fp32"])
# relative L2 against fp64: test_gpu_train.py's bf16 bounds and test_gpu_train_fp32.py's BN_BOUND.  Measured on a B200 at 16 x 228 x 304
# (C = 64 and 96 alike): bf16 output / dy 1.7e-3, statistics and d gamma / d beta <= 2.3e-7; fp32 <= 2.1e-7 for every quantity.
BN_BOUNDS = {BF: dict(out=6e-3, running=1e-4, dy=2e-2, dgamma=1e-2, dbeta=1e-2, dres=2e-2),
             torch.float32: dict(out=4e-7, running=4e-7, dy=4e-7, dgamma=4e-7, dbeta=4e-7, dres=4e-7)}
SLOPE = {0: 1.0, 1: 0.0, 2: 0.2}


def _rel(a, b):
    return float((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-30))


def _cos(a, b):
    a, b = a.double().reshape(-1), b.double().reshape(-1)
    return float((a * b).sum() / (a.norm() * b.norm() + 1e-30))


def _dump(rec):
    """RDFC_DUMP_PARITY=<file>: append the measured errors"""
    path = os.environ.get("RDFC_DUMP_PARITY")
    if path:
        with open(path, "a") as f:
            f.write(json.dumps(rec) + "\n")


def _bn(Cc, gen):
    bn = nn.BatchNorm2d(Cc).cuda().train()
    with torch.no_grad():
        bn.weight.uniform_(0.5, 1.5, generator=gen)
        bn.bias.normal_(0, 0.2, generator=gen)
    return bn


def _bn_act_run(big, off, bn0, res, act, go):
    """bn_act over the channel slice big[..., off:] (+ res, act), backward with go, on a fresh copy of the BatchNorm and leaf copies
    of the inputs -> dict of the output, the gradients and the running statistics"""
    from rdfc_gan_b200.train_ops import bn_act
    bn = copy.deepcopy(bn0)
    big = big.detach().clone().requires_grad_(True)
    r = None if res is None else res.detach().clone().requires_grad_(True)
    out = bn_act(big[..., off:], bn, r, act)
    assert out.dtype == big.dtype
    out.backward(go)
    if off:
        assert float(big.grad[..., :off].abs().max()) == 0.0
    t = dict(out=out.detach(), dy=big.grad[..., off:], dgamma=bn.weight.grad, dbeta=bn.bias.grad, running_mean=bn.running_mean,
             running_var=bn.running_var)
    if r is not None:
        t["dres"] = r.grad
    return t


def _bn_act_ref(y, bn0, res, act, go, out):
    """nn.BatchNorm2d(train) + residual + activation in fp64 autograd on the same values; the activation's derivative from the sign
    of the kernel's output ``out``, as the backward takes it (a pixel within one rounding of zero would otherwise flip its mask)"""
    ref = nn.BatchNorm2d(bn0.num_features).cuda().double().train()
    ref.load_state_dict({k: v.double() if v.is_floating_point() else v for k, v in bn0.state_dict().items()})
    yr = y.detach().double().permute(0, 3, 1, 2).requires_grad_(True)
    rr = None if res is None else res.detach().double().permute(0, 3, 1, 2).requires_grad_(True)
    z = ref(yr) + (0 if rr is None else rr)
    zr = z * torch.where(out.double().permute(0, 3, 1, 2) > 0, 1.0, SLOPE[act])
    zr.backward(go.double().permute(0, 3, 1, 2))
    t = dict(out=zr.detach().permute(0, 2, 3, 1), dy=yr.grad.permute(0, 2, 3, 1), dgamma=ref.weight.grad, dbeta=ref.bias.grad,
             running_mean=ref.running_mean, running_var=ref.running_var)
    if rr is not None:
        t["dres"] = rr.grad.permute(0, 2, 3, 1)
    return t


def _errs(got, want):
    e = {k: _rel(got[k], want[k]) for k in ("out", "dy", "dres", "dgamma", "dbeta") if k in got}
    e["running"] = max(_rel(got["running_mean"], want["running_mean"]), _rel(got["running_var"], want["running_var"]))
    return e


def _bn_inputs(B, H, W, Cc, dtype, gen, off=0):
    big = (1.5 * torch.randn(B, H, W, Cc + off, device="cuda", generator=gen) + 0.3).to(dtype)
    res = torch.randn(B, H, W, Cc, device="cuda", generator=gen).to(dtype)
    go = torch.randn(B, H, W, Cc, device="cuda", generator=gen).to(dtype)
    return big, res, go


# ------------------------------------------------------------------------------------------------ hoisted and plain forms
@DTYPES
@pytest.mark.parametrize("Cc", [8, 64, 256])
def test_bn_act_hoisted_and_plain_forms_bit_identical(Cc, dtype):
    """RDFC_BN_HOIST=0 sends every channel count to the plain form of affine_act_kernel / bn_bwd_apply_kernel: bn_act's output,
    running statistics and every gradient equal the default (hoisted) form's bit for bit.  16 x 228 x 304: several grid-stride
    iterations per thread in both forms."""
    from rdfc_gan_b200 import _cabi as C
    gen = torch.Generator(device="cuda").manual_seed(Cc)
    big, res, go = _bn_inputs(16, 228, 304, Cc, dtype, gen)
    bn = _bn(Cc, gen)
    runs = []
    try:
        for hoist in (None, 0):
            C.set_knob("RDFC_BN_HOIST", hoist)
            runs.append(_bn_act_run(big, 0, bn, res, C.ACT_LEAKY02, go))
    finally:
        C.set_knob("RDFC_BN_HOIST", None)
    assert all(torch.equal(runs[0][k], runs[1][k]) for k in runs[0]), [k for k in runs[0] if not torch.equal(runs[0][k], runs[1][k])]


# ------------------------------------------------------------------------------------------------ full-size reductions
@DTYPES
@pytest.mark.parametrize("Cc", [64, 96], ids=["C64_hoisted", "C96_plain"])
def test_bn_act_full_size_against_fp64(Cc, dtype):
    """bn_act (LeakyReLU(0.2) + residual) at 16 x 228 x 304 -- ~1 900 pixels per reduction block -- against fp64 nn.BatchNorm2d:
    output, running statistics, the gradients of y, gamma, beta and the residual; three calls bit-identical."""
    from rdfc_gan_b200 import _cabi as C
    gen = torch.Generator(device="cuda").manual_seed(Cc + 1)
    big, res, go = _bn_inputs(16, 228, 304, Cc, dtype, gen)
    bn = _bn(Cc, gen)
    runs = [_bn_act_run(big, 0, bn, res, C.ACT_LEAKY02, go) for _ in range(3)]
    for r in runs[1:]:
        assert all(torch.equal(runs[0][k], r[k]) for k in r), [k for k in r if not torch.equal(runs[0][k], r[k])]
    errs = _errs(runs[0], _bn_act_ref(big, bn, res, C.ACT_LEAKY02, go, runs[0]["out"]))
    _dump({"case": f"bn_full_{Cc}_{dtype}", "errs": errs})
    bound = BN_BOUNDS[dtype]
    assert all(v <= bound[k] for k, v in errs.items()), (errs, bound)


# ------------------------------------------------------------------------------------------------ channels that strain the statistics
# Where fp32 cancels, in units u = 2^-24 (a rounding of a value v errs by at most u |v|):
# * The kernel's mean of a channel (bn_partial_kernel, bn_final_kernel) takes one rounding of size |mean| in each block (pivot +
#   sum / n), one in each of a lane's Chan folds after its first block, which is exact, and one in each of the 5 butterfly steps:
#   k_mean = ceil(nblk / 32) + 5 roundings.  A constant channel's mean is exact: every difference from the pivot is 0.
# * The output y s + (beta - mean s), s = gamma rstd, adds the roundings of mean s and of beta - mean s: a constant offset on the
#   channel of at most (k_mean + 2) u |mean| s -- 2 u |mean| s for the constant channel, where s = gamma / sqrt(eps).
# * d gamma = sum dz (y - mean) rstd takes the mean's error times rstd sum dz; the running mean its relative error, k_mean u.
# Each such term is added to the normal bound of the quantity (BN_BOUNDS) as a relative error of that channel.
# Measured on a B200 (fp32, k_mean = 24): output 1.25e-6 on channel 0 (bound 4.4e-5) and 7.8e-7 on the constant channel (3.1e-5);
# d gamma of channel 0 1.9e-6 (6.9e-5) -- above BN_BOUND, within the counted terms; every other quantity <= 1.3e-7.


@DTYPES
def test_bn_act_special_channels(dtype):
    """One 40-channel tensor (a partial 64-channel block), passed as a channel slice, with channel 0 at |mean| = 30 std and
    channel 1 constant (variance 0), against fp64 nn.BatchNorm2d, per channel group (0, 1, 2..39): output, d y, d residual, d gamma
    and the running statistics at the normal bounds plus, in fp32, the cancellation terms counted above; d beta over all channels;
    the constant channel's d gamma exactly zero."""
    from rdfc_gan_b200 import _cabi as C
    gen = torch.Generator(device="cuda").manual_seed(40)
    B, H, W, Cc, off = 4, 96, 128, 40, 32
    big, res, go = _bn_inputs(B, H, W, Cc, torch.float32, gen, off)
    big[..., off] = 30.0 + torch.randn(big.shape[:3], device="cuda", generator=gen)
    big[..., off + 1] = 0.7
    big, res, go = big.to(dtype), res.to(dtype), go.to(dtype)
    bn = _bn(Cc, gen)
    got = _bn_act_run(big, off, bn, res, C.ACT_LEAKY02, go)
    want = _bn_act_ref(big[..., off:], bn, res, C.ACT_LEAKY02, go, got["out"])
    assert float(got["dgamma"][1]) == 0.0 and float(want["dgamma"][1]) == 0.0         # x_hat of a constant channel: exactly 0

    y64 = big[..., off:].double()
    mean, var = y64.mean((0, 1, 2)), y64.var((0, 1, 2), unbiased=False)
    rstd = (var + bn.eps).rsqrt()
    ms = (mean * bn.weight.detach().double() * rstd).abs()                                   # |mean| s
    nblk = C.lib.rdfc_bn_workspace_floats(B * H * W, Cc) // (2 * Cc)
    k_mean = (nblk + 31) // 32 + 5
    u = 2.0 ** -24 if dtype == torch.float32 else 0.0                                 # bf16: within one rounding of the output
    rms = lambda t, c: float(t[..., c].double().square().mean().sqrt())
    extra = {"out": {0: (k_mean + 2) * u * float(ms[0]) / rms(want["out"], 0), 1: 2 * u * float(ms[1]) / rms(want["out"], 1)},
             "dgamma": {0: k_mean * u * float(mean[0].abs() * rstd[0] * want["dbeta"][0].abs() / want["dgamma"][0].abs())},
             "running": {0: k_mean * u}}
    b = BN_BOUNDS[dtype]
    errs, bound = {"dbeta": _rel(got["dbeta"], want["dbeta"])}, {"dbeta": b["dbeta"]}
    for name, ch in (("bigmean", slice(0, 1)), ("const", slice(1, 2)), ("others", slice(2, None))):
        for k in ("out", "dy", "dres", "dgamma", "running"):
            if k == "dgamma" and name == "const":
                continue
            if k == "running":
                e = max(_rel(got["running_mean"][ch], want["running_mean"][ch]), _rel(got["running_var"][ch], want["running_var"][ch]))
            else:
                e = _rel(got[k][..., ch], want[k][..., ch])
            errs[f"{k}_{name}"] = e
            bound[f"{k}_{name}"] = b[k] + extra.get(k, {}).get(ch.start, 0.0)
    _dump({"case": f"bn_special_{dtype}", "errs": errs, "bounds": bound, "k_mean": k_mean})
    assert all(v <= bound[k] for k, v in errs.items()), {k: (v, bound[k]) for k, v in errs.items() if v > bound[k]}


# ------------------------------------------------------------------------------------------------ ResnetGenerator, thin layers
def _module_forward(seq, x):
    """the reference composition: ResnetGenerator.model's own modules in NCHW"""
    from rdfc_gan_b200.resnet_generator import ResnetBlock
    for m in seq:
        x = x + _module_forward(m.conv_block, x) if isinstance(m, ResnetBlock) else m(x)
    return x


@pytest.mark.parametrize("ngf", [48, 16])
def test_resnet_generator_thin_layers_bf16(ngf, monkeypatch):
    """ResnetGenerator(1, 3, ngf, n_blocks=2) in bf16 train(): its last ConvTranspose2d has 48 / 16 output channels (forward on the
    tensor cores; backward with d(output) zero-padded to 64 / 32 channels), its BatchNorms 48 / 96 / 192 channels (the plain form
    of the BatchNorm kernels) for ngf = 48.  Forward and backward finite; every parameter gradient against the same modules in
    fp32 PyTorch (TF32 off) at test_resnet_generator_against_reference's bf16 noise-floor bounds (measured on a B200: min cosine
    0.982 / 0.974, median 0.989 / 0.988 for ngf = 48 / 16)."""
    from _synth import synth_state_dict
    from rdfc_gan_b200.resnet_generator import ResnetGenerator
    monkeypatch.setattr(torch.backends.cudnn, "allow_tf32", False)
    monkeypatch.setattr(torch.backends.cuda.matmul, "allow_tf32", False)
    G = ResnetGenerator(1, 3, ngf=ngf, n_blocks=2)
    G.load_state_dict(synth_state_dict(G, seed=41, recipe="scaled"))
    G = G.cuda().train()
    R = copy.deepcopy(G)
    gen = torch.Generator(device="cuda").manual_seed(9)
    x = torch.rand(2, 1, 64, 96, device="cuda", generator=gen) * 2 - 1
    probe = torch.randn(2, 3, 64, 96, device="cuda", generator=gen)
    y = G(x)
    assert torch.isfinite(y).all()
    (y * probe).sum().backward()
    assert all(p.grad is not None and torch.isfinite(p.grad).all() for p in G.parameters())
    (_module_forward(R.model, x) * probe).sum().backward()
    want = dict(R.named_parameters())
    cos = {n: _cos(p.grad, want[n].grad) for n, p in G.named_parameters() if p.numel() >= 8}
    rep = dict(min_cos=min(cos.values()), median_cos=float(np.median(list(cos.values()))))
    _dump({"case": f"resnet_thin_{ngf}", "errs": rep, "worst": sorted((c, n) for n, c in cos.items())[:4]})
    assert rep["min_cos"] >= 0.85 and rep["median_cos"] >= 0.95, (rep, sorted((c, n) for n, c in cos.items())[:6])
