"""Frozen BatchNorm inside a train()-mode generator: a BatchNorm2d in eval() mode normalises with its running statistics and leaves
them alone, as in PyTorch.  train_ops.conv_bn_act_frozen (the BatchNorm folded into the tcgen05 conv's epilogue, backward through
rdfc_bn_frozen_backward) per op against fp64 autograd, the kernel against torch, the generators against fp32 / bf16-emulated
compositions and against the eval-mode engine, the dispatch, determinism and a training step.  The stated bounds are twice what
was measured on a B200 (DESIGN.md section 7)."""
import ctypes
import math
import os
import re
import subprocess

import numpy as np
import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
gpu = pytest.mark.gpu
BF = torch.bfloat16


def _rel(a, b):
    return float((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-30))


def _cos(a, b):
    a, b = a.double().reshape(-1), b.double().reshape(-1)
    return float((a * b).sum() / (a.norm() * b.norm() + 1e-30))


def _dump(rec):
    """RDFC_DUMP_PARITY=<file>: append the measured errors (the bounds below are twice the measured values)."""
    path = os.environ.get("RDFC_DUMP_PARITY")
    if path:
        import json
        with open(path, "a") as f:
            f.write(json.dumps(rec) + "\n")


def _freeze(module, every=1):
    """eval() on every ``every``-th BatchNorm2d of ``module`` (the usual fine-tuning recipe); -> the frozen modules"""
    bns = [m for m in module.modules() if isinstance(m, nn.BatchNorm2d)]
    for m in bns[::every]:
        m.eval()
    return bns[::every]


def _buffers(mods):
    return [(m.running_mean.clone(), m.running_var.clone(), m.num_batches_tracked.clone()) for m in mods]


def _same_buffers(mods, before):
    return all(torch.equal(m.running_mean, a) and torch.equal(m.running_var, b) and torch.equal(m.num_batches_tracked, c)
               for m, (a, b, c) in zip(mods, before))


# ------------------------------------------------------------------------------------------------ host side, no GPU
def test_frozen_backward_exported_and_validated():
    from rdfc_gan_b200 import _cabi as C
    nm = subprocess.run(["nm", "-D", "--defined-only", C.LIB_PATH], capture_output=True, text=True, check=True).stdout
    hdr = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "rdfc_b200.h")).read(), flags=re.S)
    name = "rdfc_bn_frozen_backward"
    assert re.search(rf"\b{name}\s*\(", hdr) and name in C.EXPORTS and re.search(rf" T {name}\b", nm)
    assert C.lib.rdfc_abi_version() == 2
    fake = 1 << 20                                              # never dereferenced: every case fails before a launch
    n0 = C.launch_count()
    f = ctypes.c_void_p(fake)

    def fails(rc, text):
        assert rc != 0
        assert text in C.lib.rdfc_last_error().decode(), C.lib.rdfc_last_error()

    def call(dout, out, act, dz, npix=64):
        r = lambda v: None if v is None else ctypes.byref(v)
        return C.lib.rdfc_bn_frozen_backward(r(dout), r(out), act, r(dz), f, f, npix, None)
    V = lambda dt, Cc, off=0, stride=None: C.View(fake + off, dt, Cc, stride or Cc, 0)
    fails(call(V(C.BF16, 64), V(C.F32, 64), C.ACT_RELU, V(C.BF16, 64)), "one dtype")
    fails(call(V(C.F32, 64), V(C.F32, 64), C.ACT_RELU, V(C.BF16, 64)), "one dtype")
    fails(call(V(C.BF16, 60), V(C.BF16, 60), C.ACT_RELU, V(C.BF16, 60)), "multiples of 8")
    fails(call(V(C.BF16, 64), V(C.BF16, 64, off=8), C.ACT_LEAKY02, V(C.BF16, 64)), "16-byte aligned")
    fails(call(V(C.F32, 64, stride=66), None, C.ACT_NONE, None), "16-byte aligned")
    fails(call(V(C.BF16, 64), V(C.BF16, 64), 7, V(C.BF16, 64)), "none / ReLU")
    fails(call(V(C.BF16, 64), V(C.BF16, 64), C.ACT_RELU, None), "needs a dz")
    fails(call(V(C.BF16, 64), None, C.ACT_NONE, None, npix=0), "bad argument")
    # the split conv now takes an fp32 residual of Cout channels: validation gets past it (to the missing scale vector) ...
    d = C.ConvDesc()
    d.B, d.Hi, d.Wi, d.Ho, d.Wo, d.kh, d.kw, d.stride, d.pad = 1, 8, 8, 8, 8, 3, 3, 1, 1
    d.path = C.PATH_UMMA_F32X3
    d.inp, d.out, d.residual = C.View(fake, C.F16, 128, 128, 0), C.View(fake, C.F32, 64, 64, 0), C.View(fake, C.F32, 64, 96, 0)
    d.weight, d.scale = fake, None
    fails(C.lib.rdfc_conv_forward_split(ctypes.byref(d), None), "inverse scale")
    # ... and still refuses a residual of another dtype, channel count or alignment, and a second source
    d.scale = fake
    for bad in (C.View(fake, C.BF16, 64, 64, 0), C.View(fake, C.F32, 32, 64, 0), C.View(fake + 4, C.F32, 64, 64, 0)):
        d.residual = bad
        fails(C.lib.rdfc_conv_forward_split(ctypes.byref(d), None), "residual")
    d.residual, d.in2 = C.View(None, 0, 0, 0, 0), C.View(fake, C.F16, 128, 128, 0)
    fails(C.lib.rdfc_conv_forward_split(ctypes.byref(d), None), "second source")
    assert C.launch_count() == n0, "an invalid call launched a kernel"


def test_frozen_rule():
    from rdfc_gan_b200.train_ops import bn_frozen
    bn = nn.BatchNorm2d(8)
    assert not bn_frozen(bn)
    assert bn_frozen(bn.eval())
    assert not bn_frozen(nn.BatchNorm2d(8, track_running_stats=False).eval())       # no running statistics: batch statistics


# ------------------------------------------------------------------------------------------------ per op, GPU
# B, Cin, Cout, H, W, k, stride, transposed
FORMS = [(2, 64, 64, 20, 28, 3, 1, False), (2, 64, 128, 21, 27, 3, 2, False), (1, 96, 64, 17, 23, 1, 1, False),
         (2, 64, 128, 14, 15, 1, 2, False), (2, 128, 64, 10, 13, 3, 2, True),
         # Cout % 32 != 0: dz reaches the data gradient's kernel zero-padded to 32-channel multiples
         (2, 64, 24, 20, 28, 3, 1, False), (2, 96, 48, 10, 13, 3, 2, True)]
ACTS = {0: "none", 1: "relu", 2: "leaky02"}
# Relative L2 against fp64 autograd.  bf16: one bf16 rounding of the output and of dz (measured <= 1.7e-3 output, 2.4e-3 dx,
# <= 3.5e-4 elsewhere).  fp32_tc: the split-operand contraction (measured <= 3.0e-6 output / dx, <= 2.9e-7 dW / d gamma / d beta).
OP_BOUND = {torch.bfloat16: dict(out=3.5e-3, dx=5e-3, dw=7e-4, dgamma=8e-4, dbeta=8e-4, dres=7e-4),
            torch.float32: dict(out=6e-6, dx=6e-6, dw=5e-7, dgamma=6e-7, dbeta=3e-7, dres=1.3e-8)}
# running_mean ~ 30 x sqrt(running_var): the fold's s y + t cancels in the forward (fp32_tc output measured 1.7e-5), and d gamma =
# rstd (<W, G> - rm sum dz) in the backward (measured 1.1e-5 fp32_tc; 4.9e-6 bf16, where sum dz is summed from the stored bf16 dz)
BIGMEAN_BOUND = {torch.bfloat16: dict(dgamma=1e-5), torch.float32: dict(out=3.5e-5, dgamma=2.2e-5)}


def _bn_module(Cc, gen, rm=None, rv=None):
    bn = nn.BatchNorm2d(Cc).cuda()
    with torch.no_grad():
        bn.weight.uniform_(0.5, 1.5, generator=gen)
        bn.bias.normal_(0, 0.2, generator=gen)
        bn.running_mean.copy_(torch.randn(Cc, device="cuda", generator=gen) * 0.3 if rm is None else rm)
        bn.running_var.copy_(torch.rand(Cc, device="cuda", generator=gen) + 0.5 if rv is None else rv)
        bn.num_batches_tracked.fill_(7)
    return bn.eval()


def _op_case(form, dtype, act, with_res, gen, sliced=False, big_mean=False, train_w=True, train_gb=True):
    """conv_bn_act_frozen against fp64 autograd of conv -> F.batch_norm(training=False) -> (+ res) -> act on the same operands
    (bf16-representable in the bf16 mode). -> dict of relative errors"""
    from rdfc_gan_b200.train_ops import conv_bn_act_frozen
    B, Cin, Cout, H, W, k, s, tr = form
    xs = torch.randn(B, H, W, Cin + (32 if sliced else 0), device="cuda", generator=gen)
    if big_mean:
        xs = 8 + 0.25 * xs
    big = xs.to(dtype).requires_grad_(True)
    x = big[..., 32:] if sliced else big                        # a channel slice: passed to the kernels as a view
    wshape = (Cin, Cout, k, k) if tr else (Cout, Cin, k, k)
    w = torch.randn(*wshape, device="cuda", generator=gen) / math.sqrt(Cin * k * k)
    if big_mean:
        w = w + 1.0 / (Cin * k * k)
    w = w.to(BF).float() if dtype == BF else w
    w.requires_grad_(train_w)
    xr = x.detach().double().permute(0, 3, 1, 2).requires_grad_(True)
    wr = w.detach().double().requires_grad_(train_w)
    conv = (lambda a, b: F.conv_transpose2d(a, b, stride=2, padding=1, output_padding=1)) if tr else \
        (lambda a, b: F.conv2d(a, b, stride=s, padding=(k - 1) // 2))
    rm = rv = None
    if big_mean:                                                # running statistics of the data: |rm| >> sqrt(rv)
        with torch.no_grad():
            y0 = conv(xr, wr)
            rm, rv = y0.mean((0, 2, 3)).float(), y0.var((0, 2, 3)).float()
    bn = _bn_module(Cout, gen, rm, rv)
    bn.weight.requires_grad_(train_gb)
    bn.bias.requires_grad_(train_gb)
    ref = nn.BatchNorm2d(Cout).cuda().double().eval()
    ref.load_state_dict({kk: v.double() if v.is_floating_point() else v for kk, v in bn.state_dict().items()})
    ref.weight.requires_grad_(train_gb)
    ref.bias.requires_grad_(train_gb)
    before = _buffers([bn])
    yr = conv(xr, wr)
    res = rr = None
    if with_res:
        res = torch.randn(B, yr.shape[2], yr.shape[3], Cout, device="cuda", generator=gen).to(dtype).requires_grad_(True)
        rr = res.detach().double().permute(0, 3, 1, 2).requires_grad_(True)
    out = conv_bn_act_frozen(x, w, bn, k, s, tr, res, act)
    assert out.dtype == dtype and tuple(out.shape) == (B, yr.shape[2], yr.shape[3], Cout)
    z = ref(yr) + (rr if with_res else 0)
    # the activation's derivative from the sign of the kernel's output, as the backward takes it: a pixel within one rounding of
    # zero would otherwise flip its mask and dominate the fp32_tc gradient errors
    zr = z * torch.where(out.detach().double().permute(0, 3, 1, 2) > 0, 1.0, {0: 1.0, 1: 0.0, 2: 0.2}[act])
    go = torch.randn(out.shape, device="cuda", generator=gen).to(dtype)
    if sliced:                                                  # the gradient arrives as a channel slice of a concatenation
        other = torch.zeros(B, out.shape[1], out.shape[2], 16, device="cuda", dtype=dtype)
        torch.cat([other, out], 3).backward(torch.cat([torch.randn_like(other), go], 3))
    else:
        out.backward(go)
    zr.backward(go.double().permute(0, 3, 1, 2))
    errs = {"out": _rel(out.detach().permute(0, 3, 1, 2), zr.detach()),
            "dx": _rel((big.grad[..., 32:] if sliced else big.grad).permute(0, 3, 1, 2), xr.grad)}
    if sliced:
        assert float(big.grad[..., :32].abs().max()) == 0.0
    if train_w:
        errs["dw"] = _rel(w.grad, wr.grad)
    else:
        assert w.grad is None
    if train_gb:
        errs["dgamma"], errs["dbeta"] = _rel(bn.weight.grad, ref.weight.grad), _rel(bn.bias.grad, ref.bias.grad)
    else:
        assert bn.weight.grad is None and bn.bias.grad is None
    if with_res:
        errs["dres"] = _rel(res.grad.permute(0, 3, 1, 2), rr.grad)
    assert _same_buffers([bn], before), "a frozen BatchNorm's buffers changed"
    return errs


@gpu
@pytest.mark.parametrize("dtype", [BF, torch.float32], ids=["bf16", "fp32_tc"])
@pytest.mark.parametrize("form", FORMS, ids=lambda f: f"{f[5]}x{f[5]}s{f[6]}{'T' if f[7] else ''}" + (f"o{f[2]}" if f[2] % 32 else ""))
def test_conv_bn_act_frozen_against_fp64(form, dtype):
    """Every conv form x every activation x residual on / off: output and the gradients of x, W, gamma, beta and the residual;
    the BatchNorm's running_mean / running_var / num_batches_tracked bit-identical afterwards."""
    gen = torch.Generator(device="cuda").manual_seed(sum(form[:7]) + 11)
    worst = {}
    for act in ACTS:
        for with_res in (False, True):
            for kk, v in _op_case(form, dtype, act, with_res, gen).items():
                worst[kk] = max(worst.get(kk, 0.0), v)
    _dump({"case": f"op_{form}_{dtype}", "errs": worst})
    bound = OP_BOUND[dtype]
    assert all(v <= bound[kk] for kk, v in worst.items()), (worst, bound)


@gpu
@pytest.mark.parametrize("dtype", [BF, torch.float32], ids=["bf16", "fp32_tc"])
def test_conv_bn_act_frozen_special_cases(dtype):
    """A channel-slice input and gradient; running_mean >> sqrt(running_var) (the cancellation in <W, G> - rm sum dz of d gamma);
    gamma / beta with requires_grad=False; W frozen while gamma trains."""
    gen = torch.Generator(device="cuda").manual_seed(3)
    bound = OP_BOUND[dtype]
    rep = {}
    for form in (FORMS[0], FORMS[4]):
        rep[f"slice{form[5]}{form[7]}"] = _op_case(form, dtype, 1, True, gen, sliced=True)
    for form in (FORMS[0], FORMS[2], FORMS[4]):               # no activation: an output within rounding of zero flips its mask
        rep[f"bigmean{form[5]}{form[7]}"] = _op_case(form, dtype, 0, True, gen, big_mean=True)
    rep["frozen_gb"] = _op_case(FORMS[1], dtype, 1, True, gen, train_gb=False)
    rep["frozen_w"] = _op_case(FORMS[3], dtype, 0, True, gen, train_w=False)
    _dump({"case": f"op_special_{dtype}", "errs": rep})
    for name, errs in rep.items():
        b = dict(bound, **BIGMEAN_BOUND[dtype]) if name.startswith("bigmean") else bound
        assert all(v <= b[kk] for kk, v in errs.items()), (name, errs, b)


@gpu
@pytest.mark.parametrize("dtype", [BF, torch.float32], ids=["bf16", "fp32"])
def test_frozen_backward_kernel(dtype):
    """rdfc_bn_frozen_backward against torch: dz = dout act'(out) and sum dz over channel-slice views, for every activation; with
    ACT_NONE and no dz only the sum; three calls bit-identical.  Also at the training benchmark's 16 x 228 x 304, where one
    reduction block sums ~1 900 pixels instead of 64, with 64 and 96 channels (measured sum dz <= 2.1e-7 there)."""
    from rdfc_gan_b200 import _cabi as C
    gen = torch.Generator(device="cuda").manual_seed(1)
    for B, H, W, Cc in ((3, 37, 45, 96), (16, 228, 304, 64), (16, 228, 304, 96)):
        _frozen_backward_case(C, B, H, W, Cc, dtype, gen)


def _frozen_backward_case(C, B, H, W, Cc, dtype, gen):
    dout = torch.randn(B, H, W, Cc + 32, device="cuda", generator=gen).to(dtype)[..., 32:]
    outb = torch.randn(B, H, W, Cc + 16, device="cuda", generator=gen).to(dtype)[..., :Cc]
    npix = B * H * W
    for act in ACTS:
        slope = {0: 1.0, 1: 0.0, 2: 0.2}[act]
        dz_want = (dout.float() * torch.where(outb.float() > 0, 1.0, slope)).to(dtype)
        sum_want = dz_want.double().sum((0, 1, 2))
        runs = []
        for _ in range(3):
            dz = torch.full((B, H, W, Cc + 8), float("nan"), device="cuda", dtype=dtype)[..., 8:] if act else None
            ws = torch.empty(C.lib.rdfc_bn_workspace_floats(npix, Cc), device="cuda")
            s = torch.empty(Cc, device="cuda")
            vg, vo, vz = C.view(dout), C.view(outb), C.view(dz)
            C.check(C.lib.rdfc_bn_frozen_backward(ctypes.byref(vg), ctypes.byref(vo) if act else None, act,
                                                  ctypes.byref(vz) if act else None, C.ptr(ws), C.ptr(s), npix, C.stream_ptr()))
            runs.append((None if dz is None else dz.clone(), s.clone()))
        if act:
            assert torch.equal(runs[0][0], dz_want)
        _dump({"case": f"frozen_backward_{B}x{H}x{W}x{Cc}_{act}_{dtype}", "errs": {"sum_dz": _rel(runs[0][1], sum_want)}})
        assert _rel(runs[0][1], sum_want) <= 1e-6, _rel(runs[0][1], sum_want)
        assert all(torch.equal(r[1], runs[0][1]) and (r[0] is None or torch.equal(r[0], runs[0][0])) for r in runs)


# ------------------------------------------------------------------------------------------------ generators, GPU
def _frozen_fp32_op():
    """conv_bn_act_frozen restated on fp32 PyTorch ops (TF32 off by the caller): conv -> F.batch_norm(training=False) -> + res -> act"""
    from _fp32_ops import fp32_torch_ops
    from rdfc_gan_b200 import _cabi as C
    conv, _ = fp32_torch_ops()

    def op(x, weight, bn, k=3, stride=1, transposed=False, residual=None, act=C.ACT_NONE):
        y = conv(x, weight, k, stride, transposed).permute(0, 3, 1, 2)
        z = F.batch_norm(y, bn.running_mean, bn.running_var, bn.weight, bn.bias, False, 0.0, bn.eps).permute(0, 2, 3, 1)
        if residual is not None:
            z = z + residual
        return {C.ACT_NONE: z, C.ACT_RELU: F.relu(z), C.ACT_LEAKY02: F.leaky_relu(z, 0.2)}[act]
    return op


def _frozen_bf16_op():
    """the same, rounding as the kernels do: bf16 operands, fp32 conv + BatchNorm + residual + activation, one bf16 rounding"""
    from rdfc_gan_b200 import _cabi as C

    def op(x, weight, bn, k=3, stride=1, transposed=False, residual=None, act=C.ACT_NONE):
        xn, w = x.float().permute(0, 3, 1, 2), weight.to(BF).float()
        y = (F.conv_transpose2d(xn, w, stride=2, padding=1, output_padding=1) if transposed else
             F.conv2d(xn, w, stride=stride, padding=(k - 1) // 2))
        z = F.batch_norm(y, bn.running_mean, bn.running_var, bn.weight, bn.bias, False, 0.0, bn.eps).permute(0, 2, 3, 1)
        if residual is not None:
            z = z + residual.float()
        return {C.ACT_NONE: z, C.ACT_RELU: F.relu(z), C.ACT_LEAKY02: F.leaky_relu(z, 0.2)}[act].to(BF)
    return op


def _generator(kind, seed=33):
    from make_train_golden import _NL
    from _synth import synth_state_dict
    from rdfc_gan_b200.generator import DCVGANGenerator, RDFGenerator
    if kind == "rdf":
        G = RDFGenerator(pretrained_on_imagenet=False, use_nlspn_refine=True, nlspn_configs=_NL)
    else:
        G = DCVGANGenerator(None, pretrained_on_imagenet=False, semantic_channels_in=3, use_nlpsn_refine=True, nlspn_configs=_NL)
    G.load_state_dict(synth_state_dict(G, seed=seed, recipe="scaled", nlspn_stress=True))
    return G.cuda().train()


def _run_generator(G, inputs, probes):
    out = dict(zip(G._OUTPUTS, _as_tuple(G, G(*inputs))))
    sum((out[k] * R).sum() for k, R in zip(G._OUTPUTS, probes)).backward()
    return {k: v.detach() for k, v in out.items()}, {n: p.grad.detach().clone() for n, p in G.named_parameters() if p.grad is not None}


def _gen_inputs(kind, B, H, W, seed=33):
    from _synth import synth_inputs
    rgb, normal, raw = (t.cuda() for t in synth_inputs(B, H, W, seed=seed))
    gen = torch.Generator(device="cuda").manual_seed(5)
    probes = [torch.randn(B, 1, H, W, device="cuda", generator=gen) for _ in range(5)]
    return ((rgb, raw, normal) if kind == "rdf" else (rgb, raw)), probes


# measured: min cosine 0.99381 (DCVGANGenerator, all frozen: en4.1.bn2.weight, the cancellation in d gamma = rstd (<W, G> - rm sum dz);
# >= 0.99970 elsewhere), median 0.999951, norm ratios within 0.61 %, outputs 5.8e-5 max-abs
GEN_BOUND = dict(min_cos=0.987, median_cos=0.9999, ratio=0.012, out=1.2e-4)
# bf16 against the emulation: min cosine 0.893, median 0.980, shallow layers 0.9959, norm ratios within 20 % (median 0.26 %), outputs
# 2.0e-2 -- the noise floor of two bf16 implementations (test_gpu_train.py explains it)
BF16_GEN_BOUND = dict(out=4e-2, min_cos=0.78, median_cos=0.96, min_cos_shallow=0.992, max_ratio_dev=0.4, median_ratio_dev=6e-3)


@gpu
@pytest.mark.parametrize("every", [1, 2], ids=["all_frozen", "alternate_frozen"])
@pytest.mark.parametrize("kind", ["rdf", "dcvgan"])
def test_generator_fp32_tc_matches_fp32_composition(kind, every, monkeypatch):
    """fp32_tc train()-mode generator with all / alternate BatchNorms frozen against the same walk on fp32 PyTorch ops (TF32 off;
    frozen BatchNorms as F.batch_norm(training=False)): outputs, every parameter gradient's direction and norm, and the frozen
    BatchNorms' buffers untouched while the others' move."""
    import rdfc_gan_b200.train_forward as tf
    from _fp32_ops import fp32_torch_ops
    monkeypatch.setattr(torch.backends.cudnn, "allow_tf32", False)
    monkeypatch.setattr(torch.backends.cuda.matmul, "allow_tf32", False)
    B, H, W = 2, 36, 52
    G = _generator(kind).set_train_precision('fp32_tc')
    frozen = _freeze(G, every)
    live = [m for m in G.modules() if isinstance(m, nn.BatchNorm2d) and m.training]
    assert (len(live) == 0) == (every == 1)
    inputs, probes = _gen_inputs(kind, B, H, W)
    before, live_before = _buffers(frozen), _buffers(live)
    results = []
    for composed in (False, True):
        if composed:
            conv, bn = fp32_torch_ops()
            monkeypatch.setattr(tf, "conv2d_nhwc", conv)
            monkeypatch.setattr(tf, "bn_act", bn)
            monkeypatch.setattr(tf, "conv_bn_act_frozen", _frozen_fp32_op())
        G.zero_grad(set_to_none=True)
        results.append(_run_generator(G, inputs, probes))
        assert _same_buffers(frozen, before)
    assert not live or not _same_buffers(live, live_before)
    (o0, g0), (o1, g1) = results
    assert set(g0) == set(g1) and len(g0) > 150
    cos = {n: _cos(g0[n], g1[n]) for n in g0 if g0[n].numel() >= 8}
    ratio = {n: float(g0[n].double().norm() / (g1[n].double().norm() + 1e-30)) for n in cos}
    rep = {"min_cos": min(cos.values()), "median_cos": float(np.median(list(cos.values()))),
           "max_ratio_dev": max(abs(r - 1) for r in ratio.values()), "out": max(float((o0[k] - o1[k]).abs().max()) for k in o0)}
    _dump({"case": f"gen_fp32_{kind}_{every}", "errs": rep, "worst": sorted((c, n) for n, c in cos.items())[:5]})
    assert rep["out"] <= GEN_BOUND["out"], rep
    assert rep["min_cos"] >= GEN_BOUND["min_cos"] and rep["median_cos"] >= GEN_BOUND["median_cos"], (rep, sorted((c, n) for n, c in cos.items())[:8])
    assert rep["max_ratio_dev"] <= GEN_BOUND["ratio"], (rep, sorted((abs(r - 1), n) for n, r in ratio.items())[-5:])


@gpu
@pytest.mark.parametrize("every", [1, 2], ids=["all_frozen", "alternate_frozen"])
@pytest.mark.parametrize("kind", ["rdf", "dcvgan"])
def test_generator_bf16_matches_emulation(kind, every, monkeypatch):
    """bf16 train()-mode generator with frozen BatchNorms against the same walk on PyTorch ops that round to bf16 at the same
    points (test_gpu_train.py's emulation, plus the frozen op's): the gradient cosine and norm-ratio statistics of that test."""
    import rdfc_gan_b200.train_forward as tf
    from test_gpu_train import _emulated_ops
    monkeypatch.setattr(torch.backends.cudnn, "allow_tf32", False)
    monkeypatch.setattr(torch.backends.cuda.matmul, "allow_tf32", False)
    B, H, W = 2, 36, 52
    G = _generator(kind)
    frozen = _freeze(G, every)
    inputs, probes = _gen_inputs(kind, B, H, W)
    before = _buffers(frozen)
    results = []
    for emulate in (False, True):
        if emulate:
            conv, bn = _emulated_ops()
            monkeypatch.setattr(tf, "conv2d_nhwc", conv)
            monkeypatch.setattr(tf, "bn_act", bn)
            monkeypatch.setattr(tf, "conv_bn_act_frozen", _frozen_bf16_op())
        G.zero_grad(set_to_none=True)
        results.append(_run_generator(G, inputs, probes))
    assert _same_buffers(frozen, before)
    (o0, g0), (o1, g1) = results
    assert set(g0) == set(g1) and len(g0) > 150
    cos = {n: _cos(g0[n], g1[n]) for n in g0 if g0[n].numel() >= 8}
    ratio = {n: float(g0[n].double().norm() / (g1[n].double().norm() + 1e-30)) for n in cos}
    shallow = [n for n in cos if any(t in n for t in ("_dec0.", "_dec1.", "nlspn_refine_module", ".de2."))]
    rep = {"out": max(float((o0[k] - o1[k]).abs().max()) for k in o0), "min_cos": min(cos.values()),
           "median_cos": float(np.median(list(cos.values()))), "min_cos_shallow": min(cos[n] for n in shallow),
           "max_ratio_dev": max(abs(r - 1) for r in ratio.values()), "median_ratio_dev": abs(float(np.median(list(ratio.values()))) - 1)}
    _dump({"case": f"gen_bf16_{kind}_{every}", "errs": rep, "worst": sorted((c, n) for n, c in cos.items())[:5]})
    b = BF16_GEN_BOUND
    assert rep["out"] <= b["out"], rep
    assert rep["min_cos_shallow"] >= b["min_cos_shallow"] and rep["min_cos"] >= b["min_cos"] and rep["median_cos"] >= b["median_cos"], rep
    assert rep["max_ratio_dev"] <= b["max_ratio_dev"] and rep["median_ratio_dev"] <= b["median_ratio_dev"], rep


def _as_tuple(G, out):
    return tuple(out[k] for k in G._OUTPUTS) if isinstance(out, dict) else out


EVAL_BOUND = 1.2e-4        # max-abs over the five maps (measured 5.9e-5)


@gpu
@pytest.mark.parametrize("kind", ["rdf", "dcvgan"])
def test_all_frozen_train_forward_matches_eval(kind):
    """A train()-mode generator with every BatchNorm frozen computes the reference's eval() function: its fp32_tc outputs match the
    eval-mode engine in fp32 on the same inputs."""
    B, H, W = 2, 36, 52
    G = _generator(kind).set_train_precision('fp32_tc')
    _freeze(G)
    inputs, _ = _gen_inputs(kind, B, H, W)
    with torch.no_grad():
        tr = dict(zip(G._OUTPUTS, (v.clone() for v in _as_tuple(G, G(*inputs)))))
        G.eval().set_precision('fp32')
        ev = dict(zip(G._OUTPUTS, _as_tuple(G, G(*inputs))))
    err = max(float((tr[k] - ev[k]).abs().max()) for k in tr)
    _dump({"case": f"eval_consistency_{kind}", "errs": {"out": err}})
    assert err <= EVAL_BOUND, err


@gpu
def test_dispatch_spy(monkeypatch):
    """Every BatchNorm in train(): conv_bn_act_frozen is never called.  One BatchNorm frozen: it is called once, for that layer, and
    that layer's batch-statistics op is not."""
    import rdfc_gan_b200.train_forward as tf
    from _synth import synth_state_dict
    from rdfc_gan_b200.generator import RDFGenerator
    G = RDFGenerator(pretrained_on_imagenet=False, use_nlspn_refine=False)
    G.load_state_dict(synth_state_dict(G, seed=7, recipe="scaled"))
    G = G.cuda().train()
    inputs, _ = _gen_inputs("rdf", 1, 36, 52, seed=7)
    calls, bn_calls = [], []
    real_frozen, real_bn = tf.conv_bn_act_frozen, tf.bn_act
    monkeypatch.setattr(tf, "conv_bn_act_frozen", lambda x, w, bn, *a, **k: calls.append(bn) or real_frozen(x, w, bn, *a, **k))
    monkeypatch.setattr(tf, "bn_act", lambda y, bn, *a, **k: bn_calls.append(bn) or real_bn(y, bn, *a, **k))
    G(*inputs)
    assert calls == [] and len(bn_calls) > 20
    n_bn = len(bn_calls)
    target = G.depth_branch_encoder_decoder.en3[0].bn2
    target.eval()
    bn_calls.clear()
    out = G(*inputs)
    assert calls == [target] and len(bn_calls) == n_bn - 1 and target not in bn_calls
    assert all(torch.isfinite(v).all() for v in out.values())


@gpu
@pytest.mark.parametrize("precision", ["bf16", "fp32_tc"])
def test_frozen_generator_deterministic(precision):
    """Under torch.use_deterministic_algorithms(True): three backward passes of a generator with every BatchNorm frozen give
    bit-identical parameter gradients."""
    B, H, W = 2, 36, 52
    G = _generator("rdf").set_train_precision(precision)
    _freeze(G)
    inputs, probes = _gen_inputs("rdf", B, H, W)
    saved = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    torch.use_deterministic_algorithms(True)
    try:
        runs = []
        for _ in range(3):
            G.zero_grad(set_to_none=True)
            runs.append(_run_generator(G, inputs, probes)[1])
    finally:
        torch.use_deterministic_algorithms(False)
        torch.backends.cudnn.allow_tf32 = saved
    assert all(set(r) == set(runs[0]) and all(torch.equal(r[n], runs[0][n]) for n in r) for r in runs[1:])


RESNET_BOUND = dict(out=7e-5, min_cos=0.99988, ratio=5e-3)     # measured 3.2e-5, 0.999942, 0.23 %


@gpu
@pytest.mark.parametrize("padding", ["reflect", "zero"])
def test_resnet_generator_frozen(padding, monkeypatch):
    """G_B2A in train() with every BatchNorm frozen: fp32_tc against the same walk on fp32 PyTorch ops (TF32 off) -- the frozen
    BatchNorms after the tensor-core convs fused (the explicit-pad form with its crop for 'reflect'), the one after the 7x7 conv
    on PyTorch -- and a bf16 run: finite, buffers untouched."""
    import rdfc_gan_b200.resnet_generator as rg
    from _fp32_ops import fp32_torch_ops
    from _synth import synth_state_dict
    from test_gpu_resnet_generator import _torch_pad
    monkeypatch.setattr(torch.backends.cudnn, "allow_tf32", False)
    monkeypatch.setattr(torch.backends.cuda.matmul, "allow_tf32", False)
    G = rg.ResnetGenerator(1, 3, ngf=64, n_blocks=2, padding_type=padding)
    G.load_state_dict(synth_state_dict(G, seed=41, recipe="scaled"))
    G = G.cuda().train()
    frozen = _freeze(G)
    before = _buffers(frozen)
    gen = torch.Generator(device="cuda").manual_seed(9)
    x = torch.rand(2, 1, 64, 96, device="cuda", generator=gen) * 2 - 1
    probe = torch.randn(2, 3, 64, 96, device="cuda", generator=gen)
    y = G(x)                                                    # bf16
    (y * probe).sum().backward()
    assert torch.isfinite(y).all() and all(torch.isfinite(p.grad).all() for p in G.parameters())
    G.set_train_precision('fp32_tc')
    calls = []
    real = rg.conv_bn_act_frozen
    monkeypatch.setattr(rg, "conv_bn_act_frozen", lambda *a, **k: calls.append(1) or real(*a, **k))
    grads, outs = [], []
    for composed in (False, True):
        if composed:
            conv, bn = fp32_torch_ops()
            monkeypatch.setattr(rg, "conv2d_nhwc", conv)
            monkeypatch.setattr(rg, "bn_act", bn)
            monkeypatch.setattr(rg, "pad_nhwc", _torch_pad)
            monkeypatch.setattr(rg, "conv_bn_act_frozen", _frozen_fp32_op())
        G.zero_grad(set_to_none=True)
        xi = x.clone().requires_grad_(True)
        y = G(xi)
        (y * probe).sum().backward()
        grads.append(dict({n: p.grad.detach().clone() for n, p in G.named_parameters()}, input=xi.grad))
        outs.append(y.detach())
    assert len(calls) == 2 + 2 * 2 + 2                         # down-sampling, residual-block and transposed convs
    assert _same_buffers(frozen, before)
    cos = {n: _cos(grads[0][n], grads[1][n]) for n in grads[0] if grads[0][n].numel() >= 8}
    ratio = {n: float(grads[0][n].double().norm() / (grads[1][n].double().norm() + 1e-30)) for n in cos}
    rep = dict(out=float((outs[0] - outs[1]).abs().max()), min_cos=min(cos.values()), max_ratio_dev=max(abs(r - 1) for r in ratio.values()))
    _dump({"case": f"resnet_frozen_{padding}", "errs": rep, "worst": sorted((c, n) for n, c in cos.items())[:4]})
    assert rep["out"] <= RESNET_BOUND["out"], rep
    assert rep["min_cos"] >= RESNET_BOUND["min_cos"], (rep, sorted((c, n) for n, c in cos.items())[:6])
    assert rep["max_ratio_dev"] <= RESNET_BOUND["ratio"], rep


@gpu
@pytest.mark.parametrize("precision", ["bf16", "fp32_tc"])
def test_training_step_with_frozen_generator_bn(precision):
    """One RDFGAN.optimize_parameters() with G's BatchNorms frozen: G's buffers unchanged, D's BatchNorm buffers updated, the
    losses finite."""
    from _det_step import build
    model, batch = build(2, 64, 96, precision)
    g_bns = _freeze(model.G)
    d_bns = [m for m in model.D.modules() if isinstance(m, nn.BatchNorm2d)]
    assert g_bns and d_bns
    g_before, d_before = _buffers(g_bns), _buffers(d_bns)
    model.set_input(batch)
    losses = model.optimize_parameters()
    assert all(math.isfinite(float(v)) for v in losses.values()), losses
    assert _same_buffers(g_bns, g_before)
    # D runs twice in a step (backward_D, backward_G), both times in train(): its statistics move
    assert all(int(m.num_batches_tracked) > int(c) and not torch.equal(m.running_mean, a) for m, (a, b, c) in zip(d_bns, d_before))
