"""The fp32_tc training mode (set_train_precision('fp32_tc'); train_ops.py split-operand conv / filter gradient, fp32 BatchNorm):
per op against torch in fp64 on the same fp32 tensors, the whole train-mode generator against the same composition on fp32 PyTorch
ops (TF32 off), the reference golden train_step.npz at bounds >= 10x tighter than the bf16 mode's, mode switching, and the new C
entry points' host-side validation.  The stated bounds are twice what was measured on a B200 (DESIGN.md section 7)."""
import ctypes
import math
import os
import re
import subprocess

import numpy as np
import pytest
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
gpu = pytest.mark.gpu


def _rel(a, b):
    return float((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-30))


def _cos(a, b):
    a, b = a.double().reshape(-1), b.double().reshape(-1)
    return float((a * b).sum() / (a.norm() * b.norm() + 1e-30))


# ------------------------------------------------------------------------------------------------ host side, no GPU
def test_split_entry_points_exported_and_validated():
    from rdfc_gan_b200 import _cabi as C
    nm = subprocess.run(["nm", "-D", "--defined-only", C.LIB_PATH], capture_output=True, text=True, check=True).stdout
    exported = set(re.findall(r" T (rdfc_[a-z0-9_]+)", nm))
    hdr = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "rdfc_b200.h")).read(), flags=re.S)
    new = ("rdfc_split_scaled", "rdfc_conv_forward_split", "rdfc_conv_wgrad_split_workspace_floats", "rdfc_conv_wgrad_split")
    for name in new:
        assert re.search(rf"\b{name}\s*\(", hdr), name
        assert name in C.EXPORTS and name in exported, name
    assert C.lib.rdfc_abi_version() == 2
    fake = 1 << 20                                              # never dereferenced: every case fails before a launch
    n0 = C.launch_count()

    def fails(rc, text):
        assert rc != 0
        assert text in C.lib.rdfc_last_error().decode(), C.lib.rdfc_last_error()

    # the split entry: an fp32 source only, channel counts that are multiples of 32, an fp16 destination of 2C channels
    f = ctypes.c_void_p(fake)
    fails(C.lib.rdfc_split_scaled(ctypes.byref(C.View(fake, C.BF16, 64, 64, 0)), 16, ctypes.byref(C.View(fake, C.F16, 128, 128, 0)), f, None),
          "fp32 NHWC")
    fails(C.lib.rdfc_split_scaled(ctypes.byref(C.View(fake, C.F32, 48, 48, 0)), 16, ctypes.byref(C.View(fake, C.F16, 96, 96, 0)), f, None),
          "multiple of 32")
    fails(C.lib.rdfc_split_scaled(ctypes.byref(C.View(fake, C.F32, 64, 64, 0)), 16, ctypes.byref(C.View(fake, C.F32, 128, 128, 0)), f, None),
          "fp16")
    fails(C.lib.rdfc_split_scaled(ctypes.byref(C.View(fake, C.F32, 64, 64, 0)), 16, ctypes.byref(C.View(fake + 8, C.F16, 128, 128, 0)), f, None),
          "16-byte aligned")
    # the conv entry: an fp16 [hi | lo] input of 2 x Cin channels with Cin % 32 == 0, a scale vector
    d = C.ConvDesc()
    d.B, d.Hi, d.Wi, d.Ho, d.Wo, d.kh, d.kw, d.stride, d.pad = 1, 8, 8, 8, 8, 3, 3, 1, 1
    d.path = C.PATH_UMMA_F32X3
    d.inp, d.out = C.View(fake, C.F16, 96, 96, 0), C.View(fake, C.F32, 64, 64, 0)
    d.weight, d.scale = fake, fake
    fails(C.lib.rdfc_conv_forward_split(ctypes.byref(d), None), "Cin % 32")
    d.inp = C.View(fake, C.BF16, 128, 128, 0)
    fails(C.lib.rdfc_conv_forward_split(ctypes.byref(d), None), "fp16")
    d.inp, d.scale = C.View(fake, C.F16, 128, 128, 0), None
    fails(C.lib.rdfc_conv_forward_split(ctypes.byref(d), None), "inverse scale")
    # the filter-gradient entry: unaligned workspace, bad channel count, wrong dtype
    w = C.WgradDesc()
    w.B, w.Hg, w.Wg, w.Hi, w.Wi, w.k, w.stride, w.pad = 1, 8, 8, 8, 8, 3, 1, 1
    w.grad_out, w.input = C.View(fake, C.F16, 128, 128, 0), C.View(fake, C.F16, 128, 128, 0)
    fails(C.lib.rdfc_conv_wgrad_split(ctypes.byref(w), f, f, ctypes.c_void_p(fake + 4), None), "workspace must be 16-byte aligned")
    w.input = C.View(fake, C.F16, 96, 96, 0)
    fails(C.lib.rdfc_conv_wgrad_split(ctypes.byref(w), f, f, f, None), "C % 32 == 0")
    assert C.lib.rdfc_conv_wgrad_split_workspace_floats(ctypes.byref(w)) == -1
    w.input = C.View(fake, C.BF16, 128, 128, 0)
    fails(C.lib.rdfc_conv_wgrad_split(ctypes.byref(w), f, f, f, None), "fp16")
    assert C.launch_count() == n0, "an invalid call launched a kernel"


def test_set_train_precision_interface():
    from make_train_golden import _NL
    from rdfc_gan_b200.generator import DCVGANGenerator, RDFGenerator
    G = RDFGenerator(pretrained_on_imagenet=False)
    keys = list(G.state_dict())
    assert G._train_precision == 'bf16'
    assert G.set_train_precision('fp32_tc') is G and G._train_precision == 'fp32_tc'
    assert list(G.state_dict()) == keys                        # not part of state_dict
    with pytest.raises(ValueError, match="not provided"):
        G.set_train_precision('fp32')
    for bad in ('fp16', 'FP32_TC', None):
        with pytest.raises(ValueError):
            G.set_train_precision(bad)
    assert G._train_precision == 'fp32_tc'
    assert G.set_train_precision('bf16')._train_precision == 'bf16'
    D = DCVGANGenerator(None, pretrained_on_imagenet=False, use_nlpsn_refine=True, nlspn_configs=_NL)
    assert D.set_train_precision('fp32_tc') is D


# ------------------------------------------------------------------------------------------------ per op, GPU
# the shapes of test_gpu_train.py's filter-gradient and conv-function tests: B, Cin, Cout, H, W, k, stride, transposed
CONV_CASES = [(2, 64, 64, 36, 52, 3, 1, False), (3, 64, 128, 37, 50, 3, 2, False), (2, 128, 32, 19, 45, 3, 1, False),
              (1, 192, 384, 29, 38, 1, 1, False), (2, 64, 128, 40, 41, 1, 2, False), (2, 96, 160, 17, 23, 3, 1, False),
              (1, 512, 512, 15, 19, 3, 1, False), (4, 64, 64, 228, 304, 3, 1, False), (2, 192, 64, 29, 38, 3, 2, False),
              (1, 128, 256, 58, 77, 3, 2, False), (2, 256, 96, 9, 100, 3, 1, False),
              (2, 64, 64, 20, 28, 3, 1, False), (2, 64, 128, 21, 27, 3, 2, False), (2, 128, 64, 10, 13, 3, 2, True),
              (1, 192, 384, 9, 12, 1, 1, False), (2, 64, 128, 14, 15, 1, 2, False), (2, 256, 128, 29, 38, 3, 2, True)]
# Relative L2 bounds.  Forward and data gradient: the tensor cores' fp32 accumulation costs ~5e-9 per unit of the contraction length
# K (measured 4.9e-9 .. 5.2e-9 x K on every case, K = Cin k^2 forward, Cout k^2 data gradient; 2.3e-5 at 512 -> 512 3x3, <= 8.7e-6
# elsewhere), so the bound is twice that with K = max(Cin, Cout) k^2.  Filter gradient (K = pixels, split-K partials summed in
# fp32): measured <= 2.4e-6.
def _conv_bound(case):
    B, Cin, Cout, H, W, k, s, tr = case
    return {"fwd": 1e-8 * max(Cin, Cout) * k * k, "dgrad": 1e-8 * max(Cin, Cout) * k * k, "wgrad": 5e-6}


def _conv_case(case, a, gen):
    from rdfc_gan_b200.train_ops import conv2d_nhwc
    B, Cin, Cout, H, W, k, s, tr = case
    x = (a * torch.randn(B, H, W, Cin, device="cuda", generator=gen)).requires_grad_(True)
    wshape = (Cin, Cout, k, k) if tr else (Cout, Cin, k, k)
    w = (torch.randn(*wshape, device="cuda", generator=gen) / math.sqrt(Cin * k * k)).requires_grad_(True)
    y = conv2d_nhwc(x, w, k, s, tr)
    assert y.dtype == torch.float32
    xr = x.detach().permute(0, 3, 1, 2).double().requires_grad_(True)
    wr = w.detach().double().requires_grad_(True)
    yr = F.conv_transpose2d(xr, wr, stride=2, padding=1, output_padding=1) if tr else F.conv2d(xr, wr, stride=s, padding=(k - 1) // 2)
    gy = a * torch.randn(y.shape, device="cuda", generator=gen)
    y.backward(gy)
    yr.backward(gy.permute(0, 3, 1, 2).double())
    errs = {"fwd": _rel(y.detach().permute(0, 3, 1, 2), yr.detach()), "dgrad": _rel(x.grad.permute(0, 3, 1, 2), xr.grad),
            "wgrad": _rel(w.grad, wr.grad)}
    return errs, x, w, y, gy


@gpu
@pytest.mark.parametrize("case", CONV_CASES)
def test_conv_fp32_against_fp64(case):
    """conv2d_nhwc on fp32 tensors: forward, data gradient and filter gradient of every conv form against fp64 autograd on the SAME
    fp32 tensors -- at unit scale and with x and grad_out scaled by 1e-7 and 1e5 (the power-of-two scaling keeps the split's low half
    out of fp16's subnormal range); all-zero grad_out gives exactly zero gradients; the filter gradient is bit-reproducible."""
    from rdfc_gan_b200.train_ops import conv2d_nhwc
    gen = torch.Generator(device="cuda").manual_seed(sum(case[:7]) + 17)
    worst = {}
    for a in (1.0, 1e-7, 1e5):
        errs, x, w, y, gy = _conv_case(case, a, gen)
        for k, v in errs.items():
            worst[f"{k}@{a:g}"] = v
    _dump({"case": list(case), "errs": worst})
    bound = _conv_bound(case)
    assert all(v <= bound[k.split("@")[0]] for k, v in worst.items()), (worst, bound)
    # bit-reproducible gradients (the last unit-scale-free call's tensors), exact zeros for a zero cotangent
    B, Cin, Cout, H, W, k, s, tr = case
    grads = []
    for _ in range(2):
        x.grad = w.grad = None
        conv2d_nhwc(x, w, k, s, tr).backward(gy)
        grads.append((x.grad.clone(), w.grad.clone()))
    assert torch.equal(grads[0][0], grads[1][0]) and torch.equal(grads[0][1], grads[1][1])
    x.grad = w.grad = None
    conv2d_nhwc(x, w, k, s, tr).backward(torch.zeros_like(gy))
    assert float(x.grad.abs().max()) == 0.0 and float(w.grad.abs().max()) == 0.0


BN_BOUND = 4e-7            # relative L2 of every quantity: measured <= 1.8e-7 (running statistics), <= 1.5e-7 (gradients)


@gpu
@pytest.mark.parametrize("case", [(2, 19, 27, 64, 1, True), (3, 12, 10, 128, 2, False), (1, 30, 44, 32, 0, True), (2, 114, 152, 64, 2, True)])
def test_batchnorm_activation_fp32_against_fp64(case):
    """bn_act on fp32 NHWC tensors (and a channel-sliced input) against nn.BatchNorm2d + autograd in fp64 on the same tensors:
    outputs, running statistics, and the gradients w.r.t. y, gamma, beta and the residual."""
    from rdfc_gan_b200 import _cabi as C
    from rdfc_gan_b200.train_ops import bn_act
    B, H, W, Cc, act, with_res = case
    g = torch.Generator(device="cuda").manual_seed(sum(case[:4]) + 5)
    big = (1.5 * torch.randn(B, H, W, Cc + 32, device="cuda", generator=g) + 0.3).requires_grad_(True)
    y = big[..., 32:]                                           # a channel slice: passed as a view, not copied
    res = torch.randn(B, H, W, Cc, device="cuda", generator=g).requires_grad_(True) if with_res else None
    bn = torch.nn.BatchNorm2d(Cc).cuda().train()
    with torch.no_grad():
        bn.weight.uniform_(0.5, 1.5, generator=g)
        bn.bias.normal_(0, 0.2, generator=g)
    ref = torch.nn.BatchNorm2d(Cc).cuda().double().train()
    ref.load_state_dict({k: v.double() if v.is_floating_point() else v for k, v in bn.state_dict().items()})
    out = bn_act(y, bn, res, act)
    assert out.dtype == torch.float32
    yr = y.detach().double().permute(0, 3, 1, 2).requires_grad_(True)
    rr = res.detach().double().permute(0, 3, 1, 2).requires_grad_(True) if with_res else None
    z = ref(yr) + (rr if with_res else 0)
    zr = {C.ACT_NONE: z, C.ACT_RELU: F.relu(z), C.ACT_LEAKY02: F.leaky_relu(z, 0.2)}[act]
    go = torch.randn(out.shape, device="cuda", generator=g)
    out.backward(go)
    zr.backward(go.double().permute(0, 3, 1, 2))
    errs = {"out": _rel(out.detach().permute(0, 3, 1, 2), zr.detach()),
            "running": max(_rel(bn.running_mean, ref.running_mean), _rel(bn.running_var, ref.running_var)),
            "dy": _rel(big.grad[..., 32:].permute(0, 3, 1, 2), yr.grad), "dgamma": _rel(bn.weight.grad, ref.weight.grad),
            "dbeta": _rel(bn.bias.grad, ref.bias.grad)}
    if with_res:
        errs["dres"] = _rel(res.grad.permute(0, 3, 1, 2), rr.grad)
    _dump({"case": list(case), "bn": errs})
    assert float(big.grad[..., :32].abs().max()) == 0.0
    assert all(v <= BN_BOUND for v in errs.values()), errs


# ------------------------------------------------------------------------------------------------ whole generator, GPU
# measured: min cosine 0.99989, median 0.999993, norm ratios within 0.24 %, outputs 9.8e-6 max-abs
GEN_BOUND = dict(min_cos=0.9997, median_cos=0.99998, ratio=0.005, out=2e-5)


@gpu
@pytest.mark.parametrize("fuse", ["WAdaIN", "IN"])
def test_generator_fp32_tc_matches_fp32_composition(fuse, monkeypatch):
    """The train-mode generator in fp32_tc (split-operand kernels, fp32 BatchNorm, fused NLSPN) against the same composition with
    the two kernel-backed ops on fp32 PyTorch (TF32 off): outputs and every parameter gradient's direction and norm."""
    import rdfc_gan_b200.train_forward as tf
    from make_train_golden import _NL
    from _fp32_ops import fp32_torch_ops
    from _synth import synth_inputs, synth_state_dict
    from rdfc_gan_b200.generator import RDFGenerator
    monkeypatch.setattr(torch.backends.cudnn, "allow_tf32", False)
    monkeypatch.setattr(torch.backends.cuda.matmul, "allow_tf32", False)
    B, H, W = 2, 36, 52
    G = RDFGenerator(pretrained_on_imagenet=False, fuse_depth_in_rgb_decoder=fuse, use_nlspn_refine=True, nlspn_configs=_NL)
    G.load_state_dict(synth_state_dict(G, seed=33, recipe="scaled", nlspn_stress=True))
    G = G.cuda().train().set_train_precision('fp32_tc')
    rgb, normal, raw = (t.cuda() for t in synth_inputs(B, H, W, seed=33))
    gen = torch.Generator(device="cuda").manual_seed(5)
    probes = [torch.randn(B, 1, H, W, device="cuda", generator=gen) for _ in range(5)]
    grads, outs = [], []
    for composed in (False, True):
        if composed:
            conv, bn = fp32_torch_ops()
            monkeypatch.setattr(tf, "conv2d_nhwc", conv)
            monkeypatch.setattr(tf, "bn_act", bn)
        G.zero_grad(set_to_none=True)
        out = G(rgb, raw, normal)
        sum((out[k] * R).sum() for k, R in zip(G._OUTPUTS, probes)).backward()
        grads.append({n: p.grad.detach().clone() for n, p in G.named_parameters() if p.grad is not None})
        outs.append({k: v.detach() for k, v in out.items()})
    assert set(grads[0]) == set(grads[1]) and len(grads[0]) > 150
    cos = {n: _cos(grads[0][n], grads[1][n]) for n in grads[0] if grads[0][n].numel() >= 8}
    ratio = {n: float(grads[0][n].double().norm() / (grads[1][n].double().norm() + 1e-30)) for n in cos}
    rep = {"min_cos": min(cos.values()), "median_cos": float(np.median(list(cos.values()))),
           "max_ratio_dev": max(abs(r - 1) for r in ratio.values()), "out": max(float((outs[0][k] - outs[1][k]).abs().max()) for k in outs[0])}
    _dump({"case": f"generator_{fuse}", "errs": rep, "worst": sorted((c, n) for n, c in cos.items())[:5]})
    assert rep["out"] <= GEN_BOUND["out"], rep
    assert rep["min_cos"] >= GEN_BOUND["min_cos"] and rep["median_cos"] >= GEN_BOUND["median_cos"], (rep, sorted((c, n) for n, c in cos.items())[:8])
    assert rep["max_ratio_dev"] <= GEN_BOUND["ratio"], (rep, sorted((abs(r - 1), n) for n, r in ratio.items())[-5:])


# measured: outputs 9.2e-6 max-abs, losses 1.3e-6 relative, min / median G cosine 0.99975 / 0.99994, min D cosine 0.999996, median
# norm ratio 1.00001, running mean 1.3e-7
GOLD_BOUND = dict(out=2e-5, loss=5e-6, min_cos_G=0.9995, median_cos_G=0.99987, min_cos_D=0.99999, ratio=3e-5, running_mean=3e-7)


@gpu
def test_training_step_fp32_tc_against_reference_gradients(golden_dir, monkeypatch):
    """test_gpu_train.py's reference-golden training step (train_step.npz: the reference's own modules in fp32 on the CPU) run in
    fp32_tc, at bounds at least 10x tighter than the bf16 mode's.  TF32 off, as an fp32 user runs: the PatchGAN discriminator is
    plain cuDNN (with torch's default TF32 its losses move by 3e-4 and the D gradient cosine drops to 0.9991)."""
    from make_train_golden import CASE, build_inputs, grad_sample_index, D_KW
    from _synth import synth_state_dict
    from rdfc_gan_b200.discriminator import PatchGANDiscriminator
    from rdfc_gan_b200.generator import RDFGenerator
    from rdfc_gan_b200.rdf_gan import RDFGAN
    monkeypatch.setattr(torch.backends.cudnn, "allow_tf32", False)
    monkeypatch.setattr(torch.backends.cuda.matmul, "allow_tf32", False)
    gold = np.load(f"{golden_dir}/train_step.npz")
    G = RDFGenerator(pretrained_on_imagenet=False, **CASE["kw"])
    G.load_state_dict(synth_state_dict(G, seed=CASE["seed"], recipe="scaled", nlspn_stress=True))
    G.set_train_precision('fp32_tc')
    D = PatchGANDiscriminator(**D_KW)
    D.load_state_dict(synth_state_dict(D, seed=CASE["seed"] + 1, recipe="init"))
    model = RDFGAN(G, D, device="cuda", args=CASE["args"])
    model.train()
    model.set_input(build_inputs())
    model.forward()
    outs = dict(depth_map_1=model.fake_B_rgb_branch, confidence_map_1=model.conf_map_rgb_branch, depth_map_2=model.fake_B_depth_branch,
                confidence_map_2=model.conf_map_depth_branch, pred_depth=model.final_depth)
    report = {f"out:{k}": float((v.detach().cpu() - torch.from_numpy(gold[f"out_{k}"])).abs().max()) for k, v in outs.items()}
    model.set_requires_grad(model.D, True)
    model.bucket_D.zero()
    ld = model.backward_D()
    model.set_requires_grad(model.D, False)
    model.bucket_G.zero()
    lg = model.backward_G()
    for k, v in {**ld, **lg}.items():
        report[f"loss:{k}"] = abs(float(v) - float(gold[f"loss_{k}"])) / max(abs(float(gold[f"loss_{k}"])), 1e-6)
    cos, ratio = {}, {}
    for net, mod in (("G", model.G), ("D", model.D)):
        for name, p in mod.named_parameters():
            key = f"grad_{net}_{name}"
            if key not in gold.files or p.numel() < 8:
                continue
            idx = torch.from_numpy(grad_sample_index(name, p.numel()))
            got = p.grad.detach().reshape(-1).cpu()[idx].double()
            want = torch.from_numpy(gold[key]).double()
            cos[f"{net}.{name}"] = _cos(got, want)
            ratio[f"{net}.{name}"] = float(got.norm() / (want.norm() + 1e-30))
    report["grad:min_cos_G"] = min(v for k, v in cos.items() if k.startswith("G."))
    report["grad:median_cos_G"] = float(np.median([v for k, v in cos.items() if k.startswith("G.")]))
    report["grad:min_cos_D"] = min(v for k, v in cos.items() if k.startswith("D."))
    report["grad:median_norm_ratio"] = float(np.median(list(ratio.values())))
    rm = model.G.rgb_branch_encoder_decoder.en2[0].bn1.running_mean.detach().cpu()
    report["running_mean"] = float((rm - torch.from_numpy(gold["bn_running_mean"])).abs().max())
    _dump({"case": "train_step_fp32_tc", "errs": report, "worst": sorted((c, n) for n, c in cos.items())[:8]})
    assert all(v <= GOLD_BOUND["out"] for k, v in report.items() if k.startswith("out:")), report
    assert all(v <= GOLD_BOUND["loss"] for k, v in report.items() if k.startswith("loss:")), report
    assert report["grad:min_cos_G"] >= GOLD_BOUND["min_cos_G"] and report["grad:median_cos_G"] >= GOLD_BOUND["median_cos_G"], report
    assert report["grad:min_cos_D"] >= GOLD_BOUND["min_cos_D"], report
    assert abs(report["grad:median_norm_ratio"] - 1) <= GOLD_BOUND["ratio"], report
    assert report["running_mean"] <= GOLD_BOUND["running_mean"], report


@gpu
def test_mode_switching_keeps_bf16_bits_and_eval(monkeypatch):
    """bf16 step, fp32_tc step, bf16 step: the two bf16 steps give the same bits (outputs and gradients); the eval-mode engine's
    outputs do not depend on set_train_precision."""
    from _synth import synth_inputs, synth_state_dict
    from rdfc_gan_b200.generator import RDFGenerator
    monkeypatch.setattr(torch.backends.cudnn, "deterministic", True)      # the cuDNN stems' filter gradients, run to run
    B, H, W = 2, 36, 52
    G = RDFGenerator(pretrained_on_imagenet=False, use_nlspn_refine=False)  # (the NLSPN backward scatters with fp32 atomics)
    G.load_state_dict(synth_state_dict(G, seed=7, recipe="scaled"))
    G = G.cuda().train()
    rgb, normal, raw = (t.cuda() for t in synth_inputs(B, H, W, seed=7))
    probe = torch.randn(B, 1, H, W, device="cuda", generator=torch.Generator(device="cuda").manual_seed(3))
    steps = []
    for prec in ("bf16", "fp32_tc", "bf16"):
        G.set_train_precision(prec)
        G.zero_grad(set_to_none=True)
        out = G(rgb, raw, normal)
        sum((v * probe).sum() for v in out.values()).backward()
        steps.append(({k: v.detach().clone() for k, v in out.items()}, {n: p.grad.clone() for n, p in G.named_parameters() if p.grad is not None}))
    (o1, g1), (o2, g2), (o3, g3) = steps
    assert all(torch.equal(o1[k], o3[k]) for k in o1) and set(g1) == set(g3) and all(torch.equal(g1[n], g3[n]) for n in g1)
    assert all(float((o1[k] - o2[k]).abs().max()) > 0 for k in o1)        # the fp32_tc step did run its own arithmetic
    G.eval()                                                               # (running statistics as the three steps left them)
    evs = []
    for prec in ("bf16", "fp32_tc"):
        G.set_train_precision(prec)
        with torch.no_grad():
            evs.append({k: v.clone() for k, v in G(rgb, raw, normal).items()})
    assert all(torch.equal(evs[0][k], evs[1][k]) for k in evs[0])


def _dump(rec):
    """RDFC_DUMP_PARITY=<file>: append the measured errors (the bounds above are twice the measured values)."""
    path = os.environ.get("RDFC_DUMP_PARITY")
    if path:
        import json
        with open(path, "a") as f:
            f.write(json.dumps(rec) + "\n")
