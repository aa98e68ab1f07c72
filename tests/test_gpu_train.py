"""-m gpu: the training-step kernels (filter gradient, batch-statistics BatchNorm forward / backward, the differentiable conv
Function) against PyTorch autograd on the same bf16-rounded operands, and the whole training step (generator + PatchGAN
discriminator, lsgan + L1, rdf_gan.py:135-207) against gradients taken through the REFERENCE's own modules
(tests/golden/train_step.npz, made by tests/golden/make_train_golden.py)."""
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu
BF = torch.bfloat16


def _rel(a, b):
    return float((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-30))


@pytest.mark.parametrize("case", [
    # B, Cin, Cout, H, W, k, stride
    (2, 64, 64, 36, 52, 3, 1), (3, 64, 128, 37, 50, 3, 2), (2, 128, 32, 19, 45, 3, 1), (1, 192, 384, 29, 38, 1, 1),
    (2, 64, 128, 40, 41, 1, 2), (2, 96, 160, 17, 23, 3, 1), (1, 512, 512, 15, 19, 3, 1), (4, 64, 64, 228, 304, 3, 1),
    (2, 192, 64, 29, 38, 3, 2), (1, 128, 256, 58, 77, 3, 2), (2, 256, 80, 9, 100, 3, 1),
    # Cout % 16 == 8: the kernel's N is rounded up to 16, the channels past Cout are zero fill and masked
    (2, 64, 24, 36, 52, 3, 1), (2, 64, 40, 29, 38, 3, 2), (1, 128, 8, 15, 19, 1, 1), (2, 96, 24, 20, 28, 1, 2)])
def test_filter_gradient_against_torch(case):
    from rdfc_gan_b200.train_ops import _wgrad
    B, Cin, Cout, H, W, k, s = case
    g = torch.Generator(device="cuda").manual_seed(sum(case))
    p = (k - 1) // 2
    Ho, Wo = (H + 2 * p - k) // s + 1, (W + 2 * p - k) // s + 1
    x = torch.randn(B, H, W, Cin, device="cuda", generator=g).to(BF)
    gy = torch.randn(B, Ho, Wo, Cout, device="cuda", generator=g).to(BF)
    got = _wgrad(gy, x, k, s)
    want = torch.nn.grad.conv2d_weight(x.permute(0, 3, 1, 2).double(), (Cout, Cin, k, k), gy.permute(0, 3, 1, 2).double(), stride=s, padding=p)
    assert got.shape == want.shape
    assert _rel(got, want) <= 2e-5, _rel(got, want)          # fp32 accumulation of exact bf16 products
    again = _wgrad(gy, x, k, s)
    assert torch.equal(got, again), "the split-K reduction must be deterministic"
    # every tile width of the tcgen05 kernel (csrc/wgrad_umma.cu) must give the same sums, in two launches (partials, reduction)
    from rdfc_gan_b200 import _cabi as C
    try:
        for tw in (16, 32):
            C.set_knob("RDFC_WGRAD_TW", tw)
            n0 = C.launch_count()
            other = _wgrad(gy, x, k, s)
            assert C.launch_count() - n0 == 2
            assert _rel(other, want) <= 2e-5, (tw, _rel(other, want))
    finally:
        C.set_knob("RDFC_WGRAD_TW", None)


@pytest.mark.parametrize("case", [(2, 64, 64, 20, 28, 3, 1, False), (2, 64, 128, 21, 27, 3, 2, False), (2, 128, 64, 10, 13, 3, 2, True),
                                  (1, 192, 384, 9, 12, 1, 1, False), (2, 64, 128, 14, 15, 1, 2, False)])
def test_conv_function_gradients(case):
    """conv2d_nhwc forward, data gradient (forward kernel with transformed filters) and filter gradient against autograd of
    F.conv2d / F.conv_transpose2d on the same bf16-rounded tensors."""
    from rdfc_gan_b200.train_ops import conv2d_nhwc
    B, Cin, Cout, H, W, k, s, tr = case
    g = torch.Generator(device="cuda").manual_seed(sum(case[:7]) + 3)
    x = torch.randn(B, H, W, Cin, device="cuda", generator=g).to(BF).requires_grad_(True)
    wshape = (Cin, Cout, k, k) if tr else (Cout, Cin, k, k)
    w = (torch.randn(*wshape, device="cuda", generator=g) / math.sqrt(Cin * k * k)).to(BF).float().requires_grad_(True)
    y = conv2d_nhwc(x, w, k, s, tr)
    xr = x.detach().float().permute(0, 3, 1, 2).double().requires_grad_(True)
    wr = w.detach().double().requires_grad_(True)
    yr = (F.conv_transpose2d(xr, wr, stride=2, padding=1, output_padding=1) if tr else F.conv2d(xr, wr, stride=s, padding=(k - 1) // 2))
    assert tuple(y.shape) == (B, yr.shape[2], yr.shape[3], Cout)
    assert _rel(y.float().permute(0, 3, 1, 2), yr.detach()) <= 6e-3          # bf16 output rounding
    gy = torch.randn(y.shape, device="cuda", generator=g).to(BF)
    y.backward(gy)
    yr.backward(gy.float().permute(0, 3, 1, 2).double())
    assert _rel(x.grad.float().permute(0, 3, 1, 2), xr.grad) <= 6e-3
    assert _rel(w.grad, wr.grad) <= 1e-4


@pytest.mark.parametrize("case", [(2, 64, 64, 36, 52, 1), (2, 64, 128, 37, 50, 2), (1, 128, 256, 30, 44, 2), (2, 256, 256, 19, 26, 1)])
def test_conv_input_grad_on_the_forward_kernel(case):
    """conv2d_nhwc's data gradient of the generator's 3x3 convs (stride-1 / transposed convs on the tensor-core kernel), with a filter
    that needs no gradient, against torch.nn.grad.conv2d_input on the same bf16-rounded operands."""
    from rdfc_gan_b200.train_ops import conv2d_nhwc
    B, Cin, Cout, H, W, stride = case
    gen = torch.Generator().manual_seed(sum(case))
    w = (torch.randn(Cout, Cin, 3, 3, generator=gen) / math.sqrt(Cout * 9)).bfloat16().float()
    Ho, Wo = (H + 2 - 3) // stride + 1, (W + 2 - 3) // stride + 1
    go = torch.randn(B, Cout, Ho, Wo, generator=gen).bfloat16().float()
    ref = torch.nn.grad.conv2d_input((B, Cin, H, W), w.double(), go.double(), stride=stride, padding=1).float()
    x = torch.zeros(B, H, W, Cin, dtype=BF, device="cuda", requires_grad=True)
    wd = w.cuda()
    conv2d_nhwc(x, wd, 3, stride).backward(go.permute(0, 2, 3, 1).bfloat16().contiguous().cuda())
    assert wd.grad is None
    got = x.grad.float().permute(0, 3, 1, 2).cpu()
    assert tuple(got.shape) == (B, Cin, H, W)
    err = (got - ref).abs().max().item()
    assert err <= 1.5e-2 * max(1.0, ref.abs().max().item()), (case, err)        # one bf16 rounding of the output


def test_conv_transpose_input_grad_on_the_forward_kernel():
    from rdfc_gan_b200.train_ops import conv2d_nhwc
    B, Cin, Cout, H, W = 2, 192, 64, 19, 26
    gen = torch.Generator().manual_seed(4)
    w = (torch.randn(Cin, Cout, 3, 3, generator=gen) / math.sqrt(Cout * 9)).bfloat16().float()
    xr = torch.zeros(B, Cin, H, W, dtype=torch.double, requires_grad=True)
    yr = F.conv_transpose2d(xr, w.double(), None, stride=2, padding=1, output_padding=1)
    go = torch.randn(yr.shape, generator=gen).bfloat16().float()
    (ref,) = torch.autograd.grad(yr, xr, go.double())
    x = torch.zeros(B, H, W, Cin, dtype=BF, device="cuda", requires_grad=True)
    wd = w.cuda()
    conv2d_nhwc(x, wd, 3, 2, True).backward(go.permute(0, 2, 3, 1).bfloat16().contiguous().cuda())
    assert wd.grad is None
    got = x.grad.float().permute(0, 3, 1, 2).cpu()
    assert tuple(got.shape) == (B, Cin, H, W)
    assert (got - ref.float()).abs().max().item() <= 1.5e-2 * max(1.0, ref.abs().max().item())


@pytest.mark.parametrize("dtype", [BF, torch.float32])
def test_conv_function_rejects_cin_off_the_tensor_core_rule(dtype):
    """conv2d_nhwc needs Cin % 32 == 0 (bf16 and fp32_tc alike): Cin = 24 raises a RuntimeError naming the rule before any launch."""
    from rdfc_gan_b200 import _cabi as C
    from rdfc_gan_b200.train_ops import conv2d_nhwc
    x = torch.randn(1, 8, 8, 24, device="cuda").to(dtype)
    w = torch.randn(16, 24, 3, 3, device="cuda")
    n0 = C.launch_count()
    with pytest.raises(RuntimeError, match="% 32|multiple of 32"):
        conv2d_nhwc(x, w)
    assert C.launch_count() == n0


@pytest.mark.parametrize("case", [(2, 19, 27, 64, 1, True), (3, 12, 10, 128, 2, False), (1, 30, 44, 32, 0, True), (2, 114, 152, 64, 2, True)])
def test_batchnorm_activation_function(case):
    """bn_act = act(BatchNorm2d_train(y) + residual): outputs, running statistics and the gradients w.r.t. y, gamma, beta and the
    residual against nn.BatchNorm2d + autograd in fp64 on the same bf16-rounded input."""
    from rdfc_gan_b200 import _cabi as C
    from rdfc_gan_b200.train_ops import bn_act
    B, H, W, Cc, act, with_res = case
    g = torch.Generator(device="cuda").manual_seed(sum(case[:4]))
    y = (1.5 * torch.randn(B, H, W, Cc, device="cuda", generator=g) + 0.3).to(BF).requires_grad_(True)
    res = torch.randn(B, H, W, Cc, device="cuda", generator=g).to(BF).requires_grad_(True) if with_res else None
    bn = torch.nn.BatchNorm2d(Cc).cuda().train()
    with torch.no_grad():
        bn.weight.uniform_(0.5, 1.5, generator=g)
        bn.bias.normal_(0, 0.2, generator=g)
    ref = torch.nn.BatchNorm2d(Cc).cuda().double().train()
    ref.load_state_dict({k: v.double() if v.is_floating_point() else v for k, v in bn.state_dict().items()})
    out = bn_act(y, bn, res, act)
    yr = y.detach().double().permute(0, 3, 1, 2).requires_grad_(True)
    rr = res.detach().double().permute(0, 3, 1, 2).requires_grad_(True) if with_res else None
    z = ref(yr) + (rr if with_res else 0)
    zr = {C.ACT_NONE: z, C.ACT_RELU: F.relu(z), C.ACT_LEAKY02: F.leaky_relu(z, 0.2)}[act]
    assert _rel(out.float().permute(0, 3, 1, 2), zr.detach()) <= 6e-3
    assert _rel(bn.running_mean, ref.running_mean) <= 1e-4 and _rel(bn.running_var, ref.running_var) <= 1e-4
    assert int(bn.num_batches_tracked) == 1
    go = torch.randn(out.shape, device="cuda", generator=g).to(BF)
    out.backward(go)
    zr.backward(go.double().permute(0, 3, 1, 2))
    # the activation mask comes from the bf16-rounded output: pixels within one rounding of zero may flip
    assert _rel(y.grad.float().permute(0, 3, 1, 2), yr.grad) <= 2e-2
    assert _rel(bn.weight.grad, ref.weight.grad) <= 1e-2 and _rel(bn.bias.grad, ref.bias.grad) <= 1e-2
    if with_res:
        assert _rel(res.grad.float().permute(0, 3, 1, 2), rr.grad) <= 2e-2


def _emulated_ops():
    """The two kernel-backed ops of train_ops.py re-stated with PyTorch ops that round to bf16 at the same points (bf16 operands,
    fp32 arithmetic, bf16 results; autograd supplies the backward): what the kernels must reproduce up to summation order."""
    from rdfc_gan_b200 import _cabi as C

    def conv(x, weight, k=3, stride=1, transposed=False):
        xn = x.float().permute(0, 3, 1, 2)
        w = weight.to(BF).float()
        y = (F.conv_transpose2d(xn, w, stride=2, padding=1, output_padding=1) if transposed else
             F.conv2d(xn, w, stride=stride, padding=(k - 1) // 2))
        return y.permute(0, 2, 3, 1).contiguous().to(BF)

    def bn(y, mod, residual=None, act=C.ACT_NONE):
        yf = y.float()
        mean, var = yf.mean((0, 1, 2)), yf.var((0, 1, 2), unbiased=False)
        z = (yf - mean) * torch.rsqrt(var + mod.eps) * mod.weight + mod.bias
        if residual is not None:
            z = z + residual.float()
        z = {C.ACT_NONE: z, C.ACT_RELU: F.relu(z), C.ACT_LEAKY02: F.leaky_relu(z, 0.2)}[act]
        return z.to(BF)
    return conv, bn


@pytest.mark.parametrize("fuse", ["WAdaIN", "IN"])
def test_generator_backward_matches_bf16_emulation(fuse, monkeypatch):
    """The whole train-mode generator (forward kernels, data / filter gradients, fused BatchNorm backward, fused NLSPN backward)
    against the same composition with the two kernel-backed ops replaced by PyTorch expressions that round to bf16 at the same
    points: every parameter gradient must agree closely.  (Against an fp32 reference the gradient DIRECTION of deep layers differs
    by several degrees per ReLU layer -- units whose pre-activation lies within one bf16 rounding of zero route the gradient
    differently -- which is why the reference-golden test below states a cosine bound, and this test pins the arithmetic.)"""
    import rdfc_gan_b200.train_forward as tf
    from make_train_golden import _NL
    from _synth import synth_inputs, synth_state_dict
    from rdfc_gan_b200.generator import RDFGenerator
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    B, H, W = 2, 36, 52
    G = RDFGenerator(pretrained_on_imagenet=False, fuse_depth_in_rgb_decoder=fuse, use_nlspn_refine=True, nlspn_configs=_NL)
    G.load_state_dict(synth_state_dict(G, seed=33, recipe="scaled", nlspn_stress=True))
    G = G.cuda().train()
    rgb, normal, raw = (t.cuda() for t in synth_inputs(B, H, W, seed=33))
    gen = torch.Generator(device="cuda").manual_seed(5)
    probes = [torch.randn(B, 1, H, W, device="cuda", generator=gen) for _ in range(5)]
    grads = []
    for emulate in (False, True):
        if emulate:
            conv, bn = _emulated_ops()
            monkeypatch.setattr(tf, "conv2d_nhwc", conv)
            monkeypatch.setattr(tf, "bn_act", bn)
        G.zero_grad(set_to_none=True)
        out = G(rgb, raw, normal)
        sum((out[k] * R).sum() for k, R in zip(("depth_map_1", "confidence_map_1", "depth_map_2", "confidence_map_2", "pred_depth"), probes)).backward()
        grads.append({n: p.grad.detach().clone() for n, p in G.named_parameters() if p.grad is not None})
        outs = out if not emulate else outs
    assert set(grads[0]) == set(grads[1]) and len(grads[0]) > 150
    for k in outs:
        assert float((outs[k] - out[k]).abs().max()) <= 2e-2, k
    cos = {n: float((grads[0][n].double() * grads[1][n].double()).sum() / (grads[0][n].double().norm() * grads[1][n].double().norm() + 1e-30))
           for n in grads[0] if grads[0][n].numel() >= 8}
    ratio = {n: float(grads[0][n].double().norm() / (grads[1][n].double().norm() + 1e-30)) for n in cos}
    # Two bf16 implementations that differ only in summation order already disagree by one bf16 ulp on some activations; a unit
    # whose pre-activation lies within that ulp of zero then routes its gradient differently (ReLU / LeakyReLU derivative 0 / 0.2
    # vs 1).  With eps ~ 0.4 % relative rounding noise that is ~0.3 % of the units, i.e. ~8 % relative gradient noise per
    # activation layer, accumulating in quadrature along the ~20-layer backward path: cos ~ 0.94 at the stems, ~1 at the heads
    # (measured: 0.92-0.97 / 0.998-1.0).  The per-op tests above pin the arithmetic to 1e-4..2e-2; here the bounds are the
    # noise floor, unbiased magnitude included.
    shallow = [n for n in cos if any(t in n for t in ("_dec0.", "_dec1.", "nlspn_refine_module", ".de2."))]
    assert min(cos[n] for n in shallow) >= 0.97, sorted((cos[n], n) for n in shallow)[:5]
    assert min(cos.values()) >= 0.85 and float(np.median(list(cos.values()))) >= 0.93, sorted((c, n) for n, c in cos.items())[:8]
    assert all(abs(r - 1) <= 0.3 for r in ratio.values()) and abs(float(np.median(list(ratio.values()))) - 1) <= 0.03, \
        sorted((abs(r - 1), n) for n, r in ratio.items())[-8:]


def test_training_step_against_reference_gradients(golden_dir):
    """One RDFGAN.optimize_parameters-style step at the golden's weights: train-mode generator forward (batch statistics),
    backward_D, backward_G.  Losses, the five output maps, BatchNorm running statistics and a fixed sample of every parameter's
    gradient against the reference's own modules run on the CPU (make_train_golden.py).  bf16 tensor-core arithmetic against an
    fp32 reference: the stated tolerances are twice what was measured."""
    from make_train_golden import CASE, build_inputs, grad_sample_index, D_KW
    from _synth import synth_state_dict
    from rdfc_gan_b200.discriminator import PatchGANDiscriminator
    from rdfc_gan_b200.generator import RDFGenerator
    from rdfc_gan_b200.rdf_gan import RDFGAN
    gold = np.load(f"{golden_dir}/train_step.npz")
    G = RDFGenerator(pretrained_on_imagenet=False, **CASE["kw"])
    G.load_state_dict(synth_state_dict(G, seed=CASE["seed"], recipe="scaled", nlspn_stress=True))
    D = PatchGANDiscriminator(**D_KW)
    D.load_state_dict(synth_state_dict(D, seed=CASE["seed"] + 1, recipe="init"))   # init_weights(D), as rdf_gan.py:61
    model = RDFGAN(G, D, device="cuda", args=CASE["args"])
    model.train()
    data = build_inputs()
    model.set_input(data)
    model.forward()
    outs = dict(depth_map_1=model.fake_B_rgb_branch, confidence_map_1=model.conf_map_rgb_branch, depth_map_2=model.fake_B_depth_branch,
                confidence_map_2=model.conf_map_depth_branch, pred_depth=model.final_depth)
    report = {}
    for k, v in outs.items():
        report[f"out:{k}"] = float((v.detach().cpu() - torch.from_numpy(gold[f"out_{k}"])).abs().max())
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
            if key not in gold.files or p.numel() < 8:          # one-element tensors (head biases): a direction has no meaning
                continue
            idx = torch.from_numpy(grad_sample_index(name, p.numel()))
            got = p.grad.detach().reshape(-1).cpu()[idx].double()
            want = torch.from_numpy(gold[key]).double()
            cos[f"{net}.{name}"] = float((got * want).sum() / (got.norm() * want.norm() + 1e-30))
            ratio[f"{net}.{name}"] = float(got.norm() / (want.norm() + 1e-30))
    report["grad:min_cos_G"] = min(v for k, v in cos.items() if k.startswith("G."))
    report["grad:median_cos_G"] = float(np.median([v for k, v in cos.items() if k.startswith("G.")]))
    report["grad:min_cos_D"] = min(v for k, v in cos.items() if k.startswith("D."))
    report["grad:median_norm_ratio"] = float(np.median(list(ratio.values())))
    import json, os
    if os.environ.get("RDFC_DUMP_PARITY"):
        with open(os.environ["RDFC_DUMP_PARITY"], "a") as f:
            f.write(json.dumps({"case": "train_step", "errs": report, "worst": sorted((c, n) for n, c in cos.items())[:12]}) + "\n")
    assert all(v <= 6e-2 for k, v in report.items() if k.startswith("out:")), report
    assert all(v <= 2e-2 for k, v in report.items() if k.startswith("loss:")), report
    # gradient direction: the bf16 noise floor analysed in test_generator_backward_matches_bf16_emulation (the discriminator's
    # own gradients are fp32 PyTorch on a slightly different `fake`)
    assert report["grad:min_cos_G"] >= 0.8 and report["grad:median_cos_G"] >= 0.9 and report["grad:min_cos_D"] >= 0.95, (report, sorted((c, n) for n, c in cos.items())[:8])
    assert abs(report["grad:median_norm_ratio"] - 1) <= 0.05, report
    # running statistics moved off their initial values towards the batch statistics
    rm = model.G.rgb_branch_encoder_decoder.en2[0].bn1.running_mean.detach().cpu()
    assert float((rm - torch.from_numpy(gold["bn_running_mean"])).abs().max()) <= 2e-2, (rm[:6], gold["bn_running_mean"][:6])
    # and the optimiser step runs end to end (one flattened gradient buffer per net)
    stats = model.optimize_parameters()
    assert set(stats) == {"loss_D", "loss_D_real", "loss_D_fake", "loss_G_GAN", "loss_L1_rgb_branch", "loss_L1_depth_branch", "loss_L1_fusion"}
    assert all(math.isfinite(v) for v in stats.values())


def test_resnet_generator_against_reference(golden_dir):
    """G_B2A (C/lib/models/generator/resnet_generator.py): train() and eval() outputs and the parameter gradients of a linear probe
    against the reference class on the CPU (tests/golden/resnet_generator.npz).  bf16 activations: outputs to 8e-2, gradient
    direction to the bf16 noise floor (see test_generator_backward_matches_bf16_emulation)."""
    from make_train_golden import RESNET_CASE, grad_sample_index, resnet_inputs
    from _synth import synth_state_dict
    from rdfc_gan_b200.resnet_generator import ResnetGenerator
    gold = np.load(f"{golden_dir}/resnet_generator.npz")
    G = ResnetGenerator(**RESNET_CASE["kw"])
    G.load_state_dict(synth_state_dict(G, seed=RESNET_CASE["seed"], recipe="scaled"))
    G = G.cuda().train()
    x, probe = (t.cuda() for t in resnet_inputs())
    y = G(x)
    assert tuple(y.shape) == tuple(gold["out_train"].shape)
    assert float((y.detach().cpu() - torch.from_numpy(gold["out_train"])).abs().max()) <= 8e-2          # measured 3.8e-2 (tanh outputs in +-1)
    (y * probe).sum().backward()
    cos = {}
    for n, p in G.named_parameters():
        if p.numel() < 8:
            continue
        idx = torch.from_numpy(grad_sample_index(n, p.numel()))
        got, want = p.grad.detach().reshape(-1).cpu()[idx].double(), torch.from_numpy(gold[f"grad_{n}"]).double()
        cos[n] = float((got * want).sum() / (got.norm() * want.norm() + 1e-30))
    assert min(cos.values()) >= 0.85 and float(np.median(list(cos.values()))) >= 0.95, sorted((c, n) for n, c in cos.items())[:6]
    G.eval()
    with torch.no_grad():
        ye = G(x)
    assert float((ye.cpu() - torch.from_numpy(gold["out_eval"])).abs().max()) <= 8e-2
    with pytest.raises(RuntimeError):
        G(x.cpu())


def test_channel_sliced_views_need_no_copy():
    """Autograd hands the operands of a channel concatenation back as channel SLICES of one NHWC tensor.  The training ops pass such
    tensors to the kernels as (pointer, channels, pixel stride) views: the results must be those of contiguous copies, bit for bit."""
    from rdfc_gan_b200 import _cabi as C
    from rdfc_gan_b200.train_ops import _dense, _wgrad, bn_act, conv2d_nhwc
    g = torch.Generator(device="cuda").manual_seed(11)
    big = torch.randn(2, 21, 35, 192, device="cuda", generator=g).to(BF)
    xs, gs = big[..., 64:128], big[..., 128:192]                 # two 64-channel slices, pixel stride 192
    assert not xs.is_contiguous() and C.nhwc_viewable(xs) and _dense(xs) is xs
    assert not C.nhwc_viewable(big[:, :, ::2]) and _dense(big[:, :, ::2]).is_contiguous()          # a spatial slice still gets copied
    assert torch.equal(_wgrad(gs, xs, 3, 1), _wgrad(gs.contiguous(), xs.contiguous(), 3, 1))
    assert torch.equal(_wgrad(gs, xs, 1, 1), _wgrad(gs.contiguous(), xs.contiguous(), 1, 1))
    w = (torch.randn(64, 64, 3, 3, device="cuda", generator=g) / 24).to(BF).float()
    assert torch.equal(conv2d_nhwc(xs, w, 3, 1), conv2d_nhwc(xs.contiguous(), w, 3, 1))
    bn1, bn2 = torch.nn.BatchNorm2d(64).cuda().train(), torch.nn.BatchNorm2d(64).cuda().train()
    ya = xs.detach().clone().requires_grad_(True)                 # contiguous leaf
    yb_full = big.detach().clone().requires_grad_(True)
    oa = bn_act(ya, bn1, gs.contiguous(), C.ACT_RELU)
    ob = bn_act(yb_full[..., 64:128], bn2, gs, C.ACT_RELU)        # sliced input and sliced residual
    assert torch.equal(oa, ob)
    up = torch.randn(oa.shape, device="cuda", generator=g).to(BF)
    oa.backward(up)
    ob.backward(up)
    assert torch.equal(ya.grad, yb_full.grad[..., 64:128]) and torch.equal(bn1.weight.grad, bn2.weight.grad)
    assert float(yb_full.grad[..., :64].abs().max()) == 0.0
