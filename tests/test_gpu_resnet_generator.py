"""ResnetGenerator (G_B2A) on the NHWC reflection / replication padding kernels (csrc/pad.cu, train_ops.pad_nhwc), its fp32_tc
training precision and reproducible training under torch.use_deterministic_algorithms.

Pad kernels against F.pad (forward bit for bit, backward against fp64 autograd), host-side validation, the fp32_tc generator against
the reference golden (tests/golden/resnet_generator.npz) and against the same walk on fp32 PyTorch ops, the bf16 forward against the
walk with F.pad, and bit-identical gradients under the flag, in-process and across two processes (tests/_det_cycle.py).  The stated
bounds of the fp32_tc comparisons are twice what was measured on a B200 (DESIGN.md section 7)."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest
import torch
import torch.nn.functional as F

HERE = os.path.dirname(os.path.abspath(__file__))
gpu = pytest.mark.gpu
BF = torch.bfloat16


def _cos(a, b):
    a, b = a.double().reshape(-1), b.double().reshape(-1)
    return float((a * b).sum() / (a.norm() * b.norm() + 1e-30))


def _torch_pad(x, pad, mode):
    """the parent's composition: the pad module's F.pad on the channels-last NCHW view of the NHWC tensor"""
    p = (pad,) * 4 if isinstance(pad, int) else tuple(pad)
    return F.pad(x.permute(0, 3, 1, 2), p, mode=mode).permute(0, 2, 3, 1)


def _three(fn):
    """fn() -> tuple of tensors, called three times (the second while another stream runs element-wise work); all bit-identical"""
    a = [t.clone() for t in fn()]
    side, x = torch.cuda.Stream(), torch.randn(4096, 4096, device="cuda")
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(50):
            x = torch.tanh(x * 1.0001 + 0.5)
    b = [t.clone() for t in fn()]
    c = fn()
    torch.cuda.synchronize()
    for i, (p, q, r) in enumerate(zip(a, b, c)):
        assert torch.equal(p, q) and torch.equal(p, r), i
    return a


# ------------------------------------------------------------------------------------------------ host side, no GPU
def test_pad_entry_points_validate_before_launch():
    """Invalid arguments are refused by rdfc_pad_nhwc_forward / _backward before anything touches the device (fake pointers)."""
    from rdfc_gan_b200 import _cabi as C
    assert hasattr(C.lib, "rdfc_pad_nhwc_forward") and hasattr(C.lib, "rdfc_pad_nhwc_backward")

    def v(ptr=0x10000, dtype=C.BF16, ch=8, stride=8):
        return C.View(ptr, dtype, ch, stride, 0)

    def fails(fn, small, big, B, H, W, pad, mode, text):
        n0 = C.launch_count()
        args = (ctypes.byref(small), B, H, W, pad, mode, ctypes.byref(big), None) if fn == "forward" else \
               (ctypes.byref(big), B, H, W, pad, mode, ctypes.byref(small), None)
        rc = getattr(C.lib, f"rdfc_pad_nhwc_{fn}")(*args)
        assert rc != 0 and C.launch_count() == n0
        msg = C.lib.rdfc_last_error().decode()
        assert text in msg, msg

    for fn in ("forward", "backward"):
        fails(fn, v(), v(), 2, 8, 8, -1, C.PAD_REFLECT, "padding -1 < 0")
        fails(fn, v(), v(), 2, 3, 8, 3, C.PAD_REFLECT, "padding < H and < W")
        fails(fn, v(), v(), 2, 8, 2, 2, C.PAD_REFLECT, "padding < H and < W")
        fails(fn, v(), v(), 2, 8, 8, 1, 2, "unknown mode")
        fails(fn, v(), v(dtype=C.F32), 2, 8, 8, 1, C.PAD_REPLICATE, "one dtype")
        fails(fn, v(dtype=C.F16), v(dtype=C.F16), 2, 8, 8, 1, C.PAD_REPLICATE, "one dtype")
        fails(fn, v(), v(ch=16, stride=16), 2, 8, 8, 1, C.PAD_REPLICATE, "same channel count")
        fails(fn, v(stride=4), v(), 2, 8, 8, 1, C.PAD_REPLICATE, "same channel count")
        fails(fn, v(ptr=0x10001), v(), 2, 8, 8, 1, C.PAD_REPLICATE, "aligned")
        fails(fn, v(dtype=C.F32), v(ptr=0x10002, dtype=C.F32), 2, 8, 8, 1, C.PAD_REPLICATE, "aligned")
        fails(fn, v(ptr=0), v(), 2, 8, 8, 1, C.PAD_REPLICATE, "NULL")
        fails(fn, v(), v(), 0, 8, 8, 1, C.PAD_REPLICATE, "empty")


def test_pad_op_and_precision_switch_refuse_bad_arguments():
    from rdfc_gan_b200.resnet_generator import ResnetGenerator
    from rdfc_gan_b200.train_ops import pad_nhwc
    x = torch.zeros(1, 6, 6, 4)
    with pytest.raises(RuntimeError, match="all four sides alike"):
        pad_nhwc(x, (1, 1, 2, 2), 'reflect')
    with pytest.raises(ValueError):
        pad_nhwc(x, 1, 'circular')
    G = ResnetGenerator(1, 3, n_blocks=1)
    assert G.set_train_precision('fp32_tc') is G and G._train_precision == 'fp32_tc'
    assert G.set_train_precision('bf16') is G
    for bad in ('fp32', 'fp16', None):
        with pytest.raises(ValueError):
            G.set_train_precision(bad)
    assert G._train_precision == 'bf16'
    G.set_train_precision('fp32_tc')
    sd = G.state_dict()
    assert not any('precision' in k for k in sd)
    G2 = ResnetGenerator(1, 3, n_blocks=1)
    G2.load_state_dict(sd, strict=True)
    assert G2._train_precision == 'bf16'


# ------------------------------------------------------------------------------------------------ pad kernels, GPU
def _pad_case(mode, dtype, Cc, p, H, W, B=2, seed=0):
    from rdfc_gan_b200.train_ops import pad_nhwc
    g = torch.Generator(device="cuda").manual_seed(seed * 1000 + Cc * 10 + p + H * 7 + W)
    x = torch.randn(B, H, W, Cc, device="cuda", generator=g).to(dtype)
    gy = torch.randn(B, H + 2 * p, W + 2 * p, Cc, device="cuda", generator=g).to(dtype)
    xa = x.clone().requires_grad_(True)
    y = pad_nhwc(xa, p, mode)
    assert torch.equal(y, _torch_pad(x, p, mode)), "forward is not a bit-exact copy"
    y.backward(gy)
    x64 = x.double().requires_grad_(True)
    _torch_pad(x64, p, mode).backward(gy.double())
    return x, gy, xa.grad, x64.grad


def _check_grad(got, want64, dtype):
    if dtype == torch.float32:
        err = float((got.double() - want64).abs().max())
        assert err <= 2e-7 * float(want64.abs().max()), err
    else:                               # one bf16 ulp of the fp64 result rounded to bf16
        w = want64.to(BF).double()
        ulp = torch.exp2(torch.floor(torch.log2(w.abs().clamp_min(1e-30))) - 7)
        excess = float(((got.double() - w).abs() - ulp).max())
        assert excess <= 0, excess


@gpu
@pytest.mark.parametrize("p", [1, 3])
@pytest.mark.parametrize("Cc", [1, 3, 64, 256])
@pytest.mark.parametrize("dtype", [torch.float32, BF], ids=["fp32", "bf16"])
@pytest.mark.parametrize("mode", ["reflect", "replicate"])
def test_pad_against_torch(mode, dtype, Cc, p):
    """Forward torch.equal F.pad; backward within 2e-7 relative (fp32) / one bf16 ulp (bf16) of fp64 autograd through F.pad; at odd
    sizes, H = p + 1 and W = p + 1 included (every reflected row / column maps onto a pixel that also has its own position)."""
    for H, W in ((p + 1, 13), (9, p + 1), (p + 1, p + 1), (11, 7)):
        _, _, got, want = _pad_case(mode, dtype, Cc, p, H, W)
        _check_grad(got, want, dtype)


@gpu
@pytest.mark.parametrize("dtype", [torch.float32, BF], ids=["fp32", "bf16"])
@pytest.mark.parametrize("mode", ["reflect", "replicate"])
def test_pad_channel_slices_and_reproducibility(mode, dtype):
    """A channel-slice input and a channel-slice grad_out go to the kernels as (pointer, channels, pixel stride) views: the results
    equal those of contiguous copies bit for bit.  Three backward calls are bit-identical, one with another stream busy."""
    from rdfc_gan_b200 import _cabi as C
    from rdfc_gan_b200.train_ops import _dense, pad_nhwc
    g = torch.Generator(device="cuda").manual_seed(3)
    for Cc, c0, ctot, p in ((64, 32, 96, 1), (3, 8, 16, 3)):
        B, H, W = 2, 17, 23
        big = torch.randn(B, H, W, ctot, device="cuda", generator=g).to(dtype)
        gbig = torch.randn(B, H + 2 * p, W + 2 * p, ctot, device="cuda", generator=g).to(dtype)
        xs, gs = big[..., c0:c0 + Cc], gbig[..., c0:c0 + Cc]
        assert not xs.is_contiguous() and _dense(xs) is xs and C.nhwc_viewable(gs)
        xfull = big.clone().requires_grad_(True)
        y = pad_nhwc(xfull[..., c0:c0 + Cc], p, mode)
        assert torch.equal(y, _torch_pad(xs.contiguous(), p, mode))
        y.backward(gs)
        xc = xs.contiguous().requires_grad_(True)
        pad_nhwc(xc, p, mode).backward(gs.contiguous())
        assert torch.equal(xfull.grad[..., c0:c0 + Cc], xc.grad) and float(xfull.grad[..., :c0].abs().max()) == 0.0

        def bwd():
            xa = xs.contiguous().requires_grad_(True)
            pad_nhwc(xa, p, mode).backward(gs)
            return (xa.grad,)
        _three(bwd)


@gpu
def test_reflect_pad_too_large_raises_before_launch():
    from rdfc_gan_b200 import _cabi as C
    from rdfc_gan_b200.train_ops import pad_nhwc
    x = torch.randn(1, 3, 8, 4, device="cuda")
    torch.cuda.synchronize()
    n0 = C.launch_count()
    for p, xx in ((3, x), (4, x), (8, x.transpose(1, 2).contiguous())):
        with pytest.raises(RuntimeError, match="padding < H and < W"):
            pad_nhwc(xx, p, 'reflect')
    assert C.launch_count() == n0
    assert pad_nhwc(x, 3, 'replicate').shape == (1, 9, 14, 4)           # replicate has no such limit


# ------------------------------------------------------------------------------------------------ the generator, GPU
# Measured on a B200.  Golden: outputs 2.2e-5 (train) / 3.9e-5 (eval) max-abs, min gradient cosine 0.999946, median norm ratio
# 1 + 3.5e-6.  Composition: outputs 5.0e-5, min cosine 0.999956, largest norm ratio deviation 1.06e-3.  The bounds are twice those,
# except the golden cosine, where twice the deficit (0.99989) would be looser than 0.9999.
GOLD_BOUND = dict(out=8e-5, min_cos=0.9999, ratio=7e-6)
COMP_BOUND = dict(out=1e-4, min_cos=0.99991, ratio=2.2e-3)


def _golden_generator():
    from make_train_golden import RESNET_CASE, resnet_inputs
    from _synth import synth_state_dict
    from rdfc_gan_b200.resnet_generator import ResnetGenerator
    G = ResnetGenerator(**RESNET_CASE["kw"])
    G.load_state_dict(synth_state_dict(G, seed=RESNET_CASE["seed"], recipe="scaled"))
    x, probe = resnet_inputs()
    return G.cuda(), x.cuda(), probe.cuda()


@gpu
def test_fp32_tc_against_reference_golden(golden_dir):
    """fp32_tc G_B2A against the reference class in fp32 on the CPU: train() and eval() outputs, the sampled gradients of a linear
    probe (every parameter's cosine) and the gradient norms (median ratio).  The bf16 mode's bounds are 8e-2 / cos 0.85 / 0.95."""
    from make_train_golden import grad_sample_index
    gold = np.load(f"{golden_dir}/resnet_generator.npz")
    G, x, probe = _golden_generator()
    G.train().set_train_precision('fp32_tc')
    y = G(x)
    out_train = float((y.detach().cpu() - torch.from_numpy(gold["out_train"])).abs().max())
    (y * probe).sum().backward()
    cos, ratio = {}, {}
    for n, p in G.named_parameters():
        ratio[n] = float(p.grad.double().norm()) / (float(gold[f"norm_{n}"]) + 1e-30)
        if p.numel() >= 8:
            idx = torch.from_numpy(grad_sample_index(n, p.numel()))
            cos[n] = _cos(p.grad.detach().reshape(-1).cpu()[idx], torch.from_numpy(gold[f"grad_{n}"]))
    G.eval()
    with torch.no_grad():
        out_eval = float((G(x).cpu() - torch.from_numpy(gold["out_eval"])).abs().max())
    rep = dict(out_train=out_train, out_eval=out_eval, min_cos=min(cos.values()), median_ratio_dev=abs(float(np.median(list(ratio.values()))) - 1))
    _dump({"case": "resnet_fp32_tc_golden", "errs": rep, "worst": sorted((c, n) for n, c in cos.items())[:4]})
    assert out_train <= GOLD_BOUND["out"] and out_eval <= GOLD_BOUND["out"], rep
    assert rep["min_cos"] >= GOLD_BOUND["min_cos"], (rep, sorted((c, n) for n, c in cos.items())[:6])
    assert rep["median_ratio_dev"] <= GOLD_BOUND["ratio"], rep


@gpu
def test_fp32_tc_matches_fp32_composition(monkeypatch):
    """fp32_tc G_B2A (n_blocks = 6, B = 2, 96x128) against the same walk with conv2d_nhwc / bn_act / pad_nhwc on fp32 PyTorch ops,
    TF32 off: outputs, the gradient with respect to the input and every parameter gradient's direction and norm."""
    import rdfc_gan_b200.resnet_generator as rg
    from _fp32_ops import fp32_torch_ops
    from _synth import synth_state_dict
    monkeypatch.setattr(torch.backends.cudnn, "allow_tf32", False)
    monkeypatch.setattr(torch.backends.cuda.matmul, "allow_tf32", False)
    G = rg.ResnetGenerator(1, 3, ngf=64, n_blocks=6)
    G.load_state_dict(synth_state_dict(G, seed=41, recipe="scaled"))
    G = G.cuda().train().set_train_precision('fp32_tc')
    gen = torch.Generator(device="cuda").manual_seed(9)
    x = torch.rand(2, 1, 96, 128, device="cuda", generator=gen) * 2 - 1
    probe = torch.randn(2, 3, 96, 128, device="cuda", generator=gen)
    grads, outs = [], []
    for composed in (False, True):
        if composed:
            conv, bn = fp32_torch_ops()
            monkeypatch.setattr(rg, "conv2d_nhwc", conv)
            monkeypatch.setattr(rg, "bn_act", bn)
            monkeypatch.setattr(rg, "pad_nhwc", _torch_pad)
        G.zero_grad(set_to_none=True)
        xi = x.clone().requires_grad_(True)
        y = G(xi)
        (y * probe).sum().backward()
        grads.append(dict({n: p.grad.detach().clone() for n, p in G.named_parameters()}, input=xi.grad))
        outs.append(y.detach())
    cos = {n: _cos(grads[0][n], grads[1][n]) for n in grads[0] if grads[0][n].numel() >= 8}
    ratio = {n: float(grads[0][n].double().norm() / (grads[1][n].double().norm() + 1e-30)) for n in cos}
    rep = dict(out=float((outs[0] - outs[1]).abs().max()), min_cos=min(cos.values()), input_cos=cos["input"],
               max_ratio_dev=max(abs(r - 1) for r in ratio.values()))
    _dump({"case": "resnet_fp32_tc_composition", "errs": rep, "worst": sorted((c, n) for n, c in cos.items())[:4]})
    assert rep["out"] <= COMP_BOUND["out"], rep
    assert rep["min_cos"] >= COMP_BOUND["min_cos"], (rep, sorted((c, n) for n, c in cos.items())[:6])
    assert rep["max_ratio_dev"] <= COMP_BOUND["ratio"], (rep, sorted((abs(r - 1), n) for n, r in ratio.items())[-4:])


@gpu
def test_fp32_tc_refuses_convs_off_the_tensor_cores():
    """ngf = 48: the stride-2 conv reads 48 channels, which the tensor-core conv does not take -- fp32_tc raises instead of running a
    cuDNN conv; bf16 keeps its fp32 PyTorch route for that layer, and trains (forward and backward) the 96 -> 48 transposed conv,
    whose 48 output channels the tensor-core conv takes, on the tensor cores."""
    from rdfc_gan_b200.resnet_generator import ResnetGenerator
    G = ResnetGenerator(1, 3, ngf=48, n_blocks=1).cuda().train()
    x = torch.rand(1, 1, 32, 32, device="cuda")
    y = G(x)
    assert torch.isfinite(y).all()
    y.square().sum().backward()
    assert all(p.grad is not None and torch.isfinite(p.grad).all() for p in G.parameters())
    G.set_train_precision('fp32_tc')
    with pytest.raises(RuntimeError, match="input channels % 32 == 0"):
        G(x)


@gpu
def test_bf16_forward_unchanged(monkeypatch):
    """bf16 train() and eval() outputs equal bit for bit those of the same walk with F.pad in place of pad_nhwc."""
    import rdfc_gan_b200.resnet_generator as rg
    G, x, _ = _golden_generator()
    for training in (True, False):
        outs = []
        for substitute in (False, True):
            if substitute:
                monkeypatch.setattr(rg, "pad_nhwc", _torch_pad)
            G.train(training)
            with torch.no_grad():
                outs.append(G(x))
            monkeypatch.undo()
        assert torch.equal(outs[0], outs[1]), training


@gpu
@pytest.mark.parametrize("precision", ["bf16", "fp32_tc"])
def test_deterministic_forward_backward(precision):
    """Under torch.use_deterministic_algorithms(True) (torch's NaN fill of uninitialised memory left on) G_B2A's forward and
    backward run, the output is finite, and every parameter gradient and the input gradient are bit-identical over three runs."""
    from _synth import synth_state_dict
    from rdfc_gan_b200.resnet_generator import ResnetGenerator
    G = ResnetGenerator(1, 3)
    G.load_state_dict(synth_state_dict(G, seed=5, recipe="scaled"))
    G = G.cuda().train().set_train_precision(precision)
    gen = torch.Generator(device="cuda").manual_seed(2)
    x = torch.rand(2, 1, 64, 96, device="cuda", generator=gen) * 2 - 1
    probe = torch.randn(2, 3, 64, 96, device="cuda", generator=gen)

    def run():
        G.zero_grad(set_to_none=True)
        xi = x.clone().requires_grad_(True)
        y = G(xi)
        assert torch.isfinite(y).all()
        (y * probe).sum().backward()
        return [xi.grad] + [p.grad for p in G.parameters()]
    torch.use_deterministic_algorithms(True)
    try:
        _three(run)
    finally:
        torch.use_deterministic_algorithms(False)


@gpu
@pytest.mark.parametrize("precision", ["bf16", "fp32_tc"])
def test_cycle_step_reproducible_across_processes(precision):
    """Two fresh processes, each two cycle-shaped steps (G_A2B train forward, G_B2A on depth_map_1, the RDFGAN losses plus an L1
    cycle loss, Adam on both generators) at B = 2, 96x128 under the flag: the losses and both generators' parameters and buffers
    hash the same."""
    env = dict(os.environ, CUBLAS_WORKSPACE_CONFIG=":4096:8")
    cmd = [sys.executable, os.path.join(HERE, "_det_cycle.py"), precision, "2", "96", "128", "2"]
    digests = [subprocess.run(cmd, env=env, capture_output=True, text=True, check=True).stdout.strip().splitlines()[-1] for _ in range(2)]
    assert len(digests[0]) == 64 and digests[0] == digests[1], digests


def _dump(rec):
    """RDFC_DUMP_PARITY=<file>: append the measured errors (the bounds above are twice the measured values)."""
    path = os.environ.get("RDFC_DUMP_PARITY")
    if path:
        import json
        with open(path, "a") as f:
            f.write(json.dumps(rec) + "\n")
