"""Under torch.use_deterministic_algorithms the NLSPN and DCN backwards call their *_ex entry points with RDFC_DETERMINISTIC:
fixed-point scatters, gradients bit-identical from call to call (one of three calls runs with another stream busy), at the
accuracy bounds of the default path.  The last tests run the c4 training step in two fresh processes and compare hashes."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from _synth import DCN_CASES, dcn_case_inputs, nlspn_stress_inputs
from make_golden import NLSPN_CASES, NLSPN_SHAPE

HERE = os.path.dirname(os.path.abspath(__file__))
SCALES = (1e-30, 1e-4, 3e3, 1e30)
TC_CASES = [
    # B, Cin, Cout, H, W, k, s, p, d, groups, dg, mask, magnitude: the cases of test_backward_on_tensor_cores_matches_cuda_core_kernels
    (2, 64, 128, 128, 128, 3, 1, 1, 1, 1, 2, True, 1.0), (2, 64, 64, 37, 45, 3, 2, 1, 1, 2, 4, True, 1.0), (1, 32, 64, 20, 33, 3, 1, 2, 2, 1, 1, False, 1.0),
    (3, 128, 256, 19, 26, 1, 1, 0, 1, 1, 2, True, 1.0), (2, 64, 64, 23, 31, 3, 1, 1, 1, 1, 2, True, 1e-4), (2, 64, 64, 23, 31, 3, 1, 1, 1, 1, 2, True, 3e3)]


@pytest.fixture
def deterministic():
    torch.use_deterministic_algorithms(True)
    try:
        yield
    finally:
        torch.use_deterministic_algorithms(False)


def _three(fn):
    """fn() -> tuple of tensors, called three times (the second while another stream runs matrix products); all bit-identical"""
    a = [t.clone() for t in fn()]
    side, x = torch.cuda.Stream(), torch.randn(4096, 4096, device="cuda")
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(6):
            x = torch.tanh(x @ x)
    b = [t.clone() for t in fn()]
    c = fn()
    torch.cuda.synchronize()
    for i, (p, q, r) in enumerate(zip(a, b, c)):
        assert torch.equal(p, q) and torch.equal(p, r), i
    return a


def _within(got, want, tol, floor=1.0):
    scale = max(floor, float(want.abs().max()))
    err = float((got.double() - want.double()).abs().max())
    assert err <= tol * scale, (err, scale)


# ---------------------------------------------------------------- NLSPN --------------------------------------------------------
def _prop_inputs(B, H, W, seed):
    from oracle import nlspn as onl
    x = nlspn_stress_inputs(B, H, W, seed)
    off, aff = onl.get_offset_affinity(x["guidance"], x["confidence"], x["conv_w"], x["conv_b"], np.array([4.0], np.float32))[:2]
    gout = np.random.default_rng(seed + 100).standard_normal((B, 1, H, W)).astype(np.float32)
    return x, np.ascontiguousarray(off, np.float32), np.ascontiguousarray(aff, np.float32), gout


def _prop_grads(f, o, a, fix, T, preserve, gout):
    from rdfc_gan_b200.nlspn import _PropagateFused
    f, o, a = (t.detach().requires_grad_(True) for t in (f, o, a))
    y, _ = _PropagateFused.apply(f, o, a, fix if preserve else None, T, preserve)
    return torch.autograd.grad(y, (f, o, a), gout)


def _prop_full(B, preserve):
    """B images at 228x304 tiled from the stress generator's offsets (sigma ~ 2.2 px) and affinities"""
    H, W = 228, 304
    x, off, aff, _ = _prop_inputs(2, 32, 40, 21)
    rep = lambda v: torch.from_numpy(v).cuda().repeat(2, 1, 8, 8)[:B, :, :H, :W].contiguous()
    gen = torch.Generator(device="cuda").manual_seed(5)
    f = torch.randn(B, 1, H, W, device="cuda", generator=gen)
    gout = torch.randn(B, 1, H, W, device="cuda", generator=gen)
    return f, rep(off), rep(aff), rep(x["feat_fix"]), gout


@pytest.mark.gpu
@pytest.mark.parametrize("preserve", [False, True])
def test_propagate_backward_full_size_bit_identical(preserve, deterministic):
    f, o, a, fix, gout = _prop_full(4, preserve)
    det = _three(lambda: _prop_grads(f, o, a, fix, 18, preserve, gout))
    torch.use_deterministic_algorithms(False)
    ref = _prop_grads(f, o, a, fix, 18, preserve, gout)
    for got, want in zip(det, ref):
        _within(got, want, 1e-4)


@pytest.mark.gpu
@pytest.mark.parametrize("preserve", [False, True])
def test_propagate_backward_vs_oracle(preserve, deterministic):
    from oracle import nlspn as onl
    B, H, W, T = 2, 19, 27, 5
    x, off, aff, gout = _prop_inputs(B, H, W, 11)
    ref = onl.nlspn_propagate_backward(gout, x["pred_init"], off, aff, x["feat_fix"], preserve, T)
    t = lambda v: torch.from_numpy(v).cuda()
    got = _three(lambda: _prop_grads(t(x["pred_init"]), t(off), t(aff), t(x["feat_fix"]), T, preserve, t(gout)))
    for g, r in zip(got, ref):
        _within(g.cpu(), torch.from_numpy(r), 1e-4)


def _refine_grads(cfg, x, t, gout, fused):
    import _composition as comp
    from rdfc_gan_b200.nlspn import NLSPNRefineModule
    mod = NLSPNRefineModule(prop_kernel=3, prop_time=cfg["prop_time"], affinity=cfg["affinity"], affinity_gamma=0.5,
                            conf_prop=cfg["conf_prop"], preserve_input=cfg["preserve_input"]).cuda().train()
    mod.prop_layer.conv_offset_aff.weight.data.copy_(torch.from_numpy(x["conv_w"]))
    mod.prop_layer.conv_offset_aff.bias.data.copy_(torch.from_numpy(x["conv_b"]))
    g = t["guidance"].clone().requires_grad_(True)
    p = t["pred_init"].clone().requires_grad_(True)
    cf = t["confidence"].clone().requires_grad_(True)
    y, _ = mod(p, g, cf, t["feat_fix"]) if fused else comp.refine(mod, p, g, cf, t["feat_fix"])
    y.backward(gout)
    pl = mod.prop_layer
    out = [y.detach(), g.grad, p.grad, pl.conv_offset_aff.weight.grad, pl.conv_offset_aff.bias.grad]
    if pl.aff_scale_const.grad is not None:
        out.append(pl.aff_scale_const.grad)
    if cfg["conf_prop"]:
        out.append(cf.grad)
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["tgass18", "as12_preserve", "tc12_noconf", "ass18"])
def test_refine_module_backward_matches_composition(name, deterministic):
    """The four cases of test_fused_backward_matches_composition (affinity backward with the confidence scatter and the aff_scale
    partials, propagation backward) under the flag: bit-identical, and the composition's gradients to 2e-4."""
    cfg = NLSPN_CASES[name]
    B, H, W = NLSPN_SHAPE
    x = nlspn_stress_inputs(B, H, W, cfg["seed"])
    t = {k: torch.from_numpy(v).cuda() for k, v in x.items()}
    gout = torch.randn(B, 1, H, W, generator=torch.Generator().manual_seed(3)).cuda()
    fused = _three(lambda: _refine_grads(cfg, x, t, gout, True))
    comp = _refine_grads(cfg, x, t, gout, False)
    assert len(fused) == len(comp)
    for a, b in zip(fused, comp):
        _within(a, b, 2e-4)


@pytest.mark.gpu
@pytest.mark.parametrize("scale", SCALES)
def test_nlspn_gradient_scale(scale, deterministic):
    """grad_out far from unit magnitude: the fixed-point scale follows it (no overflow, no flush to zero)"""
    cfg = NLSPN_CASES["tgass18"]
    B, H, W = NLSPN_SHAPE
    x = nlspn_stress_inputs(B, H, W, cfg["seed"])
    t = {k: torch.from_numpy(v).cuda() for k, v in x.items()}
    gout = torch.randn(B, 1, H, W, generator=torch.Generator().manual_seed(3)).cuda() * scale
    tf32 = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False            # the conv's own backward: same arithmetic whichever algorithm cuDNN picks
    try:
        det = _refine_grads(cfg, x, t, gout, True)
        torch.use_deterministic_algorithms(False)
        ref = _refine_grads(cfg, x, t, gout, True)
    finally:
        torch.backends.cudnn.allow_tf32 = tf32
    for a, b in zip(det[1:], ref[1:]):
        assert torch.isfinite(a).all()
        _within(a, b, 2e-4, floor=0.0)


@pytest.mark.gpu
def test_nlspn_zero_and_nan_gradients(deterministic):
    cfg = NLSPN_CASES["tgass18"]
    B, H, W = NLSPN_SHAPE
    x = nlspn_stress_inputs(B, H, W, cfg["seed"])
    t = {k: torch.from_numpy(v).cuda() for k, v in x.items()}
    zero = _refine_grads(cfg, x, t, torch.zeros(B, 1, H, W, device="cuda"), True)
    for g in zero[1:]:
        assert torch.equal(g, torch.zeros_like(g))
    gout = torch.randn(B, 1, H, W, device="cuda")
    gout[0, 0, H // 2, W // 3] = float("nan")
    nan = _refine_grads(cfg, x, t, gout, True)
    for g in nan[1:3]:                                     # d guidance, d pred_init
        assert not torch.isfinite(g).all()
    f, o, a, fix, _ = _prop_full(1, False)
    g = torch.zeros_like(f)
    g[0, 0, 5, 7] = float("inf")
    assert not torch.isfinite(_prop_grads(f, o, a, fix, 18, False, g)[0]).all()


# ---------------------------------------------------------------- DCN ----------------------------------------------------------
def _dcn_inputs(case, dtype=torch.float32, scale=1.0):
    B, Cin, Cout, H, W, k, s, p, d, g, dg, with_mask, mag = case
    gen = torch.Generator(device="cuda").manual_seed(sum(case[:11]) + 7)
    Ho, Wo = (H + 2 * p - (d * (k - 1) + 1)) // s + 1, (W + 2 * p - (d * (k - 1) + 1)) // s + 1
    x = torch.randn(B, Cin, H, W, device="cuda", generator=gen) * mag
    w = torch.randn(Cout, Cin // g, k, k, device="cuda", generator=gen) * 0.1
    b = torch.randn(Cout, device="cuda", generator=gen) * 0.1
    off = torch.randn(B, dg * 2 * k * k, Ho, Wo, device="cuda", generator=gen) * 2.0
    m = torch.rand(B, dg * k * k, Ho, Wo, device="cuda", generator=gen) if with_mask else None
    go = torch.randn(B, Cout, Ho, Wo, device="cuda", generator=gen) * mag * scale
    cast = lambda v: None if v is None else v.to(dtype)
    return [cast(v) for v in (x, w, b, off, m, go)], (k, k, s, s, p, p, d, d, g, dg, 64)


def _dcn_bwd(inputs, geo):
    from rdfc_gan_b200.dcn import DCN
    x, w, b, off, m, go = inputs
    if m is not None:
        return DCN.modulated_deform_conv_backward(x, w, b, off, m, go, *geo)
    return DCN.deform_conv_backward(x, w, b, off, go, *geo)


@pytest.mark.gpu
@pytest.mark.parametrize("case", TC_CASES)
def test_dcn_backward_bit_identical(case, deterministic):
    """tensor-core path, CUDA-core path (RDFC_DCN_TC = 0) and fp64: bit-identical under the flag; the tensor-core gradients match
    the CUDA-core ones (2e-4 for grad_input, 5e-5 for the others) and, at small sizes, the fp64 C oracle (1e-4); fp64 matches the fp64
    default path to 1e-10."""
    from oracle import dcn as odcn
    from rdfc_gan_b200 import _cabi as C
    inputs, geo = _dcn_inputs(case)
    res = []
    try:
        for tc in (1, 0):
            C.set_knob("RDFC_DCN_TC", tc)
            res.append(_three(lambda: _dcn_bwd(inputs, geo)))
    finally:
        C.set_knob("RDFC_DCN_TC", None)
    # fp64 against the fp64 default path: fp32 and fp64 compute the sampling positions in different precisions, and a position within
    # an fp32 ulp of an integer takes another bilinear cell there, so grad_offset / grad_mask of the two dtypes are not comparable
    inputs64 = [None if v is None else v.double() for v in inputs]
    f64 = _three(lambda: _dcn_bwd(inputs64, geo))
    torch.use_deterministic_algorithms(False)
    f64_default = _dcn_bwd(inputs64, geo)
    torch.use_deterministic_algorithms(True)
    tols = [2e-4] + [5e-5] * (len(res[0]) - 1)
    for a, r, tol in zip(res[0], res[1], tols):
        _within(a, r, tol, floor=0.0)
    for q, r in zip(f64, f64_default):
        _within(q, r, 1e-10, floor=0.0)
    H, W = case[3], case[4]
    if H * W <= 1000:
        ref = [r for r in odcn.modulated_deform_conv_backward(*[None if v is None else v.cpu().double().numpy() for v in inputs], *geo)
               if r is not None]
        for a, r in zip(res[0], ref):
            _within(a.cpu(), torch.from_numpy(r), 1e-4, floor=0.0)


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(DCN_CASES))
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_dcn_goldens(name, dtype, golden_dir, deterministic):
    from oracle import dcn as odcn
    case = DCN_CASES[name]
    t = dcn_case_inputs(case, dtype=dtype)
    gold = np.load(f"{golden_dir}/dcn_{name}.npz")
    c = {k: torch.from_numpy(v).cuda() for k, v in t.items()}
    k, s, p, d, g, dg = (case[x] for x in ("k", "s", "p", "d", "g", "dg"))
    geo = (k, k, s, s, p, p, d, d, g, dg, 64)
    grads = _three(lambda: _dcn_bwd([c["input"], c["weight"], c["bias"], c["offset"], c.get("mask"), c["grad_output"]], geo))
    names = ["grad_input", "grad_offset"] + (["grad_mask"] if case["mask"] else []) + ["grad_weight", "grad_bias"]
    ref = dict(zip(["grad_input", "grad_offset", "grad_mask", "grad_weight", "grad_bias"],
                   odcn.modulated_deform_conv_backward(t["input"], t["weight"], t["bias"], t["offset"], t.get("mask"), t["grad_output"], *geo)))
    tol = 1e-10 if dtype == np.float64 else 2e-5
    for n, gr in zip(names, grads):
        _within(gr.cpu(), torch.from_numpy(ref[n]), tol)
        _within(gr.cpu(), torch.from_numpy(gold[n]), tol, floor=max(1.0, float(np.abs(ref[n]).max())))


@pytest.mark.gpu
def test_dcn_gradcheck(deterministic):
    from torch.autograd import gradcheck
    from rdfc_gan_b200.dcn import _DeformConv, _ModulatedDeformConv
    torch.manual_seed(1)
    x = (torch.rand(2, 4, 4, 4, dtype=torch.float64).cuda() * 0.01).requires_grad_(True)
    off = (torch.randn(2, 18, 4, 4, dtype=torch.float64).cuda() * 2).requires_grad_(True)
    msk = torch.sigmoid(torch.rand(2, 9, 4, 4, dtype=torch.float64).cuda()).requires_grad_(True)
    w = torch.randn(4, 2, 3, 3, dtype=torch.float64).cuda().requires_grad_(True)
    b = torch.rand(4, dtype=torch.float64).cuda().requires_grad_(True)
    assert gradcheck(_ModulatedDeformConv, (x, off, msk, w, b, 1, 1, 1, 2, 1, 64), eps=1e-6, atol=1e-5, rtol=1e-4, nondet_tol=0.0)
    assert gradcheck(_DeformConv, (x, off, w, b, 1, 1, 1, 2, 1, 64), eps=1e-6, atol=1e-5, rtol=1e-4, nondet_tol=0.0)


@pytest.mark.gpu
@pytest.mark.parametrize("scale", SCALES)
@pytest.mark.parametrize("tc", [1, 0])
def test_dcn_gradient_scale(scale, tc, deterministic):
    from rdfc_gan_b200 import _cabi as C
    inputs, geo = _dcn_inputs(TC_CASES[1], scale=scale)
    C.set_knob("RDFC_DCN_TC", tc)
    try:
        det = _dcn_bwd(inputs, geo)
        torch.use_deterministic_algorithms(False)
        ref = _dcn_bwd(inputs, geo)
    finally:
        C.set_knob("RDFC_DCN_TC", None)
    for a, r, tol in zip(det, ref, [2e-4, 5e-5, 5e-5, 5e-5, 5e-5]):
        assert torch.isfinite(a).all()
        _within(a, r, tol, floor=0.0)


@pytest.mark.gpu
@pytest.mark.parametrize("tc", [1, 0])
def test_dcn_zero_and_nan_gradients(tc, deterministic):
    from rdfc_gan_b200 import _cabi as C
    inputs, geo = _dcn_inputs(TC_CASES[1])
    C.set_knob("RDFC_DCN_TC", tc)
    try:
        inputs[-1] = torch.zeros_like(inputs[-1])
        for g in _dcn_bwd(inputs, geo):
            assert torch.equal(g, torch.zeros_like(g))
        inputs[-1][1, 3, 4, 5] = float("nan")
        assert not torch.isfinite(_dcn_bwd(inputs, geo)[0]).all()
    finally:
        C.set_knob("RDFC_DCN_TC", None)


# ---------------------------------------------------------------- host side ----------------------------------------------------
@pytest.mark.gpu
def test_flag_off_calls_the_old_entry_points():
    """Without the flag each backward launches what its old entry point launches; with it, the deterministic kernels."""
    from rdfc_gan_b200 import _cabi as C
    inputs, geo = _dcn_inputs(TC_CASES[1])
    counts = {}
    for det in (False, True):
        torch.use_deterministic_algorithms(det)
        try:
            n0 = C.launch_count()
            _dcn_bwd(inputs, geo)
            counts[det] = C.launch_count() - n0
        finally:
            torch.use_deterministic_algorithms(False)
    x, w, b, off, m, go = inputs
    from rdfc_gan_b200.dcn import DCN
    s = DCN._shape(x, w, *geo)
    outs = [torch.empty_like(v) for v in (x, off, m, w, b)]
    n0 = C.launch_count()
    C.check(C.lib.rdfc_dcn_backward(*[C.ptr(v) for v in (x, w, off, m, go, *outs)], s, C.F32, C.stream_ptr()))
    assert counts[False] == C.launch_count() - n0 and counts[True] > counts[False], counts
    f, o, a, fix, gout = _prop_full(1, False)
    for det in (False, True):
        torch.use_deterministic_algorithms(det)
        try:
            n0 = C.launch_count()
            _prop_grads(f, o, a, fix, 18, False, gout)
            counts[det] = C.launch_count() - n0
        finally:
            torch.use_deterministic_algorithms(False)
    # forward: 18 iterations; backward: 18 scatters + 2 (default) or 1 + 18 x (scatter, conversion) + 2 (deterministic)
    assert counts[False] == 18 + 18 + 2 and counts[True] == 18 + 1 + 2 * 18 + 2, counts


@pytest.mark.gpu
def test_unknown_flags_are_refused_before_launch():
    from rdfc_gan_b200 import _cabi as C
    inputs, geo = _dcn_inputs(TC_CASES[2])
    x, w, b, off, m, go = inputs
    from rdfc_gan_b200.dcn import DCN
    s = DCN._shape(x, w, *geo)
    outs = [torch.empty_like(v) for v in (x, off, w, b)]
    n0 = C.launch_count()
    for flags in (2, -1, 1 << 8):
        assert C.lib.rdfc_dcn_backward_ex(*[C.ptr(v) for v in (x, w, off, None, go, outs[0], outs[1], None, outs[2], outs[3])], s, C.F32,
                                          C.stream_ptr(), flags) != 0
        assert b"flags" in C.lib.rdfc_last_error()
        assert C.lib.rdfc_nlspn_propagate_backward_ex(*([None] * 7), 0, *([None] * 4), 1, 8, 8, 2, None, flags) != 0
        assert b"flags" in C.lib.rdfc_last_error()
        assert C.lib.rdfc_nlspn_affinity_backward_ex(*([None] * 5), 3, 1, *([None] * 6), 1, 8, 8, None, flags) != 0
        assert b"flags" in C.lib.rdfc_last_error()
    torch.cuda.synchronize()
    assert C.launch_count() == n0


# ---------------------------------------------------------------- the training step --------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["bf16", "fp32_tc"])
def test_training_step_reproducible_across_processes(precision):
    """Two fresh processes, each two optimize_parameters steps of the c4 composition (NLSPN TGASS with conf_prop and
    preserve_input, PatchGAN) at B = 2, 96x128 under the flag (torch fills uninitialised memory with NaN there, so a kernel that
    read memory it never wrote would show): the losses, every G / D parameter and the BatchNorm buffers hash the same."""
    env = dict(os.environ, CUBLAS_WORKSPACE_CONFIG=":4096:8")
    cmd = [sys.executable, os.path.join(HERE, "_det_step.py"), precision, "2", "96", "128", "2", "1"]
    digests = [subprocess.run(cmd, env=env, capture_output=True, text=True, check=True).stdout.strip().splitlines()[-1] for _ in range(2)]
    assert len(digests[0]) == 64 and digests[0] == digests[1], digests
