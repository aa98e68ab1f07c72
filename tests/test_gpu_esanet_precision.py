"""-m gpu: the ESANet guidance network's fp32 modes ('fp32': CUDA-core fp32, 'fp32_tc': tensor cores with split fp16 operands).
The glue kernels in fp32 against torch fp64; the network against the reference's outputs (tests/golden/esanet_*.npz) and the CPU
oracle (oracle/esanet.py); precision switching; RDF-GAN (DCVGANGenerator + ESANet-34) end to end in fp32 against the CPU
composition oracle.esanet -> oracle.generator."""
import ctypes
import json
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

# ESANet logits against the reference / the oracle, relative to the RMS of the reference's logits: (RMSE, max-abs).  Twice the
# largest error measured on a B200 over the goldens and the oracle shapes below (fp32: 2.4e-6 / 2.5e-5; fp32_tc: 1.7e-4 / 1.5e-3).
ESANET_BOUND = {"fp32": (5e-6, 5e-5), "fp32_tc": (3.5e-4, 3e-3)}
# RDF-GAN end to end in fp32 (guidance network and generator), max-abs per map against oracle.esanet -> oracle.generator: twice
# the error measured on a B200.  NOT the north-star 1e-4: on this input (guidance logits of RMS 10, max 71) the generator's RGB
# decoder carries activations up to 8e6, and the fp32 CPU oracle itself lands 0.076 from an fp64 run of it on depth_map_1, so no fp32
# implementation meets 1e-4 there.  The guidance network's own share is within ESANET_BOUND (DESIGN.md section 7, rank 2).
RDFGAN_FP32_BOUND = {"depth_map_1": 0.7, "confidence_map_1": 0.19, "depth_map_2": 0.046, "confidence_map_2": 6e-5, "pred_depth": 0.35}
# RDF-GAN in fp32_tc (guidance network and generator) against the same pipeline in strict fp32 on that input, RMSE per map: twice
# the distance measured on a B200.  RMSE, not max-abs: on this ill-conditioned input single pixels of the tanh / clamped maps differ
# by up to 1.96 (fp32_tc's contractions are ~1e-5 relative where fp32's are ~1e-7), so a max-abs bound would not constrain them.
RDFGAN_FP32_TC_BOUND = {"depth_map_1": 0.034, "confidence_map_1": 0.006, "depth_map_2": 0.091, "confidence_map_2": 1.6e-4, "pred_depth": 0.057}
KEYS = ("depth_map_1", "confidence_map_1", "depth_map_2", "confidence_map_2", "pred_depth")
NL = dict(prop_kernel=3, prop_time=18, affinity="TGASS", affinity_gamma=0.5, conf_prop=True, preserve_input=False)


def _dump(case, errs):
    if os.environ.get("RDFC_DUMP_PARITY"):
        with open(os.environ["RDFC_DUMP_PARITY"], "a") as f:
            f.write(json.dumps({"case": case, "errs": errs}) + "\n")


def _rel(got, want, rms):
    d = (got.float().cpu() - want.float().cpu()).double()
    return float(d.square().mean().sqrt()) / rms, float(d.abs().max()) / rms


def _esanet(case, seed, **size):
    from make_esanet_golden import ESANET_CASES, esanet_weights
    from rdfc_gan_b200.esanet import ESANetOneModality
    net = ESANetOneModality(**dict(ESANET_CASES[case]["kw"], **size)).eval()
    sd = esanet_weights(net, seed)
    net.load_state_dict(sd)
    return net.cuda(), sd


# ---------------------------------------------------------------------------------------------------------- kernels
@pytest.mark.parametrize("case", [(2, 3, 228, 304), (1, 3, 37, 50), (3, 1, 64, 33), (2, 4, 17, 129)])
def test_first_conv_fp32(case):
    """encoder.conv1 + bn1 + ReLU to fp32 NHWC: the register-tiled kernel and the plain one against F.conv2d in fp64.  The two sum
    the 49 Cin products in different orders (channel outermost / innermost), so they agree to fp32 rounding, not bit for bit."""
    from rdfc_gan_b200 import _cabi as C
    B, Cin, H, W = case
    g = torch.Generator(device="cuda").manual_seed(sum(case))
    x = torch.randn(B, Cin, H, W, device="cuda", generator=g)
    w = torch.randn(64, Cin, 7, 7, device="cuda", generator=g) / (7 * Cin ** 0.5)
    sc, sh = torch.rand(64, device="cuda", generator=g) + 0.5, torch.randn(64, device="cuda", generator=g) * 0.1
    Ho, Wo = (H + 6 - 7) // 2 + 1, (W + 6 - 7) // 2 + 1
    want = torch.relu(F.conv2d(x.double(), w.double(), None, 2, 3) * sc.double()[None, :, None, None] + sh.double()[None, :, None, None])
    tol = 1e-5 * max(1.0, float(want.abs().max()))
    try:
        for fast in (1, 0):
            if not fast and Cin == 4:            # the plain kernel keeps the filter bank in 48 KB of shared memory (Cin <= 3)
                continue
            C.set_knob("RDFC_FIRSTCONV_FAST", fast)
            out = torch.full((B, Ho, Wo, 64), float("nan"), device="cuda")
            v = C.view(out)
            C.check(C.lib.rdfc_first_conv_forward(C.ptr(x), B, Cin, H, W, C.ptr(w), 7, 2, 3, C.ptr(sc), C.ptr(sh), 1, ctypes.byref(v), C.stream_ptr()))
            torch.cuda.synchronize()
            err = float((out.double().permute(0, 3, 1, 2) - want).abs().max())
            assert err <= tol, (fast, err)
    finally:
        C.set_knob("RDFC_FIRSTCONV_FAST", None)


@pytest.mark.parametrize("case", [(2, 64, 114, 152), (3, 64, 37, 51), (1, 128, 15, 8)])
def test_pooling_kernels_fp32(case):
    """max pool 3x3/2, adaptive average pooling (bins 1, 2, 5, 8) and nearest up-sampling into a channel slice, fp32 NHWC"""
    from rdfc_gan_b200 import _cabi as C
    B, Cc, H, W = case
    g = torch.Generator(device="cuda").manual_seed(sum(case))
    x = torch.randn(B, H, W, Cc, device="cuda", generator=g)
    xn = x.permute(0, 3, 1, 2).double()
    s = C.stream_ptr()
    Ho, Wo = (H - 1) // 2 + 1, (W - 1) // 2 + 1
    out = torch.full((B, Ho, Wo, Cc), float("nan"), device="cuda")
    vx, vo = C.view(x), C.view(out)
    C.check(C.lib.rdfc_maxpool3x3s2_forward(ctypes.byref(vx), ctypes.byref(vo), B, H, W, s))
    torch.cuda.synchronize()
    assert torch.equal(out.permute(0, 3, 1, 2).double(), F.max_pool2d(xn, 3, 2, 1))
    for bins in (1, 2, 5, 8):
        pooled = torch.full((B, bins, bins, Cc), float("nan"), device="cuda")
        vp = C.view(pooled)
        C.check(C.lib.rdfc_adaptive_avgpool_forward(ctypes.byref(vx), ctypes.byref(vp), B, H, W, bins, s))
        torch.cuda.synchronize()
        want = F.adaptive_avg_pool2d(xn, bins)
        assert float((pooled.permute(0, 3, 1, 2).double() - want).abs().max()) <= 1e-5, bins           # means of unit normals
        # nearest up-sampling of the pooled map into channels [8, 8 + Cc) of a wider buffer
        cat = torch.full((B, H, W, Cc + 16), float("nan"), device="cuda")
        vd = C.view(cat, Cc, 8)
        C.check(C.lib.rdfc_upsample_nearest_forward(ctypes.byref(vp), ctypes.byref(vd), B, bins, bins, H, W, s))
        torch.cuda.synchronize()
        up = F.interpolate(pooled.permute(0, 3, 1, 2), size=(H, W), mode="nearest")
        assert torch.equal(cat[..., 8:8 + Cc].permute(0, 3, 1, 2), up), bins
        assert torch.isnan(cat[..., :8]).all() and torch.isnan(cat[..., 8 + Cc:]).all()


@pytest.mark.parametrize("case", [(2, 40, 114, 152, 228, 304, False, True), (2, 40, 29, 38, 57, 76, True, True), (3, 128, 29, 38, 57, 76, True, False),
                                  (1, 64, 15, 19, 29, 38, False, False), (2, 40, 20, 31, 64, 65, False, True), (2, 40, 20, 31, 64, 65, True, False)])
def test_learned_upsampling_fp32(case):
    """The decoder's learned up-sampling from an fp32 NHWC input (+ fp32 skip) to fp32 NHWC or fp32 NCHW: the restructured kernels
    equal the plain one (RDFC_UPSAMPLE_FAST = 0) bit for bit, and both match torch in fp64."""
    from rdfc_gan_b200 import _cabi as C
    B, Cc, Hi, Wi, Ho, Wo, with_skip, nchw = case
    g = torch.Generator(device="cuda").manual_seed(sum(case[:6]))
    x = torch.randn(B, Hi, Wi, Cc, device="cuda", generator=g)
    w = torch.randn(Cc, 1, 3, 3, device="cuda", generator=g) * 0.3
    bias = torch.randn(Cc, device="cuda", generator=g) * 0.1
    skip = torch.randn(B, Ho, Wo, Cc, device="cuda", generator=g) if with_skip else None
    up = F.interpolate(x.double().permute(0, 3, 1, 2), size=(Ho, Wo), mode="nearest")
    want = F.conv2d(up, w.double(), bias.double(), padding=1, groups=Cc)
    if with_skip:
        want = want + skip.double().permute(0, 3, 1, 2)
    outs = []
    try:
        for fast in (1, 0):
            C.set_knob("RDFC_UPSAMPLE_FAST", fast)
            vx, vs = C.view(x), C.view(skip)
            vsp = ctypes.byref(vs) if with_skip else None
            if nchw:
                out = torch.full((B, Cc, Ho, Wo), float("nan"), device="cuda")
                C.check(C.lib.rdfc_upsample_dw_forward(ctypes.byref(vx), C.ptr(w), C.ptr(bias), vsp, None, C.ptr(out), B, Hi, Wi, Ho, Wo,
                                                       C.stream_ptr()))
                got = out
            else:
                out = torch.full((B, Ho, Wo, Cc), float("nan"), device="cuda")
                vo = C.view(out)
                C.check(C.lib.rdfc_upsample_dw_forward(ctypes.byref(vx), C.ptr(w), C.ptr(bias), vsp, ctypes.byref(vo), None, B, Hi, Wi, Ho, Wo,
                                                       C.stream_ptr()))
                got = out.permute(0, 3, 1, 2)
            torch.cuda.synchronize()
            outs.append(got.clone())
            err = float((got.double() - want).abs().max())
            assert err <= 1e-5 * max(1.0, float(want.abs().max())), (fast, err)
    finally:
        C.set_knob("RDFC_UPSAMPLE_FAST", None)
    assert torch.equal(outs[0], outs[1]), "same arithmetic order: the restructured kernels must reproduce the plain one bit for bit"


def test_glue_kernels_reject_mixed_dtypes():
    from rdfc_gan_b200 import _cabi as C
    s = C.stream_ptr()
    x32 = torch.zeros(1, 8, 8, 16, device="cuda")
    x16 = torch.zeros(1, 8, 8, 16, device="cuda", dtype=torch.bfloat16)
    o16 = torch.zeros(1, 4, 4, 16, device="cuda", dtype=torch.bfloat16)
    u16 = torch.zeros(1, 16, 16, 16, device="cuda", dtype=torch.bfloat16)
    u32 = torch.zeros(1, 16, 16, 16, device="cuda")
    w, b = torch.zeros(16, 9, device="cuda"), torch.zeros(16, device="cuda")
    v32, v16, vo16, vu16, vu32 = C.view(x32), C.view(x16), C.view(o16), C.view(u16), C.view(u32)
    calls = [lambda: C.lib.rdfc_maxpool3x3s2_forward(ctypes.byref(v32), ctypes.byref(vo16), 1, 8, 8, s),
             lambda: C.lib.rdfc_adaptive_avgpool_forward(ctypes.byref(v32), ctypes.byref(vo16), 1, 8, 8, 4, s),
             lambda: C.lib.rdfc_upsample_nearest_forward(ctypes.byref(v32), ctypes.byref(vu16), 1, 8, 8, 16, 16, s),
             lambda: C.lib.rdfc_upsample_dw_forward(ctypes.byref(v32), C.ptr(w), C.ptr(b), None, ctypes.byref(vu16), None, 1, 8, 8, 16, 16, s),
             lambda: C.lib.rdfc_upsample_dw_forward(ctypes.byref(v16), C.ptr(w), C.ptr(b), ctypes.byref(vu32), ctypes.byref(vu16), None,
                                                    1, 8, 8, 16, 16, s)]
    for i, call in enumerate(calls):
        assert call() == -1, i                   # RDFC_ERR_INVALID
        assert b"dtype" in C.lib.rdfc_last_error(), i


# ---------------------------------------------------------------------------------------------------------- network
@pytest.mark.parametrize("precision", ["fp32", "fp32_tc"])
@pytest.mark.parametrize("name", ["r18_small", "r34_full"])
def test_esanet_fp32_against_reference(name, precision, golden_dir):
    from make_esanet_golden import ESANET_CASES, esanet_input
    from _synth import state_dict_digest
    c = ESANET_CASES[name]
    gold = np.load(f"{golden_dir}/esanet_{name}.npz")
    net, sd = _esanet(name, c["seed"])
    assert state_dict_digest(sd) == int(gold["digest"][0])
    assert net.set_precision(precision) is net and net.precision == precision
    x = esanet_input(c).cuda()
    y = net(x)
    assert y.dtype == torch.float32
    got = y[:, :, ::c["stride"], ::c["stride"]]
    rmse, mx = _rel(got, torch.from_numpy(gold["logits"]), float(gold["rms"]))
    _dump(f"esanet_{precision}:{name}", {"rel_rmse": rmse, "rel_max": mx})
    bound = ESANET_BOUND[precision]
    assert rmse <= bound[0] and mx <= bound[1], (rmse, mx)
    assert torch.equal(net(x), y)                  # graph replay


@pytest.mark.parametrize("precision", ["fp32", "fp32_tc"])
@pytest.mark.parametrize("name,B,H,W", [("r18_small", 3, 37, 50), ("r18_small", 3, 64, 33), ("r34_full", 3, 37, 50), ("r34_full", 3, 64, 33)])
def test_esanet_fp32_against_oracle(name, B, H, W, precision):
    """Shapes the goldens lack (B = 3, odd level sizes) against the CPU oracle, relative to the oracle's logits' RMS"""
    from oracle.esanet import esanet_forward
    net, sd = _esanet(name, 7 + H + W, height=H, width=W)
    g = torch.Generator().manual_seed(H * W)
    x = torch.rand(B, 3, H, W, generator=g) * 2 - 1
    ref = esanet_forward(sd, x)
    y = net.set_precision(precision)(x.cuda())
    assert y.shape == ref.shape
    rmse, mx = _rel(y, ref, float(ref.square().mean().sqrt()))
    _dump(f"esanet_{precision}:oracle_{name}_{B}x{H}x{W}", {"rel_rmse": rmse, "rel_max": mx})
    bound = ESANET_BOUND[precision]
    assert rmse <= bound[0] and mx <= bound[1], (rmse, mx)


def test_esanet_precision_switching():
    """bf16 -> fp32 -> fp32_tc -> bf16 reproduces the bf16 logits bit for bit; an in-place weight change reaches an fp32 plan;
    an unknown precision raises."""
    from make_esanet_golden import ESANET_CASES, esanet_input
    from oracle.esanet import esanet_forward
    net, _ = _esanet("r18_small", 42)
    assert net.precision == "bf16"
    x = esanet_input(ESANET_CASES["r18_small"]).cuda()
    y16 = net(x)
    y32 = net.set_precision("fp32")(x)
    ytc = net.set_precision("fp32_tc")(x)
    assert torch.equal(net.set_precision("bf16")(x), y16)
    assert not torch.equal(y32, y16) and not torch.equal(ytc, y32)
    net.set_precision("fp32")
    with torch.no_grad():
        net.decoder.conv_out.bias.add_(1.0)
        net.encoder.layer2[0].bn1.running_mean.mul_(0.5)
    y32b = net(x)
    ref = esanet_forward(net.state_dict(), x.cpu())
    rmse, mx = _rel(y32b, ref, float(ref.square().mean().sqrt()))
    assert mx <= ESANET_BOUND["fp32"][1], mx
    assert float((y32b - y32).abs().max()) > 1e-2
    for bad in ("fp16", "FP32", None):
        with pytest.raises(ValueError):
            net.set_precision(bad)
    assert net.precision == "fp32"


# ---------------------------------------------------------------------------------------------------------- RDF-GAN
def _rdfgan_c2(seed):
    """DCVGANGenerator(ESANet-34) in the configuration of F/bash/test_nyuv2_Ts2T.sh: ResNet-34 encoders, adain_weighting,
    40 classes; generator weights of the 'scaled' recipe, the guidance network's those of tests/golden/make_esanet_golden.py"""
    from make_esanet_golden import ESANET_CASES, esanet_weights
    from _synth import synth_state_dict
    from rdfc_gan_b200.esanet import ESANetOneModality
    from rdfc_gan_b200.generator import DCVGANGenerator
    esa = ESANetOneModality(**ESANET_CASES["r34_full"]["kw"]).eval()
    esa.load_state_dict(esanet_weights(esa, 41))
    kw = dict(encoder_rgb="resnet34", encoder_depth="resnet34", pretrained_on_imagenet=False, semantic_channels_in=40, adain_weighting=True,
              use_nlpsn_refine=True, nlspn_configs=NL)
    G = DCVGANGenerator(esa, **kw).eval()
    sd = synth_state_dict(G, seed=seed, recipe="scaled", nlspn_stress=True)
    for k in list(sd):
        if k.startswith("global_guidance_module."):
            sd[k] = G.state_dict()[k]
    G.load_state_dict(sd)
    return G.cuda(), kw


def _rdfgan_errors(precision):
    """RDF-GAN at 228x304, guidance network and generator both in `precision`, against the CPU composition oracle.esanet ->
    oracle.generator; per stage: the guidance logits against the oracle, and the generator against the oracle fed the GPU's own
    guidance (reported to RDFC_DUMP_PARITY)."""
    from _synth import synth_inputs
    from oracle import generator as ogen
    from oracle.esanet import esanet_forward
    G, kw = _rdfgan_c2(7)
    esa = G.global_guidance_module
    rgb, _, depth = synth_inputs(1, 228, 304, seed=7)
    sd = {k: v.cpu() for k, v in G.state_dict().items()}
    esa_sd = {k[len("global_guidance_module."):]: v for k, v in sd.items() if k.startswith("global_guidance_module.")}
    gen_sd = {k: v for k, v in sd.items() if not k.startswith("global_guidance_module.")}
    guid_ref = esanet_forward(esa_sd, rgb)
    grms = float(guid_ref.square().mean().sqrt())
    ref = ogen.generator_forward(gen_sd, guid_ref, depth, adain_weighting=True, use_nlspn_refine=True, nlspn_configs=NL)
    rgb_d, depth_d = rgb.cuda(), depth.cuda()
    G.set_precision(precision)
    esa.set_precision(precision)
    with torch.no_grad():
        outs = dict(zip(KEYS, G(rgb_d, depth_d)))
        guid = esa(rgb_d)
    errs = {k: float((outs[k].cpu() - ref[k]).abs().max()) for k in KEYS}
    g_rmse, g_max = _rel(guid, guid_ref, grms)
    ref_given = ogen.generator_forward(gen_sd, guid.cpu(), depth, adain_weighting=True, use_nlspn_refine=True, nlspn_configs=NL)
    gen_errs = {k: float((outs[k].cpu() - ref_given[k]).abs().max()) for k in KEYS}
    _dump(f"rdfgan_{precision}:c2_228x304", {"end_to_end_max_abs": errs, "guidance_rel_rmse": g_rmse, "guidance_rel_max": g_max,
                                               "guidance_rms": grms, "generator_given_guidance_max_abs": gen_errs})
    return G, kw, gen_sd, (rgb_d, depth_d), errs, (g_rmse, g_max), outs


def test_rdfgan_fp32_end_to_end():
    """RDF-GAN in strict fp32 end to end against the CPU composition (bounds above); G(rgb, d) equals G2(esa(rgb), d) bit for bit"""
    from rdfc_gan_b200.generator import DCVGANGenerator
    G, kw, gen_sd, (rgb_d, depth_d), errs, (g_rmse, g_max), outs = _rdfgan_errors("fp32")
    assert g_rmse <= ESANET_BOUND["fp32"][0] and g_max <= ESANET_BOUND["fp32"][1], (g_rmse, g_max)
    assert all(errs[k] <= RDFGAN_FP32_BOUND[k] for k in KEYS), errs
    G2 = DCVGANGenerator(torch.nn.Identity(), **kw).eval()
    G2.load_state_dict(gen_sd)
    G2 = G2.cuda().set_precision("fp32")
    with torch.no_grad():
        ref2 = G2(G.global_guidance_module(rgb_d), depth_d)
    assert all(torch.equal(outs[k], b) for k, b in zip(KEYS, ref2))


def test_rdfgan_fp32_tc_end_to_end():
    """RDF-GAN in fp32_tc end to end on the input that drives the RGB decoder to activations of 8e6, beyond fp16's 65504 (every split
    input is scaled by a power of two of its own first): finite maps, the guidance within ESANET_BOUND of the oracle, and every map
    within RDFGAN_FP32_TC_BOUND (RMSE) of the same pipeline in strict fp32"""
    G, _, _, (rgb_d, depth_d), errs, (g_rmse, g_max), outs = _rdfgan_errors("fp32_tc")
    assert g_rmse <= ESANET_BOUND["fp32_tc"][0] and g_max <= ESANET_BOUND["fp32_tc"][1], (g_rmse, g_max)
    outs = {k: v.clone() for k, v in outs.items()}
    assert all(bool(torch.isfinite(outs[k]).all()) for k in KEYS), errs
    G.set_precision("fp32")
    G.global_guidance_module.set_precision("fp32")
    with torch.no_grad():
        ref = dict(zip(KEYS, G(rgb_d, depth_d)))
    dist = {k: float((outs[k] - ref[k]).double().square().mean().sqrt()) for k in KEYS}
    _dump("rdfgan_fp32_tc:c2_228x304_vs_fp32", {"rmse": dist, "max_abs": {k: float((outs[k] - ref[k]).abs().max()) for k in KEYS}})
    assert all(dist[k] <= RDFGAN_FP32_TC_BOUND[k] for k in KEYS), dist


def test_stream_with_fp32_guidance():
    """G.stream() runs an fp32 guidance module inside its pipeline: exactly forward()'s outputs"""
    from make_esanet_golden import ESANET_CASES, esanet_weights
    from _synth import synth_inputs, synth_state_dict
    from rdfc_gan_b200.esanet import ESANetOneModality
    from rdfc_gan_b200.generator import DCVGANGenerator
    esa = ESANetOneModality(**dict(ESANET_CASES["r18_small"]["kw"], height=64, width=96)).eval()
    esa.load_state_dict(esanet_weights(esa, 3))
    G = DCVGANGenerator(esa, pretrained_on_imagenet=False, semantic_channels_in=40, use_nlpsn_refine=True, nlspn_configs=NL).eval()
    sd = synth_state_dict(G, seed=4, recipe="scaled", nlspn_stress=True)
    for k in list(sd):
        if k.startswith("global_guidance_module."):
            sd[k] = G.state_dict()[k]
    G.load_state_dict(sd)
    G = G.cuda().set_precision("fp32")
    G.global_guidance_module.set_precision("fp32")
    batches = [synth_inputs(2, 64, 96, seed=s) for s in (5, 6, 5)]
    with torch.no_grad():
        want = [G(rgb.cuda(), depth.cuda()) for rgb, _, depth in batches]
    got = [{k: o[k].clone() for k in KEYS} for o in G.stream(iter([(rgb.pin_memory(), depth.pin_memory()) for rgb, _, depth in batches]),
                                                            outputs=KEYS)]
    assert len(got) == 3
    for i, w in enumerate(want):
        for k, t in zip(KEYS, w):
            assert torch.equal(got[i][k], t.cpu()), (i, k)
