"""Cost of bit-reproducible training (torch.use_deterministic_algorithms -> the RDFC_DETERMINISTIC backwards) on one GPU.
Prints one JSON line and writes it to --out.

    python scripts/train_determinism.py [--out profiles/r3_train_determinism.json] [--reps 5] [--steps 5]

Per op, default (flags 0) against deterministic (flags RDFC_DETERMINISTIC), medians of CUDA-event timings of single calls
through the *_ex entry points: the NLSPN propagation backward (B = 16, 228x304, 18 iterations, stress offsets sigma ~ 2.2 px),
the affinity backward (same size, TGASS, conf_prop) and the DCN backward at the reference's example shape (deformconv/test.py:
64 -> 128 channels, 128x128, 3x3, 2 deformable groups, mask; B = 2 and 16) on the tensor-core path.
The c4 step (bench.py config c4's composition: RDFGAN.optimize_parameters, B = 16, 228x304, bf16): flag off, flag on, and flag
on with torch.utils.deterministic.fill_uninitialized_memory = False, alternating the variants `reps` times; each sample is
`steps` steps between two CUDA events.  CUBLAS_WORKSPACE_CONFIG=:4096:8 for every variant (the flag requires it of cuBLAS).
Reproducibility: two steps from the same seeded weights and batch under the flag, hashed (tests/_det_step.py)."""
import os

os.environ.setdefault("CUBLAS_WORKSPACE_CONFIG", ":4096:8")

import argparse  # noqa: E402
import json  # noqa: E402
import statistics  # noqa: E402
import sys  # noqa: E402

import numpy as np  # noqa: E402
import torch  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

import _det_step  # noqa: E402
from train_precision import gpu_info  # noqa: E402


def timed(fn, reps, warmup=3):
    for _ in range(warmup):
        fn()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return statistics.median(ts)


def both(call, reps):
    """median ms of call(flags) for flags 0 and RDFC_DETERMINISTIC, alternating"""
    from rdfc_gan_b200 import _cabi as C
    out = {"default": [], "deterministic": []}
    for _ in range(reps):
        out["default"].append(timed(lambda: call(0), 5))
        out["deterministic"].append(timed(lambda: call(C.DETERMINISTIC), 5))
    r = {k: round(statistics.median(v), 4) for k, v in out.items()}
    r["ratio"] = round(r["deterministic"] / r["default"], 3)
    return r


def nlspn_ops(B, reps):
    from oracle import nlspn as onl
    from _synth import nlspn_stress_inputs
    from rdfc_gan_b200 import _cabi as C
    H, W, T = 228, 304, 18
    x = nlspn_stress_inputs(2, 32, 40, 21)
    off, aff = onl.get_offset_affinity(x["guidance"], x["confidence"], x["conv_w"], x["conv_b"], np.array([4.0], np.float32))[:2]
    rep = lambda v: torch.from_numpy(np.ascontiguousarray(v, np.float32)).cuda().repeat(B // 2, 1, 8, 8)[:B, :, :H, :W].contiguous()
    off, aff = rep(off), rep(aff)
    guid, conf = rep(x["guidance"]), rep(x["confidence"])
    gen = torch.Generator(device="cuda").manual_seed(5)
    f = torch.randn(B, 1, H, W, device="cuda", generator=gen)
    gout = torch.randn(B, 1, H, W, device="cuda", generator=gen)
    out, scr = torch.empty_like(f), torch.empty_like(f)
    inter = torch.empty((T, B, 1, H, W), device="cuda")
    C.check(C.lib.rdfc_nlspn_propagate_forward(C.ptr(f), C.ptr(off), C.ptr(aff), None, 0, C.ptr(out), C.ptr(scr), C.ptr(inter),
                                               B, H, W, T, 0, None, C.stream_ptr()))
    g_feat, g_off, g_aff = torch.empty_like(f), torch.empty_like(off), torch.empty_like(aff)
    scratch = torch.empty((T + 1, B, 1, H, W), device="cuda")
    prop = lambda flags: C.check(C.lib.rdfc_nlspn_propagate_backward_ex(
        C.ptr(gout), None, C.ptr(f), C.ptr(inter), C.ptr(off), C.ptr(aff), None, 0, C.ptr(g_feat), C.ptr(g_off), C.ptr(g_aff),
        C.ptr(scratch), B, H, W, T, C.stream_ptr(), flags))
    w = torch.from_numpy(x["conv_w"]).cuda()
    b = torch.from_numpy(x["conv_b"]).cuda()
    scale = torch.tensor([4.0], device="cuda")
    ga, go = torch.randn(B, 9, H, W, device="cuda", generator=gen), torch.randn(B, 18, H, W, device="cuda", generator=gen)
    g_conv, g_conf, g_scale = torch.empty(B, 24, H, W, device="cuda"), torch.empty_like(f), torch.empty(1, device="cuda")
    affb = lambda flags: C.check(C.lib.rdfc_nlspn_affinity_backward_ex(
        C.ptr(guid), C.ptr(conf), C.ptr(w), C.ptr(b), C.ptr(scale), C.AFFINITY["TGASS"], 1, C.ptr(off), C.ptr(go), C.ptr(ga),
        C.ptr(g_conv), C.ptr(g_conf), C.ptr(g_scale), B, H, W, C.stream_ptr(), flags))
    return {f"nlspn_propagate_backward_B{B}": both(prop, reps), f"nlspn_affinity_backward_B{B}": both(affb, reps)}


def dcn_op(B, reps):
    from rdfc_gan_b200 import _cabi as C
    from rdfc_gan_b200.dcn import DCN
    Cin, Cout, H, W, k, dg = 64, 128, 128, 128, 3, 2
    gen = torch.Generator(device="cuda").manual_seed(0)
    x = torch.randn(B, Cin, H, W, device="cuda", generator=gen)
    w = torch.randn(Cout, Cin, k, k, device="cuda", generator=gen) * 0.1
    bias = torch.zeros(Cout, device="cuda")
    off = torch.randn(B, dg * 2 * k * k, H, W, device="cuda", generator=gen) * 2.0
    m = torch.rand(B, dg * k * k, H, W, device="cuda", generator=gen)
    go = torch.randn(B, Cout, H, W, device="cuda", generator=gen)
    s = DCN._shape(x, w, k, k, 1, 1, 1, 1, 1, 1, 1, dg, 64)
    outs = [torch.empty_like(v) for v in (x, off, m, w, bias)]
    call = lambda flags: C.check(C.lib.rdfc_dcn_backward_ex(*[C.ptr(v) for v in (x, w, off, m, go, *outs)], s, C.F32, C.stream_ptr(), flags))
    return {f"dcn_backward_B{B}": both(call, reps)}


def c4_step(reps, steps, B=16):
    model, batch = _det_step.build(B, 228, 304, "bf16")
    variants = {"off": (False, True), "on": (True, True), "on_no_fill": (True, False)}
    fill0 = torch.utils.deterministic.fill_uninitialized_memory
    samples = {k: [] for k in variants}
    try:
        for r in range(reps + 1):                       # the first round warms every variant up and is dropped
            for name, (det, fill) in variants.items():
                torch.use_deterministic_algorithms(det)
                torch.utils.deterministic.fill_uninitialized_memory = fill
                model.set_input(batch)
                model.optimize_parameters()
                torch.cuda.synchronize()
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                for _ in range(steps):
                    model.set_input(batch)
                    stats = model.optimize_parameters()
                b.record()
                torch.cuda.synchronize()
                assert all(v == v for v in stats.values()), (name, stats)
                if r:
                    samples[name].append(a.elapsed_time(b) / steps)
    finally:
        torch.use_deterministic_algorithms(False)
        torch.utils.deterministic.fill_uninitialized_memory = fill0
    res = {k: {"ms_per_step": round(statistics.median(v), 3), "spread": round((max(v) - min(v)) / statistics.median(v), 4),
               "images_per_s": round(B * 1000 / statistics.median(v), 1)} for k, v in samples.items()}
    for k in ("on", "on_no_fill"):
        res[k]["overhead"] = round(res[k]["ms_per_step"] / res["off"]["ms_per_step"] - 1, 4)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_train_determinism.json"))
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--steps", type=int, default=5)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a GPU"
    res = dict(gpu_info(), ops={}, cublas_workspace_config=os.environ["CUBLAS_WORKSPACE_CONFIG"])
    res["ops"].update(nlspn_ops(16, args.reps))
    for B in (2, 16):
        res["ops"].update(dcn_op(B, args.reps))
    res["c4_step_B16"] = c4_step(args.reps, args.steps)
    hashes = [_det_step.run("bf16", 16, 228, 304, 1) for _ in range(2)]
    res["reproducibility"] = {"c4_step_B16_bf16_sha256": hashes, "identical": hashes[0] == hashes[1]}
    line = json.dumps(res)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
