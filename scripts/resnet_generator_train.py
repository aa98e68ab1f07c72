"""G_B2A (ResnetGenerator, the depth -> RGB half of RDFC-GAN's cycle) forward + backward as the cycle runs it, on one GPU: the
default constructor (1 -> 3 channels, ngf 64, 6 residual blocks), B = 16, 228x304, seeded weights (tests/_synth.synth_state_dict),
train(), an input that needs its gradient (G_B2A reads G_A2B's fake depth) and an L1 loss against a seeded RGB target.  Prints one
JSON line and writes it to --out.

    python scripts/resnet_generator_train.py [--out profiles/r3_resnet_generator.json] [--reps 7] [--iters 5] [--warmup 3]

Variants, alternated `reps` times in this one call (each sample: `iters` forward + backward between two CUDA events, medians):
  bf16          set_train_precision('bf16'), the pads on train_ops.pad_nhwc (this change)
  bf16_fpad     bf16 with torch.nn.functional.pad on the channels-last view in place of pad_nhwc (the parent commit's composition)
  fp32_tc       set_train_precision('fp32_tc')
  fp32_torch    the fp32_tc walk with conv2d_nhwc / bn_act / pad_nhwc on fp32 PyTorch ops, TF32 off: what an fp32 user has without it
  bf16_det      bf16 under torch.use_deterministic_algorithms(True), torch.utils.deterministic.fill_uninitialized_memory = False
Peak memory: torch.cuda.max_memory_allocated over one variant's sample.  Card name and power limit are read in the same call.
"""
import os

os.environ.setdefault("CUBLAS_WORKSPACE_CONFIG", ":4096:8")

import argparse  # noqa: E402
import contextlib  # noqa: E402
import json  # noqa: E402
import statistics  # noqa: E402
import sys  # noqa: E402

import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "scripts")):
    if p not in sys.path:
        sys.path.insert(0, p)

import rdfc_gan_b200.resnet_generator as rg  # noqa: E402
from _fp32_ops import fp32_torch_ops  # noqa: E402
from _synth import synth_state_dict  # noqa: E402
from train_precision import gpu_info  # noqa: E402

VARIANTS = ("bf16", "bf16_fpad", "fp32_tc", "fp32_torch", "bf16_det")
B, H, W = 16, 228, 304


def torch_pad(x, pad, mode):
    p = (pad,) * 4 if isinstance(pad, int) else tuple(pad)
    return F.pad(x.permute(0, 3, 1, 2), p, mode=mode).permute(0, 2, 3, 1)


@contextlib.contextmanager
def variant(G, name):
    saved = (rg.conv2d_nhwc, rg.bn_act, rg.pad_nhwc, torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32,
             torch.utils.deterministic.fill_uninitialized_memory)
    G.set_train_precision('fp32_tc' if name in ("fp32_tc", "fp32_torch") else 'bf16')
    if name == "bf16_fpad":
        rg.pad_nhwc = torch_pad
    if name == "fp32_torch":
        rg.conv2d_nhwc, rg.bn_act = fp32_torch_ops()
        rg.pad_nhwc = torch_pad
        torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    if name == "bf16_det":
        torch.use_deterministic_algorithms(True)
        torch.utils.deterministic.fill_uninitialized_memory = False
    try:
        yield
    finally:
        torch.use_deterministic_algorithms(False)
        (rg.conv2d_nhwc, rg.bn_act, rg.pad_nhwc, torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32,
         torch.utils.deterministic.fill_uninitialized_memory) = saved
        G.set_train_precision('bf16')


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_resnet_generator.json"))
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "resnet_generator_train.py measures on a GPU"
    info = gpu_info()
    G = rg.ResnetGenerator(input_channels=1, output_channels=3, ngf=64, n_blocks=6)
    G.load_state_dict(synth_state_dict(G, seed=0, recipe="scaled"))
    G = G.cuda().train()
    gen = torch.Generator(device="cuda").manual_seed(0)
    x = (torch.rand(B, 1, H, W, device="cuda", generator=gen) * 2 - 1).requires_grad_(True)
    rgb = torch.rand(B, 3, H, W, device="cuda", generator=gen) * 2 - 1

    def fwd_bwd():
        G.zero_grad(set_to_none=True)
        x.grad = None
        y = G(x)
        (y - rgb).abs().mean().backward()
        return y

    outs = {}
    for name in VARIANTS:                                    # warm-up of every variant (cuDNN algorithm choice, allocator)
        with variant(G, name):
            for _ in range(args.warmup):
                y = fwd_bwd()
            assert torch.isfinite(y).all() and torch.isfinite(x.grad).all(), name
            if name in ("bf16", "bf16_fpad"):
                with torch.no_grad():
                    outs[name] = G(x)
    samples = {n: [] for n in VARIANTS}
    peak = {}
    for _ in range(args.reps):
        for name in VARIANTS:
            with variant(G, name):
                torch.cuda.synchronize()
                torch.cuda.reset_peak_memory_stats()
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                for _ in range(args.iters):
                    fwd_bwd()
                b.record()
                torch.cuda.synchronize()
                samples[name].append(a.elapsed_time(b) / args.iters)
                peak[name] = max(peak.get(name, 0.0), torch.cuda.max_memory_allocated() / 2**30)
    res = {"workload": f"ResnetGenerator(1, 3, ngf=64, n_blocks=6) train() forward + backward (input gradient included), B = {B}, {H}x{W}",
           **info, "reps": args.reps, "iters": args.iters, "warmup": args.warmup,
           "bf16_forward_bits_equal_to_fpad": bool(torch.equal(outs["bf16"], outs["bf16_fpad"]))}
    for name in VARIANTS:
        med = statistics.median(samples[name])
        res[name] = {"ms": round(med, 3), "spread_pct": round(100 * (max(samples[name]) - min(samples[name])) / med, 2),
                     "peak_mem_gib": round(peak[name], 2)}
    res["gpu_after"] = gpu_info()
    line = json.dumps(res)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
