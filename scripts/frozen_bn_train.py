"""The c4 training step (bench.py config c4: RDFGAN step, RDFGenerator ResNet-18 x2 + W-AdaIN + NLSPN 18 it., PatchGAN, lsgan +
3 x L1, Adam, B = 16, 228x304, the bench's weights and inputs) with the generator's BatchNorms in train() mode and frozen, on one
GPU, in bf16 and fp32_tc.  Prints one JSON line and writes it to --out.

    python scripts/frozen_bn_train.py [--out profiles/r4_frozen_bn.json] [--reps 5] [--steps 5] [--warmup 3] [--batch 16]

Variants, alternated `reps` times in this one call per precision (each sample: `steps` optimize_parameters calls between two CUDA
events, medians):
  batch_stats    every BatchNorm in train(): batch statistics + running-statistics update (the step bench.py times)
  frozen_fused   every generator BatchNorm in eval() (frozen), folded into its tcgen05 conv (train_ops.conv_bn_act_frozen)
  frozen_torch   the same frozen BatchNorms as conv2d_nhwc -> F.batch_norm(training=False) -> residual / activation in PyTorch:
                 what a user could write without the fused op
fp32_tc runs with TF32 off throughout (the discriminator included), bf16 with torch's defaults, as scripts/train_precision.py.
Peak memory: torch.cuda.max_memory_allocated over one variant's sample.  Card name and power limit are read in the same call.
"""
import argparse
import json
import os
import statistics
import sys

import torch
import torch.nn as nn
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "scripts")):
    if p not in sys.path:
        sys.path.insert(0, p)

import rdfc_gan_b200.train_forward as tf  # noqa: E402
from rdfc_gan_b200 import _cabi as C  # noqa: E402
from train_precision import build, gpu_info  # noqa: E402

VARIANTS = ("batch_stats", "frozen_fused", "frozen_torch")


def frozen_torch(x, weight, bn, k=3, stride=1, transposed=False, residual=None, act=C.ACT_NONE):
    """conv_bn_act_frozen written with the repo's conv and PyTorch's eval-mode BatchNorm and activations"""
    y = tf.conv2d_nhwc(x, weight, k, stride, transposed).permute(0, 3, 1, 2)
    z = F.batch_norm(y, bn.running_mean, bn.running_var, bn.weight, bn.bias, False, 0.0, bn.eps).permute(0, 2, 3, 1)
    if residual is not None:
        z = z + residual
    return {C.ACT_NONE: z, C.ACT_RELU: F.relu(z), C.ACT_LEAKY02: F.leaky_relu(z, 0.2)}[act]


def set_variant(model, name, fused_op):
    for m in model.G.modules():
        if isinstance(m, nn.BatchNorm2d):
            m.train(name == "batch_stats")
    tf.conv_bn_act_frozen = frozen_torch if name == "frozen_torch" else fused_op


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r4_frozen_bn.json"))
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=16)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "frozen_bn_train.py measures on a GPU"
    fused_op = tf.conv_bn_act_frozen
    res = {"workload": f"c4 training step (RDFGAN.optimize_parameters), B = {args.batch}, 228x304; generator BatchNorms in train() "
                       f"vs frozen", **gpu_info(), "reps": args.reps, "steps": args.steps, "warmup": args.warmup}
    saved_tf32 = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    for prec in ("bf16", "fp32_tc"):
        model, batch = build(args.batch)
        model.G.set_train_precision(prec)
        if prec == "fp32_tc":
            torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False

        def steps(n):
            for _ in range(n):
                model.set_input(batch)
                stats = model.optimize_parameters()
            return stats
        try:
            for name in VARIANTS:                             # warm-up of every variant (cuDNN algorithm choice, allocator)
                set_variant(model, name, fused_op)
                stats = steps(args.warmup)
                assert all(float(v) == float(v) for v in stats.values()), (prec, name, stats)
            samples, peak = {n: [] for n in VARIANTS}, {}
            for _ in range(args.reps):
                for name in VARIANTS:
                    set_variant(model, name, fused_op)
                    torch.cuda.synchronize()
                    torch.cuda.reset_peak_memory_stats()
                    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    a.record()
                    steps(args.steps)
                    b.record()
                    torch.cuda.synchronize()
                    samples[name].append(a.elapsed_time(b) / args.steps)
                    peak[name] = max(peak.get(name, 0.0), torch.cuda.max_memory_allocated() / 2**30)
        finally:
            tf.conv_bn_act_frozen = fused_op
            torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = saved_tf32
        for name in VARIANTS:
            med = statistics.median(samples[name])
            res[f"{prec}:{name}"] = {"ms": round(med, 2), "spread_pct": round(100 * (max(samples[name]) - min(samples[name])) / med, 2),
                                     "peak_mem_gib": round(peak[name], 2)}
        del model, batch
        torch.cuda.empty_cache()
    res["gpu_after"] = gpu_info()
    line = json.dumps(res)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
