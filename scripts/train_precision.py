"""The training step in each arithmetic (bench.py config c4: RDFGAN step, RDFGenerator ResNet-18 x2 + W-AdaIN + NLSPN 18 it., PatchGAN,
lsgan + 3 x L1, Adam, B = 16, 228x304, the bench's weights and inputs) on one GPU.  Prints one JSON line.

    python scripts/train_precision.py [--steps 10] [--warmup 3] [--batch 16]

Modes: 'bf16' and 'fp32_tc' (set_train_precision), and 'fp32_torch': the fp32_tc composition with conv2d_nhwc / bn_act replaced
by fp32 PyTorch ops (tests/_fp32_ops.py) -- what an fp32 user of the reference runs today, cuDNN on the CUDA cores.  Both fp32
modes run with TF32 off throughout (the discriminator included); bf16 with torch's defaults, as bench.py c4.
Step times: CUDA events around `steps` optimize_parameters calls after warm-up, per step (the step's working set is far larger
than the L2).  Distances: one step from the same weights and batch in fp32_tc and in fp32_torch -- the five output maps (max-abs),
the losses (relative), every parameter gradient's cosine and norm ratio.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

import bench_train  # noqa: E402
from _fp32_ops import fp32_torch_ops  # noqa: E402
from _synth import synth_state_dict  # noqa: E402

MODES = ("bf16", "fp32_tc", "fp32_torch")


def gpu_info():
    """name and power limit of GPU 0, read-only query"""
    out = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True, check=True).stdout.strip()
    name, power = [s.strip() for s in out.split(",", 1)]
    return dict(gpu=name, power_limit=power)


class _Mode:
    """set_train_precision; TF32 off in the fp32 modes; (fp32_torch) the two kernel-backed ops swapped for fp32 PyTorch"""
    def __init__(self, model, mode):
        self.model, self.mode = model, mode

    def __enter__(self):
        import rdfc_gan_b200.train_forward as tf
        self.model.G.set_train_precision('bf16' if self.mode == 'bf16' else 'fp32_tc')
        self.saved = (tf.conv2d_nhwc, tf.bn_act, torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
        if self.mode != 'bf16':                        # an fp32 user: TF32 off (the discriminator's cuDNN convs included)
            torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
        if self.mode == 'fp32_torch':
            tf.conv2d_nhwc, tf.bn_act = fp32_torch_ops()
        return self

    def __exit__(self, *exc):
        import rdfc_gan_b200.train_forward as tf
        tf.conv2d_nhwc, tf.bn_act, torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = self.saved
        self.model.G.set_train_precision('bf16')


def build(B):
    from rdfc_gan_b200.discriminator import PatchGANDiscriminator
    from rdfc_gan_b200.generator import RDFGenerator
    from rdfc_gan_b200.rdf_gan import RDFGAN
    G = RDFGenerator(pretrained_on_imagenet=False, use_nlspn_refine=True, nlspn_configs=bench_train.NLSPN_CFG)
    G.load_state_dict(synth_state_dict(G, seed=0, recipe="init", nlspn_stress=True))
    D = PatchGANDiscriminator(in_channels=1)
    D.load_state_dict(synth_state_dict(D, seed=1, recipe="init"))
    model = RDFGAN(G, D, device="cuda", args=bench_train.ARGS)
    model.train()
    batch = {k: v.cuda() for k, v in bench_train.synth_batch(B, seed=0).items()}
    return model, batch


def step_ms(mode, B, steps, warmup):
    model, batch = build(B)
    with _Mode(model, mode):
        for _ in range(warmup):
            model.set_input(batch)
            model.optimize_parameters()
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(steps):
            model.set_input(batch)
            stats = model.optimize_parameters()
        b.record()
        torch.cuda.synchronize()
    assert all(v == v for v in stats.values()), stats
    return a.elapsed_time(b) / steps, torch.cuda.max_memory_allocated() / 2**30


def one_step(mode, B):
    """outputs, losses and parameter gradients of one step (no optimiser update) from the initial weights"""
    model, batch = build(B)
    with _Mode(model, mode):
        model.set_input(batch)
        model.forward()
        outs = dict(depth_map_1=model.fake_B_rgb_branch, confidence_map_1=model.conf_map_rgb_branch, depth_map_2=model.fake_B_depth_branch,
                    confidence_map_2=model.conf_map_depth_branch, pred_depth=model.final_depth)
        outs = {k: v.detach().clone() for k, v in outs.items()}
        model.set_requires_grad(model.D, True)
        model.bucket_D.zero()
        losses = {k: float(v) for k, v in model.backward_D().items()}
        model.set_requires_grad(model.D, False)
        model.bucket_G.zero()
        losses.update({k: float(v) for k, v in model.backward_G().items()})
        grads = {f"{net}.{n}": p.grad.detach().clone() for net, mod in (("G", model.G), ("D", model.D))
                 for n, p in mod.named_parameters() if p.grad is not None}
    return outs, losses, grads


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=16)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "train_precision.py measures on a GPU"
    info = gpu_info()
    res = {"workload": f"bench.py c4 training step on one GPU: B = {args.batch}, {bench_train.H}x{bench_train.W}, NLSPN 18 it., lsgan + L1, Adam",
           **info, "steps": args.steps, "warmup": args.warmup}
    for mode in MODES:
        ms, gib = step_ms(mode, args.batch, args.steps, args.warmup)
        res[f"step_ms_{mode}"] = round(ms, 2)
        res[f"peak_mem_gib_{mode}"] = round(gib, 2)
    o_tc, l_tc, g_tc = one_step("fp32_tc", args.batch)
    o_ref, l_ref, g_ref = one_step("fp32_torch", args.batch)
    dist = {f"out_max_abs:{k}": float((o_tc[k] - o_ref[k]).abs().max()) for k in o_tc}
    dist.update({f"loss_rel:{k}": abs(l_tc[k] - l_ref[k]) / max(abs(l_ref[k]), 1e-12) for k in l_tc})
    cos = {n: float((g_tc[n].double() * g_ref[n].double()).sum() / (g_tc[n].double().norm() * g_ref[n].double().norm() + 1e-30))
           for n in g_tc if g_tc[n].numel() >= 8 and float(g_ref[n].norm()) > 0}          # (fuse_layer5 is built but never used)
    ratio = {n: float(g_tc[n].double().norm() / (g_ref[n].double().norm() + 1e-30)) for n in cos}
    for net in ("G", "D"):
        c = [v for n, v in cos.items() if n.startswith(net + ".")]
        dist[f"grad_min_cos_{net}"] = min(c)
        dist[f"grad_median_cos_{net}"] = float(np.median(c))
    dist["grad_max_norm_ratio_dev"] = max(abs(r - 1) for r in ratio.values())
    dist["grad_median_norm_ratio"] = float(np.median(list(ratio.values())))
    dist["grad_worst_cos"] = sorted((round(c, 6), n) for n, c in cos.items())[:5]
    res["fp32_tc_vs_fp32_torch"] = dist
    res["gpu_after"] = gpu_info()
    print(json.dumps(res))


if __name__ == "__main__":
    main()
