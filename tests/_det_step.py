"""The c4 training step under torch.use_deterministic_algorithms: RDFGAN.optimize_parameters with RDFGenerator (NLSPN TGASS,
18 iterations, conf_prop), PatchGAN, lsgan + 3 x L1, Adam, from seeded weights and a seeded batch.

    python tests/_det_step.py PRECISION B H W STEPS [PRESERVE]

prints the SHA-256 of the losses of every step and, after the last, of every G / D parameter and buffer (BatchNorm running
statistics included).  Run it in a fresh process with CUBLAS_WORKSPACE_CONFIG=:4096:8 set before CUDA starts."""
import hashlib
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
for p in (os.path.dirname(HERE), HERE):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402
import torch  # noqa: E402


def build(B, H, W, precision, preserve_input=False, seed=0):
    import bench_train
    from _synth import _rng, synth_inputs, synth_state_dict
    from rdfc_gan_b200.discriminator import PatchGANDiscriminator
    from rdfc_gan_b200.generator import RDFGenerator
    from rdfc_gan_b200.rdf_gan import RDFGAN
    nl = dict(bench_train.NLSPN_CFG, preserve_input=preserve_input)
    G = RDFGenerator(pretrained_on_imagenet=False, use_nlspn_refine=True, nlspn_configs=nl)
    G.load_state_dict(synth_state_dict(G, seed=seed, recipe="init", nlspn_stress=True))
    D = PatchGANDiscriminator(in_channels=1)
    D.load_state_dict(synth_state_dict(D, seed=seed + 1, recipe="init"))
    model = RDFGAN(G, D, device="cuda", args=bench_train.ARGS)
    model.train()
    model.G.set_train_precision(precision)
    rgb, normal, raw = synth_inputs(B, H, W, seed=seed)
    coarse = torch.from_numpy(_rng(seed, "train_gt").uniform(-0.9, 0.9, (B, 1, 8, 10)).astype(np.float32))
    gt = torch.nn.functional.interpolate(coarse, size=(H, W), mode="bilinear", align_corners=True)
    batch = {k: v.cuda() for k, v in dict(rgb=rgb, normal=normal, raw_depth=raw, gt_depth=gt.contiguous()).items()}
    return model, batch


def state_digest(model, losses):
    h = hashlib.sha256()
    for stats in losses:
        for k in sorted(stats):
            h.update(k.encode() + np.float64(stats[k]).tobytes())
    for net, mod in (("G", model.G), ("D", model.D)):
        for name, t in list(mod.named_parameters()) + list(mod.named_buffers()):
            h.update(f"{net}.{name}".encode() + t.detach().cpu().contiguous().numpy().tobytes())
    return h.hexdigest()


def run(precision, B, H, W, steps, preserve_input=False):
    torch.use_deterministic_algorithms(True)
    saved = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    if precision == "fp32_tc":
        torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    try:
        model, batch = build(B, H, W, precision, preserve_input)
        losses = []
        for _ in range(steps):
            model.set_input(batch)
            losses.append(model.optimize_parameters())
        torch.cuda.synchronize()
        return state_digest(model, losses)
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = saved
        torch.use_deterministic_algorithms(False)


if __name__ == "__main__":
    prec, B, H, W, steps = sys.argv[1], *map(int, sys.argv[2:6])
    print(run(prec, B, H, W, steps, preserve_input=len(sys.argv) > 6 and sys.argv[6] == "1"))
