"""A cycle-shaped RDFC-GAN training step under torch.use_deterministic_algorithms: RDFGenerator (G_A2B: NLSPN TGASS, 18 iterations,
conf_prop) forward in train(), ResnetGenerator (G_B2A, depth -> RGB) on its depth_map_1, the RDFGAN losses (PatchGAN, lsgan +
3 x L1) plus an L1 cycle loss of G_B2A's output against the RGB input, Adam steps on the discriminator and both generators, from
seeded weights and a seeded batch (tests/_det_step.py builds G_A2B, D and the batch).

    python tests/_det_cycle.py PRECISION B H W STEPS

prints one SHA-256 of the losses of every step and, after the last, of every parameter and buffer of both generators and the
discriminator.  Run it in a fresh process with CUBLAS_WORKSPACE_CONFIG=:4096:8 set before CUDA starts."""
import hashlib
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
for p in (os.path.dirname(HERE), HERE):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

LAMBDA_CYCLE = 10.0


def cycle_step(model, G_B2A, opt_B2A):
    """RDFGAN.optimize_parameters with G_B2A(depth_map_1) and its L1 cycle loss added to the generator update"""
    from rdfc_gan_b200.parallel import reduce_losses
    model.forward()
    model.set_requires_grad(model.D, True)
    model.bucket_D.zero()
    stats = model.backward_D()
    model.bucket_D.allreduce()
    model.optimizer_D.step()
    model.set_requires_grad(model.D, False)
    model.bucket_G.zero()
    opt_B2A.zero_grad(set_to_none=False)
    rec = G_B2A(model.fake_B_rgb_branch)
    loss_cycle = (rec - model.real_A).abs().mean() * LAMBDA_CYCLE
    loss_cycle.backward(retain_graph=True)          # into G_B2A and, through depth_map_1, into G_A2B; backward_G adds its losses
    stats.update(model.backward_G())
    stats["loss_cycle"] = loss_cycle
    model.bucket_G.allreduce()
    model.optimizer_G.step()
    opt_B2A.step()
    return reduce_losses(stats)


def run(precision, B, H, W, steps, seed=0):
    import _det_step
    from _synth import synth_state_dict
    from rdfc_gan_b200.resnet_generator import ResnetGenerator
    torch.use_deterministic_algorithms(True)
    saved = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    if precision == "fp32_tc":
        torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    try:
        model, batch = _det_step.build(B, H, W, precision, seed=seed)
        G_B2A = ResnetGenerator(input_channels=1, output_channels=3)
        G_B2A.load_state_dict(synth_state_dict(G_B2A, seed=seed + 2, recipe="scaled"))
        G_B2A = G_B2A.cuda().train().set_train_precision(precision)
        a = model.args
        opt_B2A = torch.optim.Adam(G_B2A.parameters(), lr=a.lr, betas=(a.beta1, a.beta2))
        losses = []
        for _ in range(steps):
            model.set_input(batch)
            losses.append(cycle_step(model, G_B2A, opt_B2A))
        torch.cuda.synchronize()
        h = hashlib.sha256(_det_step.state_digest(model, losses).encode())
        for name, t in list(G_B2A.named_parameters()) + list(G_B2A.named_buffers()):
            h.update(f"G_B2A.{name}".encode() + t.detach().cpu().contiguous().numpy().tobytes())
        return h.hexdigest()
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = saved
        torch.use_deterministic_algorithms(False)


if __name__ == "__main__":
    prec, B, H, W, steps = sys.argv[1], *map(int, sys.argv[2:6])
    print(run(prec, B, H, W, steps))
