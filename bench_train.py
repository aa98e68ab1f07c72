"""bench.py --config c4: the RDFC-GAN training step (BASELINE config 4) on N B200s.

A step = RDFGAN.optimize_parameters (C/lib/models/rdf_gan.py:192-207): train-mode generator forward (batch-statistics
BatchNorm), discriminator update (lsgan), generator update (lsgan + three L1 terms), Adam for both nets, with ONE flattened
gradient all-reduce per net over NCCL / NVLink (parallel.GradientBucket) instead of DistributedDataParallel's buckets.
Data parallel, `batch_per_gpu` images per rank (weak scaling: the global batch grows with N, per-GPU BatchNorm statistics as in
the reference).  Rank 0 prints ONE JSON line:

  value      training images/s, inputs resident in HBM, CUDA-event timed over the K steps, max over ranks
  e2e        the same through set_input() from pinned HOST tensors (H2D inside the timed region) with the loss dict read back
  allreduce  ms per step spent in the two gradient all-reduces (CUDA events around them), elements reduced
  roofline   dense part: 3 x the forward's conv FLOPs (forward + data gradient + filter gradient) / step time vs the measured bf16 peak
  cpu_baseline / --impl reference: the reference's own modules (generator, PatchGAN, losses) doing the same step on the host cores
"""
import json
import os
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
H, W = 228, 304
NLSPN_CFG = dict(prop_kernel=3, prop_time=18, affinity="TGASS", affinity_gamma=0.5, conf_prop=True, preserve_input=False)
ARGS = dict(gan_loss_type="lsgan", lambda_l1_rgb_branch=10.0, lambda_l1_depth_branch=10.0, lambda_l1_fusion=10.0, optimizer="adam",
            lr=2e-4, beta1=0.5, beta2=0.999)
GFLOP_FWD = 221.4            # SURVEY 8d, generator forward per image at 228x304
GFLOP_D = 6.5                # PatchGAN forward per image (three forward + two backward passes per step, on cuDNN)


def workload(per_gpu, world):
    return {"workload": "BASELINE config 4: RDFC-GAN training step (RDFGenerator ResNet-18 x2 + W-AdaIN + NLSPN 18 it., PatchGAN "
                        "discriminator, lsgan + 3 x L1, Adam), data parallel with one flattened NCCL gradient all-reduce per net",
            "config": "c4", "batch_per_gpu": per_gpu, "global_batch": per_gpu * world, "height": H, "width": W,
            "weights": "synthetic (tests/_synth.py): init_weights recipe + NLSPN offsets of trained magnitude; PatchGAN init_weights",
            "cache": "per-step working set >> 126 MB L2", "parallelism": f"data parallel x{world}, gradient all-reduce (sum / world)"}


def synth_batch(B, seed):
    import numpy as np
    import torch
    from _synth import _rng, synth_inputs
    rgb, normal, raw = synth_inputs(B, H, W, seed=seed)
    r = _rng(seed, "train_gt")
    coarse = torch.from_numpy(r.uniform(-0.9, 0.9, (B, 1, 8, 10)).astype(np.float32))
    gt = torch.nn.functional.interpolate(coarse, size=(H, W), mode="bilinear", align_corners=True)
    return dict(rgb=rgb, normal=normal, raw_depth=raw, gt_depth=gt.contiguous())


def reference_step_cpu(n_images, reps, warmup=1):
    """The reference's own generator / discriminator / losses through one optimize_parameters-style step on the host cores."""
    import torch
    sys.path.insert(0, os.path.join(ROOT, "baseline"))
    import ref_loader
    from _synth import synth_state_dict
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    RefG = ref_loader.load_rdfc()
    ref_loader.differentiable_dcn_on_cpu()
    RefD, GANLoss, L1_loss = ref_loader.load_rdfc_training()
    G = RefG(pretrained_on_imagenet=False, use_nlspn_refine=True, nlspn_configs=NLSPN_CFG).train()
    G.load_state_dict(synth_state_dict(G, seed=0, recipe="init", nlspn_stress=True))
    D = RefD(in_channels=1).train()
    D.load_state_dict(synth_state_dict(D, seed=1, recipe="init"))
    oG = torch.optim.Adam(G.parameters(), lr=ARGS["lr"], betas=(ARGS["beta1"], ARGS["beta2"]))
    oD = torch.optim.Adam(D.parameters(), lr=ARGS["lr"], betas=(ARGS["beta1"], ARGS["beta2"]))
    crit = GANLoss("lsgan")
    data = synth_batch(n_images, 0)
    w = torch.ones_like(data["gt_depth"])
    w = w / (w.sum() + 1e-6)
    ts = []
    for i in range(warmup + reps):
        t0 = time.perf_counter()
        ret = G(data["rgb"], data["raw_depth"], data["normal"])
        fake = ret["depth_map_1"]
        for p in D.parameters():
            p.requires_grad = True
        oD.zero_grad()
        (0.5 * (crit(D(fake.detach()), False) + crit(D(data["gt_depth"]), True))).backward()
        oD.step()
        for p in D.parameters():
            p.requires_grad = False
        oG.zero_grad()
        (crit(D(fake), True) + 10 * L1_loss(ret["depth_map_1"], data["gt_depth"], weight=w) +
         10 * L1_loss(ret["depth_map_2"], data["gt_depth"], weight=w) + 10 * L1_loss(ret["pred_depth"], data["gt_depth"], weight=w)).backward()
        oG.step()
        if i >= warmup:
            ts.append(time.perf_counter() - t0)
    return n_images * len(ts) / sum(ts), cores, ts


def main(args, rank, world, local):
    per_gpu = args.batch or 16
    if args.impl == "reference":
        if rank != 0:
            return
        n = 1
        val, cores, ts = reference_step_cpu(n, max(1, min(args.steps, 4)), warmup=min(args.warmup, 1))
        print(json.dumps({
            "impl": "reference", "metric": "training images/sec @228x304", "value": val, "unit": "images/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * sum(ts) / len(ts), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": workload(per_gpu, world),
            "cpu_baseline": {"value": val, "unit": "images/s", "cores": cores, "kind": "reference",
                             "sample": f"{n} image per step, {len(ts)} timed steps, fp32: the reference's RDFGenerator / PatchGANDiscriminator / "
                                       "GANLoss / L1_loss on torch CPU, DCN (forward + backward) through torchvision.ops.deform_conv2d"},
            "e2e": {"value": val, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return

    import numpy as np
    import torch
    import torch.distributed as dist
    from _synth import synth_state_dict
    from rdfc_gan_b200 import _cabi as C
    from rdfc_gan_b200.discriminator import PatchGANDiscriminator
    from rdfc_gan_b200.generator import RDFGenerator
    from rdfc_gan_b200.rdf_gan import RDFGAN
    import bench
    assert torch.cuda.is_available(), "bench.py needs a GPU (no CPU fallback exists)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    G = RDFGenerator(pretrained_on_imagenet=False, use_nlspn_refine=True, nlspn_configs=NLSPN_CFG)
    G.load_state_dict(synth_state_dict(G, seed=0, recipe="init", nlspn_stress=True))
    D = PatchGANDiscriminator(in_channels=1)
    D.load_state_dict(synth_state_dict(D, seed=1, recipe="init"))
    model = RDFGAN(G, D, device=dev, distributed=world > 1, args=ARGS)
    model.train()
    host = {k: v.pin_memory() for k, v in synth_batch(per_gpu, seed=rank).items()}
    resident = {k: v.to(dev) for k, v in host.items()}

    # all-reduce timing: CUDA events around the two bucket all-reduces of every step
    ar_events = []
    for bucket in (model.bucket_G, model.bucket_D):
        orig = bucket.allreduce

        def timed(average=True, _orig=orig):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            n = _orig(average)
            b.record()
            ar_events.append((a, b))
            return n
        bucket.allreduce = timed

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def maxreduce(x):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    n0 = C.launch_count()
    for _ in range(max(args.warmup, 3)):
        model.set_input(resident)
        stats = model.optimize_parameters()
    barrier()
    launches_per_step = (C.launch_count() - n0) // max(args.warmup, 3)
    ar_events.clear()
    sampler = bench.ClockSampler(local)
    sampler.start()
    time.sleep(0.15)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(args.steps):
        model.set_input(resident)
        stats = model.optimize_parameters()
    b.record()
    barrier()
    clocks = sampler.summary()
    t_ms = maxreduce(a.elapsed_time(b))
    ar_ms = maxreduce(sum(x.elapsed_time(y) for x, y in ar_events)) / args.steps
    value = per_gpu * world * args.steps / (t_ms / 1e3)
    assert all(v == v and abs(v) < 1e6 for v in stats.values()), stats          # finite losses
    dumped = None
    if args.dump_outputs and rank == 0:         # the last timed step's generator maps and the loss dict it returned
        dumped = bench.sample_outputs(dict(zip(bench.KEYS, (model.fake_B_rgb_branch, model.conf_map_rgb_branch, model.fake_B_depth_branch,
                                                            model.conf_map_depth_branch, model.final_depth))))
        dumped.update({k: np.float64(v) for k, v in stats.items()})

    # e2e: host batch -> set_input (H2D) -> step -> loss dict on the host, wall clock
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        model.set_input(host)
        stats = model.optimize_parameters()
    barrier()
    e2e = per_gpu * world * args.steps / maxreduce(time.perf_counter() - t0)
    h2d = sum(v.numel() * 4 for v in host.values())

    pk = bench.peaks()
    tflops = 3 * GFLOP_FWD * 1e9 * per_gpu * args.steps / (t_ms / 1e3) / 1e12
    cpu = None
    import ref_loader
    if rank == 0 and world == 1 and not args.no_cpu_baseline and ref_loader.available():     # the step has no oracle restatement
        v, cores, ts = reference_step_cpu(1, 2)
        cpu = {"value": v, "unit": "images/s", "cores": cores, "kind": "reference",
               "sample": f"1 image per step x 2 timed steps, fp32, the reference's own modules on torch CPU; {sum(ts):.1f} s timed"}
    if rank == 0:
        print(json.dumps({
            "metric": "training images/sec @228x304", "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": t_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16", "data": "synthetic", "config": workload(per_gpu, world), "clocks": clocks,
            "e2e": {"value": e2e, "unit": "images/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4 * len(stats)},
            "gpu_launches": launches_per_step * args.steps,
            "allreduce": {"ms_per_step": ar_ms, "share": ar_ms / (t_ms / args.steps), "elements": model.bucket_G.numel() + model.bucket_D.numel(),
                          "backend": "nccl" if world > 1 else "none (1 rank)"},
            "losses": {k: float(v) for k, v in stats.items()},
            "roofline": {"kernel": "conv forward / dgrad (conv_umma_kernel) + filter gradient (wgrad_umma_kernel), all tcgen05: whole dense part",
                         "bound": "tensor", "achieved": tflops, "peak": pk["bf16_sustained"], "unit": "TFLOP/s",
                         "frac": tflops / pk["bf16_sustained"], "traffic": None, "peak_source": pk["src"] + " (sustained cuBLAS bf16)",
                         "note": "3 x 221.4 GFLOP per image (forward, data gradient, filter gradient) over the whole step time"},
            "cpu_baseline": cpu}))
    if dumped is not None:
        bench.write_outputs(args.dump_outputs, dumped)
    if world > 1:
        dist.destroy_process_group()
