#!/usr/bin/env python
"""bench.py -- depth maps/s of the generator forward on N B200s, with in-run parity, the NLSPN roofline and the reference beside it.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config c3|c2|c5|c4] [--batch GLOBAL] [--precision bf16|fp32]
                    [--impl reference] [--dump-outputs DIR]

Workloads (BASELINE.json `configs`; the default, c3, is the one `metric` is quoted on):
  c3  RDFC-GAN RDFGenerator (ResNet-18 x2, W-AdaIN, NLSPN TGASS 18 it.) inference, GLOBAL batch 256 @228x304, batch-sharded over
      the N ranks (256 / N images per GPU: strong scaling, no collective on the data path).
  c2  RDF-GAN DCVGANGenerator (ResNet-34 x2, 40-channel stem, W-AdaIN with `adain_weighting`, NLSPN), batch 32 @228x304.
  c5  RDFGenerator @480x640 (SUN RGB-D shape), NLSPN 18 iterations, global batch 64.
  c4  RDFC-GAN training step (generator + PatchGAN discriminator, lsgan + L1) with one NCCL gradient all-reduce (bench_train).

A step = one forward over this rank's shard.  N > 1: launched by torchrun, one rank per GPU; the timed region is bracketed by
a barrier + synchronize and the max over ranks is taken.  Rank 0 prints ONE JSON line.

  value      maps/s, inputs resident in HBM (CUDA-graph replay of the plan), CUDA-event timed per step, L2 flushed between steps.
  e2e        the same metric through the public API (G.stream(): pinned HOST batches in, all five maps back to pinned host
             memory), H2D + D2H inside the timed region.
  parity     the timed bf16 outputs of the first batch against this repo's fp32 mode (<= 1e-4 from the reference, tests/) on
             the same images: RMSE / max-abs per map; the run FAILS above PARITY_RMSE / PARITY_MAXABS.
  value_fp32 maps/s of the strict fp32 parity mode (CUDA cores; measured while computing `parity`); value_fp32_tc: the fp32 mode
             on the tensor cores (split fp16 operands) with its max-abs distance from the strict mode.
  ref_gpu    the unmodified reference (PyTorch/cuDNN + its own DCN CUDA extension, baseline/_ref) on the same GPU, maps/s.
  roofline   the NLSPN propagation kernel timed alone (CUDA events on its launch stream, >= 50 repetitions, min / median):
             achieved = 116 B x pixels per launch / launch time, against MEASURED_PEAKS.json hbm_gbs.
  cpu_baseline / --impl reference: the UNMODIFIED reference Python (baseline/_ref/rdf_generator, DCN served by
             torchvision.ops.deform_conv2d as BASELINE.json prescribes) on all host cores, on a bounded sample.

--dump-outputs DIR writes what the last timed step computed on rank 0 as DIR/<name>.npy: the five maps, float32 (beyond DUMP_BYTES,
a fixed seeded sample of the images), and for c4 also the step's losses, float64.  Inputs and weights are seeded, so two builds
run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import random
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "baseline")):
    if p not in sys.path:
        sys.path.insert(0, p)

NLSPN_CFG = dict(prop_kernel=3, prop_time=18, affinity="TGASS", affinity_gamma=0.5, conf_prop=True, preserve_input=False)
ALGO_BYTES_PER_PIXEL_ITER = 116          # SURVEY 8d: 18 offsets + 9 affinities + 1 feature read, 1 feature written, fp32
KEYS = ("depth_map_1", "confidence_map_1", "depth_map_2", "confidence_map_2", "pred_depth")
# the stated bf16 tolerance (north_star: "bf16 within a stated RMSE delta"), normalised depth units (x 5 m), against fp32 mode:
# tests/_synth.py BF16_BOUND (twice the error measured on B200), the same table the parity tests and smoke() assert
from _synth import BF16_BOUND  # noqa: E402
PARITY_RMSE, PARITY_MAXABS = BF16_BOUND["init"]

CONFIGS = {
    # gflop: SURVEY 8d, 2 x MACs of every Conv / ConvT / Linear per image
    "c3": dict(gen="rdfc", batch=256, H=228, W=304, gflop=221.4, fp32_chunk=32, cs=3, parity=(PARITY_RMSE, PARITY_MAXABS),
               name="BASELINE config 3: RDFC-GAN RDFGenerator inference (ResNet-18 x2, W-AdaIN, NLSPN TGASS 18 it.), global batch 256 "
                    "@228x304, batch-sharded"),
    # c2's weights are fan-in scaled (O(1) activations through ~70 layers, outputs span [-1, 1]): its own, wider, stated bound
    "c2": dict(gen="rdf", batch=32, H=228, W=304, gflop=415.8, fp32_chunk=16, cs=3, parity=BF16_BOUND["scaled_r34"],
               name="BASELINE config 2: RDF-GAN DCVGANGenerator forward (ESANet-34 guidance network -> 40-channel stems, ResNet-34 x2, "
                    "W-AdaIN + adain_weighting, NLSPN TGASS 18 it.), batch 32 @228x304"),
    "c5": dict(gen="rdfc", batch=64, H=480, W=640, gflop=976.9, fp32_chunk=8, cs=3, parity=(PARITY_RMSE, PARITY_MAXABS),
               name="BASELINE config 5: RDFGenerator inference @480x640 (SUN RGB-D shape), NLSPN 18 it., bf16, global batch 64, "
                    "batch-sharded"),
}


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return dict(hbm=p["hbm_gbs"], bf16=p["bf16_tflops"], bf16_sustained=p.get("bf16_tflops_sustained", p["bf16_tflops"]),
                    src="measured")
    return dict(hbm=6650.0, bf16=1590.0, bf16_sustained=1400.0, src="fallback")


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons while the timed region runs (B200_PROFILING.md recipe): one streaming
    `nvidia-smi -lms 50` process, so that even a 0.2 s timed region yields several samples."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.proc = index, [], None

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                          "-lms", "50"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                if line.strip():
                    self.rows.append([c.strip() for c in line.strip().split(",")])
        except Exception:
            pass

    def summary(self):
        if self.proc is not None:
            self.proc.terminate()
        self.join(timeout=6)
        sm = [int(r[0]) for r in self.rows if r[0].isdigit()]
        mx = [int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows for n, v in zip(names, r[2:6]) if v.lower().startswith("active")})
        return dict(sm_mhz=int(statistics.median(sm)) if sm else None, sm_max_mhz=max(mx) if mx else None, reasons=reasons,
                    samples=len(sm))


DUMP_BYTES = 48 << 20                    # --dump-outputs: at most this much array data


def sample_outputs(outputs):
    """name -> [B, ...] device tensor  =>  name -> float32 host array.  Above DUMP_BYTES in all, every map keeps the same sample
    of images, drawn with a fixed seed from B alone (so it is the same in every run with the same batch)."""
    B = next(iter(outputs.values())).shape[0]
    keep = min(B, DUMP_BYTES // sum(t[0].numel() * 4 for t in outputs.values()))
    idx = list(range(B)) if keep == B else sorted(random.Random(0).sample(range(B), keep))
    return {k: t[idx].detach().float().cpu().numpy() for k, t in outputs.items()}


def write_outputs(path, arrays):
    import numpy as np
    os.makedirs(path, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(path, k + ".npy"), a)


def gen_kwargs(cfg):
    if cfg["gen"] == "rdfc":
        return dict(pretrained_on_imagenet=False, use_nlspn_refine=True, nlspn_configs=NLSPN_CFG)
    # F/bash/test_nyuv2_Ts2T.sh:17-29
    return dict(encoder_rgb="resnet34", encoder_depth="resnet34", pretrained_on_imagenet=False, semantic_channels_in=40,
                adain_weighting=True, use_nlpsn_refine=True, nlspn_configs=NLSPN_CFG)


def synth_weights(module, cfg):
    """c3 / c5: the reference's random init (init_weights) + NLSPN offsets of trained magnitude (sigma ~ 2 px), SURVEY 8d.
    c2: fan-in scaled weights (RDF-GAN keeps torch's default init) + the same NLSPN stress."""
    from _synth import synth_state_dict
    recipe = "init" if cfg["gen"] == "rdfc" else "scaled"
    return synth_state_dict(module, seed=0, recipe=recipe, nlspn_stress=True)


ESANET_KW = dict(num_classes=40, pretrained_on_imagenet=False, encoder="resnet34", encoder_block="BasicBlock",
                 channels_decoder=[512, 256, 128], nr_decoder_blocks=[3, 3, 3], encoder_decoder_fusion="add", context_module="ppm",
                 weighting_in_encoder="SE-add", upsampling="learned-3x3-zeropad", pyramid_supervision=False)      # F/bash/test_nyuv2_Ts2T.sh:7-16


def build_product(cfg):
    from rdfc_gan_b200.generator import DCVGANGenerator, RDFGenerator
    if cfg["gen"] == "rdfc":
        G = RDFGenerator(**gen_kwargs(cfg)).eval()
    else:
        from rdfc_gan_b200.esanet import ESANetOneModality
        G = DCVGANGenerator(ESANetOneModality(height=cfg["H"], width=cfg["W"], **ESANET_KW), **gen_kwargs(cfg)).eval()
    G.load_state_dict(synth_weights(G, cfg))
    return G


def build_reference(cfg, gpu=False):
    """The reference's own generator class from baseline/_ref (no product import), same synthetic state dict."""
    import ref_loader
    if cfg["gen"] == "rdfc":
        G = ref_loader.load_rdfc(gpu)(**gen_kwargs(cfg)).eval()
    else:
        DCV, ESA = ref_loader.load_rdf_gan(gpu)
        G = DCV(ESA(height=cfg["H"], width=cfg["W"], **ESANET_KW), **gen_kwargs(cfg)).eval()
    G.load_state_dict(synth_weights(G, cfg))
    return G


def call_generator(G, cfg, rgb, stem, depth):
    """RDFGenerator.forward(rgb, depth, normal) -> dict; DCVGANGenerator.forward(rgb, depth) -> 5-tuple (its guidance network
    maps rgb to the 40-channel stem input)."""
    if cfg["gen"] == "rdfc":
        return G(rgb, depth, stem)
    return dict(zip(KEYS, G(rgb, depth)))


def reference_cpu(cfg, n_images, reps, warmup=1):
    """The unmodified reference on the host cores: returns (maps/s over the timed reps, cores, per-rep seconds, kind)."""
    import torch
    from _synth import synth_inputs
    import ref_loader
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    if ref_loader.available():
        G, kind = build_reference(cfg), "reference"
        fwd = lambda rgb, stem, depth: call_generator(G, cfg, rgb, stem, depth)
    else:                                   # baseline/_ref did not travel: the oracle restatement (RDFGenerator only)
        from oracle import generator as ogen
        sd, kind = build_product(cfg).state_dict(), "port"
        fwd = lambda rgb, stem, depth: ogen.generator_forward(sd, stem, depth, use_nlspn_refine=True, nlspn_configs=NLSPN_CFG)
    rgb, stem, depth = synth_inputs(n_images, cfg["H"], cfg["W"], seed=0, Cs=cfg["cs"])
    ts = []
    with torch.no_grad():
        for i in range(warmup + reps):
            t0 = time.perf_counter()
            fwd(rgb, stem, depth)
            if i >= warmup:
                ts.append(time.perf_counter() - t0)
    return n_images * len(ts) / sum(ts), cores, ts, kind


def workload_config(cfg, args, world, per_gpu):
    return {"workload": cfg["name"], "config": args.config, "global_batch": args.batch, "batch_per_gpu": per_gpu,
            "height": cfg["H"], "width": cfg["W"],
            "weights": "synthetic (tests/_synth.py): " + ("init_weights recipe" if cfg["gen"] == "rdfc" else "fan-in scaled") +
                       " + NLSPN offsets of trained magnitude",
            "outputs": "all five maps (depth_map_1, confidence_map_1, depth_map_2, confidence_map_2, pred_depth) in value and e2e",
            "cache": "L2 flushed (256 MiB write) between timed steps; per-step working set >> 126 MB L2",
            "parallelism": f"batch-sharded x{world}, no collective"}


def run_reference(args, cfg, rank, world):
    """--impl reference: the reference's own CPU path on this box's host cores (rank 0 only)."""
    if rank != 0:
        return
    n = 4 if cfg["H"] < 400 else 1
    val, cores, ts, kind = reference_cpu(cfg, n, args.steps, warmup=args.warmup)
    per_gpu = args.batch // world
    sample = (f"{n} images per step (a bounded sample of the {args.batch}-image batch), {args.steps} steps, fp32, unmodified reference "
              f"Python on torch CPU, DCN through torchvision.ops.deform_conv2d" if kind == "reference" else
              f"{n} images per step, {args.steps} steps, fp32, oracle port (baseline/_ref missing)")
    print(json.dumps({
        "impl": "reference", "metric": "depth maps/sec @228x304", "value": val, "unit": "maps/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * sum(ts) / len(ts), "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(cfg, args, world, per_gpu),
        "cpu_baseline": {"value": val, "unit": "maps/s", "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": val, "unit": "maps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


def reference_gpu(cfg):
    """The reference's stock GPU path (cuDNN convs + its own DCN extension) in a subprocess, before this process touches the GPU."""
    so = os.path.join(ROOT, "baseline", "_ref", "build", "DCN.so")
    if not os.path.exists(so):
        return None
    try:
        r = subprocess.run([sys.executable, os.path.join(ROOT, "baseline", "time_ref_gpu.py"), "--json", cfg["gen"],
                            str(min(32, cfg["batch"])), str(cfg["H"]), str(cfg["W"])], capture_output=True, text=True, timeout=300)
        for line in r.stdout.splitlines()[::-1]:
            if line.startswith("{"):
                return json.loads(line)
        return {"error": (r.stderr or r.stdout)[-300:]}
    except Exception as e:                                  # reporting aid only: never fail the bench on it
        return {"error": repr(e)[:300]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--config", default="c3", choices=["c3", "c2", "c5", "c4"])
    ap.add_argument("--batch", type=int, default=None, help="GLOBAL batch (default: the config's)")
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-ref-gpu", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step to DIR/<name>.npy (--impl b200 only; with several GPUs, rank 0's "
                         "shard of the batch)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs needs --impl b200")
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    if args.config == "c4":
        import bench_train
        return bench_train.main(args, rank, world, local)
    cfg = CONFIGS[args.config]
    args.batch = args.batch or cfg["batch"]
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    if args.impl == "reference":
        return run_reference(args, cfg, rank, world)

    H, W = cfg["H"], cfg["W"]
    ref_gpu = None
    if rank == 0 and world == 1 and not args.no_ref_gpu:
        ref_gpu = reference_gpu(cfg)

    import torch
    import torch.distributed as dist
    from _synth import synth_inputs
    from rdfc_gan_b200 import _cabi as C
    from rdfc_gan_b200.parallel import shard_bounds
    assert torch.cuda.is_available(), "bench.py needs a GPU (no CPU fallback exists)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    lo, hi = shard_bounds(args.batch, world, rank)          # strong scaling: this rank's slice of the GLOBAL batch
    B = hi - lo
    assert B > 0, "more ranks than images"
    G = build_product(cfg).to(dev).set_precision(args.precision)
    # every rank draws its own images (seed = first global image index): same arithmetic as slicing one global batch
    rgb, stem, depth = synth_inputs(B, H, W, seed=lo, Cs=cfg["cs"])
    rgb_d, stem_d, depth_d = rgb.to(dev), stem.to(dev), depth.to(dev)
    with torch.no_grad():
        out = call_generator(G, cfg, rgb_d, stem_d, depth_d)                 # builds + captures the plan
    eng = G.engine()
    plan = next(iter(eng._plans.values()))
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    esa_plan, n_launch = None, plan.n_launch
    if cfg["gen"] == "rdf":              # config 2: the ESANet guidance network's own plan (graph) runs in front of the generator's
        esa = G.global_guidance_module
        esa_plan = next(iter(esa._plans.values()))
        n_launch += len(esa_plan["steps"])
        with torch.no_grad():
            stem_d = esa(rgb_d)          # the 40-channel map the stems read (used by the parity section below)

    def run_step():
        if esa_plan is not None:
            esa_plan["graph"].replay()
            plan.stem_in.copy_(esa_plan["out"])
        plan.run()

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

    # ---------------- value: inputs resident, graph replay, per-step CUDA events, L2 flush between steps
    for _ in range(args.warmup):
        run_step()
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    time.sleep(0.15)                         # let nvidia-smi start streaming; the GPU keeps running warm-up work meanwhile
    for _ in range(2):
        run_step()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    for a, b in evs:
        flush.zero_()
        a.record()
        run_step()
        b.record()
    barrier()
    clocks = sampler.summary()
    t_ms = maxreduce(sum(a.elapsed_time(b) for a, b in evs))
    value = args.batch * args.steps / (t_ms / 1e3)
    dumped = sample_outputs(dict(zip(KEYS, plan.outputs))) if args.dump_outputs and rank == 0 else None

    # ---------------- e2e: public API, pinned host inputs, all five maps back to the host, H2D + D2H inside the timed region
    rgb_h, stem_h, depth_h = rgb.pin_memory(), stem.pin_memory(), depth.pin_memory()
    outs_h = {k: torch.empty(B, 1, H, W).pin_memory() for k in KEYS}

    def host_batches(n):
        for _ in range(n):
            yield (rgb_h, depth_h, stem_h) if cfg["gen"] == "rdfc" else (rgb_h, depth_h)

    last = {}

    def e2e_run(n):
        # G.stream() overlaps the H2D copy of batch i+1 and the D2H read of batch i-1 with the forward of batch i (RDF-GAN: the ESANet
        # guidance network runs on the device inside the same pipeline).
        # (the results arrive in pinned host buffers that stream() recycles two batches later; a consumer would use them in place --
        # an extra 44 MB host memcpy per 32 images here made 8 ranks on one host memory-bound, not the GPUs)
        for o in G.stream(host_batches(n), outputs=KEYS):
            for k in KEYS:
                last[k] = float(o[k][0, 0, 0, 0])         # host-side read of every returned map
    e2e_run(3)
    barrier()
    t0 = time.perf_counter()
    e2e_run(args.steps)
    barrier()
    e2e = args.batch * args.steps / maxreduce(time.perf_counter() - t0)
    # RDFGenerator's stems read `normal` and `depth` only (rdf_generator.py:286-292: `rgb` is unused), so those are the
    # tensors stream() copies; DCVGANGenerator without a guidance module reads the 40-channel map + depth
    h2d = (stem_h if cfg["gen"] == "rdfc" else rgb_h).numel() * 4 + depth_h.numel() * 4
    d2h = sum(t.numel() * 4 for t in outs_h.values())

    # ---------------- parity of what was timed: bf16 outputs vs this repo's fp32 mode, image chunk by image chunk
    parity, value_fp32, value_fp32_tc = None, None, None
    if args.precision == "bf16" and not args.no_parity:
        chunk = min(cfg["fp32_chunk"], B)
        with torch.no_grad():
            plan.stem_in.copy_(stem_d)
            plan.depth.copy_(depth_d)
            plan.run()
            out16 = [t.clone() for t in plan.outputs]
        G.set_precision("fp32")
        se = [0.0] * 5
        mx = [0.0] * 5
        t32 = []
        for c0 in range(0, B, chunk):
            c1 = min(B, c0 + chunk)
            with torch.no_grad():
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                o32 = call_generator(G, cfg, rgb_d[c0:c1], stem_d[c0:c1], depth_d[c0:c1])
                if c1 - c0 == chunk and c0 > 0:                        # a later full chunk: the plan exists, time the replay
                    a.record()
                    o32 = call_generator(G, cfg, rgb_d[c0:c1], stem_d[c0:c1], depth_d[c0:c1])
                    b.record()
                    torch.cuda.synchronize()
                    t32.append(a.elapsed_time(b))
            for i, k in enumerate(KEYS):
                d = (out16[i][c0:c1].double() - o32[k].double())
                se[i] += float((d * d).sum())
                mx[i] = max(mx[i], float(d.abs().max()))
        eng.clear_plans(precision="fp32")
        # the tensor-core fp32 mode (split fp16 operands) on the first chunk: throughput and its distance from the strict fp32 mode
        G.set_precision("fp32_tc")
        with torch.no_grad():
            o32 = call_generator(G, cfg, rgb_d[:chunk], stem_d[:chunk], depth_d[:chunk])          # strict reference of this chunk
            G.set_precision("fp32")
            ref32 = {k: v.clone() for k, v in call_generator(G, cfg, rgb_d[:chunk], stem_d[:chunk], depth_d[:chunk]).items()}
            G.set_precision("fp32_tc")
            ttc = []
            for _ in range(3):
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                o32 = call_generator(G, cfg, rgb_d[:chunk], stem_d[:chunk], depth_d[:chunk])
                b.record()
                torch.cuda.synchronize()
                ttc.append(a.elapsed_time(b))
        tc_err = max(float((o32[k] - ref32[k]).abs().max()) for k in KEYS)
        value_fp32_tc = {"value": chunk * world / (statistics.median(ttc) / 1e3), "unit": "maps/s", "batch_per_gpu": chunk,
                         "max_abs_vs_fp32": maxreduce(tc_err),
                         "note": "fp32 tensors, contractions on tcgen05 with split fp16 operands (x_hi W_hi + x_hi W_lo + x_lo W_hi)"}
        eng.clear_plans(precision="fp32")
        eng.clear_plans(precision="fp32_tc")
        G.set_precision("bf16")
        parity = {k: {"rmse": (maxreduce(se[i]) / (B * H * W)) ** 0.5, "max_abs": maxreduce(mx[i])} for i, k in enumerate(KEYS)}
        parity["against"] = "fp32 mode of this repo (<= 1e-4 from the reference's goldens, tests/test_gpu_generator.py)" + (
            "" if esa_plan is None else "; the ESANet guidance network has one (bf16) mode and is common to both sides")
        tol_rmse, tol_max = cfg["parity"]
        parity["bound"] = {"rmse": tol_rmse, "max_abs": tol_max}
        parity["images"] = args.batch
        if t32:
            value_fp32 = {"value": chunk * world / (statistics.median(t32) / 1e3), "unit": "maps/s", "batch_per_gpu": chunk,
                          "note": "strict fp32 parity mode, CUDA cores (module call incl. input copies and output clones)"}
        bad = {k: v for k, v in parity.items() if k in KEYS and (v["rmse"] > tol_rmse or v["max_abs"] > tol_max)}
        if bad:
            print(json.dumps({"error": "bf16 outputs outside the stated tolerance", "parity": parity}), file=sys.stderr)
            sys.exit(3)

    # ---------------- roofline: NLSPN propagation kernel alone (T launches per forward over the whole shard)
    T = NLSPN_CFG["prop_time"]
    P = H * W

    packed = getattr(plan, "packed", None)          # bf16 mode: fp16-packed offset / affinity stream (48 B per pixel)

    def prop_eager():
        if packed is not None:
            C.check(C.lib.rdfc_nlspn_propagate_forward_packed(C.ptr(plan.pred_init), C.ptr(packed), None, 0, C.ptr(plan.d2raw),
                                                              C.ptr(plan.scratch), B, H, W, T, 0, None, C.stream_ptr()))
        else:
            C.check(C.lib.rdfc_nlspn_propagate_forward(C.ptr(plan.pred_init), C.ptr(plan.offset), C.ptr(plan.aff), None, 0,
                                                       C.ptr(plan.d2raw), C.ptr(plan.scratch), None, B, H, W, T, 0, None, C.stream_ptr()))
    for _ in range(3):
        prop_eager()
    torch.cuda.synchronize()
    # the T launches as the product issues them: nodes of a CUDA graph (no host launch gaps between the iterations)
    prop_graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(prop_graph):
        prop_eager()
    prop = prop_graph.replay
    prop()
    torch.cuda.synchronize()
    reps = 60
    pe = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
    for a, b in pe:
        flush.zero_()
        a.record()
        prop()
        b.record()
    torch.cuda.synchronize()
    tms = sorted(a.elapsed_time(b) for a, b in pe)
    prop_ms, prop_min = statistics.median(tms), tms[0]
    algo = ALGO_BYTES_PER_PIXEL_ITER * B * P
    achieved = algo * T / (prop_ms / 1e3) / 1e9
    pk = peaks()
    kname = "nlspn_prop_packed_kernel" if packed is not None else "nlspn_prop_band_kernel"
    streamed = (56 if packed is not None else 108) * B * P      # bytes the kernel itself moves per launch (DESIGN.md 4.2)
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "nlspn_prop_traffic.json")
    if os.path.exists(tpath):
        tj = json.load(open(tpath)).get(kname)
        # ncu dram__bytes (read + write) of ONE launch, captured at tj["batch"] images of tj["pixels"] pixels: per-pixel figure
        # scaled to this launch
        if tj and tj.get("dram_bytes_per_launch"):
            traffic = tj["dram_bytes_per_launch"] * (B * P) / (tj["batch"] * tj["pixels"])
    roofline = {"kernel": kname, "bound": "hbm", "achieved": achieved, "peak": pk["hbm"], "unit": "GB/s",
                "frac": achieved / pk["hbm"], "traffic": traffic, "peak_source": pk["src"] + " (burst copy)",
                "launch_us": prop_ms * 1e3 / T, "launch_us_min": prop_min * 1e3 / T,
                "frac_best": algo * T / (prop_min / 1e3) / 1e9 / pk["hbm"], "repetitions": reps, "launches_per_forward": T,
                "algorithmic_bytes_per_launch": algo, "streamed_bytes_per_launch": streamed,
                "frac_streamed": streamed * T / (prop_ms / 1e3) / 1e9 / pk["hbm"],
                "note": "achieved = 116 B x pixels (SURVEY 8d: fp32 offsets + affinities + feature in / out) / median launch time; "
                        "the bf16-mode kernel streams the offsets / affinities as packed fp16 (56 B per pixel incl. the feature), so "
                        "`frac` can exceed 1 -- `frac_streamed` is the share of the HBM peak it really moves"}
    dense_tflops = cfg["gflop"] * 1e9 * B * args.steps / (t_ms / 1e3) / 1e12
    roofline_dense = {"kernel": "conv_umma_kernel (whole dense part, upper bound: step time includes NLSPN/norm kernels)",
                      "bound": "tensor", "achieved": dense_tflops, "peak": pk["bf16_sustained"], "unit": "TFLOP/s",
                      "frac": dense_tflops / pk["bf16_sustained"], "peak_source": pk["src"] + " (sustained cuBLAS bf16)"}

    # ---------------- CPU baseline (rank 0, N = 1 only): bounded sample of the unmodified reference
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        n = 4 if H < 400 else 1
        v, cores, ts, kind = reference_cpu(cfg, n, 4)
        cpu = {"value": v, "unit": "maps/s", "cores": cores, "kind": kind,
               "sample": f"{n}-image batch x 4 repetitions of the same forward, fp32, "
                         + ("unmodified reference Python on torch CPU + torchvision deform_conv2d" if kind == "reference" else "oracle port")
                         + f"; {sum(ts):.1f} s timed"}

    if rank == 0:
        print(json.dumps({
            "metric": "depth maps/sec @228x304" if H == 228 else f"depth maps/sec @{H}x{W}", "value": value, "unit": "maps/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": t_ms / args.steps,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": args.precision if args.precision == "bf16" else "f32", "data": "synthetic",
            "config": workload_config(cfg, args, world, B), "clocks": clocks,
            "e2e": {"value": e2e, "unit": "maps/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "gpu_launches": n_launch * args.steps, "parity": parity, "value_fp32": value_fp32, "value_fp32_tc": value_fp32_tc, "ref_gpu": ref_gpu,
            "roofline": roofline, "roofline_dense": roofline_dense, "cpu_baseline": cpu}))
    if dumped is not None:
        write_outputs(args.dump_outputs, dumped)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
