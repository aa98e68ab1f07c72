"""RDF-GAN (bench.py config c2: DCVGANGenerator + ESANet-34, B = 32, 228x304, the bench's weights and inputs) in each precision:
what the guidance network costs and how far the bf16 / fp32_tc pipelines land from strict fp32 end to end.  Prints one JSON line.

    python scripts/rdfgan_precision.py [--reps 7] [--warmup 2] [--profile DIR]

Times are CUDA events around one call after warm-up, with 256 MiB written between repetitions so that no repetition reads the
previous one's activations or weights from L2; the median is reported.  Distances compare every pixel of the five output maps
of the (bf16, bf16) and (fp32_tc, fp32_tc) pipelines -- guidance network included -- with the (fp32, fp32) pipeline.
--profile DIR writes torch.profiler's per-kernel CUDA time table of one ESANet-34 call per precision to DIR/esanet_<precision>.txt.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

import bench  # noqa: E402
from _synth import synth_inputs  # noqa: E402

PRECISIONS = ("bf16", "fp32_tc", "fp32")


def gpu_info():
    """name and power limit of GPU 0, read-only query"""
    out = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True, check=True).stdout.strip()
    name, power = [s.strip() for s in out.split(",", 1)]
    return dict(gpu=name, power_limit=power)


def median_ms(fn, reps, warmup):
    flush = torch.empty(64 << 20, dtype=torch.float32, device="cuda")             # 256 MiB, twice the L2
    for _ in range(warmup):
        fn()
    ts = []
    for _ in range(reps):
        flush.fill_(1.0)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return statistics.median(ts)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--profile", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("rdfgan_precision.py measures on a GPU; none is visible")
    cfg = bench.CONFIGS["c2"]
    B, H, W = cfg["batch"], cfg["H"], cfg["W"]
    res = dict(gpu_info(), workload=f"bench.py c2: RDF-GAN (ESANet-34 + DCVGANGenerator ResNet-34), B={B}, {H}x{W}", B=B, H=H, W=W,
               timing=f"CUDA events, median of {args.reps} after {args.warmup} warm-up calls, 256 MiB written between repetitions")
    G = bench.build_product(cfg).cuda()
    esa = G.global_guidance_module
    rgb, _, depth = synth_inputs(B, H, W, seed=0, Cs=cfg["cs"])
    rgb, depth = rgb.cuda(), depth.cuda()
    res["esanet"], res["rdfgan"], outs, guid = {}, {}, {}, {}
    with torch.no_grad():
        for p in PRECISIONS:
            esa.set_precision(p)
            G.set_precision(p)
            ms = median_ms(lambda: esa(rgb), args.reps, args.warmup)
            res["esanet"][p] = dict(ms_per_batch=round(ms, 3), maps_per_s=round(B / ms * 1e3, 1))
            ms = median_ms(lambda: G(rgb, depth), args.reps, args.warmup)
            res["rdfgan"][f"{p}+{p}"] = dict(ms_per_batch=round(ms, 3), maps_per_s=round(B / ms * 1e3, 1))
            guid[p] = esa(rgb)
            outs[p] = dict(zip(bench.KEYS, G(rgb, depth)))
            if args.profile:
                os.makedirs(args.profile, exist_ok=True)
                with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
                    esa(rgb)
                    torch.cuda.synchronize()
                with open(os.path.join(args.profile, f"esanet_{p}.txt"), "w") as f:
                    f.write(f"{res['gpu']}, power limit {res['power_limit']}; one ESANet-34 call, B={B}, {H}x{W}, precision {p}\n")
                    f.write(prof.key_averages().table(sort_by="cuda_time_total", row_limit=40))
    ref = outs["fp32"]
    res["guidance_logits_rms_fp32"] = float(guid["fp32"].double().square().mean().sqrt())
    res["guidance_vs_fp32"] = {p: dict(rmse=float((guid[p] - guid["fp32"]).double().square().mean().sqrt()),
                                       max_abs=float((guid[p] - guid["fp32"]).abs().max())) for p in ("bf16", "fp32_tc")}
    res["maps_vs_fp32_end_to_end"] = {p: {k: dict(rmse=float((outs[p][k].float() - ref[k]).double().square().mean().sqrt()),
                                                  max_abs=float((outs[p][k].float() - ref[k]).abs().max())) for k in bench.KEYS}
                                      for p in ("bf16", "fp32_tc")}
    print(json.dumps(res))


if __name__ == "__main__":
    main()
