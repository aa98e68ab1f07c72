"""Development aid: CUDA-event time of every step of the generator plan, run eagerly (one C-ABI call per step).
    python scripts/prof_plan.py [B] [precision] [--json path]
Prints the steps sorted by time plus the per-kernel-family totals; with --json writes the table for profiles/.
"""
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import bench  # noqa: E402
from rdfc_gan_b200 import _cabi as C  # noqa: E402
from _synth import synth_inputs  # noqa: E402


def main():
    args = [a for a in sys.argv[1:] if not a.startswith("--")]
    B = int(args[0]) if args else 32
    prec = args[1] if len(args) > 1 else "bf16"
    out_json = sys.argv[sys.argv.index("--json") + 1] if "--json" in sys.argv else None
    dev = torch.device("cuda", 0)
    cfg = bench.CONFIGS[os.environ.get("CONFIG", "c3")]
    G = bench.build_product(cfg).to(dev).set_precision(prec)
    rgb, normal, depth = synth_inputs(B, cfg["H"], cfg["W"], seed=0, Cs=cfg["cs"])
    with torch.no_grad():
        bench.call_generator(G, cfg, rgb.to(dev), normal.to(dev), depth.to(dev))
    plan = next(iter(G.engine()._plans.values()))
    assert len(plan.names) == len(plan.steps), (len(plan.names), len(plan.steps))
    s = C.stream_ptr()
    reps = 5
    acc = [[] for _ in plan.steps]
    for rep in range(reps + 2):
        evs = []
        for f in plan.steps:
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            f(s)
            b.record()
            evs.append((a, b))
        torch.cuda.synchronize()
        if rep >= 2:
            for i, (a, b) in enumerate(evs):
                acc[i].append(a.elapsed_time(b) * 1e3)
    med = [sorted(v)[len(v) // 2] for v in acc]
    total = sum(med)
    rows = sorted(zip(med, plan.names), reverse=True)
    print(f"plan B={B} {prec}: {len(plan.steps)} steps, sum of step medians {total/1e3:.2f} ms")
    for t, n in rows:
        print(f"  {t:9.1f} us  {100*t/total:5.1f}%  {n}")
    fam = {}
    for t, n in zip(med, plan.names):
        k = n.split()[0] + (" " + n.split()[-1] if n.startswith("conv") else "")
        fam[k] = fam.get(k, 0.0) + t
    print("families:")
    for k, t in sorted(fam.items(), key=lambda kv: -kv[1]):
        print(f"  {t/1e3:8.2f} ms  {100*t/total:5.1f}%  {k}")
    if "--timers" in sys.argv:      # needs a -DRDFC_UMMA_TIMERS build and RDFC_UMMA_DBG=1
        import ctypes
        import numpy as np
        pats = sys.argv[sys.argv.index("--timers") + 1].split(",")
        names = {0: "MMA warp lifetime", 1: "MMA wait ACC_EMPTY", 2: "MMA wait A_FULL", 3: "MMA wait B_FULL", 5: "Bload wait B_EMPTY",
                 9: "epi wait ACC_FULL", 10: "epi work", 11: "MMA issue (elected)", 12: "MMA commits", 13: "CTA lifetime"}
        for f, n in zip(plan.steps, plan.names):
            if any(pat in n for pat in pats):
                f(s)
                torch.cuda.synchronize()
                buf = (ctypes.c_longlong * (148 * 16))()
                C.lib.rdfc_dev_umma_timers(buf, 148 * 16)
                a = np.frombuffer(buf, dtype=np.int64).reshape(148, 16).astype(np.float64)
                a = a[a[:, 0] > 0]
                print(f"role timers for step '{n}' (cycles, median over {len(a)} CTAs; CTA lifetime max {a[:, 13].max():.0f}, "
                      f"last CTA end - first CTA end {(a[:, 14].max() - a[:, 14].min()) / 1e3:.1f} us, "
                      f"first start -> last end {(a[:, 14].max() - a[:, 15].min()) / 1e3:.1f} us, "
                      f"last start - first start {(a[:, 15].max() - a[:, 15].min()) / 1e3:.1f} us, "
                      f"CTA lifetime min {a[:, 13].min():.0f}):")
                for i, nm in names.items():
                    print(f"   {nm:20s} {np.median(a[:, i]):10.0f}  ({100*np.median(a[:, i])/np.median(a[:, 0]):5.1f}%)")
    if out_json:
        json.dump({"B": B, "precision": prec, "total_us": total, "steps": [{"name": n, "us": t} for t, n in zip(med, plan.names)],
                   "families_us": fam}, open(out_json, "w"), indent=1)


if __name__ == "__main__":
    main()
