"""Development aid: the filter gradient on the training step's layer shapes (B = 16 per GPU, 228x304): the tcgen05 kernel
(csrc/wgrad_umma.cu) against cuDNN's wgrad (torch.nn.grad.conv2d_weight, bf16)."""
import os, sys
import torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from rdfc_gan_b200.train_ops import _wgrad

B = int(os.environ.get("B", 16))
# (G channels, I channels, G grid, I grid, stride, count per step, name)
LAYERS = [
    (64, 64, (228, 304), (228, 304), 1, 8, "64->64 @228x304"),
    (160, 128, (228, 304), (228, 304), 1, 1, "128->160 @228x304 (d.dec1)"),
    (96, 128, (228, 304), (228, 304), 1, 1, "128->96 @228x304 (r.dec1)"),
    (128, 64, (114, 152), (228, 304), 2, 2, "64->128 s2 @228x304"),
    (128, 128, (114, 152), (114, 152), 1, 6, "128->128 @114x152"),
    (256, 128, (57, 76), (114, 152), 2, 2, "128->256 s2"),
    (256, 256, (57, 76), (57, 76), 1, 6, "256->256 @57x76"),
    (512, 256, (29, 38), (57, 76), 2, 2, "256->512 s2"),
    (512, 512, (29, 38), (29, 38), 1, 6, "512->512 @29x38"),
    (512, 512, (15, 19), (29, 38), 2, 2, "512->512 s2 (en6)"),
    (192, 64, (114, 152), (228, 304), 2, 2, "convT 192->64 (de2): G := layer input"),
    (384, 64, (57, 76), (114, 152), 2, 2, "convT 384->64 (de3)"),
    (768, 128, (29, 38), (57, 76), 2, 2, "convT 768->128 (de4)"),
    (512, 256, (15, 19), (29, 38), 2, 2, "convT 512->256 (de5)"),
]

def timeit(fn, reps=10):
    for _ in range(3): fn()
    torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
    for a, b in ev:
        a.record(); fn(); b.record()
    torch.cuda.synchronize()
    return sorted(a.elapsed_time(b) for a, b in ev)[reps // 2]

tot = {"umma": 0.0, "cuDNN": 0.0}
for O, I, (Hg, Wg), (Hi, Wi), s, cnt, name in LAYERS[:int(os.environ.get("NLAYERS", len(LAYERS)))]:
    g = torch.Generator(device="cuda").manual_seed(1)
    gy = torch.randn(B, Hg, Wg, O, device="cuda", generator=g).to(torch.bfloat16)
    x = torch.randn(B, Hi, Wi, I, device="cuda", generator=g).to(torch.bfloat16)
    flops = 2.0 * O * I * 9 * B * Hg * Wg
    t = timeit(lambda: _wgrad(gy, x, 3, s))
    tot["umma"] += cnt * t
    line = f"{name:42s} umma {t*1e3:7.1f} us ({flops/t/1e9:6.0f} TF/s)"
    if os.environ.get("CUDNN", "1") == "1":
        xn, gn = x.permute(0, 3, 1, 2), gy.permute(0, 3, 1, 2)        # channels-last views
        tc = timeit(lambda: torch.nn.grad.conv2d_weight(xn, (O, I, 3, 3), gn, stride=s, padding=1))
        tot["cuDNN"] += cnt * tc
        ref = torch.nn.grad.conv2d_weight(xn, (O, I, 3, 3), gn, stride=s, padding=1).float()
        rel = float((_wgrad(gy, x, 3, s) - ref).norm() / ref.norm())
        line += f" | cuDNN bf16 {tc*1e3:7.1f} us | rel diff {rel:.1e}"
    print(line, flush=True)
print(f"per training step (counts weighted): umma {tot['umma']:.2f} ms, cuDNN {tot['cuDNN']:.2f} ms")
