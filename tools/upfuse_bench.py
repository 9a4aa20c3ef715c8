"""Level 1 of the decoder at the benchmark shape (32 x 512 x 512 x 128 -> 32 x 1024 x 1024 x 64): upconv1 + dec1.0 as two
launches against dc_conv_upfused, CUDA events, median of N."""
import statistics
import sys

import torch

sys.path.insert(0, ".")
from unet_dc_segmentation_b200 import layers                                    # noqa: E402
from unet_dc_segmentation_b200.model import compose_upconv, pack_conv3x3, pack_upconv, pack_upfused   # noqa: E402

B, H, W = (int(v) for v in sys.argv[1:4]) if len(sys.argv) > 3 else (32, 512, 512)
dev = torch.device("cuda:0")
g = torch.Generator().manual_seed(0)
wu = torch.randn(128, 64, 2, 2, generator=g) / 128 ** 0.5
bu = torch.randn(64, generator=g) * 0.3
wd = torch.randn(64, 128, 3, 3, generator=g) / (3.0 * 128 ** 0.5)
bd = torch.randn(64, generator=g) * 0.1
comp, skipw, fb = compose_upconv(wu, bu, wd, bd)
fw, fb = pack_upfused(comp, skipw).to(dev), fb.to(dev)
pu, pd = pack_upconv(wu).to(dev), pack_conv3x3(wd).to(dev)
bu_d, bd_d = bu.to(dev), bd.to(dev)
x = torch.randn((B, H, W, 128), device=dev).bfloat16()
cat = torch.randn((B, 2 * H, 2 * W, 128), device=dev).bfloat16()
out = torch.empty((B, 2 * H, 2 * W, 64), dtype=torch.bfloat16, device=dev)
out2 = torch.empty_like(out)


def two():
    layers.upconv2x2(x, pu, bu_d, out=cat, out_offset=0)
    layers.conv3x3(cat, pd, bd_d, out=out)


def fused():
    layers.upconv_conv3x3(x, cat, fw, fb, skip_offset=64, out=out2)


def timed(fn, n=7):
    ts = []
    for _ in range(n):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); fn(); b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return statistics.median(ts[2:])


t2, tf = timed(two), timed(fused)
d = (out.float() - out2.float()).abs()
print(f"B {B} H {H} W {W}: upconv1 + dec1.0 as two launches {t2:.3f} ms, fused {tf:.3f} ms, "
      f"max |diff| {float(d.max()):.4f} mean {float(d.mean()):.5f}")


# ---- levels 2..4 at the benchmark shapes: upconv + dec.0 as two launches against conv_upfused_wide_kernel
from unet_dc_segmentation_b200.model import pack_upfused_wide                    # noqa: E402
for C, Hh in ((128, 256), (256, 128), (512, 64)):
    wu = torch.randn(2 * C, C, 2, 2, generator=g) / (2 * C) ** 0.5
    bu = torch.randn(C, generator=g) * 0.3
    wd = torch.randn(C, 2 * C, 3, 3, generator=g) / (3.0 * (2 * C) ** 0.5)
    bd = torch.randn(C, generator=g) * 0.1
    comp, skipw, fb = compose_upconv(wu, bu, wd, bd)
    wx, ws = (t.to(dev) for t in pack_upfused_wide(comp, skipw))
    fb = fb.to(dev)
    pu, pd = pack_upconv(wu).to(dev), pack_conv3x3(wd).to(dev)
    bu_d, bd_d = bu.to(dev), bd.to(dev)
    x = torch.randn((B, Hh, Hh, 2 * C), device=dev).bfloat16()
    cat = torch.randn((B, 2 * Hh, 2 * Hh, 2 * C), device=dev).bfloat16()
    o1 = torch.empty((B, 2 * Hh, 2 * Hh, C), dtype=torch.bfloat16, device=dev)
    o2 = torch.empty_like(o1)

    def two():
        layers.upconv2x2(x, pu, bu_d, out=cat, out_offset=0)
        layers.conv3x3(cat, pd, bd_d, out=o1)

    def fusedw():
        layers.upconv_conv3x3(x, cat, wx, fb, skip_offset=C, out=o2, weight_skip=ws)

    t2, tf = timed(two), timed(fusedw)
    d = (o1.float() - o2.float()).abs()
    print(f"C {C} ({Hh}^2 -> {2 * Hh}^2): two launches {t2:.3f} ms, fused {tf:.3f} ms, max |diff| {float(d.max()):.4f} mean {float(d.mean()):.5f}")
