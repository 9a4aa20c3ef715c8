"""Speed and accuracy of UNetDC.precision = "fp32" against the default bf16 forward, on one B200.

Times the two precisions alternately in one process (CUDA events around warm forwards of u8 frames through
predict_u8, the product's entry point) at 32 x 1024^2 and 8 x 256^2, and measures max / mean |p - p64| against the
float64 network on one 1024^2 frame for both, beside the CPU fp32 network's own error.  Writes a markdown report.

    python tools/fp32_forward.py [--out report.md] [--reps 5]
"""
from __future__ import annotations

import argparse
import subprocess
import sys
import time
from pathlib import Path

import numpy as np
import torch

REPO = Path(__file__).resolve().parent.parent
sys.path[:0] = [str(REPO), str(REPO / "tests")]

import oracle  # noqa: E402
import split_model as sm  # noqa: E402
from unet_dc_segmentation_b200.model import UNetDC  # noqa: E402
from unet_dc_segmentation_b200.synth import calibrated_state_dict, synthetic_image  # noqa: E402

THRESH = 0.3


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[torch.cuda.current_device()] if q else torch.cuda.get_device_name()


def frames(B, size, base):
    return torch.from_numpy(np.stack([synthetic_image(size, base + i) for i in range(B)]))


def time_forward(m, u8, mask, reps):
    """ms per call of predict_u8 on device-resident frames, mean over `reps` calls after two warm calls."""
    for _ in range(2):
        m.predict_u8(u8, THRESH, mask_out=mask)
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    start.record()
    for _ in range(reps):
        m.predict_u8(u8, THRESH, mask_out=mask)
    stop.record()
    stop.synchronize()
    return start.elapsed_time(stop) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", help="also write the report to this file")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("fp32_forward.py measures on a GPU; none is visible")
    dev = torch.device("cuda", 0)
    sd = calibrated_state_dict(seed=0, calib_size=512, n_calib=1, fit_head=True)
    m = UNetDC()
    m.load_state_dict(sd)
    m = m.to(dev).eval()
    lines = ["# fp32-precision forward vs bf16 (tools/fp32_forward.py)", "",
             f"Card: {card()} (name, power limit, max SM clock, read in the same run).", ""]

    lines += ["## Forward time", "",
              "predict_u8 on device-resident u8 grey frames, CUDA events, warm; bf16 and fp32 alternate "
              f"{args.rounds} times in one process, {args.reps} calls per sample.  img/s = frames / mean time.", "",
              "| batch | precision | ms per batch (samples) | img/s |", "|---|---|---|---|"]
    for B, size in ((32, 1024), (8, 256)):
        u8 = frames(B, size, 10).to(dev)
        mask = torch.empty((B, size, size), dtype=torch.uint8, device=dev)
        t = {"bf16": [], "fp32": []}
        for _ in range(args.rounds):
            for prec in ("bf16", "fp32"):
                m.precision = prec
                t[prec].append(time_forward(m, u8, mask, args.reps))
        for prec in ("bf16", "fp32"):
            ms = float(np.mean(t[prec]))
            lines.append(f"| {B} x {size}^2 | {prec} | {ms:.2f} ({', '.join(f'{v:.2f}' for v in t[prec])}) | "
                         f"{B * 1000.0 / ms:.1f} |")
        m.packed().workspace = None
        del u8, mask
        torch.cuda.empty_cache()

    lines += ["", "## Error against the float64 network (one 1024^2 frame)", "",
              "Input u8 / 255 in fp32 (IEEE division, as the reference preprocesses); float64 = split_model.network "
              "(tests/, BatchNorm folded in float64) on the same fp32 input; CPU fp32 = oracle.unetdc_forward (PyTorch CPU, fp32).",
              "", "| forward | max abs dp | mean abs dp | mask pixels differing from float64 |", "|---|---|---|---|"]
    u8 = frames(1, 1024, 900)
    x32 = torch.from_numpy(u8.numpy().astype(np.float32) / np.float32(255))[:, None].expand(1, 3, 1024, 1024).contiguous()
    t0 = time.time()
    p64 = sm.network(sd, x32)
    t64 = time.time() - t0
    m64 = p64 > THRESH
    rows = {"CPU fp32 network": oracle.unetdc_forward(sd, x32)[:, 0].double()}
    for prec in ("bf16", "fp32"):
        m.precision = prec
        _, prob = m.predict_u8(u8.to(dev), THRESH, return_prob=True)
        rows[f"B200 {prec}"] = prob[:, 0].double().cpu()
    for name, p in rows.items():
        d = (p - p64).abs()
        lines.append(f"| {name} | {float(d.max()):.3e} | {float(d.mean()):.3e} | {int(((p > THRESH) != m64).sum())} |")
    lines += ["", f"(float64 host reference: {t64:.1f} s.)", ""]
    text = "\n".join(lines) + "\n"
    if args.out:
        Path(args.out).write_text(text)
    print(text)


if __name__ == "__main__":
    main()
