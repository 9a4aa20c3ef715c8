"""CPU: separate the error sources of the fp32-precision forward (UNetDC.precision = "fp32").

Evaluates the forward's arithmetic exactly (tests/split_model.py network: fp32 values as three bf16 planes, the six
plane products, exact sums, fp32 stores) and with all nine products, against the float64 network.  Whatever the GPU
forward's error exceeds this by comes from summing the products in the tensor cores' fp32 accumulator.

    python tools/split_emulation.py [--frames 2] [--size 256]
"""
import argparse
import sys
from pathlib import Path

import numpy as np
import torch

REPO = Path(__file__).resolve().parent.parent
sys.path[:0] = [str(REPO), str(REPO / "tests")]

import split_model as sm  # noqa: E402
from unet_dc_segmentation_b200.synth import calibrated_state_dict, synthetic_image  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--frames", type=int, default=2)
ap.add_argument("--size", type=int, default=256)
args = ap.parse_args()
sd = calibrated_state_dict(seed=0, calib_size=256, n_calib=1, fit_head=True)
u8 = np.stack([synthetic_image(args.size, 50 + i) for i in range(args.frames)])
x32 = torch.from_numpy(u8.astype(np.float32) / np.float32(255))[:, None].expand(-1, 3, -1, -1).contiguous()
p64 = sm.network(sd, x32)
nine = sm.TERMS + ((1, 2), (2, 1), (2, 2))
for name, terms in (("six terms (the kernel's)", sm.TERMS), ("all nine terms", nine)):
    d = (sm.network(sd, x32, terms) - p64).abs()
    print(f"{args.frames} x {args.size}^2, {name}: max |dp| {float(d.max()):.3e}, mean {float(d.mean()):.3e}")
