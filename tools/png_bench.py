"""CUDA-event time of dc_png_encode per batch -- 32 masks (x 255, as qdb:58 writes them) and 32 overlays (noisy BGR
frames with painted contours, qdb:78) of 1024^2 by default -- next to the time cv2.imencode takes for the same files on a
host thread pool:
    python tools/png_bench.py [--batch 32] [--size 1024] [--reps 20] [--threads 16]"""
import argparse
import json
import subprocess
import sys
import time
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

import numpy as np
import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
from unet_dc_segmentation_b200.png import encode_png_device, png_bounds  # noqa: E402
from unet_dc_segmentation_b200.synth import synthetic_image, synthetic_mask  # noqa: E402


def frames(batch, size):
    masks = np.stack([synthetic_mask(size, 3300, seed=s) * 255 for s in range(batch)])
    grey = np.stack([synthetic_image(size, 100 + s, n_droplets=300) for s in range(batch)])
    over = np.repeat(grey[..., None], 3, 3)
    edge = (masks > 0) & ~np.roll(masks > 0, 1, axis=2)
    over[edge] = (0, 255, 0)
    return masks.astype(np.uint8), over


def time_device(x, reps):
    need, wsb = png_bounds(x.shape[0], x.shape[1], x.shape[2], 1 if x.dim() == 3 else 3)
    out = torch.empty(need, dtype=torch.uint8, device=x.device)
    ws = torch.empty(wsb, dtype=torch.uint8, device=x.device)
    for _ in range(3):
        _, off = encode_png_device(x, out, ws)
    torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ev[0].record()
    for _ in range(reps):
        encode_png_device(x, out, ws)
    ev[1].record()
    torch.cuda.synchronize()
    return ev[0].elapsed_time(ev[1]) / reps, int(off[-1].item()), out, off


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--size", type=int, default=1024)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--threads", type=int, default=16)
    a = ap.parse_args()
    import cv2
    dev = torch.device("cuda", 0)
    res = {}
    for name, host in zip(("masks", "overlays"), frames(a.batch, a.size)):
        ms, nbytes, out, off = time_device(torch.from_numpy(host).to(dev), a.reps)
        o = off.cpu().numpy()
        data = out[:int(o[-1])].cpu().numpy().tobytes()
        with ThreadPoolExecutor(a.threads) as pool:
            t0 = time.perf_counter()
            want = list(pool.map(lambda im: cv2.imencode(".png", im)[1].tobytes(), host))
            host_s = time.perf_counter() - t0
        same = all(data[o[b]:o[b + 1]] == want[b] for b in range(a.batch))
        res[name] = {"dc_png_encode_ms_per_batch": ms, "png_bytes": nbytes, "cv2_pool_ms_per_batch": host_s * 1e3,
                     "identical": same}
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    print(json.dumps({"gpu": smi[0] if smi else None, "batch": a.batch, "size": a.size, "threads": a.threads, **res}))


if __name__ == "__main__":
    main()
