"""Rolling-ball radius sweep: CUDA-event ms per batch of the tiled kernel and the banded pass (dc_rolling_ball /
dc_rolling_ball_banded) on grayscale planar batches, launches per call, and cv2's single-frame opening on the host.

    python tools/rb_radius_sweep.py [--reps 5] [--json out.json]

Prints a markdown table (the form of profiles/r03_rolling_ball_radius_sweep.md).  Both paths are bit-exact; every
timed output is checked against the other path (radii both run) before it is reported."""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))

import numpy as np  # noqa: E402
import torch  # noqa: E402

from unet_dc_segmentation_b200.morphology import (rolling_ball_device, rolling_ball_workspace_bytes,  # noqa: E402
                                                  tiled_max_radius)
from unet_dc_segmentation_b200.synth import synthetic_image  # noqa: E402

BATCHES = [(32, 1024), (64, 2048)]
BOTH = [50, 100]                       # + tiled_max_radius(): both paths, for the crossover
BANDED = [175, 256, 300, 511, 1023, 2047]
CV2_MAX_RADIUS = 300                   # cv2's opening on a 1024^2 frame grows ~x4 per doubling of the radius


def gpu_info() -> str:
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as exc:                     # the table still names torch's device
        return f"{torch.cuda.get_device_name()} (nvidia-smi: {exc})"


def launches_per_call(x, radius, method) -> int:
    from torch.profiler import ProfilerActivity, profile
    rolling_ball_device(x, radius, method=method)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        rolling_ball_device(x, radius, method=method)
        torch.cuda.synchronize()
    return sum(1 for e in prof.events() if e.device_type.name == "CUDA")          # kernels on the device


def time_ms(x, radius, method, out, ws, reps) -> float:
    rolling_ball_device(x, radius, out=out, workspace=ws, method=method)          # warm-up (module load, attributes)
    torch.cuda.synchronize()
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    times = []
    for _ in range(reps):
        start.record()
        rolling_ball_device(x, radius, out=out, workspace=ws, method=method)
        end.record()
        end.synchronize()
        times.append(start.elapsed_time(end))
    return float(np.median(times))


def main(argv=None) -> int:
    ap = argparse.ArgumentParser(description=__doc__)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--json", type=Path)
    args = ap.parse_args(argv)
    if not torch.cuda.is_available():
        raise SystemExit("rb_radius_sweep measures on the GPU; no CUDA device found")
    both = BOTH + [tiled_max_radius()]
    rows = []
    for B, n in BATCHES:
        frame = synthetic_image(n, 0)
        x = torch.from_numpy(np.ascontiguousarray(np.broadcast_to(frame, (B, n, n)))).cuda()
        out = torch.empty_like(x)
        ws = torch.empty(rolling_ball_workspace_bytes(B, n, n), dtype=torch.uint8, device="cuda")
        for r in both + BANDED:
            methods = ["tiled", "banded"] if r in both else ["banded"]
            res = {}
            for m in methods:
                res[m] = time_ms(x, r, m, out, ws, args.reps)
                if m == "tiled":
                    want = out.clone()
                elif "tiled" in res:
                    assert torch.equal(out, want), f"tiled != banded at radius {r}, {B} x {n}^2"
            rows.append({"batch": f"{B} x {n}^2", "radius": r, "tiled_ms": res.get("tiled"), "banded_ms": res["banded"],
                         "launches": launches_per_call(x[:1], r, methods[-1])})
            print(json.dumps(rows[-1]), flush=True)
        del x, out, ws
        torch.cuda.empty_cache()
    import cv2
    img = synthetic_image(1024, 0)
    cv2_ms = {}
    for r in both + BANDED:
        if r > CV2_MAX_RADIUS:
            continue
        k = cv2.getStructuringElement(cv2.MORPH_ELLIPSE, (r, r))
        t0 = time.perf_counter()
        cv2.morphologyEx(img, cv2.MORPH_OPEN, k)
        cv2_ms[r] = (time.perf_counter() - t0) * 1e3
    info = gpu_info()
    print(f"\nGPU: {info}; cv2 {cv2.__version__} with {cv2.getNumThreads()} threads\n")
    print("| batch | radius | tiled ms | banded ms | launches | cv2 opening, one 1024^2 frame, ms |")
    print("|---|---:|---:|---:|---:|---:|")
    for row in rows:
        t = f"{row['tiled_ms']:.3f}" if row["tiled_ms"] is not None else "-"
        c = f"{cv2_ms[row['radius']]:.0f}" if row["radius"] in cv2_ms and row["batch"].endswith("1024^2") else "-"
        print(f"| {row['batch']} | {row['radius']} | {t} | {row['banded_ms']:.3f} | {row['launches']} | {c} |")
    if args.json:
        args.json.parent.mkdir(parents=True, exist_ok=True)
        args.json.write_text(json.dumps({"gpu": info, "rows": rows, "cv2_ms_1024": cv2_ms}, indent=1))
    return 0


if __name__ == "__main__":
    sys.exit(main())
