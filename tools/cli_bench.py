"""Files in -> files out through the drop-in CLI (cli.main), timed on the wall clock for both loops:
    python tools/cli_bench.py [--n 8] [--size 256] [--batch 8] [--img_size 512] [--reps 3] [--excel] [--fast_only]
                              [--overlays] [--repo PATH]
BASELINE config 1 = 8 frames of 256x256, batch 8, --img_size 512 (the reference's IMG_SIZE).  --excel drops
--skip_excel (without xlsxwriter the CLI then writes all_droplets_noexcel.csv); --repo times the package of another
checkout (A/B of two versions in one process-free comparison: run the script once per tree); --overlays adds
--save_overlays (an overlay PNG per frame)."""
import argparse
import json
import shutil
import sys
import tempfile
import time
from pathlib import Path

import torch
from PIL import Image

REPO = Path(__file__).resolve().parent.parent


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repo", default=str(REPO))
    ap.add_argument("--excel", action="store_true")
    ap.add_argument("--fast_only", action="store_true")
    ap.add_argument("--overlays", action="store_true")
    ap.add_argument("--frames_dir", help="keep the generated frames and checkpoint here and reuse them on later runs")
    ap.add_argument("--n", type=int, default=8)
    ap.add_argument("--size", type=int, default=256)
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--img_size", type=int, default=512)
    ap.add_argument("--reps", type=int, default=3)
    a = ap.parse_args()
    sys.path.insert(0, str(Path(a.repo).resolve()))
    from unet_dc_segmentation_b200 import cli
    from unet_dc_segmentation_b200.synth import calibrated_state_dict, synthetic_image
    d = Path(tempfile.mkdtemp(prefix="cli_bench_"))
    src = Path(a.frames_dir) if a.frames_dir else d
    if not (src / "ckpt.pth").exists() or len(list((src / "in").glob("*.png"))) != a.n:
        (src / "in").mkdir(parents=True, exist_ok=True)
        for i in range(a.n):
            Image.fromarray(synthetic_image(a.size, i)).save(src / "in" / f"frame{i:04d}.png")
        torch.save(calibrated_state_dict(seed=0), src / "ckpt.pth")
    common = ["--img_dir", str(src / "in"), "--ckpt_path", str(src / "ckpt.pth"), "--batch", str(a.batch), "--img_size",
              str(a.img_size), "--skip_histogram", "--px_per_micron", "3.45"] + ([] if a.excel else ["--skip_excel"]) + (["--save_overlays"] if a.overlays else [])
    out = {"repo": str(a.repo), "frames": a.n, "size": a.size, "batch": a.batch, "img_size": a.img_size,
           "excel": a.excel, "overlays": a.overlays}
    loops = (("fast", []),) if a.fast_only else (("fast", []), ("reference_loop", ["--reference_loop"]))
    for tag, extra in loops:
        times = []
        for r in range(a.reps + 1):                                  # first repetition = warm-up (library load, cuda init)
            od = d / f"out_{tag}_{r}"
            t0 = time.perf_counter()
            cli.main(common + extra + ["--out_dir", str(od)])
            torch.cuda.synchronize()
            times.append(time.perf_counter() - t0)
        out[tag] = {"seconds_first": times[0], "seconds_best": min(times[1:]), "images_per_s": a.n / min(times[1:])}
    print(json.dumps(out))
    shutil.rmtree(d, ignore_errors=True)


if __name__ == "__main__":
    main()
