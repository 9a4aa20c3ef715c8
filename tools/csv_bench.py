"""CUDA-event time of dc_table_csv (droplet table -> per-image CSV text) per batch, next to the host time pandas takes
for the same text (DataFrame + insert + to_csv of every frame):
    python tools/csv_bench.py [--batch 32] [--size 1024] [--discs 3300] [--reps 50]
The default batch is the 32 x 1024^2 job of profiles/r02_cli_timing.md at about 3 k droplets per frame."""
import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np
import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
from unet_dc_segmentation_b200.quantify import (COLUMNS, MICRON_COLUMNS, csv_field, csv_text_device,  # noqa: E402
                                                label_stats_device, pack_fields, tables_to_csv)
from unet_dc_segmentation_b200.synth import synthetic_mask  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--size", type=int, default=1024)
    ap.add_argument("--discs", type=int, default=3300)
    ap.add_argument("--reps", type=int, default=50)
    a = ap.parse_args()
    dev = torch.device("cuda", 0)
    masks = torch.from_numpy(np.stack([synthetic_mask(a.size, a.discs, seed=s) for s in range(a.batch)])).to(dev)
    t = label_stats_device(masks, 1, 3.45)
    names = [f"frame{i:04d}.png" for i in range(a.batch)]
    buf, offs = pack_fields([csv_field(n) for n in names])
    d_names, d_off = torch.from_numpy(buf.copy()).to(dev), torch.from_numpy(offs).to(dev)
    for _ in range(5):
        out, off, _ = csv_text_device(t, d_names, d_off, int(offs[-1]))
    torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ev[0].record()
    for _ in range(a.reps):
        csv_text_device(t, d_names, d_off, int(offs[-1]))
    ev[1].record()
    torch.cuda.synchronize()
    dev_ms = ev[0].elapsed_time(ev[1]) / a.reps                  # includes the four launches and the buffer allocation
    texts = tables_to_csv(t, names).texts
    import pandas as pd
    cols = t.to_host()
    t0 = time.perf_counter()
    for b, c in enumerate(cols):
        df = pd.DataFrame({k: c[k] for k in COLUMNS + MICRON_COLUMNS})
        df.insert(0, "filename", names[b])
        want = df.to_csv(index=False).encode()
        assert want == texts[b], b
    host_s = time.perf_counter() - t0
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    print(json.dumps({"gpu": smi[0] if smi else None, "batch": a.batch, "size": a.size,
                      "rows": int(t.counts.sum().item()), "text_bytes": int(off[-1].item()),
                      "dc_table_csv_ms_per_batch": dev_ms, "pandas_s_per_batch": host_s}))


if __name__ == "__main__":
    main()
