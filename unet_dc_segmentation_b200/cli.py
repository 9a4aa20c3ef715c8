"""Drop-in front end for reference quantify_droplets_batch.py: same functions, same flags, same output files,
with the device work done by libunetdc_b200 (rolling ball, UNetDC, threshold, labelling, droplet table).

    python -m unet_dc_segmentation_b200.cli --img_dir IN --ckpt_path model.pth --out_dir OUT [flags as the reference]

Function-for-function (reference file:line):
    load_model   qdb:34-37     preprocess  qdb:40-46     run_batch  qdb:48-79     quantify  qdb:81-95
    main         qdb:100-201   (argparse flags qdb:101-128; report files qdb:163-199, read back by gui_qt.py:470-589)

On the device: rolling ball, both resizes (cv2.resize at qdb:44 and qdb:57 is bilinear -- the reference passes the
interpolation flag in the `dst` slot, SURVEY.md 0.2 -- reproduced bit for bit by dc_resize_linear_u8; the identity
when the frame is already IMG_SIZE), the network, the threshold, labelling, the table and the overlay contours (qdb:76-77,
bit-exact against OpenCV's findContours + drawContours).  On the host, exactly as in the reference: PIL / cv2 decode,
PNG / CSV / XLSX writing.  Added flags: `--img_size` (default 512 = the reference's
IMG_SIZE constant) and `--density_maps` (the per-image maps of the reference's second front end, quantify_pipline.py:131-141).  Under torchrun (one rank per GPU) frames are sharded i -> rank i mod N, every
rank writes the per-image files of its own frames, and the tables are gathered on rank 0, which writes the reports.

``main`` runs the FAST path (``run_fast``): frames are decoded by a thread pool, batched, and streamed through
``DropletPipeline.run_host_pipelined`` -- u8 frames up, u8 masks (+ overlay stencils) and table rows down, nothing
else crosses PCIe -- while another pool writes the PNG / CSV files.  ``preprocess`` / ``run_batch`` keep the
reference's function-by-function shape (per-image round trips) for callers that use them as a library;
``--reference_loop`` makes ``main`` use them.
"""
from __future__ import annotations

import argparse
import sys
from pathlib import Path

import numpy as np
import torch

from .model import UNetDC
from .morphology import resize_linear_u8_device, rolling_ball_device
from .density import normalize, radial_density_device, roi_mask_device, spatial_density_device
from .overlay import draw_overlay, overlay_stencil_device
from .quantify import label_stats_device
from .quantify import quantify

IMG_SIZE = 512                     # qdb:30
SUFFIXES = {".png", ".jpg", ".jpeg", ".tif", ".tiff"}     # qdb:143-144


def _device() -> torch.device:
    if not torch.cuda.is_available():
        raise RuntimeError("unet_dc_segmentation_b200 needs an sm_100 GPU; there is no CPU path")
    return torch.device("cuda", torch.cuda.current_device())


def load_model(ckpt) -> UNetDC:
    """qdb:34-37: build UNetDC(3, 1), load the checkpoint's state_dict, eval mode on the GPU."""
    dev = _device()
    with torch.device("meta"):                     # no random initialisation of 31 M parameters that are about to be replaced
        m = UNetDC(in_channels=3, out_channels=1)
    m.load_state_dict(torch.load(ckpt, map_location=dev), assign=True)
    return m.to(dev).eval()


def preprocess(path, background_radius: int, img_size: int | None = None):
    """qdb:40-46: decode to RGB, rolling-ball correct, resize to the network size, /255, HWC -> CHW.
    Returns (f32 [3,S,S] tensor on the GPU, (oh, ow))."""
    from PIL import Image
    size = IMG_SIZE if img_size is None else int(img_size)
    im = np.array(Image.open(path).convert("RGB"))
    oh, ow = im.shape[:2]
    x = torch.from_numpy(im).to(_device())[None]                               # u8 [1,oh,ow,3]
    x = rolling_ball_device(x, background_radius)                             # qdb:43
    if (oh, ow) != (size, size):
        x = resize_linear_u8_device(x, (size, size))                          # qdb:44 (effectively INTER_LINEAR)
    # IEEE division as numpy does it at qdb:45 (torch turns `/ python_scalar` into a multiply by the reciprocal)
    scale = torch.full((), 255.0, dtype=torch.float32, device=x.device)
    return torch.div(x[0].to(torch.float32), scale).permute(2, 0, 1), (oh, ow)    # qdb:45-46


@torch.no_grad()
def run_batch(tensors, meta, model, mask_dir, overlay_dir, thresh, min_area, px_per_um, per_image_rows, all_props,
              density_dir=None):
    """qdb:48-79: forward one batch, then per image: mask, PNG, droplet table, CSV, summary row, overlay.
    density_dir: also write the radial / spatial density maps of the reference's quantify_pipline.py:131-141."""
    import cv2
    dev = next(model.parameters()).device
    batch = torch.stack(tensors).to(dev)
    probs = model(batch.contiguous())
    masks_dev = (probs[:, 0] > thresh).to(torch.uint8)                        # qdb:56
    for i in range(len(tensors)):
        fpath, (oh, ow) = meta[i]
        name = Path(fpath).stem
        m = masks_dev[i:i + 1]
        if tuple(m.shape[1:]) != (oh, ow):
            m = resize_linear_u8_device(m, (ow, oh))                          # qdb:57 (effectively INTER_LINEAR)
        mask = m[0].cpu().numpy()
        cv2.imwrite(str(Path(mask_dir) / f"{name}_pred.png"), mask * 255)
        df = quantify(mask, min_area, px_per_um)
        df.insert(0, "filename", Path(fpath).name)
        df.to_csv(Path(mask_dir).parent / f"{name}_droplets.csv", index=False)
        all_props.append(df)
        per_image_rows.append({"filename": Path(fpath).name, "droplet_count": len(df),
                               "total_area_px": df["area"].sum() if not df.empty else 0})
        if overlay_dir is not None:
            img = cv2.imread(str(fpath))                                              # qdb:75
            if img is not None:
                # qdb:76-77: the pixels findContours(RETR_EXTERNAL) + drawContours(thickness 2) paint, from the GPU
                draw_overlay(img, overlay_stencil_device(m)[0].cpu().numpy())
                cv2.imwrite(str(Path(overlay_dir) / f"{name}_overlay.png"), img)      # qdb:78
        if density_dir is not None:
            save_density_maps(fpath, name, m, density_dir)


def save_density_maps(fpath, name, mask_dev, density_dir) -> None:
    """quantify_pipline.py:131-141 for one image: ROI mask of the ORIGINAL frame, its centroid, droplets per concentric
    ring and the Gaussian droplet density, all on the device.  Writes {name}_radial_density.npy / _spatial_density.npy
    (the exact f32 maps) and, when matplotlib is installed, the reference's two 'hot' PNGs of the normalised maps."""
    from PIL import Image
    orig = np.array(Image.open(fpath).convert("RGB"))                                  # qpl:131
    roi, cen = roi_mask_device(torch.from_numpy(orig).to(mask_dev.device)[None])       # qpl:132-136
    t = label_stats_device(mask_dev, 1, None)                                          # qpl:66-68 (no size filter)
    n = int(t.counts.max().item())
    if n > t.capacity:
        t = label_stats_device(mask_dev, 1, None, n)
    radial = radial_density_device(roi, cen, t, 10)[0].cpu().numpy()                   # qpl:138
    spatial = spatial_density_device(mask_dev, roi)[0].cpu().numpy()                   # qpl:139
    np.save(Path(density_dir) / f"{name}_radial_density.npy", radial)
    np.save(Path(density_dir) / f"{name}_spatial_density.npy", spatial)
    try:
        import matplotlib
        matplotlib.use("Agg")
        import matplotlib.pyplot as plt
    except ImportError:
        return
    plt.imsave(Path(density_dir) / f"{name}_radial_density.png", normalize(radial), cmap="hot")      # qpl:140
    plt.imsave(Path(density_dir) / f"{name}_spatial_density.png", normalize(spatial), cmap="hot")    # qpl:141


def combined_csv_text(all_props, csv_texts):
    """all_droplets.csv without formatting every number a second time: when every frame has droplets (so that every
    per-image table has the same columns and dtypes) the text of ``pd.concat(all_props).to_csv(index=False)`` is the
    header plus the bodies of the per-image CSVs.  Returns None when that does not hold (pandas does it then)."""
    if not csv_texts or len(csv_texts) != len(all_props) or any(t is None for t in csv_texts):
        return None
    cols = list(all_props[0].columns)
    if any(df.empty or list(df.columns) != cols for df in all_props):
        return None
    header = csv_texts[0].split("\n", 1)[0] + "\n"
    return header + "".join(t.split("\n", 1)[1] for t in csv_texts)


def write_reports(out_dir: Path, per_image_rows, all_props, skip_excel: bool, skip_histogram: bool, csv_texts=None) -> None:
    """qdb:163-199: summary_per_image.csv, all_droplets.csv (+xlsx or the noexcel copy), stats, histogram."""
    import pandas as pd
    summary_df = pd.DataFrame(per_image_rows)
    summary_df.to_csv(out_dir / "summary_per_image.csv", index=False)
    if not all_props:
        return
    combined = pd.concat(all_props, ignore_index=True)
    text = combined_csv_text(all_props, csv_texts)
    if text is not None:
        (out_dir / "all_droplets.csv").write_text(text)
    else:
        combined.to_csv(out_dir / "all_droplets.csv", index=False)
    if not skip_excel:
        try:
            import xlsxwriter  # noqa: F401
            with pd.ExcelWriter(out_dir / "all_droplets.xlsx", engine="xlsxwriter") as xw:
                combined.to_excel(xw, index=False, sheet_name="droplets")
                summary_df.to_excel(xw, index=False, sheet_name="per_image")
        except (ImportError, AttributeError):
            combined.to_csv(out_dir / "all_droplets_noexcel.csv", index=False)
            print("Skipped Excel file; install 'xlsxwriter' if you need .xlsx output.")
    size_col = "eq_diam_micron" if "eq_diam_micron" in combined.columns else "equivalent_diameter"
    if size_col in combined.columns:
        stats = combined[size_col].describe()[["mean", "50%", "std"]].rename({"50%": "median"})
        stats.to_csv(out_dir / "droplet_size_stats.csv")
        if not skip_histogram:
            try:
                import matplotlib
                matplotlib.use("Agg")
                import matplotlib.pyplot as plt
            except ImportError:
                print("Skipped histogram; matplotlib is not installed.")
                return
            plt.figure(figsize=(6, 4))
            plt.hist(combined[size_col], bins=40)
            plt.xlabel("Diameter (µm)" if "micron" in size_col else "Diameter (pixels)")
            plt.ylabel("Count")
            plt.title("Droplet size distribution")
            plt.tight_layout()
            plt.savefig(out_dir / "size_histogram.png", dpi=300)
            plt.close()


def _decode(path):
    """qdb:41: decode to RGB.  A frame whose three channels are identical (every grayscale file) is returned as one
    [H,W] plane: the rolling ball then corrects it once and the network folds the three identical input channels."""
    from PIL import Image
    im = np.array(Image.open(path).convert("RGB"))
    if np.array_equal(im[..., 0], im[..., 1]) and np.array_equal(im[..., 1], im[..., 2]):
        return np.ascontiguousarray(im[..., 0])
    return im


def _table_frame(cols: dict, px_per_um):
    """Per-image DataFrame with the reference's column contract (qdb:87-94): empty and column-less without droplets."""
    import pandas as pd
    from .quantify import COLUMNS, MICRON_COLUMNS
    if len(cols["label"]) == 0:
        return pd.DataFrame()
    return pd.DataFrame({k: cols[k] for k in COLUMNS + (MICRON_COLUMNS if px_per_um else [])})


def run_fast(images, mine, model, args, out_dir, mask_dir, overlay_dir):
    """The batched path behind ``main``: the per-image work of qdb:146-160 (preprocess + run_batch) for the frames
    ``mine`` (indices into ``images``), with every device stage batched and the host stages (decode, PNG / CSV
    writing) in thread pools around it.  Returns (indices, per_image_rows, all_props) in frame order."""
    import collections
    import os
    from concurrent.futures import ThreadPoolExecutor
    import cv2
    from .pipeline import DropletPipeline
    dev = next(model.parameters()).device
    pipe = DropletPipeline(model, args.background_radius, args.prob_thresh, args.min_area, args.px_per_micron,
                           img_size=args.img_size)
    nthreads = max(2, min(16, (os.cpu_count() or 4)))
    metas = collections.deque()                      # one entry per batch handed to the pipeline, in order
    idx, per_image_rows, all_props = [], [], []

    with ThreadPoolExecutor(nthreads) as decoders, ThreadPoolExecutor(nthreads) as writers:
        def batches():
            window = 4 * args.batch                  # decoded frames in flight (bounded host memory)
            pending = collections.deque()
            it = iter(mine)
            def refill():
                while len(pending) < window:
                    i = next(it, None)
                    if i is None:
                        return
                    pending.append((i, decoders.submit(_decode, images[i])))
            refill()
            cur, cur_meta = [], []
            while pending:
                i, fut = pending.popleft()
                refill()
                fr = fut.result()
                if cur and (fr.shape != cur[0].shape or len(cur) == args.batch):
                    metas.append(cur_meta)
                    yield np.stack(cur)
                    cur, cur_meta = [], []
                cur.append(fr)
                cur_meta.append(i)
            if cur:
                metas.append(cur_meta)
                yield np.stack(cur)

        def write_image(i, mask, stencil, df):
            name = images[i].stem
            cv2.imwrite(str(Path(mask_dir) / f"{name}_pred.png"), mask * 255)                 # qdb:58
            text = df.to_csv(index=False)                                                     # qdb:63
            (Path(mask_dir).parent / f"{name}_droplets.csv").write_text(text)
            if overlay_dir is not None:
                img = cv2.imread(str(images[i]))                                              # qdb:75
                if img is not None:
                    draw_overlay(img, stencil)                                                # qdb:76-77, from the GPU
                    cv2.imwrite(str(Path(overlay_dir) / f"{name}_overlay.png"), img)          # qdb:78
            return text

        jobs = []
        want_ov = overlay_dir is not None
        for res in pipe.run_host_pipelined(batches(), dev, copy=True, want_overlay=want_ov):
            masks, tables = res[0], res[1]
            stencils = res[2] if want_ov else None
            for b, i in enumerate(metas.popleft()):
                df = _table_frame(tables[b], args.px_per_micron)
                df.insert(0, "filename", images[i].name)                                      # qdb:62
                jobs.append(writers.submit(write_image, i, masks[b], stencils[b] if want_ov else None, df))
                idx.append(i)
                all_props.append(df)
                per_image_rows.append({"filename": images[i].name, "droplet_count": len(df),
                                       "total_area_px": df["area"].sum() if not df.empty else 0})   # qdb:67-72
                if args.density_maps:
                    save_density_maps(str(images[i]), images[i].stem, torch.from_numpy(masks[b]).to(dev)[None], out_dir)
        csv_texts = [j.result() for j in jobs]
    return idx, per_image_rows, all_props, csv_texts


def build_parser() -> argparse.ArgumentParser:
    p = argparse.ArgumentParser("Segment lipid droplets and build a report")
    p.add_argument("--img_dir", required=True)
    p.add_argument("--ckpt_path", default="best_UNetDC_focal_model.pth")
    p.add_argument("--out_dir", default="quant_results")
    p.add_argument("--batch", type=int, default=8)
    p.add_argument("--prob_thresh", type=float, default=0.3)
    p.add_argument("--min_area", type=int, default=1, help="ignore objects smaller than this (pixels²)")
    p.add_argument("--px_per_micron", type=float, help="pixels per micron for physical-unit columns")
    p.add_argument("--save_overlays", action="store_true")
    p.add_argument("--background_radius", type=int, default=50,
                   help="radius for rolling ball background correction (1..2047)")
    p.add_argument("--skip_excel", action="store_true", help="skip generation of the Excel workbook")
    p.add_argument("--skip_histogram", action="store_true", help="skip histogram plot generation")
    p.add_argument("--density_maps", action="store_true",
                   help="also write the radial / spatial droplet-density maps of the reference's quantify_pipline.py")
    p.add_argument("--reference_loop", action="store_true",
                   help="run the reference-shaped per-image loop (preprocess / run_batch) instead of the batched pipeline")
    p.add_argument("--img_size", type=int, default=IMG_SIZE,
                   help="network input size (reference constant IMG_SIZE = 512); use the frame size for native-resolution inference")
    return p


def main(argv=None) -> int:
    import os
    args = build_parser().parse_args(argv)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if torch.cuda.is_available():
        torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")))
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl")

    in_dir, out_dir = Path(args.img_dir), Path(args.out_dir)
    mask_dir = out_dir / "predicted_masks"
    overlay_dir = out_dir / "overlays" if args.save_overlays else None
    out_dir.mkdir(parents=True, exist_ok=True)
    mask_dir.mkdir(exist_ok=True)
    if overlay_dir:
        overlay_dir.mkdir(exist_ok=True)

    model = load_model(args.ckpt_path)
    images = sorted(p for p in in_dir.iterdir() if p.suffix.lower() in SUFFIXES)
    from . import shard
    mine = shard.shard_indices(len(images), rank, world)

    tensors, meta, idx = [], [], []
    per_image_rows, all_props = [], []
    csv_texts = None

    def flush():
        run_batch(tensors, meta, model, mask_dir, overlay_dir, args.prob_thresh, args.min_area, args.px_per_micron,
                  per_image_rows, all_props, density_dir=out_dir if args.density_maps else None)
        tensors.clear()
        meta.clear()

    if args.reference_loop:
        for i in mine:
            t, osize = preprocess(images[i], args.background_radius, args.img_size)
            tensors.append(t)
            meta.append((str(images[i]), osize))
            idx.append(i)
            if len(tensors) == args.batch:
                flush()
        if tensors:
            flush()
    else:
        idx, per_image_rows, all_props, csv_texts = run_fast(images, mine, model, args, out_dir, mask_dir, overlay_dir)

    texts = csv_texts if csv_texts is not None else [None] * len(idx)
    local = [(i, (row, df, t)) for i, row, df, t in zip(idx, per_image_rows, all_props, texts)]
    merged = shard.gather_results(local, len(images), dst=0)
    if rank == 0:
        write_reports(out_dir, [m[0] for m in merged], [m[1] for m in merged], args.skip_excel, args.skip_histogram,
                      csv_texts=[m[2] for m in merged])
        print("\n All done. Outputs are in ", out_dir)
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
