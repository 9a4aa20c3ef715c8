"""Drop-in front end for reference quantify_droplets_batch.py: same functions, same flags, same output files,
with the device work done by libunetdc_b200 (rolling ball, UNetDC, threshold, labelling, droplet table).

    python -m unet_dc_segmentation_b200.cli --img_dir IN --ckpt_path model.pth --out_dir OUT [flags as the reference]

Function-for-function (reference file:line):
    load_model   qdb:34-37     preprocess  qdb:40-46     run_batch  qdb:48-79     quantify  qdb:81-95
    main         qdb:100-201   (argparse flags qdb:101-128; report files qdb:163-199, read back by gui_qt.py:470-589)

On the device: rolling ball, both resizes (cv2.resize at qdb:44 and qdb:57 is bilinear -- the reference passes the
interpolation flag in the `dst` slot, SURVEY.md 0.2 -- reproduced bit for bit by dc_resize_linear_u8; the identity
when the frame is already IMG_SIZE), the network, the threshold, labelling, the table and the overlay contours (qdb:76-77,
bit-exact against OpenCV's findContours + drawContours), and in ``main`` the mask and overlay PNG files (dc_png_encode,
byte for byte what cv2.imwrite writes, whenever the installed OpenCV is found to write those bytes).  On the host, exactly
as in the reference: PIL / cv2 decode, the XLSX and the reports.  Added flags: `--img_size` (default 512 = the reference's
IMG_SIZE constant) and `--density_maps` (the per-image maps of the reference's second front end, quantify_pipline.py:131-141).  Under torchrun (one rank per GPU) frames are sharded i -> rank i mod N, every
rank writes the per-image files of its own frames, and the tables are gathered on rank 0, which writes the reports.

``main`` runs the FAST path (``run_fast``): frames are decoded by a thread pool, batched, and streamed through
``DropletPipeline.run_host_pipelined`` -- u8 frames (+ the overlay bases cv2.imread returned) up; u8 masks, overlay
stencils, the per-image CSV files as text (dc_table_csv) and the mask and overlay PNG files (dc_png_encode) down --
while another pool writes the files as bytes.  ``write_reports`` builds the reports of both loops from the per-image CSV texts.  ``preprocess`` / ``run_batch`` keep the
reference's function-by-function shape (per-image round trips) for callers that use them as a library;
``--reference_loop`` makes ``main`` use them.
"""
from __future__ import annotations

import argparse
import codecs
import functools
import io
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


@functools.lru_cache(maxsize=None)
def concat_upcasts_with_empty_frames() -> bool:
    """Whether the installed pandas turns the int64 label / area columns into float64 when pd.concat meets a per-image
    frame without droplets (pandas 3: the empty frame's missing columns count as all-NaN float64 columns; pandas 2
    left empty frames out when it chose the dtype).  Decided by one tiny concat, the way the reports are built."""
    import pandas as pd
    empty = pd.DataFrame()
    empty.insert(0, "filename", "e")
    full = pd.DataFrame({"label": np.array([1], np.int64), "area": np.array([12], np.int64), "x": [0.5]})
    full.insert(0, "filename", "f")
    text = pd.concat([empty, full], ignore_index=True).to_csv(index=False)
    if text in ("filename,label,area,x\nf,1,12,0.5\n", "filename,label,area,x\nf,1.0,12.0,0.5\n"):
        return ".0" in text
    raise RuntimeError(f"pandas {pd.__version__} concatenates the droplet tables in an unknown way: {text!r}")


def combined_csv_bytes(texts, fields) -> bytes:
    """all_droplets.csv -- ``pd.concat(per-image frames, ignore_index=True).to_csv(index=False)`` (qdb:165-166) -- from
    the per-image CSV files (bytes) without formatting a number again.  fields: each image's filename field as it
    appears in its file.  When some images have droplets and others not, pandas may write label and area as float64
    (``concat_upcasts_with_empty_frames``): then ".0" is inserted after both fields of every row, at positions that
    follow from the filename field's length."""
    full = [(t, f) for t, f in zip(texts, fields) if not t.startswith(b"filename\n")]
    if not full:
        return b"filename\n"
    header = full[0][0][:full[0][0].index(b"\n") + 1]
    if len(full) == len(texts) or not concat_upcasts_with_empty_frames():
        return header + b"".join(t[len(header):] for t, _ in full)
    dot0 = np.frombuffer(b".0", np.uint8)
    parts = [header]
    for t, f in full:
        buf = np.frombuffer(t, dtype=np.uint8)[len(header):]
        m = f.count(b"\n")                                     # a quoted field may hold line breaks: every row has m + 1
        ends = np.flatnonzero(buf == ord("\n"))[m::m + 1]
        starts = np.concatenate(([0], ends[:-1] + 1))
        commas = np.flatnonzero(buf == ord(","))
        k = np.searchsorted(commas, starts + len(f) + 1)         # the comma after the label of every row
        at = np.stack([commas[k], commas[k + 1]], 1).ravel()       # ... and the one after its area
        parts.append(np.insert(buf, np.repeat(at, 2), np.tile(dot0, at.size)).tobytes())
    return b"".join(parts)


def write_reports(out_dir: Path, per_image_rows, texts, sizes, skip_excel: bool, skip_histogram: bool,
                  encoding: str) -> None:
    """qdb:163-199: summary_per_image.csv, all_droplets.csv (+xlsx or the noexcel copy), stats, histogram, from every
    image's summary row, CSV file text (bytes in ``encoding``) and size column (f64), in frame order.  The files pandas
    writes itself are UTF-8; all_droplets.csv, when every image has droplets, is the per-image texts joined as they are
    (what the reference's concat gives then, written with write_text)."""
    import pandas as pd
    from .quantify import csv_field
    summary_df = pd.DataFrame(per_image_rows)
    summary_df.to_csv(out_dir / "summary_per_image.csv", index=False)
    if not texts:
        return
    fields = [csv_field(r["filename"], encoding) for r in per_image_rows]
    combined = combined_csv_bytes(texts, fields)
    as_pandas = combined if codecs.lookup(encoding).name == "utf-8" else combined.decode(encoding).encode("utf-8")
    every_frame = all(not t.startswith(b"filename\n") for t in texts)
    (out_dir / "all_droplets.csv").write_bytes(combined if every_frame else as_pandas)
    if not skip_excel:
        try:
            import xlsxwriter  # noqa: F401
            frame = pd.read_csv(io.BytesIO(as_pandas), dtype={"filename": str}, keep_default_na=False,
                                float_precision="round_trip")
            with pd.ExcelWriter(out_dir / "all_droplets.xlsx", engine="xlsxwriter") as xw:
                frame.to_excel(xw, index=False, sheet_name="droplets")
                summary_df.to_excel(xw, index=False, sheet_name="per_image")
        except (ImportError, AttributeError):
            (out_dir / "all_droplets_noexcel.csv").write_bytes(as_pandas)
            print("Skipped Excel file; install 'xlsxwriter' if you need .xlsx output.")
    if combined != b"filename\n":
        size_col = "eq_diam_micron" if b",eq_diam_micron\n" in combined[:combined.index(b"\n") + 1] else "equivalent_diameter"
        column = pd.Series(np.concatenate(sizes), name=size_col)
        stats = column.describe()[["mean", "50%", "std"]].rename({"50%": "median"})
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
            plt.hist(column, bins=40)
            plt.xlabel("Diameter (µm)" if "micron" in size_col else "Diameter (pixels)")
            plt.ylabel("Count")
            plt.title("Droplet size distribution")
            plt.tight_layout()
            plt.savefig(out_dir / "size_histogram.png", dpi=300)
            plt.close()


def _decode_with_base(path):
    """_decode, plus the overlay base of qdb:75 (cv2.imread; None when OpenCV cannot read the file)."""
    import cv2
    return _decode(path), cv2.imread(str(path))


def _decode(path):
    """qdb:41: decode to RGB.  A frame whose three channels are identical (every grayscale file) is returned as one
    [H,W] plane: the rolling ball then corrects it once and the network folds the three identical input channels."""
    from PIL import Image
    im = np.array(Image.open(path).convert("RGB"))
    if np.array_equal(im[..., 0], im[..., 1]) and np.array_equal(im[..., 1], im[..., 2]):
        return np.ascontiguousarray(im[..., 0])
    return im


def run_fast(images, mine, model, args, out_dir, mask_dir, overlay_dir):
    """The batched path behind ``main``: the per-image work of qdb:146-160 (preprocess + run_batch) for the frames
    ``mine`` (indices into ``images``), with every device stage batched and the host stages (decode, PNG / CSV
    writing) in thread pools around it.  The per-image CSV files are formatted on the device (dc_table_csv): no
    DataFrame and no per-row Python object.  Returns (indices, per_image_rows, texts, sizes) in frame order: the
    summary row, the CSV file's bytes and the size column of every frame."""
    import collections
    import os
    from concurrent.futures import ThreadPoolExecutor
    import cv2
    from .pipeline import DropletPipeline
    dev = next(model.parameters()).device
    pipe = DropletPipeline(model, args.background_radius, args.prob_thresh, args.min_area, args.px_per_micron,
                           img_size=args.img_size)
    nthreads = max(2, min(16, (os.cpu_count() or 4)))
    from .png import device_matches_opencv
    png = device_matches_opencv(dev.index)           # else an OpenCV on another zlib: keep writing through cv2
    want_ov = overlay_dir is not None
    bases_in = png and want_ov
    metas = collections.deque()                      # one entry per batch handed to the pipeline, in order
    idx, per_image_rows, texts, sizes = [], [], [], []

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
                    pending.append((i, decoders.submit(_decode_with_base if bases_in else _decode, images[i])))
            refill()
            cur, cur_meta, cur_base = [], [], []

            def item():
                metas.append(cur_meta)
                names = [images[j].name for j in cur_meta]
                if not bases_in:
                    return np.stack(cur), names
                # a base of another shape than the frame (an EXIF-rotated JPEG) keeps the host path: no device overlay
                ok = [b is not None and b.shape == cur[0].shape[:2] + (3,) for b in cur_base]
                bases = np.stack([b if o else np.zeros(cur[0].shape[:2] + (3,), np.uint8) for b, o in zip(cur_base, ok)])
                return np.stack(cur), names, bases, np.array(ok)
            while pending:
                i, fut = pending.popleft()
                refill()
                fr, base = fut.result() if bases_in else (fut.result(), None)
                if cur and (fr.shape != cur[0].shape or len(cur) == args.batch):
                    yield item()
                    cur, cur_meta, cur_base = [], [], []
                cur.append(fr)
                cur_meta.append(i)
                cur_base.append(base)
            if cur:
                yield item()

        def write_image(i, mask, stencil, text, mask_png, overlay_png):
            name = images[i].stem
            if mask_png is not None:                                                          # qdb:58, encoded on the GPU
                (Path(mask_dir) / f"{name}_pred.png").write_bytes(mask_png)
            else:
                cv2.imwrite(str(Path(mask_dir) / f"{name}_pred.png"), mask * 255)             # qdb:58
            (Path(mask_dir).parent / f"{name}_droplets.csv").write_bytes(text)                # qdb:62-63
            if overlay_png is not None:                                                       # qdb:75-78 on the GPU
                (Path(overlay_dir) / f"{name}_overlay.png").write_bytes(overlay_png)
            elif overlay_dir is not None:
                img = cv2.imread(str(images[i]))                                              # qdb:75
                if img is not None:
                    draw_overlay(img, stencil)                                                # qdb:76-77, from the GPU
                    cv2.imwrite(str(Path(overlay_dir) / f"{name}_overlay.png"), img)          # qdb:78

        jobs = []
        for res in pipe.run_host_pipelined(batches(), dev, copy=True, want_overlay=want_ov, csv=True, png=png):
            masks, tables = res[0], res[1]
            stencils = res[2] if want_ov else None
            files = res[-1] if png else None
            for b, i in enumerate(metas.popleft()):
                jobs.append(writers.submit(write_image, i, masks[b], stencils[b] if want_ov else None, tables.texts[b],
                                           files.masks[b] if png else None,
                                           files.overlays[b] if bases_in else None))
                idx.append(i)
                texts.append(tables.texts[b])
                sizes.append(tables.sizes[b])
                n = int(tables.counts[b])
                per_image_rows.append({"filename": images[i].name, "droplet_count": n,
                                       "total_area_px": int(tables.area_sums[b]) if n else 0})    # qdb:67-72
                if args.density_maps:
                    save_density_maps(str(images[i]), images[i].stem, torch.from_numpy(masks[b]).to(dev)[None], out_dir)
        for j in jobs:
            j.result()
    return idx, per_image_rows, texts, sizes


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
    p.add_argument("--precision", choices=("bf16", "fp32"), default="bf16",
                   help="fp32: activations and weights to fp32 accuracy (about six times the tensor-core work), for "
                        "masks and counts that match the reference's fp32 network")
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
    model.precision = args.precision
    images = sorted(p for p in in_dir.iterdir() if p.suffix.lower() in SUFFIXES)
    from . import shard
    mine = shard.shard_indices(len(images), rank, world)

    tensors, meta, idx = [], [], []
    per_image_rows, all_props = [], []

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
        # run_batch wrote its CSVs through pandas (UTF-8); the reports take the same text from its DataFrames
        encoding = "utf-8"
        size_col = "eq_diam_micron" if args.px_per_micron else "equivalent_diameter"
        texts = [df.to_csv(index=False).encode(encoding) for df in all_props]
        sizes = [df[size_col].to_numpy(np.float64) if size_col in df else np.zeros(0) for df in all_props]
    else:
        from .quantify import text_encoding
        encoding = text_encoding()
        idx, per_image_rows, texts, sizes = run_fast(images, mine, model, args, out_dir, mask_dir, overlay_dir)

    local = [(i, (row, t, s)) for i, row, t, s in zip(idx, per_image_rows, texts, sizes)]
    merged = shard.gather_results(local, len(images), dst=0)       # the CSV texts travel, not DataFrames
    if rank == 0:
        write_reports(out_dir, [m[0] for m in merged], [m[1] for m in merged], [m[2] for m in merged],
                      args.skip_excel, args.skip_histogram, encoding)
        print("\n All done. Outputs are in ", out_dir)
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
