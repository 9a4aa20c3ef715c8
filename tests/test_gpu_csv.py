"""GPU: the per-image CSV files formatted on the device (dc_table_csv) are byte for byte what pandas writes for the same
droplet tables -- the DataFrame of the column contract, the filename inserted in front, to_csv (qdb:62-63) -- for
synthetic batches, inside the pipeline (CUDA graphs, capacity overflow), and through the CLI, whose report files must
equal what the pandas-based report code writes from the same tables."""
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
REPO = Path(__file__).resolve().parent.parent
NAMES = ["f0.png", "a,b.png", 'q"u.png', "é ü 漢.tif", "new\nline.png", "plain name.jpeg", "c,\"d\",e.png", "x.png"]


def pandas_text(cols: dict, name: str, micron: bool) -> bytes:
    """The per-image file as the pandas path writes it: DataFrame (empty and column-less without droplets), insert,
    to_csv, encoded as Path.write_text encodes."""
    import pandas as pd
    from unet_dc_segmentation_b200.quantify import COLUMNS, MICRON_COLUMNS, text_encoding
    df = pd.DataFrame() if len(cols["label"]) == 0 else \
        pd.DataFrame({k: cols[k] for k in COLUMNS + (MICRON_COLUMNS if micron else [])})
    df.insert(0, "filename", name)
    return df, df.to_csv(index=False).encode(text_encoding())


def check_tables(t, names, micron):
    from unet_dc_segmentation_b200.quantify import tables_to_csv
    got = tables_to_csv(t, names)
    want = t.to_host()
    for b, name in enumerate(names):
        assert got.texts[b] == pandas_text(want[b], name, micron)[1], (b, got.texts[b][:300])
        n = len(want[b]["label"])
        assert got.counts[b] == n and got.area_sums[b] == (want[b]["area"].sum() if n else 0)
        size = want[b]["eq_diam_micron" if micron else "equivalent_diameter"]
        np.testing.assert_array_equal(got.sizes[b].view(np.int64), size.view(np.int64))
    return got


@pytest.mark.parametrize("size,discs,min_area,px", [(256, 60, 1, None), (256, 60, 5, 3.45), (1024, 3000, 1, 3.45),
                                                     (2048, 10000, 1, None), (2048, 10000, 3, 0.37)])
def test_device_text_equals_pandas(cuda_device, size, discs, min_area, px):
    import torch
    from unet_dc_segmentation_b200.quantify import label_stats_device
    from unet_dc_segmentation_b200.synth import synthetic_mask
    masks = np.stack([synthetic_mask(size, discs, seed=s) for s in range(3)] + [np.zeros((size, size), np.uint8)])
    t = label_stats_device(torch.from_numpy(masks).to(cuda_device), min_area, px, capacity=16384)
    got = check_tables(t, NAMES[:4], bool(px))
    assert got.texts[3] == b"filename\n" and min(got.counts[:3]) > 0
    if size == 2048 and min_area == 1:
        assert got.counts.max() > 5000


def test_extreme_px_per_micron_writes_inf(cuda_device):
    import torch
    from unet_dc_segmentation_b200.quantify import label_stats_device
    from unet_dc_segmentation_b200.synth import synthetic_mask
    masks = torch.from_numpy(synthetic_mask(256, 40, seed=9)[None]).to(cuda_device)
    got = check_tables(label_stats_device(masks, 1, 1e-160), ["tiny.png"], True)
    assert b",inf," in got.texts[0]


def test_capacity_overflow_never_yields_truncated_text(cuda_device):
    import torch
    from unet_dc_segmentation_b200 import _lib
    from unet_dc_segmentation_b200.quantify import (csv_field, csv_text_device, label_stats_device, pack_fields,
                                                    tables_to_csv)
    from unet_dc_segmentation_b200.synth import synthetic_mask
    masks = torch.from_numpy(np.stack([synthetic_mask(256, 60, seed=1), synthetic_mask(256, 2, seed=2)])).to(cuda_device)
    t = label_stats_device(masks, 1, None, capacity=8)
    counts = t.counts.cpu().numpy()
    assert counts[0] > 8 >= counts[1]
    with pytest.raises(_lib.DcError):
        tables_to_csv(t, ["a.png", "b.png"])
    buf, offs = pack_fields([csv_field("a.png"), csv_field("b.png")])
    out, off, asum = csv_text_device(t, torch.from_numpy(buf.copy()).to(cuda_device), torch.from_numpy(offs).to(cuda_device),
                                     int(offs[-1]))
    off, asum = off.cpu().numpy(), asum.cpu().numpy()
    assert off[1] == off[0] and asum[0] == -1                      # no text at all for the frame that did not fit
    text = out[off[1]:off[2]].cpu().numpy().tobytes()
    assert text == pandas_text(t.rows(1, 2).to_host()[0], "b.png", False)[1]


def _model(dev):
    from unet_dc_segmentation_b200 import UNetDC
    from unet_dc_segmentation_b200.synth import calibrated_state_dict
    m = UNetDC(3, 1)
    m.load_state_dict(calibrated_state_dict(seed=0, calib_size=64, n_calib=2))
    return m.to(dev).eval()


@pytest.mark.parametrize("capacity", [16384, 6])
def test_pipeline_csv_mode_with_graphs(cuda_device, capacity):
    """csv=True with use_graphs=True (captured on a slot's second use, replayed after): every frame's text, count, area
    sum and size column equal the column mode's tables through pandas -- also when batches overflow the capacity."""
    from unet_dc_segmentation_b200 import DropletPipeline
    from unet_dc_segmentation_b200.synth import synthetic_image
    model = _model(cuda_device)
    batches = [np.stack([synthetic_image(96, 10 * k + j, n_droplets=12) for j in range(4)]) for k in range(7)]
    batches[3][1] = 0                                              # a blank frame
    names = [[NAMES[(k + j) % len(NAMES)] for j in range(4)] for k in range(7)]
    ref = DropletPipeline(model, 50, 0.3, 2, 3.45, img_size=None)
    want = list(ref.run_host_pipelined(iter(batches), cuda_device))
    pipe = DropletPipeline(model, 50, 0.3, 2, 3.45, img_size=None, capacity=capacity, use_graphs=True)
    got = list(pipe.run_host_pipelined(zip(batches, names), cuda_device, csv=True, want_overlay=True))
    assert len(got) == len(want)
    for k, ((m_want, tabs), (m_got, csvt, _)) in enumerate(zip(want, got)):
        np.testing.assert_array_equal(m_got, m_want)
        for b in range(4):
            assert csvt.texts[b] == pandas_text(tabs[b], names[k][b], True)[1], (k, b)
            assert csvt.counts[b] == len(tabs[b]["label"])
            assert csvt.area_sums[b] == (tabs[b]["area"].sum() if len(tabs[b]["label"]) else 0)
            np.testing.assert_array_equal(csvt.sizes[b], tabs[b]["eq_diam_micron"])
    if capacity < 16384:
        assert pipe.capacity > capacity


# ------------------------------------------------------------------ the CLI against the pandas report code
def pandas_reports(out: Path, mask_dir: Path, frames_in: list, min_area, px, skip_excel: bool):
    """The pandas-based files of the CLI (per-image CSVs, summary, all_droplets.csv, the noexcel copy, size stats) from
    the tables of the mask PNGs the CLI wrote: per-image DataFrames written by to_csv, pd.concat of them."""
    import cv2
    import pandas as pd
    import torch
    from unet_dc_segmentation_b200 import cli
    from unet_dc_segmentation_b200.quantify import label_stats_device
    out.mkdir()
    frames, rows, texts = [], [], []
    for p in frames_in:
        mask = cv2.imread(str(mask_dir / f"{p.stem}_pred.png"), cv2.IMREAD_GRAYSCALE) // 255
        cols = label_stats_device(torch.from_numpy(mask[None]).cuda(), min_area, px).to_host()[0]
        df, _ = pandas_text(cols, p.name, bool(px))
        text = df.to_csv(index=False)
        (out / f"{p.stem}_droplets.csv").write_text(text)
        frames.append(df)
        texts.append(text)
        rows.append({"filename": p.name, "droplet_count": len(df), "total_area_px": df["area"].sum() if not df.empty else 0})
    pd.DataFrame(rows).to_csv(out / "summary_per_image.csv", index=False)
    combined = pd.concat(frames, ignore_index=True)
    text = cli.combined_csv_text(frames, texts)
    if text is not None:
        (out / "all_droplets.csv").write_text(text)
    else:
        combined.to_csv(out / "all_droplets.csv", index=False)
    if not skip_excel:
        combined.to_csv(out / "all_droplets_noexcel.csv", index=False)
    size_col = "eq_diam_micron" if "eq_diam_micron" in combined.columns else "equivalent_diameter"
    if size_col in combined.columns:
        combined[size_col].describe()[["mean", "50%", "std"]].rename({"50%": "median"}).to_csv(out / "droplet_size_stats.csv")
    return rows


def assert_same_files(got: Path, want: Path):
    names = sorted(p.name for p in want.iterdir())
    assert sorted(p.name for p in got.iterdir() if p.is_file() and not p.name.endswith(".png")) == names
    for n in names:
        assert (got / n).read_bytes() == (want / n).read_bytes(), n


@pytest.fixture(scope="module")
def cli_inputs(tmp_path_factory):
    import torch
    from PIL import Image
    from unet_dc_segmentation_b200.synth import calibrated_state_dict, synthetic_image
    d = tmp_path_factory.mktemp("cli_csv")
    (d / "in").mkdir()
    for i in range(5):
        Image.fromarray(synthetic_image(96, 600 + i, n_droplets=12)).save(d / "in" / f"f{i}.png")
    Image.fromarray(np.zeros((96, 96), np.uint8)).save(d / "in" / "f5 black, empty.png")
    Image.fromarray(synthetic_image(96, 700, n_droplets=12)).save(d / "in" / "ü \"q\".png")
    torch.save(calibrated_state_dict(seed=0, calib_size=64, n_calib=2), d / "ckpt.pth")
    return d


@pytest.mark.parametrize("skip_excel,px", [(False, "3.45"), (True, None)])
def test_cli_files_equal_pandas_reports(cuda_device, cli_inputs, skip_excel, px):
    from unet_dc_segmentation_b200 import cli
    d = cli_inputs
    out = d / f"out_{skip_excel}_{px}"
    argv = ["--img_dir", str(d / "in"), "--ckpt_path", str(d / "ckpt.pth"), "--out_dir", str(out), "--batch", "3",
            "--img_size", "96", "--skip_histogram"] + (["--skip_excel"] if skip_excel else []) + \
           (["--px_per_micron", px] if px else [])
    assert cli.main(argv) == 0
    frames = sorted(p for p in (d / "in").iterdir() if p.suffix == ".png")
    rows = pandas_reports(d / f"want_{skip_excel}_{px}", out / "predicted_masks", frames, 1, float(px) if px else None,
                          skip_excel)
    assert any(r["droplet_count"] == 0 for r in rows) and any(r["droplet_count"] > 0 for r in rows)
    assert_same_files(out, d / f"want_{skip_excel}_{px}")


def test_cli_two_ranks_files_equal_pandas_reports(cuda_device, cli_inputs):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    d = cli_inputs
    out = d / "out_two"
    env = dict(os.environ, PYTHONPATH=str(REPO), MASTER_ADDR="127.0.0.1")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", "29541", "-m", "unet_dc_segmentation_b200.cli",
                        "--img_dir", str(d / "in"), "--ckpt_path", str(d / "ckpt.pth"), "--out_dir", str(out),
                        "--batch", "2", "--img_size", "96", "--skip_histogram", "--px_per_micron", "3.45"],
                       env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    frames = sorted(p for p in (d / "in").iterdir() if p.suffix == ".png")
    pandas_reports(d / "want_two", out / "predicted_masks", frames, 1, 3.45, False)
    assert_same_files(out, d / "want_two")
