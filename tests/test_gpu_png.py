"""GPU: dc_png_encode writes, for every frame of a batch, the bytes cv2.imencode(".png", img) writes -- on the corpus of
tests/png_cases.py in mixed batches, on the crafted streams, under CUDA-graph replay, and on one BGR frame whose
deflate stream passes 2^32 bits."""
import numpy as np
import pytest

import png_cases as pc

pytestmark = pytest.mark.gpu


def encode_batch(frames, dev):
    import torch
    from unet_dc_segmentation_b200.png import encode_png_device
    buf, off = encode_png_device(torch.from_numpy(np.stack(frames)).to(dev))
    off = off.cpu().numpy()
    data = buf[:int(off[-1])].cpu().numpy().tobytes()
    return [data[off[b]:off[b + 1]] for b in range(len(frames))]


def assert_cv2(frames, got, what):
    import cv2
    for i, (img, g) in enumerate(zip(frames, got)):
        want = cv2.imencode(".png", img)[1].tobytes()
        assert g == want, f"{what} frame {i} {img.shape}: {len(g)} bytes, cv2 {len(want)}"


@pytest.mark.parametrize("shape", pc.SHAPES, ids=[f"{h}x{w}" for h, w in pc.SHAPES])
def test_mixed_batches_equal_opencv(cuda_device, shape):
    corpus = pc.corpus_for_shape(*shape)
    grey = [v for v in corpus.values() if v.ndim == 2]
    bgr = [v for v in corpus.values() if v.ndim == 3]
    for frames in (grey, bgr, grey[::-1] * 2):
        assert_cv2(frames, encode_batch(frames, cuda_device), f"{shape}")


def test_crafted_streams(cuda_device):
    for name, img in pc.crafted().items():
        assert_cv2([img, img[:, ::-1].copy()], encode_batch([img, img[:, ::-1].copy()], cuda_device), name)


def test_cuda_graph_replay(cuda_device):
    import torch
    from unet_dc_segmentation_b200.png import encode_png_device, png_bounds
    frames = list(pc.corpus_for_shape(300, 500, seed=1).values())
    bgr = [f for f in frames if f.ndim == 3]
    x = torch.from_numpy(np.stack(bgr)).to(cuda_device)
    need, wsb = png_bounds(len(bgr), 300, 500, 3)
    out = torch.empty(need, dtype=torch.uint8, device=cuda_device)
    ws = torch.empty(wsb, dtype=torch.uint8, device=cuda_device)
    s = torch.cuda.Stream(cuda_device)
    with torch.cuda.stream(s):
        encode_png_device(x, out, ws)                      # eager pass first
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=s):
            _, off = encode_png_device(x, out, ws)
    for seed in (2, 3):
        new = [f for f in pc.corpus_for_shape(300, 500, seed=seed).values() if f.ndim == 3]
        x.copy_(torch.from_numpy(np.stack(new)))
        g.replay()
        torch.cuda.synchronize()
        o = off.cpu().numpy()
        data = out[:int(o[-1])].cpu().numpy().tobytes()
        assert_cv2(new, [data[o[b]:o[b + 1]] for b in range(len(new))], f"graph replay {seed}")


def test_device_matches_opencv_probe(cuda_device):
    from unet_dc_segmentation_b200.png import device_matches_opencv, encode_png, encode_png_host, probe_images
    assert device_matches_opencv(0)
    for img in probe_images():
        assert encode_png(img, cuda_device) == encode_png_host(img)


def test_stream_past_2_to_the_32_bits(cuda_device):
    import cv2
    import torch
    from unet_dc_segmentation_b200.png import encode_png_device
    rs = np.random.default_rng(11)
    img = rs.normal(128, 40, (16384, 16384, 3)).clip(0, 255).astype(np.uint8)
    img[:4096, :4096] = 0                                   # a long run of 258-matches too
    buf, off = encode_png_device(torch.from_numpy(img[None]).to(cuda_device))
    n = int(off[1].item())
    got = buf[:n].cpu().numpy().tobytes()
    want = cv2.imencode(".png", img)[1].tobytes()
    assert len(want) * 8 > 2 ** 32
    assert got == want


@pytest.fixture(scope="module")
def model_and_frames():
    import torch
    from unet_dc_segmentation_b200 import UNetDC
    from unet_dc_segmentation_b200.synth import calibrated_state_dict, synthetic_image
    dev = torch.device("cuda", 0)
    m = UNetDC(3, 1)
    m.load_state_dict(calibrated_state_dict(seed=0, calib_size=64, n_calib=2))
    frames = np.stack([synthetic_image(128, 500 + i, n_droplets=12) for i in range(6)])
    frames[5] = 0                                            # an empty mask
    return m.to(dev).eval(), frames


@pytest.mark.parametrize("graphs", [False, True])
@pytest.mark.parametrize("overlay", [False, True])
def test_pipeline_png_equals_cv2_path(cuda_device, model_and_frames, graphs, overlay):
    import cv2
    from unet_dc_segmentation_b200.overlay import draw_overlay
    from unet_dc_segmentation_b200.pipeline import DropletPipeline
    model, frames = model_and_frames
    rs = np.random.default_rng(4)
    bases = rs.integers(0, 256, frames.shape + (3,), dtype=np.uint8)
    present = np.array([True, False, True, True, True, True])
    pipe = DropletPipeline(model, 50, 0.3, 1, None, use_graphs=graphs)
    items = [(frames[i:i + 2], bases[i:i + 2], present[i:i + 2]) if overlay else frames[i:i + 2] for i in (0, 2, 4, 0, 2)]
    n = 0
    for res in pipe.run_host_pipelined(items, cuda_device, want_overlay=overlay, png=True):
        masks, files = res[0], res[-1]
        for b in range(masks.shape[0]):
            i = (2 * n) % 6 + b
            assert files.masks[b] == cv2.imencode(".png", masks[b] * 255)[1].tobytes(), (n, b)
            if overlay:
                if present[i]:
                    want = cv2.imencode(".png", draw_overlay(bases[i].copy(), res[2][b]))[1].tobytes()
                    assert files.overlays[b] == want, (n, b)
                else:
                    assert files.overlays[b] is None
        n += 1
    assert n == 5


@pytest.mark.parametrize("overlays", [False, True])
def test_cli_output_identical_to_cv2_path(cuda_device, tmp_path, monkeypatch, overlays):
    import torch
    from PIL import Image
    from unet_dc_segmentation_b200 import cli, png
    from unet_dc_segmentation_b200.synth import calibrated_state_dict, synthetic_image
    d = tmp_path / "in"
    d.mkdir()
    for i in range(3):
        Image.fromarray(synthetic_image(96, 600 + i, n_droplets=10)).save(d / f"grey{i}.png")
    rgb = np.repeat(synthetic_image(96, 610, n_droplets=10)[..., None], 3, 2)
    rgb[..., 0] //= 2
    Image.fromarray(rgb).save(d / "colour.png")
    Image.fromarray(synthetic_image(96, 611, n_droplets=10)).save(d / "photo.jpg", quality=90)
    Image.fromarray(synthetic_image(128, 612, n_droplets=14)[:80, :112]).save(d / "wide.tif")
    Image.fromarray(np.zeros((96, 96), np.uint8)).save(d / "empty.png")
    torch.save(calibrated_state_dict(seed=0, calib_size=64, n_calib=2), tmp_path / "ckpt.pth")
    assert png.device_matches_opencv(0)

    def run(out):
        argv = ["--img_dir", str(d), "--ckpt_path", str(tmp_path / "ckpt.pth"), "--out_dir", str(out), "--batch", "2",
                "--skip_histogram", "--skip_excel", "--img_size", "96"]
        assert cli.main(argv + (["--save_overlays"] if overlays else [])) == 0
    run(tmp_path / "gpu")
    monkeypatch.setattr(png, "device_matches_opencv", lambda *a: False)
    run(tmp_path / "cv2")
    a = sorted(p.relative_to(tmp_path / "gpu") for p in (tmp_path / "gpu").rglob("*") if p.is_file())
    b = sorted(p.relative_to(tmp_path / "cv2") for p in (tmp_path / "cv2").rglob("*") if p.is_file())
    assert a == b and len(a) >= 7 * (3 if overlays else 2)
    for rel in a:
        assert (tmp_path / "gpu" / rel).read_bytes() == (tmp_path / "cv2" / rel).read_bytes(), rel
