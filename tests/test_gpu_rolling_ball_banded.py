"""GPU: the rolling ball's banded pass (csrc/morph.cu morph_band_kernel): radii past the tiled kernel up to 2047,
bit-exact against the tiled kernel, the reference's golden outputs and OpenCV's own four calls
(utils/data_loader.py:17-21); workspace, in-place, pipeline, CUDA-graph and CLI behaviour at large radii."""
import ctypes as C

import numpy as np
import pytest

from conftest import golden_cases, load_golden

pytestmark = pytest.mark.gpu


def cv2_rolling_ball(plane: np.ndarray, radius: int) -> np.ndarray:
    import cv2
    k = cv2.getStructuringElement(cv2.MORPH_ELLIPSE, (radius, radius))
    return cv2.normalize(cv2.subtract(plane, cv2.morphologyEx(plane, cv2.MORPH_OPEN, k)), None, 0, 255, cv2.NORM_MINMAX)


def _frames(shape, seed):
    from unet_dc_segmentation_b200.synth import synthetic_image
    rs = np.random.RandomState(seed)
    imgs = rs.randint(0, 256, shape).astype(np.uint8)
    if len(shape) == 3 and max(shape[1:]) <= 4096:
        H, W = shape[1:]
        imgs[0] = synthetic_image(max(H, W), seed)[:H, :W]
    imgs[(slice(None), slice(shape[1] // 3, shape[1] // 2 + 1), slice(shape[2] // 4, shape[2] // 2 + 1))] //= 4
    return imgs


def test_banded_equals_tiled_every_tiled_radius(cuda_device):
    import torch
    from unet_dc_segmentation_b200.morphology import rolling_ball_device, tiled_max_radius
    planar = torch.from_numpy(_frames((2, 193, 257), 1)).cuda()
    hwc = torch.from_numpy(_frames((1, 67, 45, 3), 2)).cuda()
    for r in range(1, tiled_max_radius() + 1):
        for x in (planar, hwc):
            a = rolling_ball_device(x, r, method="tiled")
            b = rolling_ball_device(x, r, method="banded")
            assert torch.equal(a, b), f"radius {r} shape {tuple(x.shape)}"


@pytest.mark.parametrize("case", golden_cases(load_golden("rolling_ball.npz")))
def test_golden_banded(cuda_device, case):
    import torch
    from unet_dc_segmentation_b200.morphology import rolling_ball_device
    rb = load_golden("rolling_ball.npz")
    img, radius, want = rb[f"{case}/in"], int(rb[f"{case}/radius"]), rb[f"{case}/out"]
    x = torch.from_numpy(np.ascontiguousarray(img if img.ndim == 3 else img[:, :, None]))[None].cuda()
    got = rolling_ball_device(x, radius, method="banded")[0].cpu().numpy()
    np.testing.assert_array_equal(got.reshape(want.shape), want)


def _auto_cases():
    cases = [((2, 301, 419), r) for r in (175, 176, 200, 256, 300, 511, 1023, 2047)]
    cases += [((1, 1024, 1024), 300), ((1, 1, 517), 300), ((1, 517, 1), 300), ((1, 40, 2000), 256),
              ((1, 40, 2000), 2047), ((2, 120, 97, 3), 250), ((1, 64, 80, 3), 777)]
    rs = np.random.RandomState(2047)
    for _ in range(20):
        shape = (int(rs.randint(1, 3)), int(rs.randint(1, 260)), int(rs.randint(1, 260)))
        cases.append((shape, int(rs.randint(175, 601))))
    return cases


@pytest.mark.parametrize("shape,radius", _auto_cases())
def test_auto_vs_cv2(cuda_device, shape, radius):
    import torch
    from unet_dc_segmentation_b200.morphology import rolling_ball_device
    imgs = _frames(shape, radius + shape[1])
    got = rolling_ball_device(torch.from_numpy(imgs).cuda(), radius).cpu().numpy()
    for b in range(shape[0]):
        if len(shape) == 4:
            for c in range(shape[3]):             # channels independent
                want = cv2_rolling_ball(np.ascontiguousarray(imgs[b, :, :, c]), radius)
                np.testing.assert_array_equal(got[b, :, :, c], want, err_msg=f"image {b} channel {c}")
        else:
            np.testing.assert_array_equal(got[b], cv2_rolling_ball(imgs[b], radius), err_msg=f"image {b}")


def test_constant_frame_is_zero(cuda_device):
    import torch
    from unet_dc_segmentation_b200.morphology import rolling_ball_device
    x = torch.full((2, 150, 211), 77, dtype=torch.uint8, device="cuda")
    for method in ("auto", "banded"):
        assert int(rolling_ball_device(x, 400, method=method).max()) == 0


def _call(entry, x, out, radius, ws, nbytes):
    from unet_dc_segmentation_b200 import _lib
    B, H, W = x.shape[:3]
    Cc = 1 if x.dim() == 3 else x.shape[3]
    args = _lib.RollingBallArgs(x.data_ptr(), out.data_ptr(), B, H, W, Cc, radius, ws.data_ptr(), nbytes)
    return getattr(_lib.load(), entry)(C.byref(args), _lib.stream_ptr())


@pytest.mark.parametrize("entry", ["dc_rolling_ball", "dc_rolling_ball_banded"])
def test_workspace_and_in_place(cuda_device, entry):
    import torch
    from unet_dc_segmentation_b200 import _lib
    from unet_dc_segmentation_b200.morphology import rolling_ball_workspace_bytes
    x = torch.from_numpy(_frames((2, 133, 171), 5)).cuda()
    need = rolling_ball_workspace_bytes(2, 133, 171)
    ws = torch.empty(need, dtype=torch.uint8, device="cuda")
    out = torch.empty_like(x)
    assert _call(entry, x, out, 300, ws, need) == _lib.DC_OK
    want = out.clone()
    assert _call(entry, x, out, 300, ws, need - 1) == _lib.DC_EWORKSPACE
    y = x.clone()
    assert _call(entry, y, y, 300, ws, need) == _lib.DC_OK                 # out == in
    torch.cuda.synchronize()
    assert torch.equal(y, want)
    for bad in (0, 2048):
        assert _call(entry, x, out, bad, ws, need) == _lib.DC_EINVAL


def test_row_wider_than_limit_is_refused(cuda_device):
    import torch
    from unet_dc_segmentation_b200 import _lib
    from unet_dc_segmentation_b200.morphology import rolling_ball_device, rolling_ball_workspace_bytes
    W = 32768 + 4
    x = torch.zeros((1, 2, W), dtype=torch.uint8, device="cuda")
    ws = torch.empty(rolling_ball_workspace_bytes(1, 2, W), dtype=torch.uint8, device="cuda")
    out = torch.empty_like(x)
    assert _call("dc_rolling_ball", x, out, 300, ws, ws.numel()) == _lib.DC_EINVAL
    assert "wider" in _lib.load().dc_last_error().decode()
    with pytest.raises(_lib.DcError, match="wider"):
        rolling_ball_device(x, 300, method="banded")
    # the widest accepted row runs (and the tiled kernel has no width limit)
    ok = torch.from_numpy(_frames((1, 3, 32768), 9)).cuda()
    got = rolling_ball_device(ok, 300).cpu().numpy()
    np.testing.assert_array_equal(got[0], cv2_rolling_ball(ok[0].cpu().numpy(), 300))
    assert rolling_ball_device(x, 50).shape == x.shape


def test_tiled_method_refuses_large_radius(cuda_device):
    import torch
    from unet_dc_segmentation_b200.morphology import rolling_ball_device, tiled_max_radius
    x = torch.zeros((1, 32, 32), dtype=torch.uint8, device="cuda")
    with pytest.raises(ValueError, match="tiled"):
        rolling_ball_device(x, tiled_max_radius() + 1, method="tiled")
    with pytest.raises(ValueError, match="radius must be in"):
        rolling_ball_device(x, 2048, method="banded")


def test_pipeline_radius_300_and_graphs(cuda_device):
    import torch
    from unet_dc_segmentation_b200 import DropletPipeline, UNetDC
    from unet_dc_segmentation_b200.morphology import rolling_ball_device
    from unet_dc_segmentation_b200.synth import calibrated_state_dict, synthetic_image
    m = UNetDC(3, 1)
    m.load_state_dict(calibrated_state_dict(seed=0, calib_size=64, n_calib=2))
    m = m.to(cuda_device).eval()
    frames = np.stack([synthetic_image(128, 600 + i, n_droplets=12) for i in range(2)])
    x = torch.from_numpy(frames).cuda()
    pipe = DropletPipeline(m, background_radius=300, prob_thresh=0.3, min_area=1, px_per_micron=3.45)
    res = pipe.run_device(x)
    masks, tables = res.masks.cpu().numpy(), res.tables.to_host()
    plain = DropletPipeline(m, background_radius=None, prob_thresh=0.3, min_area=1, px_per_micron=3.45)
    ref = plain.run_device(rolling_ball_device(x, 300))
    np.testing.assert_array_equal(masks, ref.masks.cpu().numpy())
    ref_tables = ref.tables.to_host()
    for i in range(2):
        assert set(tables[i]) == set(ref_tables[i])
        for c in tables[i]:
            np.testing.assert_array_equal(tables[i][c], ref_tables[i][c], err_msg=f"image {i} column {c}")
    # graph replay of the batch (the rolling ball's three launches included) against eager
    pinned = torch.from_numpy(frames).pin_memory()
    eager = [(mk.copy(), tb) for mk, tb in pipe.run_host_pipelined(pinned for _ in range(5))]
    gpipe = DropletPipeline(m, background_radius=300, prob_thresh=0.3, min_area=1, px_per_micron=3.45, use_graphs=True)
    for k, (mk, tb) in enumerate(gpipe.run_host_pipelined(pinned for _ in range(5))):
        np.testing.assert_array_equal(mk, eager[k][0], err_msg=f"graph batch {k}")
        np.testing.assert_array_equal(mk, masks, err_msg=f"graph batch {k}")
        for i in range(2):
            for c in eager[k][1][i]:
                np.testing.assert_array_equal(tb[i][c], eager[k][1][i][c], err_msg=f"graph batch {k} image {i} {c}")
    assert all(sl["graph"] is not None for sl in gpipe._slots)


def test_cli_background_radius_400(cuda_device, tmp_path):
    """--background_radius 400 writes what the CLI writes, without correction, for frames the reference's own
    rolling_ball_correction_rgb corrected (oracle/_ref where built, else cv2's four calls)."""
    import cv2
    import torch
    from PIL import Image
    from unet_dc_segmentation_b200 import cli
    from unet_dc_segmentation_b200.synth import calibrated_state_dict, synthetic_image
    try:
        from oracle import ref as oref
        ref_rb = oref.load().rolling_ball_correction_rgb if oref.available() else None
    except Exception:
        ref_rb = None
    raw, pre = tmp_path / "raw", tmp_path / "pre"
    raw.mkdir()
    pre.mkdir()
    for i in range(2):
        g = synthetic_image(96, 700 + i, n_droplets=10)
        Image.fromarray(g).save(raw / f"frame{i}.png")
        rgb = np.repeat(g[:, :, None], 3, axis=2)
        corr = ref_rb(rgb, 400) if ref_rb else np.stack([cv2_rolling_ball(rgb[:, :, c].copy(), 400) for c in range(3)], -1)
        assert np.array_equal(corr[:, :, 0], corr[:, :, 1]) and np.array_equal(corr[:, :, 0], corr[:, :, 2])
        Image.fromarray(np.ascontiguousarray(corr[:, :, 0])).save(pre / f"frame{i}.png")
    torch.save(calibrated_state_dict(seed=0, calib_size=64, n_calib=2), tmp_path / "ckpt.pth")
    common = ["--ckpt_path", str(tmp_path / "ckpt.pth"), "--batch", "2", "--skip_excel", "--skip_histogram",
              "--img_size", "96", "--px_per_micron", "3.45"]
    assert cli.main(["--img_dir", str(raw), "--out_dir", str(tmp_path / "o400"), "--background_radius", "400", *common]) == 0
    assert cli.main(["--img_dir", str(pre), "--out_dir", str(tmp_path / "o0"), "--background_radius", "0", *common]) == 0
    for i in range(2):
        a = cv2.imread(str(tmp_path / "o400" / "predicted_masks" / f"frame{i}_pred.png"), cv2.IMREAD_GRAYSCALE)
        b = cv2.imread(str(tmp_path / "o0" / "predicted_masks" / f"frame{i}_pred.png"), cv2.IMREAD_GRAYSCALE)
        np.testing.assert_array_equal(a, b, err_msg=f"frame{i} mask")
        assert (tmp_path / "o400" / f"frame{i}_droplets.csv").read_text() == (tmp_path / "o0" / f"frame{i}_droplets.csv").read_text()
    for name in ("summary_per_image.csv", "all_droplets.csv"):
        if (tmp_path / "o0" / name).exists():
            assert (tmp_path / "o400" / name).read_text() == (tmp_path / "o0" / name).read_text()
