"""GPU: every stage at the edges of the shapes it accepts.

Forward past 2^31 activation elements: a frame deep in a big batch (level-0 offsets >= 2^31) gives bit-identical
probabilities and mask to the same frame alone at B = 1, where every offset is small; the default schedule at
33 x 1024^2, 16 x 2048^2 and 4 x 4096^2, the unfused schedule at 32 x 1024^2 ([B,H,W,128] skip concatenation of 2^32
elements), the generic in/out-channel kernels at B = 65536.  Frames with tile grids hundreds of tiles wide or tall
(2048^2, 512 x 4096, 4096 x 512) against the fp32 reference network and the bf16 emulation.

Every other entry point on both sides of its grid limits, with buffers as large as the shape says: the last accepted
shape bit-exact against OpenCV / scipy / the oracle, the first refused one refused with DC_EINVAL and a message from
dc_last_error() before anything is launched.

Peak device memory is about 21 GiB (the 16 x 2048^2 and 4 x 4096^2 forwards; measured on a B200).  A test that cannot get the
memory it needs skips and names the figure."""
import ctypes as C

import numpy as np
import pytest

import oracle

pytestmark = pytest.mark.gpu

GRID_MAX = 65535            # gridDim.y / gridDim.z limit


@pytest.fixture(autouse=True)
def _free_between_tests():
    import torch
    if torch.cuda.is_available():
        torch.cuda.empty_cache()
        torch.cuda.reset_peak_memory_stats()
    yield
    if torch.cuda.is_available():
        print(f"peak device memory {torch.cuda.max_memory_allocated() / 2**30:.2f} GiB")
        torch.cuda.empty_cache()


def _need_gib(gib):
    import torch
    free, _ = torch.cuda.mem_get_info()
    if free < gib * 2**30:
        pytest.skip(f"needs {gib} GiB of free device memory, {free / 2**30:.1f} GiB free")


def _refused(rc, *words):
    """A refusal through the C ABI: DC_EINVAL, and dc_last_error() names the reason."""
    from unet_dc_segmentation_b200 import _lib
    msg = _lib.load().dc_last_error().decode()
    assert rc == _lib.DC_EINVAL, f"return code {rc} ({msg}), want DC_EINVAL"
    for w in words:
        assert w in msg, msg


def _refused_py(fn, *words):
    """The same through a Python wrapper, which raises DcError with the return code."""
    from unet_dc_segmentation_b200 import _lib
    with pytest.raises(_lib.DcError) as ei:
        fn()
    _refused(ei.value.code, *words)


# ---------------------------------------------------------------------------------------------- forward

def _model(device, **schedule):
    from unet_dc_segmentation_b200 import UNetDC
    from unet_dc_segmentation_b200.synth import calibrated_state_dict
    sd = calibrated_state_dict(seed=0)
    m = UNetDC(3, 1)
    m.load_state_dict(sd)
    for k, v in schedule.items():
        setattr(m, k, v)
    return m.to(device).eval(), sd


def _frames(B, H, W):
    """B distinct u8 frames: rolls of four synthetic bases."""
    from unet_dc_segmentation_b200.synth import synthetic_image
    base = np.stack([synthetic_image(max(H, W), 500 + i)[:H, :W] for i in range(min(B, 4))])
    return np.concatenate([np.roll(base, 37 * r, axis=2) for r in range((B + 3) // 4)])[:B]


@pytest.mark.parametrize("B,S,schedule,gib", [
    (33, 1024, "default", 14),          # the benchmark shape plus one frame: a[0] = 33 * 2^26 elements
    (32, 1024, "unfused", 20),          # cat[0] = [32,1024,1024,128] = 2^32 elements
    (16, 2048, "default", 24),
    (4, 4096, "default", 24),
])
def test_batch_past_2_31_elements_matches_solo(cuda_device, B, S, schedule, gib):
    import torch
    from unet_dc_segmentation_b200 import rolling_ball_device
    _need_gib(gib)
    kw = {} if schedule == "default" else {"fuse_level1": False, "parity_level1": False, "fuse_levels": ()}
    m, _ = _model(cuda_device, **kw)
    if schedule == "unfused":
        assert m.num_launches() == 22
    x = rolling_ball_device(torch.from_numpy(_frames(B, S, S)).to(cuda_device), 50)
    mask, prob = m.predict_u8(x, 0.3, return_prob=True)
    torch.cuda.synchronize()
    assert torch.equal(mask, (prob[:, 0] > 0.3).to(torch.uint8))
    per_frame = S * S * (128 if schedule == "unfused" else 64)        # widest level-0 tensor, elements per frame
    first_past = 2**31 // per_frame
    assert first_past < B and first_past * per_frame >= 2**31
    for i in sorted({0, first_past, B - 1}):
        m_i, p_i = m.predict_u8(x[i:i + 1], 0.3, return_prob=True)
        assert torch.equal(p_i[0], prob[i]), f"frame {i} of {B} x {S}^2 ({schedule}) differs from the frame alone"
        assert torch.equal(m_i[0], mask[i]), f"mask of frame {i}"
        del m_i, p_i
    assert 0.02 < float(mask[B - 1].float().mean()) < 0.6, "degenerate mask"
    del x, mask, prob
    m.invalidate()


def test_generic_kernels_at_batch_65536(cuda_device):
    """UNetDC(1, 2): the input conversion and the 1x1 head kernel (csrc/generic.cu) keep the batch in gridDim.y;
    past 65535 images each block walks the images b, b + 65535, ...  Frames 0, 65534 and 65535 against themselves
    alone."""
    import torch
    import unet_dc_segmentation_b200 as pkg
    _need_gib(20)
    torch.manual_seed(12)
    m = pkg.UNetDC(1, 2)
    for mod in m.modules():
        if isinstance(mod, torch.nn.BatchNorm2d):
            mod.running_mean.uniform_(-0.2, 0.2)
            mod.running_var.uniform_(0.5, 1.5)
    m.out_conv.weight.data.mul_(25.0)
    m = m.to(cuda_device).eval()
    assert m.num_launches() == 20
    B = GRID_MAX + 1
    g = torch.Generator(device=cuda_device).manual_seed(3)
    x = torch.rand((B, 1, 16, 16), generator=g, device=cuda_device)
    y = m(x)
    torch.cuda.synchronize()
    for i in (0, B - 2, B - 1):
        solo = m(x[i:i + 1])
        assert torch.equal(solo[0], y[i]), f"frame {i} of {B} differs from the frame alone"
    assert not torch.equal(y[0], y[B - 1])
    del x, y
    m.invalidate()


@pytest.mark.parametrize("H,W", [(2048, 2048), (512, 4096), (4096, 512)])
def test_large_and_non_square_frames_match_reference(cuda_device, H, W):
    """Tile grids hundreds of tiles wide or tall (256-tile rows / columns at level 0, 16 x 256 and 256 x 16 at the
    bottleneck) against the fp32 reference network and the bf16 emulation, with the tolerances and the band rule of
    test_gpu_fullsize.test_forward_parity_at_full_size."""
    import torch
    from test_gpu_forward import EMU_MEAN_TOL, EMU_TOL, MEAN_TOL, PROB_TOL, _fused
    from unet_dc_segmentation_b200 import rolling_ball_device
    _need_gib(8)
    m, sd = _model(cuda_device)
    raw = torch.from_numpy(_frames(1, H, W)).to(cuda_device)
    pre = rolling_ball_device(raw, 50)
    mask, prob = m.predict_u8(pre, 0.3, return_prob=True)
    got, mask = prob[0, 0].cpu().numpy(), mask[0].cpu().numpy()
    m.invalidate()
    x = torch.from_numpy(np.repeat(pre.cpu().numpy()[:, None], 3, 1).astype(np.float32) / 255.0)
    ref = oracle.unetdc_forward(sd, x).numpy()[0, 0]
    emu = oracle.unetdc_forward(sd, x, emulate_bf16=True, fused_levels=_fused(sd), gray_input=True).numpy()[0, 0]
    e_ref, e_emu = np.abs(got - ref), np.abs(got - emu)
    diff = mask != (ref > 0.3)
    in_band = np.abs(ref - 0.3) <= PROB_TOL
    print(f"{H}x{W}: vs fp32 max {e_ref.max():.4f} mean {e_ref.mean():.5f}; vs bf16 emulation max {e_emu.max():.4f} "
          f"mean {e_emu.mean():.5f}; mask pixels differing {int(diff.sum())} of {diff.size} "
          f"({int((diff & ~in_band).sum())} outside the band)")
    assert e_ref.max() <= PROB_TOL and e_ref.mean() <= MEAN_TOL
    assert e_emu.max() <= EMU_TOL and e_emu.mean() <= EMU_MEAN_TOL
    assert int((diff & ~in_band).sum()) == 0
    assert diff.mean() < 0.005
    assert 0.02 < float(mask.mean()) < 0.6, "degenerate mask"


# ---------------------------------------------------------------------------------------------- rolling ball

def _rb_call(entry, x, out, radius, ws):
    from unet_dc_segmentation_b200 import _lib
    B, H, W = x.shape[:3]
    Cc = 1 if x.dim() == 3 else x.shape[3]
    args = _lib.RollingBallArgs(x.data_ptr(), out.data_ptr(), B, H, W, Cc, radius, ws.data_ptr(), ws.numel())
    return getattr(_lib.load(), entry)(C.byref(args), _lib.stream_ptr())


@pytest.mark.parametrize("entry", ["dc_rolling_ball", "dc_rolling_ball_tiled", "dc_rolling_ball_banded"])
def test_rolling_ball_65535_planes(cuda_device, entry):
    import torch
    from test_gpu_rolling_ball_banded import cv2_rolling_ball
    from unet_dc_segmentation_b200.morphology import rolling_ball_workspace_bytes
    rs = np.random.RandomState(65535)
    H, W, radius = 12, 17, 7
    imgs = rs.randint(0, 256, (GRID_MAX + 1, H, W)).astype(np.uint8)
    imgs[:, 3:9, 4:12] //= 3
    x = torch.from_numpy(imgs).cuda()
    ws = torch.empty(rolling_ball_workspace_bytes(GRID_MAX + 1, H, W), dtype=torch.uint8, device="cuda")
    out = torch.empty_like(x)
    _refused(_rb_call(entry, x, out, radius, ws), "65535 planes")
    xa, outa = x[:GRID_MAX], out[:GRID_MAX]
    assert _rb_call(entry, xa, outa, radius, ws) == 0
    got = outa.cpu().numpy()
    bad = [b for b in range(GRID_MAX) if not np.array_equal(got[b], cv2_rolling_ball(imgs[b], radius))]
    assert not bad, f"{len(bad)} planes differ from cv2, first {bad[:5]}"


@pytest.mark.parametrize("radius,tile", [(50, 128), (170, 32)])
def test_rolling_ball_taller_than_tiled_grid(cuda_device, radius, tile):
    """H = 65535 * tile + 16 (65536 + 1 rows of tiles): "auto" runs the banded pass (gridDim.x holds its row bands)
    and matches cv2 on the same frame; "tiled" refuses.  65535 rows of tiles still run tiled, bit for bit what the
    banded pass gives."""
    import torch
    from test_gpu_rolling_ball_banded import cv2_rolling_ball
    from unet_dc_segmentation_b200.morphology import rolling_ball_device
    W = 4
    H = 2**23 + 16 if tile == 128 else 2**21 + 16
    assert (H + tile - 1) // tile > GRID_MAX
    rs = np.random.RandomState(radius)
    y = np.arange(H)[:, None]
    img = (96 + 80 * np.sin(y / 5000.0) + rs.randint(0, 64, (H, W))).astype(np.uint8)
    img[H // 3:H // 3 + 4000] //= 4
    x = torch.from_numpy(img[None]).cuda()
    want = cv2_rolling_ball(img, radius)
    np.testing.assert_array_equal(rolling_ball_device(x, radius).cpu().numpy()[0], want)
    np.testing.assert_array_equal(rolling_ball_device(x, radius, method="banded").cpu().numpy()[0], want)
    _refused_py(lambda: rolling_ball_device(x, radius, method="tiled"), "too tall", f"{tile}-row tiles")
    xt = x[:, :GRID_MAX * tile]                  # the tallest frame the tiled grid holds
    assert torch.equal(rolling_ball_device(xt, radius, method="tiled"), rolling_ball_device(xt, radius, method="banded"))


def test_rolling_ball_2_31_pixels_refused(cuda_device):
    import torch
    from unet_dc_segmentation_b200.morphology import rolling_ball_workspace_bytes
    _need_gib(7)
    H, W = 2**16, 2**15                         # 2^31 pixels: one too many for int32 indices
    x = torch.zeros((1, H, W), dtype=torch.uint8, device="cuda")
    ws = torch.empty(rolling_ball_workspace_bytes(1, H, W), dtype=torch.uint8, device="cuda")
    for entry in ("dc_rolling_ball", "dc_rolling_ball_tiled", "dc_rolling_ball_banded"):
        _refused(_rb_call(entry, x, x, 50, ws), "too large")


# ---------------------------------------------------------------------------------------------- labels, overlay

def _check_tables(tables, labels, masks):
    """Label images and every table column bit for bit against the oracle, image by image."""
    for b in range(masks.shape[0]):
        want_l, want = oracle.quantify_arrays(masks[b], 1, 3.45)
        np.testing.assert_array_equal(labels[b], want_l, err_msg=f"labels of image {b}")
        for c, v in want.items():
            np.testing.assert_array_equal(np.asarray(tables[b][c]), v, err_msg=f"image {b} column {c}")


def test_label_stats_and_overlay_batch_65535(cuda_device):
    import torch
    from overlay_cases import _cv2_overlay_stencil
    from unet_dc_segmentation_b200 import label_stats_device, overlay_stencil_device
    rs = np.random.RandomState(7)
    masks = (rs.rand(GRID_MAX + 1, 16, 16) < 0.4).astype(np.uint8)
    m = torch.from_numpy(masks).cuda()
    _refused_py(lambda: label_stats_device(m, 1, 3.45, capacity=128), "batch > 65535")
    _refused_py(lambda: overlay_stencil_device(m), "batch > 65535")
    t = label_stats_device(m[:GRID_MAX], 1, 3.45, capacity=128, want_labels=True)
    _check_tables(t.to_host(), t.labels.cpu().numpy(), masks[:GRID_MAX])
    got = overlay_stencil_device(m[:GRID_MAX]).cpu().numpy()
    bad = [b for b in range(GRID_MAX) if not np.array_equal(got[b], _cv2_overlay_stencil(masks[b]))]
    assert not bad, f"{len(bad)} stencils differ from OpenCV, first {bad[:5]}"


def test_label_stats_and_overlay_tallest_frame(cuda_device):
    """H = 65535 * 128 (128-row tiles, gridDim.y = 65535) against the oracle and OpenCV; one row more is refused."""
    import torch
    from overlay_cases import _cv2_overlay_stencil
    from unet_dc_segmentation_b200 import label_stats_device, overlay_stencil_device
    H = GRID_MAX * 128
    rs = np.random.RandomState(128)
    tall = (rs.rand(H + 1, 3) < 0.97).astype(np.uint8)           # long vertical runs, joined across columns
    over = np.repeat(rs.rand((H + 1) // 64 + 1, 16) < 0.5, 64, axis=0)[:H + 1].astype(np.uint8)
    for arr in (tall, over):
        m = torch.from_numpy(arr[None]).cuda()
        _refused_py(lambda: label_stats_device(m, 1, 3.45), "too tall")
        _refused_py(lambda: overlay_stencil_device(m), "too tall")
    mt = np.ascontiguousarray(tall[:H])
    t = label_stats_device(torch.from_numpy(mt[None]).cuda(), 1, 3.45, capacity=H * 3 // 2, want_labels=True)
    assert 1000 < int(t.counts[0]) <= t.capacity
    _check_tables(t.to_host(), t.labels.cpu().numpy(), mt[None])
    del t
    mo = np.ascontiguousarray(over[:H])
    got = overlay_stencil_device(torch.from_numpy(mo[None]).cuda()).cpu().numpy()[0]
    want = _cv2_overlay_stencil(mo)
    assert 0 < int(want.sum()) < want.size
    np.testing.assert_array_equal(got, want)


# ---------------------------------------------------------------------------------------------- resize

def test_resize_at_grid_limits(cuda_device):
    import cv2
    import torch
    from unet_dc_segmentation_b200.morphology import resize_linear_u8_device
    rs = np.random.RandomState(5)
    src = rs.randint(0, 256, (2, 37, 5, 3)).astype(np.uint8)
    x = torch.from_numpy(src).cuda()
    _refused_py(lambda: resize_linear_u8_device(x, (3, GRID_MAX + 1)), "dst_h")
    got = resize_linear_u8_device(x, (3, GRID_MAX)).cpu().numpy()
    for b in range(2):
        np.testing.assert_array_equal(got[b], cv2.resize(src[b], (3, GRID_MAX)), err_msg=f"dst_h 65535 image {b}")
    many = rs.randint(0, 256, (GRID_MAX + 1, 6, 9)).astype(np.uint8)
    xm = torch.from_numpy(many).cuda()
    _refused_py(lambda: resize_linear_u8_device(xm, (4, 11)), "B above 65535")
    got = resize_linear_u8_device(xm[:GRID_MAX], (4, 11)).cpu().numpy()
    bad = [b for b in range(GRID_MAX) if not np.array_equal(got[b], cv2.resize(many[b], (4, 11)))]
    assert not bad, f"{len(bad)} images differ from cv2.resize, first {bad[:5]}"


# ---------------------------------------------------------------------------------------------- density

def test_roi_mask_tallest_frame(cuda_device):
    import cv2
    import torch
    from test_gpu_density import _tissue
    from unet_dc_segmentation_b200 import density
    rs = np.random.RandomState(16)
    H, W = GRID_MAX, 24
    img = _tissue(rs, H + 1, W)
    x = torch.from_numpy(img[None]).cuda()
    _refused_py(lambda: density.roi_mask_device(x), "bad shape")
    img = np.ascontiguousarray(img[:H])
    roi, cen = density.roi_mask_device(torch.from_numpy(img[None]).cuda())
    roi, cen = roi.cpu().numpy()[0], cen.cpu().numpy()[0]
    kernel = np.ones((15, 15), np.uint8)
    blurred = cv2.GaussianBlur(cv2.cvtColor(img, cv2.COLOR_RGB2GRAY), (15, 15), 0)
    _, mk = cv2.threshold(blurred, 0, 255, cv2.THRESH_BINARY + cv2.THRESH_OTSU)
    mk = cv2.morphologyEx(cv2.morphologyEx(mk, cv2.MORPH_CLOSE, kernel), cv2.MORPH_OPEN, kernel)
    want = (mk > 0).astype(np.uint8)
    assert 0 < int(want.sum()) < want.size
    np.testing.assert_array_equal(roi, want)
    M = cv2.moments(want)
    assert tuple(cen) == (int(M["m01"] / M["m00"]), int(M["m10"] / M["m00"]))


def test_spatial_density_tallest_frame(cuda_device):
    import torch
    from scipy.ndimage import gaussian_filter
    from unet_dc_segmentation_b200 import density
    rs = np.random.RandomState(17)
    H, W = 16 * GRID_MAX, 6
    mask = (rs.rand(H + 1, W) < 0.05).astype(np.uint8)
    roi = np.repeat(rs.rand((H + 1) // 512 + 1, 1) < 0.7, 512, axis=0)[:H + 1].repeat(W, 1).astype(np.uint8)
    m, r = torch.from_numpy(mask[None]).cuda(), torch.from_numpy(roi[None]).cuda()
    _refused_py(lambda: density.spatial_density_device(m, r, 21), "too tall")
    got = density.spatial_density_device(m[:, :H], r[:, :H], 21).cpu().numpy()[0]
    mh, rh = mask[:H].astype(np.float32), roi[:H].astype(np.float32)
    want = gaussian_filter(mh, sigma=21 / 6)
    want = want / (gaussian_filter(rh, sigma=21 / 6) + 1e-5)
    want *= 100
    np.testing.assert_array_equal(got, want)
