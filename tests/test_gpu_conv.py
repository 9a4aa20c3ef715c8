"""GPU: the tensor-core layers (csrc/conv_tc.cu) and the stem (csrc/stem.cu), one layer at a time, against
a plain PyTorch fp32 CPU evaluation of the same op on the same bf16-rounded operands.

Tolerance (floating point, stated here): operands are bf16 on both sides, the kernel accumulates in fp32
(TMEM) like the fp32 CPU reference, and the only extra error is the final bf16 rounding of the output
(rel 2^-9) plus accumulation-order noise: |got - want| <= 1e-2 * max(1, |want|)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture
def conv_family():
    """dc_debug_set_conv_family for the duration of one test (the product path never calls it)."""
    from unet_dc_segmentation_b200 import _lib
    lib = _lib.load()
    codes = {"auto": _lib.DC_CONV_FAMILY_AUTO, "generic": _lib.DC_CONV_FAMILY_GENERIC}
    yield lambda name: _lib.check(lib.dc_debug_set_conv_family(codes[name]))
    _lib.check(lib.dc_debug_set_conv_family(_lib.DC_CONV_FAMILY_AUTO))


def _close(got, want, what=""):
    import torch
    got = got.float().cpu()
    err = (got - want).abs()
    tol = 1e-2 * want.abs().clamp(min=1.0)
    bad = err > tol
    assert not bool(bad.any()), (f"{what}: {int(bad.sum())}/{bad.numel()} elements off, max err {float(err.max()):.4g}, "
                                 f"first bad index {tuple(int(v) for v in bad.nonzero()[0])}")


def _rand_layer(cin, cout, seed):
    import torch
    g = torch.Generator().manual_seed(seed)
    w = (torch.randn(cout, cin, 3, 3, generator=g) / (3.0 * cin ** 0.5)).bfloat16().float()
    b = torch.randn(cout, generator=g) * 0.1
    return w, b


def _rand_act(B, H, W, C, seed):
    import torch
    g = torch.Generator().manual_seed(seed)
    return torch.randn(B, H, W, C, generator=g).bfloat16()


CONV_CASES = [
    # B, H, W, Cin, Cout, dilation
    (1, 8, 16, 64, 64, 1),        # exactly one tile
    (2, 16, 32, 64, 64, 1),
    (1, 24, 40, 64, 128, 2),      # partial tiles in both directions
    (2, 16, 16, 128, 128, 2),
    (1, 32, 48, 128, 256, 4),
    (1, 16, 16, 256, 512, 8),     # two N tiles
    (2, 8, 8, 512, 1024, 16),     # dilation > map: only the centre tap is in bounds
    (1, 16, 32, 1024, 512, 1),    # long K
    (3, 40, 24, 192, 64, 3),      # Cin not a power of two, odd dilation; single-CTA halo kernel, weights streamed
    (2, 48, 24, 128, 64, 1),      # dec1.0 shape: halo kernel, two chunks, weights resident
    (1, 40, 40, 64, 128, 2),      # enc2.0 shape: halo kernel, BN = 128, dilation 2
    (1, 32, 16, 64, 64, 4),       # halo kernel, dilation 4
    (2, 16, 8, 64, 64, 1),        # exactly one 16 x 8 halo tile per image
    (1, 48, 40, 256, 512, 1),     # CTA-pair kernel, BN = 256, two n-tiles, odd number of m-tiles (15)
    (3, 16, 24, 128, 256, 4),     # CTA-pair kernel, BN = 256, dilation 4
    (1, 16, 8, 512, 256, 2),      # CTA-pair kernel, a single m-tile (the peer CTA redoes it)
    (1, 64, 64, 512, 1024, 16),   # bottleneck.0 of a 1024^2 frame (model_2.py:16): dilation 16 with every tap in bounds
    (1, 48, 80, 1024, 1024, 16),  # bottleneck.3: ragged map, taps partly in the padding
    (2, 32, 48, 256, 512, 8),     # enc4.0 (model_2.py:13): dilation 8, non-centre taps in bounds
    (1, 128, 128, 512, 512, 8),   # enc4.3 at its 1024^2-frame size
]


@pytest.mark.parametrize("B,H,W,cin,cout,d", CONV_CASES)
def test_conv3x3_store(cuda_device, B, H, W, cin, cout, d):
    import torch
    import torch.nn.functional as F
    from unet_dc_segmentation_b200 import layers
    from unet_dc_segmentation_b200.model import pack_conv3x3
    w, b = _rand_layer(cin, cout, 1000 + cin + cout + d)
    x = _rand_act(B, H, W, cin, 7 + H * W)
    want = F.relu(F.conv2d(x.float().permute(0, 3, 1, 2), w, b, padding=d, dilation=d)).permute(0, 2, 3, 1)
    got = layers.conv3x3(x.cuda(), pack_conv3x3(w).cuda(), b.cuda(), dilation=d, relu=True)
    torch.cuda.synchronize()
    _close(got, want, f"conv {cin}->{cout} d{d} {B}x{H}x{W}")


@pytest.mark.parametrize("B,H,W,cin,cout,d", [(2, 16, 32, 64, 64, 1), (1, 24, 40, 64, 128, 2), (1, 32, 48, 128, 256, 4)])
def test_conv3x3_generic_path_forced(cuda_device, conv_family, B, H, W, cin, cout, d):
    """Most layers take the CTA-pair halo kernel; the test-only family switch keeps the per-tap kernel covered."""
    conv_family("generic")
    test_conv3x3_store(cuda_device, B, H, W, cin, cout, d)


@pytest.mark.parametrize("family", ["generic", "single_cta"])
def test_fused_epilogues_on_the_fallback_kernels(cuda_device, conv_family, family):
    """Pool, head and transposed-conv epilogues through the per-tap kernel (forced), and pool and head through the
    single-CTA halo kernel, which AUTO picks for 256 -> 64 at dilation 1."""
    if family == "generic":
        conv_family("generic")
        _store_pool(1, 16, 32, 64, 64, 1)
        _store_pool(2, 24, 48, 128, 128, 2)
        _head(64)
        test_upconv2x2(cuda_device, 1, 8, 16, 128, 64)
    else:
        _store_pool(2, 24, 32, 256, 64, 1)
        _head(256)


def test_conv3x3_no_relu_and_channel_slices(cuda_device):
    """Reads channels [0,64) of a 128-wide buffer and writes channels [64,128) of another (the concat layout)."""
    import torch
    import torch.nn.functional as F
    from unet_dc_segmentation_b200 import layers
    from unet_dc_segmentation_b200.model import pack_conv3x3
    w, b = _rand_layer(64, 64, 5)
    xin = _rand_act(2, 16, 32, 128, 9)
    out = torch.full((2, 16, 32, 128), 7.0, dtype=torch.bfloat16).cuda()
    want = F.conv2d(xin[..., :64].float().permute(0, 3, 1, 2), w, b, padding=1).permute(0, 2, 3, 1)
    layers.conv3x3(xin.cuda(), pack_conv3x3(w).cuda(), b.cuda(), relu=False, cin=64, out=out, out_offset=64)
    torch.cuda.synchronize()
    _close(out[..., 64:], want, "sliced conv")
    assert bool((out[..., :64].float() == 7.0).all()), "wrote outside its channel slice"


def _store_pool(B, H, W, cin, cout, d):
    import torch
    import torch.nn.functional as F
    from unet_dc_segmentation_b200 import layers
    from unet_dc_segmentation_b200.model import pack_conv3x3
    w, b = _rand_layer(cin, cout, 77 + cin)
    x = _rand_act(B, H, W, cin, 3 + cin)
    full = F.relu(F.conv2d(x.float().permute(0, 3, 1, 2), w, b, padding=d, dilation=d))
    got, pooled = layers.conv3x3(x.cuda(), pack_conv3x3(w).cuda(), b.cuda(), dilation=d, pool=True)
    torch.cuda.synchronize()
    _close(got, full.permute(0, 2, 3, 1), "pool: full-res output")
    # the pooled tensor must be EXACTLY the 2x2 max of the bf16 full-res tensor the kernel wrote
    want_pool = F.max_pool2d(got.float().cpu().permute(0, 3, 1, 2), 2).permute(0, 2, 3, 1)
    assert torch.equal(pooled.float().cpu(), want_pool)


@pytest.mark.parametrize("B,H,W,c,d", [(1, 16, 32, 64, 1), (2, 24, 48, 128, 2), (1, 16, 16, 256, 4)])
def test_conv3x3_store_pool(cuda_device, B, H, W, c, d):
    _store_pool(B, H, W, c, c, d)


@pytest.mark.parametrize("B,H,W,cin,cout", [(1, 8, 16, 128, 64), (2, 12, 20, 256, 128), (1, 8, 8, 1024, 512)])
def test_upconv2x2(cuda_device, B, H, W, cin, cout):
    import torch
    import torch.nn.functional as F
    from unet_dc_segmentation_b200 import layers
    from unet_dc_segmentation_b200.model import pack_upconv
    g = torch.Generator().manual_seed(cin + cout)
    w = (torch.randn(cin, cout, 2, 2, generator=g) / cin ** 0.5).bfloat16().float()
    b = torch.randn(cout, generator=g) * 0.1
    x = _rand_act(B, H, W, cin, 11 + cin)
    want = F.conv_transpose2d(x.float().permute(0, 3, 1, 2), w, b, stride=2).permute(0, 2, 3, 1)
    cat = torch.zeros((B, 2 * H, 2 * W, 2 * cout), dtype=torch.bfloat16).cuda()
    layers.upconv2x2(x.cuda(), pack_upconv(w).cuda(), b.cuda(), out=cat, out_offset=0)
    torch.cuda.synchronize()
    _close(cat[..., :cout], want, f"upconv {cin}->{cout}")
    assert bool((cat[..., cout:] == 0).all())


UPFUSED_CASES = [
    # B, H, W of the transposed conv's input (the output is twice that)
    (1, 16, 8),       # exactly one tile: its pair partner redoes it
    (2, 16, 8),       # one pair
    (1, 40, 24),      # ragged rows, three tile columns, odd tile count
    (3, 24, 20),      # ragged in both directions
    (2, 64, 64),      # several waves of pairs on a small grid
    (1, 8, 8),        # smaller than a tile
]


@pytest.mark.parametrize("B,H,W", UPFUSED_CASES)
def test_upconv_conv3x3_fused(cuda_device, B, H, W):
    """dc_conv_upfused (upconv1 + dec1.0 as one launch) against the CPU evaluation of the same composed blobs, and
    loosely against the unfused fp32 chain conv_transpose2d -> cat -> conv2d it stands for."""
    import torch
    import torch.nn.functional as F
    import oracle
    from unet_dc_segmentation_b200 import layers
    from unet_dc_segmentation_b200.model import compose_upconv, pack_upfused
    g = torch.Generator().manual_seed(B * 1000 + H * 10 + W)
    wu = torch.randn(128, 64, 2, 2, generator=g) / 128 ** 0.5
    bu = torch.randn(64, generator=g) * 0.3
    wd = torch.randn(64, 128, 3, 3, generator=g) / (3.0 * 128 ** 0.5)
    bd = torch.randn(64, generator=g) * 0.1
    comp, skipw, bias9 = compose_upconv(wu, bu, wd, bd)
    weight = pack_upfused(comp, skipw)
    x = _rand_act(B, H, W, 128, 5)
    cat = _rand_act(B, 2 * H, 2 * W, 128, 6)              # skip = channels [64,128) of a 128-channel buffer
    xs, ss = x.float().permute(0, 3, 1, 2), cat[..., 64:].float().permute(0, 3, 1, 2)
    for relu in (True, False):
        want = oracle.composed_upconv_conv3x3(xs, ss, comp, skipw, bias9, relu=relu).permute(0, 2, 3, 1)
        out = torch.full((B, 2 * H, 2 * W, 96), 7.0, dtype=torch.bfloat16).cuda()
        layers.upconv_conv3x3(x.cuda(), cat.cuda(), weight.cuda(), bias9.cuda(), relu=relu, skip_offset=64, out=out,
                              out_offset=16)
        torch.cuda.synchronize()
        _close(out[..., 16:80], want, f"fused upconv+conv {B}x{H}x{W} relu={relu}")
        assert bool((out[..., :16] == 7).all()) and bool((out[..., 80:] == 7).all())
    chain = F.relu(F.conv2d(torch.cat([F.conv_transpose2d(xs, wu, bu, stride=2), ss], 1), wd, bd, padding=1)).permute(0, 2, 3, 1)
    err = (out[..., 16:80].float().cpu().clamp(min=0) - chain).abs().max()
    assert float(err) < 0.05, f"fused layer vs unfused fp32 chain: max err {float(err):.4f}"


WIDE_CASES = [
    # C, B, H, W of the transposed conv's input
    (128, 1, 16, 8), (128, 2, 24, 20), (128, 1, 40, 24),
    (256, 1, 16, 8), (256, 2, 24, 12), (256, 1, 8, 8),
    (512, 1, 16, 8), (512, 2, 16, 16), (512, 1, 24, 20),
]


@pytest.mark.parametrize("C,B,H,W", WIDE_CASES)
def test_upconv_conv3x3_fused_wide(cuda_device, C, B, H, W):
    """dc_conv_upfused for the deeper decoder levels (upconv{2,3,4} + dec{2,3,4}.0: conv_upfused_wide_kernel, the
    parity classes walked in passes) against the CPU evaluation of the same composed weights and, loosely, the
    unfused fp32 chain."""
    import torch
    import torch.nn.functional as F
    import oracle
    from unet_dc_segmentation_b200 import layers
    from unet_dc_segmentation_b200.model import compose_upconv, pack_upfused_wide
    g = torch.Generator().manual_seed(C + B * 1000 + H * 10 + W)
    wu = torch.randn(2 * C, C, 2, 2, generator=g) / (2 * C) ** 0.5
    bu = torch.randn(C, generator=g) * 0.3
    wd = torch.randn(C, 2 * C, 3, 3, generator=g) / (3.0 * (2 * C) ** 0.5)
    bd = torch.randn(C, generator=g) * 0.1
    comp, skipw, bias9 = compose_upconv(wu, bu, wd, bd)
    wx, ws = pack_upfused_wide(comp, skipw)
    x = _rand_act(B, H, W, 2 * C, 5)
    cat = _rand_act(B, 2 * H, 2 * W, 2 * C, 6)            # skip = channels [C, 2C) of a 2C-channel buffer
    xs, ss = x.float().permute(0, 3, 1, 2), cat[..., C:].float().permute(0, 3, 1, 2)
    for relu in (True, False):
        want = oracle.composed_upconv_conv3x3(xs, ss, comp, skipw, bias9, relu=relu).permute(0, 2, 3, 1)
        out = torch.full((B, 2 * H, 2 * W, C + 32), 7.0, dtype=torch.bfloat16).cuda()
        layers.upconv_conv3x3(x.cuda(), cat.cuda(), wx.cuda(), bias9.cuda(), relu=relu, skip_offset=C, out=out,
                              out_offset=16, weight_skip=ws.cuda())
        torch.cuda.synchronize()
        _close(out[..., 16:16 + C], want, f"fused upconv+conv C={C} {B}x{H}x{W} relu={relu}")
        assert bool((out[..., :16] == 7).all()) and bool((out[..., 16 + C:] == 7).all())
    chain = F.relu(F.conv2d(torch.cat([F.conv_transpose2d(xs, wu, bu, stride=2), ss], 1), wd, bd, padding=1)).permute(0, 2, 3, 1)
    err = (out[..., 16:16 + C].float().cpu().clamp(min=0) - chain).abs().max()
    assert float(err) < 0.06, f"fused layer vs unfused fp32 chain: max err {float(err):.4f}"


PARITY_CASES = [(1, 32, 16), (2, 32, 16), (1, 80, 48), (3, 48, 40), (2, 128, 128), (1, 16, 16), (1, 2, 2)]


@pytest.mark.parametrize("B,H,W", PARITY_CASES)
def test_conv3x3_parity_class_kernel(cuda_device, B, H, W):
    """dc_conv_tc with weight_par: a 64 -> 64 channel 3x3 layer computed per output parity class with shared windows
    (conv_par2_kernel, what enc1.3 / dec1.3 run): plain store (+ channel slices, no ReLU), store + 2x2 max pool, and
    the out_conv + sigmoid + threshold head, each against the fp32 evaluation and the generic kernel's contract."""
    import torch
    import torch.nn.functional as F
    from unet_dc_segmentation_b200 import layers
    from unet_dc_segmentation_b200.model import pack_conv3x3, pack_par3x3
    w, b = _rand_layer(64, 64, 31 + H)
    wp = pack_par3x3(w).cuda()
    xin = _rand_act(B, H, W, 128, 9 + W)                      # the layer reads channels [0,64) of a 128-wide buffer
    xs = xin[..., :64].float().permute(0, 3, 1, 2)
    lin = F.conv2d(xs, w, b, padding=1)
    # store, no ReLU, into a channel slice
    out = torch.full((B, H, W, 160), 7.0, dtype=torch.bfloat16).cuda()
    layers.conv3x3(xin.cuda(), pack_conv3x3(w).cuda(), b.cuda(), relu=False, cin=64, out=out, out_offset=64, weight_par=wp)
    torch.cuda.synchronize()
    _close(out[..., 64:128], lin.permute(0, 2, 3, 1), f"parity store {B}x{H}x{W}")
    assert bool((out[..., :64] == 7).all()) and bool((out[..., 128:] == 7).all()), "wrote outside its channel slice"
    # store + pool
    got, pooled = layers.conv3x3(xin.cuda(), pack_conv3x3(w).cuda(), b.cuda(), cin=64, pool=True, weight_par=wp)
    torch.cuda.synchronize()
    _close(got, F.relu(lin).permute(0, 2, 3, 1), "parity pool: full-res output")
    want_pool = F.max_pool2d(got.float().cpu().permute(0, 3, 1, 2), 2).permute(0, 2, 3, 1)
    assert torch.equal(pooled.float().cpu(), want_pool)       # EXACTLY the 2x2 max of the bf16 tensor the kernel wrote
    # head
    g = torch.Generator().manual_seed(3)
    hw, hb = torch.randn(64, generator=g) * 0.2, 0.1
    want = torch.sigmoid((F.relu(lin) * hw.view(1, -1, 1, 1)).sum(1) + hb)
    x64 = xin[..., :64].contiguous()
    prob, mask = layers.conv3x3_head(x64.cuda(), pack_conv3x3(w).cuda(), b.cuda(), hw.cuda(), hb, 0.3, weight_par=wp)
    torch.cuda.synchronize()
    err = (prob.cpu() - want).abs().max()
    assert float(err) < 2e-3, f"parity head prob max err {float(err)}"
    assert torch.equal(mask.cpu(), (prob.cpu() > 0.3).to(torch.uint8))


def _head(cin):
    import torch
    import torch.nn.functional as F
    from unet_dc_segmentation_b200 import layers
    from unet_dc_segmentation_b200.model import pack_conv3x3
    w, b = _rand_layer(cin, 64, 31)
    g = torch.Generator().manual_seed(2)
    hw = torch.randn(64, generator=g) * 0.3
    hb = -0.2
    x = _rand_act(2, 24, 32, cin, 13)
    feat = F.relu(F.conv2d(x.float().permute(0, 3, 1, 2), w, b, padding=1))
    want = torch.sigmoid((feat * hw.view(1, -1, 1, 1)).sum(1) + hb)
    prob, mask = layers.conv3x3_head(x.cuda(), pack_conv3x3(w).cuda(), b.cuda(), hw.cuda(), hb, 0.3)
    torch.cuda.synchronize()
    err = (prob.cpu() - want).abs().max()
    assert float(err) < 2e-3, f"head prob max err {float(err)}"             # no bf16 rounding of the features here
    assert torch.equal(mask.cpu(), (prob.cpu() > 0.3).to(torch.uint8))     # mask is exactly `prob > thresh`


def test_head_epilogue(cuda_device):
    _head(64)


@pytest.mark.parametrize("kind", ["f32_nchw", "u8_gray", "u8_hwc"])
@pytest.mark.parametrize("d", [1, 2])
def test_stem(cuda_device, kind, d):
    import torch
    import torch.nn.functional as F
    from unet_dc_segmentation_b200 import layers
    g = torch.Generator().manual_seed(5)
    w = torch.randn(64, 3, 3, 3, generator=g) * 0.2
    b = torch.randn(64, generator=g) * 0.1
    B, H, W = 2, 20, 36
    if kind == "f32_nchw":
        x = torch.rand(B, 3, H, W, generator=g)
        ref_in, dev_in = x, x.cuda()
    elif kind == "u8_gray":
        u = torch.randint(0, 256, (B, H, W), generator=g, dtype=torch.uint8)
        ref_in, dev_in = (u.float() / 255.0)[:, None].expand(B, 3, H, W), u.cuda()
    else:
        u = torch.randint(0, 256, (B, H, W, 3), generator=g, dtype=torch.uint8)
        ref_in, dev_in = (u.float() / 255.0).permute(0, 3, 1, 2), u.cuda()
    want = F.relu(F.conv2d(ref_in, w, b, padding=d, dilation=d)).permute(0, 2, 3, 1)
    got = layers.stem(dev_in, w.reshape(64, 27).contiguous().cuda(), b.cuda(), dilation=d)
    torch.cuda.synchronize()
    _close(got, want, f"stem {kind} d{d}")


def test_bad_arguments_raise(cuda_device):
    import torch
    from unet_dc_segmentation_b200 import _lib, layers
    x = torch.zeros((1, 8, 16, 48), dtype=torch.bfloat16).cuda()
    w = torch.zeros((64, 9 * 48), dtype=torch.bfloat16).cuda()
    with pytest.raises(_lib.DcError) as ei:
        layers.conv3x3(x, w, torch.zeros(64).cuda())
    assert ei.value.code == _lib.DC_EINVAL and "multiple of 64" in str(ei.value)


def test_upfused_bad_arguments_raise(cuda_device):
    """dc_conv_upfused refuses what it cannot run: channel counts outside 64 / 128 / 256 / 512, a wide level without its
    skip-weight blob, strides smaller than the channels read, misaligned output slices."""
    import torch
    from unet_dc_segmentation_b200 import _lib, layers
    z = lambda *s: torch.zeros(s, dtype=torch.bfloat16).cuda()
    with pytest.raises(_lib.DcError) as ei:                               # C = 96
        layers.upconv_conv3x3(z(1, 8, 8, 192), z(1, 16, 16, 96), z(16, 64), torch.zeros(9, 96).cuda())
    assert ei.value.code == _lib.DC_EINVAL and "channels" in str(ei.value)
    with pytest.raises(_lib.DcError) as ei:                               # C = 128 without weight_skip
        layers.upconv_conv3x3(z(1, 8, 8, 256), z(1, 16, 16, 128), z(8192, 64), torch.zeros(9, 128).cuda())
    assert ei.value.code == _lib.DC_EINVAL and "weight_skip" in str(ei.value)
    with pytest.raises(_lib.DcError) as ei:                               # x narrower than 2 C
        layers.upconv_conv3x3(z(1, 8, 8, 64), z(1, 16, 16, 64), z(2, 2176, 64), torch.zeros(9, 64).cuda())
    assert ei.value.code == _lib.DC_EINVAL and "x_stride" in str(ei.value)
    with pytest.raises(_lib.DcError) as ei:                               # output slice not 16-byte aligned
        layers.upconv_conv3x3(z(1, 8, 8, 128), z(1, 16, 16, 64), z(2, 2176, 64), torch.zeros(9, 64).cuda(),
                              out=z(1, 16, 16, 80), out_offset=4)
    assert ei.value.code == _lib.DC_EINVAL and "out_offset" in str(ei.value)
