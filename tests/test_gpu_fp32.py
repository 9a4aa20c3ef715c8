"""GPU: the fp32-precision forward (UNetDC.precision = "fp32", dc_conv_args.planes = 3, DC_PRECISION_FP32).

Exact tier: on the operand families of tests/split_model.py (every one of the six plane products carries part of some
compared output, every partial sum exact in fp32) each split layer must store the three planes of the float64 result
bit for bit; on integer networks whose activations need more than 8 bits (12-bit input frames) the whole forward must
give the float64 logits.  Outputs sit between sentinel guards, unread input channels hold bf16 NaN, the forward's
workspace is filled with 0xFF.  Tolerance tier: a calibrated network (real-valued weights) against float64 (P_TOL below
says why it is 1e-3, not the 1e-4 first aimed at)."""
import ctypes

import numpy as np
import pytest
import torch

import exact_net as en
import split_model as sm

pytestmark = pytest.mark.gpu

GUARD, SENT, SENT16 = en.GUARD, en.SENT, en.SENT16
THRESH = 0.3


def _L():
    from unet_dc_segmentation_b200 import _lib
    return _lib


_guarded, _check_guards, _conv, _assert_planes = en.guarded, en.check_guards, en.conv_tc, sm.assert_planes


# (B, H, W, Cin, Cout, dilation): the Cin / Cout families and dilations of the network, odd shapes for the borders
CONV_CASES = [(1, 16, 16, 64, 64, 1), (2, 24, 40, 64, 128, 2), (1, 32, 24, 128, 256, 4), (1, 16, 16, 256, 512, 8),
              (2, 8, 8, 512, 1024, 16), (1, 16, 32, 1024, 512, 1), (1, 12, 20, 128, 64, 3), (1, 40, 24, 128, 128, 1),
              (2, 16, 8, 1024, 1024, 16), (1, 8, 48, 256, 256, 2)]


@pytest.mark.parametrize("i", range(len(CONV_CASES)))
@pytest.mark.parametrize("kind", sm.KINDS)
def test_split_conv_store_exact(cuda_device, i, kind):
    from unet_dc_segmentation_b200.model import pack_conv3x3_split
    L = _L()
    B, H, W, cin, cout, d = CONV_CASES[i]
    relu = i % 2 == 0
    x, w, b = sm.operands(kind, B, H, W, cin, cout, seed=100 * i + len(kind))
    want = sm.conv64(x, w, b, d, relu)
    ips = cin + 64
    xin = sm.plane_buffer(x, ips, 3 * ips).cuda()                # unread channels between the planes: bf16 NaN
    ops = cout + 32
    raw, out = _guarded((B, H, W, 3 * ops), torch.bfloat16)
    wp, bias = pack_conv3x3_split(w).cuda(), b.float().cuda()
    _conv(kind=L.DC_KIND_CONV3X3, epilogue=L.DC_EPI_STORE, relu=int(relu), B=B, H=H, W=W, Cin=cin, Cout=cout, dilation=d,
          in_=xin.data_ptr(), in_stride=3 * ips, weight=wp.data_ptr(), bias=bias.data_ptr(), out=out.data_ptr(),
          out_stride=3 * ops, out_offset=16, planes=3, in_plane_stride=ips, out_plane_stride=ops)
    case = f"split conv {cin}->{cout} d{d} {B}x{H}x{W} {kind} relu={relu}"
    _assert_planes(out, want, ops, 16, case)
    _check_guards(raw, case)


POOL_CASES = [(1, 16, 32, 64, 1), (2, 24, 40, 128, 2), (1, 16, 16, 256, 4), (1, 8, 16, 512, 8), (2, 10, 18, 64, 1)]


@pytest.mark.parametrize("i", range(len(POOL_CASES)))
@pytest.mark.parametrize("kind", sm.KINDS)
def test_split_conv_pool_exact(cuda_device, i, kind):
    """STORE_POOL: the pooled planes are the split of the fp32 max of the window, into the [up | enc] layout of the
    forward's skip buffers (encoder half at channel offset C, plane stride 2C)."""
    from unet_dc_segmentation_b200.model import pack_conv3x3_split
    L = _L()
    B, H, W, c, d = POOL_CASES[i]
    x, w, b = sm.operands(kind, B, H, W, c, c, seed=7 + i)
    want = sm.conv64(x, w, b, d)
    xin = sm.plane_buffer(x, c, 3 * c).cuda()
    raw, out = _guarded((B, H, W, 6 * c), torch.bfloat16)
    praw, pooled = _guarded((B, H // 2, W // 2, 3 * c + 64), torch.bfloat16)
    wp, bias = pack_conv3x3_split(w).cuda(), b.float().cuda()
    _conv(kind=L.DC_KIND_CONV3X3, epilogue=L.DC_EPI_STORE_POOL, relu=1, B=B, H=H, W=W, Cin=c, Cout=c, dilation=d,
          in_=xin.data_ptr(), in_stride=3 * c, weight=wp.data_ptr(), bias=bias.data_ptr(), out=out.data_ptr(),
          out_stride=6 * c, out_offset=c, pool_out=pooled.data_ptr(), pool_stride=3 * c + 64, planes=3,
          in_plane_stride=c, out_plane_stride=2 * c, pool_plane_stride=c)
    case = f"split pool {c} d{d} {B}x{H}x{W} {kind}"
    _assert_planes(out, want, 2 * c, c, case)
    _check_guards(raw, case)
    _assert_planes(pooled, sm.pool_split(want), c, 0, f"{case}: pooled")
    _check_guards(praw, f"{case}: pooled")


@pytest.mark.parametrize("c", [64, 128, 256, 512])
@pytest.mark.parametrize("kind", sm.KINDS)
def test_split_upscatter_exact(cuda_device, c, kind):
    """The transposed conv (GEMM N = 4 Cout) into the up half of a [up | enc] skip buffer, per plane."""
    from unet_dc_segmentation_b200.model import pack_upconv_split
    L = _L()
    B, H, W = 2, 6, 10
    x, w, b = sm.operands(kind, B, H, W, 2 * c, c, seed=c, upconv=True)
    want = sm.upconv64(x, w, b)
    xin = sm.plane_buffer(x, 2 * c, 6 * c).cuda()
    raw, out = _guarded((B, 2 * H, 2 * W, 6 * c), torch.bfloat16)
    wp, bias = pack_upconv_split(w).cuda(), b.float().cuda()
    _conv(kind=L.DC_KIND_UPCONV2, epilogue=L.DC_EPI_UPSCATTER, relu=0, B=B, H=H, W=W, Cin=2 * c, Cout=c, dilation=1,
          in_=xin.data_ptr(), in_stride=6 * c, weight=wp.data_ptr(), bias=bias.data_ptr(), out=out.data_ptr(),
          out_stride=6 * c, out_offset=0, planes=3, in_plane_stride=2 * c, out_plane_stride=2 * c)
    case = f"split upconv {2 * c}->{c} {kind}"
    _assert_planes(out, want, 2 * c, 0, case)
    _check_guards(raw, case)


@pytest.mark.parametrize("kind", sm.KINDS)
@pytest.mark.parametrize("cin,d", [(64, 1), (128, 1), (64, 3)])
def test_split_head_exact(cuda_device, kind, cin, d):
    """HEAD: fp32 accumulator + bias + ReLU -> 1x1 conv -> sigmoid; the logits are exact on both sides."""
    from unet_dc_segmentation_b200.model import pack_conv3x3_split
    L = _L()
    B, H, W = 2, 16, 24
    x, w, b = sm.operands(kind, B, H, W, cin, 64, seed=cin + d)
    feat = sm.conv64(x, w, b, d)
    g = torch.Generator().manual_seed(3)
    k = torch.zeros(64, dtype=torch.float64)               # four non-zeros: the head's fp32 sum of 18-bit features is exact
    k[torch.randperm(64, generator=g)[:4]] = torch.tensor([3.0, -2.0, 1.0, -4.0], dtype=torch.float64)
    raw = feat @ k
    s = 6
    while float(raw.std()) / 2 ** s > 2.5:
        s += 1
    hw, hb = k / 2 ** s, float(torch.round(-raw.mean() / 2 ** s * 64) / 64)
    logits = feat @ hw + hb
    xin = sm.plane_buffer(x, cin + 64, 3 * cin + 192).cuda()
    wp, bias, hwd = pack_conv3x3_split(w).cuda(), b.float().cuda(), hw.float().cuda()
    praw, prob = _guarded((B, H, W), torch.float32)
    mraw, mask = _guarded((B, H, W), torch.uint8)
    _conv(kind=L.DC_KIND_CONV3X3, epilogue=L.DC_EPI_HEAD, relu=1, B=B, H=H, W=W, Cin=cin, Cout=64, dilation=d,
          in_=xin.data_ptr(), in_stride=3 * cin + 192, weight=wp.data_ptr(), bias=bias.data_ptr(), head_w=hwd.data_ptr(),
          head_b=hb, thresh=THRESH, prob_out=prob.data_ptr(), mask_out=mask.data_ptr(), planes=3,
          in_plane_stride=cin + 64)
    case = f"split head {cin} d{d} {kind}"
    en.assert_probs(prob, mask, logits, THRESH, case)
    _check_guards(praw, case)
    _check_guards(mraw, case)


def test_split_arguments_are_checked(cuda_device):
    L = _L()
    lib = L.load()
    x = torch.zeros(1, 8, 8, 192, dtype=torch.bfloat16, device="cuda")
    w = torch.zeros(64, 27 * 64, dtype=torch.bfloat16, device="cuda")
    b = torch.zeros(64, device="cuda")
    base = dict(kind=L.DC_KIND_CONV3X3, epilogue=L.DC_EPI_STORE, relu=1, B=1, H=8, W=8, Cin=64, Cout=64, dilation=1,
                in_=x.data_ptr(), in_stride=192, weight=w.data_ptr(), bias=b.data_ptr(), out=x.data_ptr(), out_stride=192,
                planes=3, in_plane_stride=64, out_plane_stride=64)
    for bad in (dict(planes=2), dict(in_plane_stride=72), dict(out_plane_stride=80), dict(in_plane_stride=60)):
        a = L.ConvArgs()
        for k, v in {**base, **bad}.items():
            setattr(a, k, v)
        assert lib.dc_conv_tc(ctypes.byref(a), L.stream_ptr()) == L.DC_EINVAL, bad


# ----------------------------------------------------------------------------- whole forward, exact tier

def _wide_input(B, H, W, cin, seed):
    """Integer frames in [0, 4096): activations need up to 13 bits, so the mid plane is in use."""
    return torch.randint(0, 4096, (B, cin, H, W), generator=torch.Generator().manual_seed(seed)).double()


def _wide_net(cin, cout, dil, seed):
    """exact_net's integer network with out_conv recalibrated for 12-bit input frames."""
    sd = en.exact_state_dict(cin, cout, dil, seed)
    k = torch.randint(-4, 5, (cout, 64), generator=torch.Generator().manual_seed(seed + 9)).double()
    sd["out_conv.weight"] = torch.zeros(cout, 64, 1, 1)
    sd["out_conv.bias"] = torch.zeros(cout)
    feat = en.forward64(sd, _wide_input(1, 64, 64, cin, 77 + seed), dil)["dec1.3"]
    raw = torch.einsum("oc,bchw->bohw", k, feat)
    s = 6
    while float(raw.std()) / 2 ** s > 2.5:
        s += 1
    sd["out_conv.weight"] = (k / 2 ** s).float().reshape(cout, 64, 1, 1)
    sd["out_conv.bias"] = (torch.round(-raw.mean((0, 2, 3)) / 2 ** s * 64) / 64).float()
    return sd


def _model(cls, sd, cin=3, cout=1):
    m = cls(cin, cout)
    m.load_state_dict(sd)
    m = m.cuda().eval()
    m.precision = "fp32"
    return m


def _fill_workspace(m, B, H, W):
    m.packed().workspace_for(B, H, W).fill_(0xFF)


NETS = {"unetdc": (3, 1, en.DEFAULT_DIL, 0), "unet": (3, 1, (1, 1, 1, 1, 1), 0), "unetdc_1_2": (1, 2, en.DEFAULT_DIL, 2)}


@pytest.mark.parametrize("name", sorted(NETS))
@pytest.mark.parametrize("shape", [(2, 48, 80), (1, 64, 128), (1, 16, 16)])
def test_forward_exact(cuda_device, name, shape):
    from unet_dc_segmentation_b200.model import UNet, UNetDC
    cin, cout, dil, seed = NETS[name]
    sd = _wide_net(cin, cout, dil, seed)
    m = _model(UNet if name == "unet" else UNetDC, sd, cin, cout)
    B, H, W = shape
    x = _wide_input(B, H, W, cin, 5 + H)
    bounds = {}
    logits = en.forward64(sd, x, dil, bounds=bounds)["logits"]
    assert max(bounds.values()) <= en.BOUND
    _fill_workspace(m, B, H, W)
    prob = m(x.float().cuda())
    en.assert_probs(prob, None, logits, THRESH, f"fp32 forward {name} {shape}")
    assert m.num_launches() == 23 + (cout != 1)


def test_forward_u8_kinds_match_fp32_input(cuda_device):
    """u8 grey [B,H,W] and u8 HWC [B,H,W,3] enter as u8 / 255 in IEEE fp32: the same bits as the fp32 NCHW entry fed
    torch's u8 / 255 (with the exact 8-bit integer network the fp32 entry is held to float64 above)."""
    from unet_dc_segmentation_b200.model import UNetDC
    sd = _wide_net(3, 1, en.DEFAULT_DIL, 0)
    m = _model(UNetDC, sd)
    hwc = en.frames(2, 48, 64, 3).cuda()
    gray = en.gray_frames(2, 48, 64, 4).cuda()
    for u8, x in ((hwc, hwc.permute(0, 3, 1, 2)), (gray, gray[:, None].expand(2, 3, 48, 64))):
        xf = torch.from_numpy(x.cpu().numpy().astype(np.float32) / np.float32(255)).cuda()    # IEEE division
        _fill_workspace(m, 2, 48, 64)
        mask, prob = m.predict_u8(u8, THRESH, return_prob=True)
        _fill_workspace(m, 2, 48, 64)
        want = m(xf.contiguous())
        assert torch.equal(prob, want) and torch.equal(mask, (want[:, 0] > THRESH).to(torch.uint8))


def test_fused_blobs_with_fp32_are_rejected(cuda_device):
    """dc_model_create refuses any fused or parity blob together with DC_PRECISION_FP32."""
    L = _L()
    lib = L.load()
    buf = torch.zeros(1024, device="cuda")
    desc = L.ModelDesc()
    for i in range(L.DC_NUM_LAYERS):
        desc.weight[i] = desc.bias[i] = buf.data_ptr()
    for i, d in enumerate(en.DEFAULT_DIL):
        desc.dilations[i] = d
    desc.base_channels = 64
    desc.precision = L.DC_PRECISION_FP32
    h = ctypes.c_void_p()
    L.check(lib.dc_model_create(ctypes.byref(h), 0, ctypes.byref(desc)))
    lib.dc_model_destroy(h)
    for field, idx in (("fused_weight1", None), ("par_weight", 0), ("par_weight", 1), ("fused_wide_x", 1)):
        if idx is None:
            setattr(desc, field, buf.data_ptr())
        else:
            getattr(desc, field)[idx] = buf.data_ptr()
        assert lib.dc_model_create(ctypes.byref(h), 0, ctypes.byref(desc)) == L.DC_EINVAL, field
        assert b"DC_PRECISION_FP32" in lib.dc_last_error()
        if idx is None:
            setattr(desc, field, None)
        else:
            getattr(desc, field)[idx] = None


def test_precision_switch_repacks(cuda_device):
    from unet_dc_segmentation_b200.model import UNetDC
    m = UNetDC().cuda().eval()
    x = torch.rand(1, 3, 32, 32, device="cuda")
    a = m(x)
    assert m.num_launches() == 18
    m.precision = "fp32"
    b = m(x)
    assert m.num_launches() == 23 and m.packed().precision == "fp32"
    m.precision = "bf16"
    assert torch.equal(m(x), a) and m.num_launches() == 18
    assert not torch.equal(a, b)
    m.precision = "fp16"
    with pytest.raises(ValueError):
        m(x)


# ----------------------------------------------------------------------------- tolerance tier

def _calibrated():
    from unet_dc_segmentation_b200.synth import calibrated_state_dict
    return calibrated_state_dict(seed=0, calib_size=256, n_calib=1, fit_head=True)


def _frames(B, size, base):
    from unet_dc_segmentation_b200.synth import synthetic_image
    return torch.from_numpy(np.stack([synthetic_image(size, base + i) for i in range(B)]))


# The 1e-4 target was not met.  Measured on a B200: max |p - p64| 1.55e-4 at 4 x 256^2, 3.6e-4 on one 512^2 frame and
# 1.84e-4 on one 1024^2 frame, against 2.9e-6 / 3.8e-6 / 3.4e-6 for the CPU fp32 network (profiles/r04_fp32_forward.md);
# the bar leaves room above the largest of these, since the value moves with the frames.  Cause: the same
# arithmetic evaluated exactly (fp32 planes, the six terms, exact sums, fp32 stores) reaches 7.1e-7 at 2 x 256^2, 6.8e-7
# with all nine terms, so neither the dropped terms nor the plane storage account for it.  What remains is measured:
# tcgen05 truncates toward zero at every K = 16 step (tests/tc_accum_model.py), and tests/test_gpu_tc_accum.py shows
# the whole fp32 forward is that model, layer by layer and bit for bit (9.7e-5 at 64^2 against 4.9e-7 with exact sums).
# At 512^2 and 1024^2 tests/test_gpu_tc_accum_fullsize.py shows it too: every layer of the chain equals the model at
# sampled sites (every tile, the borders, interior samples), and predict_u8 equals the chain, so the errors quoted
# above are the model's, not a kernel's.
P_TOL = 1e-3


@pytest.mark.parametrize("B,size", [(4, 256), (1, 512)])
def test_fp32_matches_float64(cuda_device, B, size):
    """Max |p - p64| <= P_TOL against the float64 network on the same fp32 input; masks differ only within P_TOL of
    the threshold.  The CPU fp32 network's own error and the bf16 forward's are printed beside it."""
    import oracle
    from unet_dc_segmentation_b200.model import UNetDC
    sd = _calibrated()
    m = _model(UNetDC, sd)
    u8 = _frames(B, size, 50)
    x32 = torch.from_numpy(u8.numpy().astype(np.float32) / np.float32(255))[:, None].expand(B, 3, size, size).contiguous()
    p64 = sm.network(sd, x32)
    p32 = oracle.unetdc_forward(sd, x32)[:, 0].double()
    mask, prob = m.predict_u8(u8.cuda(), THRESH, return_prob=True)
    p = prob[:, 0].double().cpu()
    err, cpu_err = float((p - p64).abs().max()), float((p32 - p64).abs().max())
    m.precision = "bf16"
    bf16_err = float((m.predict_u8(u8.cuda(), THRESH, return_prob=True)[1][:, 0].double().cpu() - p64).abs().max())
    print(f"{B}x{size}^2: max |dp| vs float64: fp32 mode {err:.3e} (mean {float((p - p64).abs().mean()):.3e}), "
          f"CPU fp32 network {cpu_err:.3e}, bf16 mode {bf16_err:.3e}")
    assert err <= P_TOL, f"max |dp| {err}"
    bad = (mask.cpu() != (p64 > THRESH).to(torch.uint8)) & ((p64 - THRESH).abs() > P_TOL)
    assert not bool(bad.any()), f"{int(bad.sum())} mask pixels differ away from the threshold"


def test_fp32_envelope_past_2_31_elements(cuda_device):
    """11 x 1024^2: the three-plane level-0 activations hold 11 * 2^20 * 192 > 2^31 elements; the last frame of the
    batch gives the bits it gives alone."""
    from unet_dc_segmentation_b200.model import UNetDC
    m = _model(UNetDC, _calibrated())
    u8 = _frames(11, 1024, 300).cuda()
    mask, prob = m.predict_u8(u8, THRESH, return_prob=True)
    last = prob[-1].clone()
    m.packed().workspace = None
    torch.cuda.empty_cache()
    mask1, prob1 = m.predict_u8(u8[-1:].contiguous(), THRESH, return_prob=True)
    assert torch.equal(last, prob1[0]) and torch.equal(mask[-1], mask1[0])


def test_pipeline_graph_replay_fp32(cuda_device):
    """DropletPipeline follows the model's precision; a replayed CUDA graph gives the bits of the eager pass."""
    from unet_dc_segmentation_b200 import DropletPipeline
    from unet_dc_segmentation_b200.model import UNetDC
    m = _model(UNetDC, _calibrated())
    frames = _frames(4, 128, 700).numpy()
    pipe = DropletPipeline(m, background_radius=50, prob_thresh=THRESH, use_graphs=True)
    batches = [torch.from_numpy(frames)] * 3
    outs = [masks.copy() for masks, _ in pipe.run_host_pipelined(batches)]
    assert np.array_equal(outs[0], outs[1]) and np.array_equal(outs[0], outs[2])
    eager = DropletPipeline(m, background_radius=50, prob_thresh=THRESH).run_device(torch.from_numpy(frames).cuda())
    assert np.array_equal(eager.masks.cpu().numpy(), outs[0])
    m.precision = "bf16"
    bf = DropletPipeline(m, background_radius=50, prob_thresh=THRESH).run_device(torch.from_numpy(frames).cuda())
    print(f"pipeline 4 x 128^2: {int((bf.masks.cpu().numpy() != outs[0]).sum())} mask pixels differ bf16 vs fp32")


def test_cli_precision_fp32(cuda_device, tmp_path):
    """cli --precision fp32 writes the masks and droplet tables DropletPipeline gives in fp32 mode."""
    import cv2
    import pandas as pd
    from PIL import Image
    from unet_dc_segmentation_b200 import DropletPipeline, cli
    from unet_dc_segmentation_b200.synth import synthetic_image
    (tmp_path / "in").mkdir()
    frames = [synthetic_image(96, 800 + i, n_droplets=10) for i in range(3)]
    for i, f in enumerate(frames):
        Image.fromarray(f).save(tmp_path / "in" / f"frame{i}.png")
    torch.save(_calibrated(), tmp_path / "ckpt.pth")
    out = tmp_path / "out"
    assert cli.main(["--img_dir", str(tmp_path / "in"), "--ckpt_path", str(tmp_path / "ckpt.pth"), "--out_dir", str(out),
                     "--batch", "2", "--img_size", "96", "--skip_histogram", "--skip_excel", "--precision", "fp32"]) == 0
    m = cli.load_model(tmp_path / "ckpt.pth")
    m.precision = "fp32"
    res = DropletPipeline(m, 50, THRESH, 1, None, img_size=96).run_device(torch.from_numpy(np.stack(frames)).cuda())
    tables = res.tables.to_host()
    for i in range(3):
        got = cv2.imread(str(out / "predicted_masks" / f"frame{i}_pred.png"), cv2.IMREAD_GRAYSCALE)
        np.testing.assert_array_equal(got // 255, res.masks[i].cpu().numpy(), err_msg=f"frame{i} mask")
        df = pd.read_csv(out / f"frame{i}_droplets.csv", float_precision="round_trip")
        assert len(df) == len(tables[i]["label"])
        np.testing.assert_array_equal(df["area"].to_numpy(), np.asarray(tables[i]["area"]))
