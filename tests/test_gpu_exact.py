"""GPU: the tensor-core layers and the whole forward held BIT FOR BIT to a float64 reference, on integer-valued operands
(tests/exact_net.py).  Every operand is an integer or a multiple of 1/4 and sum |w x| <= 2^20, so the fp32 accumulation is
exact in any order and the bf16 store (round to nearest even) of each layer must equal ``float64 -> float32 -> bf16``:
a dropped MMA chunk, a wrong border-class bias or a store that rounds toward zero is a mismatch, not noise inside a
tolerance.  Every schedule of the forward must give the same bits.

Around every launch: outputs are views of larger buffers whose guard bytes and unwritten channels hold a sentinel that
must survive; the input channels a layer does not read (and the skip channels outside its slice) hold bf16 NaN; the
forward's cached workspace is filled with 0xFF (bf16 NaN) before every call."""
import ctypes
import functools

import pytest
import torch
from hypothesis import HealthCheck, given, settings
from hypothesis import strategies as st

import exact_net as en

pytestmark = pytest.mark.gpu

GUARD, SENT, SENT16 = en.GUARD, en.SENT, en.SENT16
THRESH = 0.3
FAMILIES = ("auto", "generic")

CONV_CASES = [
    (1, 8, 16, 64, 64, 1), (2, 16, 32, 64, 64, 1), (1, 24, 40, 64, 128, 2), (2, 16, 16, 128, 128, 2),
    (1, 32, 48, 128, 256, 4), (1, 16, 16, 256, 512, 8), (2, 8, 8, 512, 1024, 16), (1, 16, 32, 1024, 512, 1),
    (3, 40, 24, 192, 64, 3), (2, 48, 24, 128, 64, 1), (1, 40, 40, 64, 128, 2), (1, 32, 16, 64, 64, 4),
    (2, 16, 8, 64, 64, 1), (1, 48, 40, 256, 512, 1), (3, 16, 24, 128, 256, 4), (1, 16, 8, 512, 256, 2),
    (1, 64, 64, 512, 1024, 16), (1, 48, 80, 1024, 1024, 16), (2, 32, 48, 256, 512, 8), (1, 128, 128, 512, 512, 8),
]                                              # the shapes of test_gpu_conv.CONV_CASES
UPFUSED_CASES = [(1, 16, 8), (2, 16, 8), (1, 40, 24), (3, 24, 20), (2, 64, 64), (1, 8, 8)]
WIDE_CASES = [(128, 1, 16, 8), (128, 2, 24, 20), (128, 1, 40, 24), (256, 1, 16, 8), (256, 2, 24, 12), (256, 1, 8, 8),
              (512, 1, 16, 8), (512, 2, 16, 16), (512, 1, 24, 20)]
PARITY_CASES = [(1, 32, 16), (2, 32, 16), (1, 80, 48), (3, 48, 40), (2, 128, 128), (1, 16, 16), (1, 2, 2)]


def _lib():
    from unet_dc_segmentation_b200 import _lib as L
    return L


family = en.family


# ----------------------------------------------------------------------------- buffers

_guarded, _check_guards, _check_outside = en.guarded, en.check_guards, en.check_outside


def _nan_padded(x64, width, off=0):
    """bf16 NHWC [..., width] on the device holding x64 at channels [off, off + C) and NaN everywhere else."""
    buf = torch.full(tuple(x64.shape[:-1]) + (width,), float("nan"), dtype=torch.bfloat16)
    buf[..., off:off + x64.shape[-1]] = en.bf16(x64)
    return buf.cuda()


_conv = en.conv_tc


def _head_weights(feat64, seed):
    """Dyadic out_conv weights k / 2^s (k in [-4, 4]) and bias for a [B,H,W,64] feature map: logits of a few units."""
    g = torch.Generator().manual_seed(seed)
    k = torch.randint(-4, 5, (64,), generator=g).double()
    raw = feat64 @ k
    s = 6
    while float(raw.std()) / 2 ** s > 2.5:
        s += 1
    hb = float(torch.round(-raw.mean() / 2 ** s * 64) / 64)
    return k / 2 ** s, hb


# ----------------------------------------------------------------------------- single layers

@functools.lru_cache(maxsize=4)
def _conv_ref(B, H, W, cin, cout, d, kind, seed):
    """Operands and the pre-activation float64 output of one layer (computed once per case)."""
    x = en.acts((B, H, W, cin), seed)
    w = en.conv_weight(cout, cin, kind, seed + 1)
    b = en.biases(cout, seed + 2)
    en.assert_bound(lambda *o: en.conv3x3_ref(*o, d, False), x, w, b)
    return x, w, b, en.conv3x3_ref(x, w, b, d, relu=False)


def _store_case(B, H, W, cin, cout, d, kind, relu, case, seed=0, weight=None):
    from unet_dc_segmentation_b200.model import pack_conv3x3
    L = _lib()
    x64, w64, b64, pre = _conv_ref(B, H, W, cin, cout, d, kind, seed)
    want = pre.clamp(min=0) if relu else pre
    x = _nan_padded(x64, cin + 64)
    wp = pack_conv3x3(w64).cuda() if weight is None else weight
    raw, out = _guarded((B, H, W, cout + 32), torch.bfloat16)
    bias = b64.float().cuda()
    _conv(kind=L.DC_KIND_CONV3X3, epilogue=L.DC_EPI_STORE, relu=int(relu), B=B, H=H, W=W, Cin=cin, Cout=cout, dilation=d,
          in_=x.data_ptr(), in_stride=cin + 64, weight=wp.data_ptr(), bias=bias.data_ptr(), out=out.data_ptr(),
          out_stride=cout + 32, out_offset=16)
    en.assert_exact(out[..., 16:16 + cout], want, case)
    _check_outside(raw, out, 16, cout, case)


@pytest.mark.parametrize("i", range(len(CONV_CASES)))
def test_conv_store_exact(cuda_device, family, i):
    """Plain store, ReLU on and off, into a channel slice, under every kernel family; dense weights on even cases
    (long K, large sums, bf16 rounding of the output), sparse +-1 on odd ones."""
    B, H, W, cin, cout, d = CONV_CASES[i]
    kind = "dense" if i % 2 == 0 else "sparse"
    for fam in FAMILIES:
        family(fam)
        for relu in (True, False):
            _store_case(B, H, W, cin, cout, d, kind, relu,
                        f"conv {cin}->{cout} d{d} {B}x{H}x{W} {kind} relu={relu} family={fam}")


COMMON = dict(deadline=None, suppress_health_check=[HealthCheck.function_scoped_fixture, HealthCheck.too_slow],
              derandomize=True)


@settings(max_examples=40, **COMMON)
@given(B=st.integers(1, 3), H=st.integers(1, 40), W=st.integers(1, 40),
       cin=st.sampled_from([64, 128, 192, 256, 320, 512, 1024]), cout=st.sampled_from([64, 128, 192, 256, 512, 1024]),
       d=st.integers(1, 20), relu=st.booleans(), kind=st.sampled_from(["dense", "sparse"]), seed=st.integers(0, 10 ** 6))
def test_conv_store_exact_random(cuda_device, B, H, W, cin, cout, d, relu, kind, seed):
    _store_case(B, H, W, cin, cout, d, kind, relu, f"conv {cin}->{cout} d{d} {B}x{H}x{W} {kind} relu={relu} seed={seed}",
                seed=seed)


def _pool_case(B, H, W, cin, c, d, kind, case, par=False):
    from unet_dc_segmentation_b200.model import pack_conv3x3, pack_par3x3
    L = _lib()
    x64, w64, b64, pre = _conv_ref(B, H, W, cin, c, d, kind, 7)
    want = pre.clamp(min=0)
    x = _nan_padded(x64, cin + 64)
    raw, out = _guarded((B, H, W, c + 32), torch.bfloat16)
    praw, pooled = _guarded((B, H // 2, W // 2, c), torch.bfloat16)
    wp, bias = pack_conv3x3(w64).cuda(), b64.float().cuda()
    wpar = pack_par3x3(w64.float()).cuda() if par else None
    _conv(kind=L.DC_KIND_CONV3X3, epilogue=L.DC_EPI_STORE_POOL, relu=1, B=B, H=H, W=W, Cin=cin, Cout=c, dilation=d,
          in_=x.data_ptr(), in_stride=cin + 64, weight=wp.data_ptr(), bias=bias.data_ptr(), out=out.data_ptr(),
          out_stride=c + 32, out_offset=16, pool_out=pooled.data_ptr(), pool_stride=c,
          weight_par=wpar.data_ptr() if par else None)
    en.assert_exact(out[..., 16:16 + c], want, f"{case}: full-res output")
    _check_outside(raw, out, 16, c, case)
    want_pool = torch.nn.functional.max_pool2d(want.permute(0, 3, 1, 2), 2).permute(0, 2, 3, 1)
    en.assert_exact(pooled, want_pool, f"{case}: pooled output")
    _check_guards(praw, f"{case}: pooled output")


def _head_case(B, H, W, cin, d, case, par=False):
    from unet_dc_segmentation_b200.model import pack_conv3x3, pack_par3x3
    L = _lib()
    x64, w64, b64, pre = _conv_ref(B, H, W, cin, 64, d, "sparse", 11)
    feat = pre.clamp(min=0)
    hw, hb = _head_weights(feat, 3)
    logits = feat @ hw + hb
    x = _nan_padded(x64, cin + 64)
    wp, bias = pack_conv3x3(w64).cuda(), b64.float().cuda()
    wpar = pack_par3x3(w64.float()).cuda() if par else None
    hwd = hw.float().cuda()
    praw, prob = _guarded((B, H, W), torch.float32)
    mraw, mask = _guarded((B, H, W), torch.uint8)
    _conv(kind=L.DC_KIND_CONV3X3, epilogue=L.DC_EPI_HEAD, relu=1, B=B, H=H, W=W, Cin=cin, Cout=64, dilation=d,
          in_=x.data_ptr(), in_stride=cin + 64, weight=wp.data_ptr(), bias=bias.data_ptr(), head_w=hwd.data_ptr(), head_b=hb,
          thresh=THRESH, prob_out=prob.data_ptr(), mask_out=mask.data_ptr(), weight_par=wpar.data_ptr() if par else None)
    en.assert_probs(prob, mask, logits, THRESH, case)
    _check_guards(praw, f"{case}: prob")
    _check_guards(mraw, f"{case}: mask")


@pytest.mark.parametrize("fam", FAMILIES)
def test_pool_and_head_epilogues_exact(cuda_device, family, fam):
    """256 -> 64 at dilation 1 is a single-CTA halo layer (conv_halo_kernel) in AUTO."""
    family(fam)
    for B, H, W, cin, c, d in [(1, 16, 32, 64, 64, 1), (2, 24, 48, 128, 128, 2), (1, 16, 16, 256, 256, 4),
                               (1, 18, 34, 64, 64, 1), (2, 24, 32, 256, 64, 1)]:
        _pool_case(B, H, W, cin, c, d, "dense" if cin > 64 else "sparse", f"pool {cin}->{c} d{d} {B}x{H}x{W} family={fam}")
    for B, H, W, cin, d in [(2, 24, 32, 64, 1), (1, 17, 29, 64, 1), (2, 16, 8, 64, 2), (1, 24, 40, 256, 1)]:
        _head_case(B, H, W, cin, d, f"head {cin}->64 {B}x{H}x{W} d{d} family={fam}")


@pytest.mark.parametrize("B,H,W", PARITY_CASES)
def test_parity_class_kernel_exact(cuda_device, B, H, W):
    """conv_par2_kernel (weight_par): store without ReLU into a slice, store + pool, and the head."""
    from unet_dc_segmentation_b200.model import pack_conv3x3, pack_par3x3
    L = _lib()
    case = f"parity {B}x{H}x{W}"
    x64, w64, b64, pre = _conv_ref(B, H, W, 64, 64, 1, "dense", 5)
    x = _nan_padded(x64, 128)
    raw, out = _guarded((B, H, W, 96), torch.bfloat16)
    wp, bias, wpar = pack_conv3x3(w64).cuda(), b64.float().cuda(), pack_par3x3(w64.float()).cuda()
    _conv(kind=L.DC_KIND_CONV3X3, epilogue=L.DC_EPI_STORE, relu=0, B=B, H=H, W=W, Cin=64, Cout=64, dilation=1,
          in_=x.data_ptr(), in_stride=128, weight=wp.data_ptr(), bias=bias.data_ptr(), out=out.data_ptr(), out_stride=96,
          out_offset=16, weight_par=wpar.data_ptr())
    en.assert_exact(out[..., 16:80], pre, f"{case}: store")
    _check_outside(raw, out, 16, 64, case)
    _pool_case(B, H, W, 64, 64, 1, "dense", f"{case}: pool", par=True)
    _head_case(B, H, W, 64, 1, f"{case}: head", par=True)


@pytest.mark.parametrize("fam", FAMILIES)
@pytest.mark.parametrize("B,H,W,cin,cout", [(1, 8, 16, 128, 64), (2, 12, 20, 256, 128), (1, 8, 8, 1024, 512),
                                            (3, 5, 7, 128, 64)])
def test_upconv_exact(cuda_device, family, fam, B, H, W, cin, cout):
    """The transposed conv (DC_EPI_UPSCATTER) into a channel slice of a wider buffer."""
    from unet_dc_segmentation_b200.model import pack_upconv
    L = _lib()
    family(fam)
    case = f"upconv {cin}->{cout} {B}x{H}x{W} family={fam}"
    x64 = en.acts((B, H, W, cin), cin + H)
    w64 = en.upconv_weight(cin, cout, "dense", cout + W)
    b64 = en.biases(cout, B)
    en.assert_bound(en.upconv_ref, x64, w64, b64)
    x = _nan_padded(x64, cin + 64)
    raw, out = _guarded((B, 2 * H, 2 * W, cout + 32), torch.bfloat16)
    wp, bias = pack_upconv(w64).cuda(), b64.float().cuda()
    _conv(kind=L.DC_KIND_UPCONV2, epilogue=L.DC_EPI_UPSCATTER, relu=0, B=B, H=H, W=W, Cin=cin, Cout=cout, dilation=1,
          in_=x.data_ptr(), in_stride=cin + 64, weight=wp.data_ptr(), bias=bias.data_ptr(), out=out.data_ptr(),
          out_stride=cout + 32, out_offset=16)
    en.assert_exact(out[..., 16:16 + cout], en.upconv_ref(x64, w64, b64), case)
    _check_outside(raw, out, 16, cout, case)


def _upfused_case(C, B, H, W, kind, relu, case, bias9_edit=None):
    """dc_conv_upfused on integer operands against the unfused float64 chain.  x is read at channels [0, 2C) of a
    2C + 64 wide buffer, skip at [64, 64 + C) of a C + 128 wide one; everything else is NaN."""
    from unet_dc_segmentation_b200.model import compose_upconv, pack_upfused, pack_upfused_wide
    L = _lib()
    lib = L.load()
    wu, bu, wd, bd = en.upfused_operands(C, 100 + C + H, kind)
    x64, s64 = en.acts((B, H, W, 2 * C), C + W), en.acts((B, 2 * H, 2 * W, C), C + B)
    en.assert_bound(lambda *o: en.upfused_ref(*o, relu=False), x64, s64, wu, bu, wd, bd)
    want = en.upfused_ref(x64, s64, wu, bu, wd, bd, relu)
    comp, skipw, bias9 = compose_upconv(wu.float(), bu.float(), wd.float(), bd.float())
    if bias9_edit is not None:
        bias9 = bias9.clone()
        bias9[bias9_edit] += 1.0
    ws = None
    if C == 64:
        wx = pack_upfused(comp, skipw).cuda()
    else:
        wx, ws = (t.cuda() for t in pack_upfused_wide(comp, skipw))
    x = _nan_padded(x64, 2 * C + 64)
    skip = _nan_padded(s64, C + 128, off=64)
    raw, out = _guarded((B, 2 * H, 2 * W, C + 32), torch.bfloat16)
    b9 = bias9.cuda()
    a = L.UpfuseArgs()
    a.B, a.H, a.W, a.channels = B, H, W, C
    a.x, a.x_stride = x.data_ptr(), 2 * C + 64
    a.skip, a.skip_stride = skip.data_ptr() + 2 * 64, C + 128
    a.weight, a.bias9, a.relu = wx.data_ptr(), b9.data_ptr(), int(relu)
    if ws is not None:
        a.weight_skip = ws.data_ptr()
    a.out, a.out_stride, a.out_offset = out.data_ptr(), C + 32, 16
    L.check(lib.dc_conv_upfused(ctypes.byref(a), L.stream_ptr()))
    torch.cuda.synchronize()
    en.assert_exact(out[..., 16:16 + C], want, case)
    _check_outside(raw, out, 16, C, case)


@pytest.mark.parametrize("B,H,W", UPFUSED_CASES)
def test_upfused_level1_exact(cuda_device, B, H, W):
    """conv_upfused2_kernel (C = 64)."""
    for relu, kind in ((True, "dense"), (False, "sparse")):
        _upfused_case(64, B, H, W, kind, relu, f"upfused C=64 {B}x{H}x{W} {kind} relu={relu}")


@pytest.mark.parametrize("C,B,H,W", WIDE_CASES)
def test_upfused_wide_exact(cuda_device, C, B, H, W):
    """conv_upfused_wide_kernel (C = 128 / 256 / 512)."""
    for relu, kind in ((True, "dense"), (False, "sparse")):
        _upfused_case(C, B, H, W, kind, relu, f"upfused C={C} {B}x{H}x{W} {kind} relu={relu}")


@pytest.mark.parametrize("in_kind", [0, 1, 2])
@pytest.mark.parametrize("d", [1, 2, 3])
def test_stem_exact(cuda_device, in_kind, d):
    """dc_stem for f32 NCHW, u8 grey and u8 HWC frames (u8 stem weights 255 v), into a channel slice."""
    L = _lib()
    case = f"stem in_kind={in_kind} d{d}"
    for B, H, W in [(2, 20, 36), (1, 37, 53)]:
        w64 = en.conv_weight(64, 3, "dense", d)
        b64 = en.biases(64, d + 1)
        if in_kind == 1:
            u = en.gray_frames(B, H, W, 3 + d)
            x64 = u.double()[:, None].expand(B, 3, H, W)
            dev = u.cuda()
        else:
            u = en.frames(B, H, W, 3 + d)
            x64 = u.permute(0, 3, 1, 2).double()
            dev = x64.float().contiguous().cuda() if in_kind == 0 else u.cuda()
        want = en.conv3x3_ref(x64.permute(0, 2, 3, 1), w64, b64, d, relu=True)
        wdev = (w64 * (255.0 if in_kind else 1.0)).reshape(64, 27).float().cuda()
        bias = b64.float().cuda()
        raw, out = _guarded((B, H, W, 128), torch.bfloat16)
        a = L.StemArgs(in_kind, B, H, W, 64, d, dev.data_ptr(), wdev.data_ptr(), bias.data_ptr(), out.data_ptr(), 128, 32)
        L.check(L.load().dc_stem(ctypes.byref(a), L.stream_ptr()))
        torch.cuda.synchronize()
        en.assert_exact(out[..., 32:96], want, f"{case} {B}x{H}x{W}")
        _check_outside(raw, out, 32, 64, f"{case} {B}x{H}x{W}")


def test_mutated_blobs_are_caught(cuda_device):
    """The comparison has teeth on the device: one weight of one (tap, chunk) block changed by +1 in the packed blob,
    and one border class of bias9 changed by 1, are each reported at the layer and position they touch."""
    from unet_dc_segmentation_b200.model import pack_conv3x3
    B, H, W, cin, cout, d = 2, 16, 32, 128, 64, 1
    x64, w64, b64, _ = _conv_ref(B, H, W, cin, cout, d, "sparse", 0)
    wp = pack_conv3x3(w64)
    wp[5, 8 * cin + 64 + 3] += 1.0                        # output channel 5, tap 8 (ky = kx = 2), chunk 1
    with pytest.raises(AssertionError, match=r"mutated tap 8 chunk 1: .* differ; first at \(b=\d+, y=\d+, x=\d+, c=5\)"):
        _store_case(B, H, W, cin, cout, d, "sparse", False, "mutated tap 8 chunk 1", weight=wp.cuda())
    # bias9 row 2 * 3 + 1: last output row, interior column -- the first mismatch is on row 2H - 1
    with pytest.raises(AssertionError, match=rf"mutated bias9: .* differ; first at \(b=0, y={2 * 8 - 1}, x=\d+, c=7\)"):
        _upfused_case(64, 1, 8, 8, "sparse", False, "mutated bias9", bias9_edit=(7, 7))


# ----------------------------------------------------------------------------- whole forward

SWITCHES = [(("enc1",), (2,)), (("dec1",), (3, 4)), ((), (2, 3, 4)), (("enc1", "dec1"), ())]   # test_gpu_forward


@pytest.fixture(scope="module")
def refs():
    """(network, shape) -> (state_dict, dilations, u8 HWC frames, float64 NCHW input, float64 logits), computed once."""
    nets, cache = {}, {}

    def get(name, shape):
        if name not in nets:
            nets[name] = en.net(name)
        if (name, shape) not in cache:
            sd, dil = nets[name]
            B, H, W = shape
            seed = 40 + B * H + W
            x64 = en.net_input(B, H, W, seed, en.NETS[name][0])
            u8 = en.frames(B, H, W, seed) if en.NETS[name][0] == 3 else None
            cache[(name, shape)] = (sd, dil, u8, x64, en.forward64(sd, x64, dil)["logits"])
        return cache[(name, shape)]
    return get


def _model(name, sd, dil):
    import unet_dc_segmentation_b200 as pkg
    cin, cout = en.NETS[name][:2]
    base = pkg.UNet if name == "unet" else pkg.UNetDC
    cls = base if dil == base.dilations else type(f"UNetDC_{name}", (pkg.UNetDC,), {"dilations": dil})
    m = cls(cin, cout)
    m.load_state_dict(sd)
    return m.cuda().eval()


def _forward(m, in_kind, x, B, H, W, want_prob=True, want_mask=True):
    """dc_forward with a workspace full of 0xFF (bf16 NaN) and prob / mask in guarded sentinel-filled buffers."""
    L = _lib()
    pk = m.packed()
    ws = pk.workspace_for(B, H, W)
    ws.fill_(0xFF)
    praw, prob = _guarded((B, m.out_channels, H, W), torch.float32)
    mraw, mask = _guarded((B, H, W), torch.uint8)
    L.check(L.load().dc_forward(pk.handle, in_kind, x.data_ptr(), B, H, W, THRESH,
                                prob.data_ptr() if want_prob else None, mask.data_ptr() if want_mask else None,
                                ws.data_ptr(), ws.numel(), L.stream_ptr()))
    torch.cuda.synchronize()
    _check_guards(praw, "prob")
    _check_guards(mraw, "mask")
    if not want_prob:
        assert bool((praw == SENT).all()), "prob written though not asked for"
    if not want_mask:
        assert bool((mraw == SENT).all()), "mask written though not asked for"
    return (prob.cpu() if want_prob else None), (mask.cpu() if want_mask else None)


def _schedules():
    """(label, setup(model, lib)) of every schedule: default, the switch combinations, fully unfused; then all of them
    with the per-tap kernel forced."""
    base = [("default", {})]
    base += [(f"parity={layers} fused={levels}", {"parity_layers": layers, "fuse_levels": levels}) for layers, levels in SWITCHES]
    base += [("unfused", {"fuse_level1": False, "parity_level1": False, "fuse_levels": ()})]
    return [(lbl, attrs, fam) for fam in FAMILIES for lbl, attrs in base]


def _run_schedule(m, attrs, fam, fn):
    import unet_dc_segmentation_b200 as pkg
    L = _lib()
    lib = L.load()
    codes = {"auto": L.DC_CONV_FAMILY_AUTO, "generic": L.DC_CONV_FAMILY_GENERIC}
    for k, v in attrs.items():
        setattr(m, k, v)
    try:
        L.check(lib.dc_debug_set_conv_family(codes[fam]))
        m.invalidate()
        if attrs.get("fuse_level1") is False:
            assert m.num_launches() == 22 + (m.in_channels != 3) + (m.out_channels != 1)
        return fn()
    finally:
        L.check(lib.dc_debug_set_conv_family(L.DC_CONV_FAMILY_AUTO))
        for k in attrs:
            setattr(m, k, getattr(pkg.UNetDC, k))
        m.invalidate()


@pytest.mark.parametrize("shape", en.FORWARD_SHAPES)
def test_forward_every_schedule_exact(cuda_device, refs, shape):
    """UNetDC on frames that differ within the batch: every schedule equals the float64 reference and gives the same
    bits as every other (probabilities and masks)."""
    sd, dil, u8, x64, logits = refs("unetdc", shape)
    B, H, W = shape
    m = _model("unetdc", sd, dil)
    rgb = u8.cuda()
    mu = _model("unetdc", en.u8_stem(sd), dil)
    first = None
    for lbl, attrs, fam in _schedules():
        case = f"forward {B}x{H}x{W} schedule {lbl} family={fam}"
        prob, mask = _run_schedule(mu, attrs, fam, lambda: _forward(mu, 2, rgb, B, H, W))
        en.assert_probs(prob[:, 0], mask, logits[:, 0], THRESH, case)
        if first is None:
            first = (prob, mask)
        assert torch.equal(prob, first[0]) and torch.equal(mask, first[1]), f"{case}: not bit-identical to the default"
    # the f32 entry point on the same integers gives the same bits
    prob, mask = _forward(m, 0, x64.float().contiguous().cuda(), B, H, W)
    assert torch.equal(prob, first[0]) and torch.equal(mask, first[1]), f"f32 entry {shape}: differs from u8 HWC"


@pytest.mark.parametrize("name", [n for n in en.NETS if n != "unetdc"])
def test_forward_other_networks_exact(cuda_device, refs, name):
    """UNet, the dilation sets of test_forward_other_dilation_sets and UNetDC(1,1), (4,2), (7,1): default and unfused
    schedules, equal to the float64 reference and to each other."""
    for shape in (en.TEETH_SHAPE, (2, 48, 80)):
        sd, dil, u8, x64, logits = refs(name, shape)
        B, H, W = shape
        m = _model(name, sd, dil)
        x = x64.float().contiguous().cuda()
        prob, mask = _forward(m, 0, x, B, H, W)
        en.assert_probs(prob, mask, logits, THRESH, f"{name} {shape} default")
        p2, m2 = _run_schedule(m, {"fuse_level1": False, "parity_level1": False, "fuse_levels": ()}, "auto",
                               lambda: _forward(m, 0, x, B, H, W))
        assert torch.equal(prob, p2) and torch.equal(mask, m2), f"{name} {shape}: unfused schedule differs"


def test_forward_in_kinds_exact(cuda_device, refs):
    """All three in_kinds of the (3, 1) model: f32 NCHW and u8 HWC on the same integers give the same bits; u8 grey
    frames equal the reference of the frames replicated to three channels."""
    B, H, W = 2, 48, 80
    sd, dil, u8, x64, logits = refs("unetdc", (B, H, W))
    m, mu = _model("unetdc", sd, dil), _model("unetdc", en.u8_stem(sd), dil)
    p0, m0 = _forward(m, 0, x64.float().contiguous().cuda(), B, H, W)
    p2, m2 = _forward(mu, 2, u8.cuda(), B, H, W)
    en.assert_probs(p0[:, 0], m0, logits[:, 0], THRESH, "in_kind 0")
    assert torch.equal(p0, p2) and torch.equal(m0, m2), "in_kind 2 differs from in_kind 0"
    g = en.gray_frames(B, H, W, 17)
    lg = en.forward64(sd, g.double()[:, None].expand(B, 3, H, W), dil)["logits"]
    p1, m1 = _forward(mu, 1, g.cuda(), B, H, W)
    en.assert_probs(p1[:, 0], m1, lg[:, 0], THRESH, "in_kind 1")


def test_forward_poisoned_workspace_and_outputs(cuda_device, refs):
    """A larger forward first, then smaller ones in the same workspace refilled with 0xFF: nothing read that the
    forward did not write.  dc_forward with prob only, mask only and both, in guarded buffers."""
    sd, dil = refs("unetdc", (1, 256, 256))[:2]
    mu = _model("unetdc", en.u8_stem(sd), dil)
    for shape in [(1, 256, 256), (2, 48, 80), (1, 16, 16)]:
        _, _, u8, _, logits = refs("unetdc", shape)
        B, H, W = shape
        for wp, wm in ((True, True), (True, False), (False, True)):
            prob, mask = _forward(mu, 2, u8.cuda(), B, H, W, wp, wm)
            en.assert_probs(None if prob is None else prob[:, 0], mask, logits[:, 0], THRESH,
                            f"poisoned workspace {shape} prob={wp} mask={wm}")
