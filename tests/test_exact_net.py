"""CPU: the integer networks and layer operands of tests/exact_net.py keep the fp32 arithmetic of the tensor-core path
exact, the host-side folds and packers keep it exact, the oracle's fp32 and bf16-emulation paths agree with the float64
reference on them, and every layer of every network used is visible in the output (the GPU comparisons have teeth)."""
import numpy as np
import pytest
import torch

import exact_net as en
import oracle


@pytest.fixture(scope="module")
def nets():
    return {}


def _net(nets, name):
    if name not in nets:
        nets[name] = en.net(name)
    return nets[name]


def _cases():
    out = [("unetdc", s) for s in en.FORWARD_SHAPES]
    out += [(n, en.TEETH_SHAPE) for n in en.NETS if n != "unetdc"]
    return out


@pytest.mark.parametrize("name,shape", _cases())
def test_network_invariants(nets, name, shape):
    """Every value an integer, every stored tensor <= 256 and >= 20 % non-zero, sum |w x| <= 2^20 in every layer, every
    (tap, chunk) block covered, and at least 30 % of the pixels with p in [0.02, 0.98]."""
    sd, dil = _net(nets, name)
    cin = en.NETS[name][0]
    for layer in en.CONV_LAYERS:
        assert en.blocks_covered(sd[f"{layer}.weight"]), f"{name} {layer}: a (tap, chunk) block without a weight"
    for lvl in (1, 2, 3, 4):
        assert en.blocks_covered(sd[f"upconv{lvl}.weight"], upconv=True), f"{name} upconv{lvl}"
    bounds = {}
    t = en.forward64(sd, en.net_input(*shape, 3, cin), dil, bounds)
    for k in en.STORED:
        v = t[k]
        assert torch.equal(v, v.round()), f"{name} {shape} {k}: not integer-valued"
        assert float(v.abs().max()) <= en.STORE_MAX, f"{name} {shape} {k}: max {float(v.abs().max())}"
        nz = float((v != 0).double().mean())
        assert nz >= 0.2, f"{name} {shape} {k}: only {100 * nz:.1f} % non-zero"
    for k, b in bounds.items():
        assert b <= en.BOUND, f"{name} {shape} {k}: sum |w x| = {b}"
    p = torch.sigmoid(t["logits"])
    frac = float(((p >= 0.02) & (p <= 0.98)).double().mean())
    assert frac >= 0.3, f"{name} {shape}: only {100 * frac:.1f} % of the pixels have p in [0.02, 0.98]"
    s = t["logits"] * 2 ** 12
    assert torch.equal(s, s.round()), "logits not dyadic"


def test_batchnorm_fold_is_the_identity():
    """gamma 1, mean 0, running_var float32(1 - 1e-5): model.fold_conv_bn returns the conv weights and beta bit for bit."""
    sd = en.exact_state_dict()
    for layer in en.CONV_LAYERS:
        p, idx = layer.split(".")
        w, b = en.folded(sd, layer)
        assert torch.equal(w, sd[f"{layer}.weight"].double()), layer
        assert torch.equal(b, sd[f"{p}.{int(idx) + 1}.bias"].double()), layer


def test_u8_stem_weights_are_exact():
    """The stem kernel multiplies the weights by 1.0f/255.0f and rounds to bf16: 255 * v gives v for every integer v in
    [-64, 64] and, summed over the three grey channels first, v_r + v_g + v_b."""
    v = torch.arange(-64, 65, dtype=torch.float32)
    scale = torch.tensor(1.0, dtype=torch.float32) / torch.tensor(255.0, dtype=torch.float32)
    assert torch.equal(((v * 255.0) * scale).bfloat16().float(), v)
    vr, vg, vb = torch.meshgrid(torch.arange(-2, 3.0), torch.arange(-2, 3.0), torch.arange(-2, 3.0), indexing="ij")
    s = ((vr * 255.0 + vg * 255.0 + vb * 255.0) * scale).bfloat16().float()
    assert torch.equal(s, vr + vg + vb)
    sd = en.u8_stem(en.exact_state_dict())
    w = sd["enc1.0.weight"].reshape(64, 27)
    assert torch.equal((w * scale).bfloat16().float(), (w / 255).round())


@pytest.mark.parametrize("C", [64, 128, 256, 512])
@pytest.mark.parametrize("kind", ["sparse", "dense"])
def test_composition_and_packers_exact(C, kind):
    """compose_upconv of integer weights is integer-valued and <= 256 (so its bf16 blobs are the float64 composition),
    the packers only move those values, and oracle.composed_upconv_conv3x3 equals the unfused chain exactly."""
    from unet_dc_segmentation_b200.model import compose_upconv, pack_upfused, pack_upfused_wide, pack_par3x3
    wu, bu, wd, bd = en.upfused_operands(C, 10 + C, kind)
    comp, skipw, bias9 = compose_upconv(wu.float(), bu.float(), wd.float(), bd.float())
    c64 = comp.double()
    assert torch.equal(c64, c64.round()) and float(c64.abs().max()) <= 256
    assert torch.equal(skipw.double(), wd[:, C:].permute(2, 3, 0, 1))
    assert torch.equal(bias9.double() * 4, (bias9.double() * 4).round())
    if C == 64:                  # these two only select and reorder tiles; test_upf_model_level1_exact pins the order
        for blob in (pack_upfused(comp, skipw), pack_par3x3(wd[:, C:].float())):
            assert torch.equal(blob.double(), blob.double().round()) and float(blob.double().abs().max()) <= 256
    else:
        wx, ws = pack_upfused_wide(comp, skipw)
        assert torch.equal(wx.double().flatten().sort().values, c64.flatten().sort().values)
        assert torch.equal(ws.double().flatten().sort().values, skipw.double().flatten().sort().values)
    B, H, W = 2, 6, 5
    x = en.acts((B, H, W, 2 * C), C)
    skip = en.acts((B, 2 * H, 2 * W, C), C + 1)
    want = en.upfused_ref(x, skip, wu, bu, wd, bd, relu=False)
    en.assert_bound(lambda *a: en.upfused_ref(*a, relu=False), x, skip, wu, bu, wd, bd)
    got = oracle.composed_upconv_conv3x3(x.permute(0, 3, 1, 2).float(), skip.permute(0, 3, 1, 2).float(), comp, skipw,
                                         bias9, relu=False)
    assert torch.equal(got.double().permute(0, 2, 3, 1), want)


def _upf_want(x, skip, comp, skipw):
    zero = torch.zeros(9, skip.shape[-1])
    y = oracle.composed_upconv_conv3x3(x.permute(2, 0, 1)[None].float(), skip.permute(2, 0, 1)[None].float(), comp,
                                       skipw, zero, relu=False)
    return y[0].permute(1, 2, 0).numpy()


def test_upf_model_level1_exact():
    """The numpy replay of one tile pair of conv_upfused2_kernel (tests/upf_model.py) gives the exact result."""
    import upf_model as um
    from unet_dc_segmentation_b200 import model as M
    from unet_dc_segmentation_b200.model import compose_upconv
    wu, bu, wd, bd = en.upfused_operands(64, 3, "dense")
    comp, skipw, _ = compose_upconv(wu.float(), bu.float(), wd.float(), bd.float())
    x, skip = en.acts((20, 12, 128), 4), en.acts((40, 24, 64), 5)
    blob = M.pack_upfused(comp, skipw).float().numpy()
    got = np.zeros((40, 24, 64), np.float32)
    for tiles in ([(0, 0), (0, 8)], [(16, 0), (16, 8)]):
        acc = um.level1_tile_pair(x.float().numpy(), skip.float().numpy(), blob, tiles)
        for c, (h0, w0) in enumerate(tiles):
            um.scatter_level1(acc[c], h0, w0, got)
    np.testing.assert_array_equal(got, _upf_want(x, skip, comp, skipw))


@pytest.mark.parametrize("C", [128, 256, 512])
def test_upf_model_wide_exact(C):
    import upf_model as um
    from unet_dc_segmentation_b200 import model as M
    wu, bu, wd, bd = en.upfused_operands(C, C, "dense")
    comp, skipw, _ = M.compose_upconv(wu.float(), bu.float(), wd.float(), bd.float())
    x, skip = en.acts((16, 12, 2 * C), C + 1), en.acts((32, 24, C), C + 2)
    wx, ws = (t.float().numpy() for t in M.pack_upfused_wide(comp, skipw))
    bn = min(C, 256)
    ncls, ntiles = 256 // bn, C // bn
    tiles = [(0, 0), (0, 8)]
    got = np.zeros((32, 24, C), np.float32)
    for grp in range(4 // ncls):
        for nt in range(ntiles):
            acc = um.wide_pass(x.float().numpy(), skip.float().numpy(), wx, ws, C, tiles, grp, nt)
            for c, (h0, w0) in enumerate(tiles):
                for half in range(ncls):
                    cls = grp * ncls + half
                    for lane in range(128):
                        y, xx = 2 * (h0 + lane // 8) + (cls >> 1), 2 * (w0 + lane % 8) + (cls & 1)
                        if y < 32 and xx < 24:
                            got[y, xx, nt * bn:(nt + 1) * bn] = acc[c, half, lane]
    np.testing.assert_array_equal(got, _upf_want(x, skip, comp, skipw))


@pytest.mark.parametrize("name", ["unetdc", "unet", "dil_3_1_5_2_7", "unetdc_4_2"])
def test_oracle_equals_float64_reference(nets, name):
    """On these networks the bf16 emulation IS the truth: oracle.unetdc_forward in fp32, emulated with and without the
    fused decoder levels (and, for three channels, from grey u8 frames) all equal the float64 reference within 1e-6."""
    from unet_dc_segmentation_b200.model import fused_level_blobs
    sd, dil = _net(nets, name)
    cin = en.NETS[name][0]
    B, H, W = 2, 32, 48
    x = en.net_input(B, H, W, 9, cin)
    want = torch.sigmoid(en.forward64(sd, x, dil)["logits"])
    fused = {lvl: fused_level_blobs(sd, lvl) for lvl in (1, 2, 3, 4)}
    # the oracle takes frames / 255 and the stem weights of the u8 entry points only through gray_input; otherwise
    # the integer frames and the integer stem weights
    runs = {"fp32": oracle.unetdc_forward(sd, x.float(), dil),
            "bf16": oracle.unetdc_forward(sd, x.float(), dil, emulate_bf16=True, round_last=en.NETS[name][1] != 1),
            "bf16 fused": oracle.unetdc_forward(sd, x.float(), dil, emulate_bf16=True, fused_levels=fused,
                                                round_last=en.NETS[name][1] != 1)}
    if cin == 3:
        g = en.gray_frames(B, H, W, 9).double()
        xg = g[:, None].expand(B, 3, H, W)
        want_g = torch.sigmoid(en.forward64(sd, xg, dil)["logits"])
        got_g = oracle.unetdc_forward(en.u8_stem(sd), (xg / 255).float(), dil, emulate_bf16=True, gray_input=True,
                                      fused_levels=fused)
        assert float((got_g.double() - want_g).abs().max()) <= 1e-6
    for k, v in runs.items():
        err = float((v.double() - want).abs().max())
        assert err <= 1e-6, f"{name} {k}: max |dp| {err}"


@pytest.mark.parametrize("name", list(en.NETS))
def test_every_layer_is_visible(nets, name):
    """The teeth of the GPU comparisons: for every layer, one in-bounds non-zero weight moved by one unit, and
    separately one bias moved by 1, moves the float64 output by >= 1e-4 somewhere.  Sparse wiring could otherwise hide a
    layer (or a dead channel) from the output, and a kernel bug there from every forward test."""
    sd, dil = _net(nets, name)
    B, H, W = en.TEETH_SHAPE
    x = en.net_input(B, H, W, 5, en.NETS[name][0])
    p0 = torch.sigmoid(en.forward64(sd, x, dil)["logits"])
    weak = []
    for layer, what, m in en.mutations(sd, dil, H, W):
        d = float((torch.sigmoid(en.forward64(m, x, dil)["logits"]) - p0).abs().max())
        if d < 1e-4:
            weak.append(f"{layer} {what}: max |dp| {d:.2e}")
    assert not weak, f"{name}: layers the output does not see: {weak}"
