"""Integer-valued layers and networks on which the tensor-core path is exact -- test infrastructure, CPU only.

The product of two bf16 values is exact in fp32.  When every operand is an integer (or a multiple of one small power of
two) and sum |w * x| of every output stays below 2^24, every fp32 partial sum is exact too, in any summation order: the
tensor-core K order, the halves of a CTA pair, the passes of the wide decoder kernel, the shared windows of the parity
kernel cannot change the result.  bias + ReLU in fp32 are then exact, and the store (round to nearest even) gives the
same bits as a float64 reference converted with ``.float().bfloat16()``.  The generators here keep that bound at 2^20
(``BOUND``), so a kernel is held to the float64 value by ``torch.equal`` instead of a tolerance.

Networks: ``exact_state_dict`` builds the 136-key state_dict of ``UNetDC`` / ``UNet`` / ``UNetDC(cin, cout)`` / the
dilation-set subclasses so that every stored activation is an integer of magnitude <= 256 (``STORE_MAX``, lossless in
bf16).  Then every schedule of the forward (fused or unfused decoder levels, parity layers, kernel families, upfuse
modes) must give identical bits, equal to the plain float64 evaluation ``forward64``.
  3x3 conv: per output channel exactly one +1 weight and one or more -1 weights, every input channel read, every
            (tap, 64-channel chunk) block holding a non-zero; bias (BatchNorm beta) in {0, 1, 2}.  With non-negative
            inputs and a positive weight mass of 1 the maximum grows by at most the bias per layer.
  BatchNorm: gamma 1, mean 0, running_var float32(1 - 1e-5), so that var + 1e-5 == 1.0f and the fold is the identity.
  upconv:   one +1 per (output channel, parity) on an input channel (every input channel read), bias in {0..3}.
  out_conv: dense k / 2^s, k in [-4, 4], dyadic bias, calibrated so that the logits spread over a few units.
  stem:     for the u8 entry points the stem weights are 255 * v: the kernel's 1/255 gives bf16 weight v exactly.
"""
from __future__ import annotations

import ctypes

import pytest
import torch
import torch.nn.functional as F

BOUND = 1 << 20
STORE_MAX = 256
BN_VAR = float(torch.tensor(1.0 - 1e-5, dtype=torch.float32))     # float32(var) + 1e-5 rounds to exactly 1.0f
FRAME_MAX = 127
CONV_LAYERS = ("enc1.0", "enc1.3", "enc2.0", "enc2.3", "enc3.0", "enc3.3", "enc4.0", "enc4.3", "bottleneck.0",
               "bottleneck.3", "dec4.0", "dec4.3", "dec3.0", "dec3.3", "dec2.0", "dec2.3", "dec1.0", "dec1.3")
ALL_LAYERS = CONV_LAYERS + ("upconv4", "upconv3", "upconv2", "upconv1", "out_conv")
_ENC = (("enc1", 64), ("enc2", 128), ("enc3", 256), ("enc4", 512))


def _gen(seed):
    return torch.Generator().manual_seed(int(seed))


# ----------------------------------------------------------------------------- single-layer operands

def acts(shape, seed, lo=-8, hi=8):
    """Integer activations in [lo, hi], float64."""
    return torch.randint(lo, hi + 1, tuple(shape), generator=_gen(seed)).double()


def biases(n, seed):
    """Multiples of 1/4 in [-4, 4]."""
    return torch.randint(-16, 17, (n,), generator=_gen(seed)).double() / 4


def conv_weight(cout, cin, kind, seed):
    """[cout, cin, 3, 3] float64.  'dense': integers in [-2, 2] (long K, large partial sums, outputs that round in bf16);
    'sparse': 16 entries of +-1 per output channel (outputs <= 256 on activations <= 8, so any single wrong term
    shows), spread so that every (tap, 64-channel chunk) block holds one."""
    g = _gen(seed)
    if kind == "dense":
        return torch.randint(-2, 3, (cout, cin, 3, 3), generator=g).double()
    assert kind == "sparse"
    w = torch.zeros(cout, cin, 3, 3, dtype=torch.float64)
    nchunk = -(-cin // 64)
    nblk = 9 * nchunk
    for o in range(cout):
        for j in range(16):
            blk = (o * 16 + j) % nblk
            tap, chunk = blk // nchunk, blk % nchunk
            c = chunk * 64 + int(torch.randint(0, min(64, cin - chunk * 64), (1,), generator=g))
            w[o, c, tap // 3, tap % 3] = 1.0 if int(torch.randint(0, 2, (1,), generator=g)) else -1.0
    return w


def upconv_weight(cin, cout, kind, seed):
    """ConvTranspose2d weight [cin, cout, 2, 2]: 'dense' integers in [-2, 2] or 'sparse' (one +1 per output channel and
    parity, every input channel read: the network recipe)."""
    g = _gen(seed)
    if kind == "dense":
        return torch.randint(-2, 3, (cin, cout, 2, 2), generator=g).double()
    w = torch.zeros(cin, cout, 2, 2, dtype=torch.float64)
    perm = torch.randperm(cin, generator=g)
    for p in range(4):
        for o in range(cout):
            if p < 2 and cin >= 2 * cout:
                c = int(perm[(p * cout + o) % cin])
            else:
                c = int(torch.randint(0, cin, (1,), generator=g))
            w[c, o, p // 2, p % 2] = 1.0
    return w


def upfused_operands(C, seed, kind="sparse"):
    """(wu, bu, wd, bd) of an upconv(2C -> C) + 3x3 conv(2C -> C) pair whose composition (model.compose_upconv) is
    integer-valued and exact in bf16: a sparse transposed conv (one +1 per output channel and parity), the 3x3 conv
    'sparse' or 'dense', integer biases of the transposed conv, quarter biases of the conv."""
    wu = upconv_weight(2 * C, C, "sparse", seed)
    bu = torch.randint(0, 4, (C,), generator=_gen(seed + 1)).double()
    wd = conv_weight(C, 2 * C, kind, seed + 2)
    bd = biases(C, seed + 3)
    return wu, bu, wd, bd


def bf16(t64):
    """float64 -> the bf16 the kernels store (round to nearest even), asserting the float32 step is exact."""
    f = t64.float()
    assert torch.equal(f.double(), t64), "reference value not exact in fp32"
    return f.bfloat16()


def conv3x3_ref(x, w, b, d=1, relu=True):
    """x NHWC float64 -> NHWC float64."""
    y = F.conv2d(x.permute(0, 3, 1, 2), w, b, padding=d, dilation=d)
    return (y.clamp(min=0) if relu else y).permute(0, 2, 3, 1)


def upconv_ref(x, w, b):
    return F.conv_transpose2d(x.permute(0, 3, 1, 2), w, b, stride=2).permute(0, 2, 3, 1)


def upfused_ref(x, skip, wu, bu, wd, bd, relu=True):
    """The unfused chain conv_transpose2d -> cat -> conv2d, NHWC float64."""
    xs, ss = x.permute(0, 3, 1, 2), skip.permute(0, 3, 1, 2)
    y = F.conv2d(torch.cat([F.conv_transpose2d(xs, wu, bu, stride=2), ss], 1), wd, bd, padding=1)
    return (y.clamp(min=0) if relu else y).permute(0, 2, 3, 1)


def assert_bound(fn, *operands):
    """sum |w * x| (+ |b|) of every output of fn(*operands) is at most BOUND: fn evaluated on the absolute values."""
    m = float(fn(*(o.abs() if torch.is_tensor(o) else o for o in operands)).max())
    assert m <= BOUND, f"operand bound {m} > {BOUND}"
    return m


# ----------------------------------------------------------------------------- comparison

def _where(bad, names):
    idx = tuple(int(v) for v in bad.nonzero()[0])
    return idx, ", ".join(f"{n}={i}" for n, i in zip(names, idx))


def assert_exact(got, want64, case, names=("b", "y", "x", "c")):
    """A stored bf16 tensor against the float64 reference, bit for bit (-0 equals +0).  The report names the case and
    the first mismatching (b, y, x, c)."""
    g = got.detach().float().cpu()
    w = bf16(want64).float()
    assert g.shape == w.shape, f"{case}: shape {tuple(g.shape)} != {tuple(w.shape)}"
    bad = ~(g == w)
    if bool(bad.any()):
        idx, where = _where(bad, names)
        raise AssertionError(f"{case}: {int(bad.sum())}/{bad.numel()} elements differ; first at ({where}): "
                             f"got {float(g[idx])!r}, want {float(w[idx])!r}")


def assert_probs(prob, mask, logits64, thresh, case, names=("b", "y", "x")):
    """Probabilities within 1e-6 of the float64 sigmoid (the logits are exact on both sides: what is left is expf and
    one division); the mask exact wherever |p - thresh| > 1e-6."""
    want = torch.sigmoid(logits64)
    if prob is not None:
        p = prob.detach().double().cpu()
        assert p.shape == want.shape, f"{case}: prob shape {tuple(p.shape)} != {tuple(want.shape)}"
        bad = ~((p - want).abs() <= 1e-6)
        if bool(bad.any()):
            idx, where = _where(bad, names if p.dim() == len(names) else ("b", "o", "y", "x"))
            raise AssertionError(f"{case}: {int(bad.sum())}/{bad.numel()} probabilities off by > 1e-6; first at ({where}): "
                                 f"got {float(p[idx])!r}, want {float(want[idx])!r} (logit {float(logits64[idx])!r})")
    if mask is not None:
        w0 = want[:, 0] if want.dim() == 4 else want
        m = mask.detach().cpu()
        bad = (m != (w0 > thresh).to(torch.uint8)) & ((w0 - thresh).abs() > 1e-6)
        if bool(bad.any()):
            idx, where = _where(bad, names)
            raise AssertionError(f"{case}: {int(bad.sum())} mask pixels differ; first at ({where}): got {int(m[idx])}, "
                                 f"p = {float(w0[idx])!r}")


# ----------------------------------------------------------------------------- networks

def frames(B, H, W, seed):
    """u8 [B,H,W,3] in [0, FRAME_MAX]: three different channels, every frame different."""
    return torch.randint(0, FRAME_MAX + 1, (B, H, W, 3), generator=_gen(seed), dtype=torch.uint8)


def gray_frames(B, H, W, seed):
    return torch.randint(0, FRAME_MAX + 1, (B, H, W), generator=_gen(seed), dtype=torch.uint8)


def _net_conv(cout, cin, g, centre):
    """Network 3x3 conv: one +1 and n_neg >= 1 -1 weights per output channel.  The +1 weights read one permutation of the
    input channels, the -1 weights continue it, so every input channel is read; per 64-channel chunk the -1 weights take
    every tap.  The +1 sits on the centre tap when `centre` (large dilations: the outer taps of a small map fall in the
    padding) and otherwise on the centre tap for about half of the channels."""
    n_neg = max(1, -(-cin // cout) - 1)
    w = torch.zeros(cout, cin, 3, 3, dtype=torch.float64)
    chans = torch.cat([torch.randperm(cin, generator=g) for _ in range(-(-cout * (1 + n_neg) // cin))])
    pos, neg = chans[:cout], chans[cout:cout * (1 + n_neg)]
    taps = torch.zeros(len(neg), dtype=torch.long)
    chunk = neg // 64
    for k in chunk.unique():
        sel = (chunk == k).nonzero()[:, 0]
        taps[sel[torch.randperm(len(sel), generator=g)]] = torch.arange(len(sel)) % 9
    for s in range(len(neg)):
        o, c, t = s % cout, int(neg[s]), int(taps[s])
        while w[o, c, t // 3, t % 3] != 0:
            t = (t + 1) % 9
        w[o, c, t // 3, t % 3] = -1.0
    for o in range(cout):
        c = int(pos[o])
        t = 4 if centre or int(torch.randint(0, 2, (1,), generator=g)) else int(torch.randint(0, 9, (1,), generator=g))
        while w[o, c, t // 3, t % 3] != 0:
            t = (t + 1) % 9
        w[o, c, t // 3, t % 3] = 1.0
    return w


def blocks_covered(w, upconv=False):
    """Every (tap, 64-channel chunk) block (transposed conv: (parity, chunk)) holds a non-zero weight."""
    if upconv:
        w = w.permute(1, 0, 2, 3)                          # [cout, cin, 2, 2]
    nz = w.ne(0).any(0)                                    # [cin, k, k]
    cin = nz.shape[0]
    return all(bool(nz[c0:c0 + 64].any(0).all()) for c0 in range(0, cin, 64))


def _conv_layer_names(in_channels):
    names = []
    cin = in_channels
    for name, width in _ENC + (("bottleneck", 1024),):
        names += [(f"{name}.0", cin, width), (f"{name}.3", width, width)]
        cin = width
    for lvl, width in ((4, 512), (3, 256), (2, 128), (1, 64)):
        names += [(f"dec{lvl}.0", 2 * width, width), (f"dec{lvl}.3", width, width)]
    return names


def exact_state_dict(in_channels=3, out_channels=1, dilations=(1, 2, 4, 8, 16), seed=0, calib=(64, 64)):
    """The 136-key state_dict of the integer network (see the module docstring), float32 like a checkpoint."""
    from unet_dc_segmentation_b200.model import UNetDC
    g = _gen(1000 + seed)
    sd = {k: v.clone() for k, v in UNetDC(in_channels, out_channels).state_dict().items()}
    level = {"enc1": 0, "enc2": 1, "enc3": 2, "enc4": 3, "bottleneck": 4}
    for name, cin, cout in _conv_layer_names(in_channels):
        p, idx = name.rsplit(".", 1)
        bn = f"{p}.{int(idx) + 1}"
        sd[f"{name}.weight"] = _net_conv(cout, cin, g, dilations[level[p]] >= 4 if p in level else False).float()
        sd[f"{name}.bias"] = torch.zeros(cout)
        sd[f"{bn}.weight"] = torch.ones(cout)
        sd[f"{bn}.bias"] = torch.randint(0, 3, (cout,), generator=g).float()
        sd[f"{bn}.running_mean"] = torch.zeros(cout)
        sd[f"{bn}.running_var"] = torch.full((cout,), BN_VAR)
    for lvl, width in ((4, 512), (3, 256), (2, 128), (1, 64)):
        sd[f"upconv{lvl}.weight"] = upconv_weight(2 * width, width, "sparse", int(torch.randint(0, 1 << 30, (1,), generator=g))).float()
        sd[f"upconv{lvl}.bias"] = torch.randint(0, 4, (width,), generator=g).float()
    # out_conv: logits = (k . feat) / 2^s + b, calibrated on one frame so that they spread over a few units around 0
    k = torch.randint(-4, 5, (out_channels, 64), generator=g).double()
    H, W = calib
    x = net_input(1, H, W, 77 + seed, in_channels)
    sd["out_conv.weight"] = torch.zeros(out_channels, 64, 1, 1)
    sd["out_conv.bias"] = torch.zeros(out_channels)
    feat = forward64(sd, x, dilations)["dec1.3"]
    raw = torch.einsum("oc,bchw->bohw", k, feat)
    s = 6
    while float(raw.std()) / 2 ** s > 2.5:
        s += 1
    sd["out_conv.weight"] = (k / 2 ** s).float().reshape(out_channels, 64, 1, 1)
    sd["out_conv.bias"] = (torch.round(-raw.mean((0, 2, 3)) / 2 ** s * 64) / 64).float()
    return sd


def u8_stem(sd):
    """The same network for the u8 entry points: stem weights 255 * v (the kernel multiplies by 1/255)."""
    sd = dict(sd)
    sd["enc1.0.weight"] = sd["enc1.0.weight"] * 255.0
    return sd


def folded(sd, name):
    """(w, b) of a conv + BatchNorm pair folded as the product folds them (model.fold_conv_bn, fp32), as float64."""
    from unet_dc_segmentation_b200.model import fold_conv_bn
    p, idx = name.rsplit(".", 1)
    bn = f"{p}.{int(idx) + 1}"
    w, b = fold_conv_bn(sd[f"{name}.weight"], sd[f"{name}.bias"], sd[f"{bn}.weight"], sd[f"{bn}.bias"],
                        sd[f"{bn}.running_mean"], sd[f"{bn}.running_var"])
    return w.double(), b.double()


def forward64(sd, x, dilations=(1, 2, 4, 8, 16), bounds=None):
    """Plain float64 evaluation of the network: x float64 [B, cin, H, W] (integer grey levels, not /255).
    Returns every intermediate NCHW tensor by layer name ('enc1.0' ... 'dec1.3', 'pool1' ... 'pool4', 'upconv4' ...
    'upconv1') plus 'logits'; `bounds` (a dict), when given, receives sum |w * x| + |b| of each layer."""
    t = {}

    def conv(name, inp, d):
        w, b = folded(sd, name)
        if bounds is not None:
            bounds[name] = float(F.conv2d(inp.abs(), w.abs(), b.abs(), padding=d, dilation=d).max())
        t[name] = F.relu(F.conv2d(inp, w, b, padding=d, dilation=d))
        return t[name]

    cur = x
    for i, (name, _) in enumerate(_ENC):
        cur = conv(f"{name}.3", conv(f"{name}.0", cur, dilations[i]), dilations[i])
        cur = t[f"pool{i + 1}"] = F.max_pool2d(cur, 2)
    cur = conv("bottleneck.3", conv("bottleneck.0", cur, dilations[4]), dilations[4])
    for lvl in (4, 3, 2, 1):
        wu, bu = sd[f"upconv{lvl}.weight"].double(), sd[f"upconv{lvl}.bias"].double()
        if bounds is not None:
            bounds[f"upconv{lvl}"] = float(F.conv_transpose2d(cur.abs(), wu.abs(), bu.abs(), stride=2).max())
        up = t[f"upconv{lvl}"] = F.conv_transpose2d(cur, wu, bu, stride=2)
        cur = conv(f"dec{lvl}.3", conv(f"dec{lvl}.0", torch.cat([up, t[f"enc{lvl}.3"]], 1), 1), 1)
    hw, hb = sd["out_conv.weight"].double(), sd["out_conv.bias"].double()
    if bounds is not None:
        bounds["out_conv"] = float(F.conv2d(cur.abs(), hw.abs(), hb.abs()).max())
    t["logits"] = F.conv2d(cur, hw, hb)
    return t


STORED = tuple(n for n in CONV_LAYERS) + ("pool1", "pool2", "pool3", "pool4", "upconv4", "upconv3", "upconv2", "upconv1")


def net_input(B, H, W, seed, in_channels=3):
    """float64 NCHW integer frames in [0, FRAME_MAX] for the reference and the f32 entry point: for three channels the
    frames of `frames(B, H, W, seed)` (so that the u8 entry points see the same integers), else independent channels."""
    if in_channels == 3:
        return frames(B, H, W, seed).permute(0, 3, 1, 2).double().contiguous()
    return torch.randint(0, FRAME_MAX + 1, (B, in_channels, H, W), generator=_gen(seed)).double()


def _in_bounds_taps(d, h, w):
    return [(ky, kx) for ky in range(3) for kx in range(3) if abs(ky - 1) * d < h and abs(kx - 1) * d < w]


def mutations(sd, dilations, H, W, seed=0):
    """For every layer of the network: (layer, what, mutated state_dict) with one non-zero weight on a tap inside an
    H x W frame's map moved by one unit (+-1; the head by its 1/2^s) and, separately, one bias moved by 1."""
    g = _gen(5000 + seed)
    out = []
    level = {"enc1": 0, "enc2": 1, "enc3": 2, "enc4": 3, "bottleneck": 4}
    for name in ALL_LAYERS:
        wkey = f"{name}.weight"
        w = sd[wkey]
        nz = w.ne(0)
        if name in CONV_LAYERS:
            p, idx = name.split(".")
            lvl = level[p] if p in level else int(p[3]) - 1
            d = dilations[lvl] if p in level else 1
            ok = torch.zeros(3, 3, dtype=torch.bool)
            for ky, kx in _in_bounds_taps(d, H >> lvl, W >> lvl):
                ok[ky, kx] = True
            nz &= ok.view(1, 1, 3, 3)
            bkey = f"{p}.{int(idx) + 1}.bias"
        else:
            bkey = f"{name}.bias"
        cand = nz.nonzero()
        pick = tuple(int(v) for v in cand[int(torch.randint(0, len(cand), (1,), generator=g))])
        step = float(w.abs()[w.ne(0)].min()) if name == "out_conv" else 1.0
        sign = 1.0 if int(torch.randint(0, 2, (1,), generator=g)) else -1.0
        m = dict(sd)
        m[wkey] = w.clone()
        m[wkey][pick] += sign * step
        out.append((name, f"weight {pick} {sign * step:+g}", m))
        m = dict(sd)
        m[bkey] = sd[bkey].clone()
        m[bkey][int(torch.randint(0, len(sd[bkey]), (1,), generator=g))] += 1.0
        out.append((name, "bias +1", m))
    return out


# The networks the GPU tests run: name -> (in_channels, out_channels, dilations, seed).  The seeds are ones for which
# every layer moves the output (tests/test_exact_net.py::test_every_layer_is_visible at TEETH_SHAPE).
DEFAULT_DIL = (1, 2, 4, 8, 16)
NETS = {
    "unetdc": (3, 1, DEFAULT_DIL, 0),
    "unet": (3, 1, (1, 1, 1, 1, 1), 0),
    "dil_1_2_2_4_4": (3, 1, (1, 2, 2, 4, 4), 0),
    "dil_2_4_8_16_32": (3, 1, (2, 4, 8, 16, 32), 0),
    "dil_3_1_5_2_7": (3, 1, (3, 1, 5, 2, 7), 0),
    "unetdc_1_1": (1, 1, DEFAULT_DIL, 2),
    "unetdc_4_2": (4, 2, DEFAULT_DIL, 2),
    "unetdc_7_1": (7, 1, DEFAULT_DIL, 0),
}
FORWARD_SHAPES = [(1, 16, 16), (2, 48, 80), (1, 80, 48), (3, 112, 208), (1, 16, 272), (2, 272, 16), (1, 256, 256),
                  (1, 64, 128)]
TEETH_SHAPE = (1, 64, 128)            # the shape every network is also run at on the GPU


def net(name):
    cin, cout, dil, seed = NETS[name]
    return exact_state_dict(cin, cout, dil, seed), dil


# ----------------------------------------------------------------------------- device buffers and launches (GPU tests)

GUARD = 4096                                   # bytes of sentinel before and after every output view
SENT = 0xA5
SENT16 = -23131                                # int16 view of the bytes 0xA5 0xA5


def _lib():
    from unet_dc_segmentation_b200 import _lib as L
    return L


@pytest.fixture
def family():
    """dc_debug_set_conv_family for one test, restored to auto afterwards (import it into a test module to use it)."""
    L = _lib()
    codes = {"auto": L.DC_CONV_FAMILY_AUTO, "generic": L.DC_CONV_FAMILY_GENERIC}
    try:
        yield lambda name: L.check(L.load().dc_debug_set_conv_family(codes[name]))
    finally:
        L.check(L.load().dc_debug_set_conv_family(L.DC_CONV_FAMILY_AUTO))


def guarded(shape, dtype):
    """(raw uint8 buffer, view of `shape`) on the device: the view sits between GUARD sentinel bytes, and is itself
    sentinel-filled."""
    n = torch.Size(shape).numel() * torch.empty((), dtype=dtype).element_size()
    raw = torch.full((n + 2 * GUARD,), SENT, dtype=torch.uint8, device="cuda")
    return raw, raw[GUARD:GUARD + n].view(dtype).view(shape)


def check_guards(raw, case):
    r = raw.cpu()
    assert bool((r[:GUARD] == SENT).all()), f"{case}: wrote before its output buffer"
    assert bool((r[-GUARD:] == SENT).all()), f"{case}: wrote after its output buffer"


def check_outside(raw, view, off, n, case):
    """Guards intact and channels [0, off) and [off + n, S) of a bf16 NHWC view untouched."""
    check_guards(raw, case)
    v = view.cpu().view(torch.int16)
    assert bool((v[..., :off] == SENT16).all()) and bool((v[..., off + n:] == SENT16).all()), \
        f"{case}: wrote outside channels [{off}, {off + n})"


def conv_tc(**kw):
    """dc_conv_tc with the given dc_conv_args fields, synchronised."""
    L = _lib()
    a = L.ConvArgs()
    for k, v in kw.items():
        setattr(a, k, v)
    L.check(L.load().dc_conv_tc(ctypes.byref(a), L.stream_ptr()))
    torch.cuda.synchronize()
