"""Model of the fp32-precision (three bf16 planes) conv layer -- test infrastructure, CPU only.

``replay_conv`` / ``replay_upconv`` walk K exactly as conv_tc_split_kernel does: per tap, per term
(activation plane ``PLANE_A[t]`` x weight plane ``PLANE_B[t]``, the six products with i + j <= 2), per 64-channel chunk,
reading the activation planes ``in_plane_stride`` channels apart in the pixel and the weight columns
``(3 * tap + plane) * Cin + chunk * 64`` of the packed blob (model.pack_conv3x3_split / pack_upconv_split).  The sums
are float64, which on the operands below is what the tensor core's fp32 accumulation gives.

Exact operands (``operands``): three families whose every product a_i * b_j and every partial sum are exact in fp32
and whose dropped terms (a1 b2, a2 b1, a2 b2) are zero, so that the split layer equals the float64 conv bit for bit and
each of the six terms carries part of the result somewhere:
  'a3'  activations with three non-zero planes (2^17 + 2^8 + 1 = (131072, 256, 1), 2^18 + 2^9 + 3 = (262144, 516, -1))
        x sparse +-1 weights: terms (0,0) (1,0) (2,0)
  'w3'  weights with three non-zero planes x activations in {0, +-1, +-2}: terms (0,0) (0,1) (0,2)
  'mid' both with two planes (513 = (512, 1)): terms (0,0) (0,1) (1,0) (1,1)
Every output's sum |w x| + |b| stays below 2^20, the envelope of tests/exact_net.py.
"""
from __future__ import annotations

import numpy as np
import torch
import torch.nn.functional as F

PLANE_A = (0, 0, 0, 1, 1, 2)          # conv_tc.cu split_plane_a
PLANE_B = (0, 1, 2, 0, 1, 0)
TERMS = tuple(zip(PLANE_A, PLANE_B))
KINDS = ("a3", "w3", "mid")
_A3 = (131329.0, 262659.0, 1.0)        # 2^17 + 2^8 + 1, 2^18 + 2^9 + 3 (an integer needs 18 bits for a non-zero lo)
_MID = (513.0, 1.0)


def _gen(seed):
    return torch.Generator().manual_seed(int(seed))


def _pick(values, shape, g, zero_frac=0.0):
    v = torch.tensor(values, dtype=torch.float64)
    out = v[torch.randint(0, len(values), tuple(shape), generator=g)]
    out = out * (torch.randint(0, 2, tuple(shape), generator=g) * 2 - 1)
    if zero_frac:
        out = out * (torch.rand(tuple(shape), generator=g) >= zero_frac)
    return out


def _sparse(cout, cin, k, taps, per_out, values, g):
    """[cout, cin, k, k] with `per_out` non-zeros per output channel drawn from +-values, spread over taps and chunks."""
    w = torch.zeros(cout, cin, k, k, dtype=torch.float64)
    for o in range(cout):
        for j in range(per_out):
            c = int(torch.randint(0, cin, (1,), generator=g))
            t = taps[(o * per_out + j) % len(taps)]
            w[o, c, t // k, t % k] = float(_pick(values, (1,), g)[0])
    return w


def operands(kind, B, H, W, cin, cout, seed, upconv=False):
    """(x NHWC float64, w float64 [cout, cin, 3, 3] or ConvTranspose2d [cin, cout, 2, 2], bias float64) of `kind`."""
    g = _gen(seed)
    k, taps = (2, (0, 1, 2, 3)) if upconv else (3, (4, 0, 1, 2, 3, 5, 6, 7, 8))
    if kind == "a3":
        x = _pick(_A3 + (0.0,), (B, H, W, cin), g)
        w = _sparse(cout, cin, k, taps, 3, (1.0,), g)
    elif kind == "w3":
        x = _pick((0.0, 1.0, 2.0), (B, H, W, cin), g)
        w = _sparse(cout, cin, k, taps, 3, _A3[::2], g)
    else:
        assert kind == "mid"
        x = _pick(_MID + (2.0, 0.0), (B, H, W, cin), g)
        w = _sparse(cout, cin, k, taps, 3, _MID, g)
    if upconv:
        w = w.permute(1, 0, 2, 3).contiguous()          # [cin, cout, 2, 2]
    b = torch.randint(-16, 17, (cout,), generator=g).double() / 4
    return x, w, b


def split64(t):
    """float64 -> the three planes of model.split_bf16 as float64 [3, ...]."""
    from unet_dc_segmentation_b200.model import split_bf16
    return torch.stack([p.double() for p in split_bf16(t)])


def plane_buffer(x64, plane_stride, width, fill=float("nan"), off=0):
    """bf16 NHWC [..., width] holding plane p of x64 at channels [off + p * plane_stride, + C) and `fill` elsewhere."""
    buf = torch.full(tuple(x64.shape[:-1]) + (width,), fill, dtype=torch.bfloat16)
    C = x64.shape[-1]
    for p, pl in enumerate(split64(x64)):
        buf[..., off + p * plane_stride:off + p * plane_stride + C] = pl.bfloat16()
    return buf


def assert_planes(buf, want64, plane_stride, off, case, others=True):
    """Plane p of a bf16 buffer at channels [off + p * plane_stride, + C) equals plane p of split(want64), bit for bit
    (-0 == +0); others: every channel outside the three ranges still holds the sentinel of exact_net.guarded."""
    from exact_net import SENT16
    g = buf.detach().cpu()
    C = want64.shape[-1]
    want = split64(want64.cpu())
    for p in range(3):
        got = g[..., off + p * plane_stride:off + p * plane_stride + C].float()
        bad = ~(got == want[p].float())
        if bool(bad.any()):
            idx = tuple(int(v) for v in bad.nonzero()[0])
            raise AssertionError(f"{case}: plane {p}: {int(bad.sum())}/{bad.numel()} differ; first at {idx}: got "
                                 f"{float(got[idx])!r}, want {float(want[p][idx])!r} (value {float(want64[idx])!r})")
    if others:
        keep = torch.ones(g.shape[-1], dtype=torch.bool)
        for p in range(3):
            keep[off + p * plane_stride:off + p * plane_stride + C] = False
        assert bool((g.view(torch.int16)[..., keep] == SENT16).all()), f"{case}: wrote outside its channel ranges"


def join(buf, plane_stride, C, off=0):
    """Three bf16 planes of a buffer -> float64 values hi + (mid + lo)."""
    f = buf.double()
    return sum(f[..., off + p * plane_stride:off + p * plane_stride + C] for p in (2, 1, 0))


def replay_conv(buf, in_plane_stride, cin, blob, cout, d, bias, relu=True, terms=TERMS, plane_a=None):
    """The split 3x3 layer's K walk on a plane buffer (bf16 [B,H,W,S]) and a pack_conv3x3_split blob."""
    x = buf.double().numpy()
    Bn, H, W, _ = x.shape
    w = blob.double().numpy()
    xp = np.pad(x, ((0, 0), (d, d), (d, d), (0, 0)))
    acc = np.zeros((Bn, H, W, cout))
    for tap in range(9):
        ky, kx = divmod(tap, 3)
        win = xp[:, ky * d:ky * d + H, kx * d:kx * d + W, :]
        for pa, pb in terms:
            a0 = (plane_a or {}).get(pa, pa) * in_plane_stride
            for ch in range(0, cin, 64):
                A = win[..., a0 + ch:a0 + ch + 64]
                Bm = w[:, (3 * tap + pb) * cin + ch:(3 * tap + pb) * cin + ch + 64]
                acc += A @ Bm.T
    y = torch.from_numpy(acc) + bias.view(1, 1, 1, -1)
    return y.clamp(min=0) if relu else y


def replay_upconv(buf, in_plane_stride, cin, blob, cout, bias, terms=TERMS):
    """The split transposed conv (GEMM N = 4 Cout, parity scatter) on a plane buffer and a pack_upconv_split blob."""
    x = buf.double().numpy()
    Bn, H, W, _ = x.shape
    w = blob.double().numpy()                                   # [4 cout][3 cin]
    acc = np.zeros((Bn, H, W, 4 * cout))
    for pa, pb in terms:
        for ch in range(0, cin, 64):
            acc += x[..., pa * in_plane_stride + ch:pa * in_plane_stride + ch + 64] @ w[:, pb * cin + ch:pb * cin + ch + 64].T
    y = torch.from_numpy(acc).reshape(Bn, H, W, 2, 2, cout) + bias.view(1, 1, 1, 1, 1, -1)
    return y.permute(0, 1, 3, 2, 4, 5).reshape(Bn, 2 * H, 2 * W, cout)


def conv64(x, w, b, d=1, relu=True):
    y = F.conv2d(x.permute(0, 3, 1, 2), w, b, padding=d, dilation=d)
    return (y.clamp(min=0) if relu else y).permute(0, 2, 3, 1)


def upconv64(x, w, b):
    return F.conv_transpose2d(x.permute(0, 3, 1, 2), w, b, stride=2).permute(0, 2, 3, 1)


def pool_split(y64):
    """The split epilogue's 2x2 pool: the max of the fp32 values, then split (NHWC)."""
    return F.max_pool2d(y64.permute(0, 3, 1, 2), 2).permute(0, 2, 3, 1)


def pool_per_plane(y64):
    """A per-plane max (wrong: the max of each plane is not a plane of the max), joined back to values."""
    pl = split64(y64)
    return sum(pool_split(pl[p]) for p in (2, 1, 0))


def network(sd, x, terms=None, dilations=(1, 2, 4, 8, 16)):
    """UNetDC evaluated on the host in float64: x NCHW, returns channel 0 of the probabilities.  terms=None: the
    float64 network (BatchNorm folded in float64), the reference of the fp32-precision forward.  terms = TERMS: the
    forward's arithmetic evaluated exactly -- weights and every stored activation rounded to fp32 and split into
    three bf16 planes, only the listed plane products summed (exactly), bias, ReLU and pooling as the kernels do them.
    What the GPU forward adds to the error of the latter comes from summing the products in the tensor cores' fp32
    accumulator (tools/split_emulation.py)."""
    from unet_dc_segmentation_b200.model import fold_conv_bn
    sdd = {k: v.detach().double().cpu() for k, v in sd.items()}
    f32 = (lambda t: t) if terms is None else (lambda t: t.float().double())

    def mix(op, t, w):
        if terms is None:
            return op(t, w)
        ts, ws = split64(f32(t)), split64(f32(w))
        return sum(op(ts[i], ws[j]) for i, j in terms)

    def conv(t, p, idx, d):
        w, b = fold_conv_bn(sdd[f"{p}.{idx}.weight"], sdd[f"{p}.{idx}.bias"], sdd[f"{p}.{idx + 1}.weight"],
                            sdd[f"{p}.{idx + 1}.bias"], sdd[f"{p}.{idx + 1}.running_mean"],
                            sdd[f"{p}.{idx + 1}.running_var"], dtype=torch.float64)
        y = mix(lambda a, k: F.conv2d(a, k, None, padding=d, dilation=d), t, w) + f32(b).view(1, -1, 1, 1)
        return f32(F.relu(y))

    t, skips = f32(x.double().cpu()), []
    for i, name in enumerate(("enc1", "enc2", "enc3", "enc4")):
        t = conv(conv(t, name, 0, dilations[i]), name, 3, dilations[i])
        skips.append(t)
        t = F.max_pool2d(t, 2)
    t = conv(conv(t, "bottleneck", 0, dilations[4]), "bottleneck", 3, dilations[4])
    for lvl in (4, 3, 2, 1):
        up = mix(lambda a, k: F.conv_transpose2d(a, k, None, stride=2), t, sdd[f"upconv{lvl}.weight"])
        up = f32(up + f32(sdd[f"upconv{lvl}.bias"]).view(1, -1, 1, 1))
        t = conv(conv(torch.cat([up, skips[lvl - 1]], 1), f"dec{lvl}", 0, 1), f"dec{lvl}", 3, 1)
    logits = F.conv2d(t, f32(sdd["out_conv.weight"]), f32(sdd["out_conv.bias"]))
    return torch.sigmoid(logits)[:, 0]
