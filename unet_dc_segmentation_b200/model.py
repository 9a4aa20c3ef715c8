"""``UNetDC`` -- drop-in for the reference ``models/model_2.py`` nn.Module, computed by libunetdc_b200.

Same constructor, same 136 ``state_dict`` keys and shapes, same call contract
(``f32 [B,3,H,W] in [0,1] -> f32 [B,1,H,W]`` probabilities, reference models/model_2.py:56-80), so
``load_model`` of reference quantify_droplets_batch.py:34-37 works unchanged with this class.  The
parameters live in ordinary ``nn.Conv2d`` / ``nn.BatchNorm2d`` / ``nn.ConvTranspose2d`` holders (that is
what fixes the state_dict), but ``forward`` never calls them: on the first call in eval mode the weights
are BatchNorm-folded in fp32, repacked K-major to bf16 and handed to ``dc_model_create``; every call then
runs ``dc_forward`` (18 kernel launches with the decoder levels fused, 22 without; see csrc/api.cu).  There is no PyTorch or CPU fallback.

``UNet`` is the reference's plain ``models/model.py`` network: identical state_dict, dilation 1 everywhere.

``precision = "fp32"`` (class or instance attribute) runs the same network to fp32 accuracy, still on tcgen05: every
activation and weight is held as three bf16 planes (``split_bf16``), each layer sums the six plane products that matter,
and BatchNorm is folded in float64.  About six times the MMAs and three times the workspace of the bf16 forward.
"""
from __future__ import annotations

import ctypes as C

import torch
import torch.nn as nn

from . import _lib

_ENCODER = (("enc1", 64), ("enc2", 128), ("enc3", 256), ("enc4", 512), ("bottleneck", 1024))
# blob order of dc_model_desc_t (include/unetdc_b200.h)
_LAYER_ORDER = (
    ("enc1", 0), ("enc1", 3), ("enc2", 0), ("enc2", 3), ("enc3", 0), ("enc3", 3), ("enc4", 0), ("enc4", 3),
    ("bottleneck", 0), ("bottleneck", 3),
    ("upconv4", None), ("dec4", 0), ("dec4", 3), ("upconv3", None), ("dec3", 0), ("dec3", 3),
    ("upconv2", None), ("dec2", 0), ("dec2", 3), ("upconv1", None), ("dec1", 0), ("dec1", 3),
)


def _conv_pair(cin: int, cout: int, d: int) -> nn.Sequential:
    # indices 0/1 and 3/4 are what the reference's state_dict names (models/model_2.py:40-54)
    return nn.Sequential(
        nn.Conv2d(cin, cout, 3, padding=d, dilation=d), nn.BatchNorm2d(cout), nn.ReLU(inplace=True),
        nn.Conv2d(cout, cout, 3, padding=d, dilation=d), nn.BatchNorm2d(cout), nn.ReLU(inplace=True))


def fold_conv_bn(conv_w, conv_b, bn_w, bn_b, bn_mean, bn_var, eps: float = 1e-5, dtype=torch.float32):
    """Eval-mode BatchNorm folded into the preceding conv, in fp32 (model_2.py:41-46); the fp32-precision forward folds
    in float64 (dtype)."""
    scale = bn_w.to(dtype) / torch.sqrt(bn_var.to(dtype) + eps)
    w = conv_w.to(dtype) * scale.view(-1, 1, 1, 1)
    b = (conv_b.to(dtype) - bn_mean.to(dtype)) * scale + bn_b.to(dtype)
    return w, b


BF16_MAX = float(torch.finfo(torch.bfloat16).max)


def split_bf16(t):
    """float32(t) as three bf16 planes (hi, mid, lo): hi = bf16(x), mid = bf16(x - hi), lo = bf16(x - hi - mid), round to
    nearest even, every residual exact in fp32, so that hi + (mid + lo) == x bit for bit in fp32 (also (hi + mid) + lo
    below the overflow threshold).  Where bf16(x) would overflow (|x| within half a bf16 ulp of FLT_MAX) hi is the
    largest finite bf16 instead, as the device's split does (csrc/generic.cu split3)."""
    x = t.float()
    hi = x.bfloat16()
    over = hi.float().isinf() & ~x.isinf()
    if bool(over.any()):
        hi = torch.where(over, x.sign() * BF16_MAX, hi.float()).bfloat16()
    r = x - hi.float()
    mid = r.bfloat16()
    lo = (r - mid.float()).bfloat16()
    return hi, mid, lo


def pack_conv3x3(w):
    """[Cout,Cin,3,3] -> bf16 [Cout, (ky*3+kx)*Cin + ci] (DC_KIND_CONV3X3 layout)."""
    co, ci = w.shape[:2]
    return w.permute(0, 2, 3, 1).reshape(co, 9 * ci).to(torch.bfloat16).contiguous()


def pack_upconv(w):
    """ConvTranspose2d weight [Cin,Cout,2,2] -> bf16 [(a*2+b)*Cout + co, ci] (DC_KIND_UPCONV2 layout)."""
    ci, co = w.shape[:2]
    return w.float().permute(2, 3, 1, 0).reshape(4 * co, ci).to(torch.bfloat16).contiguous()


def pack_conv3x3_split(w):
    """[Cout,Cin,3,3] (float64 or float32) -> bf16 [Cout, ((ky*3+kx)*3 + plane)*Cin + ci]: the three planes of
    split_bf16 per tap (DC_KIND_CONV3X3 layout of the fp32-precision forward)."""
    co, ci = w.shape[:2]
    return torch.stack(split_bf16(w.permute(0, 2, 3, 1)), 3).reshape(co, 27 * ci).contiguous()


def pack_upconv_split(w):
    """ConvTranspose2d weight [Cin,Cout,2,2] -> bf16 [(a*2+b)*Cout + co, plane*Cin + ci] (the fp32-precision
    DC_KIND_UPCONV2 layout)."""
    ci, co = w.shape[:2]
    return torch.stack(split_bf16(w.permute(2, 3, 1, 0)), 3).reshape(4 * co, 3 * ci).contiguous()


def compose_upconv(wu, bu, wd, bd):
    """ConvTranspose2d(k=2, s=2) followed by cat([up, skip]) and a 3x3 conv, folded into one layer (dc_conv_upfused).

    wu [Cx,C,2,2], bu [C]: the transposed conv (model_2.py:29); wd [Co,2C,3,3], bd [Co]: the 3x3 conv with BatchNorm
    already folded (model_2.py:40-46), input channels [0,C) = up, [C,2C) = skip (torch.cat order, model_2.py:76).
    up[Y,X] = bu + x[Y>>1, X>>1] . wu[:, :, Y&1, X&1], so output pixel (2i+py, 2j+px) sees x only at the 2x2
    neighbourhood (i-1+py+a, j-1+px+b): the weights of that tap are the sum, over the 3x3 taps (ky, kx) that land
    on it, of wu[..., ry, rx] . wd[..., ky, kx] with (ry, rx) the parity of the upsampled pixel.  Composed in fp64,
    rounded to bf16 once.  Returns
      comp  bf16 [4 classes (py*2+px)][2][2 taps (a, b)][Co][Cx]   composed weights over x
      skipw bf16 [3][3][Co][C]                                     the skip half of the 3x3 weights
      bias9 f32  [9][Co]   row (row class * 3 + col class), class 0 / 1 / 2 = first / interior / last output row
                           (column): bd plus bu through the taps that lie inside the upsampled image."""
    cx, c = wu.shape[:2]
    co = wd.shape[0]
    assert cx == 2 * c and co == c and wd.shape[1] == 2 * c and c in (64, 128, 256, 512), "UNet decoder shapes only"
    wu64, wd64 = wu.double(), wd.double()
    wd_up, wd_skip = wd64[:, :c], wd64[:, c:]
    comp = torch.zeros((4, 2, 2, co, cx), dtype=torch.float64, device=wd.device)
    for py in range(2):
        for px in range(2):
            for ky in range(3):
                for kx in range(3):
                    ty, tx = py + ky - 1, px + kx - 1                  # offset of the upsampled pixel from (2i, 2j)
                    a, b = ty // 2 - (py - 1), tx // 2 - (px - 1)      # which of the 2x2 x-taps it reads
                    comp[py * 2 + px, a, b] += torch.einsum("oc,ic->oi", wd_up[:, :, ky, kx], wu64[:, :, ty % 2, tx % 2])
    skipw = wd_skip.permute(2, 3, 0, 1)                                                   # [ky][kx][co][c]
    tb = torch.einsum("ockl,c->klo", wd_up, bu.double())                                  # bias of `up` through tap (ky, kx)
    bias9 = torch.zeros((3, 3, co), dtype=torch.float64, device=wd.device)
    valid = ((1, 2), (0, 1, 2), (0, 1))            # taps inside the image for the first / interior / last row (column)
    for rc in range(3):
        for cc in range(3):
            bias9[rc, cc] = bd.double() + sum(tb[ky, kx] for ky in valid[rc] for kx in valid[cc])
    return (comp.to(torch.bfloat16).contiguous(), skipw.to(torch.bfloat16).contiguous(),
            bias9.reshape(9, co).float().contiguous())


def upfuse_schedule():
    """The MMA schedule of dc_conv_upfused (host-only library call): rows (chunk, r, c, slot0, nslots).  Accumulator
    slot s holds parity class s ^ (s >> 1) (Gray order 0, 1, 3, 2)."""
    buf = (C.c_int * (5 * 128))()
    n = _lib.load().dc_debug_upfuse_schedule(buf, len(buf))
    _lib.check(min(n, 0))
    return [tuple(buf[5 * i:5 * i + 5]) for i in range(n)]


def pack_upfused(comp, skipw):
    """Weights of compose_upconv in the order the kernel's MMAs consume them: bf16 [2 CTAs][2176 rows][64 ci].
    An MMA on window (r, c) covering accumulator slots slot0 .. slot0+n-1 (slot s = class s ^ (s >> 1)) takes, for class
    (py, px), tap (r - py, c - px) of chunk 0 / 1 (x channels [0,64) / [64,128)) or of the skip weights (chunk 2); its
    B operand is those [64 co][64 ci] tiles stacked in slot order, the first half of the rows in CTA 0's blob and the
    second half in CTA 1's.
    comp = None: the skip part alone = a plain 64 -> 64 channel 3x3 layer by parity class, [2][1152][64]
    (dc_conv_args.weight_par)."""
    halves = ([], [])
    for chunk, r, c, cls0, ncls in upfuse_schedule():
        if comp is None and chunk != 2:
            continue
        tiles = []
        for slot in range(cls0, cls0 + ncls):
            cls = slot ^ (slot >> 1)
            py, px = cls >> 1, cls & 1
            tiles.append(skipw[r - py, c - px] if chunk == 2 else comp[cls, r - py, c - px][:, chunk * 64:(chunk + 1) * 64])
        rows = torch.cat(tiles, 0)                                   # [64 * ncls][64]
        half = rows.shape[0] // 2
        halves[0].append(rows[:half])
        halves[1].append(rows[half:])
    blob = torch.stack([torch.cat(h, 0) for h in halves], 0).contiguous()
    assert blob.shape == (2, 2176 if comp is not None else 1152, 64) and blob.dtype == torch.bfloat16
    return blob


def pack_par3x3(w):
    """[64,64,3,3] (BatchNorm folded) -> the parity-class layout of dc_conv_args.weight_par."""
    assert tuple(w.shape) == (64, 64, 3, 3)
    return pack_upfused(None, w.permute(2, 3, 0, 1).to(torch.bfloat16).contiguous())


def pack_upfused_wide(comp, skipw):
    """compose_upconv weights for C = 128 / 256 / 512 in the order conv_upfused_wide_kernel streams them
    (include/unetdc_b200.h dc_upfuse_args): returns (weight, weight_skip),
      weight      [class group][n-tile][CTA][x chunk][tap a*2+b][classes of the group x BN/2 rows][64]
      weight_skip [n-tile][CTA][chunk][tap ky*3+kx][BN/2 rows][64]
    with BN = min(C, 256), 256 / BN classes per group, row r of a tile = output channel n-tile*BN + CTA*BN/2 + r."""
    c = comp.shape[3]
    bn = min(c, 256)
    ncls, nt, hb = 256 // bn, c // bn, bn // 2
    xc, sc = 2 * c // 64, c // 64
    # comp [cls][a][b][co][cx] -> [group][cls in group][tap][n-tile][cta][hb][x chunk][64]
    w = comp.reshape(4 // ncls, ncls, 4, nt, 2, hb, xc, 64)
    w = w.permute(0, 3, 4, 6, 2, 1, 5, 7).contiguous()                 # [group][nt][cta][xchunk][tap][cls][hb][64]
    weight = w.reshape(-1, 64)
    s = skipw.reshape(9, nt, 2, hb, sc, 64).permute(1, 2, 4, 0, 3, 5).contiguous()   # [nt][cta][chunk][tap][hb][64]
    return weight, s.reshape(-1, 64)


def fused_level_blobs(sd, lvl: int = 1, eps: float = 1e-5):
    """(comp, skipw, bias9) of the composed upconv{lvl} + dec{lvl}.0 layer from a state_dict (on the tensors' device)."""
    wd, bd = fold_conv_bn(sd[f"dec{lvl}.0.weight"], sd[f"dec{lvl}.0.bias"], sd[f"dec{lvl}.1.weight"], sd[f"dec{lvl}.1.bias"],
                          sd[f"dec{lvl}.1.running_mean"], sd[f"dec{lvl}.1.running_var"], eps)
    return compose_upconv(sd[f"upconv{lvl}.weight"].float(), sd[f"upconv{lvl}.bias"].float(), wd, bd)


def fused_level1_blobs(sd, eps: float = 1e-5):
    return fused_level_blobs(sd, 1, eps)


class _Packed:
    """Device blobs + the dc_model handle built from one state of the parameters."""

    def __init__(self, module: "UNetDC", device: torch.device):
        lib = _lib.load()
        sd = {k: v.detach().to(device) for k, v in module.state_dict().items()}
        self.blobs = []          # keeps the device tensors alive for the lifetime of the handle
        self.precision = module.precision
        if self.precision not in ("bf16", "fp32"):
            raise ValueError(f"UNetDC.precision must be 'bf16' or 'fp32', got {self.precision!r}")
        fp32 = self.precision == "fp32"
        desc = _lib.ModelDesc()
        for i, (name, idx) in enumerate(_LAYER_ORDER):
            if fp32:
                # every layer on the per-tap kernel in three bf16 planes, BatchNorm folded in float64; enc1.0 runs as an
                # ordinary 3x3 layer on the input planes padded to 64 channels
                if idx is None:
                    w = pack_upconv_split(sd[f"{name}.weight"].double())
                    b = sd[f"{name}.bias"].float().contiguous()
                else:
                    wf, b = fold_conv_bn(sd[f"{name}.{idx}.weight"], sd[f"{name}.{idx}.bias"],
                                         sd[f"{name}.{idx + 1}.weight"], sd[f"{name}.{idx + 1}.bias"],
                                         sd[f"{name}.{idx + 1}.running_mean"], sd[f"{name}.{idx + 1}.running_var"],
                                         module._bn_eps(name, idx + 1), dtype=torch.float64)
                    if i == 0:
                        wp = torch.zeros((wf.shape[0], 64, 3, 3), dtype=wf.dtype, device=wf.device)
                        wp[:, :module.in_channels] = wf
                        wf = wp
                    w = pack_conv3x3_split(wf)
                    b = b.float().contiguous()
            elif idx is None:
                w = pack_upconv(sd[f"{name}.weight"])
                b = sd[f"{name}.bias"].float().contiguous()
            else:
                wf, b = fold_conv_bn(sd[f"{name}.{idx}.weight"], sd[f"{name}.{idx}.bias"],
                                     sd[f"{name}.{idx + 1}.weight"], sd[f"{name}.{idx + 1}.bias"],
                                     sd[f"{name}.{idx + 1}.running_mean"], sd[f"{name}.{idx + 1}.running_var"],
                                     module._bn_eps(name, idx + 1))
                if i == 0 and module.in_channels == 3:
                    w = wf.reshape(wf.shape[0], -1).contiguous()          # stem: fp32 [64][27]
                elif i == 0:
                    # other input channel counts: enc1.0 runs as an ordinary 3x3 layer on the input padded to 64 channels
                    wp = torch.zeros((wf.shape[0], 64, 3, 3), dtype=wf.dtype, device=wf.device)
                    wp[:, :module.in_channels] = wf
                    w = pack_conv3x3(wp)
                else:
                    w = pack_conv3x3(wf)
                    if module.parity_level1 and idx == 3 and name in module.parity_layers:
                        wp = pack_par3x3(wf)
                        self.blobs.append(wp)
                        desc.par_weight[0 if name == "enc1" else 1] = wp.data_ptr()
                b = b.contiguous()
            self.blobs += [w, b]
            desc.weight[i] = w.data_ptr()
            desc.bias[i] = b.data_ptr()
        hw = sd["out_conv.weight"].float().reshape(-1).contiguous()
        hb = sd["out_conv.bias"].float().reshape(-1).contiguous()
        self.blobs += [hw, hb]
        desc.weight[22] = hw.data_ptr()
        desc.bias[22] = hb.data_ptr()
        for i, d in enumerate(module.dilations):
            desc.dilations[i] = int(d)
        desc.base_channels = 64
        desc.in_channels = module.in_channels
        desc.out_channels = module.out_channels
        desc.precision = _lib.DC_PRECISION_FP32 if fp32 else _lib.DC_PRECISION_BF16
        if module.fuse_level1 and not fp32:
            comp, skipw, fb = fused_level1_blobs(sd, module._bn_eps("dec1", 1))
            fw = pack_upfused(comp, skipw)
            self.blobs += [fw, fb]
            desc.fused_weight1 = fw.data_ptr()
            desc.fused_bias1 = fb.data_ptr()
        for lvl in (2, 3, 4):
            if lvl in module.fuse_levels and not fp32:
                comp, skipw, fb = fused_level_blobs(sd, lvl, module._bn_eps(f"dec{lvl}", 1))
                wx, ws = pack_upfused_wide(comp, skipw)
                self.blobs += [wx, ws, fb]
                desc.fused_wide_x[lvl - 2] = wx.data_ptr()
                desc.fused_wide_s[lvl - 2] = ws.data_ptr()
                desc.fused_wide_b[lvl - 2] = fb.data_ptr()
        self.device = device
        self.handle = C.c_void_p()
        with torch.cuda.device(device):
            torch.cuda.synchronize(device)
            _lib.check(lib.dc_model_create(C.byref(self.handle), device.index, C.byref(desc)))
        self.workspace = None

    def workspace_for(self, B: int, H: int, W: int) -> torch.Tensor:
        need = C.c_size_t()
        _lib.check(_lib.load().dc_forward_workspace_bytes(self.handle, B, H, W, C.byref(need)))
        if self.workspace is None or self.workspace.numel() < need.value:
            self.workspace = None
            self.workspace = torch.empty(need.value, dtype=torch.uint8, device=self.device)
        return self.workspace

    def __del__(self):
        try:
            if self.handle:
                _lib.load().dc_model_destroy(self.handle)
        except Exception:
            pass


class UNetDC(nn.Module):
    """Dilated U-Net of reference models/model_2.py:5-80 (dilations 1/2/4/8/16 in the encoder)."""

    dilations = (1, 2, 4, 8, 16)
    # upconv1 + dec1.0 as one launch with host-composed weights (csrc/conv_tc.cu conv_upfused2_kernel); False runs the
    # two layers separately (set it before the first forward, or call invalidate())
    fuse_level1 = True
    # upconv{l} + dec{l}.0 as one launch for l in fuse_levels (2, 3, 4: conv_upfused_wide_kernel)
    fuse_levels = (2, 3, 4)
    # enc1.3 and dec1.3 per output parity class with shared windows (conv_par2_kernel; taken when dilations[0] == 1)
    parity_level1 = True
    parity_layers = ("enc1", "dec1")
    # "bf16" (activations and weights in bf16) or "fp32" (three bf16 planes each, products to ~2^-24 relative, the
    # unfused schedule on the per-tap kernel; the fuse / parity settings above are then ignored).  Read when the weights
    # are packed; changing it repacks on the next call.
    precision = "bf16"

    def __init__(self, in_channels: int = 3, out_channels: int = 1):
        super().__init__()
        if not (1 <= in_channels <= 64 and 1 <= out_channels <= 64):
            raise ValueError("UNetDC (sm_100a): in_channels and out_channels must be in [1, 64]")
        # (3, 1) -- what quantify_droplets_batch.py:35 builds -- is the fused fast path (tcgen05 stem, out_conv + sigmoid
        # + threshold in dec1.3's epilogue); other counts wrap the same layers in two plain kernels (csrc/generic.cu)
        self.in_channels, self.out_channels = int(in_channels), int(out_channels)
        cin = in_channels
        for (name, width), d in zip(_ENCODER, self.dilations):
            setattr(self, name, _conv_pair(cin, width, d))
            cin = width
        for lvl, width in ((4, 512), (3, 256), (2, 128), (1, 64)):
            setattr(self, f"upconv{lvl}", nn.ConvTranspose2d(2 * width, width, kernel_size=2, stride=2))
            setattr(self, f"dec{lvl}", _conv_pair(2 * width, width, 1))
        self.out_conv = nn.Conv2d(64, out_channels, kernel_size=1)
        self._packed: _Packed | None = None

    # ------------------------------------------------------------------ packing
    def _bn_eps(self, name: str, idx: int) -> float:
        return float(getattr(self, name)[idx].eps)

    def invalidate(self) -> None:
        """Drop the packed device weights (call after changing parameters in place)."""
        self._packed = None

    def load_state_dict(self, *args, **kwargs):
        self._packed = None
        return super().load_state_dict(*args, **kwargs)

    def _apply(self, fn, *args, **kwargs):
        self._packed = None
        return super()._apply(fn, *args, **kwargs)

    def packed(self) -> _Packed:
        dev = self.out_conv.weight.device
        _lib.require_cuda(self.out_conv.weight, "UNetDC parameters (call .to('cuda') first)")
        if self._packed is None or self._packed.device != dev or self._packed.precision != self.precision:
            self._packed = _Packed(self, dev)
        return self._packed

    # ------------------------------------------------------------------ inference
    def _run(self, in_kind: int, x: torch.Tensor, B: int, H: int, W: int, thresh: float,
             want_prob: bool, want_mask: bool, mask_out: torch.Tensor | None = None):
        if self.training:
            raise RuntimeError("UNetDC (sm_100a) implements eval-mode inference only; call .eval() "
                               "(reference quantify_droplets_batch.py:37)")
        if H % 16 or W % 16:
            raise ValueError(f"H and W must be multiples of 16 (four 2x2 pools), got {H}x{W}")
        pk = self.packed()
        dev = pk.device
        with torch.cuda.device(dev):
            ws = pk.workspace_for(B, H, W)
            prob = torch.empty((B, self.out_channels, H, W), dtype=torch.float32, device=dev) if want_prob else None
            mask = None
            if want_mask:
                if mask_out is not None:
                    if mask_out.shape != (B, H, W) or mask_out.dtype != torch.uint8 or not mask_out.is_contiguous():
                        raise ValueError("mask_out must be a contiguous uint8 [B,H,W] tensor")
                    mask = _lib.require_cuda(mask_out, "mask_out")
                else:
                    mask = torch.empty((B, H, W), dtype=torch.uint8, device=dev)
            _lib.check(_lib.load().dc_forward(
                pk.handle, in_kind, x.data_ptr(), B, H, W, float(thresh),
                prob.data_ptr() if want_prob else None, mask.data_ptr() if want_mask else None,
                ws.data_ptr(), ws.numel(), _lib.stream_ptr(dev)))
        return prob, mask

    @torch.no_grad()
    def forward(self, x: torch.Tensor) -> torch.Tensor:
        """f32 [B,in_channels,H,W] -> f32 [B,out_channels,H,W] probabilities (sigmoid applied, model_2.py:80)."""
        _lib.require_cuda(x, "UNetDC input")
        if x.dim() != 4 or x.shape[1] != self.in_channels:
            raise ValueError(f"expected [B,{self.in_channels},H,W], got {tuple(x.shape)}")
        x = x.to(torch.float32).contiguous()
        B, _, H, W = x.shape
        prob, _ = self._run(0, x, B, H, W, 0.5, True, False)
        return prob

    @torch.no_grad()
    def predict_u8(self, images: torch.Tensor, prob_thresh: float, return_prob: bool = False,
                   mask_out: torch.Tensor | None = None):
        """Fused path of quantify_droplets_batch.py:45,51-52,56 for device-resident u8 images.

        images: u8 [B,H,W] (grayscale, replicated to RGB as ``Image.convert("RGB")`` does, qdb:41)
                or u8 [B,H,W,3]; the /255 is done in the first kernel.
        Returns (mask u8 [B,H,W] {0,1}, probs f32 [B,1,H,W] or None)."""
        _lib.require_cuda(images, "images")
        if self.in_channels != 3:
            raise ValueError("predict_u8 feeds u8 frames as RGB (qdb:41): it needs a model with in_channels == 3")
        if images.dtype != torch.uint8:
            raise TypeError("predict_u8 takes uint8 images")
        images = images.contiguous()
        if images.dim() == 3:
            kind = 1
        elif images.dim() == 4 and images.shape[-1] == 3:
            kind = 2
        else:
            raise ValueError(f"expected u8 [B,H,W] or [B,H,W,3], got {tuple(images.shape)}")
        B, H, W = images.shape[:3]
        prob, mask = self._run(kind, images, B, H, W, prob_thresh, return_prob, True, mask_out)
        return mask, prob

    def num_launches(self) -> int:
        return int(_lib.load().dc_forward_num_launches(self.packed().handle))


class UNet(UNetDC):
    """Plain U-Net of reference models/model.py:7-50: the same state_dict with dilation 1 everywhere."""

    dilations = (1, 1, 1, 1, 1)
