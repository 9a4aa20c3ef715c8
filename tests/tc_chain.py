"""The calibrated network's forward as a chain of single-layer launches, every layer held to the tcgen05 accumulator
model (tc_accum_model) -- test infrastructure, GPU.

One launch sequence serves the default bf16 forward (as dc_forward's forward_impl runs it, csrc/api.cu: the stem,
enc1.3 STORE_POOL, enc2-4 and the bottleneck, upconv + dec.0 fused per level, each dec.3, dec1.3 HEAD) and the fp32
forward (split input, 18 convs, 4 transposed convs into [up | enc] plane buffers, HEAD).  After each launch the check
passed in picks the layer's sites: None replays the whole map (test_gpu_tc_accum.py's small chains), sites replay
those outputs only (test_gpu_tc_accum_fullsize.py).  Either way every checked output must equal the model's replay of
the layer's own GPU input bit for bit (probabilities within 1e-6 of the sigmoid of the exact logit)."""

import time
from typing import NamedTuple

import torch

import exact_net as en
import split_model as sm
import tc_accum_model as tm

THRESH = 0.3


def _L():
    from unet_dc_segmentation_b200 import _lib
    return _lib


class Geom(NamedTuple):
    """A launch as a check sees it: the grid its sites live on (B frames of h x w: the output map, or the half-resolution
    map for the parity-class kernels, the fused kernels and the transposed conv, whose sites stand for 2 x 2 output
    blocks), the dilation on that grid, the kernel's tile (rows, columns) on it, the MMA products one site replays
    and the kernel's name."""
    case: str
    B: int
    h: int
    w: int
    d: int
    tile: tuple
    cost: int
    kernel: str


def whole_map(geom):
    """The check that replays every output of every layer."""
    return None


class Sites:
    """The check that replays sampled sites (tc_accum_model.select_sites) of the given frames, seeded per layer, and
    prints per layer the sites, MMA products and replay time.  teeth: the kernels at whose first non-HEAD layer a
    wrong walk is replayed at the same sites; ``wrong[kernel]`` = (outputs it changes, outputs compared)."""

    def __init__(self, frames, teeth=()):
        self.frames = list(frames)
        self.teeth = set(teeth)
        self.wrong = {}
        self.layers = 0

    def __call__(self, geom):
        self.layers += 1
        return tm.select_sites((geom.B, geom.h, geom.w), geom.d, geom.tile, self.frames, geom.cost, seed=self.layers)

    def report(self, geom, sites, replayed, seconds):
        """One line per layer; every tile of the kernel's grid in the checked frames holds a site."""
        b, y, x = sites
        th, tw = geom.tile
        tiles = torch.unique(torch.stack([b, y // th, x // tw]), dim=1).shape[1]
        want = len(self.frames) * -(-geom.h // th) * -(-geom.w // tw)
        n = replayed[0].numel()
        print(f"{geom.case}: {geom.kernel}, {n} sites, {tiles}/{want} tiles, {n * geom.cost:.3e} products, "
              f"replay {seconds:.2f} s")
        assert tiles == want, f"{geom.case}: the sites miss {want - tiles} tiles"


def _at(t, s):
    return t if s is None else t[s[0], s[1], s[2]]


def bf16_blobs(m):
    """The packed bf16 model's blobs by role (model._Packed: per layer [parity blob], weight, bias; the head; the fused
    level-1 blob and bias9; per wide level x weights, skip weights, bias9)."""
    from unet_dc_segmentation_b200.model import _LAYER_ORDER
    it = iter(m.packed().blobs)
    wts, bss, par = [], [], {}
    for i, (name, idx) in enumerate(_LAYER_ORDER):
        if m.parity_level1 and idx == 3 and name in m.parity_layers:
            par[i] = next(it)
        wts.append(next(it))
        bss.append(next(it))
    hw, hb = next(it), next(it)
    fused = {1: (next(it), None, next(it))}
    for lvl in (2, 3, 4):
        fused[lvl] = (next(it), next(it), next(it))
    assert next(it, None) is None and set(par) == {1, 21} and tuple(par[1].shape) == (2, 1152, 64)
    return wts, bss, par, hw, float(hb[0]), fused


def forward_chain(m, precision, fam, u8, x32, pick, in_kind=1):
    """Run m's forward one launch at a time and check every layer with `pick` (whole_map or a Sites).  precision "bf16"
    (the default forward; in_kind: the stem's input, 1 = u8 grey, 0 = fp32) or "fp32" (m.precision already "fp32");
    fam: the conv family already set (dc_debug_set_conv_family); u8 [B, H, W] grey frames and x32 [B, 3, H, W] the
    same frames as fp32.  Under family generic conv_par2_kernel and the pair / halo kernels are off (launch_conv_tc),
    the fused kernels are not.  Returns the chain's (prob [B, H, W], mask)."""
    import ctypes
    from unet_dc_segmentation_b200.model import fused_level_blobs, pack_upfused, pack_upfused_wide
    L = _L()
    fp32 = precision == "fp32"
    B, H, W = u8.shape
    dil = m.dilations
    P = 3 if fp32 else 1                               # planes per tensor
    name = f"{precision} chain {B}x{H}x{W}" + ("" if fp32 else f" {fam}")
    teeth = getattr(pick, "teeth", set())
    if fp32:
        pk = m.packed()
        wts = [pk.blobs[2 * i] for i in range(22)]
        bss = [pk.blobs[2 * i + 1] for i in range(22)]
        hw, hb, par, fused = pk.blobs[44], float(pk.blobs[45][0]), {}, {}
    else:
        wts, bss, par, hw, hb, fused = bf16_blobs(m)
        sdd = {k: v.detach().cuda() for k, v in m.state_dict().items()}

    def buf(h, w, c):
        return torch.full((B, h, w, P * c), float("nan"), dtype=torch.bfloat16, device="cuda")

    def check(geom, acc_fn, store, out=None, pool=None, head=None):
        """acc_fn(sites, wrong) -> the model's accumulators (a wrong walk if `wrong`); store(acc, sites, out_sites) ->
        the stored values.  out = (tensor, plane stride, channel offset, C) the launch wrote; pool the pooled tensor;
        head = (prob, mask)."""
        sites = pick(geom)
        if sites is not None:
            sites = tuple(t.cuda() for t in sites)
            written = [t[..., o + p * ps:o + p * ps + c] for t, ps, o, c in [out] for p in range(P)] if out else []
            written += [pool] if pool is not None else []
            written += [head[0]] if head else []
            for t in written:
                assert not bool(torch.isnan(t).any()), f"{geom.case}: the launch left outputs unwritten (NaN)"
            if head:
                assert bool((head[1] <= 1).all()), f"{geom.case}: the launch left mask pixels unwritten"
        t0 = time.perf_counter()
        rs, half = sites, geom.kernel in HALF_GRID
        if sites is not None and pool is not None and not half:        # pooling at a site: its 2 x 2 block
            b, y, x = sites
            rs = tuple(torch.unique(torch.stack([b, y // 2, x // 2]), dim=1).unbind(0))
        os = rs if sites is None or (rs is sites and not half) else tm.class_sites(rs)
        acc = acc_fn(rs if half else os, False)
        y = store(acc, rs, os)
        if sites is not None:
            torch.cuda.synchronize()
            pick.report(geom, sites, rs, time.perf_counter() - t0)
        names = ("b", "y", "x", "c") if sites is None else ("site", "c")
        if head:
            en.assert_probs(_at(head[0], os), _at(head[1], os), y.cpu(), THRESH, geom.case, names[:-1])
            return
        t, ps, off, _ = out
        got = _at(t, os)
        if fp32:
            sm.assert_planes(got, y, ps, off, geom.case, others=False)
        else:
            en.assert_exact(got, y.cpu(), geom.case, names)
        if pool is not None:
            yp = tm.pool_bf16(y, blocks=sites is not None)
            if fp32:
                sm.assert_planes(_at(pool, rs), yp, pool.shape[-1] // 3, 0, f"{geom.case}: pooled", others=False)
            else:
                en.assert_exact(_at(pool, rs), yp.cpu(), f"{geom.case}: pooled", names)
        if sites is not None and geom.kernel in teeth:
            teeth.discard(geom.kernel)
            yw = store(acc_fn(rs if half else os, True), rs, os)
            ref = sm.join(got, ps, yw.shape[-1], off) if fp32 else got.double()
            ywr = yw if fp32 else yw.float().bfloat16().double()
            pick.wrong[geom.kernel] = (int((ref != ywr).sum()), ref.numel())
            print(f"{geom.case}: a wrong walk of {geom.kernel} changes {pick.wrong[geom.kernel][0]} of "
                  f"{ref.numel()} outputs")

    def conv(i, epi, relu, h, w, cin, cout, d, src, ss, dst=None, ds=0, doff=0, pool=None, prob=None, mask=None):
        wpar = par.get(i)
        kw = dict(kind=L.DC_KIND_CONV3X3, epilogue=epi, relu=relu, B=B, H=h, W=w, Cin=cin, Cout=cout, dilation=d,
                  in_=src.data_ptr(), in_stride=src.shape[-1], weight=wts[i].data_ptr(), bias=bss[i].data_ptr())
        if fp32:
            kw.update(planes=3, in_plane_stride=ss, out_plane_stride=ds)
        elif wpar is not None:
            kw.update(weight_par=wpar.data_ptr())
        if dst is not None:
            kw.update(out=dst.data_ptr(), out_stride=dst.shape[-1], out_offset=doff)
        if pool is not None:
            kw.update(pool_out=pool.data_ptr(), pool_stride=pool.shape[-1], pool_plane_stride=cout if fp32 else 0)
        head = epi == L.DC_EPI_HEAD
        if head:
            kw.update(head_w=hw.data_ptr(), head_b=hb, thresh=THRESH, prob_out=prob.data_ptr(), mask_out=mask.data_ptr())
        en.conv_tc(**kw)
        xs = [src[..., p * ss:p * ss + cin] for p in range(P)]
        bias = bss[i].double()
        case = f"{name} layer {i}"
        par2 = wpar is not None and fam == "auto" and d == 1          # launch_conv_tc's test for conv_par2_kernel
        if fp32:
            ws = wts[i].double().reshape(cout, 9, 3, cin).permute(2, 0, 1, 3)
            kernel, tile = "split", (8, 16)
        else:
            ws = [wts[i].double().reshape(cout, 9, cin)]
            if par2:
                kernel, tile = "par2", (16, 8)
            elif fam == "auto" and d <= 4:
                kernel, tile = ("pair" if cin >= 128 else "pair, Cin 64"), (16, 8)
            else:
                kernel, tile = f"per-tap d{d}", (8, 16)
        tm.assert_normal_products(xs, ws)
        if par2:
            wc = ws[0].reshape(cout, 3, 3, cin).permute(1, 2, 0, 3)
            geom = Geom(case, B, h // 2, w // 2, 1, tile, 4 * 36 * 16 * cout, kernel)

            def acc_fn(s, wrong):
                return tm.class_acc(None, xs[0], None, wc, tm.upf_walks(tm.PAR_CHUNKS, reverse_groups=wrong), sites=s)
        else:
            order = "chunk" if kernel.startswith("pair") else "tap"
            cost = 9 * len(sm.TERMS if fp32 else ((0, 0),)) * cin * cout * (4 if pool is not None else 1)
            geom = Geom(case, B, h, w, d, tile, cost, kernel)

            def acc_fn(s, wrong):
                if fp32:
                    return tm.run_steps(tm.conv_steps(xs, ws, d, sm.TERMS[::-1] if wrong else sm.TERMS, sites=s))
                o = {"tap": "chunk", "chunk": "tap"}[order] if wrong else order
                return tm.run_steps(tm.conv_steps(xs, ws, d, order=o, sites=s))

        def store(acc, rs, os):
            if head:
                return tm.head_logit(tm.store_split(acc, bias, True), hw, hb)
            return (tm.store_split if fp32 else tm.store_bf16)(acc, bias, relu)

        check(geom, acc_fn, store, None if head else (dst, ds, doff, cout), pool, (prob, mask) if head else None)

    def stem(dst):
        """The bf16 forward's first layer: dc_stem on the u8 grey or fp32 frames."""
        dev = u8 if in_kind == 1 else x32
        s = L.StemArgs(in_kind, B, H, W, 64, dil[0], dev.data_ptr(), wts[0].data_ptr(), bss[0].data_ptr(),
                       dst.data_ptr(), 64, 0)
        L.check(L.load().dc_stem(ctypes.byref(s), L.stream_ptr()))
        torch.cuda.synchronize()
        x = u8[:, None] if in_kind == 1 else x32.bfloat16()
        wk = tm.stem_weights(wts[0].double(), in_kind)
        geom = Geom(f"{name} stem {in_kind}", B, H, W, dil[0], (8, 16), wk.numel(), "stem")
        check(geom, lambda s, wrong: tm.run_steps(tm.stem_steps(tm.stem_cols(x, dil[0], s), wk)),
              lambda acc, rs, os: tm.store_bf16(acc, bss[0].double(), True), (dst, 0, 0, 64))

    def upconv(i, h, w, cin, cout, src, ss, dst, ds):
        """The fp32 forward's transposed conv (split, UPSCATTER) into channels [0, cout) of the [up | enc] buffer."""
        en.conv_tc(kind=L.DC_KIND_UPCONV2, epilogue=L.DC_EPI_UPSCATTER, relu=0, B=B, H=h, W=w, Cin=cin, Cout=cout,
                   dilation=1, in_=src.data_ptr(), in_stride=src.shape[-1], weight=wts[i].data_ptr(),
                   bias=bss[i].data_ptr(), out=dst.data_ptr(), out_stride=dst.shape[-1], out_offset=0, planes=3,
                   in_plane_stride=ss, out_plane_stride=ds)
        xs = [src[..., p * ss:p * ss + cin] for p in range(3)]
        ws = wts[i].double().reshape(4 * cout, 3, cin).permute(1, 0, 2)
        tm.assert_normal_products(xs, ws)
        bias = bss[i].double().repeat(4)

        def store(acc, rs, os):
            y = tm.store_split(acc, bias, False)
            if rs is None:
                return y.reshape(B, h, w, 2, 2, cout).permute(0, 1, 3, 2, 4, 5).reshape(B, 2 * h, 2 * w, cout)
            return y.view(-1, 4, cout).transpose(0, 1).reshape(-1, cout)      # class-major, as class_sites

        geom = Geom(f"{name} layer {i}", B, h, w, 1, (8, 16), 6 * cin * 4 * cout, "split upconv")
        check(geom, lambda s, wrong: tm.run_steps(tm.upconv_steps(xs, ws, sm.TERMS[::-1] if wrong else sm.TERMS, s)),
              store, (dst, ds, 0, cout))

    def upfused(lvl, h, w, c, src, skip, dst):
        """The bf16 forward's upconv + dec.0 of a level: conv_upfused2_kernel (level 1) or conv_upfused_wide_kernel."""
        wx, wsk, b9 = fused[lvl]
        comp, skipw, bias9 = fused_level_blobs(sdd, lvl, m._bn_eps(f"dec{lvl}", 1))
        if lvl == 1:
            assert torch.equal(pack_upfused(comp, skipw), wx)
        else:
            assert all(torch.equal(p, q) for p, q in zip(pack_upfused_wide(comp, skipw), (wx, wsk)))
        assert torch.equal(bias9, b9)
        a = L.UpfuseArgs()
        a.B, a.H, a.W, a.channels = B, h // 2, w // 2, c
        a.x, a.x_stride, a.skip, a.skip_stride = src.data_ptr(), 2 * c, skip.data_ptr(), c
        a.weight, a.bias9, a.relu = wx.data_ptr(), b9.data_ptr(), 1
        if wsk is not None:
            a.weight_skip = wsk.data_ptr()
        a.out, a.out_stride, a.out_offset = dst.data_ptr(), c, 0
        L.check(L.load().dc_conv_upfused(ctypes.byref(a), L.stream_ptr()))
        torch.cuda.synchronize()
        comp, skipw = comp.double(), skipw.double()
        tm.assert_normal_products([src, skip], [comp, skipw])
        walks = tm.upf_walks(tm.UPF_CHUNKS) if lvl == 1 else tm.wide_walks(c)
        wrong = tm.skip_first(walks) if lvl == 1 else tm.wide_walks(c, reverse_groups=True)
        geom = Geom(f"{name} fused level {lvl}", B, h // 2, w // 2, 1, (16, 8), 4 * len(walks[0]) * 16 * c,
                    "fused" if lvl == 1 else "fused wide")
        check(geom, lambda s, bad: tm.class_acc(src, skip, comp, skipw, wrong if bad else walks, sites=s),
              lambda acc, rs, os: tm.store_border_bf16(acc, bias9.double(), True, os, (h, w)), (dst, 0, 0, c))

    a = [buf(H >> l, W >> l, 64 << l) for l in range(5)]
    # fp32: [up | enc] buffers of both halves; bf16: the skip half alone (the fused kernels read the upconv input)
    cat = [buf(H >> l, W >> l, (128 if fp32 else 64) << l) for l in range(4)]
    pool = [buf(H >> (l + 1), W >> (l + 1), 64 << l) for l in range(4)]
    if fp32:
        xin = torch.zeros(B, H, W, 192, dtype=torch.bfloat16)
        for p, pl in enumerate(sm.split64(x32.cpu().permute(0, 2, 3, 1).double())):
            xin[..., 64 * p:64 * p + 3] = pl.bfloat16()
        conv(0, L.DC_EPI_STORE, 1, H, W, 64, 64, dil[0], xin.cuda(), 64, a[0], 64)
    else:
        stem(a[0])
    conv(1, L.DC_EPI_STORE_POOL, 1, H, W, 64, 64, dil[0], a[0], 64, cat[0], 128 if fp32 else 0, 64 if fp32 else 0,
         pool[0])
    for l in range(1, 4):
        h, w, c = H >> l, W >> l, 64 << l
        conv(2 * l, L.DC_EPI_STORE, 1, h, w, c // 2, c, dil[l], pool[l - 1], c // 2, a[l], c)
        conv(2 * l + 1, L.DC_EPI_STORE_POOL, 1, h, w, c, c, dil[l], a[l], c, cat[l], 2 * c if fp32 else 0,
             c if fp32 else 0, pool[l])
    bott = buf(H >> 4, W >> 4, 1024)
    conv(8, L.DC_EPI_STORE, 1, H >> 4, W >> 4, 512, 1024, dil[4], pool[3], 512, a[4], 1024)
    conv(9, L.DC_EPI_STORE, 1, H >> 4, W >> 4, 1024, 1024, dil[4], a[4], 1024, bott, 1024)
    src = bott
    prob = torch.full((B, H, W), float("nan"), device="cuda")
    mask = torch.full((B, H, W), 7, dtype=torch.uint8, device="cuda")
    for l in (3, 2, 1, 0):
        h, w, c = H >> l, W >> l, 64 << l
        ad = buf(h, w, c)
        if fp32:
            upconv(10 + 3 * (3 - l), h // 2, w // 2, 2 * c, c, src, 2 * c, cat[l], 2 * c)
            conv(11 + 3 * (3 - l), L.DC_EPI_STORE, 1, h, w, 2 * c, c, 1, cat[l], 2 * c, ad, c)
        else:
            upfused(l + 1, h, w, c, src, cat[l], ad)
        if l > 0:
            src = buf(h, w, c)
            conv(12 + 3 * (3 - l), L.DC_EPI_STORE, 1, h, w, c, c, 1, ad, c, src, c)
        else:
            conv(21, L.DC_EPI_HEAD, 1, h, w, c, c, 1, ad, c, prob=prob, mask=mask)
    return prob, mask


HALF_GRID = {"par2", "fused", "fused wide", "split upconv"}     # kernels whose sites stand for 2 x 2 output blocks
