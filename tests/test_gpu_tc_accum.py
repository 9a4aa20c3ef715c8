"""GPU: how tcgen05 kind::f16 MMAs add into an fp32 accumulator, and real-valued layers held to that model bit for bit.

Probes (tests/tc_accum_model.py, "probes"): the split kernel with three output planes, bias -0.0 and no ReLU stores the
accumulator's fp32 bits exactly, so one launch of B = 1, H = 8, W = 16, Cin = 64, dilation 16 runs 128 x N independent
experiments of 24 MMA steps each.  Every output must equal tc_accum_model.MEASURED; each probe family prints which
candidate models (tc_accum_model.CANDIDATES) it rules out, and together they must rule out every one.

Layers: real-valued operands (ReLU-like activations, He-scaled weights, real biases), which the exact tier of
test_gpu_exact.py / test_gpu_fp32.py cannot use, each stored output equal to the model's replay of the kernel's K walk
and epilogue, inside sentinel guards, with unread channels holding bf16 NaN: the split kernel's epilogues, the bf16
per-tap / halo / pair kernels (STORE and STORE_POOL), the unfused bf16 transposed conv, the stem, conv_par2_kernel
(STORE, STORE_POOL, HEAD) and the fused upconv + conv kernels (conv_upfused2_kernel, conv_upfused_wide_kernel).
Forward: the calibrated network's fp32 forward and its default bf16 forward, each as a chain of single-layer launches,
every layer equal to the model's replay of its own GPU input, and m(x) bit-identical to the chain.  The replay runs in
torch float64 on the GPU as a plain reference."""

import pytest
import torch

import exact_net as en
import split_model as sm
import tc_accum_model as tm
import tc_chain as tc
from exact_net import family  # noqa: F401  (fixture)
from test_gpu_exact import PARITY_CASES, UPFUSED_CASES, WIDE_CASES
from test_gpu_fp32 import CONV_CASES, POOL_CASES

pytestmark = pytest.mark.gpu

THRESH = 0.3


def _L():
    from unet_dc_segmentation_b200 import _lib
    return _lib


# ----------------------------------------------------------------------------- probes

def probe_launch(A, W):
    """The probe launch (tc_accum_model): A [128, 3, 64], W [N, 3, 64] bf16 values -> the fp32 accumulators [128, N]
    (float64), read back from the three stored planes (disjoint bit ranges: their float64 sum is exact)."""
    L = _L()
    N = W.shape[0]
    xin = A.bfloat16().reshape(1, 8, 16, 192).contiguous().cuda()
    assert torch.equal(xin.cpu().double().reshape(128, 3, 64), A), "probe activations are not bf16 values"
    blob = torch.full((N, 9, 3, 64), float("nan"), dtype=torch.bfloat16)     # taps other than the centre: never read
    blob[:, 4] = W.bfloat16()
    assert torch.equal(blob[:, 4].double(), W), "probe weights are not bf16 values"
    bias = torch.full((N,), -0.0, dtype=torch.float32).cuda()
    raw, out = en.guarded((1, 8, 16, 3 * N), torch.bfloat16)
    en.conv_tc(kind=L.DC_KIND_CONV3X3, epilogue=L.DC_EPI_STORE, relu=0, B=1, H=8, W=16, Cin=64, Cout=N, dilation=16,
              in_=xin.data_ptr(), in_stride=192, weight=blob.reshape(N, 27 * 64).cuda().data_ptr(), bias=bias.data_ptr(),
              out=out.data_ptr(), out_stride=3 * N, out_offset=0, planes=3, in_plane_stride=64, out_plane_stride=N)
    en.check_guards(raw, "probe")
    o = out.cpu().reshape(128, 3, N).double()
    acc = o.sum(1)
    zero = acc == 0
    return torch.where(zero, o[:, 0], acc)          # keeps the sign of a zero accumulator (hi plane of -0.0 is -0.0)


def _same(got, want):
    return (got == want) & (torch.signbit(got) == torch.signbit(want))


def _report(got, want, labels, case, ok):
    bad = ~_same(got, want) & ok
    if bool(bad.any()):
        p, n = (int(v) for v in bad.nonzero()[0])
        raise AssertionError(f"{case}: {int(bad.sum())}/{bad.numel()} accumulators differ from the model; first: probe "
                             f"{labels[n]!r} at pixel scale {float(tm.probe_activations()[p, 0, 0])!r}: got "
                             f"{float(got[p, n])!r}, model {float(want[p, n])!r}")


def test_accumulator_probes(cuda_device):
    """Every probe family on every pixel scale equals MEASURED wherever all products are normal fp32 numbers; together
    the families rule out every candidate."""
    A = tm.probe_activations()
    ruled_out = set()
    for fam, rows in tm.probe_rows().items():
        labels = [r[0] for r in rows]
        W = torch.stack([r[1] for r in rows])
        W = torch.cat([W, torch.zeros((-len(rows)) % 64, 3, 64, dtype=torch.float64)])
        got = torch.cat([probe_launch(A, W[i:i + 256]) for i in range(0, W.shape[0], 256)], 1)[:, :len(rows)]
        want = tm.run_steps(tm.probe_steps(A, W[:len(rows)]))
        ok = tm.compared(A, W[:len(rows)], want)
        _report(got, want, labels, f"probes {fam}", ok)
        out = [name for name, c in tm.CANDIDATES.items()
               if not bool((_same(got, tm.run_steps(tm.probe_steps(A, W[:len(rows)]), c)) | ~ok).all())]
        print(f"{fam}: {len(rows)} rows x 128 scales, rules out {out}")
        ruled_out |= set(out)
    assert ruled_out == set(tm.CANDIDATES), f"no probe rules out {set(tm.CANDIDATES) - ruled_out}"


@pytest.mark.parametrize("seed", range(4))
def test_accumulator_random_operands(cuda_device, seed):
    """Arbitrary bf16 values in all three planes, exponents over +-4, +-12 and +-30: 24 steps of 16 products each."""
    g = torch.Generator().manual_seed(seed)
    for e in (4, 12, 30):
        A, W = (tm.random_bf16(s, e, g) for s in ((128, 3, 64), (256, 3, 64)))
        got, want = probe_launch(A, W), tm.run_steps(tm.probe_steps(A, W))
        _report(got, want, [f"random e{e} row {n}" for n in range(256)], f"random operands e{e} seed {seed}",
                tm.compared(A, W, want))


# ----------------------------------------------------------------------------- real-valued split layers

def _planes(x64):
    return [p.double() for p in sm.split64(x64)]


def _split_conv_acc(x, blob, cin, cout, d):
    """The model's fp32 accumulator of conv_tc_split_kernel on the GPU: planes of x against the packed blob's planes."""
    ws = blob.double().reshape(cout, 9, 3, cin).permute(2, 0, 1, 3).cuda()
    xs = [p.cuda() for p in _planes(x)]
    tm.assert_normal_products(xs, ws)
    return tm.run_steps(tm.conv_steps(xs, ws, d, sm.TERMS))


@pytest.mark.parametrize("i", range(len(CONV_CASES)))
@pytest.mark.parametrize("relu", [0, 1])
def test_split_conv_store_real(cuda_device, i, relu):
    from unet_dc_segmentation_b200.model import pack_conv3x3_split
    L = _L()
    B, H, W, cin, cout, d = CONV_CASES[i]
    x, w, b = tm.real_operands(B, H, W, cin, cout, seed=10 * i + relu)
    wp = pack_conv3x3_split(w)
    want = tm.store_split(_split_conv_acc(x, wp, cin, cout, d), b.cuda(), relu).cpu()
    ips, ops = cin + 64, cout + 32
    xin = sm.plane_buffer(x, ips, 3 * ips).cuda()
    raw, out = en.guarded((B, H, W, 3 * ops), torch.bfloat16)
    bias = b.float().cuda()
    en.conv_tc(kind=L.DC_KIND_CONV3X3, epilogue=L.DC_EPI_STORE, relu=relu, B=B, H=H, W=W, Cin=cin, Cout=cout,
              dilation=d, in_=xin.data_ptr(), in_stride=3 * ips, weight=wp.cuda().data_ptr(), bias=bias.data_ptr(),
              out=out.data_ptr(), out_stride=3 * ops, out_offset=16, planes=3, in_plane_stride=ips, out_plane_stride=ops)
    case = f"real split conv {cin}->{cout} d{d} {B}x{H}x{W} relu={relu}"
    sm.assert_planes(out, want, ops, 16, case)
    en.check_guards(raw, case)


@pytest.mark.parametrize("i", range(len(POOL_CASES)))
def test_split_pool_real(cuda_device, i):
    from unet_dc_segmentation_b200.model import pack_conv3x3_split
    L = _L()
    B, H, W, c, d = POOL_CASES[i]
    x, w, b = tm.real_operands(B, H, W, c, c, seed=300 + i)
    wp = pack_conv3x3_split(w)
    want = tm.store_split(_split_conv_acc(x, wp, c, c, d), b.cuda(), True).cpu()
    xin = sm.plane_buffer(x, c, 3 * c).cuda()
    raw, out = en.guarded((B, H, W, 6 * c), torch.bfloat16)
    praw, pooled = en.guarded((B, H // 2, W // 2, 3 * c + 64), torch.bfloat16)
    bias = b.float().cuda()
    en.conv_tc(kind=L.DC_KIND_CONV3X3, epilogue=L.DC_EPI_STORE_POOL, relu=1, B=B, H=H, W=W, Cin=c, Cout=c, dilation=d,
              in_=xin.data_ptr(), in_stride=3 * c, weight=wp.cuda().data_ptr(), bias=bias.data_ptr(), out=out.data_ptr(),
              out_stride=6 * c, out_offset=c, pool_out=pooled.data_ptr(), pool_stride=3 * c + 64, planes=3,
              in_plane_stride=c, out_plane_stride=2 * c, pool_plane_stride=c)
    case = f"real split pool {c} d{d} {B}x{H}x{W}"
    sm.assert_planes(out, want, 2 * c, c, case)
    en.check_guards(raw, case)
    sm.assert_planes(pooled, sm.pool_split(want), c, 0, f"{case}: pooled")
    en.check_guards(praw, f"{case}: pooled")


@pytest.mark.parametrize("c", [64, 128, 256, 512])
def test_split_upscatter_real(cuda_device, c):
    from unet_dc_segmentation_b200.model import pack_upconv_split
    L = _L()
    B, H, W = 2, 6, 10
    x, w, b = tm.real_operands(B, H, W, 2 * c, c, seed=c, upconv=True)
    wp = pack_upconv_split(w)
    ws = wp.double().reshape(4 * c, 3, 2 * c).permute(1, 0, 2).cuda()
    acc = tm.run_steps(tm.upconv_steps([p.cuda() for p in _planes(x)], ws, sm.TERMS))
    y = tm.store_split(acc, b.repeat(4).cuda(), False).cpu()
    want = y.reshape(B, H, W, 2, 2, c).permute(0, 1, 3, 2, 4, 5).reshape(B, 2 * H, 2 * W, c)
    xin = sm.plane_buffer(x, 2 * c, 6 * c).cuda()
    raw, out = en.guarded((B, 2 * H, 2 * W, 6 * c), torch.bfloat16)
    bias = b.float().cuda()
    en.conv_tc(kind=L.DC_KIND_UPCONV2, epilogue=L.DC_EPI_UPSCATTER, relu=0, B=B, H=H, W=W, Cin=2 * c, Cout=c,
              dilation=1, in_=xin.data_ptr(), in_stride=6 * c, weight=wp.cuda().data_ptr(), bias=bias.data_ptr(),
              out=out.data_ptr(), out_stride=6 * c, out_offset=0, planes=3, in_plane_stride=2 * c,
              out_plane_stride=2 * c)
    case = f"real split upconv {2 * c}->{c}"
    sm.assert_planes(out, want, 2 * c, 0, case)
    en.check_guards(raw, case)


@pytest.mark.parametrize("cin,d", [(64, 1), (128, 1), (64, 3)])
def test_split_head_real(cuda_device, cin, d):
    """HEAD: the model's features, the exact fmaf chain to the logit; probabilities within 1e-6 of its sigmoid."""
    from unet_dc_segmentation_b200.model import pack_conv3x3_split
    L = _L()
    B, H, W = 2, 16, 24
    x, w, b = tm.real_operands(B, H, W, cin, 64, seed=500 + cin + d)
    wp = pack_conv3x3_split(w)
    feat = tm.store_split(_split_conv_acc(x, wp, cin, 64, d), b.cuda(), True)
    g = torch.Generator().manual_seed(cin + d)
    hw = (torch.randn(64, generator=g) * 0.3).float()
    hb = float(torch.tensor(-float((feat.cpu() @ hw.double()).mean())).float())
    logits = tm.head_logit(feat, hw.cuda(), hb).cpu()
    xin = sm.plane_buffer(x, cin + 64, 3 * cin + 192).cuda()
    bias, hwd = b.float().cuda(), hw.cuda()
    praw, prob = en.guarded((B, H, W), torch.float32)
    mraw, mask = en.guarded((B, H, W), torch.uint8)
    en.conv_tc(kind=L.DC_KIND_CONV3X3, epilogue=L.DC_EPI_HEAD, relu=1, B=B, H=H, W=W, Cin=cin, Cout=64, dilation=d,
              in_=xin.data_ptr(), in_stride=3 * cin + 192, weight=wp.cuda().data_ptr(), bias=bias.data_ptr(),
              head_w=hwd.data_ptr(), head_b=hb, thresh=THRESH, prob_out=prob.data_ptr(), mask_out=mask.data_ptr(),
              planes=3, in_plane_stride=cin + 64)
    case = f"real split head {cin} d{d}"
    en.assert_probs(prob, mask, logits, THRESH, case)
    en.check_guards(praw, case)
    en.check_guards(mraw, case)


# ----------------------------------------------------------------------------- real-valued bf16 layers

# (B, H, W, Cin, Cout, dilation, family, K order): pair kernel (auto, d <= 4, BN 64 / 128 / 256 resident or streamed),
# single-CTA halo (auto, Cout = 64 with long K), per-tap kernel (generic; auto at dilation 8 / 16)
BF16_CASES = [(1, 16, 16, 64, 64, 1, "auto", "chunk"), (2, 24, 40, 128, 128, 2, "auto", "chunk"),
              (1, 32, 24, 64, 128, 4, "auto", "chunk"), (1, 16, 32, 256, 256, 1, "auto", "chunk"),
              (1, 12, 20, 512, 512, 3, "auto", "chunk"), (1, 12, 20, 256, 64, 3, "auto", "chunk"),
              (1, 16, 16, 64, 64, 1, "generic", "tap"), (2, 24, 40, 128, 256, 2, "generic", "tap"),
              (1, 16, 16, 256, 512, 8, "auto", "tap"), (2, 8, 8, 512, 512, 16, "auto", "tap"),
              (1, 16, 32, 1024, 512, 1, "generic", "tap")]


@pytest.mark.parametrize("i", range(len(BF16_CASES)))
def test_bf16_conv_store_real(cuda_device, family, i):
    from unet_dc_segmentation_b200.model import pack_conv3x3
    L = _L()
    B, H, W, cin, cout, d, fam, order = BF16_CASES[i]
    family(fam)
    x, w, b = tm.real_operands(B, H, W, cin, cout, seed=700 + i)
    x = x.bfloat16().double()
    wp = pack_conv3x3(w)
    ws = wp.double().reshape(cout, 9, cin).cuda()
    relu = i % 2 == 0
    want = tm.store_bf16(tm.run_steps(tm.conv_steps([x.cuda()], [ws], d, order=order)), b.cuda(), relu).cpu()
    xin = torch.full((B, H, W, cin + 64), float("nan"), dtype=torch.bfloat16)
    xin[..., 32:32 + cin] = x.bfloat16()
    xin = xin.cuda()
    raw, out = en.guarded((B, H, W, cout + 64), torch.bfloat16)
    bias = b.float().cuda()
    en.conv_tc(kind=L.DC_KIND_CONV3X3, epilogue=L.DC_EPI_STORE, relu=int(relu), B=B, H=H, W=W, Cin=cin, Cout=cout,
              dilation=d, in_=xin[..., 32:].data_ptr(), in_stride=cin + 64, weight=wp.cuda().data_ptr(),
              bias=bias.data_ptr(), out=out.data_ptr(), out_stride=cout + 64, out_offset=32)
    case = f"real bf16 conv {cin}->{cout} d{d} {B}x{H}x{W} {fam} relu={relu}"
    en.assert_exact(out[..., 32:32 + cout], want, case)
    en.check_outside(raw, out, 32, cout, case)


@pytest.mark.parametrize("cin,cout", [(128, 64), (256, 128), (512, 256), (1024, 512)])
def test_bf16_upconv_real(cuda_device, cin, cout):
    """The unfused bf16 transposed conv (GEMM N = 4 Cout, one tap): (chunk, k16) into a channel slice."""
    from unet_dc_segmentation_b200.model import pack_upconv
    L = _L()
    B, H, W = 2, 6, 10
    x, w, b = tm.real_operands(B, H, W, cin, cout, seed=900 + cin, upconv=True)
    x = x.bfloat16().double()
    wp = pack_upconv(w)
    acc = tm.run_steps(tm.upconv_steps([x.cuda()], [wp.double().cuda()]))
    y = tm.store_bf16(acc, b.repeat(4).cuda(), False).cpu()
    want = y.reshape(B, H, W, 2, 2, cout).permute(0, 1, 3, 2, 4, 5).reshape(B, 2 * H, 2 * W, cout)
    xin = torch.full((B, H, W, cin + 64), float("nan"), dtype=torch.bfloat16)
    xin[..., 32:32 + cin] = x.bfloat16()
    xin = xin.cuda()
    raw, out = en.guarded((B, 2 * H, 2 * W, cout + 64), torch.bfloat16)
    bias = b.float().cuda()
    en.conv_tc(kind=L.DC_KIND_UPCONV2, epilogue=L.DC_EPI_UPSCATTER, relu=0, B=B, H=H, W=W, Cin=cin, Cout=cout,
               dilation=1, in_=xin[..., 32:].data_ptr(), in_stride=cin + 64, weight=wp.cuda().data_ptr(),
               bias=bias.data_ptr(), out=out.data_ptr(), out_stride=cout + 64, out_offset=32)
    case = f"real bf16 upconv {cin}->{cout}"
    en.assert_exact(out[..., 32:32 + cout], want, case)
    en.check_outside(raw, out, 32, cout, case)


@pytest.mark.parametrize("in_kind", [0, 1, 2])
@pytest.mark.parametrize("d", [1, 3])
def test_stem_real(cuda_device, in_kind, d):
    """dc_stem for f32 NCHW, u8 grey and u8 HWC frames with real-valued fp32 weights: the kernel's own fp32 -> bf16
    weight conversion (1/255 for u8, the grey channel sum), K = 27 -> 32 or 9 -> 16, bias + ReLU, bf16 store."""
    import ctypes
    L = _L()
    B, H, W = 2, 20, 36
    g = torch.Generator().manual_seed(40 + 3 * in_kind + d)
    w = (torch.randn(64, 27, generator=g) * (2.0 / 27) ** 0.5).float()
    b = (torch.randn(64, generator=g) * 0.1).float()
    if in_kind == 0:
        xf = torch.rand(B, 3, H, W, generator=g)
        x64, dev = xf.bfloat16().double(), xf.contiguous().cuda()
    else:
        u = torch.randint(0, 256, (B, H, W) if in_kind == 1 else (B, H, W, 3), generator=g, dtype=torch.uint8)
        x64 = u.double()[:, None] if in_kind == 1 else u.permute(0, 3, 1, 2).double()
        dev = u.cuda()
    acc = tm.run_steps(tm.stem_steps(tm.stem_cols(x64, d).cuda(), tm.stem_weights(w.double(), in_kind).cuda()))
    want = tm.store_bf16(acc, b.double().cuda(), True).cpu()
    wdev, bias = w.cuda(), b.cuda()
    raw, out = en.guarded((B, H, W, 128), torch.bfloat16)
    a = L.StemArgs(in_kind, B, H, W, 64, d, dev.data_ptr(), wdev.data_ptr(), bias.data_ptr(), out.data_ptr(), 128, 32)
    L.check(L.load().dc_stem(ctypes.byref(a), L.stream_ptr()))
    torch.cuda.synchronize()
    case = f"real stem in_kind={in_kind} d{d}"
    en.assert_exact(out[..., 32:96], want, case)
    en.check_outside(raw, out, 32, 64, case)


# ----------------------------------------------------------------------------- the fp32 forward as a chain of layers

@pytest.mark.parametrize("B,H,W", [(1, 64, 64), (2, 48, 80)])
def test_fp32_forward_chain(cuda_device, B, H, W):
    """The calibrated network's fp32 forward run as the forward runs it (split input, 18 convs, 4 transposed convs into
    [up | enc] plane buffers, HEAD), one dc_conv_tc launch at a time (tc_chain.forward_chain): every layer equals the
    model's replay of its own GPU input bit for bit, and m(x) / predict_u8 give exactly the chain's probabilities and
    mask.  The model forward is then the GPU forward, so the model accounts for all of its error; the printed line
    compares it with float64."""
    import oracle
    import test_gpu_fp32 as t32
    sd = t32._calibrated()
    m = t32._model(__import__("unet_dc_segmentation_b200").UNetDC, sd)
    u8 = t32._frames(B, max(H, W), 60)[:, :H, :W].contiguous()
    x32 = torch.from_numpy(u8.numpy().astype("float32") / __import__("numpy").float32(255))[:, None]
    x32 = x32.expand(B, 3, H, W).contiguous()
    prob, mask = tc.forward_chain(m, "fp32", "auto", u8.cuda(), x32.cuda(), tc.whole_map)
    mk, pr = m.predict_u8(u8.cuda(), THRESH, return_prob=True)
    assert torch.equal(pr[:, 0], prob) and torch.equal(mk, mask), "predict_u8 differs from the layer chain"
    assert torch.equal(m(x32.cuda())[:, 0], prob), "m(x) differs from the layer chain"
    p64 = sm.network(sd, x32)
    six = sm.network(sd, x32, terms=sm.TERMS)
    cpu = oracle.unetdc_forward(sd, x32)[:, 0].double()
    err = {k: float((v.double().cpu() - p64).abs().max()) for k, v in
           (("GPU forward = model forward", prob), ("six terms, exact sums", six), ("CPU fp32 network", cpu))}
    print(f"{B}x{H}x{W}: max |dp| vs float64: " + ", ".join(f"{k} {v:.3e}" for k, v in err.items()))


# ----------------------------------------------------------------------------- real-valued parity-class and fused layers

def _nan_buf(x64, width, off):
    """bf16 NHWC [..., width] on the device: x64 at channels [off, off + C), bf16 NaN everywhere else."""
    buf = torch.full(tuple(x64.shape[:-1]) + (width,), float("nan"), dtype=torch.bfloat16)
    buf[..., off:off + x64.shape[-1]] = x64.bfloat16()
    return buf.cuda()


@pytest.mark.parametrize("i", range(len(PARITY_CASES)))
def test_bf16_par2_real(cuda_device, i):
    """conv_par2_kernel (weight_par) on a real-valued 64 -> 64 layer: STORE without ReLU into a slice, STORE_POOL with
    ReLU and HEAD, each equal to the model's replay of the parity-class walk (tc_accum_model.upf_walks(PAR_CHUNKS))."""
    from unet_dc_segmentation_b200.model import pack_conv3x3, pack_par3x3
    L = _L()
    B, H, W = PARITY_CASES[i]
    x, w, b = tm.real_operands(B, H, W, 64, 64, seed=1300 + i)
    x = x.bfloat16().double()
    ws = w.permute(2, 3, 0, 1).bfloat16().double()
    tm.assert_normal_products([x], [ws])
    acc = tm.class_acc(None, x.cuda(), None, ws.cuda(), tm.upf_walks(tm.PAR_CHUNKS))
    xin = _nan_buf(x, 128, 32)
    wp, wpar, bias = pack_conv3x3(w).cuda(), pack_par3x3(w.float()).cuda(), b.float().cuda()
    common = dict(kind=L.DC_KIND_CONV3X3, B=B, H=H, W=W, Cin=64, Cout=64, dilation=1, in_=xin[..., 32:].data_ptr(),
                  in_stride=128, weight=wp.data_ptr(), bias=bias.data_ptr(), weight_par=wpar.data_ptr())
    case = f"real par2 {B}x{H}x{W}"
    raw, out = en.guarded((B, H, W, 128), torch.bfloat16)
    en.conv_tc(epilogue=L.DC_EPI_STORE, relu=0, out=out.data_ptr(), out_stride=128, out_offset=32, **common)
    en.assert_exact(out[..., 32:96], tm.store_bf16(acc, b.cuda(), False).cpu(), f"{case}: store")
    en.check_outside(raw, out, 32, 64, f"{case}: store")
    raw, out = en.guarded((B, H, W, 128), torch.bfloat16)
    praw, pooled = en.guarded((B, H // 2, W // 2, 64), torch.bfloat16)
    en.conv_tc(epilogue=L.DC_EPI_STORE_POOL, relu=1, out=out.data_ptr(), out_stride=128, out_offset=32,
               pool_out=pooled.data_ptr(), pool_stride=64, **common)
    y = tm.store_bf16(acc, b.cuda(), True).cpu()
    en.assert_exact(out[..., 32:96], y, f"{case}: store_pool")
    en.check_outside(raw, out, 32, 64, f"{case}: store_pool")
    en.assert_exact(pooled, tm.pool_bf16(y), f"{case}: pooled")
    en.check_guards(praw, f"{case}: pooled")
    feat = tm.store_split(acc, b.cuda(), True)
    g = torch.Generator().manual_seed(1400 + i)
    hw = (torch.randn(64, generator=g) * 0.3).float()
    hb = float(torch.tensor(-float((feat.cpu() @ hw.double()).mean())).float())
    logits = tm.head_logit(feat, hw.cuda(), hb).cpu()
    hwd = hw.cuda()
    praw, prob = en.guarded((B, H, W), torch.float32)
    mraw, mask = en.guarded((B, H, W), torch.uint8)
    en.conv_tc(epilogue=L.DC_EPI_HEAD, relu=1, head_w=hwd.data_ptr(), head_b=hb, thresh=THRESH,
               prob_out=prob.data_ptr(), mask_out=mask.data_ptr(), **common)
    en.assert_probs(prob, mask, logits, THRESH, f"{case}: head")
    en.check_guards(praw, f"{case}: head")
    en.check_guards(mraw, f"{case}: head")


def _upfused_real(C, B, Hh, Wh, seed, relu):
    """dc_conv_upfused on a real-valued level: x at channels [0, 2C) of a 2C + 64 wide buffer, skip at [64, 64 + C) of a
    C + 128 wide one (NaN elsewhere), the output in a slice; equal to the model's walk and border-class epilogue."""
    import ctypes
    from unet_dc_segmentation_b200.model import pack_upfused, pack_upfused_wide
    L = _L()
    x, s, comp, skipw, bias9 = tm.upfused_real_operands(C, B, Hh, Wh, seed)
    tm.assert_normal_products([x, s], [comp, skipw])
    walks = tm.upf_walks(tm.UPF_CHUNKS) if C == 64 else tm.wide_walks(C)
    want = tm.store_border_bf16(tm.class_acc(x.cuda(), s.cuda(), comp.cuda(), skipw.cuda(), walks), bias9.cuda(), relu).cpu()
    ws = None
    if C == 64:
        wx = pack_upfused(comp.bfloat16(), skipw.bfloat16()).cuda()
    else:
        wx, ws = (t.cuda() for t in pack_upfused_wide(comp.bfloat16(), skipw.bfloat16()))
    xin, skip = _nan_buf(x, 2 * C + 64, 0), _nan_buf(s, C + 128, 64)
    raw, out = en.guarded((B, 2 * Hh, 2 * Wh, C + 32), torch.bfloat16)
    b9 = bias9.float().cuda()
    a = L.UpfuseArgs()
    a.B, a.H, a.W, a.channels = B, Hh, Wh, C
    a.x, a.x_stride = xin.data_ptr(), 2 * C + 64
    a.skip, a.skip_stride = skip.data_ptr() + 2 * 64, C + 128
    a.weight, a.bias9, a.relu = wx.data_ptr(), b9.data_ptr(), int(relu)
    if ws is not None:
        a.weight_skip = ws.data_ptr()
    a.out, a.out_stride, a.out_offset = out.data_ptr(), C + 32, 16
    L.check(L.load().dc_conv_upfused(ctypes.byref(a), L.stream_ptr()))
    torch.cuda.synchronize()
    case = f"real upfused C={C} {B}x{Hh}x{Wh} relu={relu}"
    en.assert_exact(out[..., 16:16 + C], want, case)
    en.check_outside(raw, out, 16, C, case)


@pytest.mark.parametrize("i", range(len(UPFUSED_CASES)))
def test_bf16_upfused_real(cuda_device, i):
    """conv_upfused2_kernel (C = 64): tiles of 16 x 8 half-resolution pixels, ragged in either axis, B > 1."""
    B, Hh, Wh = UPFUSED_CASES[i]
    _upfused_real(64, B, Hh, Wh, 1100 + i, i % 2 == 0)


@pytest.mark.parametrize("i", range(len(WIDE_CASES)))
def test_bf16_upfused_wide_real(cuda_device, i):
    """conv_upfused_wide_kernel: C = 128 (BN = 128, two classes per pass), 256 and 512 (BN = 256, one class per pass)."""
    C, B, Hh, Wh = WIDE_CASES[i]
    _upfused_real(C, B, Hh, Wh, 1200 + i, i % 2 == 0)


def _bf16_order(fam, d):
    """K order of a bf16 3x3 layer outside conv_par2_kernel: the pair / halo kernels in auto at dilation <= 4, else the
    per-tap kernel (launch_conv_tc)."""
    return "chunk" if fam == "auto" and d <= 4 else "tap"


# enc2.3, enc3.3, enc4.3 of the default network (pair kernel, pair kernel, per-tap kernel in auto)
POOL_BF16_CASES = [(2, 24, 40, 128, 2), (1, 32, 24, 256, 4), (2, 16, 16, 512, 8)]


@pytest.mark.parametrize("fam", ["auto", "generic"])
@pytest.mark.parametrize("i", range(len(POOL_BF16_CASES)))
def test_bf16_pool_real(cuda_device, family, fam, i):
    """STORE_POOL of the bf16 pair / halo / per-tap kernels: the full-resolution store and the 2x2 max of it."""
    from unet_dc_segmentation_b200.model import pack_conv3x3
    L = _L()
    B, H, W, c, d = POOL_BF16_CASES[i]
    family(fam)
    x, w, b = tm.real_operands(B, H, W, c, c, seed=1500 + i)
    x = x.bfloat16().double()
    wp = pack_conv3x3(w)
    ws = wp.double().reshape(c, 9, c)
    tm.assert_normal_products([x], [ws])
    y = tm.store_bf16(tm.run_steps(tm.conv_steps([x.cuda()], [ws.cuda()], d, order=_bf16_order(fam, d))), b.cuda(), True).cpu()
    xin = _nan_buf(x, c + 64, 32)
    raw, out = en.guarded((B, H, W, 2 * c), torch.bfloat16)
    praw, pooled = en.guarded((B, H // 2, W // 2, c + 64), torch.bfloat16)
    bias = b.float().cuda()
    en.conv_tc(kind=L.DC_KIND_CONV3X3, epilogue=L.DC_EPI_STORE_POOL, relu=1, B=B, H=H, W=W, Cin=c, Cout=c, dilation=d,
               in_=xin[..., 32:].data_ptr(), in_stride=c + 64, weight=wp.cuda().data_ptr(), bias=bias.data_ptr(),
               out=out.data_ptr(), out_stride=2 * c, out_offset=c, pool_out=pooled.data_ptr(), pool_stride=c + 64)
    case = f"real bf16 pool {c} d{d} {B}x{H}x{W} {fam}"
    en.assert_exact(out[..., c:2 * c], y, case)
    en.check_outside(raw, out, c, c, case)
    en.assert_exact(pooled[..., :c], tm.pool_bf16(y), f"{case}: pooled")
    en.check_outside(praw, pooled, 0, c, f"{case}: pooled")


# ----------------------------------------------------------------------------- the bf16 forward as a chain of layers

@pytest.mark.parametrize("fam", ["auto", "generic"])
@pytest.mark.parametrize("B,H,W", [(1, 64, 64), (2, 48, 80)])
def test_bf16_forward_chain(cuda_device, family, fam, B, H, W):
    """The calibrated network's default bf16 forward run as dc_forward runs it (forward_impl, csrc/api.cu): the stem,
    enc1.3 STORE_POOL (conv_par2_kernel in auto), enc2-4 and the bottleneck, upconv + dec.0 fused for levels 4-2
    (conv_upfused_wide_kernel) and level 1 (conv_upfused2_kernel), each dec.3, dec1.3 HEAD (conv_par2_kernel in auto),
    one launch at a time from the model's own blobs (tc_chain.forward_chain).  Every layer equals the model's replay of
    its own GPU input bit for bit, and predict_u8 (u8 grey stem) and m(x) (fp32 stem) give exactly the chain's
    probabilities and mask.  Under family generic conv_par2_kernel and the pair / halo kernels are off
    (launch_conv_tc), the fused kernels are not."""
    import numpy as np
    import test_gpu_fp32 as t32
    from unet_dc_segmentation_b200 import UNetDC
    family(fam)
    sd = t32._calibrated()
    m = UNetDC()
    m.load_state_dict(sd)
    m = m.cuda().eval()
    u8 = t32._frames(B, max(H, W), 60)[:, :H, :W].contiguous()
    x32 = torch.from_numpy(u8.numpy().astype("float32") / np.float32(255))[:, None].expand(B, 3, H, W).contiguous()
    prob, mask = tc.forward_chain(m, "bf16", fam, u8.cuda(), x32.cuda(), tc.whole_map, in_kind=1)
    mk, pr = m.predict_u8(u8.cuda(), THRESH, return_prob=True)
    assert torch.equal(pr[:, 0], prob) and torch.equal(mk, mask), "predict_u8 differs from the layer chain"
    prob0, _ = tc.forward_chain(m, "bf16", fam, u8.cuda(), x32.cuda(), tc.whole_map, in_kind=0)
    assert torch.equal(m(x32.cuda())[:, 0], prob0), "m(x) differs from the layer chain"
    p64 = sm.network(sd, x32)
    err = {k: float((v.double().cpu() - p64).abs().max()) for k, v in (("u8 grey entry", prob), ("fp32 entry", prob0))}
    print(f"{B}x{H}x{W} {fam}: bf16 forward max |dp| vs float64: " + ", ".join(f"{k} {v:.3e}" for k, v in err.items()))
