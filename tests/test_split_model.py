"""CPU: the three-plane (fp32-precision) arithmetic of UNetDC.precision = "fp32" -- the split of model.split_bf16, the
split weight packers, the kernel's (tap, term, chunk) walk replayed by tests/split_model.py against a float64 conv, and
the fp32 max of the pooled epilogue."""
import pytest
import torch

import split_model as sm
from unet_dc_segmentation_b200.model import (fold_conv_bn, pack_conv3x3_split, pack_upconv_split, split_bf16, UNetDC)

FLT_MAX = float(torch.finfo(torch.float32).max)
TINY = float(torch.finfo(torch.float32).tiny)


def _same_bits(a, b):
    """Bit for bit, except that -0 may come back as +0 (hi = -0 plus mid + lo = +0)."""
    nz = b != 0
    return torch.equal(a[nz].view(torch.int32), b[nz].view(torch.int32)) and bool((a[~nz] == 0).all())


def _assert_split_exact(x32):
    hi, mid, lo = split_bf16(x32)
    assert hi.dtype == mid.dtype == lo.dtype == torch.bfloat16
    assert _same_bits(hi.float() + (mid.float() + lo.float()), x32), "hi + (mid + lo) != x"
    small = x32.abs() < 2.0 ** 127
    assert _same_bits(((hi.float() + mid.float()) + lo.float())[small], x32[small]), "(hi + mid) + lo != x"
    # each plane is the round-to-nearest bf16 of what the planes before it leave
    assert torch.equal(mid, (x32 - hi.float()).bfloat16()) and torch.equal(lo, (x32 - hi.float() - mid.float()).bfloat16())


def test_split_exact_random():
    g = torch.Generator().manual_seed(0)
    mant = torch.rand(200000, generator=g) + 1.0
    expo = torch.randint(-100, 100, (200000,), generator=g).float()
    sign = torch.randint(0, 2, (200000,), generator=g).float() * 2 - 1
    _assert_split_exact((sign * mant * torch.exp2(expo)).float())
    _assert_split_exact(torch.randn(100000, generator=g))
    _assert_split_exact(torch.randint(-(1 << 24), 1 << 24, (100000,), generator=g).float())


def test_split_exact_edges():
    x = torch.tensor([FLT_MAX, -FLT_MAX, TINY, -TINY, 0.0, -0.0, 1.0, -1.0, 2.0 ** 19 + 2 ** 9 + 1, -(2.0 ** 19 + 2 ** 10),
                      float(torch.tensor(1 / 3, dtype=torch.float32)), -255.0 / 256, 2.0 ** 100, -(2.0 ** -100)],
                     dtype=torch.float32)
    _assert_split_exact(x)
    hi, mid, lo = split_bf16(x)
    assert not hi.float().isinf().any(), "the largest finite value split into an infinite hi"
    # values whose lo is 0: up to 16 significant bits
    y = torch.tensor([2.0 ** 19 + 2 ** 10, 513.0, -65535.0, 0.75], dtype=torch.float32)
    _assert_split_exact(y)
    assert torch.equal(split_bf16(y)[2].float(), torch.zeros(4))
    # three non-zero planes, including a negative lo
    z = torch.tensor([2.0 ** 19 + 2 ** 9 + 1, 2.0 ** 18 + 2 ** 9 + 3], dtype=torch.float32)
    assert all(bool((p.float() != 0).all()) for p in split_bf16(z))


def test_weight_split_from_float64():
    """BatchNorm folded in float64, rounded to fp32 once, split: the planes rebuild float32(w64) exactly, and the packers
    put plane p of tap t at column (3 t + p) Cin (3x3) / p Cin (transposed conv)."""
    g = torch.Generator().manual_seed(1)
    w, b = torch.randn(16, 64, 3, 3, generator=g), torch.randn(16, generator=g)
    gam, bet = torch.rand(16, generator=g) + 0.5, torch.randn(16, generator=g)
    mu, var = torch.randn(16, generator=g), torch.rand(16, generator=g) + 0.1
    w64, b64 = fold_conv_bn(w, b, gam, bet, mu, var, dtype=torch.float64)
    assert w64.dtype == torch.float64
    ref = ((w.double() * (gam.double() / torch.sqrt(var.double() + 1e-5)).view(-1, 1, 1, 1)))
    assert torch.equal(w64, ref)
    blob = pack_conv3x3_split(w64)
    assert blob.shape == (16, 27 * 64) and blob.dtype == torch.bfloat16
    r = blob.float().reshape(16, 9, 3, 64)
    rebuilt = r[:, :, 0] + (r[:, :, 1] + r[:, :, 2])
    assert torch.equal(rebuilt, w64.float().permute(0, 2, 3, 1).reshape(16, 9, 64))
    wu = torch.randn(128, 64, 2, 2, generator=g).double()
    ub = pack_upconv_split(wu).float().reshape(4, 64, 3, 128)
    want = wu.float().permute(2, 3, 1, 0).reshape(4, 64, 128)
    assert torch.equal(ub[:, :, 0] + (ub[:, :, 1] + ub[:, :, 2]), want)


@pytest.mark.parametrize("kind", sm.KINDS)
@pytest.mark.parametrize("cin,cout,d", [(64, 64, 1), (128, 64, 2), (64, 128, 4)])
def test_replay_equals_float64_conv(kind, cin, cout, d):
    """The kernel's K walk over the packed blob and the plane strides equals the float64 conv on the exact operands."""
    x, w, b = sm.operands(kind, 2, 9, 11, cin, cout, seed=cin + cout + d)
    ips = cin + 8
    buf = sm.plane_buffer(x, ips, 3 * ips, fill=0.0)
    got = sm.replay_conv(buf, ips, cin, pack_conv3x3_split(w), cout, d, b)
    assert torch.equal(got, sm.conv64(x, w, b, d))
    # the operands need the planes they claim: each kind has a term whose removal changes the output
    assert bool(split_bf16(x)[2].float().ne(0).any()) == (kind == "a3")
    assert bool(split_bf16(w)[2].float().ne(0).any()) == (kind == "w3")


@pytest.mark.parametrize("kind", sm.KINDS)
def test_replay_upconv_equals_float64(kind):
    x, w, b = sm.operands(kind, 2, 5, 7, 128, 64, seed=3, upconv=True)
    buf = sm.plane_buffer(x, 128, 384, fill=0.0)
    got = sm.replay_upconv(buf, 128, 128, pack_upconv_split(w), 64, b)
    assert torch.equal(got, sm.upconv64(x, w, b))


def test_mutations_are_seen():
    """Dropping any one of the six terms, swapping two activation planes or reading with a wrong plane stride changes
    a compared output on one of the operand families."""
    cases = {k: sm.operands(k, 1, 8, 8, 64, 64, seed=11) for k in sm.KINDS}
    packed = {k: pack_conv3x3_split(w) for k, (x, w, b) in cases.items()}

    def differs(**kw):
        stride = kw.pop("stride", 72)
        out = False
        for k, (x, w, b) in cases.items():
            buf = sm.plane_buffer(x, 72, 216, fill=0.0)
            out |= not torch.equal(sm.replay_conv(buf, stride, 64, packed[k], 64, 1, b, relu=False, **kw),
                                   sm.conv64(x, w, b, 1, relu=False))
        return out

    assert not differs()
    for t in range(6):
        assert differs(terms=sm.TERMS[:t] + sm.TERMS[t + 1:]), f"dropping term {sm.TERMS[t]} went unseen"
    assert differs(plane_a={1: 2, 2: 1}), "swapped activation planes went unseen"
    assert differs(plane_a={0: 1, 1: 0}), "swapped activation planes went unseen"
    assert differs(stride=64), "a wrong plane stride went unseen"


def test_pool_counter_example():
    """2^19 + 2^9 + 1 = (2^19, 512, 1) and 2^19 + 2^10 = (2^19, 1024, 0): a per-plane max gives 2^19 + 1025, the max of
    the values 2^19 + 1024."""
    y = torch.tensor([2.0 ** 19 + 2 ** 9 + 1, 2.0 ** 19 + 2 ** 10, 0.0, 1.0], dtype=torch.float64).view(1, 2, 2, 1)
    assert float(sm.pool_split(y)) == 2.0 ** 19 + 2 ** 10
    assert float(sm.pool_per_plane(y)) == 2.0 ** 19 + 1025


def test_precision_defaults_to_bf16_per_instance():
    m = UNetDC()
    assert UNetDC.precision == "bf16" and m.precision == "bf16"
    m.precision = "fp32"
    assert UNetDC.precision == "bf16"
