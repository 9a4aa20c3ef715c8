"""GPU: the forward at full frame size held to the tcgen05 accumulator model bit for bit, layer by layer.

test_gpu_tc_accum.py replays whole maps of 64^2 and 48 x 80 chains.  At those sizes no persistent CTA reaches a second
tile, the deep layers' dilated taps are never in bounds and the parity-class and border-class epilogues see few tiles.
Here the same launch sequence (tc_chain.forward_chain) runs at the benchmark's 1024^2 frame, at 2 x 784 x 1296 (partial
tiles at levels 1-4, a 49 x 81 bottleneck map on which every dilated tap is in bounds somewhere), at 33 x 1024^2
(level-0 offsets past 2^31 from frame 32 on) and in fp32 precision at 512^2 and 1024^2.  A float64 replay of whole
1024^2 layers is out of reach (each conv layer is about 3.9e10 multiply-adds), so each layer is replayed at the sites of
tc_accum_model.select_sites: the border ring, the rows and columns where dilated taps cross the edge, one pixel of
every tile of the kernel's grid at a rotating in-tile position, and seeded interior pixels up to a product budget.
Every launch must also have written its whole output (the buffers start as NaN), and predict_u8 / m(x) / the
pipeline must give exactly the chain's result.  Teeth: for each kernel family the chain reaches, a wrong K walk
replayed at the same sites differs from the GPU's bits."""

import numpy as np
import pytest
import torch

import tc_chain as tc
from exact_net import family  # noqa: F401  (fixture)

pytestmark = pytest.mark.gpu

THRESH = 0.3
# each kernel family of the default bf16 forward at 1024^2 (pair kernel at Cin >= 128, per-tap kernel at dilation 8
# and 16, conv_par2_kernel, both fused kernels) and of the fp32 forward (the split kernel, its transposed conv)
BF16_TEETH = ("pair", "per-tap d8", "per-tap d16", "par2", "fused", "fused wide")
FP32_TEETH = ("split", "split upconv")


@pytest.fixture(autouse=True)
def _free_between_tests():
    torch.cuda.empty_cache()
    yield
    torch.cuda.empty_cache()


def _need_gib(gib):
    free, _ = torch.cuda.mem_get_info()
    if free < gib * 2**30:
        pytest.skip(f"needs {gib} GiB of free device memory, {free / 2**30:.1f} GiB free")


def _bf16_model(sd):
    from unet_dc_segmentation_b200 import UNetDC
    m = UNetDC()
    m.load_state_dict(sd)
    return m.cuda().eval()


def _x32(u8):
    """The fp32 entry's frames: u8 / 255 correctly rounded in fp32, as the u8 entries compute it (a device division by
    a scalar multiplies by its reciprocal instead), on three channels."""
    x = torch.from_numpy(u8.cpu().numpy().astype(np.float32) / np.float32(255))
    return x[:, None].expand(-1, 3, -1, -1).contiguous().cuda()


def _assert_teeth(check, kernels):
    assert set(check.wrong) == set(kernels), f"no layer of {set(kernels) - set(check.wrong)} reached"
    for k, (n, total) in check.wrong.items():
        assert n > 0, f"a wrong walk of {k} gives the GPU's bits at all {total} outputs: the sites cannot see order"


def _bench_frame():
    """The benchmark's frame and network: synthetic_image(1024, 0) and calibrated_state_dict(seed=0)."""
    from unet_dc_segmentation_b200.synth import calibrated_state_dict, synthetic_image
    return torch.from_numpy(synthetic_image(1024, 0))[None].cuda(), calibrated_state_dict(seed=0)


def test_bf16_bench_frame_auto(cuda_device, family):
    """The benchmark's frame after the rolling ball (radius 50), both entries, auto family; the pipeline's mask is the
    chain's; a wrong walk of each kernel family differs somewhere."""
    from unet_dc_segmentation_b200.morphology import rolling_ball_device
    from unet_dc_segmentation_b200.pipeline import DropletPipeline
    family("auto")
    raw, sd = _bench_frame()
    m = _bf16_model(sd)
    u8 = rolling_ball_device(raw, 50)
    check = tc.Sites([0], teeth=BF16_TEETH)
    prob, mask = tc.forward_chain(m, "bf16", "auto", u8, _x32(u8), check, in_kind=1)
    _assert_teeth(check, BF16_TEETH)
    mk, pr = m.predict_u8(u8, THRESH, return_prob=True)
    assert torch.equal(pr[:, 0], prob) and torch.equal(mk, mask), "predict_u8 differs from the layer chain"
    assert torch.equal(DropletPipeline(m, 50, THRESH, 1, 3.45).run_device(raw).masks, mask), \
        "the pipeline's mask differs from the layer chain"
    prob0, _ = tc.forward_chain(m, "bf16", "auto", u8, _x32(u8), tc.Sites([0]), in_kind=0)
    assert torch.equal(m(_x32(u8))[:, 0], prob0), "m(x) differs from the layer chain"


def test_bf16_bench_frame_generic(cuda_device, family):
    """The same frame with the pair / halo kernels and conv_par2_kernel off: every 3x3 layer on the per-tap kernel."""
    from unet_dc_segmentation_b200.morphology import rolling_ball_device
    family("generic")
    raw, sd = _bench_frame()
    m = _bf16_model(sd)
    u8 = rolling_ball_device(raw, 50)
    prob, mask = tc.forward_chain(m, "bf16", "generic", u8, _x32(u8), tc.Sites([0]), in_kind=1)
    mk, pr = m.predict_u8(u8, THRESH, return_prob=True)
    assert torch.equal(pr[:, 0], prob) and torch.equal(mk, mask), "predict_u8 differs from the layer chain"


def test_bf16_partial_tiles(cuda_device, family):
    """2 x 784 x 1296: partial tiles at levels 1-4 and a 49 x 81 bottleneck map; sites in both frames."""
    import test_gpu_fp32 as t32
    family("auto")
    m = _bf16_model(t32._calibrated())
    u8 = t32._frames(2, 1296, 60)[:, :784].contiguous().cuda()
    prob, mask = tc.forward_chain(m, "bf16", "auto", u8, _x32(u8), tc.Sites([0, 1]), in_kind=1)
    mk, pr = m.predict_u8(u8, THRESH, return_prob=True)
    assert torch.equal(pr[:, 0], prob) and torch.equal(mk, mask), "predict_u8 differs from the layer chain"


def test_bf16_past_2_31(cuda_device, family):
    """33 x 1024^2: from frame 32 on, level-0 element offsets are >= 2^31; sites in frames 0 and 32."""
    import test_gpu_fp32 as t32
    _need_gib(80)
    family("auto")
    m = _bf16_model(t32._calibrated())
    u8 = t32._frames(33, 1024, 300).cuda()
    prob, mask = tc.forward_chain(m, "bf16", "auto", u8, _x32(u8), tc.Sites([0, 32]), in_kind=1)
    mk, pr = m.predict_u8(u8, THRESH, return_prob=True)
    assert torch.equal(pr[:, 0], prob) and torch.equal(mk, mask), "predict_u8 differs from the layer chain"


@pytest.mark.parametrize("size", [512, 1024])
def test_fp32_forward(cuda_device, size):
    """fp32 precision on one frame of the sizes test_gpu_fp32.py's P_TOL note quotes; a wrong term order of the split
    kernel and of its transposed conv differs somewhere."""
    import test_gpu_fp32 as t32
    from unet_dc_segmentation_b200 import UNetDC
    m = t32._model(UNetDC, t32._calibrated())
    u8 = t32._frames(1, size, 50).cuda()
    check = tc.Sites([0], teeth=FP32_TEETH)
    prob, mask = tc.forward_chain(m, "fp32", "auto", u8, _x32(u8), check)
    _assert_teeth(check, FP32_TEETH)
    mk, pr = m.predict_u8(u8, THRESH, return_prob=True)
    assert torch.equal(pr[:, 0], prob) and torch.equal(mk, mask), "predict_u8 differs from the layer chain"
    assert torch.equal(m(_x32(u8))[:, 0], prob), "m(x) differs from the layer chain"
