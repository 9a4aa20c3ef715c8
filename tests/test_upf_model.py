"""CPU: the numpy model of the fused upconv + conv kernels (tests/upf_model.py) -- regions, generated MMA issue code,
weight blobs row by row -- against the oracle's evaluation of the composed layer.  Pins the host-side packers, the
schedule generator and the slot -> class mapping without a GPU."""
import numpy as np
import pytest

import oracle
import upf_model as um


def _layer(C, seed):
    import torch
    from unet_dc_segmentation_b200.model import compose_upconv
    g = torch.Generator().manual_seed(seed)
    wu = torch.randn(2 * C, C, 2, 2, generator=g) / (2 * C) ** 0.5
    bu = torch.randn(C, generator=g) * 0.3
    wd = torch.randn(C, 2 * C, 3, 3, generator=g) / (3.0 * (2 * C) ** 0.5)
    bd = torch.randn(C, generator=g) * 0.1
    return compose_upconv(wu, bu, wd, bd)


def _acts(C, H, W, seed):
    import torch
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(H, W, 2 * C, generator=g).bfloat16().float()
    skip = torch.randn(2 * H, 2 * W, C, generator=g).bfloat16().float()
    return x, skip


def _want(x, skip, comp, skipw, bias9):
    import torch
    zero = torch.zeros_like(bias9)                      # the model stops before the epilogue's bias
    y = oracle.composed_upconv_conv3x3(x.permute(2, 0, 1)[None], skip.permute(2, 0, 1)[None], comp, skipw, zero, relu=False)
    return y[0].permute(1, 2, 0).numpy()


def test_level1_model():
    """Level 1 (C = 64): image of 20 x 12 half-resolution pixels = tiles (0,0), (0,8) (ragged) and (16,0), (16,8):
    every border class, zero fill on all four sides, both CTAs of a pair."""
    from unet_dc_segmentation_b200 import model as M
    comp, skipw, bias9 = _layer(64, 1)
    x, skip = _acts(64, 20, 12, 2)
    blob = M.pack_upfused(comp, skipw).float().numpy()
    got = np.zeros((40, 24, 64), np.float32)
    for tiles in ([(0, 0), (0, 8)], [(16, 0), (16, 8)]):
        acc = um.level1_tile_pair(x.numpy(), skip.numpy(), blob, tiles)
        for c, (h0, w0) in enumerate(tiles):
            um.scatter_level1(acc[c], h0, w0, got)
    want = _want(x, skip, comp, skipw, bias9)
    assert np.abs(got - want).max() < 2e-3 * max(1.0, np.abs(want).max())


@pytest.mark.parametrize("C", [128, 256, 512])
def test_wide_model(C):
    """Levels 2-4: one tile pair of a 16 x 12 half-resolution image, every class group and n-tile."""
    from unet_dc_segmentation_b200 import model as M
    comp, skipw, bias9 = _layer(C, C)
    x, skip = _acts(C, 16, 12, C + 1)
    wx, ws = (t.float().numpy() for t in M.pack_upfused_wide(comp, skipw))
    bn = min(C, 256)
    ncls, ntiles = 256 // bn, C // bn
    tiles = [(0, 0), (0, 8)]
    got = np.zeros((32, 24, C), np.float32)
    for grp in range(4 // ncls):
        for nt in range(ntiles):
            acc = um.wide_pass(x.numpy(), skip.numpy(), wx, ws, C, tiles, grp, nt)
            for c, (h0, w0) in enumerate(tiles):
                for half in range(ncls):
                    cls = grp * ncls + half
                    for lane in range(128):
                        y, xx = 2 * (h0 + lane // 8) + (cls >> 1), 2 * (w0 + lane % 8) + (cls & 1)
                        if y < 32 and xx < 24:
                            got[y, xx, nt * bn:(nt + 1) * bn] = acc[c, half, lane]
    want = _want(x, skip, comp, skipw, bias9)
    assert np.abs(got - want).max() < 2e-3 * max(1.0, np.abs(want).max())
