"""CPU: host-side logic of the product -- weight folding / packing, the module's state_dict contract,
the FLOP model behind roofline.achieved, the synthetic inputs."""
import json
from pathlib import Path

import numpy as np
import pytest
import torch
import torch.nn.functional as F

GOLDEN = Path(__file__).resolve().parent / "golden"


def test_state_dict_contract_matches_reference():
    """Same 136 keys, shapes and dtypes as reference models/model_2.py UNetDC (keys captured by make_golden.py)."""
    from unet_dc_segmentation_b200 import UNet, UNetDC
    want = json.loads((GOLDEN / "state_dict_keys.json").read_text())
    for cls in (UNetDC, UNet):
        sd = cls(3, 1).state_dict()
        got = [[k, list(v.shape), str(v.dtype)] for k, v in sd.items()]
        assert got == want
    assert len(want) == 136
    assert sum(int(np.prod(s)) for k, s, _ in want if "running" not in k and "num_batches" not in k) == 31_043_521


def test_load_state_dict_roundtrip_and_constructor_contract():
    from unet_dc_segmentation_b200 import UNetDC
    from unet_dc_segmentation_b200.synth import calibrated_state_dict
    sd = calibrated_state_dict(seed=1, calib_size=32, n_calib=1)
    m = UNetDC(in_channels=3, out_channels=1)
    missing = m.load_state_dict(sd)
    assert not missing.missing_keys and not missing.unexpected_keys
    for k, v in m.state_dict().items():
        assert torch.equal(v, sd[k]), k
    assert UNetDC(1, 2).state_dict()["enc1.0.weight"].shape == (64, 1, 3, 3)          # any channel counts, as the reference
    with pytest.raises(ValueError):
        UNetDC(0, 1)
    with pytest.raises(ValueError):
        UNetDC(3, 65)


def test_bn_fold_equals_conv_then_bn():
    from unet_dc_segmentation_b200.model import fold_conv_bn
    g = torch.Generator().manual_seed(0)
    w, b = torch.randn(8, 4, 3, 3, generator=g), torch.randn(8, generator=g)
    gamma, beta = torch.rand(8, generator=g) + 0.5, torch.randn(8, generator=g)
    mean, var = torch.randn(8, generator=g), torch.rand(8, generator=g) + 0.1
    x = torch.randn(2, 4, 9, 9, generator=g)
    want = F.batch_norm(F.conv2d(x, w, b, padding=2, dilation=2), mean, var, gamma, beta, False, 0.0, 1e-5)
    wf, bf = fold_conv_bn(w, b, gamma, beta, mean, var)
    np.testing.assert_allclose(F.conv2d(x, wf, bf, padding=2, dilation=2).numpy(), want.numpy(), atol=2e-5)


def test_pack_layouts():
    from unet_dc_segmentation_b200.model import pack_conv3x3, pack_upconv
    w = torch.arange(2 * 3 * 9, dtype=torch.float32).reshape(2, 3, 3, 3)
    p = pack_conv3x3(w).float()
    assert p.shape == (2, 27)
    for co in range(2):
        for ci in range(3):
            for ky in range(3):
                for kx in range(3):
                    assert p[co, (ky * 3 + kx) * 3 + ci] == w[co, ci, ky, kx]
    wt = torch.arange(4 * 5 * 4, dtype=torch.float32).reshape(4, 5, 2, 2)        # [Cin, Cout, 2, 2]
    q = pack_upconv(wt).float()
    assert q.shape == (20, 4)
    for ci in range(4):
        for co in range(5):
            for a in range(2):
                for b in range(2):
                    assert q[(a * 2 + b) * 5 + co, ci] == wt[ci, co, a, b]
    # the packed matrix reproduces conv_transpose2d(k=2, s=2): out[.., 2i+a, 2j+b] = W_q @ x[.., i, j]
    x = torch.randn(1, 4, 3, 3)
    y = F.conv_transpose2d(x, wt, None, stride=2)
    yq = torch.einsum("nk,bkij->bnij", q, x).reshape(1, 2, 2, 5, 3, 3)
    for a in range(2):
        for b in range(2):
            np.testing.assert_allclose(y[0, :, a::2, b::2].numpy(), yq[0, a, b].numpy(), rtol=1e-5, atol=1e-4)


def test_flop_model_matches_baseline_md():
    from unet_dc_segmentation_b200 import workload as wl
    for size, tflop, frac in ((256, 0.0963, 0.8905), (512, 0.3853, 0.9363), (1024, 1.5414, 0.9659),
                              (2048, 6.1654, 0.9824), (4096, 24.662, 0.9911)):
        nominal = wl.forward_flops(size, size, in_bounds=False)
        assert nominal == 2 * 734_976 * size * size
        assert abs(nominal / 1e12 - tflop) / tflop < 5e-4          # BASELINE.md prints 4 significant digits
        assert abs(wl.forward_flops(size, size) / nominal - frac) < 1e-4
    names, fl = wl.launch_flops(1024, 1024)
    assert len(names) == 22 and names[0] == "enc1.0" and names[-1] == "dec1.3"
    assert abs(sum(fl) - wl.forward_flops(1024, 1024)) < 1.0
    # plain UNet (models/model.py) = dilation 1 everywhere: same nominal FLOPs, more in-bounds taps
    assert wl.forward_flops(256, 256, (1, 1, 1, 1, 1)) > wl.forward_flops(256, 256)
    # decoder levels run as one composed launch each: names merge, the algorithmic FLOPs stay, the issued ones drop
    names_f, fl_f = wl.launch_flops(1024, 1024, fused_level1=True, fused_levels=(2, 3, 4))
    assert len(names_f) == 18 and "upconv3+dec3.0" in names_f and abs(sum(fl_f) - sum(fl)) < 1.0
    assert wl.forward_flops_issued(1024, 1024) == wl.forward_flops(1024, 1024)
    r = wl.forward_flops_issued(1024, 1024, fused_levels=(1, 2, 3, 4)) / wl.forward_flops(1024, 1024)
    assert 0.92 < r < 0.94              # 4 levels x 11 % of the FLOPs x (1 - 17/20)


def test_synthetic_inputs_are_seeded():
    from unet_dc_segmentation_b200.synth import synthetic_image, synthetic_mask, synthetic_rgb
    a, b = synthetic_image(64, 5), synthetic_image(64, 5)
    assert a.dtype == np.uint8 and a.shape == (64, 64) and np.array_equal(a, b)
    assert not np.array_equal(a, synthetic_image(64, 6))
    img, truth = synthetic_image(64, 5, with_truth=True)
    assert np.array_equal(img, a) and set(np.unique(truth)) <= {0, 1} and 0 < truth.mean() < 0.5
    rgb = synthetic_rgb(32, 1)
    assert rgb.shape == (32, 32, 3) and np.array_equal(rgb[..., 0], rgb[..., 2])
    m = synthetic_mask(128, 50, seed=2)
    assert set(np.unique(m)) == {0, 1}


def test_shard_helpers():
    from unet_dc_segmentation_b200 import shard
    assert shard.shard_indices(10, 1, 4) == [1, 5, 9]
    assert sum((shard.shard_indices(4096, r, 8) for r in range(8)), []).__len__() == 4096
    assert shard.batches([0, 2, 4, 6, 8], 2) == [[0, 2], [4, 6], [8]]
    per_rank = [[(i, f"t{i}") for i in shard.shard_indices(7, r, 3)] for r in range(3)]
    assert shard.merge_in_frame_order(per_rank, 7) == [f"t{i}" for i in range(7)]
    with pytest.raises(ValueError):
        shard.merge_in_frame_order(per_rank[:2], 7)
    with pytest.raises(ValueError):
        shard.merge_in_frame_order(per_rank + [[(0, "dup")]], 7)
    assert shard.gather_results([(0, "a"), (1, "b")], 2) == ["a", "b"]       # no process group: identity


def test_combined_csv_text_equals_pandas_concat():
    """cli.combined_csv_text (all_droplets.csv from the per-image CSV bodies) is byte-identical to what the reference
    writes (pd.concat(all_props).to_csv, qdb:165-166), and declines whenever a frame has no droplets."""
    import numpy as np
    import pandas as pd
    from unet_dc_segmentation_b200 import cli
    rs = np.random.RandomState(0)
    frames = []
    for k in range(4):
        n = int(rs.randint(1, 40))
        a = rs.randint(1, 500, n).astype(np.int64)
        df = pd.DataFrame({"label": np.arange(1, n + 1), "area": a, "equivalent_diameter": np.sqrt(4 * a / np.pi),
                           "centroid-0": rs.rand(n) * 1024, "centroid-1": rs.rand(n) * 1e-7,
                           "area_sqmicron": a / (3.45 ** 2), "eq_diam_micron": np.sqrt(4 * a / np.pi) / 3.45})
        df.insert(0, "filename", f"f{k}.png")
        frames.append(df)
    texts = [df.to_csv(index=False) for df in frames]
    assert cli.combined_csv_text(frames, texts) == pd.concat(frames, ignore_index=True).to_csv(index=False)
    empty = pd.DataFrame()
    empty.insert(0, "filename", "none.png")
    assert cli.combined_csv_text(frames + [empty], texts + [empty.to_csv(index=False)]) is None
    assert cli.combined_csv_text(frames, None) is None


def test_compose_upconv_equals_the_two_layers():
    """model.compose_upconv: the composed 2x2-over-x + 3x3-over-skip layer (evaluated on the CPU from the blobs the
    kernel consumes) is conv_transpose2d -> cat -> conv2d(padding=1) of models/model_2.py:76-77, border bias included."""
    import torch
    import torch.nn.functional as F
    import oracle
    from unet_dc_segmentation_b200 import model as M
    g = torch.Generator().manual_seed(3)
    wu = torch.randn(128, 64, 2, 2, generator=g) * 0.1
    bu = torch.randn(64, generator=g)
    wd = torch.randn(64, 128, 3, 3, generator=g) * 0.05
    bd = torch.randn(64, generator=g)
    x = torch.randn(2, 128, 5, 7, generator=g)
    skip = torch.randn(2, 64, 10, 14, generator=g)
    want = F.conv2d(torch.cat([F.conv_transpose2d(x, wu, bu, stride=2), skip], 1), wd, bd, padding=1)
    comp, skipw, b9 = M.compose_upconv(wu, bu, wd, bd)
    assert comp.dtype == torch.bfloat16 and tuple(comp.shape) == (4, 2, 2, 64, 128) and tuple(b9.shape) == (9, 64)
    got = oracle.composed_upconv_conv3x3(x, skip, comp, skipw, b9, relu=False)
    assert float((got - want).abs().max()) < 0.05                  # bf16 rounding of the composed weights only
    # without that rounding the two are the same linear map
    class _NoRound:
        def __getattr__(self, k):
            return torch.float32 if k == "bfloat16" else getattr(torch, k)
    real, M.torch = M.torch, _NoRound()
    try:
        c32, s32, b932 = M.compose_upconv(wu, bu, wd, bd)
    finally:
        M.torch = real
    got32 = oracle.composed_upconv_conv3x3(x, skip, c32, s32, b932, relu=False)
    assert float((got32 - want).abs().max()) < 1e-4


def test_pack_upfused_follows_the_kernel_schedule():
    """The weight blob of dc_conv_upfused: every MMA of the schedule the library reports (host-only call) gets the
    tiles of the classes it covers, split between the two CTAs of a pair; 17 groups of 128 rows per CTA; every
    (class, tap, chunk) of the composed weights and every (class, 3x3 tap) of the skip weights is used exactly once."""
    import torch
    from unet_dc_segmentation_b200 import model as M
    sched = M.upfuse_schedule()
    assert len(sched) == 2 * 10 + 18
    seen = set()
    rows = 0
    for chunk, r, c, slot0, nslots in sched:
        assert nslots in (1, 2, 4) and slot0 + nslots <= 4
        for slot in range(slot0, slot0 + nslots):
            cls = slot ^ (slot >> 1)                        # accumulators in Gray order: 0, 1, 3, 2
            ky, kx = r - (cls >> 1), c - (cls & 1)
            assert 0 <= ky < (3 if chunk == 2 else 2) and 0 <= kx < (3 if chunk == 2 else 2)
            assert (chunk, cls, ky, kx) not in seen
            seen.add((chunk, cls, ky, kx))
        rows += 32 * nslots
    assert len(seen) == 2 * 4 * 4 + 4 * 9 and rows == 2176
    comp = torch.arange(4 * 2 * 2 * 64 * 128, dtype=torch.float32).reshape(4, 2, 2, 64, 128).bfloat16()
    skipw = -torch.arange(9 * 64 * 64, dtype=torch.float32).reshape(3, 3, 64, 64).bfloat16()
    blob = M.pack_upfused(comp, skipw)
    assert tuple(blob.shape) == (2, 2176, 64)
    # first MMA: window (1, 1) of x chunk 0, all four slots -> classes 0, 1 in CTA 0, classes 3, 2 in CTA 1
    assert torch.equal(blob[0, :64], comp[0, 1, 1][:, :64]) and torch.equal(blob[0, 64:128], comp[1, 1, 0][:, :64])
    assert torch.equal(blob[1, :64], comp[3, 0, 0][:, :64]) and torch.equal(blob[1, 64:128], comp[2, 0, 1][:, :64])


def test_upf_schedule_include_is_current(tmp_path):
    """csrc/upf_schedule.inc is generated (tools/gen_upf_schedule.py); the committed copy must be what the generator writes."""
    import subprocess
    import sys
    from pathlib import Path
    repo = Path(__file__).resolve().parent.parent
    out = tmp_path / "upf_schedule.inc"
    subprocess.run([sys.executable, str(repo / "tools" / "gen_upf_schedule.py"), str(out)], check=True, capture_output=True)
    assert out.read_text() == (repo / "unet_dc_segmentation_b200" / "csrc" / "upf_schedule.inc").read_text()


def test_pack_upfused_wide_layout():
    """Weight blobs of the deeper fused decoder levels: every (class group, n-tile, CTA, chunk, tap, class, row) lands
    where conv_upfused_wide_kernel's producers read it (include/unetdc_b200.h dc_upfuse_args)."""
    import torch
    from unet_dc_segmentation_b200 import model as M
    g = torch.Generator().manual_seed(7)
    for C in (128, 256, 512):
        bn = min(C, 256)
        ncls, nt, hb = 256 // bn, C // bn, bn // 2
        xc, sc = 2 * C // 64, C // 64
        comp = torch.randn(4, 2, 2, C, 2 * C, generator=g).bfloat16()
        skipw = torch.randn(3, 3, C, C, generator=g).bfloat16()
        wx, ws = M.pack_upfused_wide(comp, skipw)
        assert tuple(wx.shape) == ((4 // ncls) * nt * 2 * xc * 4 * 128, 64) and tuple(ws.shape) == (nt * 2 * sc * 9 * hb, 64)
        for _ in range(200):
            grp, t, cta, ch, tap, ci, r = (int(torch.randint(0, n, (1,), generator=g)) for n in (4 // ncls, nt, 2, xc, 4, ncls, hb))
            row = (((((grp * nt + t) * 2 + cta) * xc + ch) * 4 + tap) * ncls + ci) * hb + r
            cls, co = grp * ncls + ci, t * bn + cta * hb + r
            assert torch.equal(wx[row], comp[cls, tap >> 1, tap & 1, co, ch * 64:(ch + 1) * 64])
            ch_s, tap_s = ch % sc, int(torch.randint(0, 9, (1,), generator=g))
            row = (((t * 2 + cta) * sc + ch_s) * 9 + tap_s) * hb + r
            assert torch.equal(ws[row], skipw[tap_s // 3, tap_s % 3, co, ch_s * 64:(ch_s + 1) * 64])


def test_upf_schedule_issue_code_matches_its_tables():
    """The straight-line MMA issue code of csrc/upf_schedule.inc (literal descriptor offsets) against the definitions:
    per (chunk kind, group) every MMA reads the window of its table entry (x chunk: (r*10 + c)*8; skip chunk:
    column-parity plane (c & 1), row r, column c >> 1 of a 9-wide plane), takes its weights from the next free 32-row
    sub-tile of the group's ring slot, writes the accumulator of its first class with N = 64 * classes, and only the
    first MMA to touch a class in a tile's first chunk may overwrite."""
    import re
    from pathlib import Path
    txt = (Path(__file__).resolve().parent.parent / "unet_dc_segmentation_b200" / "csrc" / "upf_schedule.inc").read_text()
    ops = {}
    for m in re.finditer(r"upf_(u|s)_op\(int i\) \{\s*switch \(i\) \{(.*?)default", txt, re.S):
        ops[m.group(1)] = [tuple(int(v) for v in t) for t in re.findall(r"UpfOp\{(\d+), (\d+), (\d+), (\d+)\}", m.group(2))]
    assert len(ops) == 2
    plane = (9 * 34 * 128) >> 4
    groups = 0
    for m in re.finditer(r"upf_issue_group<(\d), (\d)>\(.*?\) \{(.*?)\n\}", txt, re.S):
        kind, g = int(m.group(1)), int(m.group(2))
        groups += 1
        calls = re.findall(r"umma_bf16_2sm\(d \+ (\d+)u, a \+ (\d+)ull, b \+ (\d+)ull, 0x([0-9a-f]+)u, ([^)]*)\);", m.group(3))
        table = ops["u" if kind == 0 else "s"]
        # the group's entries: groups are consecutive runs of the table whose classes add up to 4
        runs, cur, tot = [], [], 0
        for o in table:
            cur.append(o); tot += o[3]
            if tot == 4:
                runs.append(cur); cur, tot = [], 0
        grp = runs[g]
        assert len(calls) == 4 * len(grp)
        for k in range(4):
            sub = 0
            for j, (r, c, cls0, ncls) in enumerate(grp):
                d, a, b, idesc, acc = calls[k * len(grp) + j]
                want_a = (r * 10 + c) * 8 if kind == 0 else (c & 1) * plane + (r * 9 + (c >> 1)) * 8
                assert (int(d), int(a), int(b)) == (cls0 * 64, want_a + 2 * k, sub * 256 + 2 * k)
                assert (int(idesc, 16) >> 17) & 0x3F == (64 * ncls) >> 3 and (int(idesc, 16) >> 24) & 0x1F == 256 >> 4
                if "fresh" in acc:
                    assert k == 0 and kind != 1
                sub += ncls
        if kind != 1 and g == 0:
            assert any("fresh" in c[4] for c in calls)
    assert groups == 4 + 2 * 9          # x chunk; skip chunk after the x chunks and on its own
