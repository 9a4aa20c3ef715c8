"""CPU: bench.py --dump-outputs -- the last timed step's masks and droplet tables as float arrays, sampled with a fixed
seed to stay within the size budget."""
import numpy as np
import torch

import bench
from unet_dc_segmentation_b200.quantify import DropletTables


def _step(B=3, H=16, W=24, cap=40, seed=0):
    g = torch.Generator().manual_seed(seed)
    masks = (torch.rand((B, H, W), generator=g) < 0.4).to(torch.uint8)
    counts = torch.randint(0, cap + 1, (B,), dtype=torch.int32, generator=g)
    col = lambda: torch.rand((B, cap), dtype=torch.float64, generator=g)          # noqa: E731
    area = torch.randint(1, 100, (B, cap), generator=g)
    return masks, DropletTables(counts, area, col(), col(), col(), col(), col(), None, cap)


def test_dump_holds_every_row_and_droplet_within_budget():
    masks, t = _step()
    out = bench.last_step_outputs(masks, t)
    assert all(a.dtype in (np.float32, np.float64) for a in out.values())
    np.testing.assert_array_equal(out["mask_rows"], masks.reshape(-1, masks.shape[2]).numpy())
    np.testing.assert_array_equal(out["mask_row_index"][:, 0], np.repeat(np.arange(3), 16))
    np.testing.assert_array_equal(out["droplet_counts"], t.counts.numpy())
    host = t.to_host()
    for c in host[0]:
        np.testing.assert_array_equal(out[f"droplets_{c}"], np.concatenate([np.asarray(h[c], np.float64) for h in host]))
    np.testing.assert_array_equal(out["droplets_image"], np.repeat(np.arange(3), t.counts.numpy()))


def test_dump_samples_with_a_fixed_seed_past_the_budget(monkeypatch):
    monkeypatch.setattr(bench, "DUMP_MASK_BYTES", 10 * 4 * 24)
    monkeypatch.setattr(bench, "DUMP_BYTES", 10 * 4 * 24 + 10 * 2 * 8 + 3 * 8 + 25 * 8 * 8)
    masks, t = _step()
    out = bench.last_step_outputs(masks, t)
    assert sum(a.nbytes for a in out.values()) <= bench.DUMP_BYTES
    assert out["mask_rows"].shape == (10, 24) and len(out["droplets_image"]) == 25
    b, r = out["mask_row_index"].astype(np.int64).T
    np.testing.assert_array_equal(out["mask_rows"], masks[b, r].numpy())
    host = t.to_host()
    for i, lab, dia in zip(out["droplets_image"].astype(int), out["droplets_label"].astype(int),
                           out["droplets_equivalent_diameter"]):
        assert host[i]["equivalent_diameter"][lab - 1] == dia
    again = bench.last_step_outputs(*_step())
    assert all(np.array_equal(again[k], v) for k, v in out.items())
