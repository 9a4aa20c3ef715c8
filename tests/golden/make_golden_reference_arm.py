"""Stored outputs for tests/test_reference_arm.py, so that its comparisons also run where the original project's
compiled modules (oracle/_ref, see oracle/ref.py) are absent -- which is every fresh checkout.

    python tests/golden/make_golden_reference_arm.py

Writes
    reference_arm.npz   the path of quantify_droplets_batch.py on the test's two frames (synthetic_image(96, 30 + i),
                        calibrated_state_dict(seed=0, calib_size=64, n_calib=2)): probs f32, masks bit-packed, and for
                        both parametrizations (min_area, px) = (1, 3.45) and (4, None) every table column as f64
    reference_arm.json  the state_dict contract (key, shape, dtype) of UNetDC(cin, cout) for the test's channel counts

Source: with oracle/_ref present, the original's own functions (ref.run_path, the original UNetDC class).  Without it,
the port (oracle.run_path in fp32, with the C rolling ball) and unet_dc_segmentation_b200.UNetDC, whose results
test_reference_arm requires to equal the original's bit for bit whenever the original is present.  `source` in both
files says which one wrote them.  Either way the (3, 1) contract must equal state_dict_keys.json, which
make_golden.py took from the original.
"""
from __future__ import annotations

import json
import sys
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
REPO = HERE.parent.parent
sys.path.insert(0, str(REPO))

CASES = {"min1_px3.45": (1, 3.45), "min4_none": (4, None)}
CHANNELS = [(3, 1), (1, 1), (5, 2)]


def frames():
    from unet_dc_segmentation_b200.synth import synthetic_image
    return np.stack([synthetic_image(96, 30 + i) for i in range(2)])


def main():
    import oracle
    from oracle import ref
    from unet_dc_segmentation_b200.model import UNetDC
    from unet_dc_segmentation_b200.synth import calibrated_state_dict

    source = "reference" if ref.available() else "port"
    run_path = ref.run_path if source == "reference" else oracle.run_path
    module = ref.load().UNetDC if source == "reference" else UNetDC

    sd = calibrated_state_dict(seed=0, calib_size=64, n_calib=2)
    imgs = frames()
    rgb = [np.repeat(im[:, :, None], 3, 2) for im in imgs]
    out = {"source": np.array(source), "images": imgs}
    for case, (min_area, px) in CASES.items():
        probs, masks, tables = run_path(sd, rgb, 50, 0.3, min_area, px)
        if "probs" not in out:
            out["probs"] = probs.astype(np.float32)
            for i, m in enumerate(masks):
                out[f"mask{i}"] = np.packbits(m, axis=None)
        for i, df in enumerate(tables):
            assert len(df) > 0
            out[f"{case}/columns"] = np.array(list(df.columns))
            out[f"{case}/t{i}/n"] = np.int64(len(df))
            for c in df.columns:
                out[f"{case}/t{i}/{c}"] = df[c].to_numpy().astype(np.float64)
    np.savez_compressed(HERE / "reference_arm.npz", **out)

    contracts = {f"{cin},{cout}": [[k, list(v.shape), str(v.dtype)] for k, v in module(cin, cout).state_dict().items()]
                 for cin, cout in CHANNELS}
    assert contracts["3,1"] == json.loads((HERE / "state_dict_keys.json").read_text())
    (HERE / "reference_arm.json").write_text(json.dumps({"source": source, "contracts": contracts}, indent=0) + "\n")
    print("source", source, "droplets", [int(out[f"{c}/t{i}/n"]) for c in CASES for i in range(2)])


if __name__ == "__main__":
    main()
