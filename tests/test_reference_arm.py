"""CPU: the oracle port against the original project's path.  Where the original's compiled modules (oracle/_ref) are
present, the port's whole path must reproduce them bit for bit: probabilities, masks and every table column -- the
unmodified reference code over real cv2 and real torch (skimage.measure through the scipy-backed shim of
oracle/shims.py).  Elsewhere the same comparisons run against the outputs stored in tests/golden/reference_arm.*
(tests/golden/make_golden_reference_arm.py; `source` there says what wrote them), with the fp32 probabilities held
to the 2e-4 of test_oracle_golden, as CPU convolution kernels differ between machines in the last bits."""
import json

import numpy as np
import pytest

import oracle
from conftest import GOLDEN, assert_table_equal, golden_table, load_golden
from oracle import ref


@pytest.fixture(scope="module")
def reference_or_none():
    if not ref.available() and not ref.build_ref():
        return None
    return ref.load()


@pytest.fixture(scope="module")
def reference(reference_or_none):
    if reference_or_none is None:
        pytest.skip("the original project's compiled modules (oracle/_ref) are absent")
    return reference_or_none


def test_reference_modules_are_the_reference(reference):
    assert reference.qdb.IMG_SIZE == 512 and reference.qdb.__name__ == "quantify_droplets_batch"
    assert reference.UNetDC.__module__ == "models.model_2"
    assert list(reference.UNetDC(3, 1).state_dict().keys())[:2] == ["enc1.0.weight", "enc1.0.bias"]


@pytest.mark.parametrize("min_area,px", [(1, 3.45), (4, None)])
def test_port_reproduces_the_reference_path(reference_or_none, min_area, px):
    from unet_dc_segmentation_b200.synth import calibrated_state_dict, synthetic_image
    sd = calibrated_state_dict(seed=0, calib_size=64, n_calib=2)
    imgs = [np.repeat(synthetic_image(96, 30 + i)[:, :, None], 3, 2) for i in range(2)]
    p_port, m_port, t_port = oracle.run_path(sd, imgs, 50, 0.3, min_area, px, use_cv2=False)     # the C rolling ball
    if reference_or_none is not None:
        p_ref, m_ref, t_ref = ref.run_path(sd, imgs, 50, 0.3, min_area, px)
        np.testing.assert_array_equal(p_ref, p_port)
        np.testing.assert_array_equal(m_ref, m_port)
        for a, b in zip(t_ref, t_port):
            assert list(a.columns) == list(b.columns) and len(a) == len(b) > 0
            for c in a.columns:
                np.testing.assert_array_equal(a[c].to_numpy(), b[c].to_numpy(), err_msg=c)
        return
    g = load_golden("reference_arm.npz")
    case = f"min{min_area}_{'px' + str(px) if px else 'none'}"
    np.testing.assert_array_equal(np.stack([im[:, :, 0] for im in imgs]), g["images"])
    np.testing.assert_allclose(p_port, g["probs"], atol=2e-4, rtol=0)
    for i in range(2):
        want_mask = np.unpackbits(g[f"mask{i}"])[: 96 * 96].reshape(96, 96)
        near = np.abs(g["probs"][i] - 0.3) < 1e-3
        assert np.all((m_port[i] == want_mask) | near)
        want = golden_table(g, f"{case}/t{i}/")
        assert list(t_port[i].columns) == list(g[f"{case}/columns"]) and int(want["n"]) > 0
        if np.array_equal(m_port[i], want_mask):
            got = {c: t_port[i][c].to_numpy() for c in t_port[i].columns}
        else:       # a pixel within 1e-3 of the threshold flipped: the table of the stored mask is what must match
            got = oracle.quantify_arrays(want_mask, min_area, px)[1]
        assert_table_equal(got, want, f"{case} image {i}")


def test_reference_quantify_empty_and_filtered(reference_or_none):
    """An empty frame gives an empty, column-less DataFrame; a frame whose droplets are all below min_area an empty one
    (qdb:87-88).  Without the original, the port must give what the original gives."""
    import pandas as pd
    quantify = reference_or_none.quantify if reference_or_none is not None else oracle.quantify
    assert quantify(np.zeros((16, 16), np.uint8), 1, None).equals(pd.DataFrame())
    cb = (np.add.outer(np.arange(16), np.arange(16)) % 2).astype(np.uint8)
    assert quantify(cb, 2, 3.0).empty and oracle.quantify(cb, 2, 3.0).empty


@pytest.mark.parametrize("cin,cout", [(3, 1), (1, 1), (5, 2)])
def test_module_contract_matches_the_reference_for_any_channel_count(reference_or_none, cin, cout):
    """Same constructor, same state_dict keys / shapes / dtypes as the reference class it replaces (model_2.py:6-32)."""
    from unet_dc_segmentation_b200.model import UNetDC
    ours = UNetDC(cin, cout).state_dict()
    if reference_or_none is not None:
        theirs = reference_or_none.UNetDC(cin, cout).state_dict()
        assert list(ours.keys()) == list(theirs.keys())
        for k in ours:
            assert ours[k].shape == theirs[k].shape and ours[k].dtype == theirs[k].dtype, k
        return
    want = json.loads((GOLDEN / "reference_arm.json").read_text())["contracts"][f"{cin},{cout}"]
    assert [[k, list(v.shape), str(v.dtype)] for k, v in ours.items()] == want
