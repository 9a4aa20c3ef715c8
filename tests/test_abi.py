"""CPU: the C-ABI shared library loads and exports every symbol include/unetdc_b200.h declares; the ctypes
structures mirror the C structs byte for byte; entry points fail loudly (no fallback) without a GPU.
No compute is launched here."""
import ctypes as C
import re
import subprocess
import sys
from pathlib import Path

import pytest

REPO = Path(__file__).resolve().parent.parent
HEADER = REPO / "include" / "unetdc_b200.h"


def declared_functions():
    text = HEADER.read_text()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(dc_[a-z0-9_]+)\s*\(", text)))


def test_header_cites_reference_lines():
    text = HEADER.read_text()
    for needle in ("models/model_2.py:56-80", "utils/data_loader.py:11-24", "quantify_droplets_batch.py:81-95"):
        assert needle in text


def test_library_exports_every_declared_symbol():
    from unet_dc_segmentation_b200 import _lib
    lib = _lib.load()
    fns = declared_functions()
    assert len(fns) >= 15
    for name in fns:
        assert hasattr(lib, name), f"{name} declared in the header but not exported"
    assert sorted(_lib.EXPORTS) == fns, "the ctypes binding and the header disagree on the entry points"
    assert lib.dc_version() >= 100


def test_ctypes_structs_match_c_layout(tmp_path):
    """sizeof / offsetof of every argument struct, as gcc lays them out, equals the ctypes mirror."""
    from unet_dc_segmentation_b200 import _lib
    structs = {"dc_conv_args_t": _lib.ConvArgs, "dc_stem_args_t": _lib.StemArgs, "dc_model_desc_t": _lib.ModelDesc,
               "dc_rolling_ball_args_t": _lib.RollingBallArgs, "dc_label_args_t": _lib.LabelArgs,
               "dc_resize_args_t": _lib.ResizeArgs}
    lines = ['#include <stdio.h>', '#include <stddef.h>', f'#include "{HEADER}"', "int main(void) {"]
    for cname, cls in structs.items():
        lines.append(f'  printf("{cname} %zu\\n", sizeof({cname}));')
        for fname, _ in cls._fields_:
            cfield = fname.rstrip("_")
            lines.append(f'  printf("{cname}.{fname} %zu\\n", offsetof({cname}, {cfield}));')
    lines += ["  return 0;", "}"]
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-o", str(exe), str(src)], check=True)
    out = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout
    got = dict(line.split() for line in out.strip().splitlines())
    for cname, cls in structs.items():
        assert int(got[cname]) == C.sizeof(cls), cname
        for fname, _ in cls._fields_:
            assert int(got[f"{cname}.{fname}"]) == getattr(cls, fname).offset, f"{cname}.{fname}"


def test_workspace_queries_and_argument_errors_need_no_gpu():
    from unet_dc_segmentation_b200 import _lib
    lib = _lib.load()
    n = C.c_size_t()
    assert lib.dc_label_workspace_bytes(2, 64, 64, C.byref(n)) == _lib.DC_OK and n.value >= 2 * 2 * 4 * 64 * 64
    assert lib.dc_rolling_ball_workspace_bytes(2, 64, 64, 1, C.byref(n)) == _lib.DC_OK and n.value >= 2 * 2 * 64 * 64
    assert lib.dc_label_workspace_bytes(0, 64, 64, C.byref(n)) == _lib.DC_EINVAL
    assert b"bad argument" in lib.dc_last_error()
    with pytest.raises(_lib.DcError) as ei:
        _lib.check(lib.dc_rolling_ball_workspace_bytes(1, -1, 8, 1, C.byref(n)))
    assert ei.value.code == _lib.DC_EINVAL
    for family in (-1, 1, 3):           # the family numbers are ABI: AUTO = 0, GENERIC = 2, 1 is unassigned
        assert lib.dc_debug_set_conv_family(family) == _lib.DC_EINVAL
    assert lib.dc_debug_set_conv_family(_lib.DC_CONV_FAMILY_AUTO) == _lib.DC_OK


NO_GPU_CHECK = r"""
import ctypes as C, sys
import numpy as np
import pytest
import torch
sys.path.insert(0, sys.argv[1])
import unet_dc_segmentation_b200 as pkg
assert not torch.cuda.is_available()
m = pkg.UNetDC(3, 1).eval()
with pytest.raises(RuntimeError, match="no CPU"):
    m(torch.zeros(1, 3, 16, 16))
with pytest.raises((RuntimeError, AssertionError)):
    pkg.quantify(np.zeros((8, 8), np.uint8), 1, None)
with pytest.raises((RuntimeError, AssertionError)):
    pkg.rolling_ball_correction_rgb(np.zeros((8, 8, 3), np.uint8), 5)
from unet_dc_segmentation_b200 import _lib
lib = _lib.load()
args = _lib.LabelArgs()
rc = lib.dc_label_stats(C.byref(args), None)
assert rc in (_lib.DC_ECUDA, _lib.DC_EDEVICE) and lib.dc_last_error()
print("NO_FALLBACK_OK")
"""


def test_no_cpu_fallback():
    """Without a GPU the product raises; it never routes to the oracle or to PyTorch ops.  Checked in a child process
    that sees no CUDA device, so that it holds on machines with and without one."""
    import os
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    r = subprocess.run([sys.executable, "-c", NO_GPU_CHECK, str(REPO)], env=env, capture_output=True, text=True,
                       timeout=300)
    assert r.returncode == 0 and "NO_FALLBACK_OK" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]


def test_product_never_imports_the_oracle():
    """oracle/ is test infrastructure: no product source may import it."""
    pkg = REPO / "unet_dc_segmentation_b200"
    for f in pkg.rglob("*.py"):
        text = f.read_text()
        assert not re.search(r"^\s*(import oracle|from oracle)", text, flags=re.M), f
    for f in (pkg / "csrc").glob("*"):
        assert "oracle" not in f.read_text().lower(), f
