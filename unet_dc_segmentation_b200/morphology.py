"""Rolling-ball background correction on the GPU (reference utils/data_loader.py:11-24).

``rolling_ball_correction_rgb`` keeps the reference's numpy-in / numpy-out signature;
``rolling_ball_device`` is the same operation on device-resident batches for the fused pipeline.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib



def max_radius() -> int:
    """Largest background radius the GPU path accepts (2047).  Radii up to ``tiled_max_radius()`` run the tiled
    chord kernel, larger ones the banded pass, which takes rows of at most 32768 pixels."""
    return int(_lib.load().dc_rolling_ball_max_radius())


def tiled_max_radius() -> int:
    """Largest radius the tiled chord kernel runs (170: the haloed tile of the element has to fit in shared memory)."""
    return int(_lib.load().dc_rolling_ball_tiled_max_radius())


def rolling_ball_workspace_bytes(B: int, H: int, W: int, Cc: int = 1) -> int:
    need = C.c_size_t()
    _lib.check(_lib.load().dc_rolling_ball_workspace_bytes(B, H, W, Cc, C.byref(need)))
    return int(need.value)


def rolling_ball_device(images: torch.Tensor, radius: int = 50, out: torch.Tensor | None = None,
                        workspace: torch.Tensor | None = None, method: str = "auto") -> torch.Tensor:
    """images: CUDA u8 [B,H,W] (planar) or [B,H,W,C] (interleaved).  Returns the corrected images, same shape.

    Per plane: opening with cv2's radius x radius ellipse, saturating subtract, min-max stretch to 0..255.
    method: "auto" (the tiled kernel up to ``tiled_max_radius()``, the banded pass above and for frames taller than
    the tiled kernel's grid: more than 65535 rows of tiles), "tiled" or "banded" (either kernel on its own; both are
    bit-exact, so the choice only changes the speed; "tiled" refuses what it cannot run)."""
    _lib.require_cuda(images, "images")
    if images.dtype != torch.uint8:
        raise TypeError("rolling ball works on uint8 images")
    if images.dim() == 3:
        B, H, W = images.shape
        Cc = 1
    elif images.dim() == 4:
        B, H, W, Cc = images.shape
    else:
        raise ValueError(f"expected u8 [B,H,W] or [B,H,W,C], got {tuple(images.shape)}")
    if method not in ("auto", "tiled", "banded"):
        raise ValueError(f"method must be 'auto', 'tiled' or 'banded', got {method!r}")
    if not 1 <= int(radius) <= max_radius():
        raise ValueError(f"radius must be in [1, {max_radius()}] (the structuring element is radius x radius pixels)")
    if method == "tiled" and int(radius) > tiled_max_radius():
        raise ValueError(f"method='tiled' takes radius 1..{tiled_max_radius()} (the haloed tile of a larger element does "
                         "not fit in shared memory); use 'auto' or 'banded'")
    images = images.contiguous()
    lib = _lib.load()
    entry = {"auto": lib.dc_rolling_ball, "tiled": lib.dc_rolling_ball_tiled, "banded": lib.dc_rolling_ball_banded}[method]
    need = rolling_ball_workspace_bytes(B, H, W, Cc)
    dev = images.device
    with torch.cuda.device(dev):
        if workspace is None or workspace.numel() < need:
            workspace = torch.empty(need, dtype=torch.uint8, device=dev)
        if out is None:
            out = torch.empty_like(images)
        args = _lib.RollingBallArgs(images.data_ptr(), out.data_ptr(), B, H, W, Cc, int(radius),
                                    workspace.data_ptr(), workspace.numel())
        _lib.check(entry(C.byref(args), _lib.stream_ptr(dev)))
    return out


def rolling_ball_correction_rgb(image: np.ndarray, radius: int = 50, device: str | torch.device = "cuda") -> np.ndarray:
    """Drop-in for reference utils/data_loader.py:11: u8 [H,W,3] (or [H,W]) numpy in, same shape out."""
    arr = np.ascontiguousarray(image, dtype=np.uint8)
    squeeze = arr.ndim == 2
    if squeeze:
        arr = arr[:, :, None]
    t = torch.from_numpy(arr).to(device)[None]
    out = rolling_ball_device(t, radius)[0].cpu().numpy()
    return out[:, :, 0] if squeeze else out


def resize_linear_u8_device(images: torch.Tensor, dsize, out: torch.Tensor | None = None) -> torch.Tensor:
    """cv2.resize(img, dsize) with the default INTER_LINEAR on u8, bit-exact, for a device batch -- what the two
    resize calls of reference quantify_droplets_batch.py:44 and :57 effectively do (flag in the `dst` slot).
    images: CUDA u8 [B,H,W] or [B,H,W,3]; dsize = (width, height) as in cv2.  Returns [B,dh,dw(,3)]."""
    _lib.require_cuda(images, "images")
    if images.dtype != torch.uint8 or images.dim() not in (3, 4):
        raise TypeError("resize works on uint8 [B,H,W] or [B,H,W,3]")
    images = images.contiguous()
    B, sh, sw = images.shape[:3]
    cn = 1 if images.dim() == 3 else images.shape[3]
    dw, dh = int(dsize[0]), int(dsize[1])
    shape = (B, dh, dw) if images.dim() == 3 else (B, dh, dw, cn)
    if out is None:
        out = torch.empty(shape, dtype=torch.uint8, device=images.device)
    elif tuple(out.shape) != shape or out.dtype != torch.uint8 or not out.is_contiguous():
        raise ValueError(f"out must be a contiguous uint8 tensor of shape {shape}")
    args = _lib.ResizeArgs(images.data_ptr(), out.data_ptr(), B, cn, sh, sw, dh, dw)
    with torch.cuda.device(images.device):
        _lib.check(_lib.load().dc_resize_linear_u8(C.byref(args), _lib.stream_ptr(images.device)))
    return out
