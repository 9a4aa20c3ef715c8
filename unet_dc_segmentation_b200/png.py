"""PNG files of u8 frames encoded on the GPU (dc_png_encode), byte for byte what ``cv2.imwrite`` writes with its
default parameters: the mask PNGs of reference quantify_droplets_batch.py:58 and the overlays of :78.

``encode_png_device`` encodes a batch into one device buffer; ``encode_png`` is ``cv2.imencode(".png", img)[1]
.tobytes()`` for one host frame.  ``device_matches_opencv`` compares both on probe images once per process: an OpenCV
built on another zlib (zlib-ng, for example) writes other bytes, and callers then keep writing through cv2.
"""
from __future__ import annotations

import ctypes as C
import functools

import numpy as np
import torch

from . import _lib


def png_bounds(B: int, H: int, W: int, C_: int) -> tuple[int, int]:
    """(out_bytes, workspace_bytes) for a batch of B frames [H,W] (C_ = 1) or [H,W,3] (C_ = 3): static worst cases."""
    out, ws = C.c_int64(), C.c_size_t()
    _lib.check(_lib.load().dc_png_bounds(int(B), int(H), int(W), int(C_), C.byref(out), C.byref(ws)))
    return int(out.value), int(ws.value)


def _shape(images: torch.Tensor) -> tuple[int, int, int, int]:
    if images.dtype != torch.uint8 or images.dim() not in (3, 4) or (images.dim() == 4 and images.shape[3] != 3):
        raise TypeError("images must be uint8 [B,H,W] or BGR [B,H,W,3]")
    B, H, W = (int(x) for x in images.shape[:3])
    return B, H, W, 1 if images.dim() == 3 else 3


def encode_png_device(images: torch.Tensor, out: torch.Tensor | None = None, workspace: torch.Tensor | None = None,
                      offsets: torch.Tensor | None = None):
    """images: CUDA u8 [B,H,W] or BGR [B,H,W,3] -> (buffer, offsets): frame b's PNG file is
    buffer[offsets[b]:offsets[b+1]] (u8 and int64 CUDA tensors).  out / workspace / offsets: preallocated buffers (out and
    workspace of at least ``png_bounds`` bytes, the workspace 256-byte aligned as torch allocations are; offsets int64
    [B+1]), for CUDA-graph capture.  Runs on the current stream."""
    _lib.require_cuda(images, "images")
    B, H, W, C_ = _shape(images)
    images = images.contiguous()
    dev = images.device
    need, wsb = png_bounds(B, H, W, C_)
    with torch.cuda.device(dev):
        if out is None:
            out = torch.empty(need, dtype=torch.uint8, device=dev)
        if workspace is None:
            workspace = torch.empty(wsb, dtype=torch.uint8, device=dev)
        for name, t, n in (("out", out, need), ("workspace", workspace, wsb)):
            if t.dtype != torch.uint8 or t.device != dev or not t.is_contiguous() or t.numel() < n:
                raise ValueError(f"{name} must be a contiguous uint8 tensor of at least {n} bytes on the images' device")
        if offsets is None:
            offsets = torch.empty(B + 1, dtype=torch.int64, device=dev)
        elif offsets.dtype != torch.int64 or offsets.device != dev or not offsets.is_contiguous() or offsets.numel() != B + 1:
            raise ValueError("offsets must be a contiguous int64 [B+1] tensor on the images' device")
        args = _lib.PngArgs(images.data_ptr(), B, H, W, C_, out.data_ptr(), out.numel(), offsets.data_ptr(),
                            workspace.data_ptr(), workspace.numel())
        _lib.check(_lib.load().dc_png_encode(C.byref(args), _lib.stream_ptr(dev)))
    return out, offsets


def encode_png(img: np.ndarray, device: torch.device | str = "cuda") -> bytes:
    """``cv2.imencode(".png", img)[1].tobytes()`` for one u8 [H,W] or BGR [H,W,3] frame, encoded on the GPU."""
    img = np.ascontiguousarray(img)
    buf, off = encode_png_device(torch.from_numpy(img[None]).to(device))
    off = off.cpu().numpy()
    return buf[int(off[0]):int(off[1])].cpu().numpy().tobytes()


def encode_png_host(img: np.ndarray, stats: bool = False):
    """The encoder's code compiled for the host (a test aid, no GPU needed): the same bytes as ``encode_png``.
    stats: also return every deflate block's type | 4 (code lengths limited to 15) | 8 (bit lengths limited to 7)."""
    img = np.ascontiguousarray(img)
    if img.dtype != np.uint8 or img.ndim not in (2, 3) or (img.ndim == 3 and img.shape[2] != 3):
        raise TypeError("img must be uint8 [H,W] or BGR [H,W,3]")
    H, W = img.shape[:2]
    C_ = 1 if img.ndim == 2 else 3
    need, _ = png_bounds(1, H, W, C_)
    out = np.empty(need, dtype=np.uint8)
    n, nb = C.c_int64(), C.c_int64()
    cap = (H * (1 + W * C_)) // 16383 + 2
    st = np.zeros(cap, dtype=np.int32)
    _lib.check(_lib.load().dc_debug_png_host(img.ctypes.data, H, W, C_, out.ctypes.data, out.size, C.byref(n),
                                             st.ctypes.data, cap, C.byref(nb)))
    data = out[:n.value].tobytes()
    return (data, st[:nb.value].copy()) if stats else data


def probe_images() -> list[np.ndarray]:
    """Small frames whose encodings use stored, fixed and dynamic blocks between them."""
    rs = np.random.default_rng(7)
    mask = np.zeros((40, 60), np.uint8)
    mask[10:25, 15:40] = 255
    grey = (rs.normal(120, 20, (64, 96)).clip(0, 255)).astype(np.uint8)
    tiny = np.zeros((4, 4), np.uint8)
    return [tiny,                                                           # fixed
            rs.integers(0, 256, (24, 32, 3), dtype=np.uint8),               # stored
            mask, grey,                                                     # dynamic
            np.dstack([grey, grey // 2, mask[:1].repeat(64, 0)[:, :1].repeat(96, 1)])]


@functools.lru_cache(maxsize=None)
def device_matches_opencv(device_index: int = 0) -> bool:
    """Whether the installed OpenCV writes the bytes dc_png_encode writes, on the probe images (once per process)."""
    import cv2
    dev = torch.device("cuda", device_index)
    for img in probe_images():
        ok, want = cv2.imencode(".png", img)
        if not ok or encode_png(img, dev) != want.tobytes():
            return False
    return True
