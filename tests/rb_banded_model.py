"""numpy model of csrc/morph.cu's morph_band_kernel (the rolling ball's banded pass for radii past the tiled kernel),
driven by the ACTUAL rectangle table the C++ host code builds (dc_debug_rolling_ball_bands, host only).  Test
infrastructure: it pins the rectangle builder and the kernel's data path (bands of T output rows, 4-pixel words,
van Herk blocks scanned in pieces with carries between pieces, identity padding) on the CPU."""
from __future__ import annotations

import ctypes as C

import numpy as np


def load_bands(radius: int) -> dict:
    from unet_dc_segmentation_b200 import _lib
    lib = _lib.load()
    cap = 3 + 4 * 1024
    buf = (C.c_int * cap)()
    n = lib.dc_debug_rolling_ball_bands(radius, buf, cap)
    if n < 0:
        raise RuntimeError(lib.dc_last_error().decode())
    v = list(buf[:n])
    k, K, piece = v[:3]
    assert n == 3 + 4 * K
    rects = [tuple(v[3 + 4 * m: 7 + 4 * m]) for m in range(K)]
    return {"k": k, "K": K, "piece": piece, "rects": rects}


def smem_pitches(W: int, bands: dict) -> tuple[int, int, int]:
    """(vp, lp, cp): bytes per output row of V / A, of P / S and of the piece carries, as the launcher sizes them."""
    G = bands["piece"]
    vp = 4 * ((W + 3) // 4)
    wmax, cmax = 0, 0
    for ya, yb, xa, xb in bands["rects"]:
        w = xb - xa + 1
        L = W + w - 1
        npc = -(-w // G)
        wmax = max(wmax, w)
        if npc > 1:
            cmax = max(cmax, -(-L // w) * npc)
    return vp, (vp + wmax + 8 + 15) & ~15, (cmax + 15) & ~15


def band_pass(img: np.ndarray, bands: dict, is_max: bool, T: int) -> np.ndarray:
    """One erode (is_max False) / dilate pass over a u8 [H,W] plane, band of T rows by band, as the kernel does it."""
    H, W = img.shape
    G = bands["piece"]
    ident = 0 if is_max else 255
    op = np.maximum if is_max else np.minimum
    vp, lp, cp = smem_pitches(W, bands)
    rects = bands["rects"]
    out = np.empty_like(img)
    for y0 in range(0, H, T):
        rows = y0 + np.arange(T)

        def fold(V, dys):
            for dy in dys:
                yy = rows + dy
                ok = (yy >= 0) & (yy < H)
                word_row = np.full((T, vp), ident, np.uint8)          # 4-pixel words, bytes past W are the identity
                word_row[ok, :W] = img[yy[ok]]
                V = op(V, word_row)
            return V

        ya, yb = rects[0][:2]
        V = fold(np.full((T, vp), ident, np.uint8), range(ya, yb + 1))
        A = np.full((T, vp), ident, np.uint8)
        pya, pyb = ya, yb
        for m, (ya, yb, xa, xb) in enumerate(rects):
            assert (ya, yb) == (pya, pyb)
            w = xb - xa + 1
            L = W + w - 1
            nb, npc = -(-L // w), -(-w // G)
            # padded coordinate u = x' - xa: identity outside the image's columns
            u = np.arange(L)
            x = u + xa
            vals = np.full((T, L), ident, np.uint8)
            inside = (x >= 0) & (x < W)
            vals[:, inside] = V[:, x[inside]]
            # pieces: block blk = u // w, piece pc = (u % w) // G, slot j = (u % w) % G
            blk = u // w
            off = u - blk * w
            pc, j = off // G, off % G
            pid = blk * npc + pc
            assert pid.max() < nb * npc and (npc == 1 or nb * npc <= cp)
            pieces = np.full((T, nb * npc, G), ident, np.uint8)
            pieces[:, pid, j] = vals
            pre = op.accumulate(pieces, axis=2)
            suf = op.accumulate(pieces[:, :, ::-1], axis=2)[:, :, ::-1]
            # carries: extremum of the earlier (later) pieces of the same block
            tot = pre[:, :, -1].reshape(T, nb, npc)
            pc_carry = np.full_like(tot, ident)
            sc_carry = np.full_like(tot, ident)
            if npc > 1:
                pc_carry[:, :, 1:] = op.accumulate(tot, axis=2)[:, :, :-1]
                sc_carry[:, :, :-1] = op.accumulate(tot[:, :, ::-1], axis=2)[:, :, ::-1][:, :, 1:]
            P = op(pre[:, pid, j], pc_carry.reshape(T, -1)[:, pid])
            S = op(suf[:, pid, j], sc_carry.reshape(T, -1)[:, pid])
            # output x takes S[x] and P[x + w - 1]; the kernel reads P as two words up to byte 4 ww + w + 6 < lp
            assert (vp - 4) + w - 1 + 7 < lp
            A[:, :W] = op(A[:, :W], op(S[:, :W], P[:, w - 1:w - 1 + W]))
            if m + 1 < len(rects):
                nya, nyb = rects[m + 1][:2]
                assert nya <= pya and nyb >= pyb, "bands must grow along the walk"
                V = fold(V, list(range(nya, pya)) + list(range(pyb + 1, nyb + 1)))
                pya, pyb = nya, nyb
        hh = min(T, H - y0)
        out[y0:y0 + hh] = A[:hh, :W]
    return out
