"""Pure-numpy model of the fused upconv + conv kernels' data path (csrc/conv_tc.cu conv_upfused2_kernel and
conv_upfused_wide_kernel) -- test infrastructure, CPU only.

It replays, for ONE tile pair, exactly what the kernels address: the regions as TMA lays them out (haloed x region per
64-channel chunk; the skip tensor as two column-parity planes; zero fill outside the image), the weight blobs row by
row as the producers fetch them (per CTA of the pair), and every MMA of the generated issue code
(csrc/upf_schedule.inc) with its LITERAL descriptor offsets decoded back into (plane, row, column) windows, 32-row
weight sub-tiles, accumulator slots and N.  What comes out is compared with the oracle's evaluation of the composed
layer, so the packer (model.pack_upfused / pack_upfused_wide), the schedule generator and the epilogue's
slot -> parity-class mapping are pinned on a machine without a GPU."""
from __future__ import annotations

import re
from pathlib import Path

import numpy as np

HT_H, HT_W = 16, 8                       # tile of the half-resolution grid
U_W, U_H = HT_W + 2, HT_H + 2            # x region
S_W, S_H = HT_W + 1, 2 * HT_H + 2        # one column-parity plane of the skip region
PLANE16 = (S_W * S_H * 128) >> 4         # plane size in descriptor units (16 bytes)
INC = Path(__file__).resolve().parent.parent / "unet_dc_segmentation_b200" / "csrc" / "upf_schedule.inc"


def issue_code(kind: int):
    """[(group, [(d, a, b, N, fresh_at_k0), ...])] parsed from the generated issue functions."""
    txt = INC.read_text()
    out = []
    for m in re.finditer(rf"upf_issue_group<{kind}, (\d)>\(.*?\) \{{(.*?)\n\}}", txt, re.S):
        calls = re.findall(r"umma_bf16_2sm\(d \+ (\d+)u, a \+ (\d+)ull, b \+ (\d+)ull, 0x([0-9a-f]+)u, ([^)]*)\);", m.group(2))
        out.append((int(m.group(1)), [(int(d), int(a), int(b), ((int(i, 16) >> 17) & 0x3F) << 3, "fresh" in acc)
                                      for d, a, b, i, acc in calls]))
    return out


def x_region(x, h0, w0, chunk):
    """TMA box (64 ch, U_W, U_H) of x [H,W,Cx] at (w0 - 1, h0 - 1), zero filled: [U_H, U_W, 64]."""
    H, W, _ = x.shape
    r = np.zeros((U_H, U_W, 64), np.float32)
    for i in range(U_H):
        for j in range(U_W):
            y, xx = h0 - 1 + i, w0 - 1 + j
            if 0 <= y < H and 0 <= xx < W:
                r[i, j] = x[y, xx, chunk * 64:(chunk + 1) * 64]
    return r


def skip_planes(skip, h0, w0, chunk):
    """The two plane boxes: plane 0 = odd columns 2 w0 - 1, 2 w0 + 1, ...; plane 1 = even columns 2 w0, ...; rows from 2 h0 - 1."""
    H2, W2, _ = skip.shape
    p = np.zeros((2, S_H, S_W, 64), np.float32)
    for q, (par, j0) in enumerate(((1, w0 - 1), (0, w0))):
        for i in range(S_H):
            for j in range(S_W):
                y, xx = 2 * h0 - 1 + i, 2 * (j0 + j) + par
                if 0 <= y < H2 and 0 <= xx < W2 and j0 + j >= 0:
                    p[q, i, j] = skip[y, xx, chunk * 64:(chunk + 1) * 64]
    return p


def window(region_flat_rows, start_row16, sbo_rows):
    """A operand of one MMA for one CTA: 16 groups of 8 consecutive 128-byte rows, groups `sbo_rows` rows apart, from
    the region viewed as a flat list of 128-byte rows; start in descriptor units (8 per row)."""
    assert start_row16 % 8 == 0
    s = start_row16 // 8
    return np.stack([region_flat_rows[s + g * sbo_rows + r] for g in range(16) for r in range(8)])      # [128, 64]


def level1_tile_pair(x, skip, blob, tiles):
    """conv_upfused2_kernel for one pair of tiles [(h0, w0) of CTA 0, (h0, w0) of CTA 1]; x [H,W,128], skip [2H,2W,64],
    blob [2, 2176, 64] (model.pack_upfused).  Returns per CTA the four accumulators [4 slots][128 px][64]."""
    acc = np.zeros((2, 256, 128), np.float32)             # [cta][tmem column = slot * 64 + co][lane = pixel]
    started = np.zeros(4, bool)
    row = 0
    kinds = [(0, 0), (0, 1), (1, None)]                   # (issue kind, x chunk)
    for kind, chunk in kinds:
        if kind == 0:
            flat = [x_region(x, h0, w0, chunk).reshape(-1, 64) for h0, w0 in tiles]
        else:
            flat = [skip_planes(skip, h0, w0, 0).reshape(-1, 64) for h0, w0 in tiles]
        for g, calls in issue_code(kind):
            slot_rows = [blob[c, row:row + 128].astype(np.float32) for c in range(2)]      # this group's ring slot per CTA
            row += 128
            per_k = len(calls) // 4
            for k in range(4):
                for d, a, b, n, fresh in calls[k * per_k:(k + 1) * per_k]:
                    assert (a - 2 * k) % 8 == 0 and (b - 2 * k) % 256 == 0
                    sub = (b - 2 * k) // 256
                    # B: rows [0, N/2) from CTA 0's slot, [N/2, N) from CTA 1's, both at the same offset
                    bt = np.concatenate([slot_rows[c][sub * 32:sub * 32 + n // 2, 16 * k:16 * k + 16] for c in range(2)])   # [N, 16]
                    sbo = U_W if kind == 0 else 2 * S_W
                    for c in range(2):
                        aw = window(flat[c], a - 2 * k, sbo)[:, 16 * k:16 * k + 16]      # [128 px, 16]
                        upd = bt @ aw.T                                                  # [N, 128]
                        if fresh and kind == 0 and chunk == 0 and k == 0:
                            acc[c, d:d + n] = upd
                        else:
                            acc[c, d:d + n] += upd
                    if kind == 0 and chunk == 0 and k == 0:
                        assert fresh == (not started[d // 64:(d + n) // 64].any())
                    started[d // 64:(d + n) // 64] = True
    assert row == 2176 and started.all()
    return acc.reshape(2, 4, 64, 128).transpose(0, 1, 3, 2)           # [cta][slot][px][co]


def scatter_level1(acc_cta, h0, w0, out):
    """Epilogue mapping: slot s = class s ^ (s >> 1) = (py, px); lane = row * 8 + col of the 16 x 8 tile."""
    H2, W2, _ = out.shape
    for s in range(4):
        cls = s ^ (s >> 1)
        py, px = cls >> 1, cls & 1
        for lane in range(128):
            y, xx = 2 * (h0 + lane // HT_W) + py, 2 * (w0 + lane % HT_W) + px
            if y < H2 and xx < W2:
                out[y, xx] = acc_cta[s, lane]


def wide_pass(x, skip, wx, ws, C, h0w0, grp, nt):
    """conv_upfused_wide_kernel: one pass (class group `grp`, n-tile `nt`) of one tile pair; returns [cta][class in group][px][BN]."""
    bn = min(C, 256)
    ncls, ntiles, hb = 256 // bn, C // bn, bn // 2
    sc = C // 64
    acc = np.zeros((2, ncls, 128, bn), np.float32)
    nt_eff = grp * ntiles + nt
    for g in range(sc):
        for r in range(2):
            chunk = 2 * g + r
            flat = [x_region(x, h0, w0, chunk).reshape(-1, 64) for h0, w0 in h0w0]
            for tap in range(4):
                rows = [wx[(((nt_eff * 2 + c) * 2 * sc + chunk) * 4 + tap) * 128:][:128].astype(np.float32) for c in range(2)]
                for half in range(ncls):
                    cls = grp * ncls + half
                    py, px = cls >> 1, cls & 1
                    off = (py * U_W + px) * 8 + ((tap >> 1) * U_W + (tap & 1)) * 8
                    bt = np.concatenate([rows[c][half * hb:(half + 1) * hb] for c in range(2)])          # [BN, 64]
                    for c in range(2):
                        acc[c, half] += window(flat[c], off, U_W) @ bt.T
        planes = [skip_planes(skip, h0, w0, g).reshape(-1, 64) for h0, w0 in h0w0]
        for tap in range(9):
            rows = [ws[(((nt * 2 + c) * sc + g) * 9 + tap) * hb:][:hb].astype(np.float32) for c in range(2)]
            bt = np.concatenate(rows)
            for half in range(ncls):
                cls = grp * ncls + half
                py, px = cls >> 1, cls & 1
                cx = px + tap % 3
                off = (cx & 1) * PLANE16 + ((tap // 3) * S_W + (cx >> 1)) * 8 + py * S_W * 8
                for c in range(2):
                    acc[c, half] += window(planes[c], off, 2 * S_W) @ bt.T
    return acc
