"""Frames for the PNG encoder's tests (tests/test_png_format.py, tests/test_gpu_png.py), and the zlib oracle: what
cv2.imencode(".png", img) writes, rebuilt from the standard library's zlib (level 1, Z_RLE, memLevel 8 on the
SUB-filtered rows, libpng's zlib-header window rewrite, 8192-byte IDAT chunks)."""
import heapq
import struct
import zlib

import numpy as np


def png_like_cv2(img: np.ndarray) -> bytes:
    H, W = img.shape[:2]
    c = 1 if img.ndim == 2 else 3
    rows = (img if c == 1 else img[..., ::-1]).reshape(H, W * c).astype(np.int16)
    ft = 0 if W == 1 else 1                  # SUB, except None for one-pixel-wide images
    f = rows.copy()
    if ft:
        f[:, c:] = (rows[:, c:] - rows[:, :-c]) % 256
    raw = np.concatenate([np.full((H, 1), ft, np.uint8), f.astype(np.uint8)], 1).tobytes()
    co = zlib.compressobj(1, zlib.DEFLATED, 15, 8, zlib.Z_RLE)
    z = bytearray(co.compress(raw) + co.flush())
    if len(raw) <= 16384:                    # libpng optimize_cmf
        cinfo = z[0] >> 4
        half = 1 << (cinfo + 7)
        if len(raw) <= half:
            while True:
                half >>= 1
                cinfo -= 1
                if not (cinfo > 0 and len(raw) <= half):
                    break
            z[0] = (z[0] & 0x0F) | (cinfo << 4)
            t = z[1] & 0xE0
            z[1] = t + 0x1F - ((z[0] << 8) + t) % 0x1F

    def chunk(tag, data):
        return struct.pack(">I", len(data)) + tag + data + struct.pack(">I", zlib.crc32(tag + data))
    z = bytes(z)
    ihdr = struct.pack(">IIBBBBB", W, H, 8, 0 if c == 1 else 2, 0, 0, 0)
    return (b"\x89PNG\r\n\x1a\n" + chunk(b"IHDR", ihdr)
            + b"".join(chunk(b"IDAT", z[i:i + 8192]) for i in range(0, len(z), 8192)) + chunk(b"IEND", b""))


def from_filtered(f: np.ndarray) -> np.ndarray:
    """The grey image [H,W] whose SUB-filtered rows are f [H,W] (each row's stream is then 1, f[y])."""
    return (np.cumsum(f.astype(np.int64), axis=1) % 256).astype(np.uint8)


def no_repeat_sequence(counts: dict, seed: int = 0) -> np.ndarray:
    """counts[v] copies of every byte v with no two neighbours equal: every byte is a literal of the RLE parse."""
    rs = np.random.default_rng(seed)
    h = [(-c, rs.random(), v) for v, c in counts.items() if c > 0]
    heapq.heapify(h)
    out, prev = [], None
    while h:
        c, r, v = heapq.heappop(h)
        if v == prev:
            c2, r2, v2 = heapq.heappop(h)
            heapq.heappush(h, (c, r, v))
            c, r, v = c2, r2, v2
        out.append(v)
        prev = v
        if c + 1:
            heapq.heappush(h, (c + 1, r, v))
    return np.array(out, np.uint8)


def paint_overlay(img: np.ndarray, stencil: np.ndarray) -> np.ndarray:
    out = img.copy()
    out[stencil.astype(bool)] = (0, 255, 0)
    return out


def corpus_for_shape(H: int, W: int, seed: int = 0) -> dict:
    """Every kind of frame the CLI writes, and the extremes, at one shape."""
    rs = np.random.default_rng(seed + 1000 * H + W)
    yy, xx = np.mgrid[:H, :W]
    mask = (((yy - H / 3) ** 2 + (xx - W / 2) ** 2) < (min(H, W) / 4) ** 2).astype(np.uint8) * 255
    grey = rs.normal(120, 20, (H, W)).clip(0, 255).astype(np.uint8)
    bgr = rs.normal(120, 20, (H, W, 3)).clip(0, 255).astype(np.uint8)
    ring = (mask > 0) & ~np.roll(mask > 0, 2, axis=1)
    return {"mask": mask, "zeros": np.zeros((H, W), np.uint8), "full": np.full((H, W), 255, np.uint8),
            "checker": (((yy + xx) % 2) * 255).astype(np.uint8), "grey": grey, "bgr": bgr,
            "overlay": paint_overlay(bgr, ring), "uniform": rs.integers(0, 256, (H, W, 3), dtype=np.uint8)}


SHAPES = [(1, 1), (1, 9), (13, 1), (2, 2), (40, 60), (90, 181), (128, 128), (276, 408), (1024, 1024)]


def run_row(runs) -> np.ndarray:
    """One filtered row made of runs [(value, length)]."""
    parts = [np.full(n, v, np.uint8) for v, n in runs]
    return np.concatenate(parts)


def crafted() -> dict:
    """Filtered streams built through the inverse filter, each reaching one corner of the parse or the trees."""
    out = {}
    lens = [1, 2, 3, 4, 258, 259, 260, 261, 262, 516, 517]
    for n in lens:
        # a run of n at the stream start: the filter byte 1 followed by n - 1 more ones, then other bytes
        row = np.concatenate([np.ones(n - 1, np.uint8), np.array([7, 9, 7], np.uint8)])
        out[f"start_run_{n}"] = from_filtered(row[None])
        # ... and at the end of the stream
        out[f"end_run_{n}"] = from_filtered(np.concatenate([np.array([7, 9], np.uint8), np.full(n, 5, np.uint8)])[None])
    # runs of every length in one row, and runs that cross rows (row end 1 + next row's filter byte 1)
    row = run_row([(v % 200 + 2, n) for v, n in enumerate(lens * 3)])
    out["runs_mixed"] = from_filtered(row[None])
    rows = np.full((6, 300), 1, np.uint8)
    rows[:, :5] = np.arange(5, 10)
    out["runs_across_rows"] = from_filtered(rows)
    # exactly 2 * 16383 literal symbols: two full blocks and an empty final one
    out["empty_final_block"] = from_filtered(np.tile(np.array([2, 3], np.uint8), 16383)[None, :32765])
    # small masks: fixed codes win
    m = np.zeros((12, 20), np.uint8)
    m[3:9, 4:15] = 255
    out["small_mask"] = m
    # Fibonacci literal frequencies (the filter byte and END_BLOCK are the two 1s): code lengths past 15 bits
    fib = [1, 1]
    while len(fib) < 19:
        fib.append(fib[-1] + fib[-2])
    out["fib_15_bits"] = from_filtered(no_repeat_sequence({10 + i: c for i, c in enumerate(fib[2:])})[None])
    # power-law literal frequencies on shuffled byte values: bit-length code lengths past 7 bits
    vals = np.random.default_rng(1).permutation(256)
    fr = np.floor(3000 / (np.arange(256) + 1) ** 1.1).astype(int)
    out["bl_7_bits"] = from_filtered(no_repeat_sequence({int(v): int(c) for v, c in zip(vals, fr) if c > 0}, 1)[None])
    # a stored block holding a match (of 29 bytes, with extra length bits), then a compressed block
    rs = np.random.default_rng(2)
    f = np.zeros(59999, np.uint8)
    f[:20000] = no_repeat_sequence({v: 80 for v in range(256)}, 2)[:20000]
    f[5000:5030] = f[4999] ^ 1 if f[5030] != f[4999] ^ 1 else f[4999] ^ 2
    out["stored_match_then_dynamic"] = from_filtered(f[None])
    # uniform bytes (stored blocks) with a painted horizontal line (0, 255, 0 filters to runs of zeros)
    u = rs.integers(0, 256, (64, 700, 3), dtype=np.uint8)
    u[20, 50:650] = (0, 255, 0)
    u[41:43, :] = (0, 255, 0)
    out["uniform_with_line"] = u
    return out
