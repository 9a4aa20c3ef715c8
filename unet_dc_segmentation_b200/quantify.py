"""Mask -> droplet table on the GPU (reference quantify_droplets_batch.py:81-95).

``quantify`` keeps the reference signature and DataFrame contract (columns ``label, area,
equivalent_diameter, centroid-0, centroid-1`` [+ ``area_sqmicron, eq_diam_micron``]; an empty,
column-less frame when nothing is left, qdb:87-88).  ``label_stats_device`` is the batched device
entry the fused pipeline uses; both run ``dc_label_stats``.  ``tables_to_csv`` turns a device table into the
per-image CSV files (``dc_table_csv``), byte for byte what pandas writes for those DataFrames (qdb:62-63).
"""
from __future__ import annotations

import ctypes as C
import csv
import io
import locale
from dataclasses import dataclass

import numpy as np
import torch

from . import _lib

COLUMNS = ["label", "area", "equivalent_diameter", "centroid-0", "centroid-1"]
MICRON_COLUMNS = ["area_sqmicron", "eq_diam_micron"]
DEFAULT_CAPACITY = 16384


@dataclass
class DropletTables:
    """Device-resident result of one dc_label_stats call (row r of image b = label r + 1)."""
    counts: torch.Tensor          # int32 [B]
    area: torch.Tensor            # int64 [B, capacity]
    centroid0: torch.Tensor       # f64   [B, capacity]  (row)
    centroid1: torch.Tensor       # f64   [B, capacity]  (col)
    eq_diam: torch.Tensor         # f64   [B, capacity]
    area_um2: torch.Tensor | None
    diam_um: torch.Tensor | None
    labels: torch.Tensor | None   # int32 [B,H,W]
    capacity: int

    def rows(self, a: int, b: int) -> "DropletTables":
        """Views of images [a, b) of this table (same memory): lets a caller archive many batches in one allocation."""
        cut = lambda t: None if t is None else t[a:b]           # noqa: E731
        return DropletTables(self.counts[a:b], self.area[a:b], self.centroid0[a:b], self.centroid1[a:b], self.eq_diam[a:b],
                             cut(self.area_um2), cut(self.diam_um), cut(self.labels), self.capacity)

    def compact_rows(self):
        """Device-side compaction: (counts int64 [B], rows f64 [sum(min(counts, capacity)), C]) with the columns area (bit
        pattern of the int64), equivalent_diameter, centroid-0, centroid-1 [, area_sqmicron, eq_diam_micron], image by
        image.  One boolean-mask gather per column; synchronises (the row count is data dependent)."""
        n = torch.clamp(self.counts.to(torch.int64), max=self.capacity)
        # flat positions of the rows in use: image b, row r -> b * capacity + r, image by image (one data-dependent
        # size, one synchronisation; every column is then a plain gather)
        start = torch.cumsum(n, 0) - n
        total = int(n.sum().item())
        img = torch.repeat_interleave(torch.arange(n.shape[0], device=n.device), n, output_size=total)
        flat = img * self.capacity + (torch.arange(total, device=n.device) - start[img])
        cols = [self.area.view(torch.float64), self.eq_diam, self.centroid0, self.centroid1]
        if self.area_um2 is not None:
            cols += [self.area_um2, self.diam_um]
        out = torch.empty((total, len(cols)), dtype=torch.float64, device=n.device)
        for j, c in enumerate(cols):
            out[:, j] = c.reshape(-1).index_select(0, flat)
        return n, out

    def to_host(self):
        """One D2H per column; returns a list (per image) of dicts of numpy columns."""
        counts = self.counts.cpu().numpy()
        nmax = int(counts.max()) if counts.size else 0
        if nmax > self.capacity:
            raise _lib.DcError(_lib.DC_ECAPACITY, f"droplet table capacity {self.capacity} < {nmax} droplets")
        cols = {"area": self.area[:, :nmax].cpu().numpy(),
                "equivalent_diameter": self.eq_diam[:, :nmax].cpu().numpy(),
                "centroid-0": self.centroid0[:, :nmax].cpu().numpy(),
                "centroid-1": self.centroid1[:, :nmax].cpu().numpy()}
        if self.area_um2 is not None:
            cols["area_sqmicron"] = self.area_um2[:, :nmax].cpu().numpy()
            cols["eq_diam_micron"] = self.diam_um[:, :nmax].cpu().numpy()
        out = []
        for b, n in enumerate(counts):
            n = int(n)
            d = {"label": np.arange(1, n + 1, dtype=np.int64)}
            for k, v in cols.items():
                d[k] = v[b, :n].copy()
            out.append(d)
        return out


def label_workspace_bytes(B: int, H: int, W: int) -> int:
    need = C.c_size_t()
    _lib.check(_lib.load().dc_label_workspace_bytes(B, H, W, C.byref(need)))
    return int(need.value)


def alloc_tables(B: int, capacity: int, micron: bool, device) -> DropletTables:
    """Device buffers for one dc_label_stats call (reusable across calls via label_stats_device(out=...))."""
    counts = torch.empty(B, dtype=torch.int32, device=device)
    area = torch.empty((B, capacity), dtype=torch.int64, device=device)
    c0, c1, dia = (torch.empty((B, capacity), dtype=torch.float64, device=device) for _ in range(3))
    aum = torch.empty((B, capacity), dtype=torch.float64, device=device) if micron else None
    dum = torch.empty((B, capacity), dtype=torch.float64, device=device) if micron else None
    return DropletTables(counts, area, c0, c1, dia, aum, dum, None, capacity)


def label_stats_device(masks: torch.Tensor, min_area: int = 1, px_per_um: float | None = None,
                       capacity: int = DEFAULT_CAPACITY, want_labels: bool = False,
                       workspace: torch.Tensor | None = None, out: DropletTables | None = None) -> DropletTables:
    """masks: CUDA u8 [B,H,W] (non-zero = foreground).  No host synchronisation.
    out: buffers from alloc_tables() to fill instead of allocating (their capacity wins)."""
    _lib.require_cuda(masks, "masks")
    if masks.dtype != torch.uint8 or masks.dim() != 3:
        raise TypeError("masks must be uint8 [B,H,W]")
    masks = masks.contiguous()
    B, H, W = masks.shape
    capacity = int(max(1, min(capacity, (H * W + 1) // 2))) if out is None else out.capacity
    lib = _lib.load()
    dev = masks.device
    need = label_workspace_bytes(B, H, W)
    with torch.cuda.device(dev):
        if workspace is None or workspace.numel() < need:
            workspace = torch.empty(need, dtype=torch.uint8, device=dev)
        micron = bool(px_per_um)
        t = out if out is not None else alloc_tables(B, capacity, micron, dev)
        if t.counts.shape[0] != B or (micron and t.area_um2 is None):
            raise ValueError("out tables do not match this call (batch size / micron columns)")
        counts, area, c0, c1, dia, aum, dum = t.counts, t.area, t.centroid0, t.centroid1, t.eq_diam, t.area_um2, t.diam_um
        labels = torch.empty((B, H, W), dtype=torch.int32, device=dev) if want_labels else None
        args = _lib.LabelArgs(
            masks.data_ptr(), B, H, W, int(min_area), float(px_per_um) if micron else 0.0,
            labels.data_ptr() if want_labels else None, capacity, counts.data_ptr(),
            area.data_ptr(), c0.data_ptr(), c1.data_ptr(), dia.data_ptr(),
            aum.data_ptr() if micron else None, dum.data_ptr() if micron else None,
            workspace.data_ptr(), workspace.numel())
        _lib.check(lib.dc_label_stats(C.byref(args), _lib.stream_ptr(dev)))
    return DropletTables(counts, area, c0, c1, dia, aum if micron else None, dum if micron else None, labels, capacity)


def quantify_arrays(masks: torch.Tensor, min_area: int = 1, px_per_um: float | None = None,
                    want_labels: bool = False, capacity: int = DEFAULT_CAPACITY):
    """Batched quantify with automatic capacity growth.  Returns (list of column dicts, labels or None)."""
    t = label_stats_device(masks, min_area, px_per_um, capacity, want_labels)
    nmax = int(t.counts.max().item())
    if nmax > t.capacity:   # counts are exact even on overflow: rerun once with room for everything
        t = label_stats_device(masks, min_area, px_per_um, nmax, want_labels)
    return t.to_host(), (t.labels if want_labels else None)


def quantify(bin_mask, min_area: int = 1, px_per_um: float | None = None, device: str | torch.device = "cuda"):
    """Drop-in for reference quantify_droplets_batch.py:81: u8 [H,W] mask -> pandas.DataFrame."""
    import pandas as pd
    if isinstance(bin_mask, torch.Tensor):
        m = bin_mask.to(device=device, dtype=torch.uint8)
    else:
        m = torch.from_numpy(np.ascontiguousarray(bin_mask).astype(np.uint8, copy=False)).to(device)
    if m.dim() != 2:
        raise ValueError(f"quantify takes one [H,W] mask, got {tuple(m.shape)}")
    tables, _ = quantify_arrays(m[None], min_area, px_per_um)
    cols = tables[0]
    if len(cols["label"]) == 0:
        return pd.DataFrame()                                   # qdb:87-88
    order = COLUMNS + (MICRON_COLUMNS if px_per_um else [])
    return pd.DataFrame({k: cols[k] for k in order})


# ------------------------------------------------------------------ table -> CSV text (dc_table_csv)
def text_encoding() -> str:
    """The encoding Path.write_text uses (UTF-8 mode: UTF-8; otherwise the locale's)."""
    enc = io.text_encoding(None)
    return locale.getencoding() if enc == "locale" else enc


def csv_field(name: str, encoding: str | None = None) -> bytes:
    """`name` as the filename field of pandas' to_csv (csv QUOTE_MINIMAL: quoted, quotes doubled, when it holds a comma,
    a quote or a line break), encoded as Path.write_text would (``encoding`` None) or in ``encoding``."""
    buf = io.StringIO()
    csv.writer(buf, lineterminator="\n", quoting=csv.QUOTE_MINIMAL).writerow([name, ""])
    return buf.getvalue()[:-2].encode(encoding or text_encoding())


def pack_fields(fields) -> tuple[np.ndarray, np.ndarray]:
    """Filename fields (bytes) -> (u8 buffer, int64 offsets [B+1]) as dc_table_csv takes them."""
    offsets = np.zeros(len(fields) + 1, dtype=np.int64)
    offsets[1:] = np.cumsum([len(f) for f in fields])
    return np.frombuffer(b"".join(fields) or b"\0", dtype=np.uint8), offsets


def table_csv_bounds(B: int, capacity: int, micron: bool, names_bytes: int) -> tuple[int, int]:
    """(text bytes that always suffice, workspace bytes) for dc_table_csv."""
    out, ws = C.c_int64(), C.c_size_t()
    _lib.check(_lib.load().dc_table_csv_bounds(B, capacity, int(micron), names_bytes, C.byref(out), C.byref(ws)))
    return int(out.value), int(ws.value)


def table_csv_device(t: "DropletTables", names: torch.Tensor, name_offsets: torch.Tensor, names_bytes: int,
                     out: torch.Tensor, frame_offsets: torch.Tensor, area_sum: torch.Tensor, workspace: torch.Tensor):
    """Enqueue dc_table_csv on the current stream (no synchronisation, no allocation): frame b's file text lands in
    out[frame_offsets[b]:frame_offsets[b+1]], its area sum in area_sum[b].  names / name_offsets: device copies of
    pack_fields(); names_bytes: the largest names total these buffers will hold (sizes the bound)."""
    B = t.counts.shape[0]
    micron = t.area_um2 is not None
    args = _lib.TableCsvArgs(
        B, t.capacity, t.counts.data_ptr(), t.area.data_ptr(), t.eq_diam.data_ptr(), t.centroid0.data_ptr(),
        t.centroid1.data_ptr(), t.area_um2.data_ptr() if micron else None, t.diam_um.data_ptr() if micron else None,
        names.data_ptr(), name_offsets.data_ptr(), int(names_bytes), out.data_ptr(), out.numel(),
        frame_offsets.data_ptr(), area_sum.data_ptr(), workspace.data_ptr(), workspace.numel())
    _lib.check(_lib.load().dc_table_csv(C.byref(args), _lib.stream_ptr(t.counts.device)))


@dataclass
class CsvTables:
    """Per-image CSV files of one batch, read back to the host."""
    texts: list                   # bytes per image: the file quantify_droplets_batch.py:63 writes
    counts: np.ndarray            # int64 [B] droplets per image
    area_sums: np.ndarray         # int64 [B] sum of the area column (summary_per_image.csv's total_area_px)
    sizes: list                   # f64 per image: eq_diam_micron with micron columns, else equivalent_diameter


def csv_text_device(t: "DropletTables", names: torch.Tensor, name_offsets: torch.Tensor, names_bytes: int):
    """dc_table_csv into fresh device buffers on the current stream: (text u8, frame_offsets int64 [B+1], area_sum)."""
    dev = t.counts.device
    B = t.counts.shape[0]
    nbytes, wsb = table_csv_bounds(B, t.capacity, t.area_um2 is not None, names_bytes)
    out = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    off = torch.empty(B + 1, dtype=torch.int64, device=dev)
    asum = torch.empty(B, dtype=torch.int64, device=dev)
    ws = torch.empty(wsb, dtype=torch.uint8, device=dev)
    table_csv_device(t, names, name_offsets, names_bytes, out, off, asum, ws)
    return out, off, asum


def tables_to_csv(t: "DropletTables", filenames) -> CsvTables:
    """Device droplet table + one filename per image -> the per-image CSV files as bytes (synchronises).  A table whose
    capacity some image exceeds raises DC_ECAPACITY (re-run label_stats_device with room for every droplet)."""
    counts = t.counts.cpu().numpy().astype(np.int64)
    if counts.size and int(counts.max()) > t.capacity:
        raise _lib.DcError(_lib.DC_ECAPACITY, f"droplet table capacity {t.capacity} < {int(counts.max())} droplets")
    buf, offs = pack_fields([csv_field(f) for f in filenames])
    dev = t.counts.device
    with torch.cuda.device(dev):
        names = torch.from_numpy(buf.copy()).to(dev)
        name_off = torch.from_numpy(offs).to(dev)
        out, off, asum = csv_text_device(t, names, name_off, int(offs[-1]))
    off = off.cpu().numpy()
    text = out[:int(off[-1])].cpu().numpy()
    size = t.diam_um if t.area_um2 is not None else t.eq_diam
    sizes = [size[b, :n].cpu().numpy() for b, n in enumerate(counts)]
    return CsvTables([text[off[b]:off[b + 1]].tobytes() for b in range(counts.size)], counts, asum.cpu().numpy(), sizes)
