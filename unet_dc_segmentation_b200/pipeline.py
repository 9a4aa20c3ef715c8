"""Fused device pipeline: u8 images -> (u8 masks, droplet tables).

The device-side composition of reference quantify_droplets_batch.py: ``preprocess`` (:40-46, at native
size, where both cv2.resize calls are the identity) -> ``model(batch)`` (:52) -> ``> thresh`` (:56) ->
``quantify`` (:61, :81-95), for a whole batch at a time with nothing but the u8 images going up and
the u8 masks + per-droplet rows coming back.

Stages, all on the current CUDA stream (no host synchronisation until the tables are fetched):
  dc_rolling_ball   (grayscale input: one plane per image -- the three RGB channels the reference
                     builds with Image.convert("RGB") are identical, so they are corrected once)
  dc_forward        stem reads the corrected u8 plane and does the /255 (qdb:45); the last conv's
                     epilogue does out_conv + sigmoid + `> prob_thresh` and writes the u8 mask
  dc_label_stats    labelling, min_area filter, compaction, area / centroid / diameter (+ micron columns)
  dc_table_csv      (run_host_pipelined(csv=True)) the per-image CSV files as text, formatted on the device
  dc_png_encode     (run_host_pipelined(png=True)) the mask PNGs (x 255) and the painted overlays as PNG files
"""
from __future__ import annotations

from contextlib import contextmanager
from dataclasses import dataclass

import numpy as np
import torch

from . import _lib
from .model import UNetDC
from .morphology import resize_linear_u8_device, rolling_ball_device, rolling_ball_workspace_bytes
from .overlay import OVERLAY_BGR, overlay_stencil_device, overlay_workspace_bytes
from .png import encode_png_device, png_bounds
from .quantify import (DEFAULT_CAPACITY, CsvTables, DropletTables, alloc_tables, csv_field, csv_text_device,
                       label_stats_device, label_workspace_bytes, pack_fields, table_csv_bounds, table_csv_device)


@contextmanager
def _nvtx(name: str):
    """NVTX range per stage (visible to nsys / ncu --nvtx; free otherwise), closed even when the stage raises."""
    torch.cuda.nvtx.range_push(name)
    try:
        yield
    finally:
        torch.cuda.nvtx.range_pop()


@dataclass
class PngFiles:
    masks: list                    # bytes of every frame's {name}_pred.png (cv2.imwrite of mask * 255, qdb:58)
    overlays: list | None          # bytes of every frame's overlay PNG (qdb:78); None where the frame had no base


@dataclass
class BatchResult:
    masks: torch.Tensor            # u8 [B,H,W] {0,1} (device)
    tables: DropletTables          # device-resident table
    probs: torch.Tensor | None     # f32 [B,1,H,W] when requested
    stencil: torch.Tensor | None = None   # u8 [B,H,W] overlay stencil (qdb:76-77) when requested


class DropletPipeline:
    def __init__(self, model: UNetDC, background_radius: int | None = 50, prob_thresh: float = 0.3,
                 min_area: int = 1, px_per_micron: float | None = None, capacity: int = DEFAULT_CAPACITY,
                 img_size: int | None = None, use_graphs: bool = False):
        """img_size: network input size.  None = native resolution (frames must be multiples of 16; both resizes of
        the reference are then the identity).  An integer reproduces the as-shipped flow (IMG_SIZE = 512, qdb:30):
        corrected frames are resized to img_size x img_size (qdb:44) and the mask is resized back to the frame size
        (qdb:57), both with cv2's effective INTER_LINEAR, on the device.
        use_graphs: ``run_host_pipelined`` captures the ~35 kernel launches of a batch into one CUDA graph per buffer
        slot (after one eager pass) and replays it: the launch-bound small-batch configurations (8 x 256^2 is 0.3 ms of
        GPU work behind 35 launches) then cost one launch per batch."""
        self.model = model
        self.img_size = img_size
        self.background_radius = background_radius
        self.prob_thresh = float(prob_thresh)
        self.min_area = int(min_area)
        self.px_per_micron = px_per_micron
        self.capacity = int(capacity)
        self._rb_ws = None
        self._rb_out = None
        self._ccl_ws = None
        self._ovl_ws = None
        self._staging = None
        self._slots = [None, None]       # run_host_pipelined's device / pinned buffers, kept across calls
        self._streams = None
        self.use_graphs = bool(use_graphs)

    # ------------------------------------------------------------------ device-resident entry
    def run_device(self, images: torch.Tensor, return_prob: bool = False, want_labels: bool = False,
                   mask_out: torch.Tensor | None = None, tables_out: DropletTables | None = None,
                   want_overlay: bool = False, stencil_out: torch.Tensor | None = None) -> BatchResult:
        """images: CUDA u8 [B,H,W] grayscale or [B,H,W,3].  mask_out / tables_out / stencil_out: preallocated outputs.
        want_overlay: also compute the pixels the reference's findContours + drawContours paint (qdb:76-77)."""
        _lib.require_cuda(images, "images")
        x = images
        with _nvtx("dc:rolling_ball"):
            if self.background_radius:
                if self._rb_out is None or self._rb_out.shape != x.shape or self._rb_out.device != x.device:
                    self._rb_out = torch.empty_like(x)
                    self._rb_ws = None
                if self._rb_ws is None:
                    need = rolling_ball_workspace_bytes(x.shape[0], x.shape[1], x.shape[2], 1 if x.dim() == 3 else x.shape[3])
                    self._rb_ws = torch.empty(need, dtype=torch.uint8, device=x.device)
                x = rolling_ball_device(x, self.background_radius, out=self._rb_out, workspace=self._rb_ws)
        with _nvtx("dc:forward"):
            oh, ow = int(images.shape[1]), int(images.shape[2])
            resized = self.img_size is not None and (oh, ow) != (self.img_size, self.img_size)
            if resized:
                x = resize_linear_u8_device(x, (self.img_size, self.img_size))                     # qdb:44
                masks, probs = self.model.predict_u8(x, self.prob_thresh, return_prob=return_prob)
                masks = resize_linear_u8_device(masks, (ow, oh), out=mask_out)                     # qdb:57
            else:
                masks, probs = self.model.predict_u8(x, self.prob_thresh, return_prob=return_prob, mask_out=mask_out)
        with _nvtx("dc:label_stats"):
            need = label_workspace_bytes(*masks.shape)
            if self._ccl_ws is None or self._ccl_ws.device != masks.device or self._ccl_ws.numel() < need:
                self._ccl_ws = torch.empty(need, dtype=torch.uint8, device=masks.device)
            tables = label_stats_device(masks, self.min_area, self.px_per_micron, self.capacity,
                                        want_labels=want_labels, workspace=self._ccl_ws, out=tables_out)
        stencil = None
        if want_overlay:
            need = overlay_workspace_bytes(*masks.shape)
            if self._ovl_ws is None or self._ovl_ws.device != masks.device or self._ovl_ws.numel() < need:
                self._ovl_ws = torch.empty(need, dtype=torch.uint8, device=masks.device)
            stencil = overlay_stencil_device(masks, out=stencil_out, workspace=self._ovl_ws)
        return BatchResult(masks, tables, probs, stencil)

    # ------------------------------------------------------------------ host entry (what a user calls)
    def run_host(self, images: torch.Tensor | np.ndarray, device: torch.device | str = "cuda"):
        """images: host u8 [B,H,W] or [B,H,W,3] (pinned for async copies).  Returns
        (masks u8 numpy [B,H,W], list of per-image column dicts).  H2D of the images and D2H of the
        masks and table rows are part of this call."""
        if isinstance(images, np.ndarray):
            images = torch.from_numpy(np.ascontiguousarray(images))
        if images.dtype != torch.uint8:
            raise TypeError("images must be uint8")
        dev = torch.device(device)
        if self._staging is None or self._staging.shape != images.shape or self._staging.device != dev:
            self._staging = torch.empty(images.shape, dtype=torch.uint8, device=dev)
        self._staging.copy_(images, non_blocking=True)
        res = self.run_device(self._staging)
        masks = res.masks.to("cpu", non_blocking=False)
        tables = res.tables
        nmax = int(tables.counts.max().item())
        if nmax > tables.capacity:
            self.capacity = nmax
            tables = label_stats_device(res.masks, self.min_area, self.px_per_micron, nmax)
        return masks.numpy(), tables.to_host()

    # ------------------------------------------------------------------ pipelined host entry
    def run_host_pipelined(self, batches, device: torch.device | str = "cuda", copy: bool = True,
                           want_overlay: bool = False, tables_archive: DropletTables | None = None, csv: bool = False,
                           png: bool = False):
        """Generator over host batches (each u8 [B,H,W] or [B,H,W,3], ideally pinned; all the same shape):
        yields (masks u8 numpy [B,H,W], list of per-image column dicts) per batch, in order.

        Four streams (copy-in, compute, one read-back stream per slot) and two buffer slots: the H2D copy of batch
        k+1 and the D2H copy of batch k-1 run while
        batch k computes, so the steady-state rate is the device rate, not device + PCIe.

        Everything yielded is owned by the caller (``list(pipe.run_host_pipelined(...))`` is safe).  ``copy=False``
        yields the masks as a VIEW of the pipeline's two-slot pinned read-back buffer instead: that view is valid
        only until the generator is advanced again (the next batch's read-back is queued into the other slot and the
        one after that into this one).  ``want_overlay``: yields (masks, tables, stencils) with the overlay stencil
        of every mask (u8 [B,H,W], qdb:76-77).  ``tables_archive`` (from ``alloc_tables(total_frames, ...)``): the
        tables stay on the DEVICE, batch after batch in consecutive rows of the archive, and ``None`` is yielded in
        their place -- for jobs whose tables are merged elsewhere (sharded runs gather them to one rank) instead of being
        read back batch by batch; the archive's capacity applies and is not grown.

        ``csv``: every item of ``batches`` is (images, filenames), and the tables come back as a ``CsvTables`` -- the
        per-image CSV files (qdb:62-63) formatted on the device by dc_table_csv inside the batch's own stream (and CUDA
        graph), their counts and area sums, and the one size column the reports need -- in place of the column dicts;
        only those cross PCIe.

        ``png``: one more element is yielded, a ``PngFiles`` with every frame's mask PNG (the x 255 of qdb:58 and
        dc_png_encode in the batch's stream and CUDA graph), byte for byte what cv2.imwrite writes.  With ``want_overlay``
        every item also ends with the overlay bases cv2.imread returned (qdb:75) -- u8 BGR [B,H,W,3] and a per-frame
        present flag -- and the overlays are painted (0, 255, 0) and encoded on the device too (frames without a base get
        None).  The masks and stencils are still yielded."""
        dev = torch.device(device)
        if dev.index is None:
            dev = torch.device("cuda", torch.cuda.current_device())
        it = iter(batches)
        if self._streams is None or self._streams[0].device != dev:
            self._streams = tuple(torch.cuda.Stream(dev) for _ in range(4))
            self._slots = [None, None]
        # one read-back stream PER SLOT: finishing batch k-1 must not wait behind batch k's mask copy, which is
        # queued as soon as batch k is launched and cannot start before batch k has been computed
        s_in, s_run, s_out0, s_out1 = self._streams
        s_outs = (s_out0, s_out1)
        slots = self._slots              # pinned allocations cost milliseconds: made once, reused by later calls
        micron = bool(self.px_per_micron)
        if csv and tables_archive is not None:
            raise ValueError("csv=True reads the tables back as text; it cannot keep them in a tables_archive")

        def make_slot(shape, names_cap=0):
            B, H, W = shape[:3]
            d = {"dev_in": torch.empty(shape, dtype=torch.uint8, device=dev),
                 "masks": torch.empty(tuple(shape[:3]), dtype=torch.uint8, device=dev),
                 "stencil": torch.empty(tuple(shape[:3]), dtype=torch.uint8, device=dev) if want_overlay else None,
                 "h_stencil": torch.empty(tuple(shape[:3]), dtype=torch.uint8).pin_memory() if want_overlay else None,
                 "tables": alloc_tables(B, self.capacity, micron, dev),
                 "h_masks": torch.empty(tuple(shape[:3]), dtype=torch.uint8).pin_memory(),
                 "h_counts": torch.empty(B, dtype=torch.int32).pin_memory(),
                 "h_cols": torch.empty((1 if csv else 7 if micron else 5, B, self.capacity), dtype=torch.float64).pin_memory(),
                 "ev_in": torch.cuda.Event(), "ev_run": torch.cuda.Event(), "ev_counts": torch.cuda.Event(),
                 "ev_free": torch.cuda.Event(), "graph": None, "uses": 0, "names_cap": names_cap}
            if csv:
                # text buffer sized for the widest rows of names_cap bytes of filename fields: static for graph replay
                nbytes, wsb = table_csv_bounds(B, self.capacity, micron, names_cap)
                d.update({"d_names": torch.empty(names_cap, dtype=torch.uint8, device=dev),
                          "d_name_off": torch.empty(B + 1, dtype=torch.int64, device=dev),
                          "d_text": torch.empty(nbytes, dtype=torch.uint8, device=dev),
                          "d_frame_off": torch.empty(B + 1, dtype=torch.int64, device=dev),
                          "d_area_sum": torch.empty(B, dtype=torch.int64, device=dev),
                          "csv_ws": torch.empty(wsb, dtype=torch.uint8, device=dev),
                          "h_frame_off": torch.empty(B + 1, dtype=torch.int64).pin_memory(),
                          "h_area_sum": torch.empty(B, dtype=torch.int64).pin_memory()})
            if png:
                nbytes, wsb = png_bounds(B, H, W, 1)
                d.update({"m255": torch.empty((B, H, W), dtype=torch.uint8, device=dev),
                          "png_out": torch.empty(nbytes, dtype=torch.uint8, device=dev),
                          "png_ws": torch.empty(wsb, dtype=torch.uint8, device=dev),
                          "png_off": torch.empty(B + 1, dtype=torch.int64, device=dev),
                          "h_png_off": torch.empty(B + 1, dtype=torch.int64).pin_memory()})
                if want_overlay:
                    nbytes, wsb = png_bounds(B, H, W, 3)
                    d.update({"d_base": torch.empty((B, H, W, 3), dtype=torch.uint8, device=dev),
                              "painted": torch.empty((B, H, W, 3), dtype=torch.uint8, device=dev),
                              "green": torch.tensor(OVERLAY_BGR, dtype=torch.uint8, device=dev),
                              "ov_out": torch.empty(nbytes, dtype=torch.uint8, device=dev),
                              "ov_ws": torch.empty(wsb, dtype=torch.uint8, device=dev),
                              "ov_off": torch.empty(B + 1, dtype=torch.int64, device=dev),
                              "h_ov_off": torch.empty(B + 1, dtype=torch.int64).pin_memory()})
            d["ev_free"].record(s_run)
            return d

        h_text = [torch.empty(0, dtype=torch.uint8)]     # pinned text read-back buffer, grown on demand
        h_png = [torch.empty(0, dtype=torch.uint8), torch.empty(0, dtype=torch.uint8)]   # mask / overlay PNG read-back
        bases_in = png and want_overlay

        def stage(k, item):
            parts = tuple(item) if (csv or bases_in) else (item,)
            host, names = parts[0], (parts[1] if csv else None)
            if bases_in:
                bases, present = parts[-2], np.asarray(parts[-1], dtype=bool)
                bases = torch.from_numpy(np.ascontiguousarray(bases)) if isinstance(bases, np.ndarray) else bases
            host = torch.from_numpy(np.ascontiguousarray(host)) if isinstance(host, np.ndarray) else host
            if csv:
                if len(names) != host.shape[0]:
                    raise ValueError(f"{host.shape[0]} images but {len(names)} filenames")
                name_buf, name_off = pack_fields([csv_field(n) for n in names])
            sl = slots[k % 2]
            if (sl is None or sl["dev_in"].shape != host.shape or sl["tables"].capacity != self.capacity
                    or (sl["tables"].area_um2 is not None) != micron or (sl["stencil"] is not None) != want_overlay
                    or ("d_text" in sl) != csv or (csv and name_off[-1] > sl["names_cap"])
                    or ("png_out" in sl) != png or ("d_base" in sl) != bases_in):
                names_cap = 2 * int(name_off[-1]) + 256 if csv else 0
                sl = slots[k % 2] = make_slot(tuple(host.shape), names_cap)
            with torch.cuda.stream(s_in):
                s_in.wait_event(sl["ev_free"])            # the slot's previous batch has been computed and read back
                sl["dev_in"].copy_(host, non_blocking=True)
                if csv:
                    sl["d_names"][:name_buf.size].copy_(torch.from_numpy(name_buf.copy()), non_blocking=True)
                    sl["d_name_off"].copy_(torch.from_numpy(name_off), non_blocking=True)
                if bases_in:
                    if tuple(bases.shape) != tuple(host.shape[:3]) + (3,) or bases.dtype != torch.uint8:
                        raise ValueError(f"overlay bases must be uint8 {tuple(host.shape[:3]) + (3,)}")
                    sl["d_base"].copy_(bases, non_blocking=True)
                    sl["present"] = present.copy()
                sl["ev_in"].record(s_in)

        archive_pos = [0]

        def compute(k):
            sl = slots[k % 2]
            s_out = s_outs[k % 2]
            tables_out = sl["tables"]
            if tables_archive is not None:
                nb = sl["dev_in"].shape[0]
                tables_out = tables_archive.rows(archive_pos[0], archive_pos[0] + nb)
                if tables_out.counts.shape[0] != nb:
                    raise ValueError("tables_archive is too small for the frames streamed through it")
                archive_pos[0] += nb
            def work():
                self.run_device(sl["dev_in"], mask_out=sl["masks"], tables_out=tables_out, want_overlay=want_overlay,
                                stencil_out=sl["stencil"])
                if csv:
                    table_csv_device(tables_out, sl["d_names"], sl["d_name_off"], sl["names_cap"], sl["d_text"],
                                     sl["d_frame_off"], sl["d_area_sum"], sl["csv_ws"])
                if png:
                    torch.mul(sl["masks"], 255, out=sl["m255"])                                   # qdb:58
                    encode_png_device(sl["m255"], sl["png_out"], sl["png_ws"], sl["png_off"])
                    if want_overlay:                                                             # qdb:77-78
                        torch.where(sl["stencil"].bool()[..., None], sl["green"], sl["d_base"], out=sl["painted"])
                        encode_png_device(sl["painted"], sl["ov_out"], sl["ov_ws"], sl["ov_off"])
            if self.use_graphs and tables_archive is None and sl["graph"] is None and sl["uses"] >= 1:
                # second use of the slot: every buffer the batch touches exists and is static -> capture once
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    work()
                sl["graph"] = g
            with torch.cuda.stream(s_run):
                s_run.wait_event(sl["ev_in"])
                if sl["graph"] is not None:
                    sl["graph"].replay()
                else:
                    work()
                sl["uses"] += 1
                sl["ev_run"].record(s_run)
            with torch.cuda.stream(s_out):
                s_out.wait_event(sl["ev_run"])
                sl["h_counts"].copy_(sl["tables"].counts, non_blocking=True)
                if csv:
                    sl["h_frame_off"].copy_(sl["d_frame_off"], non_blocking=True)
                    sl["h_area_sum"].copy_(sl["d_area_sum"], non_blocking=True)
                if png:
                    sl["h_png_off"].copy_(sl["png_off"], non_blocking=True)
                    if want_overlay:
                        sl["h_ov_off"].copy_(sl["ov_off"], non_blocking=True)
                sl["ev_counts"].record(s_out)
                sl["h_masks"].copy_(sl["masks"], non_blocking=True)
                if want_overlay:
                    sl["h_stencil"].copy_(sl["stencil"], non_blocking=True)

        def finish(k):
            if not png:
                return finish_tables(k)
            sl = slots[k % 2]
            sl["ev_counts"].synchronize()
            offs = [sl["h_png_off"].numpy().copy()]
            bufs = [sl["png_out"]]
            if want_overlay:
                offs.append(sl["h_ov_off"].numpy().copy())
                bufs.append(sl["ov_out"])
            with torch.cuda.stream(s_outs[k % 2]):       # queued before finish_tables releases the slot
                for j, (o, buf) in enumerate(zip(offs, bufs)):
                    total = int(o[-1])
                    if h_png[j].numel() < total:
                        h_png[j] = torch.empty(total + total // 2, dtype=torch.uint8).pin_memory()
                    h_png[j][:total].copy_(buf[:total], non_blocking=True)
            present = sl.get("present")
            res = finish_tables(k)                        # synchronises the read-back stream
            files = [[h_png[j].numpy()[o[b]:o[b + 1]].tobytes() for b in range(o.size - 1)] for j, o in enumerate(offs)]
            ov = [f if p else None for f, p in zip(files[1], present)] if want_overlay else None
            return tuple(res) + (PngFiles(files[0], ov),)

        def finish_tables(k):
            sl = slots[k % 2]
            s_out = s_outs[k % 2]
            t = sl["tables"]
            if tables_archive is not None:
                with torch.cuda.stream(s_out):
                    sl["ev_free"].record(s_out)
                s_out.synchronize()
                masks = sl["h_masks"].numpy()
                if want_overlay:
                    st = sl["h_stencil"].numpy()
                    return (masks.copy() if copy else masks), None, (st.copy() if copy else st)
                return (masks.copy() if copy else masks), None
            sl["ev_counts"].synchronize()
            counts = sl["h_counts"].numpy().copy()
            nmax = int(counts.max()) if counts.size else 0
            if csv:
                text_dev, frame_off, area_sums = sl["d_text"], sl["h_frame_off"].numpy(), sl["h_area_sum"].numpy()
            if nmax > t.capacity:        # rare: rerun the table with room for everything (counts are exact)
                with torch.cuda.stream(s_run):
                    t = label_stats_device(sl["masks"], self.min_area, self.px_per_micron, nmax)
                    self.capacity = max(self.capacity, nmax)
                    if csv:              # the batch's own text left those frames out: format the complete table
                        text_dev, off_dev, asum_dev = csv_text_device(t, sl["d_names"], sl["d_name_off"], sl["names_cap"])
                s_run.synchronize()
                if csv:
                    frame_off, area_sums = off_dev.cpu().numpy(), asum_dev.cpu().numpy()
            if csv:
                return finish_csv(sl, s_out, t, counts, nmax, text_dev, frame_off.copy(), area_sums.copy())
            cols_dev = [t.area.view(torch.float64), t.eq_diam, t.centroid0, t.centroid1]
            names = ["area", "equivalent_diameter", "centroid-0", "centroid-1"]
            if micron:
                cols_dev += [t.area_um2, t.diam_um]
                names += ["area_sqmicron", "eq_diam_micron"]
            if nmax > sl["h_cols"].shape[2]:
                sl["h_cols"] = torch.empty((7 if micron else 5, counts.size, nmax), dtype=torch.float64).pin_memory()
            with torch.cuda.stream(s_out):
                for j, c in enumerate(cols_dev):
                    sl["h_cols"][j, :, :nmax].copy_(c[:, :nmax], non_blocking=True)
                sl["ev_free"].record(s_out)
            s_out.synchronize()
            masks = sl["h_masks"].numpy()
            if copy:
                masks = masks.copy()
            out = []
            for b, n in enumerate(counts):
                n = int(n)
                d = {"label": np.arange(1, n + 1, dtype=np.int64)}
                for j, name in enumerate(names):
                    col = sl["h_cols"][j, b, :n].numpy()
                    d[name] = col.view(np.int64).copy() if name == "area" else col.copy()
                out.append(d)
            if want_overlay:
                st = sl["h_stencil"].numpy()
                return masks, out, (st.copy() if copy else st)
            return masks, out

        def finish_csv(sl, s_out, t, counts, nmax, text_dev, frame_off, area_sums):
            total = int(frame_off[-1])
            if h_text[0].numel() < total:
                h_text[0] = torch.empty(total + total // 2, dtype=torch.uint8).pin_memory()
            if nmax > sl["h_cols"].shape[2]:
                sl["h_cols"] = torch.empty((1, counts.size, nmax), dtype=torch.float64).pin_memory()
            size = t.diam_um if micron else t.eq_diam
            with torch.cuda.stream(s_out):
                h_text[0][:total].copy_(text_dev[:total], non_blocking=True)
                sl["h_cols"][0, :, :nmax].copy_(size[:, :nmax], non_blocking=True)
                sl["ev_free"].record(s_out)
            s_out.synchronize()
            text = h_text[0].numpy()
            masks = sl["h_masks"].numpy()
            out = CsvTables([text[frame_off[b]:frame_off[b + 1]].tobytes() for b in range(counts.size)],
                            counts.astype(np.int64), area_sums,
                            [sl["h_cols"][0, b, :n].numpy().copy() for b, n in enumerate(counts)])
            if want_overlay:
                st = sl["h_stencil"].numpy()
                return (masks.copy() if copy else masks), out, (st.copy() if copy else st)
            return (masks.copy() if copy else masks), out

        k = 0
        pending = []                      # batch indices staged / computed but not yet yielded
        first = next(it, None)
        if first is None:
            return
        stage(0, first)
        nxt = next(it, None)
        while True:
            compute(k)
            pending.append(k)
            if nxt is not None:
                if len(pending) == 2:     # slot (k+1) % 2 still holds batch k-1: read it back first
                    yield finish(pending.pop(0))
                stage(k + 1, nxt)
                nxt = next(it, None)
                k += 1
                continue
            break
        for j in pending:
            yield finish(j)
