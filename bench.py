#!/usr/bin/env python
"""bench.py -- images/sec of the droplet-quantification hot path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--batch 32] [--size 1024]

One "step" = one batch of synthetic grayscale frames through the whole path of reference
quantify_droplets_batch.py: rolling-ball correction -> UNetDC forward -> `> prob_thresh` -> 4-connected
labelling -> per-droplet table.  Workload at N = 1: BASELINE.json configs[1] (UNetDC 1024x1024, batch 32,
bf16, threshold + CCL + stats).  N > 1 (torchrun, one rank per GPU): every rank runs its own shard of
independent batches -- no data-path collective (SURVEY.md 8e), NCCL only for the barrier / max-over-ranks.

`value`  : frames already resident in HBM when the timed region starts (device-timed, CUDA events).
`e2e`    : the same metric through DropletPipeline.run_host with pinned HOST buffers -- the H2D copy of the
           frames and the D2H copy of masks + table rows are inside the timed region.
`--impl reference` : the reference's OWN modules (oracle/_ref: quantify_droplets_batch.py, models/model_2.py,
           utils/data_loader.py byte-compiled where they lie; rolling_ball_correction_rgb, UNetDC fp32, `> thresh`,
           quantify with its O(labels x pixels) filter loop) on this box's host cores; rank 0 only.  Falls back to the
           oracle port (kind "port") when oracle/_ref is absent.
`parity`  : GPU outputs against the reference's on the cpu_baseline frames: |dp|, mask pixels / droplets differing.
`config4` : BASELINE configs[3] -- `--frames 4096` frames sharded round-robin over the ranks (strong scaling), tables
           gathered to rank 0 in frame order inside the timed region, merged-table checksum (equal for every N).
`--dump-outputs DIR` : after the timed steps, rank 0 writes what the device-resident arm returned in its last step as
           DIR/<name>.npy (float32 / float64, under 64 MB; see last_step_outputs).  The inputs depend only on the
           arguments, so two builds run with the same arguments can be compared output for output.  With N > 1 the
           files hold rank 0's frames only, and each rank's frames depend on its rank: compare dumps taken with the
           same --gpus.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

REPO = Path(__file__).resolve().parent
sys.path.insert(0, str(REPO))

_OUT = sys.stdout
METRIC = "images/sec end-to-end (mask + droplet table)"
UNIT = "images/s"
PROB_THRESH = 0.3
MIN_AREA = 1
RADIUS = 50
PX_PER_UM = 3.45


def workload_name(batch, size):
    return (f"configs[1]: UNetDC inference {size}x{size} batch {batch} bf16 on B200, rolling_ball radius {RADIUS} + "
            f"threshold {PROB_THRESH} + CCL + per-droplet stats")


def peaks():
    p = REPO / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return d, "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


# ------------------------------------------------------------------------------------ clocks
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int, period_ms: int = 100):
        self.index = index
        self.period_ms = period_ms
        self.proc = None
        self.lines = []
        self.thread = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                 "-lms", str(self.period_ms)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None
            return
        self.thread = threading.Thread(target=self._pump, daemon=True)
        self.thread.start()

    def wait_ready(self, timeout: float = 15.0):
        """Block until nvidia-smi has initialised (NVML start-up takes 0.2-2 s on a fresh box and, overlapping the
        timed region, was measured to stretch it by 10-30 %) and is delivering samples."""
        if self.proc is None:
            return
        t0 = time.time()
        while len(self.lines) < 2 and time.time() - t0 < timeout and self.proc.poll() is None:
            time.sleep(0.05)

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self, t0: float, t1: float):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, line in self.lines:
            if ts < t0 or ts > t1 + 0.15:
                continue
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0])); mx.append(float(parts[1])); pw.append(float(parts[2]))
            except ValueError:
                continue
            for n, v in zip(names, parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples in the timed region"]}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "power_w_max": max(pw), "samples": len(sm),
                "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------ inputs
def make_frames(n: int, size: int) -> np.ndarray:
    from unet_dc_segmentation_b200.synth import synthetic_image
    return np.stack([synthetic_image(size, i) for i in range(n)])


# ------------------------------------------------------------------------------------ CPU arm
def cpu_reference_step(sd, frames_u8, use_threads, want_outputs=False):
    """The reference's CPU path on `frames_u8` (u8 [n,H,W]).  Returns (seconds, droplets, kind[, probs, masks, tables]).
    kind "reference": the reference's own modules from oracle/_ref; "port": the oracle restatement."""
    import oracle
    import torch
    from oracle import ref
    torch.set_num_threads(use_threads)
    rgb = [np.repeat(f[:, :, None], 3, 2) for f in frames_u8]          # Image.convert("RGB"), qdb:41
    kind = "reference" if ref.available() else "port"
    if kind == "reference":
        try:
            ref.load()
        except Exception as exc:  # noqa: BLE001  (compiled by another Python, a clashing `utils` package, ...)
            print(f"bench.py: oracle/_ref cannot be loaded ({exc}); timing the port instead", file=sys.stderr)
            kind = "port"
    t0 = time.perf_counter()
    if kind == "reference":
        probs, masks, tables = ref.run_path(sd, rgb, radius=RADIUS, prob_thresh=PROB_THRESH, min_area=MIN_AREA,
                                            px_per_um=PX_PER_UM)
    else:
        probs, masks, tables = oracle.run_path(sd, rgb, radius=RADIUS, prob_thresh=PROB_THRESH, min_area=MIN_AREA,
                                               px_per_um=PX_PER_UM, use_cv2=True)
    dt = time.perf_counter() - t0
    n = sum(len(t) for t in tables)
    return (dt, n, kind, probs, masks, tables) if want_outputs else (dt, n, kind)


CPU_SAMPLE = {"reference": "the reference's own rolling_ball_correction_rgb + UNetDC fp32 + `> thresh` + quantify (oracle/_ref)",
              "port": "cv2 rolling ball + torch fp32 UNetDC + threshold + oracle quantify (oracle/_ref absent)"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    import torch
    from unet_dc_segmentation_b200.synth import calibrated_state_dict
    cores = os.cpu_count() or 1
    sd = calibrated_state_dict(seed=0)
    frames = make_frames(2, args.size)
    per_step = 1
    kind = "port"
    for w in range(args.warmup):
        cpu_reference_step(sd, frames[:per_step], cores)
    times = []
    for k in range(args.steps):
        dt, _, kind = cpu_reference_step(sd, frames[k % 2:k % 2 + per_step], cores)
        times.append(dt)
    total = sum(times)
    value = per_step * args.steps / total
    sample = (f"{per_step} frame of {args.size}x{args.size} per step (of the batch-{args.batch} workload): {CPU_SAMPLE[kind]}")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(args.batch, args.size), "batch": args.batch, "size": args.size,
                   "sample_frames_per_step": per_step},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample,
                         "torch_threads": torch.get_num_threads()},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    _OUT.write(json.dumps(line) + "\n")
    _OUT.flush()
    return 0


# ------------------------------------------------------------------------------------ parity (GPU vs the reference)
def parity_report(probs, masks, tables, probs_ref, masks_ref, tables_ref, kind):
    """How far the GPU path is from the reference on the same frames (north_star: probabilities within a stated bf16
    tolerance, mask disagreements only near prob_thresh, tables bit-exact given the same mask)."""
    import oracle
    err = np.abs(probs - probs_ref)
    diff = masks != masks_ref
    dist = np.abs(probs_ref - PROB_THRESH)
    exact = True
    for i in range(len(masks)):
        _, cols = oracle.quantify_arrays(masks[i], MIN_AREA, PX_PER_UM)
        exact = exact and all(np.array_equal(np.asarray(tables[i][c]), v) for c, v in cols.items())
    n_gpu = [int(len(t["label"])) for t in tables]
    n_ref = [int(len(t)) for t in tables_ref]
    a_gpu = [int(np.asarray(t["area"]).sum()) for t in tables]
    a_ref = [int(t["area"].sum()) if len(t) else 0 for t in tables_ref]
    return {
        "against": f"{kind} ({CPU_SAMPLE[kind]})", "frames": int(len(masks)), "pixels": int(masks.size),
        "prob_max_abs_diff": float(err.max()), "prob_mean_abs_diff": float(err.mean()),
        "prob_tolerance": {"this_checkpoint": 0.08, "survey_checkpoint": 0.03,
                           "note": "bench weights have a least-squares out_conv (logits -6..+4); tests/test_gpu_forward.py"},
        "mask_pixels_differing": int(diff.sum()), "mask_pixels_differing_frac": float(diff.mean()),
        "of_which_within_0.03_of_thresh": int((diff & (dist <= 0.03)).sum()),
        "of_which_within_0.08_of_thresh": int((diff & (dist <= 0.08)).sum()),
        "outside_0.08_band": int((diff & (dist > 0.08)).sum()),
        "droplets_per_frame_gpu": n_gpu, "droplets_per_frame_reference": n_ref,
        "droplet_count_delta": [g - r for g, r in zip(n_gpu, n_ref)],
        "total_area_px_gpu": a_gpu, "total_area_px_reference": a_ref,
        "total_area_delta_frac": [float((g - r) / max(1, r)) for g, r in zip(a_gpu, a_ref)],
        "tables_bit_exact_given_gpu_mask": bool(exact),
    }


# ------------------------------------------------------------------------------------ config 4 (strong scaling)
def frame_content(base, i):
    """Frame i of the config-4 job: a function of the GLOBAL frame index only, so every sharding sees the same job."""
    n = len(base)
    return np.roll(base[i % n], 37 * ((i // n) % 16), axis=1)


def run_config4(pipe, dev, rank, world, frames_total, batch, size, barrier, dist, expect_per_frame=2):
    """BASELINE configs[3]: frames_total frames, frame i -> rank i mod world (shard.py).  Each rank streams its batches
    through DropletPipeline.run_host_pipelined (pinned host frames up, host masks down; the masks stay with the rank that
    computed them, as qdb:58 writes them there) with the tables archived on the device; at the end the per-droplet
    tables are compacted, gathered on rank 0 over NCCL, put into frame order and read back to the host once -- all
    inside the timed region."""
    import torch
    from unet_dc_segmentation_b200 import shard
    from unet_dc_segmentation_b200.quantify import alloc_tables
    base = make_frames(8, size)
    mine = shard.shard_indices(frames_total, rank, world)
    groups = shard.batches(mine, batch)
    uniq = {}
    def content(i):
        key = (i % 8, (i // 8) % 16)
        if key not in uniq:
            uniq[key] = frame_content(base, i)
        return uniq[key]
    staged = [torch.from_numpy(np.stack([content(i) for i in g])).pin_memory() for g in groups]
    ncol = 6
    archive = alloc_tables(len(mine), pipe.capacity, True, dev)
    host_rows = torch.empty((frames_total * 4096, ncol), dtype=torch.float64).pin_memory() if rank == 0 else None
    # first use of a collective sets up its connections, first use of a torch op loads its kernels and the first
    # allocation of a size goes to cudaMalloc: run the tail once before the clock starts, on a dummy archive of the
    # job's own shape (as many rows per frame as the bench step found), so that the timed tail reuses cached blocks
    per = int(min(max(expect_per_frame, 2), pipe.capacity))
    dummy = alloc_tables(len(mine), pipe.capacity, True, dev)
    dummy.counts.fill_(per)
    for t in (dummy.area, dummy.centroid0, dummy.centroid1, dummy.eq_diam, dummy.area_um2, dummy.diam_um):
        t.zero_()
    shard.gather_tables_in_frame_order(dummy, frames_total, host_rows)
    del dummy
    barrier(); torch.cuda.synchronize()
    t0 = time.perf_counter()
    mask_px = 0
    for (m_h, _) in pipe.run_host_pipelined(iter(staged), dev, copy=False, tables_archive=archive):
        mask_px += int(m_h.size)
    torch.cuda.synchronize()
    t_stream_own = time.perf_counter() - t0
    barrier()                                                  # (the gather below would wait for the slowest rank anyway)
    t_stream = time.perf_counter() - t0
    timing = {}
    merged, merged_counts = shard.gather_tables_in_frame_order(archive, frames_total, host_rows, timing)
    timing = {k: v + t_stream for k, v in timing.items()}      # (relative to the start of the job)
    torch.cuda.synchronize(); barrier()
    dt = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([dt], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dt = float(t.item())
    out = {"frames_total": frames_total, "seconds": dt, "value": frames_total / dt, "unit": UNIT, "scaling": "strong",
           "seconds_streaming_rank0": t_stream_own, "seconds_streaming_slowest_rank": t_stream,
           "seconds_gather_merge_readback": dt - t_stream,
           "seconds_tail_rank0": {"compact": timing["compact"] - t_stream, "nccl_gather": timing["gather"] - timing["compact"],
                                  "order_and_readback": dt - timing["gather"]},
           "batches_per_rank": len(groups), "tail_batch": len(groups[-1]) if groups else 0,
           "sharding": f"frame i -> rank i mod {world}; tables gathered to rank 0 and merged in frame order inside the timed region"}
    if rank == 0:
        import hashlib
        # frames repeat with period 128 (frame_content): every repeat must give the same table rows
        offs = np.concatenate([[0], np.cumsum(merged_counts)])
        mism = 0
        for i in range(128, frames_total):
            a, b = merged[offs[i - 128]:offs[i - 128 + 1]], merged[offs[i]:offs[i + 1]]
            mism += int(a.shape != b.shape or not np.array_equal(a.view(np.int64), b.view(np.int64)))
        out["repeat_mismatches"] = mism
        h = hashlib.sha256()
        h.update(merged_counts.tobytes())
        h.update(np.ascontiguousarray(merged).tobytes())
        out.update({"droplets_total": int(merged_counts.sum()), "table_bytes": int(merged.nbytes),
                    "merged_table_sha256": h.hexdigest()[:16]})
    return out


# ------------------------------------------------------------------------------------ --dump-outputs
DUMP_BYTES = 60 << 20           # all arrays together: with the .npy headers, under 64 MB
DUMP_MASK_BYTES = 16 << 20      # of which the mask rows


def last_step_outputs(masks, tables):
    """The timed path's results (masks u8 [B,H,W] and the droplet tables) as host float32 / float64 arrays.

    mask_rows [n, W] holds whole mask rows, mask_row_index [n, 2] their (image, row): every row while the batch fits in
    DUMP_MASK_BYTES as float32, otherwise a sample of rows drawn with seed 0.  droplet_counts [B] is the number of
    droplets per image; droplets_<column> holds one entry per droplet, image by image, for the columns of
    DropletTables.to_host() plus `image`; past the remaining budget a seed-0 sample of droplets is kept (their
    `image` and `label` say which)."""
    import torch
    rng = np.random.default_rng(0)
    B, H, W = masks.shape
    n_rows = min(B * H, max(1, DUMP_MASK_BYTES // (4 * W)))
    rows = np.sort(rng.choice(B * H, n_rows, replace=False))
    picked = masks.reshape(B * H, W).index_select(0, torch.from_numpy(rows).to(masks.device))
    out = {"mask_rows": picked.cpu().numpy().astype(np.float32),
           "mask_row_index": np.stack([rows // H, rows % H], 1).astype(np.float64)}
    per_image = tables.to_host()
    out["droplet_counts"] = np.array([len(t["label"]) for t in per_image], np.float64)
    cols = {"image": np.concatenate([np.full(len(t["label"]), b, np.float64) for b, t in enumerate(per_image)])}
    for c in per_image[0]:
        cols[c] = np.concatenate([np.asarray(t[c], np.float64) for t in per_image])
    n = len(cols["image"])
    room = (DUMP_BYTES - sum(a.nbytes for a in out.values())) // (8 * len(cols))
    if n > room:
        keep = np.sort(rng.choice(n, room, replace=False))
        cols = {c: v[keep] for c, v in cols.items()}
    out.update({f"droplets_{c}": v for c, v in cols.items()})
    return out


def write_outputs(directory, arrays):
    d = Path(directory)
    d.mkdir(parents=True, exist_ok=True)
    for name, a in arrays.items():
        np.save(d / f"{name}.npy", a)
    total = sum(a.nbytes for a in arrays.values())
    print(f"bench.py: wrote {len(arrays)} arrays ({total / 2**20:.1f} MiB) to {d}", file=sys.stderr)


# ------------------------------------------------------------------------------------ B200 arm
def run_b200(args):
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the B200 arm has no CPU fallback (use --impl reference for the CPU path)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    from unet_dc_segmentation_b200 import DropletPipeline, UNetDC, _lib
    from unet_dc_segmentation_b200.morphology import rolling_ball_device
    from unet_dc_segmentation_b200.quantify import alloc_tables, label_stats_device
    from unet_dc_segmentation_b200.synth import calibrated_state_dict
    from unet_dc_segmentation_b200 import workload as wl

    B, S, K, Wm = args.batch, args.size, args.steps, args.warmup
    # torchrun pins OMP_NUM_THREADS=1; the one-off CPU calibration of the synthetic checkpoint can use this rank's share
    torch.set_num_threads(max(1, (os.cpu_count() or 1) // max(1, world)))
    sd = calibrated_state_dict(seed=0)
    model = UNetDC(3, 1)
    model.load_state_dict(sd)
    model = model.to(dev).eval()
    pipe = DropletPipeline(model, RADIUS, PROB_THRESH, MIN_AREA, PX_PER_UM, capacity=args.capacity,
                           use_graphs=args.graphs)

    # distinct frames per rank; NVAR variants of the batch so consecutive steps never see the same input
    base = make_frames(min(B, args.unique_frames), S)
    reps = (B + len(base) - 1) // len(base)
    batch0 = np.concatenate([np.roll(base, 17 * r + 5 * rank, axis=2) for r in range(reps)])[:B]
    NVAR = 4
    host_batches = [torch.from_numpy(np.ascontiguousarray(np.roll(batch0, 61 * v, axis=1))).pin_memory() for v in range(NVAR)]
    dev_batches = [h.to(dev) for h in host_batches]
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- device-resident arm
    for w in range(Wm):
        pipe.run_device(dev_batches[w % NVAR])
    torch.cuda.synchronize()
    sampler = ClockSampler(local, int(os.environ.get("DC_BENCH_SMI_MS", "100")))
    sampler.start()
    sampler.wait_ready()
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(4)] for _ in range(K)]
    # steady-state serving loop: outputs are preallocated (a fresh 60 MB of masks + tables per step sends the second
    # step into cudaMalloc, a 30-60 ms stall with the first step's results still referenced)
    mask_buf = torch.empty((B, S, S), dtype=torch.uint8, device=dev)
    tables_buf = alloc_tables(B, pipe.capacity, PX_PER_UM is not None, dev)
    barrier(); torch.cuda.synchronize()
    t_wall0 = time.time()
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    last = None
    for k in range(K):
        x = dev_batches[k % NVAR]
        ev[k][0].record()
        xc = rolling_ball_device(x, RADIUS, out=pipe._rb_out, workspace=pipe._rb_ws)
        ev[k][1].record()
        masks, _ = model.predict_u8(xc, PROB_THRESH, mask_out=mask_buf)
        ev[k][2].record()
        last = label_stats_device(masks, MIN_AREA, PX_PER_UM, pipe.capacity, workspace=pipe._ccl_ws, out=tables_buf)
        ev[k][3].record()
    end.record()
    torch.cuda.synchronize(); barrier()
    t_wall1 = time.time()
    ms_total = max_over_ranks(start.elapsed_time(end))
    clocks = sampler.stop(t_wall0, t_wall1)
    stage_ms = [sum(ev[k][i].elapsed_time(ev[k][i + 1]) for k in range(K)) / K for i in range(3)]
    step_ms = [ev[k][0].elapsed_time(ev[k + 1][0]) if k + 1 < K else ev[k][0].elapsed_time(end) for k in range(K)]
    counts = last.counts.cpu().numpy()
    dumped = last_step_outputs(masks, last) if args.dump_outputs and rank == 0 else None
    value = world * B * K / (ms_total / 1e3)

    # ---- end-to-end arm: pinned host frames in, host masks + table rows out, every copy inside the timed region.
    # DropletPipeline.run_host_pipelined is the public streaming entry: H2D of batch k+1 and D2H of batch k-1
    # overlap the compute of batch k (three streams, pinned buffers).
    def host_batches_iter(n):
        for k in range(n):
            yield host_batches[k % NVAR]

    for _ in pipe.run_host_pipelined(host_batches_iter(max(2, Wm)), dev):
        pass
    barrier(); torch.cuda.synchronize()
    s2, e2 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s2.record()
    t_e2e0 = time.perf_counter()
    d2h = 0
    n_out = 0
    for m_h, tabs in pipe.run_host_pipelined(host_batches_iter(K), dev, copy=False):      # consumed before advancing
        d2h = m_h.nbytes + sum(sum(v.nbytes for c, v in t.items() if c != "label") for t in tabs) + 4 * B
        n_out += len(tabs)
    torch.cuda.synchronize()
    e2.record()
    torch.cuda.synchronize(); barrier()
    assert n_out == B * K
    ms_e2e = max_over_ranks(max(s2.elapsed_time(e2), 1e3 * (time.perf_counter() - t_e2e0)))
    e2e_value = world * B * K / (ms_e2e / 1e3)

    # ---- per-launch profile of the forward (one extra, untimed pass) for the roofline table
    pk, ptype = peaks()
    names, fl = wl.launch_flops(S, S, model.dilations, in_bounds=True, fused_level1=model.fuse_level1,
                                fused_levels=model.fuse_levels)
    import ctypes as C
    n_launch = model.num_launches()
    ms_arr = (C.c_float * n_launch)()
    mk = torch.empty((B, S, S), dtype=torch.uint8, device=dev)
    ws = model.packed().workspace_for(B, S, S)
    passes = []
    for _ in range(5):
        _lib.check(_lib.load().dc_forward_profile(model.packed().handle, 1, pipe._rb_out.data_ptr(), B, S, S, PROB_THRESH,
                                                  None, mk.data_ptr(), ws.data_ptr(), ws.numel(), _lib.stream_ptr(dev), ms_arr))
        passes.append([float(v) for v in ms_arr])
    med = [statistics.median(p[i] for p in passes) for i in range(n_launch)]
    layers = [{"launch": n, "ms": round(med[i], 4), "tflops": round(B * fl[i] / (med[i] * 1e9), 1)}
              for i, n in enumerate(names)]

    fwd_flops = B * wl.forward_flops(S, S, model.dilations, in_bounds=True)
    issued_flops = B * wl.forward_flops_issued(S, S, model.dilations, in_bounds=True,
                                               fused_levels=tuple(model.fuse_levels) + ((1,) if model.fuse_level1 else ()))
    fwd_ms = stage_ms[1]
    achieved = fwd_flops / (fwd_ms * 1e-3) / 1e12
    peak = pk.get("bf16_tflops_sustained", pk["bf16_tflops"])
    px = B * S * S
    rb_gbs = px * wl.ROLLING_BALL_BYTES_PER_PX / (stage_ms[0] * 1e-3) / 1e9
    ccl_bytes = px * (wl.LABEL_BYTES_PER_PX + wl.STATS_BYTES_PER_PX) + int(counts.sum()) * wl.STATS_BYTES_PER_DROPLET
    ccl_gbs = ccl_bytes / (stage_ms[2] * 1e-3) / 1e9
    launches_per_step = 3 + n_launch + 7          # rolling ball (erode, dilate, stretch) + dc_forward + dc_label_stats
    # DRAM bytes of the forward launches of THIS configuration, from the newest committed ncu capture
    # (profiles/forward_traffic.json, written by tools/summarize_profiles.py from the per-launch
    # dram__bytes_read.sum + dram__bytes_write.sum); null when no capture of this configuration is committed
    traffic, traffic_src = None, None
    tj = REPO / "profiles" / "forward_traffic.json"
    if tj.exists():
        for rec in json.loads(tj.read_text()):
            if (rec["batch"], rec["size"]) == (B, S) and tuple(rec["dilations"]) == tuple(model.dilations):
                traffic, traffic_src = rec["dram_bytes"], rec["source"]
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": Wm,
        "ms_per_step": ms_total / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16", "data": "synthetic",
        "config": {"workload": workload_name(B, S), "batch_per_gpu": B, "size": S, "sharding": f"{world} independent per-GPU streams, no collective",
                   "weights": "random-init UNetDC + BN calibration (seed 0)",
                   "l2": f"{NVAR} distinct input batches rotated; per-step activation traffic (tens of GB) >> 126 MB L2",
                   "droplets_per_image": float(counts.mean())},
        "roofline": {"kernel": f"dc_forward = {n_launch} tcgen05 launches (stem, conv, fused upconv+conv kernels)", "bound": "tensor",
                     "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                     "frac_note": "algorithmic FLOPs of the reference network / time / peak; the kernels issue fewer FLOPs "
                                  "than that (see `issued`), so this can exceed 1",
                     "traffic": traffic,
                     "traffic_note": f"DRAM bytes per dc_forward ({n_launch} launches) from the ncu capture {traffic_src}; "
                                     "activations written once + read once would be ~84 GB unfused (SURVEY 8d)",
                     "peak_source": f"{ptype} MEASURED_PEAKS.json bf16_tflops_sustained (kernel timed inside a long step)",
                     "flops_per_launch_group": fwd_flops,
                     "flops_model": "ALGORITHMIC = the reference network's layers, in-bounds taps (conservative), SURVEY.md 8d",
                     "issued": {"flops_per_launch_group": issued_flops, "TFLOPs": issued_flops / (fwd_ms * 1e-3) / 1e12,
                                "frac": issued_flops / (fwd_ms * 1e-3) / 1e12 / peak,
                                "note": "what the kernels execute: each decoder level runs upconv + conv composed into one "
                                        "layer with K = 17 C instead of 20 C per output pixel and channel (DESIGN.md 3.1), "
                                        "so `achieved` (reference FLOPs / time) can exceed the cuBLAS-measured peak"},
                     "ms": fwd_ms},
        "stages": {"rolling_ball": {"ms": stage_ms[0], "GBps_algorithmic": rb_gbs, "frac_hbm": rb_gbs / pk["hbm_gbs"]},
                   "forward": {"ms": stage_ms[1], "TFLOPs": achieved},
                   "label_stats": {"ms": stage_ms[2], "GBps_algorithmic": ccl_gbs, "frac_hbm": ccl_gbs / pk["hbm_gbs"]}},
        "layers": layers,
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": B * S * S, "d2h_bytes_per_step": int(d2h),
                "ms_per_step": ms_e2e / K, "api": "DropletPipeline.run_host_pipelined(copy=False) (pinned host frames -> host masks + tables, each batch "
                              "consumed before the generator is advanced)"
                       + (", CUDA-graph replay per batch" if args.graphs else "")},
        "gpu_launches": launches_per_step * K,
        "clocks": clocks,
        "step_ms": [round(x, 2) for x in step_ms],
    }

    if args.frames > 0:
        # (a failure of this extra job must not cost the headline line; every rank takes the same branch because
        #  the job fails or succeeds collectively only on deterministic conditions such as memory)
        try:
            line["config4"] = run_config4(pipe, dev, rank, world, args.frames, B, S, barrier, dist,
                                          expect_per_frame=int(1.1 * float(counts.max())) + 1)
        except Exception as exc:  # noqa: BLE001
            if world > 1:
                raise
            line["config4"] = {"error": f"{type(exc).__name__}: {exc}"}

    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cores = os.cpu_count() or 1
        nfr = args.cpu_frames
        frames = batch0[:nfr]
        try:
            cpu_reference_step(sd, frames[:1], cores)                       # warm the conv primitives
            dt, _, kind, probs_ref, masks_ref, tables_ref = cpu_reference_step(sd, frames, cores, want_outputs=True)
            line["cpu_baseline"] = {"value": nfr / dt, "unit": UNIT, "cores": cores, "kind": kind,
                                    "sample": f"{nfr} of the batch's {S}x{S} frames, once ({torch.get_num_threads()} torch "
                                              f"threads): {CPU_SAMPLE[kind]}; {dt:.1f} s"}
            # the same frames through the GPU path: how far is it from the reference?
            res = pipe.run_device(torch.from_numpy(np.ascontiguousarray(frames)).to(dev), return_prob=True)
            torch.cuda.synchronize()
            line["parity"] = parity_report(res.probs[:, 0].cpu().numpy(), res.masks.cpu().numpy(), res.tables.to_host(),
                                           probs_ref, masks_ref, tables_ref, kind)
        except Exception as exc:  # noqa: BLE001  (the CPU leg must not cost the GPU line)
            line.setdefault("cpu_baseline", {"error": f"{type(exc).__name__}: {exc}"})
            line.setdefault("parity", {"error": f"{type(exc).__name__}: {exc}"})
    if dumped is not None:
        write_outputs(args.dump_outputs, dumped)
    if rank == 0:
        _OUT.write(json.dumps(line) + "\n")
        _OUT.flush()
    if world > 1:
        dist.destroy_process_group()
    return 0


def _claim_stdout():
    """Libraries (NCCL's version banner, for one) write to fd 1; the driver wants exactly ONE JSON line there.
    Point fd 1 at stderr for the duration of the run and return a writer for the real stdout."""
    sys.stdout.flush()
    real = os.dup(1)
    os.dup2(2, 1)
    return os.fdopen(real, "w")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--size", type=int, default=1024)
    ap.add_argument("--capacity", type=int, default=16384)
    ap.add_argument("--unique-frames", type=int, default=8)
    ap.add_argument("--cpu-frames", type=int, default=3)
    ap.add_argument("--frames", type=int, default=4096,
                    help="BASELINE configs[3]: total frames of the strong-scaling job reported under `config4` (0 = skip)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--graphs", action="store_true",
                    help="e2e arm: replay each batch's launches as one CUDA graph (DropletPipeline(use_graphs=True))")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the last timed step's masks and droplet tables to DIR/<name>.npy (rank 0, --impl b200)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the B200 path (--impl b200)")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    global _OUT
    _OUT = _claim_stdout()
    if args.impl == "reference":
        return run_reference(args)
    return run_b200(args)


if __name__ == "__main__":
    sys.exit(main())
