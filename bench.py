#!/usr/bin/env python
"""Benchmark of the AprilGroup tracking hot path (BASELINE.json metric: refined poses/sec).

  python bench.py --gpus N --steps K --warmup W            # this repo (CUDA, sm_100a)
  python bench.py --impl reference --gpus N --steps K ...    # CPU arm: the oracle on the host cores

Workload (BASELINE.json configs[1]): batched dense pose refinement of 4096 independent
synthetic 1080p frames per GPU (12-tag dodecahedron, 20 172 surface samples), one
hypothesis per frame, initial pose = truth + N(0, 0.01 rad) + N(0, 0.5 mm).  One step =
build the Gaussian pyramid of every frame (K1) + refine every frame (K4); frames are
resident in HBM for ``value`` and in pinned host memory for ``e2e`` (which goes through
the host-buffer C-ABI entry point agt_refine_host: H2D of every frame, D2H of every pose).
Other workloads of BASELINE.json (--workload lk / multihyp) are secondary lines.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

from accurate_aprilgroup_tracking_b200 import synth  # noqa: E402

CAM = synth.CAMERA_1080P
BYTES_PER_SAMPLE_EVAL = 36          # SURVEY.md 8d: 16 B model record + 4 B intensity taps + 16 B gradient taps
BYTES_PER_POSE_FIXED = 156
LK_BYTES_PER_CORNER = 5008          # SURVEY.md 8d
PYR_BYTES_PER_1080P = 2754000       # SURVEY.md 8d
# Per-pose figures of one dpr_kernel launch that only a profiler can give (DRAM bytes, warp instructions issued) are NOT
# constants of this file: they are read from the summary of the latest `ncu --set full` capture of this very command,
# profiles/ncu_dpr_kernel.json (written by scripts/ncu_summary.py from the .ncu-rep; it records the git revision of
# csrc/agt_dpr.cu it was taken from).  Without that file `roofline.traffic` and `roofline.issue_frac` are null.
NCU_DPR_SUMMARY = ROOT / "profiles" / "ncu_dpr_kernel.json"
SM_COUNT, SCHEDULERS_PER_SM = 148, 4


def ncu_dpr_summary():
    try:
        return json.loads(NCU_DPR_SUMMARY.read_text())
    except (OSError, ValueError):
        return None


def dpr_config(world: int, frames_per_gpu: int) -> dict:
    """The `config` object of the headline workload - the same for the CUDA arm and the CPU (--impl reference) arm."""
    return {"workload": "batched dense pose refinement: 1080p frames, 12-tag dodecahedron, 20172 surface samples, 1 hypothesis",
            "frames_per_gpu": frames_per_gpu,
            "step": "K4 LM refinement to convergence with K1 fused into it (each refinement builds the region of interest of its own pyramid level from the frame, cv2.pyrDown arithmetic) + exact redo on a full pyramid of frames that left their ROI",
            "l2": "inputs (%.1f GB of frames per GPU) are larger than L2; no flush needed" % (frames_per_gpu * CAM.width * CAM.height / 1e9),
            "parallelism": f"frames sharded over {world} GPU(s), no collective on the path; one NCCL all-gather of the final poses of all steps"}


def measured_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return float(d["hbm_gbs"]), "measured"
    return 6650.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.FIELDS}",
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1])); smax.append(float(parts[2]))
            except ValueError:
                continue
            for nm, val in zip(names, parts[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm)}


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir: str, arrays: dict, rank: int, world: int) -> None:
    """Write each array as <out_dir>/<name>.npy (<out_dir>/rank<r>/ when several ranks run): float64 stays float64, every
    other dtype becomes float32 (the integer outputs are far below 2^24, so exactly).  When the whole set exceeds 64 MB, every
    array keeps the same fixed, seeded sample of frames (first axis), and sample_index.npy holds their indices."""
    host = {k: v.cpu().numpy() for k, v in arrays.items()}
    host = {k: v if v.dtype == np.float64 else v.astype(np.float32) for k, v in host.items()}
    n = len(next(iter(host.values())))
    per_frame = sum(v.nbytes for v in host.values()) / max(n, 1)
    budget = DUMP_LIMIT_BYTES - (64 << 10)                        # room for the .npy headers
    if n * per_frame > budget:
        keep = int(budget // (per_frame + 8))
        idx = np.sort(np.random.default_rng(0).choice(n, keep, replace=False))
        host = {k: v[idx] for k, v in host.items()}
        host["sample_index"] = idx.astype(np.float64)
    d = Path(out_dir) / (f"rank{rank}" if world > 1 else "")
    d.mkdir(parents=True, exist_ok=True)
    for k, v in host.items():
        np.save(d / f"{k}.npy", v)


def make_poses(n: int, seed: int):
    rng = np.random.default_rng(seed)
    truth = np.array([synth.random_pose(rng) for _ in range(n)])
    init = truth + np.concatenate([rng.normal(0, 0.01, (n, 3)), rng.normal(0, 0.0005, (n, 3))], axis=1)
    return truth, init


# ------------------------------------------------------------------------------------------
# CPU arm: the oracle (there is no reference implementation of dense refinement, see oracle/)
# ------------------------------------------------------------------------------------------
_CPU = {}


def _cpu_refine_one(i):
    import cv2
    from oracle import dpr_oracle, lk_oracle
    cv2.setNumThreads(1)
    t0 = time.perf_counter()
    pyr = lk_oracle.pyramid_cv(_CPU["frames"][i])
    out = dpr_oracle.refine(pyr, _CPU["model"], CAM.mtx, _CPU["init"][i])
    return time.perf_counter() - t0, out["pose"], out["evals"]


def cpu_refine(frames: np.ndarray, init: np.ndarray, workers: int, repeats: int = 1):
    """Refine frames with the oracle on `workers` processes (forked: frames and model are inherited, not pickled).
    Returns (list of wall seconds per repeat, poses)."""
    from oracle import dpr_oracle
    s, tg, n, c = synth.surface_model()
    _CPU.update(frames=frames, init=init, model=dpr_oracle.Model(s, tg, n, c, synth.model_pitch()))
    idx = list(range(len(frames)))
    walls = []
    # one BLAS thread per process: `cores` then means what it says, and 16 processes do not fight over 16 x 16 threads
    # (measured on the GPU box: 265 poses/s with the default pool, 688 with one thread each; scripts/cpu_probe.py)
    try:
        from threadpoolctl import threadpool_limits
        _CPU["blas_limit"] = threadpool_limits(1)
    except Exception:
        pass
    if workers <= 1:
        for _ in range(repeats):
            t0 = time.perf_counter()
            res = [_cpu_refine_one(i) for i in idx]
            walls.append(time.perf_counter() - t0)
        return walls, np.array([r[1] for r in res])
    import multiprocessing as mp
    with mp.get_context("fork").Pool(workers) as pool:
        pool.map(_cpu_refine_one, idx[:workers])                   # warm the workers (imports)
        for _ in range(repeats):
            t0 = time.perf_counter()
            res = pool.map(_cpu_refine_one, idx, chunksize=1)
            walls.append(time.perf_counter() - t0)
    return walls, np.array([r[1] for r in res])


def _render_one(args):
    pose, seed = args
    return synth.render(pose, CAM, seed)


def sample_frames_for_cpu(n: int, seed: int, workers: int):
    """Frames for the CPU arm: the numpy specification of the renderer (synth.render), in this process tree only - the CPU arm
    must not touch the CUDA library (its record lists the native libraries the process mapped)."""
    truth, init = make_poses(n, seed)
    jobs = [(truth[i], seed + i) for i in range(n)]
    if workers > 1:
        import multiprocessing as mp
        with mp.get_context("fork").Pool(workers) as pool:
            frames = np.stack(pool.map(_render_one, jobs, chunksize=1))
    else:
        frames = np.stack([_render_one(j) for j in jobs])
    return frames, truth, init


def native_library_mapped() -> bool:
    try:
        return "libagt" in Path("/proc/self/maps").read_text()
    except OSError:
        return False


def run_reference(args):
    """CPU arm: oracle/dpr_oracle.py (there is no reference code for dense refinement) on every host core, same metric,
    config object and step count as the CUDA arm; a step refines a bounded sample of the 4096-frame batch."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    workers = max(1, min(cores, 64))
    n = max(workers * 8, 32)                       # frames per step: a bounded sample of the 4096-frame workload
    frames, truth, init = sample_frames_for_cpu(n, 2000, workers)
    steps = args.steps                             # the CUDA arm's step count (a step takes ~0.2 s on 16 cores)
    walls, _ = cpu_refine(frames, init, workers, repeats=max(args.warmup, 1) + steps)
    times = walls[max(args.warmup, 1):]
    total = sum(times)
    value = n * len(times) / total
    assert not native_library_mapped(), "the CPU arm must not load libagt.so"
    line = {
        "impl": "reference", "metric": "refined poses/sec", "value": value, "unit": "poses/s", "n_gpus": args.gpus,
        "steps": len(times), "warmup": args.warmup, "ms_per_step": 1e3 * total / len(times), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": dpr_config(args.gpus, args.frames),
        "cpu_baseline": {"value": value, "unit": "poses/s", "cores": workers, "kind": "port",
                         "sample": f"{n} frames of the batch per step (synth.render, the numpy specification of the frame generator), "
                                   f"{workers} processes with one BLAS thread each, cv2.pyrDown pyramid + oracle/dpr_oracle.py; "
                                   "no reference code exists for this stage"},
        "e2e": {"value": value, "unit": "poses/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "native_library_mapped": native_library_mapped(),
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------
def run_gpu(args):
    import torch
    import torch.distributed as dist
    from accurate_aprilgroup_tracking_b200.context import AgtContext
    from accurate_aprilgroup_tracking_b200.cv_compat import HostContext

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a B200: the tracking path has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    B = args.frames
    ctx = AgtContext(local, CAM.mtx, None)
    ctx.set_synthetic_model()
    truth, init = make_poses(B, 2000 + 7919 * rank)
    pyr = ctx.alloc_pyramid(B, CAM.width, CAM.height, 4)
    for b0 in range(0, B, 512):                                   # synthetic frames, generated on device
        nb = min(512, B - b0)
        ctx.render(pyr, truth[b0:b0 + nb], np.arange(b0, b0 + nb) + 2000 + 7919 * rank, offset=b0, batch=nb)
    d_init = torch.as_tensor(init, dtype=torch.float64, device=ctx.tdev).reshape(B, 1, 6)
    # every step's poses are kept on the device ([steps][B][6] f64 per rank) and gathered ONCE, after the last step and inside
    # the timed region: the path itself has no exchange step (SURVEY.md 8e), and a per-step collective only coupled the
    # ranks step by step (round 1: 5.8 % slower at 8 GPUs)
    n_keep = max(args.steps, 1)
    all_poses = torch.zeros((n_keep, B, 6), dtype=torch.float64, device=ctx.tdev)
    gathered = torch.empty((world, n_keep, B, 6), dtype=torch.float64, device=ctx.tdev) if world > 1 else None
    step_no = [0]
    torch.cuda.synchronize()

    redo = torch.empty(B, dtype=torch.uint8, device=ctx.tdev)

    def step(ev=None):
        # K4 with K1 fused into it (every refinement builds the region of interest of its own pyramid level from the
        # frame), then the exactness net: frames whose refinement read outside that region get the full pyramid and
        # are refined again (both launches exit at once otherwise)
        if ev: ev[0].record()
        res = ctx.refine(pyr, d_init, 1, fused=True)
        if ev: ev[1].record()
        ctx._check(ctx.lib.agt_any_flag(ctx.h, ctx._p(res["left_roi"]), 1, ctx._p(redo), B))
        ctx.build_pyramid_masked(pyr, redo)
        ctx.refine(pyr, d_init, 1, mask=redo, out=res)
        if ev: ev[2].record()
        all_poses[step_no[0] % n_keep].copy_(res["pose"].reshape(B, 6))
        step_no[0] += 1
        return res

    def drain():
        if world > 1:
            dist.all_gather_into_tensor(gathered.reshape(world * n_keep * B, 6), all_poses.reshape(n_keep * B, 6))

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()          # sampled from the warm-up on, so short timed regions still see clocks under load
    for _ in range(max(args.warmup, 3)):
        res = step()
    drain()
    step_no[0] = 0
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(args.steps)]
    l0 = ctx.launch_count()
    t_begin = torch.cuda.Event(enable_timing=True)
    t_end = torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    t_begin.record()
    for k in range(args.steps):
        res = step(ev[k])
    drain()                                                       # the one gather of all poses is inside the timed region
    t_end.record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    launches = ctx.launch_count() - l0
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs:
        # what a caller of the refinement receives for the batch of the last timed step
        dump_outputs(args.dump_outputs, {k: res[k] for k in ("pose", "cost", "n_valid", "evals", "status", "left_roi")}, rank, world)
    gather_ok = True
    if world > 1:
        # every rank holds every rank's poses: its own block is bit-identical, and all ranks agree on a checksum of the whole
        gather_ok = bool(torch.equal(gathered[rank], all_poses))
        chk = gathered.sum(dim=(1, 2, 3)).clone()
        ref = chk.clone()
        dist.broadcast(ref, 0)
        gather_ok = gather_ok and bool(torch.equal(chk, ref)) and bool(torch.isfinite(chk).all())
        flag = torch.tensor([1.0 if gather_ok else 0.0], dtype=torch.float64, device=ctx.tdev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        gather_ok = bool(flag.item() == 1.0)
    elapsed_ms = t_begin.elapsed_time(t_end)
    t = torch.tensor([elapsed_ms], dtype=torch.float64, device=ctx.tdev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    elapsed_ms = float(t.item())
    dpr_ms = sum(e[0].elapsed_time(e[1]) for e in ev) / args.steps
    redo_ms = sum(e[1].elapsed_time(e[2]) for e in ev) / args.steps
    n_redo = int(redo.sum().item())
    # the full-frame pyramid kernel (what the LK stage consumes), timed on the same batch outside the step
    fe0, fe1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ctx.build_pyramid(pyr)
    fe0.record()
    for _ in range(5):
        ctx.build_pyramid(pyr)
    fe1.record()
    torch.cuda.synchronize()
    full_pyr_ms = fe0.elapsed_time(fe1) / 5
    # K4 alone on the pyramid just built (no K1 inside), for comparison with the fused launch of the step
    ke0, ke1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    plain = ctx.refine(pyr, d_init, 1)
    ke0.record()
    for _ in range(5):
        plain = ctx.refine(pyr, d_init, 1)
    ke1.record()
    torch.cuda.synchronize()
    k4_only_ms = ke0.elapsed_time(ke1) / 5
    inside = res["left_roi"] == 0
    fused_equals_plain = bool(all(torch.equal(res[k][inside], plain[k][inside]) for k in ("pose", "cost", "n_valid", "evals", "status")))

    # parity guard on the measured batch: the refined poses must sit near the truth they were rendered from
    pose = res["pose"].reshape(B, 6).cpu().numpy()
    evals = res["evals"].reshape(B).cpu().numpy().astype(np.int64)
    nvalid = res["n_valid"].reshape(B).cpu().numpy().astype(np.int64)
    status = res["status"].reshape(B).cpu().numpy()
    dt = np.linalg.norm(pose[:, 3:] - truth[:, 3:], axis=1)
    algo_bytes = float((BYTES_PER_SAMPLE_EVAL * nvalid * evals).sum() + BYTES_PER_POSE_FIXED * B)
    peak, peak_kind = measured_peaks()
    achieved = algo_bytes / (dpr_ms * 1e-3) / 1e9
    ncu = ncu_dpr_summary()

    # ---- e2e through the host-buffer C-ABI entry point: every rank at once (they share the host's memory and PCIe
    #      root complexes), timed by wall clock around the blocking call, max over ranks ----
    e2e = None
    import psutil
    enough_ram = psutil.virtual_memory().available > world * (B * CAM.width * CAM.height + (4 << 30))
    if not args.no_e2e and enough_ram:
        hctx = HostContext(local)
        s, tg, n, c = synth.surface_model()
        hctx.set_model(s, tg, n, c, synth.model_pitch())
        # the pinned frames of a rank live on the NUMA node of its GPU (one process per GPU: first-touch allocation)
        from accurate_aprilgroup_tracking_b200 import sharding as _sh
        with _sh.on_gpu_numa_node(local) as numa:
            host_frames = torch.empty((B, CAM.height, CAM.width), dtype=torch.uint8, pin_memory=True)
            host_frames.copy_(pyr.frames)
        torch.cuda.synchronize()
        hf = host_frames.numpy()
        e2e_steps = max(3, min(args.steps, 5))
        for _ in range(2):
            out = hctx.refine_poses(hf, init, CAM.mtx)              # warm-up (allocates device staging)
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            out = hctx.refine_poses(hf, init, CAM.mtx)
        e2e_s = (time.perf_counter() - t0) / e2e_steps
        tt = torch.tensor([e2e_s], dtype=torch.float64, device=ctx.tdev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        e2e_s = float(tt.item())
        same = float(np.abs(out["pose"].reshape(B, 6) - pose).max())
        h2d = hctx.last_h2d_bytes()
        e2e = {"value": B * world / e2e_s, "unit": "poses/s", "h2d_bytes_per_step": int(h2d),
               "d2h_bytes_per_step": int(B * (48 + 4 + 4 + 4 + 1 + 1)), "ms_per_step": 1e3 * e2e_s,
               "max_abs_diff_vs_device_path": same, "host_frame_bytes_per_step": int(B * CAM.width * CAM.height),
               "host_numa_node": numa,
               "note": "agt_refine_host on pinned host frames (allocated on the NUMA node of the rank's GPU when the host exposes one: host_numa_node), all ranks concurrently, max over ranks; per frame only the "
                       "rectangle the refinement can read is copied (frames that leave it are redone from the full frame)"}
        # the same call on PAGEABLE frames (what a numpy caller holds): host threads pack each chunk's rectangles into pinned
        # staging, one copy per chunk (agt_set_upload_threads); next to it the one-2-D-copy-per-frame path it replaces
        if world == 1 and psutil.virtual_memory().available > B * CAM.width * CAM.height + (8 << 30):
            hp = np.array(hf)                                        # pageable copy
            legs = {}
            for label, threads in (("staged", None), ("copy_per_frame", 0)):
                if threads is not None:
                    hctx.set_upload_threads(threads)
                outp = hctx.refine_poses(hp, init, CAM.mtx)         # warm-up (allocates the staging buffers)
                t0 = time.perf_counter()
                for _ in range(3):
                    outp = hctx.refine_poses(hp, init, CAM.mtx)
                legs[label] = (time.perf_counter() - t0) / 3
                assert float(np.abs(outp["pose"].reshape(B, 6) - pose).max()) == 0.0
            e2e["pageable"] = {"value": B / legs["staged"], "unit": "poses/s", "ms_per_step": 1e3 * legs["staged"],
                               "h2d_bytes_per_step": int(hctx.last_h2d_bytes()),
                               "upload_threads": min(8, os.cpu_count() or 4),
                               "copy_per_frame_ms_per_step": 1e3 * legs["copy_per_frame"],
                               "note": "agt_refine_host on frames in pageable host memory (a plain numpy array), same poses bit for bit"}
            del hp
        hctx.close()
        del host_frames

    # ---- BASELINE config 5 next to it, on every N the driver runs: the full pipeline (predictor -> PnP / LK fallback -> dense
    #      refinement, one frame of every stream per step), 64 streams per GPU (weak) and 64 streams in all (strong) ----
    streams = None
    secondary = {}
    if not args.no_streams:
        from accurate_aprilgroup_tracking_b200 import sharding as _sh
        frames_s = pyr.frames[:args.cpu_sample].cpu().numpy() if (rank == 0 and not args.no_cpu) else None
        del pyr, res, plain
        torch.cuda.empty_cache()
        F = 32
        weak = streams_measure(torch, dist, world, rank, ctx, 64 * world, list(range(64 * rank, 64 * rank + 64)), F, 2)
        torch.cuda.empty_cache()
        strong = streams_measure(torch, dist, world, rank, ctx, 64, _sh.local_streams(64, rank, world), F, 2) if world > 1 else weak
        torch.cuda.empty_cache()
        # the same 64 streams per GPU from pixels alone: the tag detector (N3) runs on the device in front of the path
        pixels = streams_measure(torch, dist, world, rank, ctx, 64 * world, list(range(64 * rank, 64 * rank + 64)), F, 2, from_pixels=True)
        torch.cuda.empty_cache()
        secondary["lk"] = dict(lk_measure(torch, dist, world, rank, ctx, 8192, 3, 3), metric="tracked corners/sec (BASELINE config 3)",
                               config=dict(LK_CONFIG, frame_pairs_per_gpu=8192))
        torch.cuda.empty_cache()
        secondary["multihyp"] = dict(multihyp_measure(torch, dist, world, rank, ctx, 64, 64, 3, 3),
                                     metric="refined poses/sec, 64 hypotheses per frame (BASELINE config 4)")
        torch.cuda.empty_cache()
        streams = {"metric": "refined poses/sec (full APE+LK+DPR pipeline, BASELINE config 5)",
                   "weak_64_streams_per_gpu": weak, "strong_64_streams": strong, "weak_64_streams_per_gpu_from_pixels": pixels,
                   "note": "one frame of every stream per step (frames of a stream are sequential: predictor and LK need the previous "
                           "frame), CUDA graph per step, frame ingest + K1 of the next frame on a side stream; streams pinned to GPUs, one "
                           "all-gather of all poses per sequence; from_pixels: no detections are handed in, agt_detect_tags_roi finds the "
                           "tags on a window around each stream's predicted pose and agt_pack_detections filters and maps them on the device"}
    else:
        frames_s = pyr.frames[:args.cpu_sample].cpu().numpy() if (rank == 0 and not args.no_cpu) else None

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- CPU baseline on a bounded sample of the same frames (rank 0, one core) ----
    cpu = None
    if not args.no_cpu:
        ns = args.cpu_sample
        walls, cpu_pose = cpu_refine(frames_s, init[:ns], 1)
        wall = walls[0]
        dr = [2 * math.asin(min(1.0, 0.5 * np.linalg.norm(synth.rodrigues(cpu_pose[i, :3]) - synth.rodrigues(pose[i, :3]))))
              for i in range(ns)]
        cpu = {"value": ns / wall, "unit": "poses/s", "cores": 1, "kind": "port",
               "sample": f"first {ns} frames of the batch: cv2.pyrDown pyramid + oracle/dpr_oracle.py (numpy, float64), 1 process",
               "max_rot_diff_vs_gpu_rad": float(max(dr)),
               "max_trans_diff_vs_gpu_m": float(np.abs(cpu_pose[:, 3:] - pose[:ns, 3:]).max())}

    value = B * world * args.steps / (elapsed_ms * 1e-3)
    sm_mhz = (clocks or {}).get("sm_mhz") or None
    roofline = {"bound": "hbm", "kernel": "dpr_kernel", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": None, "issue_frac": None, "peak_kind": peak_kind, "algorithmic_bytes": algo_bytes,
                "note": "per launch of the step (setup launch + dpr_kernel including its fused pyrDown); algorithmic bytes = 36 B x valid samples x "
                        "evaluations + 156 B per pose (SURVEY.md 8d), evaluation and sample counts returned by the kernel.  The ROI is read once (and "
                        "its pyramid level built) into shared memory and reused by every LM evaluation, so real DRAM traffic (`traffic`) is far "
                        "BELOW the algorithmic bytes and the kernel is bound by instruction issue: `issue_frac` = warp instructions issued / "
                        "(148 SMs x 4 schedulers x SM clock x kernel time) is the binding roofline"}
    if ncu is not None:
        scale = float((nvalid * evals).sum()) / max(float(ncu.get("sample_evals", 0.0)), 1.0)      # work of this launch / work of the captured one
        roofline["traffic"] = float(ncu["dram_bytes"]) * B / float(ncu["poses"])
        if sm_mhz:
            roofline["issue_frac"] = float(ncu["warp_instructions"]) * scale / (SM_COUNT * SCHEDULERS_PER_SM * sm_mhz * 1e6 * dpr_ms * 1e-3)
        roofline["ncu"] = {k: ncu.get(k) for k in ("source", "poses", "dram_bytes", "warp_instructions", "sample_evals", "issue_active_pct",
                                                  "kernel_ms_under_ncu", "agt_dpr_cu_sha256")}
    line = {
        "metric": "refined poses/sec", "value": value, "unit": "poses/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": elapsed_ms / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": dpr_config(world, B),
        "gpu_launches": int(launches), "all_ranks_hold_all_poses": gather_ok,
        "kernel_ms": {"dense_refinement_with_fused_pyramid": dpr_ms, "redo_pass": redo_ms,
                      "dense_refinement_on_built_pyramid": k4_only_ms, "full_frame_pyramid": full_pyr_ms},
        "fused_equals_built_pyramid_path": fused_equals_plain,
        "frames_redone_on_full_pyramid": n_redo,
        "lm": {"mean_evals": float(evals.mean()), "max_evals": int(evals.max()), "mean_samples": float(nvalid.mean()),
               "sample_evals": float((nvalid * evals).sum()),
               "converged_frac": float((status == 1).mean()), "median_trans_err_vs_truth_m": float(np.median(dt))},
        "roofline": roofline,
        "pyramid_roofline": {"kernel": "pyr_down_stream_kernel (full frames, 3 levels)", "bound": "hbm",
                             "achieved": PYR_BYTES_PER_1080P * B / (full_pyr_ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                             "frac": PYR_BYTES_PER_1080P * B / (full_pyr_ms * 1e-3) / 1e9 / peak},
        "clocks": clocks,
    }
    if streams is not None:
        line["streams"] = streams
    line.update(secondary)
    if e2e is not None:
        line["e2e"] = e2e
    if cpu is not None:
        line["cpu_baseline"] = cpu
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------
# secondary workloads (BASELINE.json configs 3-5); the driver's contract line is --workload dpr
# ------------------------------------------------------------------------------------------
def _dist_setup():
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a B200: the tracking path has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1 and not dist.is_initialized():
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    return torch, dist, world, rank, local


def _timed(torch, dist, world, fn, steps, warmup):
    for _ in range(max(warmup, 3)):
        fn()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def lk_measure(torch, dist, world, rank, ctx, B, steps, warmup):
    """Config 3 on this rank: B frame pairs x 48 corners.  -> dict (identical on every rank)."""
    traj = np.array([synth.trajectory(3000 + 7919 * rank + i, 2) for i in range(B)])
    pa, pb = ctx.alloc_pyramid(B, CAM.width, CAM.height, 4), ctx.alloc_pyramid(B, CAM.width, CAM.height, 4)
    for b0 in range(0, B, 512):
        nb = min(512, B - b0)
        ctx.render(pa, traj[b0:b0 + nb, 0], np.arange(nb) + b0, offset=b0, batch=nb)
        ctx.render(pb, traj[b0:b0 + nb, 1], np.arange(nb) + b0 + 1, offset=b0, batch=nb)
    ctx.build_pyramid(pa)
    obj = synth.object_points()
    pts = torch.as_tensor(np.stack([synth.project(obj, traj[i, 0], CAM) for i in range(B)]).astype(np.float32), device=ctx.tdev)
    holder = {}

    def step_full():
        ctx.build_pyramid(pb)                       # complete pyramid of the new frames (the previous one is reused)
        holder["full"] = ctx.lk(pa, pb, pts)

    def step():
        # pyramid of the new frames only where the corners can look + LK + exact redo of frames that looked outside
        holder["out"] = ctx.lk_roi(pa, pb, pts)

    full_ms = _timed(torch, dist, world, step_full, steps, 3) / steps
    l0 = ctx.launch_count()
    ms = _timed(torch, dist, world, step, steps, warmup)
    launches = (ctx.launch_count() - l0) * steps // (steps + max(warmup, 3))
    same = all(bool(torch.equal(a.view(torch.int32) if a.dtype == torch.float32 else a, b.view(torch.int32) if b.dtype == torch.float32 else b))
               for a, b in zip(holder["out"][:3], holder["full"]))
    redone = int(holder["out"][4].sum())
    ctx.build_pyramid(pb)
    lk_ms = _timed(torch, dist, world, lambda: holder.__setitem__("k", ctx.lk(pa, pb, pts)), steps, 3) / steps
    st = holder["out"][1]
    peak, kind = measured_peaks()
    corners = B * 48
    ach = LK_BYTES_PER_CORNER * corners / (lk_ms * 1e-3) / 1e9
    res = {"value": corners * world * steps / (ms * 1e-3), "unit": "corners/s", "ms_per_step": ms / steps, "steps": steps,
           "frame_pairs_per_gpu": B, "gpu_launches": int(launches), "kernel_ms": {"lk": lk_ms, "step_with_complete_pyramid": full_ms},
           "roi_equals_complete_pyramid_path": same, "frames_redone_on_complete_pyramid": redone, "tracked_frac": float(st.float().mean()),
           "roofline": {"bound": "hbm", "kernel": "lk_kernel", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                        "traffic": None, "peak_kind": kind,
                        "note": "5008 B per corner (SURVEY.md 8d); bound by instruction issue and the dependent float32 chains that make it "
                                "bit-identical to cv2.calcOpticalFlowPyrLK, not by bandwidth"}}
    del pa, pb, holder
    return res


LK_CONFIG = {"workload": "pyramidal LK: 4 levels, 21x21 window, 48 corners per 1080p frame pair",
             "step": "K1 pyramid of the new frames below the rectangles the corners can look at (32 px of flow) + K2 LK + "
                     "exact redo on complete pyramids of frames that looked outside", "l2": "inputs larger than L2"}


def run_lk(args):
    """Config 3: pyramidal LK, 4 levels, 21x21, 48 corners per frame pair."""
    torch, dist, world, rank, local = _dist_setup()
    from accurate_aprilgroup_tracking_b200.context import AgtContext
    ctx = AgtContext(local, CAM.mtx, None)
    r = lk_measure(torch, dist, world, rank, ctx, args.frames, args.steps, args.warmup)
    if rank == 0:
        print(json.dumps({
            "metric": "tracked corners/sec", "value": r["value"], "unit": "corners/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": r["ms_per_step"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "i32/f32", "data": "synthetic",
            "config": dict(LK_CONFIG, frame_pairs_per_gpu=args.frames),
            **{k: r[k] for k in ("gpu_launches", "kernel_ms", "roi_equals_complete_pyramid_path", "frames_redone_on_complete_pyramid",
                                 "tracked_frac", "roofline")}}), flush=True)


def multihyp_measure(torch, dist, world, rank, ctx, B, H, steps, warmup):
    """Config 4 on this rank: B frames x H hypotheses.  -> dict."""
    rng = np.random.default_rng(4000 + rank)
    truth = np.array([synth.random_pose(rng) for _ in range(B)])
    init = truth[:, None, :] + np.concatenate([rng.normal(0, 0.03, (B, H, 3)), rng.normal(0, 0.002, (B, H, 3))], axis=2)
    pyr = ctx.alloc_pyramid(B, CAM.width, CAM.height, 4)
    ctx.render(pyr, truth, np.arange(B) + 4000)
    d_init = torch.as_tensor(init, device=ctx.tdev)
    holder = {}

    def step():
        ctx.build_pyramid(pyr)
        res = ctx.refine(pyr, d_init, H)
        holder["res"], holder["best"] = res, ctx.select_best(res)

    l0 = ctx.launch_count()
    ms = _timed(torch, dist, world, step, steps, warmup)
    launches = ctx.launch_count() - l0
    res, (best, bp) = holder["res"], holder["best"]
    bp = bp.cpu().numpy()
    ev, nv = res["evals"].double(), res["n_valid"].double()
    dt = np.linalg.norm(bp[:, 3:] - truth[:, 3:], axis=1)
    out = {"value": B * world * steps / (ms * 1e-3), "unit": "poses/s", "ms_per_step": ms / steps, "steps": steps, "frames_per_gpu": B,
           "hypotheses": H, "gpu_launches": int(launches), "hypothesis_refinements_per_s": B * H * world * steps / (ms * 1e-3),
           "lm": {"mean_evals": float(ev.mean()), "converged_frac": float((res["status"] == 1).double().mean()),
                  "median_trans_err_vs_truth_m": float(np.median(dt)),
                  "algorithmic_GBps": float((BYTES_PER_SAMPLE_EVAL * ev * nv).sum()) * steps / (ms * 1e-3) / 1e9}}
    del pyr, holder
    return out


def run_multihyp(args):
    """Config 4: 64 perturbed hypotheses per frame, LM to convergence, arg-min selection."""
    torch, dist, world, rank, local = _dist_setup()
    from accurate_aprilgroup_tracking_b200.context import AgtContext
    ctx = AgtContext(local, CAM.mtx, None)
    ctx.set_synthetic_model()
    H = 64
    r = multihyp_measure(torch, dist, world, rank, ctx, max(1, args.frames // H), H, args.steps, args.warmup)
    if rank == 0:
        print(json.dumps({
            "metric": "refined poses/sec (64 hypotheses per frame)", "value": r["value"], "unit": "poses/s",
            "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": r["ms_per_step"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "multi-hypothesis dense refinement: 64 inits per 1080p frame (0.03 rad, 2 mm), LM to convergence",
                       "frames_per_gpu": r["frames_per_gpu"], "hypotheses": H},
            **{k: r[k] for k in ("gpu_launches", "hypothesis_refinements_per_s", "lm")}}), flush=True)


def streams_measure(torch, dist, world, rank, ctx, s_total, mine, n_frames, steps, from_pixels=False, groups=1):
    """Config 5 on this rank's streams `mine` (global stream ids): the whole sequence `steps` times, timed on the device, max
    over ranks.  -> dict (identical on every rank).  from_pixels: the tag detector runs on the device in front of the path
    (BatchedPoseDetector.step_frames: detect -> decision-margin filter -> id mapping -> APE ...) instead of detections handed in."""
    from accurate_aprilgroup_tracking_b200 import sharding
    from accurate_aprilgroup_tracking_b200.batched import BatchedPoseDetector
    S, F = len(mine), n_frames
    trajs = [synth.trajectory(5000 + s, F) for s in mine]
    rngs = [np.random.default_rng(5000 + s) for s in mine]
    bank = ctx.alloc_pyramid(S * F, CAM.width, CAM.height, 1)           # pre-rendered frames [F][S]
    for f in range(F):
        ctx.render(bank, np.array([trajs[i][f] for i in range(S)]), np.array([1000 * s + f for s in mine]), offset=f * S, batch=S)
    bpd = BatchedPoseDetector(ctx, S, CAM.width, CAM.height, synth.object_points())
    det_img, det_valid, det_n, det_packed = [], [], [], []
    for f in range(F):
        dets = []
        for i in range(S):
            d = synth.detections(trajs[i][f], CAM, rngs[i])
            if (f + 3 * i) % 17 == 16:
                d = d[:1]                                               # periodic detector dropouts exercise the LK path
            dets.append(d)
        a, b, c = bpd.pack(dets)
        det_img.append(torch.as_tensor(a, device=ctx.tdev)); det_valid.append(torch.as_tensor(b, device=ctx.tdev))
        det_n.append(torch.as_tensor(c, device=ctx.tdev))
        det_packed.append(bpd.pack_inputs(det_img[-1], det_valid[-1], det_n[-1]))      # one copy per step instead of three
    bank_frames = bank.frames.reshape(F, S, CAM.height, CAM.width)
    holder = {}
    hist = torch.zeros((S, F, 6), dtype=torch.float64, device=ctx.tdev)     # every stream's poses, frame by frame

    # frame ingest (device to device) and its pyramid are double-buffered: frame f+1 lands in the free slot, and K1 builds its
    # pyramid, on a side stream while the latency-bound rest of step f runs
    # from pixels: the detector of frame f+1 (search windows from the states before step f) runs on the side stream as well, under the
    # chain of step f, and K1 of frame f+1 - which the detector does not read - on a third stream.  The detector is then the longest
    # chain of the step (0.28 ms next to the refinement chain and K1, 0.19 ms alone), so its stream gets the high priority too.
    pipelined = from_pixels and os.environ.get("AGT_BENCH_PIPELINED_DETECT", "1") == "1"
    side, landed, stepped = torch.cuda.Stream(priority=-1 if pipelined else 0), torch.cuda.Event(), torch.cuda.Event()
    third, prepared, copied, built = torch.cuda.Stream(), torch.cuda.Event(), torch.cuda.Event(), torch.cuda.Event()

    def run_sequence():
        bpd.reset()
        main = torch.cuda.current_stream()
        acc = 0
        bpd.frames.copy_(bank_frames[0])
        stepped.record(main)
        for f in range(F):
            if f + 1 < F and os.environ.get("AGT_BENCH_SERIAL_INGEST") == "1":     # (probe: no overlap, the chain alone)
                bpd.ingest_next(bank_frames[f + 1])
                landed.record(main)
            elif f + 1 < F and os.environ.get("AGT_BENCH_SERIAL_INGEST") == "2":   # (probe: no ingest at all - stale frames)
                landed.record(main)
            elif f + 1 < F and pipelined:
                bpd.next_windows()                                      # where to look in frame f+1: from the states before step f
                prepared.record(main)
                side.wait_event(stepped)                                # the free slot was last read by step f-1
                side.wait_event(prepared)
                with torch.cuda.stream(side):
                    bpd.ingest_next(bank_frames[f + 1], build=False)    # ingest copy of the next frame
                    copied.record(side)
                    bpd.detect_next()                                   # its tags, into the input buffers of its slot
                    landed.record(side)
                k1s = third if os.environ.get("AGT_BENCH_K1_THIRD", "1") == "1" else side
                k1s.wait_event(copied)
                with torch.cuda.stream(k1s):
                    bpd.build_next()                                    # K1 of the next frame
                    built.record(k1s)
            elif f + 1 < F:
                side.wait_event(stepped)                                # the free slot was last read by step f-1
                with torch.cuda.stream(side):
                    bpd.ingest_next(bank_frames[f + 1])                 # ingest copy + K1 of the next frame
                    landed.record(side)
            if pipelined and f > 0:
                out = bpd.step(None)                                    # detections are in place (detect_next of the last iteration)
            else:
                out = bpd.step_frames() if from_pixels else bpd.step(det_packed[f])
            hist[:, f].copy_(out["pose"])
            stepped.record(main)
            if f + 1 < F:
                main.wait_event(landed)
                if pipelined:
                    main.wait_event(built)
            acc = out
        if world > 1:
            # NCCL: the final poses only - one all-gather of the whole sequence ([streams, frames x 6]), nothing per frame
            holder["all"] = sharding.gather_stream_poses(hist.reshape(S, F * 6), s_total)
        return acc

    if groups > 1:
        # the streams of this GPU as `groups` independent batches in flight at once (batched.StreamGroups): same poses, the
        # latency-bound chains of the groups overlap
        from accurate_aprilgroup_tracking_b200.batched import StreamGroups
        from accurate_aprilgroup_tracking_b200.context import AgtContext
        del bpd
        gctx = [AgtContext(ctx.device, CAM.mtx, None) for _ in range(groups)]
        for c in gctx:
            c.set_synthetic_model()
        sg = StreamGroups(gctx, S, CAM.width, CAM.height, synth.object_points())
        bpd = sg.dets[0]
        det_img_t, det_valid_t, det_n_t = torch.stack(det_img), torch.stack(det_valid), torch.stack(det_n)
        acc_last = torch.zeros(S, dtype=torch.int32, device=ctx.tdev)

        def run_sequence():                                             # noqa: F811
            sg.reset()
            sg.load(bank_frames[0])
            sg.fork()
            for f in range(F):
                nxt = bank_frames[f + 1] if f + 1 < F else None
                if from_pixels:
                    sg.step(next_frames=nxt, pose_out=hist[:, f], accepted_out=acc_last)
                else:
                    sg.step(det_img_t[f], det_valid_t[f], det_n_t[f], next_frames=nxt, pose_out=hist[:, f], accepted_out=acc_last)
            sg.join()
            if world > 1:
                holder["all"] = sharding.gather_stream_poses(hist.reshape(S, F * 6), s_total)
            return {"pose": hist[:, F - 1], "accepted": acc_last}

    # the steps run on a high-priority stream (the ingest of the next frame on a normal one): the latency-bound chain of a step
    # is not held up by the bandwidth-bound copy + K1 it overlaps with
    hp = torch.cuda.Stream(priority=-1) if os.environ.get("AGT_BENCH_STREAM_PRIORITY", "1") == "1" else torch.cuda.current_stream()
    with torch.cuda.stream(hp):
        run_sequence()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            out = run_sequence()
        e1.record()
        torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=ctx.tdev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    pose = out["pose"].cpu().numpy()
    dt = np.array([np.linalg.norm(pose[i, 3:] - trajs[i][F - 1][3:]) for i in range(S)])
    # the steps replay CUDA graphs of the same launch sequence; the three pyrDown launches of a frame run outside the graph
    res = {"value": s_total * F * steps / (ms * 1e-3), "unit": "poses/s", "ms_per_frame_step": ms / steps / F, "ms_per_sequence": ms / steps,
           "streams": s_total, "streams_per_gpu": S, "frames_per_stream": F, "sequences_timed": steps,
           "gpu_launches": int((bpd.kernels_per_step + 3) * F * steps), "kernels_per_frame_step": int(bpd.kernels_per_step) + 3,
           "cuda_graphs": True, "stream_groups": int(groups), "detector_one_frame_ahead": bool(pipelined),
           "pose_checksum": float(hist.sum().item()),
           "final_frame_median_trans_err_m": float(np.median(dt)),
           "accepted_frac_last": float(out["accepted"].float().mean())}
    del bank, bpd
    return res


def run_streams(args):
    """Config 5: concurrent 1080p streams, full APE + LK + DPR per frame.  --stream-scaling strong: 64 streams in all, stream s
    on GPU s mod G (BASELINE config 5); weak: 64 streams PER GPU (what a box serving more cameras than one GPU holds does)."""
    torch, dist, world, rank, local = _dist_setup()
    from accurate_aprilgroup_tracking_b200 import sharding
    from accurate_aprilgroup_tracking_b200.context import AgtContext
    ctx = AgtContext(local, CAM.mtx, None)
    ctx.set_synthetic_model()
    weak = args.stream_scaling == "weak"
    s_total = args.streams * world if weak else args.streams
    mine = list(range(rank * args.streams, (rank + 1) * args.streams)) if weak else sharding.local_streams(s_total, rank, world)
    pixels = args.stream_input == "pixels"
    r = streams_measure(torch, dist, world, rank, ctx, s_total, mine, args.stream_frames, args.steps, from_pixels=pixels,
                        groups=args.stream_groups)
    if rank == 0:
        print(json.dumps({
            "metric": "refined poses/sec (full APE+LK+DPR pipeline)", "value": r["value"], "unit": "poses/s",
            "n_gpus": world, "steps": args.steps, "warmup": 1, "ms_per_step": r["ms_per_sequence"], "higher_is_better": True,
            "scaling": "weak" if weak else "strong", "vs_baseline": None, "dtype": "f32/f64", "data": "synthetic",
            "config": {"workload": ("concurrent 1080p camera streams, " + ("tag detector (search window around the predicted pose) -> " if pixels else "")
                                    + "predictor -> PnP / LK fallback -> dense refinement per frame"),
                       "input": "frames only (tags detected on the device)" if pixels else "frames + tag detections",
                       "streams": s_total, "frames_per_stream": args.stream_frames, "step": "one pass over all frames of all streams",
                       "parallelism": (f"{args.streams} streams per GPU" if weak else f"streams s mod {world} -> GPU")
                                      + "; one NCCL all-gather of all poses at the end of the sequence"},
            **{k: r[k] for k in ("gpu_launches", "kernels_per_frame_step", "cuda_graphs", "stream_groups", "detector_one_frame_ahead", "pose_checksum", "ms_per_frame_step",
                                 "final_frame_median_trans_err_m", "accepted_frac_last")}}), flush=True)


def run_config1(args):
    """Config 1: the reference's own shape - one 640x480 camera stream, 300 frames, APE + LK + dense refinement per frame
    through the drop-in ``PoseDetector`` (host buffers in, attributes out, one frame at a time) - next to the CPU
    composition of the stage oracles (the reference's ``_estimate_pose`` state machine + OpenCV LK + dense oracle)."""
    import logging
    import tempfile
    import torch
    from accurate_aprilgroup_tracking_b200.aprilgroup_pose_estimation import PoseDetector
    from accurate_aprilgroup_tracking_b200.context import AgtContext
    cam = synth.CAMERA_VGA
    n = 300
    traj = synth.trajectory(1000, n)
    rng = np.random.default_rng(1000)
    ctx = AgtContext(0, cam.mtx, None)
    ctx.set_synthetic_model()
    pyr = ctx.alloc_pyramid(n, cam.width, cam.height, 1)
    ctx.render(pyr, traj, np.arange(n) + 1000)
    frames = pyr.frames.cpu().numpy()
    ctx.close()
    dets_all = []
    for f in range(n):
        d = synth.detections(traj[f], cam, rng)
        if f % 17 == 16:
            d = d[:1]                                   # periodic detector dropouts exercise the LK path
        dets_all.append(d)

    class _Det:
        def __init__(self, tag_id, corners):
            self.tag_id, self.corners, self.decision_margin = int(tag_id), np.asarray(corners, dtype=np.float64), 100.0
            self.center = self.corners.mean(axis=0)

    lg = logging.getLogger("agt-bench")
    lg.handlers[:] = [logging.NullHandler()]
    lg.propagate = False
    tmp = tempfile.mkdtemp()
    synth.write_april_group_json(tmp)
    cls = type("PD", (PoseDetector,), {"DIRPATH": os.path.join(tmp, "aprilgroup_tracking", "aprilgroup_pose_estimation")})

    def run_gpu_sequence():
        det = cls(lg, cam.mtx, None, True, use_lk=True, use_dense_refine=True)
        poses, t_frames = [], []
        for f in range(n):
            t0 = time.perf_counter()
            det.img = None
            det._set_gray(frames[f])
            lists = det._lists_from_detections([_Det(t, c) for t, c in dets_all[f]])
            if len(lists[0]) < 2:
                lists = det._track_lost_tags(*lists)
            det._estimate_pose(lists[0], lists[1])
            t_frames.append(time.perf_counter() - t0)
            pt = det.prev_transform
            poses.append(None if pt[0] is None else np.concatenate([pt[0].ravel(), pt[1].ravel().astype(np.float64)]))
        return poses, np.array(t_frames)

    run_gpu_sequence()                                   # warm-up: library load, scratch buffers, kernels
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    poses, t_frames = run_gpu_sequence()
    wall = time.perf_counter() - t0

    cpu = None
    if not args.no_cpu:
        from oracle import ape_oracle, dpr_oracle, pipeline_oracle
        sm, tg, nn, c = synth.surface_model()
        po = pipeline_oracle.PipelineOracle(ape_oracle.group_from_json(synth.april_group_dict()), cam.mtx,
                                            dpr_oracle.Model(sm, tg, nn, c, synth.model_pitch()))
        n_cpu = 60                                       # a bounded sample of the sequence: ~20 ms of oracle per frame
        worst_r = worst_t = 0.0
        t0 = time.perf_counter()
        for f in range(n_cpu):
            po.frame(frames[f], dets_all[f])
            if po.prev[0] is not None and poses[f] is not None:
                want = np.concatenate([po.prev[0].ravel(), po.prev[1].ravel().astype(np.float64)])
                dr = np.linalg.norm(synth.rodrigues(poses[f][:3]) - synth.rodrigues(want[:3]))
                worst_r, worst_t = max(worst_r, float(dr)), max(worst_t, float(np.abs(poses[f][3:] - want[3:]).max()))
        cpu_wall = time.perf_counter() - t0
        cpu = {"value": n_cpu / cpu_wall, "unit": "poses/s", "cores": 1, "kind": "port",
               "sample": f"first {n_cpu} frames of the sequence: reference APE state machine (cv2.solvePnP) + cv2.calcOpticalFlowPyrLK + oracle/dpr_oracle.py",
               "max_rot_diff_vs_gpu_rad": worst_r, "max_trans_diff_vs_gpu_m": worst_t}
    dt = np.array([np.linalg.norm(p[3:] - traj[f][3:]) for f, p in enumerate(poses) if p is not None])
    line = {"metric": "refined poses/sec (one 640x480 stream through the drop-in PoseDetector)", "value": n / wall, "unit": "poses/s",
            "n_gpus": 1, "steps": 1, "warmup": 1, "ms_per_step": 1e3 * wall, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32/f64", "data": "synthetic",
            "config": {"workload": "BASELINE config 1: 300-frame 640x480 synthetic sequence, APE + LK fallback + dense refinement per frame, "
                                   "one frame at a time through PoseDetector (host numpy in, attributes out)",
                       "frames": n},
            "ms_per_frame": {"median": float(np.median(t_frames) * 1e3), "p95": float(np.percentile(t_frames, 95) * 1e3)},
            "poses_accepted": int(sum(p is not None for p in poses)), "median_trans_err_vs_truth_m": float(np.median(dt))}
    if cpu:
        line["cpu_baseline"] = cpu
    print(json.dumps(line), flush=True)


def ensure_library():
    """libagt.so normally travels with the tree; if it is absent build it once (local rank 0) and let the others wait."""
    from accurate_aprilgroup_tracking_b200 import _build, _lib
    if _lib.LIB_PATH.exists():
        return
    if int(os.environ.get("LOCAL_RANK", "0")) == 0:
        _build.build()
        return
    for _ in range(600):
        if _lib.LIB_PATH.exists():
            time.sleep(1.0)
            return
        time.sleep(0.5)
    raise RuntimeError("libagt.so was not built")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--frames", type=int, default=None,
                    help="frames per GPU per step (default: 4096, BASELINE config 2; 8192 frame pairs for --workload lk, config 3)")
    ap.add_argument("--cpu-sample", type=int, default=96)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--workload", default="dpr", choices=["dpr", "lk", "multihyp", "streams", "config1"])
    ap.add_argument("--streams", type=int, default=64)
    ap.add_argument("--stream-frames", type=int, default=64)
    ap.add_argument("--stream-scaling", default="strong", choices=["strong", "weak"])
    ap.add_argument("--stream-groups", type=int, default=1,
                    help="streams of a GPU as this many independent batches in flight at once (batched.StreamGroups)")
    ap.add_argument("--stream-input", default="detections", choices=["detections", "pixels"],
                    help="streams workload: tag detections handed in (BASELINE config 5), or frames only - the detector runs on the device")
    ap.add_argument("--no-streams", action="store_true", help="skip the config-3/4/5 legs of the default line")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="default workload: write the refinement outputs of the last timed step to DIR/<name>.npy (float32/float64), "
                         "to compare two builds on the same seeded inputs")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.workload != "dpr"):
        ap.error("--dump-outputs applies to the default workload (--workload dpr) of this implementation")
    if args.frames is None:
        args.frames = 8192 if args.workload == "lk" else 4096
    ensure_library()
    if args.impl == "reference":
        run_reference(args)
    elif args.workload == "lk":
        run_lk(args)
    elif args.workload == "multihyp":
        run_multihyp(args)
    elif args.workload == "streams":
        run_streams(args)
    elif args.workload == "config1":
        run_config1(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
