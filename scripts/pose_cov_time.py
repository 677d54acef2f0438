"""Time agt_pose_covariance on the bench's batch: 4096 synthetic 1080p frames (bench.py's poses and seeds), refined with
agt_refine_fused (+ the left_roi redo), then the covariance of every refined pose.  The two launches alternate in the same
process, each between its own pair of CUDA events; the card's name and power limit are read in the same run.

  python scripts/pose_cov_time.py [--frames 4096] [--reps 30] [--out profiles/r03_pose_cov.log]
"""
import argparse
import subprocess
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))


def card():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as exc:
        q = f"power limit not read ({exc})"
    return f"{name}, power limit / max SM clock: {q}"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=4096)
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    from accurate_aprilgroup_tracking_b200 import synth
    from accurate_aprilgroup_tracking_b200.context import AgtContext
    cam = synth.CAMERA_1080P
    B = a.frames
    ctx = AgtContext(0, cam.mtx, None)
    ctx.set_synthetic_model()
    rng = np.random.default_rng(2000)                       # bench.py make_poses(B, 2000)
    truth = np.array([synth.random_pose(rng) for _ in range(B)])
    init = truth + np.concatenate([rng.normal(0, 0.01, (B, 3)), rng.normal(0, 0.0005, (B, 3))], axis=1)
    pyr = ctx.alloc_pyramid(B, cam.width, cam.height, 4)
    for b0 in range(0, B, 512):
        nb = min(512, B - b0)
        ctx.render(pyr, truth[b0:b0 + nb], np.arange(b0, b0 + nb) + 2000, offset=b0, batch=nb)
    d_init = torch.as_tensor(init, dtype=torch.float64, device=ctx.tdev).reshape(B, 1, 6)
    res = ctx.refine_fused(pyr, d_init, 1)                  # the pyramid as the step leaves it, and the poses
    pose = res["pose"].clone()
    out = ctx.pose_covariance(pyr, d_init, pose)
    torch.cuda.synchronize()
    n_redo = int(res["redo"].sum())
    ok = int(out["ok"].sum())
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    t_ref, t_cov = [], []
    for rep in range(a.reps + 3):
        ev[0].record()
        ctx.refine(pyr, d_init, 1, fused=True, out={k: v for k, v in res.items() if k != "redo"})
        ev[1].record()
        ev[2].record()
        ctx.pose_covariance(pyr, d_init, pose, out=out)
        ev[3].record()
        torch.cuda.synchronize()
        if rep >= 3:                                        # warm-up
            t_ref.append(ev[0].elapsed_time(ev[1]))
            t_cov.append(ev[2].elapsed_time(ev[3]))
    t_ref, t_cov = np.array(t_ref), np.array(t_cov)
    s = [f"# python scripts/pose_cov_time.py --frames {B} --reps {a.reps}",
         f"card: {card()}",
         f"batch: {B} synthetic 1080p frames (bench.py poses, seeds 2000..), 1 hypothesis; {n_redo} frames redone after left_roi; "
         f"covariance ok for {ok} of {B}",
         f"agt_refine_fused:    median {np.median(t_ref):.3f} ms  (min {t_ref.min():.3f}, max {t_ref.max():.3f}) per {B} poses",
         f"agt_pose_covariance: median {np.median(t_cov):.3f} ms  (min {t_cov.min():.3f}, max {t_cov.max():.3f}) per {B} poses",
         f"ratio covariance / refinement: {np.median(t_cov) / np.median(t_ref):.3f}"]
    print("\n".join(s))
    if a.out:
        Path(a.out).write_text("\n".join(s) + "\n")


if __name__ == "__main__":
    main()
