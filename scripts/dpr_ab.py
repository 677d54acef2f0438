"""bench.py's dense-refinement step, two builds of libagt.so in one process: python scripts/dpr_ab.py OTHER_LIBAGT_SO [--rounds N]

Both builds refine the bench's batch (4096 1080p frames of bench.make_poses(4096, 2000), one pyramid each) with bench.py's
step: the refinement with K1 fused, the flag reduction, the masked pyramid of the frames whose refinement left its ROI and
their redo.  Rounds alternate the in-tree library and OTHER (CUDA events, 20 steps per round after a warm-up), and report
the median, min and max per step of the whole step and of the fused refinement launch alone.  Every output of the last
step of each round is compared byte for byte between the two builds.  Prints the card's name, power limit and SM clock."""
import argparse
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, ".")
import bench  # noqa: E402
from accurate_aprilgroup_tracking_b200 import synth  # noqa: E402
from scripts.dpr_bits_golden import context_on  # noqa: E402

FIELDS = ("pose", "cost", "n_valid", "evals", "status", "left_roi")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("other")
    ap.add_argument("--rounds", type=int, default=12)
    ap.add_argument("--steps", type=int, default=20)
    args = ap.parse_args()
    q = "name,power.limit,clocks.max.sm,clocks.sm"
    print(subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv"], capture_output=True, text=True).stdout)
    cam = synth.CAMERA_1080P
    B = 4096
    truth, init = bench.make_poses(B, 2000)
    runs = {}
    for name, path in (("branch", None), ("other", args.other)):
        ctx = context_on(path, cam.mtx)
        ctx.set_synthetic_model()
        pyr = ctx.alloc_pyramid(B, cam.width, cam.height, 4)
        for b0 in range(0, B, 512):
            nb = min(512, B - b0)
            ctx.render(pyr, truth[b0:b0 + nb], np.arange(b0, b0 + nb) + 2000, offset=b0, batch=nb)
        d_init = torch.as_tensor(init, dtype=torch.float64, device=ctx.tdev).reshape(B, 1, 6)
        redo = torch.empty(B, dtype=torch.uint8, device=ctx.tdev)

        def step(ev=None, ctx=ctx, pyr=pyr, d_init=d_init, redo=redo):
            if ev: ev[0].record()
            res = ctx.refine(pyr, d_init, 1, fused=True)
            if ev: ev[1].record()
            ctx._check(ctx.lib.agt_any_flag(ctx.h, ctx._p(res["left_roi"]), 1, ctx._p(redo), B))
            ctx.build_pyramid_masked(pyr, redo)
            ctx.refine(pyr, d_init, 1, mask=redo, out=res)
            if ev: ev[2].record()
            return res

        for _ in range(5):
            step()
        runs[name] = step
    torch.cuda.synchronize()
    times = {(n, w): [] for n in runs for w in ("step", "fused")}
    identical = True
    for _ in range(args.rounds):
        outs = {}
        for name, step in runs.items():
            ev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(args.steps)]
            for k in range(args.steps):
                res = step(ev[k])
            torch.cuda.synchronize()
            times[(name, "step")].append(np.mean([e[0].elapsed_time(e[2]) for e in ev]))
            times[(name, "fused")].append(np.mean([e[0].elapsed_time(e[1]) for e in ev]))
            outs[name] = {k: res[k].cpu().numpy().tobytes() for k in FIELDS}
        identical &= outs["branch"] == outs["other"]
    print(subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv"], capture_output=True, text=True).stdout)
    print(f"outputs of both builds byte-identical in every round: {identical}")
    for (name, which), t in times.items():
        print(f"{name:6s} {which:5s}: median {np.median(t):.4f} ms, min {np.min(t):.4f}, max {np.max(t):.4f} "
              f"per {B}-frame step ({args.rounds} rounds of {args.steps})")


if __name__ == "__main__":
    main()
