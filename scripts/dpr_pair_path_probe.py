"""Share of warp-pairs that take the dense refinement's fast pair body, on the bench's batch (CPU only):
python scripts/dpr_pair_path_probe.py [--frames N]

For the seeded batch bench.py refines (bench.make_poses(4096, 2000)), every active sample is projected at the initial pose
in float64, on the level and against the staged tile of the refinement's plan (tests/test_gpu_dpr_forms.dpr_plan, the numpy
restatement of agt_dpr_plan).  The samples are dealt to the threads of the one-CTA form as dpr_kernel<1> deals them (thread
t takes samples t, t + 256, ... of the concatenated active tags), and a warp-pair counts as fast when all 32 lanes hold two
samples whose footprints lie inside the tile.  That is the share of the first evaluation's pairs that skip eval_sample;
later evaluations move the pose by a fraction of a pixel."""
import argparse
import math
import sys

import numpy as np

sys.path.insert(0, ".")
import bench  # noqa: E402
from accurate_aprilgroup_tracking_b200 import synth  # noqa: E402
from oracle import dpr_oracle  # noqa: E402
from tests.test_gpu_dpr_forms import dpr_plan  # noqa: E402

THREADS = 256


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=4096)
    args = ap.parse_args()
    cam = synth.CAMERA_1080P
    s, tg, n, c = synth.surface_model()
    model = dpr_oracle.Model(s, tg, n, c, synth.model_pitch())
    radius = float(np.linalg.norm(s[:, :3].astype(np.float64), axis=1).max())
    _, init = bench.make_poses(args.frames, 2000)
    pairs = fast = 0
    samples = in_tile = 0
    for p in init:
        lvl, _, (tx0, ty0, tw, th) = dpr_plan(cam, p[3:], radius)
        act = dpr_oracle.active_tags(model, dpr_oracle.rodrigues(p[:3]), p[3:])
        x = s[np.isin(tg, np.nonzero(act)[0]), :3].astype(np.float64)    # tag-major: the kernel's concatenated order
        xc = x @ dpr_oracle.rodrigues(p[:3]).T + p[3:]
        sc = 1.0 / (1 << lvl)
        z = np.where(xc[:, 2] > 1e-6, xc[:, 2], 1.0)
        ul = (cam.fx * xc[:, 0] / z + cam.cx) * sc
        vl = (cam.fy * xc[:, 1] / z + cam.cy) * sc
        lx, ly = np.floor(ul) - tx0 - 1, np.floor(vl) - ty0 - 1
        ok = (xc[:, 2] > 2e-6) & (lx >= 0) & (lx < tw - 3) & (ly >= 0) & (ly < th - 3)
        samples += len(ok)
        in_tile += int(ok.sum())
        # thread t, pair k: samples t + 256 * 2k and t + 256 * (2k + 1)
        n_s = len(ok)
        per = math.ceil(n_s / THREADS)
        grid = np.zeros((THREADS, per + (per & 1)), bool)              # [thread, sample of the thread], False = no sample
        idx = np.arange(n_s)
        grid[idx % THREADS, idx // THREADS] = ok
        lane_pairs = grid[:, 0::2] & grid[:, 1::2]                     # [thread, pair]
        warp_pairs = lane_pairs.reshape(THREADS // 32, 32, -1).all(axis=1)
        # pairs a warp runs: the most any of its lanes holds (a lane past its last sample forces eval_sample)
        left = np.maximum(0, (n_s - np.arange(THREADS) + THREADS - 1) // THREADS)
        n_pairs = ((left + 1) // 2).reshape(THREADS // 32, 32).max(axis=1)
        for w in range(THREADS // 32):
            pairs += int(n_pairs[w])
            fast += int(warp_pairs[w, :n_pairs[w]].sum())
    print(f"{args.frames} frames of bench.make_poses({args.frames}, 2000), 1080p, first evaluation, dpr_kernel<1>")
    print(f"samples with the footprint inside the tile: {in_tile} of {samples} ({100.0 * in_tile / samples:.2f} %)")
    print(f"warp-pairs on the fast body: {fast} of {pairs} ({100.0 * fast / pairs:.2f} %)")


if __name__ == "__main__":
    main()
