"""K3 latency probe (run on the GPU box): one warp per frame, so a 64-frame step is one dependent chain per warp and the launch time is
the latency of the slowest frame.  Times agt_pnp back to back for a stream-sized batch (64) and for batches that fill the machine.
    python scripts/pnp_probe.py"""
import sys, numpy as np
sys.path.insert(0, '.')
import torch
from accurate_aprilgroup_tracking_b200 import synth
from accurate_aprilgroup_tracking_b200.context import AgtContext
cam = synth.CAMERA_1080P
ctx = AgtContext(0, cam.mtx, None)
t = torch
obj = synth.object_points().astype(np.float32)


def inputs(n, seed, sig_r, sig_t):
    rng = np.random.default_rng(seed)
    img = np.zeros((n, 48, 2), np.float32); valid = np.zeros((n, 48), np.uint8); poses = np.zeros((n, 6))
    for i in range(n):
        while True:
            p = synth.random_pose(rng); vis = synth.visible_tags(p)
            if len(vis) >= 2: break
        poses[i] = p
        img[i] = synth.project(obj.astype(np.float64), p, cam) + rng.normal(0, 0.1, (48, 2))
        for k in vis: valid[i, 4 * k:4 * k + 4] = 1
    guess = poses + np.concatenate([rng.normal(0, sig_r, (n, 3)), rng.normal(0, sig_t, (n, 3))], axis=1)
    return img, valid, guess


def run(n, with_guess, sig_r=0.01, sig_t=0.001, reps=200):
    img, valid, guess = inputs(n, 5, sig_r, sig_t)
    d = lambda a, dt: t.as_tensor(a, dtype=dt, device="cuda").contiguous()
    o, i, v, g = d(obj, t.float32), d(img, t.float32), d(valid, t.uint8), d(guess, t.float64)
    ug = t.ones(n, dtype=t.uint8, device="cuda")
    pose = t.empty((n, 6), dtype=t.float64, device="cuda"); ok = t.empty(n, dtype=t.uint8, device="cuda")
    err = t.empty(n, dtype=t.float32, device="cuda"); it = t.empty(n, dtype=t.int32, device="cuda")
    P = ctx._p
    ctx._use_current_stream()
    def call():
        ctx._check(ctx.lib.agt_pnp(ctx.h, P(o), P(i), P(v), P(g) if with_guess else None, P(ug) if with_guess else None, P(pose), P(ok), P(err), P(it), n, 48))
    for _ in range(5): call()
    e0, e1 = t.cuda.Event(enable_timing=True), t.cuda.Event(enable_timing=True)
    t.cuda.synchronize(); e0.record()
    for _ in range(reps): call()
    e1.record(); t.cuda.synchronize()
    us = e0.elapsed_time(e1) / reps * 1e3
    itn = it.cpu().numpy()
    print(f"batch {n:6d} guess {int(with_guess)} (sigma {sig_r} rad): {us:8.1f} us per launch, iterations mean {itn.mean():.2f} max {itn.max()}, "
          f"ok {int(ok.sum())}/{n}, checksum {float(pose.double().sum()):.12f}")


run(64, True)
run(64, True, 0.001, 0.0001)
run(64, False)
run(4096, True, reps=50)
run(4096, False, reps=50)
