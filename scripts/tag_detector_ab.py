"""Detector time and output, two builds of libagt.so in one process: python scripts/tag_detector_ab.py OTHER_LIBAGT_SO

Times agt_detect_tags per 64 windowed and per 64 whole 1080p frames (the frames and windows of scripts/tag_time_probe.py),
alternating the in-tree library and OTHER round by round (CUDA events, 20 calls per round, 10 rounds), and checks that both give
the same tags (ids and corner bytes, per frame, sorted) on those frames and on the frames of test_detect_tags_against_aruco_and_truth.
Prints the card's name and power limit with the numbers."""
import ctypes as C
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, ".")
from accurate_aprilgroup_tracking_b200 import _lib, synth  # noqa: E402
from accurate_aprilgroup_tracking_b200.context import AgtContext  # noqa: E402


def context_on(path, mtx):
    """AgtContext bound to the library at `path` (prototypes of the symbols it has)."""
    lib = C.CDLL(path)
    for name, (res, args) in _lib.PROTOTYPES.items():
        if hasattr(lib, name):
            getattr(lib, name).restype = res
            getattr(lib, name).argtypes = args
    saved, _lib._lib = _lib._lib, lib
    try:
        return AgtContext(0, mtx, None)
    finally:
        _lib._lib = saved


def tags(det):
    d = {k: v.cpu().numpy() for k, v in det.items()}
    return [sorted((int(d["id"][f, j]), d["corners"][f, j].tobytes()) for j in range(int(d["n"][f]))) for f in range(len(d["n"]))]


def main():
    other = sys.argv[1]
    print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"], capture_output=True, text=True).stdout)
    cam = synth.CAMERA_1080P
    ctxs = {"branch": AgtContext(0, cam.mtx, None), "other": context_on(other, cam.mtx)}
    n = 64
    poses = np.array([synth.trajectory(5000 + s, 1)[0] for s in range(n)])
    data = {}
    for name, ctx in ctxs.items():
        pyr = ctx.alloc_pyramid(n, cam.width, cam.height, 1)
        ctx.render(pyr, poses, np.arange(n))
        state = ctx.new_stream_state(n)
        st = state.cpu().numpy(); st[:, 0] = 1.0; st[:, 1:7] = poses
        state.copy_(torch.tensor(st, device=state.device))
        rects = ctx.track_rects(state, cam.width, cam.height, float(np.linalg.norm(synth.object_points(), axis=1).max()), 48)
        data[name] = (pyr, rects)
    for which in ("window", "whole"):
        outs = {}
        for name, ctx in ctxs.items():
            pyr, rects = data[name]
            outs[name] = tags(ctx.detect_tags(pyr, rects=rects if which == "window" else None))
        print(f"{which}: identical tags {outs['branch'] == outs['other']}, {sum(map(len, outs['branch']))} tags")
    for cam_t in (synth.CAMERA_VGA, synth.CAMERA_1080P):
        ps = np.array([synth.trajectory(s, 1)[0] for s in range(700, 724)])
        res = {}
        for name, ctx in ctxs.items():
            ctx.set_camera(cam_t.mtx)
            pyr = ctx.alloc_pyramid(len(ps), cam_t.width, cam_t.height, 1)
            ctx.render(pyr, ps, np.arange(700, 724))
            res[name] = tags(ctx.detect_tags(pyr, refine_win=4))
        print(f"seeds 700-723 {cam_t.width}x{cam_t.height}: identical tags {res['branch'] == res['other']}, {sum(map(len, res['branch']))} tags")
    # frames with more than 4096 components (tests/tag_quad_cases.py): which of the tags quads_np + decode_np find each build finds
    from oracle import tag_oracle
    from tests import tag_quad_cases
    for case in tag_quad_cases.max_component_cases():
        g = case["gray"]
        r = tag_oracle.quads_np(g, case["rect"], case["local"])
        want = {tag_oracle.decode_np(g, q["alts"][0]["corners"].astype(np.float64))[0] for q in r["quads"]} - {-1}
        found = {}
        for name, ctx in ctxs.items():
            ctx.set_tag_threshold("local" if case["local"] else "window")
            pyr = ctx.alloc_pyramid(1, g.shape[1], g.shape[0], 1)
            ctx.upload_frames(pyr, g[None])
            found[name] = sorted({i for i, _ in tags(ctx.detect_tags(pyr, max_tags=1024))[0]})
            ctx.set_tag_threshold("auto")
        print(f"{case['name']}: oracle tags {sorted(want)}; branch {found['branch']}; other {found['other']}")
    times = {(name, which): [] for name in ctxs for which in ("window", "whole")}
    for name, ctx in ctxs.items():
        pyr, rects = data[name]
        for _ in range(5):
            ctx.detect_tags(pyr, rects=rects); ctx.detect_tags(pyr)
    torch.cuda.synchronize()
    for _ in range(10):
        for name, ctx in ctxs.items():
            pyr, rects = data[name]
            for which in ("window", "whole"):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(20):
                    ctx.detect_tags(pyr, rects=rects if which == "window" else None)
                e1.record()
                torch.cuda.synchronize()
                times[(name, which)].append(e0.elapsed_time(e1) / 20)
    for (name, which), t in times.items():
        print(f"{name:6s} {which:6s}: median {np.median(t):.4f} ms, min {np.min(t):.4f}, max {np.max(t):.4f} per {n} frames")


if __name__ == "__main__":
    main()
