"""The dense-refinement runs whose outputs tests/test_gpu_dpr_bits.py pins to the bit, and the golden file they are pinned to.

- 256 frames of the bench's seeded 1080p batch (bench.make_poses, frames rendered on the device as bench.py renders them),
  refined with K1 fused (every level above 0 built by the refinement itself) and from a complete pyramid.  256 jobs run as
  the one-CTA form, dpr_kernel<1>.
- The case frames of tests/test_gpu_dpr_forms.py (1080p and VGA, good / moderate / poor starts) in each of the four launch
  forms, fused and plain, one hypothesis per frame, at the high end of each form's job range.  Their off-axis views, image
  corners and the start whose answer lies outside the planned ROI put samples outside the staged tile, so every kind of
  warp-pair of the sample loop occurs: all lanes in the tile, none, some, and a thread's odd last sample.

Outputs per run: pose, cost, n_valid, evals, status, left_roi (the fused runs also after their redo from a complete
pyramid, as bench.py's step does it).  scripts/dpr_bits_golden.py writes them to GOLDEN."""
import numpy as np

from accurate_aprilgroup_tracking_b200 import synth
from tests import test_gpu_dpr_forms as forms
from tests import util

GOLDEN = util.ROOT / "tests" / "golden" / "dpr_bits.npz"
FIELDS = ("pose", "cost", "n_valid", "evals", "status", "left_roi")
BENCH_FRAMES = 256


class CaseFrames:
    """The frames and starts of test_gpu_dpr_forms.CaseSet (same seeds, same order of draws), without its oracle runs:
    what _run_form reads."""

    def __init__(self, ctx, cam_name, seed):
        self.ctx, self.cam_name = ctx, cam_name
        self.cam = cam = synth.CAMERA_1080P if cam_name == "1080p" else synth.CAMERA_VGA
        self.specs = forms._case_specs(cam_name)
        rng = np.random.default_rng(seed)
        truth, init = [], []
        for _, t, pin, _, _ in self.specs:
            pose = synth.random_pose(rng)
            if t is not None:
                pose[6 - len(t):] = t
            truth.append(pose)
            starts = []
            for _, sr, st in forms.STARTS:
                start = pose + np.concatenate([rng.normal(0, sr, 3), rng.normal(0, st, 3)])
                for k, v in pin.items():
                    start[k] = v
                starts.append(start)
            init.append(starts)
        self.truth, self.init = np.array(truth), np.array(init)
        self.n = len(self.specs)
        self.src = ctx.alloc_pyramid(self.n, cam.width, cam.height, forms.LEVELS)
        ctx.render(self.src, self.truth, np.arange(self.n) + seed)
        ctx.build_pyramid(self.src)
        ctx.sync()


def _bench_runs(ctx):
    import bench
    cam = synth.CAMERA_1080P
    truth, init = bench.make_poses(BENCH_FRAMES, 2000)
    pyr = ctx.alloc_pyramid(BENCH_FRAMES, cam.width, cam.height, forms.LEVELS)
    ctx.render(pyr, truth, np.arange(BENCH_FRAMES) + 2000)
    for l in range(1, forms.LEVELS):
        pyr.levels[l].fill_(255)          # what a fused refinement reads outside the region it built is fixed, not stale memory
    d_init = ctx.torch.as_tensor(init, dtype=ctx.torch.float64, device=ctx.tdev).reshape(BENCH_FRAMES, 1, 6)
    out = {}
    fused = ctx.refine(pyr, d_init, 1, fused=True)
    out["bench_fused"] = {k: fused[k].cpu().numpy() for k in FIELDS}
    ctx.build_pyramid(pyr)
    plain = ctx.refine(pyr, d_init, 1)
    out["bench_plain"] = {k: plain[k].cpu().numpy() for k in FIELDS}
    del pyr
    return out


def run_all(ctx1080, ctxvga):
    """-> {"<run>/<field>": array} for every run above."""
    import torch
    out = _bench_runs(ctx1080)
    ranges = forms._form_ranges(torch.cuda.get_device_properties(0).multi_processor_count)
    for cam_name, ctx, seed in (("1080p", ctx1080, 3100), ("vga", ctxvga, 3200)):
        cs = CaseFrames(ctx, cam_name, seed)
        for form in forms.FORMS:
            jobs = ranges[form][1]
            for fused in (False, True):
                r = forms._run_form(cs, form, jobs, 1, fused, 9000 + 10 * form + fused)
                name = f"{cam_name}_form{form}_{'fused' if fused else 'plain'}"
                out[name] = r["out"]
                if fused:
                    out[name + "_redo"] = r["redo"]
        del cs
        torch.cuda.empty_cache()
    return {f"{run}/{k}": np.ascontiguousarray(v[k]) for run, v in out.items() for k in FIELDS}
