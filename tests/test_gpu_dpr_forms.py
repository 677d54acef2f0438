"""K4 dense refinement in each of its four launch forms, against oracle/dpr_oracle.py.

refine_impl (csrc/agt_dpr.cu) picks the form from the job count batch * n_hyp and the number of CTA slots, twice the SM
count: one CTA per refinement with a separate setup launch (dpr_kernel<1> after dpr_prep_kernel) when the jobs outnumber
half the slots, otherwise a cluster of 2, 4 or 8 CTAs that derives the setup in the kernel and splits the samples by rank.
Each form is run here on purpose, at both ends of its job range, with the case frames at different positions of a larger
batch padded with masked frames, for one and for three hypotheses per frame, with and without K1 fused into it.

The case set aims at the places where the kernel has code of its own: starts 1 mm either side of each pyramid-level
boundary (the level is frozen at the start), a level-3 close-up and a level-0 far view, off-axis views whose level ROI
is wider than the shared-memory tile (samples outside it take the global-memory fetch), objects cut by an image corner
down to a sliver with few valid samples, and poor starts that end at the evaluation cap.  Each frame is refined from a
good (0.01 rad, 0.5 mm), a moderate (0.03 rad, 2 mm) and a poor (0.08 rad, 5 mm) start.
"""
import math

import numpy as np
import pytest

from accurate_aprilgroup_tracking_b200 import synth
from tests import util

pytestmark = pytest.mark.gpu

STARTS = (("good", 0.01, 0.0005), ("moderate", 0.03, 0.002), ("poor", 0.08, 0.005))
FORMS = (1, 2, 4, 8)
C1_TOP = 4096                   # the high end of the one-CTA form: the bench batch
LEVELS = 4
# agt_dpr_plan.cuh
TILE_ROWS, TILE_PITCH, DRIFT_MARGIN = 270, 288, 8
# a sentinel in every output of a masked frame: the kernel must leave them as they are
SENTINEL = {"pose": -7.25, "cost": -3.5, "n_valid": -11, "evals": -13, "status": 201, "left_roi": 202}
ST_CONVERGED, ST_MAX_EVALS = 1, 2
MAX_EVALS = 50
# An oracle run compared pose for pose has converged with this many evaluations to spare: the float32 trajectory of a
# run that creeps to its fixed point (a 1.4 cm close-up with 90 valid samples, a corner sliver) takes a few evaluations
# more or fewer than the oracle's and may end at the cap a few um from it; such runs are checked like capped ones.
EVAL_MARGIN = 10
# Late runs are still held to the parity bar where the kernel converges too, unless the oracle's answer rests on fewer
# valid samples than this: the VGA view 1.4 cm from the tag surface (89 samples) has several fixed points, and the forms
# converge to ones 2e-2 rad from the oracle's (logged, not asserted).
MIN_SAMPLES_LATE = 100


def _at_fixed_point(ref):
    return ref["status"] == ST_CONVERGED and ref["evals"] <= MAX_EVALS - EVAL_MARGIN


# ------------------------------------------------------------------------------------------
# the case set
# ------------------------------------------------------------------------------------------
def _boundaries(cam):
    """Depths where the level changes: q = fx * pitch / z crosses 2, 4, 8 (0.42 / 0.21 / 0.105 m at 1080p)."""
    return [cam.fx * synth.model_pitch() / q for q in (2.0, 4.0, 8.0)]


def _case_specs(cam_name):
    """(name, translation (or whole pose) or None for a random working-volume pose, start coordinates fixed by the case
    {index: value}, expected level or None, what the case aims at: "cut" (tile cut), "border" (cut by the image border),
    "sliver" (few valid samples), "exit" (samples outside the ROI at the answer))."""
    cam = synth.CAMERA_1080P if cam_name == "1080p" else synth.CAMERA_VGA
    specs = []
    for lvl, zb in enumerate(_boundaries(cam)):
        specs.append((f"boundary {zb:.4f} m -1 mm", (0.004, -0.003, zb - 1e-3), {5: zb - 1e-3}, lvl + 1, None))
        specs.append((f"boundary {zb:.4f} m +1 mm", (-0.003, 0.004, zb + 1e-3), {5: zb + 1e-3}, lvl, None))
    if cam_name == "1080p":
        # tile cuts: the start is where the level ROI is widest (the plan cuts 16 px off its left side); the object
        # lies 3-4 mm to the left of it, so that the refinement reads samples left of the tile (and of the ROI)
        specs += [("level-3 close-up", (0.004, 0.002, 0.08), {}, 3, None),
                  ("level-0 far", (-0.02, 0.01, 0.58), {}, 0, None),
                  ("off-axis above 0.42 m, tile cut", (0.195, 0.0, 0.421), {3: 0.198, 5: 0.421}, 0, "cut"),
                  ("off-axis above 0.21 m, tile cut", (0.0927, 0.0, 0.211), {3: 0.0967, 5: 0.211}, 1, "cut"),
                  ("cut by a corner", (0.16, 0.09, 0.27), {}, 1, "border"),
                  ("sliver in a corner", (0.197, 0.116, 0.27), {}, 1, "sliver")]
        n_random = 4
        # an exit the kernel must report: the start 5 mm to the left of the object, so that at the answer 8 samples, all in
        # the second half of the split when the samples are shared by 2 CTAs, lie right of the ROI planned at the start
        edge = [("few samples leave the ROI", (0.1765, 0.0171, 0.328, -0.0074, -0.0293, 0.3105), (-0.005, 0.0))]
    else:
        specs += [("cut by a corner", (0.11, 0.085, 0.25), {}, 0, "border"),
                  ("sliver in a corner", (-0.148, -0.115, 0.25), {}, 0, "sliver")]
        n_random = 2
    specs += [(f"random {k}", None, {}, None, None) for k in range(n_random)]
    if cam_name == "1080p":
        specs += [(name, pose, {3: pose[3] + dx, 4: pose[4] + dy, 5: pose[5]}, 1, "exit") for name, pose, (dx, dy) in edge]
    return specs


def _level_sizes(cam):
    ws, hs = [cam.width], [cam.height]
    for _ in range(LEVELS - 1):
        ws.append((ws[-1] + 1) // 2)
        hs.append((hs[-1] + 1) // 2)
    return ws, hs


def dpr_plan(cam, t, radius):
    """numpy restatement of agt_make_dpr_plan: level, predicted ROI (x0, y0, x1, y1) and staged tile (x0, y0, w, h)."""
    ws, hs = _level_sizes(cam)
    q = cam.fx * synth.model_pitch() / t[2]
    lvl = 0 if q < 2 else 1 if q < 4 else 2 if q < 8 else 3
    lvl = min(lvl, LEVELS - 1)
    lw, lh, sc = ws[lvl], hs[lvl], 1.0 / (1 << lvl)
    ext = []
    for c, f, pp in ((t[0], cam.fx, cam.cx), (t[1], cam.fy, cam.cy)):
        sb = min(radius / math.hypot(c, t[2]), 0.95)
        al, be = math.atan2(c, t[2]), math.asin(sb)
        lo, hi = max(al - be, -1.5), min(al + be, 1.5)
        ext += [(f * math.tan(lo) + pp) * sc - DRIFT_MARGIN - 2, (f * math.tan(hi) + pp) * sc + DRIFT_MARGIN + 2]
    x0, x1 = math.floor(ext[0]), math.ceil(ext[1]) + 1
    y0, y1 = math.floor(ext[2]), math.ceil(ext[3]) + 1
    x0, y0 = max(x0, 0) & ~15, max(y0, 0)
    x1, y1 = max(min(x1, lw), x0), max(min(y1, lh), y0)
    roi = (x0, y0, x1, y1)
    tw, th = x1 - x0, y1 - y0
    if tw > TILE_PITCH:
        x0 += (tw - TILE_PITCH + 31) // 32 * 16
        tw = min(lw - x0, TILE_PITCH)
    if th > TILE_ROWS:
        y0 += (th - TILE_ROWS) // 2
        th = TILE_ROWS
    return lvl, roi, (x0, y0, max(tw, 0), max(th, 0))


def _rect_l0(cam, plan):
    """agt_dpr_rect_l0 of one hypothesis: the plan's ROI at level 0 plus the pyrDown halo (what agt_dpr_rects returns)."""
    lvl, (x0, y0, x1, y1), _ = plan
    if x1 <= x0 or y1 <= y0:
        return (0, 0, 0, 0)
    pad = 2 << lvl
    return ((max((x0 << lvl) - pad, 0) & ~15), max((y0 << lvl) - pad, 0),
            min((((x1 - 1) << lvl) + pad + 1 + 15) & ~15, cam.width), min(((y1 - 1) << lvl) + pad + 1, cam.height))


def _samples_outside_tile(ev, pose, tile):
    """Valid samples of the oracle's evaluator at `pose` whose 4x4 footprint is not inside the staged tile."""
    from oracle import dpr_oracle
    xc = ev.x @ dpr_oracle.rodrigues(pose[:3]).T + pose[3:]
    z = np.where(xc[:, 2] > 1e-6, xc[:, 2], 1.0)
    x0 = np.floor((ev.fx * xc[:, 0] / z + ev.cx) * ev.scale)
    y0 = np.floor((ev.fy * xc[:, 1] / z + ev.cy) * ev.scale)
    ok = (xc[:, 2] > 1e-6) & (x0 >= 1) & (x0 <= ev.w - 3) & (y0 >= 1) & (y0 <= ev.h - 3)
    tx0, ty0, tw, th = tile
    inside = (x0 - 1 >= tx0) & (x0 + 3 <= tx0 + tw) & (y0 - 1 >= ty0) & (y0 + 3 <= ty0 + th)
    return int((ok & ~inside).sum())


def _roi_exits(ev, pose, roi):
    """Valid samples of the oracle's evaluator at `pose` whose 4x4 footprint leaves the planned ROI: the kernel reads them
    with the global-memory fetch and must report left_roi.  -> (active-sample indices, footprint x0).  Samples within
    1e-3 px of a pixel edge are left out (float32 projection may floor them the other way)."""
    from oracle import dpr_oracle
    xc = ev.x @ dpr_oracle.rodrigues(pose[:3]).T + pose[3:]
    z = np.where(xc[:, 2] > 1e-6, xc[:, 2], 1.0)
    ul, vl = (ev.fx * xc[:, 0] / z + ev.cx) * ev.scale, (ev.fy * xc[:, 1] / z + ev.cy) * ev.scale
    x0, y0 = np.floor(ul), np.floor(vl)
    clear = (np.minimum(ul - x0, x0 + 1 - ul) > 1e-3) & (np.minimum(vl - y0, y0 + 1 - vl) > 1e-3)
    ok = (xc[:, 2] > 1e-6) & (x0 >= 1) & (x0 <= ev.w - 3) & (y0 >= 1) & (y0 <= ev.h - 3) & clear
    rx0, ry0, rx1, ry1 = roi
    out = ok & ((x0 - 1 < rx0) | (y0 - 1 < ry0) | (x0 + 3 > rx1) | (y0 + 3 > ry1))
    return np.nonzero(out)[0], x0[out]


class CaseSet:
    """Frames of one camera rendered on the device, their starts, plans and oracle runs."""

    def __init__(self, ctx, cam_name, seed):
        from oracle import dpr_oracle
        self.ctx, self.cam_name = ctx, cam_name
        self.cam = cam = synth.CAMERA_1080P if cam_name == "1080p" else synth.CAMERA_VGA
        self.specs = _case_specs(cam_name)
        rng = np.random.default_rng(seed)
        truth, init = [], []
        for name, t, pin, _, _ in self.specs:
            pose = synth.random_pose(rng)
            if t is not None:
                pose[6 - len(t):] = t
            truth.append(pose)
            starts = []
            for _, sr, st in STARTS:
                start = pose + np.concatenate([rng.normal(0, sr, 3), rng.normal(0, st, 3)])
                for k, v in pin.items():
                    start[k] = v
                starts.append(start)
            init.append(starts)
        self.truth, self.init = np.array(truth), np.array(init)          # [F, 6], [F, 3, 6]
        self.n = len(self.specs)
        self.src = ctx.alloc_pyramid(self.n, cam.width, cam.height, LEVELS)
        ctx.render(self.src, self.truth, np.arange(self.n) + seed)
        ctx.build_pyramid(self.src)
        ctx.sync()
        self.model = util.dpr_model()
        self.radius = float(np.linalg.norm(self.model.samples[:, :3].astype(np.float64), axis=1).max())
        self.levels = [[self.src.level(l)[b].cpu().numpy() for l in range(LEVELS)] for b in range(self.n)]
        self.plans = [[dpr_plan(cam, self.init[f, s, 3:], self.radius) for s in range(3)] for f in range(self.n)]
        self.oracle = [[dpr_oracle.refine(self.levels[f], self.model, cam.mtx, self.init[f, s]) for s in range(3)]
                       for f in range(self.n)]
        first = [[dpr_oracle.refine(self.levels[f], self.model, cam.mtx, self.init[f, s], max_evals=1) for s in range(3)]
                 for f in range(self.n)]
        self.start_cost = np.array([[r["cost"] for r in row] for row in first])
        self.start_n = np.array([[r["n_valid"] for r in row] for row in first])
        self.ev = [[dpr_oracle.Evaluator(self.levels[f], self.model, cam.mtx, self.init[f, s]) for s in range(3)]
                   for f in range(self.n)]
        self.outside_tile = [[_samples_outside_tile(self.ev[f][s], self.oracle[f][s]["pose"], self.plans[f][s][2])
                              for s in range(3)] for f in range(self.n)]

    def exits(self, f, s, pose):
        return _roi_exits(self.ev[f][s], pose, self.plans[f][s][1])

    def label(self, f, s):
        return f"{self.cam_name} frame {f} ({self.specs[f][0]}), {STARTS[s][0]} start"


# ------------------------------------------------------------------------------------------
# every form, on purpose
# ------------------------------------------------------------------------------------------
def _form_ranges(sm_count):
    """Job range of each form (refine_impl: the cluster doubles while jobs * 2 * cluster <= 2 * SMs, up to 8)."""
    slots = 2 * sm_count
    return {1: (slots // 2 + 1, C1_TOP), 2: (slots // 4 + 1, slots // 2), 4: (slots // 8 + 1, slots // 4), 8: (1, slots // 8)}


def _ends(lo, hi, n_hyp):
    """The smallest and the largest job count of [lo, hi] that n_hyp divides."""
    return (lo + n_hyp - 1) // n_hyp * n_hyp, hi // n_hyp * n_hyp


def _run_form(cs, form, jobs, n_hyp, fused, seed, profile=False):
    """Refine the whole case set at `jobs` jobs per launch: the case frames at seeded positions of a batch of
    jobs / n_hyp frames, the rest masked, in as many launches as it takes.  -> outputs [F, 3] (numpy), launch-count
    increments, kernel names seen by the profiler, and whether every masked output kept its sentinel."""
    ctx, torch = cs.ctx, cs.ctx.torch
    b = jobs // n_hyp
    units = [(f, s) for f in range(cs.n) for s in range(3)] if n_hyp == 1 else [(f, None) for f in range(cs.n)]
    rng = np.random.default_rng(seed)
    res = {k: None for k in SENTINEL}
    res.update(pose=np.zeros((cs.n, 3, 6)), cost=np.zeros((cs.n, 3)), n_valid=np.zeros((cs.n, 3), np.int64),
               evals=np.zeros((cs.n, 3), np.int64), status=np.zeros((cs.n, 3), np.int64), left_roi=np.zeros((cs.n, 3), np.int64))
    redo_res = {k: np.zeros_like(v) for k, v in res.items()}
    best = np.full(cs.n, -1)
    launches, names, masked_ok = [], set(), True
    for c0 in range(0, len(units), b):
        chunk = units[c0:c0 + b]
        pos = np.sort(rng.choice(b, len(chunk), replace=False))
        pyr = ctx.alloc_pyramid(b, cs.cam.width, cs.cam.height, LEVELS)
        init = np.zeros((b, n_hyp, 6))
        mask = np.zeros(b, np.uint8)
        mask[pos] = 1
        src = torch.as_tensor([f for f, _ in chunk], device=ctx.tdev)
        dst = torch.as_tensor(pos, device=ctx.tdev)
        for l in range(LEVELS):
            if l == 0 or not fused:
                pyr.levels[l][dst] = cs.src.levels[l][src]
            else:
                pyr.levels[l].fill_(255)      # poison: a fused refinement that reads what it did not build goes visibly wrong
        for (f, s), p in zip(chunk, pos):
            init[p] = cs.init[f, s] if s is not None else cs.init[f]
        out = {k: torch.full(shape, v, dtype=dt, device=ctx.tdev) for k, v, shape, dt in (
            ("pose", SENTINEL["pose"], (b, n_hyp, 6), torch.float64), ("cost", SENTINEL["cost"], (b, n_hyp), torch.float32),
            ("n_valid", SENTINEL["n_valid"], (b, n_hyp), torch.int32), ("evals", SENTINEL["evals"], (b, n_hyp), torch.int32),
            ("status", SENTINEL["status"], (b, n_hyp), torch.uint8), ("left_roi", SENTINEL["left_roi"], (b, n_hyp), torch.uint8))}
        ctx.sync()
        n0 = ctx.launch_count()
        if profile:
            from torch.profiler import ProfilerActivity, profile as tprofile
            with tprofile(activities=[ProfilerActivity.CUDA]) as prof:
                ctx.refine(pyr, init, n_hyp, mask=mask, out=out, fused=fused)
                ctx.sync()
            names |= {e.name for e in prof.events() if "dpr_" in e.name}
            profile = False
        else:
            ctx.refine(pyr, init, n_hyp, mask=mask, out=out, fused=fused)
        launches.append(ctx.launch_count() - n0)
        skipped = torch.as_tensor(mask == 0, device=ctx.tdev)
        for k, v in out.items():
            masked_ok &= bool((v[skipped] == torch.tensor(SENTINEL[k], dtype=v.dtype, device=ctx.tdev)).all())
        o = {k: v.cpu().numpy() for k, v in out.items()}
        if n_hyp == 3:
            best[[f for f, _ in chunk]] = ctx.select_best(out)[0].cpu().numpy()[pos]
        if fused:
            # the exactness net: frames whose refinement left its ROI get the full pyramid and are refined again
            for l in range(1, LEVELS):
                pyr.levels[l].fill_(255)
            r2 = {k: v.cpu().numpy() for k, v in ctx.refine_fused(pyr, init, n_hyp, mask=mask).items() if k in SENTINEL}
        for (f, s), p in zip(chunk, pos):
            sl = slice(None) if s is None else s
            for k in SENTINEL:
                res[k][f, sl] = o[k][p] if s is None else o[k][p, 0]
                if fused:
                    redo_res[k][f, sl] = r2[k][p] if s is None else r2[k][p, 0]
        del pyr, out
    return {"out": res, "redo": redo_res if fused else None, "launches": launches, "names": names, "masked_ok": masked_ok,
            "best": best}


@pytest.fixture(scope="module")
def case_sets(ctx1080, ctxvga):
    return {"1080p": CaseSet(ctx1080, "1080p", 3100), "vga": CaseSet(ctxvga, "vga", 3200)}


@pytest.fixture(scope="module")
def form_runs(case_sets):
    """(camera, form, end, n_hyp, fused) -> _run_form result; end 0 / 1: the low / high end of the form's job range."""
    import torch
    ranges = _form_ranges(torch.cuda.get_device_properties(0).multi_processor_count)
    runs = {}
    for cam_name, cs in case_sets.items():
        for form in FORMS:
            for n_hyp in (1, 3):
                for end, jobs in enumerate(_ends(*ranges[form], n_hyp)):
                    for fused in (False, True):
                        seed = 7000 + 100 * form + 10 * end + n_hyp
                        runs[cam_name, form, end, n_hyp, fused] = _run_form(
                            cs, form, jobs, n_hyp, fused, seed, profile=(n_hyp == 1 and not fused))
                        runs[cam_name, form, end, n_hyp, fused]["jobs"] = jobs
        torch.cuda.empty_cache()
    return runs


# ------------------------------------------------------------------------------------------
# the assertions
# ------------------------------------------------------------------------------------------
def test_case_set_hits_its_targets(case_sets):
    """Each special case reaches what it is aimed at, by the numpy restatement of the plan, which in turn agrees with the
    device's own plan (agt_dpr_rects)."""
    for cam_name, cs in case_sets.items():
        for s in range(3):
            rects = cs.ctx.dpr_rects(cs.src, np.ascontiguousarray(cs.init[:, s:s + 1]), 1).cpu().numpy()
            for f in range(cs.n):
                assert tuple(rects[f]) == _rect_l0(cs.cam, cs.plans[f][s]), (cs.label(f, s), rects[f], cs.plans[f][s])
                assert cs.plans[f][s][0] == cs.oracle[f][s]["level"], cs.label(f, s)
        n_valid = cs.start_n
        n_active = np.array([[int(r["active"].sum()) * synth.MODEL_GRID ** 2 for r in row] for row in cs.oracle])
        for f, (name, _, _, lvl, aim) in enumerate(cs.specs):
            for s in range(3):
                lv, (x0, y0, x1, y1), (_, _, tw, th) = cs.plans[f][s]
                if lvl is not None:
                    assert lv == lvl, (cs.label(f, s), lv)
                if aim == "cut":
                    assert tw < x1 - x0 or th < y1 - y0, (cs.label(f, s), cs.plans[f][s])
                if aim in ("border", "sliver"):
                    assert n_valid[f, s] < n_active[f, s], cs.label(f, s)
                if aim == "sliver":
                    assert 0 < n_valid[f, s] <= 0.25 * n_active[f, s], (cs.label(f, s), n_valid[f, s], n_active[f, s])
            if aim == "exit":
                j, x0 = cs.exits(f, 0, cs.oracle[f][0]["pose"])
                assert len(j) > 0, cs.label(f, 0)
                print(f"{cs.label(f, 0)}: {len(j)} samples outside the ROI at the oracle's answer, in rank "
                      f"{sorted(set((j // 256 % 2).tolist()))} of 2 / {sorted(set((j // 256 % 4).tolist()))} of 4, "
                      f"{int((x0 == cs.ev[f][0].w - 3).sum())} on the last valid column")
        levels = {p[0] for row in cs.plans for p in row}
        assert levels == {0, 1, 2, 3}, (cam_name, levels)
        capped = [(f, s) for f in range(cs.n) for s in range(3) if cs.oracle[f][s]["status"] == ST_MAX_EVALS]
        late = [(f, s) for f in range(cs.n) for s in range(3)
                if cs.oracle[f][s]["status"] == ST_CONVERGED and not _at_fixed_point(cs.oracle[f][s])]
        outside = sum(1 for row in cs.outside_tile for v in row if v > 0)
        print(f"{cam_name}: {cs.n} frames x 3 starts; oracle at the evaluation cap: {len(capped)} "
              f"({', '.join(cs.label(f, s) for f, s in capped)}); converged after more than {MAX_EVALS - EVAL_MARGIN} evaluations: "
              f"{', '.join(f'{cs.label(f, s)} ({cs.oracle[f][s]['evals']})' for f, s in late) or 'none'}; "
              f"runs reading samples outside their tile: {outside}")


def test_every_form_ran(form_runs):
    """The form of each run is the one it was aimed at: its launch count (setup + refinement for one CTA per pose, one
    cluster launch otherwise) and, where the profiler sees kernels, the kernel's name."""
    names_seen = set()
    for (cam_name, form, end, n_hyp, fused), r in form_runs.items():
        want = 2 if form == 1 else 1
        assert all(n == want for n in r["launches"]), (cam_name, form, end, n_hyp, fused, r["launches"])
        for name in r["names"]:
            if "dpr_kernel<" in name:
                names_seen.add(name[name.index("dpr_kernel<"):name.index(">") + 1])
                assert f"dpr_kernel<{form}>" in name, (cam_name, form, end, r["names"])
        if r["names"] and form == 1:
            assert any("dpr_prep_kernel" in n for n in r["names"]), r["names"]
    print("kernels in the profiler trace:", sorted(names_seen) if names_seen else "none (no CUDA activity recorded)")
    print("job counts per launch:", sorted({(k[1], k[3], r["jobs"]) for k, r in form_runs.items()}))
    if names_seen:
        assert names_seen == {f"dpr_kernel<{c}>" for c in FORMS}, names_seen


def _stats(form_runs, case_sets):
    """Per camera and form: worst difference to the oracle on converged runs."""
    rows = {}
    for (cam_name, form, end, n_hyp, fused), r in form_runs.items():
        cs = case_sets[cam_name]
        o = r["redo"] if fused else r["out"]
        st = rows.setdefault((cam_name, form), {"rot": 0.0, "trans": 0.0, "cost": 0.0, "n": 0, "status_eq": 0, "not_conv": 0})
        for f in range(cs.n):
            for s in range(3):
                ref = cs.oracle[f][s]
                if not _at_fixed_point(ref):
                    st["not_conv"] += 1
                    st["status_eq"] += int(o["status"][f, s] == ref["status"])
                    continue
                dr, dt = util.pose_diff(o["pose"][f, s], ref["pose"])
                st["rot"], st["trans"] = max(st["rot"], dr), max(st["trans"], dt)
                st["cost"] = max(st["cost"], abs(o["cost"][f, s] - ref["cost"]) / ref["cost"])
                st["n"] += 1
    return rows


def test_forms_match_oracle(form_runs, case_sets):
    failures, late, late_n = [], {}, {}
    for (cam_name, form, end, n_hyp, fused), r in form_runs.items():
        cs = case_sets[cam_name]
        o = r["redo"] if fused else r["out"]        # (a fused run that left its ROI is only exact after the redo)
        for f in range(cs.n):
            for s in range(3):
                ref = cs.oracle[f][s]
                what = f"{cs.label(f, s)}, form {form} end {end} n_hyp {n_hyp} fused {fused}"
                dr, dt = util.pose_diff(o["pose"][f, s], ref["pose"])
                if ref["status"] == ST_CONVERGED and not _at_fixed_point(ref):
                    late[what] = (ref["evals"], int(o["status"][f, s]), int(o["evals"][f, s]), dr, dt)
                    late_n[what] = ref["n_valid"]
                    if (o["status"][f, s] == ST_CONVERGED and ref["n_valid"] >= MIN_SAMPLES_LATE
                            and (dr > util.ROT_TOL or dt > util.TRANS_TOL)):
                        failures.append(f"{what} (late): {dr:.2e} rad, {dt:.2e} m")
                if not _at_fixed_point(ref):
                    continue            # not at a fixed point: float32 projection may take the trajectory elsewhere
                if (o["n_valid"][f, s] != ref["n_valid"] or o["status"][f, s] != ref["status"] or dr > util.ROT_TOL
                        or dt > util.TRANS_TOL or abs(o["cost"][f, s] - ref["cost"]) > 1e-3 * ref["cost"]):
                    failures.append(f"{what}: n_valid {o['n_valid'][f, s]} / {ref['n_valid']}, status {o['status'][f, s]} / "
                                    f"{ref['status']}, {dr:.2e} rad, {dt:.2e} m, cost {o['cost'][f, s]:.6g} / {ref['cost']:.6g}")
    for (cam_name, form), st in sorted(_stats(form_runs, case_sets).items()):
        print(f"{cam_name} dpr_kernel<{form}> vs oracle: {st['n']} converged runs, worst {st['rot']:.2e} rad {st['trans']:.2e} m, "
              f"cost {st['cost']:.1e} relative; runs not at a fixed point in the oracle {st['not_conv']} (cap, or converged after "
              f"more than {MAX_EVALS - EVAL_MARGIN} evaluations), kernel status equal on {st['status_eq']}")
    seen = set()
    for what, (ev_ref, st, ev, dr, dt) in late.items():
        key = what.split(", form")[0] + f" form {what.split('form ')[1].split()[0]}"
        if key not in seen:
            seen.add(key)
            print(f"converged late in the oracle ({ev_ref} evaluations, {late_n[what]} valid samples): {key}: kernel status {st} "
                  f"after {ev}, {dr:.2e} rad {dt:.2e} m")
    assert not failures, "\n".join(failures[:20])


def test_left_roi_reports_every_exit(form_runs, case_sets):
    """left_roi against an independent count: a run whose answer has samples outside the planned ROI read them at its last
    evaluation, so left_roi must be set, by every form (the cluster forms OR it over their ranks)."""
    failures, n_exit = [], {}
    for (cam_name, form, end, n_hyp, fused), r in form_runs.items():
        cs = case_sets[cam_name]
        for o in (r["out"], r["redo"]) if fused else (r["out"],):
            for f in range(cs.n):
                for s in range(3):
                    if o["n_valid"][f, s] > 0 and len(cs.exits(f, s, o["pose"][f, s])[0]) > 0:
                        n_exit[cam_name, form] = n_exit.get((cam_name, form), 0) + 1
                        if o["left_roi"][f, s] != 1:
                            failures.append(f"{cs.label(f, s)}, form {form} end {end} n_hyp {n_hyp} fused {fused}: "
                                            f"{len(cs.exits(f, s, o['pose'][f, s])[0])} samples outside the ROI, left_roi 0")
    for (cam_name, form), n in sorted(n_exit.items()):
        n_set = sum(int((r["out"]["left_roi"] == 1).sum()) for k, r in form_runs.items() if k[0] == cam_name and k[1] == form)
        print(f"{cam_name} dpr_kernel<{form}>: left_roi set on {n_set} of {8 * 3 * case_sets[cam_name].n} runs; "
              f"{n} results with samples outside the ROI at the answer")
    assert not failures, "\n".join(failures[:20])


def test_multi_hypothesis_selection(form_runs, case_sets):
    from oracle import dpr_oracle
    for (cam_name, form, end, n_hyp, fused), r in form_runs.items():
        if n_hyp != 3:
            continue
        cs = case_sets[cam_name]
        for f in range(cs.n):
            want = dpr_oracle.select(cs.oracle[f])
            assert r["best"][f] == want, (cs.label(f, 0), form, end, fused, r["best"][f], want)


def test_masked_frames_untouched(form_runs):
    for key, r in form_runs.items():
        assert r["masked_ok"], key


def test_position_independent(form_runs):
    """The two ends of a form place the case frames at different positions of batches of different sizes."""
    for (cam_name, form, end, n_hyp, fused), r in form_runs.items():
        if end == 0:
            other = form_runs[cam_name, form, 1, n_hyp, fused]["out"]
            for k, v in r["out"].items():
                assert np.array_equal(v, other[k]), (cam_name, form, n_hyp, fused, k)


def test_fused_equals_unfused(form_runs):
    for (cam_name, form, end, n_hyp, fused), r in form_runs.items():
        if not fused:
            continue
        want, got = form_runs[cam_name, form, end, n_hyp, False]["out"], r["out"]
        inside = got["left_roi"] == 0
        assert np.array_equal(got["left_roi"], want["left_roi"]), (cam_name, form, end, n_hyp)
        for k in SENTINEL:
            assert np.array_equal(got[k][inside], want[k][inside]), (cam_name, form, end, n_hyp, k)
            assert np.array_equal(r["redo"][k], want[k]), (cam_name, form, end, n_hyp, k, "after the redo")


def test_forms_agree(form_runs, case_sets):
    """Across forms, on the runs the oracle brings to a fixed point (see EVAL_MARGIN): the same decisions, and poses within
    the bar of the scipy pin (1e-5 rad, 2 um); bits may differ (the sample partition changes the float32 partial sums).
    Runs that end at the evaluation cap are not at a fixed point, and the forms' trajectories part there as they part
    from the oracle's."""
    failures = []
    for cam_name, cs in case_sets.items():
        for n_hyp in (1, 3):
            base = form_runs[cam_name, 1, 0, n_hyp, False]["out"]
            for form in FORMS[1:]:
                o = form_runs[cam_name, form, 0, n_hyp, False]["out"]
                worst, same_evals, n_conv = np.zeros(2), 0, 0
                for f in range(cs.n):
                    for s in range(3):
                        same_evals += int(o["evals"][f, s] == base["evals"][f, s])
                        if not _at_fixed_point(cs.oracle[f][s]):
                            continue
                        n_conv += 1
                        for k in ("n_valid", "status", "left_roi"):
                            if o[k][f, s] != base[k][f, s]:
                                failures.append(f"{cs.label(f, s)}: {k} {o[k][f, s]} (form {form}) vs {base[k][f, s]} (form 1)")
                        d = util.pose_diff(o["pose"][f, s], base["pose"][f, s])
                        worst = np.maximum(worst, d)
                        if d[0] > 1e-5 or d[1] > 2e-6:
                            failures.append(f"{cs.label(f, s)}: form {form} is {d[0]:.2e} rad {d[1]:.2e} m from form 1")
                print(f"{cam_name} n_hyp {n_hyp} dpr_kernel<{form}> vs dpr_kernel<1>: {n_conv} converged runs, worst {worst[0]:.2e} rad "
                      f"{worst[1]:.2e} m; equal evaluation counts {same_evals}/{3 * cs.n}")
    assert not failures, "\n".join(failures[:30])


def test_cost_never_ends_above_its_start(form_runs, case_sets):
    for cam_name, cs in case_sets.items():
        for f in range(cs.n):
            for s in range(3):
                assert cs.oracle[f][s]["cost"] <= cs.start_cost[f, s], cs.label(f, s)
    worst = (0.0, None)
    for (cam_name, form, end, n_hyp, fused), r in form_runs.items():
        cs = case_sets[cam_name]
        cost = (r["redo"] if fused else r["out"])["cost"]
        ratio = np.where(cs.start_cost > 0, cost / np.maximum(cs.start_cost, 1e-30), 0.0)
        f, s = np.unravel_index(np.argmax(ratio), ratio.shape)
        if ratio[f, s] > worst[0]:
            worst = (float(ratio[f, s]), f"{cs.label(f, s)}, form {form}, status {r['out']['status'][f, s]}")
        bad = np.argwhere(cost > cs.start_cost * (1 + 1e-6))
        assert len(bad) == 0, [(cs.label(f, s), form, cost[f, s], cs.start_cost[f, s]) for f, s in bad]
    print(f"highest final / starting cost: {worst[0]:.6f} ({worst[1]})")
