"""Covariance of a refined pose (agt_pose_covariance, csrc/agt_dpr.cu:pose_cov_kernel) against oracle/dpr_cov_oracle.py,
in its launch forms, in the batched pipeline and in the drop-in class."""
import ctypes as C
import sys
from pathlib import Path

import numpy as np
import pytest

from accurate_aprilgroup_tracking_b200 import _lib, synth
from tests import util
from tests.test_gpu_dropin import _Det, _logger, detector_factory, host  # noqa: F401  (fixtures)

pytestmark = pytest.mark.gpu

BAND = (0.15, 5.0)          # eigenvalues of the scatter against sigma_noise^2 H^-1 (tests/test_cpu_pose_cov.py)


def _render(ctx, cam, poses, seeds):
    pyr = ctx.alloc_pyramid(len(poses), cam.width, cam.height, 4)
    ctx.render(pyr, poses, seeds)
    ctx.build_pyramid(pyr)
    return pyr


def _case(ctx, cam, n, seed, sig_r, sig_t, n_hyp):
    """The DPR parity cases (tests/test_gpu_kernels.py:_dpr_case): n noisy renders, n_hyp starts each, refined on the device."""
    rng = np.random.default_rng(seed)
    truth = np.array([synth.random_pose(rng) for _ in range(n)])
    pyr = _render(ctx, cam, truth, np.arange(n) + seed)
    init = truth[:, None, :] + np.concatenate([rng.normal(0, sig_r, (n, n_hyp, 3)), rng.normal(0, sig_t, (n, n_hyp, 3))], axis=2)
    res = ctx.refine(pyr, init, n_hyp)
    return pyr, init, res


def _whitened(a, b):
    """|| L^-1 (a - b) L^-T ||_2 with L = chol(b)."""
    low = np.linalg.cholesky(b)
    m = np.linalg.solve(low, np.linalg.solve(low, (a - b).T).T)
    return float(np.linalg.norm(m, 2))


@pytest.mark.parametrize("n_hyp", [1, 3])
@pytest.mark.parametrize("cam_name", ["1080p", "vga"])
def test_covariance_matches_oracle(ctx1080, ctxvga, cam_name, n_hyp):
    from oracle import dpr_cov_oracle
    ctx, cam = (ctx1080, synth.CAMERA_1080P) if cam_name == "1080p" else (ctxvga, synth.CAMERA_VGA)
    n, seed, sr, st = (24, 2000, 0.01, 0.0005) if cam_name == "1080p" else (12, 2100, 0.005, 0.0003)
    pyr, init, res = _case(ctx, cam, n, seed, sr, st, n_hyp)
    cov = {k: v.cpu().numpy() for k, v in ctx.pose_covariance(pyr, init, res["pose"], n_hyp).items()}
    pose = res["pose"].cpu().numpy()
    model = util.dpr_model()
    worst = np.zeros(3)
    for b in range(n):
        levels = [pyr.level(l)[b].cpu().numpy() for l in range(4)]
        for h in range(n_hyp):
            ref = dpr_cov_oracle.covariance(levels, model, cam.mtx, init[b, h], pose[b, h])
            what = f"{cam_name} frame {b} hypothesis {h}"
            assert int(cov["n_valid"][b, h]) == ref["n"], what
            assert bool(cov["ok"][b, h]) == ref["ok"], what
            if not ref["ok"]:
                assert np.isnan(cov["cov"][b, h]).all()
                continue
            c_gpu = 0.5 * float(cov["sigma2"][b, h]) * (ref["n"] - 6)
            e = [abs(c_gpu - ref["c"]) / ref["c"], _whitened(cov["cov"][b, h], ref["cov"]), _whitened(cov["info"][b, h], ref["H"])]
            worst = np.maximum(worst, e)
            assert e[0] <= 1e-4 and e[1] <= 1e-3 and e[2] <= 1e-3, (what, e)
            assert np.array_equal(cov["cov"][b, h], cov["cov"][b, h].T)
    print(f"{cam_name} x{n_hyp}: worst relative c {worst[0]:.2e}, whitened Sigma {worst[1]:.2e}, whitened H {worst[2]:.2e}")


def test_launch_forms_are_bit_identical(ctx1080):
    """Full pyramid vs ROI pyramid vs fused refinement (frames with left_roi = 0), a frame at two batch positions, and
    masked frames whose outputs keep what was there."""
    torch = ctx1080.torch
    cam = synth.CAMERA_1080P
    n = 20
    rng = np.random.default_rng(2500)
    truth = np.array([synth.random_pose(rng) for _ in range(n)])
    truth[0, 3:] = (0.16, 0.09, 0.27)           # cut by the image corner
    init = (truth + np.concatenate([rng.normal(0, 0.01, (n, 3)), rng.normal(0, 0.0005, (n, 3))], axis=1)).reshape(n, 1, 6)
    init[2, 0, 3] += 0.010                      # leaves its ROI: redone on the full pyramid
    full = _render(ctx1080, cam, truth, np.arange(n) + 2500)
    res = ctx1080.refine(full, init, 1)
    want = ctx1080.pose_covariance(full, init, res["pose"])
    for form in ("roi", "fused"):
        pyr = ctx1080.alloc_pyramid(n, cam.width, cam.height, 4)
        pyr.levels[0].copy_(full.levels[0])
        for l in (1, 2, 3):
            pyr.levels[l].fill_(255)            # poison: what the ROI / fused pyramid does not build stays visibly wrong
        got_ref = ctx1080.refine_roi(pyr, init, 1) if form == "roi" else ctx1080.refine_fused(pyr, init, 1)
        assert torch.equal(got_ref["pose"], res["pose"])
        redo = got_ref["redo"].cpu().numpy()
        assert redo[2] == 1
        # the kernel on the pyramid as the refinement left it: frames redone on a full pyramid are exact as well, the
        # others because their refinement stayed inside the region it built
        got = ctx1080.pose_covariance(pyr, init, res["pose"])
        for k in want:
            assert torch.equal(got[k], want[k]), (form, k)
    # one frame at two batch positions of a larger batch, the rest masked with sentinels in their outputs
    b = 8
    pyr = ctx1080.alloc_pyramid(b, cam.width, cam.height, 4)
    for l in range(4):
        pyr.levels[l][1] = full.levels[l][5]
        pyr.levels[l][6] = full.levels[l][5]
    ini = np.zeros((b, 1, 6)); ini[:, 0, 5] = 0.3
    ps = torch.zeros((b, 1, 6), dtype=torch.float64, device=ctx1080.tdev); ps[:, 0, 5] = 0.3
    ini[1] = ini[6] = init[5]
    ps[1] = ps[6] = res["pose"][5]
    mask = np.zeros(b, np.uint8); mask[[1, 6]] = 1
    sentinel = {"cov": -7.25, "info": -3.5, "sigma2": -1.5, "n_valid": -11, "ok": 201}
    out = {k: torch.full_like(v[:1].expand(b, *v.shape[1:]).contiguous(), s) for (k, v), s in zip(want.items(), sentinel.values())}
    ctx1080.pose_covariance(pyr, ini, ps, mask=mask, out=out)
    for k, v in out.items():
        assert torch.equal(v[1], want[k][5]) and torch.equal(v[6], want[k][5]), k
        skipped = torch.as_tensor(mask == 0, device=ctx1080.tdev)
        assert bool((v[skipped] == torch.tensor(sentinel[k], dtype=v.dtype, device=ctx1080.tdev)).all()), k


def test_statistics_on_the_device(ctx1080):
    """256 noise seeds at two 1080p poses (agt_render), refined and evaluated on the device: the seed-to-seed scatter of the
    refined pose against sigma_level^2 H^-1 (the pixel noise at the pyramid level the refinement reads), same band as the CPU
    calibration."""
    from scipy.linalg import eigh
    from oracle import dpr_cov_oracle, dpr_oracle
    cam = synth.CAMERA_1080P
    rng = np.random.default_rng(7300)
    n = 256
    for k in range(2):
        truth = synth.random_pose(rng)
        pyr = _render(ctx1080, cam, np.repeat(truth[None], n, axis=0), np.arange(n) + 40000 + 1000 * k)
        # one start for every seed: it fixes the cost function (oracle/dpr_cov_oracle.py:calibration)
        start = truth + np.concatenate([rng.normal(0, 0.01, 3), rng.normal(0, 0.0005, 3)])
        init = np.repeat(start[None, None], n, axis=0)
        res = ctx1080.refine(pyr, init, 1)
        cov = ctx1080.pose_covariance(pyr, init, res["pose"])
        assert bool(cov["ok"].all())
        pose = res["pose"].cpu().numpy().reshape(n, 6)
        offs = np.array([dpr_cov_oracle.tangent_offset(p, truth) for p in pose])
        scatter = np.cov(offs.T)
        level = dpr_oracle.select_level(cam.fx, synth.model_pitch(), start[5], 4)
        predicted = dpr_cov_oracle.level_noise_var(level, synth.NOISE_SIGMA) * np.linalg.inv(cov["info"].cpu().numpy().reshape(n, 6, 6).mean(axis=0))
        eig = eigh(scatter, predicted, eigvals_only=True)
        print(f"pose {k} z={truth[5]:.3f} level {level}: eigenvalues of the scatter against sigma_level^2 H^-1 {np.round(eig, 3)}, "
              f"residual sigma {np.sqrt(cov['sigma2'].cpu().numpy()).mean():.1f}")
        assert BAND[0] <= eig.min() and eig.max() <= BAND[1], eig


def _stream_run(ctx, use_graphs, pose_covariance, n_streams=64, n_frames=16):
    """64 streams x 16 1080p frames through BatchedPoseDetector.  With pose_covariance, every step's covariance is also
    recomputed by a standalone call on the inputs the step's launch read (its pyramid, the PnP pose, the refined pose and
    the gate: static buffers of the step, or of the slot's graph)."""
    from accurate_aprilgroup_tracking_b200.batched import BatchedPoseDetector, pack_detections
    cam = synth.CAMERA_1080P
    real = ctx.pose_covariance
    calls = {}

    def spy(pyr, init, pose, n_hyp=1, mask=None, out=None):
        calls[id(pyr)] = (pyr, init, pose, mask)
        return real(pyr, init, pose, n_hyp, mask=mask, out=out)
    if pose_covariance:
        ctx.pose_covariance = spy
    try:
        bpd = BatchedPoseDetector(ctx, n_streams, cam.width, cam.height, synth.object_points(), use_graphs=use_graphs,
                                  pose_covariance=pose_covariance)
        trajs = [synth.trajectory(9100 + s, n_frames) for s in range(n_streams)]
        rngs = [np.random.default_rng(9100 + s) for s in range(n_streams)]
        steps = []
        for f in range(n_frames):
            poses = np.array([trajs[s][f] for s in range(n_streams)])
            ctx.render(bpd.pyr[bpd.cur], poses, np.arange(n_streams) + 100 * f)
            dets = [synth.detections(trajs[s][f], cam, rngs[s]) for s in range(n_streams)]
            if f == 5:
                dets[3] = dets[3][:1]
            slot_pyr = bpd.pyr[bpd.cur]
            out = bpd.step(*pack_detections(dets))
            rec = {"pose": out["pose"].clone(), "accepted": out["accepted"].clone(),
                   "refine": {k: v.clone() for k, v in out["refine"].items()}, "kernels": bpd.kernels_per_step}
            if pose_covariance:
                rec["covariance"], rec["covariance_ok"] = out["covariance"].clone(), out["covariance_ok"].clone()
                pyr, init, pose, mask = calls[id(slot_pyr)]
                rec["standalone"] = {k: v.clone() for k, v in real(pyr, init, pose, 1, mask=mask).items()}
            steps.append(rec)
    finally:
        ctx.__dict__.pop("pose_covariance", None)
    return steps


@pytest.mark.parametrize("use_graphs", [False, True])
def test_pipeline_unchanged_and_covariance_matches_standalone(ctx1080, use_graphs):
    torch = ctx1080.torch
    base = _stream_run(ctx1080, use_graphs, False)
    cov = _stream_run(ctx1080, use_graphs, True)
    refined = 0
    for f, (a, b) in enumerate(zip(base, cov)):
        assert torch.equal(a["pose"], b["pose"]) and torch.equal(a["accepted"], b["accepted"]), f
        gate = b["refine"]["status"].reshape(-1) != 0
        assert torch.equal(a["refine"]["status"].reshape(-1) != 0, gate), f
        for k in ("pose", "cost", "n_valid", "evals", "status", "left_roi"):
            assert torch.equal(a["refine"][k][gate], b["refine"][k][gate]), (f, k)     # masked frames' outputs are not written
        assert b["kernels"] == a["kernels"] + 1
        st = b["standalone"]
        assert torch.equal(b["covariance"][gate], st["cov"].reshape(-1, 6, 6)[gate]), f
        assert torch.equal(b["covariance_ok"][gate], st["ok"].reshape(-1)[gate]), f
        assert not bool(b["covariance_ok"][~gate].any()), f
        refined += int(gate.sum())
    assert refined > 64 * 8


def test_dropin_pose_covariance(detector_factory, host, ctxvga):
    """PoseDetector(pose_covariance=True) decides and poses exactly as without it; self.pose_covariance equals
    HostContext.pose_covariance on the same gray frame."""
    stub_dir = str(Path(__file__).resolve().parent.parent / "oracle" / "apriltag_stub")
    sys.path.insert(0, stub_dir)
    try:
        import apriltag as stub
        cam = synth.CAMERA_VGA
        dets_on = [detector_factory(cam.mtx, use_lk=True, use_dense_refine=True, pose_covariance=flag) for flag in (False, True)]
        n = 8
        traj = synth.trajectory(4322, n)
        pyr = ctxvga.alloc_pyramid(n, cam.width, cam.height, 1)
        ctxvga.render(pyr, traj, np.arange(n) + 60)
        frames = pyr.frames.cpu().numpy()
        seen = 0
        for f in range(n):
            rng = np.random.default_rng(f)
            dets = synth.detections(traj[f], cam, rng)
            poses = []
            for det in dets_on:
                stub.push_detections(stub.Detection(t, c, 100.0) for t, c in dets)
                pnp = {}
                orig = det._refine_in_place

                def spy(tr, orig=orig, pnp=pnp):
                    pnp["init"] = np.concatenate([np.asarray(v, dtype=np.float64).reshape(3) for v in tr])
                    orig(tr)
                det._refine_in_place = spy
                det._detect_and_get_pose(np.repeat(frames[f][:, :, None], 3, axis=2))     # (it draws on the frame it is given)
                del det._refine_in_place
                poses.append((np.concatenate([det.prev_transform[0].ravel(), det.prev_transform[1].ravel()]), bool(det._prev_corners),
                              pnp.get("init")))
            assert np.array_equal(poses[0][0], poses[1][0]) and poses[0][1] == poses[1][1], f
            assert dets_on[0].pose_covariance is None
            if dets_on[1].pose_covariance is not None:
                seen += 1
                # the refined pose in float64 (prev_transform may hold the translation in the guess's float32)
                init = poses[1][2]
                ok, r, t, _, _ = host.refine_pose(dets_on[1]._gray, init[:3], init[3:], cam.mtx)
                want = host.pose_covariance(dets_on[1]._gray, init, np.concatenate([r.ravel(), t.ravel()]), cam.mtx)
                assert want["ok"][0, 0]
                assert np.array_equal(dets_on[1].pose_covariance, want["cov"][0, 0])
        assert seen >= n - 1
    finally:
        sys.path.remove(stub_dir)
        sys.modules.pop("apriltag", None)


def test_argument_errors(ctx1080):
    lib, torch = ctx1080.lib, ctx1080.torch
    cam = synth.CAMERA_1080P
    pyr = ctx1080.alloc_pyramid(2, cam.width, cam.height, 4)
    pyr.levels[0].fill_(128)
    ctx1080.build_pyramid(pyr)
    dev = ctx1080.tdev
    init = torch.zeros((2, 1, 6), dtype=torch.float64, device=dev); init[..., 5] = 0.3
    cov = torch.zeros((2, 1, 36), dtype=torch.float64, device=dev)
    ok = torch.zeros((2, 1), dtype=torch.uint8, device=dev)
    p = ctx1080._p
    args = lambda n_hyp, d_cov: (ctx1080.h, C.byref(pyr.desc), p(init), p(init), n_hyp, None, d_cov, None, None, None, p(ok), 2)
    assert lib.agt_pose_covariance(*args(0, p(cov))) == _lib.AGT_ERR_INVALID
    assert lib.agt_pose_covariance(*args(1, None)) == _lib.AGT_ERR_INVALID
    assert lib.agt_pose_covariance(*args(1, p(cov))) == _lib.AGT_OK
    with pytest.raises(ValueError):
        ctx1080.pose_covariance(pyr, init, init, n_hyp=0)
    with pytest.raises(ValueError):
        ctx1080.pose_covariance(pyr, np.zeros((3, 1, 6)), np.zeros((3, 1, 6)))       # 3 frames of poses, 2 in the pyramid
    # a flat grey frame: every sample valid but H singular -> ok = 0, Sigma NaN; a pose that sees nothing -> n = 0
    out = ctx1080.pose_covariance(pyr, init, init)
    assert int(out["n_valid"][0, 0]) > 6 and int(out["ok"][0, 0]) == 0 and bool(out["cov"][0, 0].isnan().all())
    far = init.clone(); far[..., 3] = 5.0
    out = ctx1080.pose_covariance(pyr, far, far)
    assert int(out["n_valid"][0, 0]) == 0 and int(out["ok"][0, 0]) == 0 and bool(out["cov"].isnan().all())
