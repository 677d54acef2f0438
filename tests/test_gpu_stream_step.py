"""The stream step launch by launch.

  * agt_ape_update on scripted poses against ``ApeOracle.step_given`` (the reference's state machine, detect_pose.py:490-574),
    slot by slot of the state record, in every branch it has;
  * agt_ape_commit against agt_ape_update, bit for bit, with and without a refined pose and the hand-over of the corners;
  * agt_streams_front against its parts lk_merge -> ape_prepare -> pnp -> accept_gate, bit for bit;
  * BatchedPoseDetector.step (eager and from replayed graphs) against the same chain driven launch by launch;
  * agt_track_rects against a numpy restatement.

Equality owed: the fused launches inline the same device code as their parts, so they must equal them bit for bit.  Against the
oracle, slots that copy a pose handed in are exact, computed float64 slots agree to 1e-12 and the float32-rounded tvec of a
prediction is exact unless its float64 value lies within 1e-12 (relative) of a float32 rounding midpoint (counted and printed)."""
import math

import cv2
import numpy as np
import pytest

from accurate_aprilgroup_tracking_b200 import synth
from accurate_aprilgroup_tracking_b200._lib import AGT_STREAM_STATE_DOUBLES, DPR_NONE
from oracle import ape_oracle
from tests import util

pytestmark = pytest.mark.gpu

F64_TOL = 1e-12
NEAR_PI = 1e-6       # angles this close to pi: rotation vectors compared as rotations ...
NEAR_PI_TOL = 1e-7   # ... to what cv::Rodrigues resolves there (its angle is acos of the trace: steps of ~1.5e-8 rad near pi)
ERR_BELOW_2 = float(np.nextafter(np.float32(2.0), np.float32(0.0)))


def _rvec(rmat):
    return cv2.Rodrigues(np.asarray(rmat, dtype=np.float64))[0].ravel()


def _rmat(rvec):
    return cv2.Rodrigues(np.asarray(rvec, dtype=np.float64).reshape(3, 1))[0]


def _pose(rmat, t):
    return np.concatenate([_rvec(rmat), np.asarray(t, dtype=np.float64)])


def _random_rot(rng, scale=1.0):
    return _rmat(rng.normal(0.0, scale, 3))


def _bits(x):
    """float tensor / array -> integer view (bitwise comparison, NaN included)."""
    a = x.cpu().numpy() if hasattr(x, "cpu") else np.asarray(x)
    a = np.ascontiguousarray(a)
    return a.view({8: np.int64, 4: np.int32, 2: np.int16, 1: np.uint8}[a.dtype.itemsize])


# ------------------------------------------------------------------------------------------
# scripted scenarios: per stream a list of frames (n_tags, pose (6,), ok, err)
# ------------------------------------------------------------------------------------------
def _accelerating(rng, n_frames, dr=0.05, dt=5e-3):
    """Poses whose rotational and translational velocities change by ~dr rad and ~dt m every frame."""
    rot, t = _random_rot(rng, 0.6), np.array([rng.uniform(-0.05, 0.05), rng.uniform(-0.03, 0.03), rng.uniform(0.3, 0.5)])
    w, v = rng.normal(0, 0.03, 3), rng.normal(0, 3e-3, 3)
    out = []
    for _ in range(n_frames):
        out.append(_pose(rot, t))
        w, v = w + rng.normal(0, dr, 3), v + rng.normal(0, dt, 3)
        rot, t = rot @ _rmat(w), t + v
    return out


def _gimbal(rng, sign):
    """Three poses whose rotational acceleration rv_new^T rv_old has a pitch of sign * pi/2 (the Euler gimbal branch)."""
    r1 = _random_rot(rng, 0.6)
    rv_old = _random_rot(rng, 0.3)
    racc = _rmat([0.0, sign * math.pi / 2, 0.0]) @ _rmat([0.4, 0.0, 0.0])
    rv_new = rv_old @ racc.T
    r0 = r1 @ rv_old
    r2 = r1 @ rv_new.T
    t = [np.array([0.01, -0.02, 0.4]), np.array([0.013, -0.018, 0.41]), np.array([0.021, -0.019, 0.43])]
    return [_pose(r0, t[0]), _pose(r1, t[1]), _pose(r2, t[2])]


def _near_pi(rng, eps):
    """Three poses at a constant angular velocity whose prediction (R2^T R1 R1) is a rotation of pi - eps."""
    axis = np.array([0.48, -0.6, 0.64])
    rstar = _rmat(axis / np.linalg.norm(axis) * (math.pi - eps))
    r1 = _random_rot(rng, 0.5)
    r2 = r1 @ r1 @ rstar.T
    r0 = r1 @ r2.T @ r1
    t = [np.array([0.02, 0.01, 0.4]), np.array([0.024, 0.012, 0.405]), np.array([0.029, 0.015, 0.411])]
    return [_pose(r0, t[0]), _pose(r1, t[1]), _pose(r2, t[2])]


def _scenarios():
    rng = np.random.default_rng(20261022)
    ok = lambda p, err=0.5, n=3: (n, p, True, err)             # noqa: E731
    sc = {}
    sc["acceleration"] = (1, [[ok(p) for p in _accelerating(rng, 7)] for _ in range(5)])
    # same pose twice -> zero translation velocity (aliased guess); identity rotations -> exact zeros in the rotation velocity;
    # a rotation about z twice -> zeros in the rotation velocity; the same pose twice after a prediction (guess not aliased)
    p = _accelerating(rng, 5)
    ident = [_pose(np.eye(3), [0.01, 0.02, 0.4]), _pose(np.eye(3), [0.012, 0.021, 0.41]), _pose(np.eye(3), [0.015, 0.02, 0.43])]
    rz = [_pose(_rmat([0, 0, 0.3]), [0.01, 0.0, 0.4]), _pose(_rmat([0, 0, 0.35]), [0.012, 0.001, 0.41])] + [p[2], p[3]]
    p32 = [q.copy() for q in p]
    p32[3][3:] = p32[3][3:].astype(np.float32)             # float32-exact tvec: written unchanged into the float32 guess
    sc["zero_velocity"] = (1, [[ok(p[0]), ok(p[0]), ok(p[1]), ok(p[2])],
                               [ok(q) for q in ident] + [ok(p[4])],
                               [ok(q) for q in rz],
                               [ok(q) for q in p32[:4]] + [ok(p32[3]), ok(p32[4])]])
    sc["gimbal"] = (1, [[ok(q) for q in _gimbal(rng, 1.0)], [ok(q) for q in _gimbal(rng, -1.0)]])
    sc["near_pi"] = (1, [[ok(q) for q in _near_pi(rng, 1e-10)], [ok(q) for q in _near_pi(rng, 3e-11)]])
    p = _accelerating(rng, 5)
    sc["gate"] = (1, [[ok(p[0], ERR_BELOW_2), ok(p[1], 2.0), ok(p[2], ERR_BELOW_2), ok(p[3], ERR_BELOW_2), ok(p[4], 2.0)],
                      [ok(p[0], 2.0), ok(p[1], ERR_BELOW_2), ok(p[2], float("nan")), ok(p[3]), ok(p[4], 1e30)]])
    # ok = 0: PnP writes zeros (or what it returns) into the guess arrays, and through them into prev when they alias it
    p = _accelerating(rng, 6)
    z = np.zeros(6)
    sc["pnp_failed"] = (1, [[(3, z, False, 0.0), ok(p[0]), ok(p[1])],
                            [ok(p[0]), (3, z, False, 0.0), ok(p[1]), ok(p[2])],
                            [ok(p[0]), ok(p[1]), ok(p[2]), (3, p[3] + 1e-3 / 3, False, 0.0), ok(p[4]), ok(p[5])],
                            [ok(p[0]), ok(p[1]), ok(p[2]), (3, z, False, 0.0), ok(p[3]), ok(p[4])]])
    p = _accelerating(rng, 9)
    sc["n_tags"] = (1, [[ok(p[0], n=2), ok(p[1], n=0), ok(p[2], n=2), ok(p[3], n=2), ok(p[4], n=1), ok(p[5], n=2), ok(p[6], n=2),
                         ok(p[7], n=2), ok(p[8], n=2)],
                        [ok(q, n=[2, 2, 2, 1, 2, 2, 2, 0, 2][k]) for k, q in enumerate(p)]])
    sc["enhance_off"] = (0, [[ok(q) for q in _accelerating(rng, 5)] for _ in range(3)])
    p = _accelerating(rng, 6)
    nan = np.full(6, np.nan)
    half_nan = p[2].copy()
    half_nan[4] = np.nan
    sc["nan_pose"] = (1, [[ok(nan), ok(p[0]), ok(p[1]), ok(p[2]), ok(p[3])],
                          [ok(p[0]), ok(p[1]), ok(p[2]), ok(half_nan), ok(p[3]), ok(p[4]), ok(p[5])],
                          [ok(p[0]), ok(p[1]), (3, nan, False, 0.0), ok(p[2]), ok(p[3])]])
    return sc


def _frames(streams):
    """Pad every stream to the longest with n_tags = 0 frames -> per frame (n_tags [S], pose [S,6], ok [S], err [S])."""
    n = max(len(s) for s in streams)
    out = []
    for f in range(n):
        rows = [s[f] if f < len(s) else (0, np.zeros(6), False, 0.0) for s in streams]
        out.append((np.array([r[0] for r in rows], np.int32), np.array([r[1] for r in rows], np.float64),
                    np.array([r[2] for r in rows], np.uint8), np.array([r[3] for r in rows], np.float32)))
    return out


def _f32_midpoint(x):
    """x (float64) lies within 1e-12 (relative) of a point halfway between two float32 values."""
    f = np.float32(x)
    for nb in (np.nextafter(f, np.float32(np.inf)), np.nextafter(f, np.float32(-np.inf))):
        mid = 0.5 * (float(f) + float(nb))
        if abs(x - mid) <= 1e-12 * max(abs(x), 1e-300):
            return True
    return False


def _rot_close(a, b, tol):
    return util.rot_angle(a, b) <= tol


class _Counts(dict):
    def add(self, k, n=1):
        self[k] = self.get(k, 0) + int(n)


def _compare_to_oracle(got, orc, accepted, flag, err_flag_want, what, counts):
    """One stream's state record (float64 [64]) and decisions against the oracle after the same frame."""
    want = orc.state_record()
    assert bool(accepted) == orc.last_accepted, f"{what}: accepted"
    assert bool(flag) == err_flag_want, f"{what}: error flag"
    for k in (0, 7, 16):
        assert got[k] == want[k], f"{what}: slot {k} = {got[k]}, oracle {want[k]}"
    assert np.array_equal(got[1:7], want[1:7], equal_nan=True), f"{what}: prev {got[1:7]} vs {want[1:7]}"
    if want[7]:
        assert got[14] == want[14] and got[15] == want[15], f"{what}: alias / t32 {got[14:16]} vs {want[14:16]}"
        if orc.last_t64 is None:                              # the guess holds a pose handed in (possibly float32-rounded)
            assert np.array_equal(got[8:14], want[8:14], equal_nan=True), f"{what}: guess {got[8:14]} vs {want[8:14]}"
        else:                                                 # a prediction
            counts.add("t32 roundings", np.sum(np.float32(orc.last_t64).astype(np.float64) != orc.last_t64))
            ang = float(np.linalg.norm(want[8:11]))
            if np.all(np.isfinite(want[8:11])) and abs(ang - math.pi) < NEAR_PI:
                counts.add("near-pi predictions")
                assert _rot_close(got[8:11], want[8:11], NEAR_PI_TOL), f"{what}: guess rotation {got[8:11]} vs {want[8:11]}"
            else:
                assert np.allclose(got[8:11], want[8:11], rtol=F64_TOL, atol=F64_TOL, equal_nan=True), \
                    f"{what}: guess rvec {got[8:11]} vs {want[8:11]}"
            for k in range(3):
                if np.isfinite(orc.last_t64[k]) and _f32_midpoint(orc.last_t64[k]):
                    counts.add("rounding midpoints")
                    assert abs(got[11 + k] - want[11 + k]) <= abs(np.spacing(np.float32(want[11 + k]))), what
                else:
                    assert np.array_equal(got[11 + k:12 + k], want[11 + k:12 + k], equal_nan=True), \
                        f"{what}: guess tvec[{k}] {got[11 + k]!r} vs {want[11 + k]!r} (float64 {orc.last_t64[k]!r})"
    assert np.allclose(got[17:41], want[17:41], rtol=F64_TOL, atol=F64_TOL, equal_nan=True), \
        f"{what}: velocities differ by {np.nanmax(np.abs(got[17:41] - want[17:41]))}"
    assert got[41] == want[41], f"{what}: prev tvec float32 {got[41]} vs {want[41]}"
    assert not np.any(got[42:]), f"{what}: slots beyond 41"


def _branches(orc, counts):
    """Which branches of the predictor the oracle's state makes the next prediction take (after an accepted frame)."""
    if len(orc.rot_vel) < 2 or orc.last_t64 is None:
        return
    rv_new, rv_old = orc.rot_vel[1], orc.rot_vel[0]
    tacc = rv_new.T @ (orc.tran_vel[0] - orc.tran_vel[1])
    racc = rv_new.T @ rv_old
    counts.add("predictions")
    if np.all(np.isfinite(racc)):
        if math.sqrt(racc[0, 0] ** 2 + racc[1, 0] ** 2) < 1e-6:
            counts.add("gimbal")
        counts["max |0.5 tacc| m"] = max(counts.get("max |0.5 tacc| m", 0.0), float(np.linalg.norm(0.5 * tacc)))
        counts["max racc angle rad"] = max(counts.get("max racc angle rad", 0.0), float(np.linalg.norm(_rvec(racc))))


def _run_scenario(ctx, name, enhance, streams):
    torch = ctx.torch
    group = ape_oracle.group_from_json(synth.april_group_dict())
    orcs = [ape_oracle.ApeOracle(group, synth.CAMERA_VGA.mtx, None, bool(enhance)) for _ in streams]
    state = ctx.new_stream_state(len(streams))
    counts = _Counts()
    for f, (nt, pose, ok, err) in enumerate(_frames(streams)):
        acc, flag = ctx.ape_update(state, ctx._dev(nt, torch.int32), ctx._dev(pose, torch.float64), ctx._dev(ok, torch.uint8),
                                   ctx._dev(err, torch.float32), enhance_ape=bool(enhance))
        st, acc, flag = state.cpu().numpy(), acc.cpu().numpy(), flag.cpu().numpy()
        for s, orc in enumerate(orcs):
            flag_want = orc.step_given(int(nt[s]), pose[s], bool(ok[s]), float(err[s]))
            counts.add("accepted", orc.last_accepted)
            counts.add("error flags", flag_want)
            _compare_to_oracle(st[s], orc, acc[s], flag[s], flag_want, f"{name} frame {f} stream {s}", counts)
            if orc.last_accepted and not flag_want:
                _branches(orc, counts)
    return counts


def test_ape_update_matches_state_machine_on_scripted_poses(ctxvga):
    """agt_ape_update against ApeOracle.step_given, slot by slot, in every branch of the reference's state machine."""
    report = {}
    for name, (enhance, streams) in _scenarios().items():
        report[name] = _run_scenario(ctxvga, name, enhance, streams)
        print(f"ape_update {name}: " + ", ".join(f"{k} {v:.3g}" if isinstance(v, float) else f"{k} {v}" for k, v in report[name].items()))
    # every branch was taken where it was meant to be
    assert report["acceleration"]["max |0.5 tacc| m"] >= 100 * util.TRANS_TOL
    assert report["acceleration"]["max racc angle rad"] >= 100 * util.ROT_TOL
    assert report["acceleration"]["predictions"] >= 5 * 4
    assert report["zero_velocity"]["error flags"] >= 4
    assert report["gimbal"].get("gimbal", 0) == 2
    assert report["near_pi"].get("near-pi predictions", 0) == 2
    assert report["gate"]["accepted"] == 5
    assert report["enhance_off"].get("predictions", 0) == 0 and report["enhance_off"]["accepted"] == 15
    assert sum(r.get("t32 roundings", 0) for r in report.values()) >= 20


# ------------------------------------------------------------------------------------------
# agt_ape_commit == agt_ape_update (+ refined pose where status != 0, + hand-over), bit for bit
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("form", ["refined+handover", "refined", "handover", "plain"])
def test_ape_commit_equals_ape_update(ctxvga, form):
    torch = ctxvga.torch
    dev = ctxvga.tdev
    rng = np.random.default_rng(77)
    cases = [(name, enhance, streams) for name, (enhance, streams) in _scenarios().items()]
    for b in (13, 130):                                              # batches that are not a multiple of the 4 warps of a block
        cases.append((f"batch{b}", 1, [[(3 if rng.random() > 0.1 else 1, p, rng.random() > 0.05, float(rng.uniform(0, 2.4)))
                                        for p in _accelerating(rng, 6)] for _ in range(b)]))
    with_ref, with_hand = form.startswith("refined"), form.endswith("handover")
    n_pts = 48
    used = 0
    for name, enhance, streams in cases:
        s_n = len(streams)
        st_u, st_c = ctxvga.new_stream_state(s_n), ctxvga.new_stream_state(s_n)
        for f, (nt, pose, ok, err) in enumerate(_frames(streams)):
            nt_d, pose_d = ctxvga._dev(nt, torch.int32), ctxvga._dev(pose, torch.float64)
            ok_d, err_d = ctxvga._dev(ok, torch.uint8), ctxvga._dev(err, torch.float32)
            refined, pose_u = None, pose_d
            if with_ref:
                status = ((np.arange(s_n) + f) % 4).astype(np.uint8)          # DPR_NONE, DPR_CONVERGED, DPR_MAX_EVALS, DPR_LAMBDA
                rp = pose + np.concatenate([rng.normal(0, 1e-3, (s_n, 3)), rng.normal(0, 1e-4, (s_n, 3))], axis=1)
                refined = {"pose": ctxvga._dev(rp, torch.float64).reshape(s_n, 1, 6), "status": ctxvga._dev(status, torch.uint8).reshape(s_n, 1)}
                use = status != DPR_NONE
                pose_u = ctxvga._dev(np.where(use[:, None], rp, pose), torch.float64)
                used += int((use & (ok != 0) & (nt >= 2)).sum())
            img = valid = prev_pts = prev_valid = None
            if with_hand:
                img = torch.as_tensor(rng.normal(300, 100, (s_n, n_pts, 2)).astype(np.float32), device=dev)
                valid = torch.as_tensor((rng.random((s_n, n_pts)) > 0.3).astype(np.uint8), device=dev)
                prev_pts = torch.full((s_n, n_pts, 2), float("nan"), dtype=torch.float32, device=dev)
                prev_valid = torch.full((s_n, n_pts), 7, dtype=torch.uint8, device=dev)
            acc_u, flag_u = ctxvga.ape_update(st_u, nt_d, pose_u, ok_d, err_d, enhance_ape=bool(enhance))
            acc_c, flag_c, pose_out = ctxvga.ape_commit(st_c, nt_d, pose_d, ok_d, err_d, refined, img, valid, prev_pts, prev_valid,
                                                        enhance_ape=bool(enhance))
            what = f"{form} {name} frame {f}"
            assert np.array_equal(_bits(st_c), _bits(st_u)), what
            assert torch.equal(acc_c, acc_u) and torch.equal(flag_c, flag_u), what
            assert np.array_equal(_bits(pose_out), _bits(st_c[:, 1:7].contiguous())), what
            if with_hand:
                assert np.array_equal(_bits(prev_pts), _bits(img)), what
                want_valid = torch.where(acc_c[:, None] != 0, valid, torch.zeros_like(valid))
                assert torch.equal(prev_valid, want_valid), what
    if with_ref:
        print(f"ape_commit {form}: refined poses used by accepted-or-failed frames: {used}")
        assert used >= 100


# ------------------------------------------------------------------------------------------
# agt_streams_front == lk_merge -> ape_prepare -> pnp -> accept_gate, bit for bit
# ------------------------------------------------------------------------------------------
def _front_inputs(batch, seed, cam=synth.CAMERA_VGA):
    """Frames of ``batch`` streams with 0..3 detected tags, the corners LK tracked (some corners lost, some not tracked in the
    previous frame), NaN corners and frames on which PnP fails, and state records with and without a guess."""
    rng = np.random.default_rng(seed)
    obj = synth.object_points()
    n_pts = obj.shape[0]
    img = rng.normal(320, 200, (batch, n_pts, 2)).astype(np.float32)          # undetected slots hold garbage
    valid = np.zeros((batch, n_pts), np.uint8)
    tracked = np.zeros((batch, n_pts, 2), np.float32)
    status = np.zeros((batch, n_pts), np.uint8)
    prev_valid = np.zeros((batch, n_pts), np.uint8)
    n_in = np.zeros(batch, np.int32)
    state = np.zeros((batch, AGT_STREAM_STATE_DOUBLES))
    truth = np.array([synth.random_pose(rng) for _ in range(batch)])
    for b in range(batch):
        vis = synth.visible_tags(truth[b]).tolist()
        rng.shuffle(vis)
        n_det = min(int(rng.integers(0, 4)), len(vis))
        proj = synth.project(obj, truth[b], cam)
        tracked[b] = proj + rng.normal(0, 0.2, proj.shape)
        for k in vis:
            prev_valid[b, 4 * k:4 * k + 4] = 1
            status[b, 4 * k:4 * k + 4] = 1
        for k in vis[:n_det]:                                   # detected: their own corners, never overwritten by LK
            img[b, 4 * k:4 * k + 4] = proj[4 * k:4 * k + 4] + rng.normal(0, 0.1, (4, 2))
            valid[b, 4 * k:4 * k + 4] = 1
        n_in[b] = n_det
        if len(vis) > n_det + 1 and b % 3 == 0:
            k = vis[n_det]
            status[b, 4 * k + int(rng.integers(0, 4))] = 0              # one corner not tracked
        if len(vis) > n_det + 2 and b % 4 == 1:
            k = vis[n_det + 1]
            prev_valid[b, 4 * k + int(rng.integers(0, 4))] = 0          # one corner not in the previous accepted frame
        if b % 5 == 2:
            prev_valid[b] = 0                                           # nothing to re-admit: PnP on < 2 tags or fails
            status[b] = 0
        if b % 11 == 3 and n_det:
            img[b, 4 * vis[0] + 1, 0] = np.nan                          # NaN corner
        if b % 13 == 5:
            tracked[b] = np.nan                                         # NaN tracked corners (re-admitted as NaN)
        if b % 2 == 0:
            state[b, 7] = 1.0
            state[b, 8:14] = truth[b] + np.concatenate([rng.normal(0, 0.02, 3), rng.normal(0, 2e-3, 3)])
            if b % 17 == 6:
                state[b, 9] = np.nan                                    # a non-finite guess: PnP fails
    return dict(img=img, valid=valid, tracked=tracked, status=status, prev_valid=prev_valid, n_in=n_in, state=state,
                obj=obj.astype(np.float32))


@pytest.mark.parametrize("batch", [1, 7, 64, 1000])
def test_streams_front_equals_its_launches(ctxvga, batch):
    torch = ctxvga.torch
    checked = 0
    for seed, merge, enhance in ((batch, True, 1), (batch + 1, False, 1), (batch + 2, True, 0)):
        d = _front_inputs(batch, seed)
        dv = {k: ctxvga._dev(v, {np.float32: torch.float32, np.uint8: torch.uint8, np.int32: torch.int32,
                                  np.float64: torch.float64}[v.dtype.type]) for k, v in d.items()}
        img_f, valid_f = dv["img"].clone(), dv["valid"].clone()
        fr = ctxvga.streams_front(dv["obj"], dv["state"], enhance, img_f, valid_f, dv["n_in"],
                                  tracked=dv["tracked"] if merge else None, lk_status=dv["status"] if merge else None,
                                  prev_valid=dv["prev_valid"] if merge else None)
        img_c, valid_c, nt_c = dv["img"].clone(), dv["valid"].clone(), dv["n_in"].clone()
        tt_c = torch.full((batch,), -99, dtype=torch.int32, device=ctxvga.tdev)
        if merge:
            ctxvga.lk_merge(dv["tracked"], dv["status"], dv["prev_valid"], img_c, valid_c, nt_c, tt_c)
        guess, use = ctxvga.ape_prepare(dv["state"], bool(enhance))
        pose, ok, err, iters = ctxvga.pnp(dv["obj"], img_c, valid_c, guess, use)
        gate = ctxvga.accept_gate(ok, err, nt_c)
        what = f"batch {batch} seed {seed} merge {merge} enhance {enhance}"
        assert np.array_equal(_bits(fr["pose"]), _bits(pose)), what
        for k, v in (("ok", ok), ("iters", iters), ("n_tags", nt_c), ("gate", gate)):
            assert torch.equal(fr[k], v), f"{what}: {k}"
        assert np.array_equal(_bits(fr["err"]), _bits(err)), what
        assert not fr["status"].any(), what
        assert np.array_equal(_bits(img_f), _bits(img_c)) and torch.equal(valid_f, valid_c), what
        if merge:
            assert torch.equal(fr["tracked_tags"], tt_c), what
            # detected tags keep their corners; only fully tracked, fully valid tags of frames with < 2 detections come in
            v0 = d["valid"].reshape(batch, -1, 4).all(axis=2)
            full = (d["prev_valid"].reshape(batch, -1, 4) != 0).all(axis=2) & (d["status"].reshape(batch, -1, 4) == 1).all(axis=2)
            want = v0 | (full & (d["n_in"] < 2)[:, None])
            assert np.array_equal(valid_c.cpu().numpy().reshape(batch, -1, 4).all(axis=2), want), what
            assert np.array_equal(nt_c.cpu().numpy(), want.sum(axis=1)), what
            im = img_c.cpu().numpy()
            assert np.array_equal(_bits(im[np.repeat(v0, 4, axis=1)]), _bits(d["img"][np.repeat(v0, 4, axis=1)])), what
        else:
            assert torch.equal(fr["n_tags"], dv["n_in"]), what
        # sanity anchor: cv2.solvePnP on the merged point sets, at the pose tolerance of the suite
        okh, gh, poseh, useh = ok.cpu().numpy(), gate.cpu().numpy(), pose.cpu().numpy(), use.cpu().numpy()
        im, va, gs = img_c.cpu().numpy(), valid_c.cpu().numpy(), guess.cpu().numpy()
        cam = synth.CAMERA_VGA
        for b in range(min(batch, 64)):
            m = va[b] != 0
            if not gh[b] or not np.all(np.isfinite(im[b][m])):
                continue
            if useh[b]:
                r0, t0 = gs[b, :3].reshape(3, 1).copy(), gs[b, 3:].reshape(3, 1).copy()
                okr, r, t = cv2.solvePnP(d["obj"][m], im[b][m], cam.mtx, None, r0, t0, True, flags=cv2.SOLVEPNP_ITERATIVE)
            else:
                okr, r, t = cv2.solvePnP(d["obj"][m], im[b][m], cam.mtx, None, flags=cv2.SOLVEPNP_ITERATIVE)
            assert okr
            util.assert_pose_close(poseh[b], np.concatenate([r.ravel(), t.ravel()]), f"{what} stream {b}")
            checked += 1
        if merge:
            print(f"streams_front {what}: tags re-admitted {int(tt_c.sum())}, PnP failed {int((okh == 0).sum())}, "
                  f"gate open {int(gh.sum())}, guesses used {int(useh.sum())}")
    if batch >= 64:
        assert checked >= 20


# ------------------------------------------------------------------------------------------
# BatchedPoseDetector.step == the chain of its launches, eager and from replayed graphs
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("use_graphs", [False, True])
def test_captured_step_equals_its_launches(ctxvga, use_graphs):
    from accurate_aprilgroup_tracking_b200.batched import BatchedPoseDetector, pack_detections
    torch = ctxvga.torch
    cam = synth.CAMERA_VGA
    n_streams, n_frames = 8, 12
    trajs = [synth.trajectory(8300 + s, n_frames) for s in range(n_streams)]
    rngs = [np.random.default_rng(8300 + s) for s in range(n_streams)]
    obj = synth.object_points()
    bpd = BatchedPoseDetector(ctxvga, n_streams, cam.width, cam.height, obj, use_graphs=use_graphs)
    pyrs = [ctxvga.alloc_pyramid(n_streams, cam.width, cam.height, 4) for _ in range(2)]
    obj_d = ctxvga._dev(obj, torch.float32)
    state = ctxvga.new_stream_state(n_streams)
    prev_pts = torch.zeros((n_streams, obj.shape[0], 2), dtype=torch.float32, device=ctxvga.tdev)
    prev_valid = torch.zeros((n_streams, obj.shape[0]), dtype=torch.uint8, device=ctxvga.tdev)
    readmitted = used = 0
    for f in range(n_frames):
        poses = np.array([trajs[s][f] for s in range(n_streams)])
        seeds = np.arange(n_streams) + 100 * f
        ctxvga.render(bpd.pyr[bpd.cur], poses, seeds)
        cur, prv = pyrs[f % 2], pyrs[(f + 1) % 2]
        ctxvga.render(cur, poses, seeds)
        dets = []
        for s in range(n_streams):
            d = synth.detections(trajs[s][f], cam, rngs[s])
            if (f + s) % 5 == 3:
                d = d[:1]                                      # one tag left: LK carries the others
            if (f + 2 * s) % 9 == 4:
                d = []                                         # nothing detected
            dets.append(d)
        img, valid, ntags = pack_detections(dets)
        out = bpd.step(img, valid, ntags)
        got = {k: out[k].clone() for k in ("pose", "accepted", "tracked_tags")}
        got_state = bpd.state.clone()
        # the same frame launch by launch
        ctxvga.build_pyramid(cur)
        img_d, valid_d, nt_d = ctxvga._dev(img, torch.float32), ctxvga._dev(valid, torch.uint8), ctxvga._dev(ntags, torch.int32)
        nxt, st, _ = ctxvga.lk(prv if f else cur, cur, prev_pts, n_tags=nt_d)
        tt = torch.empty(n_streams, dtype=torch.int32, device=ctxvga.tdev)
        ctxvga.lk_merge(nxt, st, prev_valid, img_d, valid_d, nt_d, tt)
        guess, use = ctxvga.ape_prepare(state)
        pose, ok, err, _ = ctxvga.pnp(obj_d, img_d, valid_d, guess, use)
        gate = ctxvga.accept_gate(ok, err, nt_d)
        res = ctxvga.refine(cur, pose.reshape(n_streams, 1, 6), 1, mask=gate)
        refined = res["status"].reshape(-1) != 0
        pose_in = torch.where(refined[:, None], res["pose"].reshape(n_streams, 6), pose)
        acc, _ = ctxvga.ape_update(state, nt_d, pose_in, ok, err)
        prev_pts.copy_(img_d)
        prev_valid.copy_(torch.where(acc[:, None] != 0, valid_d, torch.zeros_like(valid_d)))
        what = f"graphs {use_graphs} frame {f}"
        assert np.array_equal(_bits(got_state), _bits(state)), what
        assert np.array_equal(_bits(got["pose"]), _bits(state[:, 1:7].contiguous())), what
        assert torch.equal(got["accepted"], acc), what
        assert torch.equal(got["tracked_tags"], tt), what
        assert torch.equal(bpd.prev_pts, prev_pts) and torch.equal(bpd.prev_valid, prev_valid), what
        readmitted += int(tt.sum())
        used += int(refined.sum())
    print(f"captured step (graphs {use_graphs}): {n_frames} frames x {n_streams} streams, tags re-admitted {readmitted}, "
          f"refined poses used {used}")
    assert readmitted >= 5 and used >= n_frames * n_streams // 2


# ------------------------------------------------------------------------------------------
# agt_track_rects against a numpy restatement
# ------------------------------------------------------------------------------------------
def _track_rect_np(s, cam, radius, margin, w, h):
    """-> ((x0, y0, x1, y1), ambiguous): ambiguous where a float64 extent lies within 1e-9 of an integer."""
    t = s[8 + 3:8 + 6] if s[7] != 0 else (s[1 + 3:1 + 6] if s[0] != 0 else None)
    if t is None or not t[2] > 1e-6 or math.isnan(t[0]) or math.isnan(t[1]):
        return (0, 0, 0, 0), False
    ext = []
    for a in range(2):
        c, f, pp = t[a], (cam.fx, cam.fy)[a], (cam.cx, cam.cy)[a]
        sb = min(radius / math.sqrt(c * c + t[2] * t[2]), 0.95)
        al, be = math.atan2(c, t[2]), math.asin(sb)
        ext += [f * math.tan(max(al - be, -1.5)) + pp - margin, f * math.tan(min(al + be, 1.5)) + pp + margin]
    amb = any(abs(e - round(e)) < 1e-9 for e in ext)
    x0, y0 = int(max(math.floor(ext[0]), 0)), int(max(math.floor(ext[2]), 0))
    x1, y1 = int(min(math.ceil(ext[1]) + 1, w)), int(min(math.ceil(ext[3]) + 1, h))
    return ((x0, y0, x1, y1) if x1 > x0 and y1 > y0 else (0, 0, 0, 0)), amb


def test_track_rects_match_restatement(ctx1080):
    cam = synth.CAMERA_1080P
    rng = np.random.default_rng(31)
    radius, margin = float(np.linalg.norm(synth.object_points(), axis=1).max()), 32
    rows, kinds = [], []

    def add(kind, prev=None, guess=None):
        s = np.zeros(AGT_STREAM_STATE_DOUBLES)
        if prev is not None:
            s[0], s[1:7] = 1.0, prev
        if guess is not None:
            s[7], s[8:14] = 1.0, guess
        rows.append(s)
        kinds.append(kind)

    for _ in range(40):
        add("guess over prev", prev=synth.random_pose(rng), guess=synth.random_pose(rng))
        add("prev only", prev=synth.random_pose(rng))
    add("neither")
    for tz in (1e-6, 0.0, -0.3, np.nan):
        add("t_z <= 1e-6", guess=np.array([0.1, 0.2, 0.3, 0.01, 0.02, tz]))
    add("NaN", guess=np.array([0, 0, 0, np.nan, 0.0, 0.4]))
    add("NaN", prev=np.array([0, 0, 0, 0.0, np.nan, 0.4]))
    add("NaN guess, prev set", prev=synth.random_pose(rng), guess=np.array([0, 0, 0, np.nan, 0.0, 0.4]))
    for tz in (0.04, 0.03, 0.02):
        add("0.95 cap", guess=np.array([0, 0, 0, 0.005, -0.003, tz]))
    for tx in (-2.0, 2.0, -0.8):
        add("1.5 rad clamp", prev=np.array([0, 0, 0, tx, 0.01, 0.1]))
    for tx, ty in ((-0.35, 0.0), (0.0, 0.2), (0.38, -0.2)):
        add("frame edge", prev=np.array([0, 0, 0, tx, ty, 0.5]))
    for tx, ty in ((3.0, 0.0), (0.0, -3.0)):
        add("empty", guess=np.array([0, 0, 0, tx, ty, 0.5]))
    state = ctx1080._dev(np.array(rows), ctx1080.torch.float64)
    got = ctx1080.track_rects(state, cam.width, cam.height, radius, margin).cpu().numpy()
    per_kind, ambiguous = {}, 0
    for s, kind, g in zip(rows, kinds, got):
        want, amb = _track_rect_np(s, cam, radius, margin, cam.width, cam.height)
        if amb:
            ambiguous += 1
            continue
        assert tuple(int(v) for v in g) == want, f"{kind}: {s[:14]} -> {g.tolist()} vs {want}"
        per_kind.setdefault(kind, []).append(want)
    print(f"track_rects: {len(rows)} states, {ambiguous} with an extent within 1e-9 of an integer (skipped)")
    # (a NaN guess is still the guess: prev does not stand in for it)
    assert all(r == (0, 0, 0, 0) for k in ("neither", "t_z <= 1e-6", "NaN", "NaN guess, prev set", "empty") for r in per_kind[k])
    assert all(r[0] == 0 or r[1] == 0 or r[2] == cam.width or r[3] == cam.height for r in per_kind["frame edge"])
    assert len(per_kind["guess over prev"]) >= 35 and any(r != (0, 0, 0, 0) for r in per_kind["0.95 cap"] + per_kind["1.5 rad clamp"])
