"""CPU tests (no GPU): the oracle against the reference / OpenCV / scipy and the golden vectors."""
import numpy as np
import pytest

from accurate_aprilgroup_tracking_b200 import synth
from oracle import ape_oracle, dpr_oracle, lk_oracle, make_golden
from tests import util

GOLDEN = make_golden.GOLDEN


# ---------------------------------------------------------------------------- APE
def _run_ape_oracle(ids, corners, mtx):
    orc = ape_oracle.ApeOracle(ape_oracle.group_from_json(synth.april_group_dict()), mtx, None, True)
    snaps = []
    for f in range(ids.shape[0]):
        orc.step(make_golden.unpack_detections(ids, corners, f))
        snaps.append(orc.snapshot())
    return snaps


def test_ape_oracle_reproduces_reference_golden_bit_exact():
    g = np.load(GOLDEN / "ape_sequence.npz")
    snaps = _run_ape_oracle(g["ids"], g["corners"], g["mtx"])
    for f, s in enumerate(snaps):
        for key in ("prev", "guess"):
            want = g[key][f]
            if np.isnan(want[0]):
                assert s[key] is None, (f, key)
            else:
                assert s[key] is not None, (f, key)
                assert np.array_equal(np.concatenate(s[key]), want), (f, key)     # same OpenCV build -> identical bits
        assert s["n_vel"] == g["n_vel"][f]
    # the sequence exercises the reset paths: guess dropped at the loss frames and at the gate failure
    lost = np.nonzero(np.isnan(g["guess"][:, 0]))[0].tolist()
    assert lost == [30, 31, 50]


def test_ape_oracle_state_record_follows_the_golden_sequence():
    """state_record() (the device's layout) carries the same prev / guess / n_vel as the snapshots of the golden run."""
    g = np.load(GOLDEN / "ape_sequence.npz")
    orc = ape_oracle.ApeOracle(ape_oracle.group_from_json(synth.april_group_dict()), g["mtx"], None, True)
    for f in range(g["ids"].shape[0]):
        orc.step(make_golden.unpack_detections(g["ids"], g["corners"], f))
        s = orc.state_record()
        assert s.shape == (64,) and not s[42:].any()
        assert s[0] == (not np.isnan(g["prev"][f][0])) and s[7] == (not np.isnan(g["guess"][f][0])) and s[16] == g["n_vel"][f]
        if s[0]:
            assert np.array_equal(s[1:7], g["prev"][f])
        if s[7]:
            assert np.array_equal(s[8:14], g["guess"][f])
            assert s[15] == (orc.last_t64 is not None)    # a float32 tvec exactly when the guess is a prediction
            assert s[14] == (orc.last_t64 is None)        # otherwise the guess arrays are prev's


def test_ape_oracle_step_given_models_the_guess_write_and_the_raise():
    """step_given on poses it is handed: the write of solvePnP into the (aliased, float32) guess arrays, and the state the
    reference is left in when a zero velocity raises."""
    rng = np.random.default_rng(4)
    orc = ape_oracle.ApeOracle(ape_oracle.group_from_json(synth.april_group_dict()), synth.CAMERA_VGA.mtx, None, True)
    poses = [np.concatenate([rng.normal(0, 0.5, 3), [0.01 * k, -0.02, 0.4 + 0.01 * k * k]]) for k in range(5)]
    assert not orc.step_given(3, poses[0], True, 0.5)
    s = orc.state_record()
    assert s[0] == s[7] == s[14] == 1 and s[15] == 0 and np.array_equal(s[1:7], poses[0]) and np.array_equal(s[8:14], poses[0])
    # the same pose again: a zero translation velocity raises in the reference -> error flag, nothing appended
    assert orc.step_given(3, poses[0], True, 0.5) and orc.last_accepted and orc.state_record()[16] == 0
    # PnP fails: its zeros land in the guess arrays and, aliased, in prev
    assert not orc.step_given(3, np.zeros(6), False, 0.0) and not orc.last_accepted
    s = orc.state_record()
    assert not s[1:7].any() and not s[8:14].any() and s[14] == 1
    for k in (1, 2, 3):
        assert not orc.step_given(3, poses[k], True, 0.5)
    s = orc.state_record()
    assert s[16] == 2 and s[14] == 0 and s[15] == 1 and orc.guess[1].dtype == np.float32
    # (the pose of the frame after the prediction came through the float32 guess arrays)
    assert np.array_equal(s[1:4], poses[3][:3]) and np.array_equal(s[4:7], poses[3][3:].astype(np.float32))
    # with a float32 guess, the pose handed in is rounded on its way into it; prev (not aliased) keeps its value
    assert not orc.step_given(3, poses[4], False, 0.0)
    s = orc.state_record()
    assert np.array_equal(s[11:14], poses[4][3:].astype(np.float32)) and np.array_equal(s[8:11], poses[4][:3])
    assert np.array_equal(s[1:4], poses[3][:3]) and np.array_equal(s[4:7], poses[3][3:].astype(np.float32))
    # fewer than two tags drop the guess; the velocities stay
    assert not orc.step_given(1, poses[4], True, 0.5)
    s = orc.state_record()
    assert s[7] == 0 and not s[8:16].any() and s[16] == 2


def test_object_points_match_reference_golden():
    g = np.load(GOLDEN / "ape_sequence.npz")
    assert np.allclose(synth.object_points(), g["all_objpts"], atol=1e-9)


def test_decision_margin_filter():
    assert ape_oracle.filter_detections(["a", "b", "c"], [100.0, 49.9, 50.0]) == ["a", "c"]


# ---------------------------------------------------------------------------- pyramid / LK
def test_pyramid_and_scharr_restatement_equal_opencv():
    import cv2
    g = np.load(GOLDEN / "lk_pair.npz")
    img = g["prev"]
    for size in (img, img[:239, :317], img[:31, :23]):
        lv = size
        for _ in range(3):
            assert np.array_equal(lk_oracle.pyr_down_np(lv), cv2.pyrDown(lv))
            assert np.array_equal(lk_oracle.scharr_np(lv), lk_oracle.scharr_cv(lv))
            lv = cv2.pyrDown(lv)
    assert np.array_equal(cv2.pyrDown(img), g["level1"])
    assert np.array_equal(lk_oracle.scharr_cv(img), g["scharr0"])


def test_lk_restatement_matches_opencv_and_golden():
    g = np.load(GOLDEN / "lk_pair.npz")
    nxt, st, err = lk_oracle.lk_cv(g["prev"], g["next"], g["pts"])
    assert np.array_equal(st, g["status"]) and np.array_equal(nxt, g["next_pts"])      # OpenCV is deterministic
    n2, s2, e2 = lk_oracle.lk_np(g["prev"], g["next"], g["pts"])
    assert np.array_equal(s2, st)
    m = st == 1
    assert np.abs(n2[m] - nxt[m]).max() < 2e-3
    assert np.abs(e2[m] - err[m]).max() < 2e-3
    assert st.sum() >= 40 and (st == 0).sum() >= 1          # the fixture has tracked and lost points


# ---------------------------------------------------------------------------- dense refinement
def test_dpr_oracle_reproduces_golden():
    g = np.load(GOLDEN / "dpr_case.npz")
    model = util.dpr_model()
    for i in range(len(g["frames"])):
        out = dpr_oracle.refine(lk_oracle.pyramid_cv(g["frames"][i], 4), model, g["mtx"], g["init"][i])
        want = g["result"][i]
        assert np.allclose(out["pose"], want[:6], atol=1e-12)
        assert out["n_valid"] == int(want[7]) and out["evals"] == int(want[8]) and out["status"] == int(want[9])
        assert out["level"] == int(want[10])
        # and it actually refines: closer to the truth than the initial pose
        d0 = util.pose_diff(g["init"][i], g["truth"][i])
        d1 = util.pose_diff(out["pose"], g["truth"][i])
        assert d1[0] < d0[0] and d1[1] < d0[1] * 1.5


def test_dpr_oracle_jacobian_is_derivative_of_smoothed_cost():
    """The analytic 1x6 Jacobian against central differences of the residual it linearises
    (residual rebuilt with the same Scharr-interpolated gradient => compare J to dI/dp numerically on a smooth image)."""
    import cv2
    cam = make_golden.SMALL_CAM
    model = util.dpr_model()
    rng = np.random.default_rng(5)
    pose = np.array([0.3, -0.2, 0.1, 0.002, 0.001, 0.24])
    # a smooth synthetic image (quadratic ramp) so bilinear interpolation and Scharr/32 are exact derivatives
    ys, xs = np.mgrid[0:240, 0:320].astype(np.float64)
    img = np.clip(0.3 * xs + 0.2 * ys + 20, 0, 255).astype(np.uint8)
    ev = dpr_oracle.Evaluator([img], model, cam.mtx, pose)
    rmat, t = dpr_oracle.rodrigues(pose[:3]), pose[3:]
    r0, ok, jac = ev.residuals(rmat, t)
    eps = 1e-6
    for k in range(6):
        d = np.zeros(6); d[k] = eps
        rp, okp, _ = ev.residuals(dpr_oracle.rodrigues(d[:3]) @ rmat, t + d[3:], want_jac=False)
        rm, okm, _ = ev.residuals(dpr_oracle.rodrigues(-d[:3]) @ rmat, t - d[3:], want_jac=False)
        num = (rp - rm) / (2 * eps)
        sel = ok & okp & okm
        # uint8 quantisation of the ramp makes the image piecewise constant +-0.5: compare in the mean
        assert abs(np.mean(num[sel] - jac[sel, k])) < 0.02 * max(1.0, np.abs(jac[sel, k]).mean())


def test_dpr_multi_hypothesis_tie_breaks_to_lowest_index():
    g = np.load(GOLDEN / "dpr_case.npz")
    model = util.dpr_model()
    pyr = lk_oracle.pyramid_cv(g["frames"][1], 4)
    init = np.stack([g["init"][1], g["init"][1], g["truth"][1]])
    best, runs = dpr_oracle.refine_multi(pyr, model, g["mtx"], init)
    score = np.array([2 * r["cost"] / r["n_valid"] for r in runs])
    # the lowest index within SELECT_TIE of the best score: runs 0 and 1 are identical, run 2 (started at the truth) ends in
    # the same fixed point with a score that differs in the 6th digit or so - still a tie, so index 0 wins
    assert best == int(np.nonzero(score <= score.min() * (1 + dpr_oracle.SELECT_TIE))[0][0])
    assert score[0] == score[1] and best == 0


# ---------------------------------------------------------------------------- whole path (BASELINE config 1 shape)
def test_pipeline_oracle_reduces_to_ape_and_tracks_through_dropout():
    from oracle import pipeline_oracle
    g = np.load(GOLDEN / "ape_sequence.npz")
    group = ape_oracle.group_from_json(synth.april_group_dict())
    # with both extra stages off the composition is exactly the reference's APE state machine
    po = pipeline_oracle.PipelineOracle(group, g["mtx"], util.dpr_model(), use_lk=False, use_dense_refine=False)
    for f in range(40):
        po.frame(np.zeros((8, 8), np.uint8), make_golden.unpack_detections(g["ids"], g["corners"], f))
        snap = po.snapshot()
        want = g["prev"][f]
        assert (snap["prev"] is None) == bool(np.isnan(want[0]))
        if snap["prev"] is not None:
            assert np.array_equal(np.concatenate(snap["prev"]), want)
    # full path on a short rendered VGA sequence with a detector dropout: LK carries the tags, refinement runs
    cam = synth.CAMERA_VGA
    po = pipeline_oracle.PipelineOracle(group, cam.mtx, util.dpr_model())
    traj = synth.trajectory(777, 6)
    rng = np.random.default_rng(777)
    for f in range(6):
        dets = synth.detections(traj[f], cam, rng)
        if f == 4:
            dets = dets[:1]
        po.frame(synth.render(traj[f], cam, seed=f), dets)
        assert po.last_accepted, f
        dr, dt = util.pose_diff(np.concatenate([po.prev[0].ravel(), po.prev[1].ravel().astype(np.float64)]), traj[f])
        assert dr < 0.02 and dt < 2e-3, (f, dr, dt)
        if f == 4:
            assert po.tracked >= 1


# ------------------------------------------------------------------------------------------
# frame ingest with undistortion (row N2): the restatement of cv::undistort against the installed cv2,
# i.e. against the very call the reference makes (detect_pose.py:174)
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("w,h,f", [(333, 201, 300.0), (640, 480, 600.0), (97, 64, 80.0)])
def test_undistort_oracle_matches_cv2(w, h, f):
    import cv2
    from oracle import undistort_oracle as uo
    rng = np.random.default_rng(w)
    mtx = np.array([[f, 0, w / 2 + 3.3], [0, f * 1.01, h / 2 - 2.1], [0, 0, 1]])
    for dist in ([-0.28, 0.11, 0.0007, -0.0004, -0.02], [0.05, -0.1, 0.001, 0.002, 0.03], [0, 0, 0, 0, 0]):
        dist = np.array(dist, np.float64).reshape(1, 5)
        new_mtx, roi = cv2.getOptimalNewCameraMatrix(mtx, dist, (w, h), 1, (w, h))
        x, y, rw, rh = roi
        for shape in ((h, w, 3), (h, w)):
            frame = rng.integers(0, 256, shape, dtype=np.uint8)
            und = cv2.undistort(frame, mtx, dist, None, new_mtx)
            assert np.array_equal(uo.undistort(frame, mtx, dist, new_mtx), und)
            want = und[y:y + rh, x:x + rw]
            want = cv2.cvtColor(want, cv2.COLOR_BGR2GRAY) if want.ndim == 3 else want
            assert np.array_equal(uo.undistort_frame_gray(frame, mtx, dist, new_mtx, roi), want)


def test_remap_table_sums_to_one():
    from oracle import undistort_oracle as uo
    tab = uo.bilinear_table()
    assert tab.shape == (1024, 4) and (tab.sum(axis=1) == 32768).all() and tab.min() >= 0
    assert tab[0].tolist() == [32767, 0, 0, 1]          # saturation of 1.0 * 2^15 and the remainder fix-up


def test_undistort_oracle_matches_golden():
    from oracle import make_golden, undistort_oracle as uo
    g = np.load(make_golden.GOLDEN / "undistort_case.npz")
    for k in range(2):
        x, y, w, h = g["roi"][k]
        got = uo.undistort_frame_gray(g["frame"], g["mtx"], g["dist"][k], g["new_mtx"][k], g["roi"][k])
        assert np.array_equal(got.ravel(), g[f"gray{k}"]) and got.shape == (h, w)



def test_roi_exactness_rule_of_the_pyramid_chain():
    """The rule behind agt_build_pyramid_roi / agt_lk_roi (include/agt.h): a level-l pixel depends only on the level-0
    pixels 2^l x +- (2^(l+1) - 2) of its pyrDown chain (reflected at the image border).  Checked with cv2.pyrDown itself:
    randomising everything outside a rectangle leaves the window the kernels treat as exact untouched."""
    import cv2
    rng = np.random.default_rng(5)
    w, h = 208, 144
    base = rng.integers(0, 256, (h, w), dtype=np.uint8)

    def window(lo, hi, n0, n, level):
        reach = (2 << level) - 2
        a = 0 if lo <= 0 else (lo + reach + (1 << level) - 1) >> level
        b = n if hi >= n0 else ((hi - 1 - reach) >> level) + 1
        return a, max(b, 0)

    for x0, y0, x1, y1 in ((48, 30, 160, 120), (0, 0, 96, 80), (112, 64, w, h), (0, 40, w, 100)):
        other = rng.integers(0, 256, (h, w), dtype=np.uint8)
        other[y0:y1, x0:x1] = base[y0:y1, x0:x1]
        a, b = base, other
        for level in (1, 2, 3):
            a, b = cv2.pyrDown(a), cv2.pyrDown(b)
            lh, lw = a.shape
            ax, bx = window(x0, x1, w, lw, level)
            ay, by = window(y0, y1, h, lh, level)
            assert bx > ax and by > ay
            assert np.array_equal(a[ay:by, ax:bx], b[ay:by, ax:bx]), (level, (x0, y0, x1, y1))


# ---------------------------------------------------------------------------- corner refinement (row N3, first step)
def test_corner_subpix_restatement_equals_opencv():
    from oracle import corner_oracle
    cam = synth.CAMERA_VGA
    rng = np.random.default_rng(3)
    worst = 0.0
    for s in range(4):
        pose = synth.trajectory(600 + s, 1)[0]
        img = synth.render(pose, cam, s)
        true = np.concatenate([synth.project(synth.object_points()[4 * k:4 * k + 4], pose, cam) for k in synth.visible_tags(pose)])
        pts = (true + rng.normal(0, 1.0, true.shape)).astype(np.float32)
        for win in (3, 5):
            a = corner_oracle.corner_subpix_cv(img, pts, win)
            b = corner_oracle.corner_subpix_np(img, pts, win)
            worst = max(worst, float(np.abs(a - b).max()))
    border = np.array([[2.3, 3.1], [637.2, 476.9], [0.5, 240.0], [320.0, 0.2], [639.4, 100.0]], np.float32)
    a, b = corner_oracle.corner_subpix_cv(img, border), corner_oracle.corner_subpix_np(img, border)
    worst = max(worst, float(np.abs(a - b).max()))
    assert worst <= 1e-4, worst           # float32 resampling order: identical on almost every corner


# ---------------------------------------------------------------------------- tag identification / detection (row N3)
def test_tag_decoder_restatement_agrees_with_aruco():
    """decode_np (the frozen specification of agt_decode_tags) against OpenCV's ArUco module, the one implementation of the
    tag36h11 family in the image: on every tag aruco finds, decoding aruco's own corners returns aruco's id (hamming 0,
    rotation 0 once the corners are in the reference's order); decoding the true corners returns the true id; a quad that
    starts at the tag's corner k comes back with rotation k; the committed aruco output (tests/golden/tag_case.npz) is
    reproduced by the installed cv2."""
    from oracle import tag_oracle
    cam = synth.CAMERA_VGA
    obj = synth.object_points()
    g = np.load(make_golden.GOLDEN / "tag_case.npz")
    at = 0
    for frame, pose, cnt in zip(g["frames"], g["poses"], g["counts"]):
        live = sorted(tag_oracle.detect_cv(frame), key=lambda d: d[0])
        assert [i for i, _ in live] == g["ids"][at:at + cnt].tolist()
        assert np.abs(np.array([c for _, c in live]) - g["corners"][at:at + cnt]).max() < 1e-3
        at += cnt
    n_aruco = 0
    for s in range(8):
        pose = synth.trajectory(720 + s, 1)[0]
        img = synth.render(pose, cam, seed=s)
        facing = set(synth.visible_tags(pose, cos_limit=0.0).tolist())          # aruco also reads tags seen at a grazing angle
        for tag, corners in tag_oracle.detect_cv(img):
            assert tag in facing
            n_aruco += 1
            assert tag_oracle.decode_np(img, corners)[:3] == (tag, 0, 0)
            true = synth.project(obj[4 * tag:4 * tag + 4], pose, cam)
            assert np.abs(corners - true).max() < 3.0            # aruco's corners are contour points
            tid, rot, ham, margin = tag_oracle.decode_np(img, true)
            assert (tid, rot, ham) == (tag, 0, 0) and margin > 50.0          # the reference's decision-margin bar
            for k in range(1, 4):
                assert tag_oracle.decode_np(img, np.roll(true, -k, axis=0))[:3] == (tag, k, 0)
    assert n_aruco >= 20
    # not a tag: a flat patch, a quad across two faces, a quad that leaves the image
    assert tag_oracle.decode_np(img, np.array([[10, 40], [10, 10], [40, 10], [40, 40]], float))[0] == -1
    assert tag_oracle.decode_np(img, np.array([[-5, 40], [-5, 10], [40, 10], [40, 40]], float)) == (-1, 0, 255, 0.0)


def test_pack_detections_host_rules():
    """The A0 rules the device kernel agt_pack_detections has to reproduce (tests/test_gpu_tags.py compares it with this
    function): position = index of the id in the group's JSON order, unknown ids raise, a tag seen twice fills one slot."""
    from accurate_aprilgroup_tracking_b200.batched import pack_detections
    group = [7, 3, 11, 0]
    c = np.arange(8, dtype=np.float32).reshape(4, 2)
    img, valid, n = pack_detections([[(3, c), (0, c + 100)], [], [(11, c + 5), (11, c + 6)]], group)
    assert n.tolist() == [2, 0, 1]
    assert np.array_equal(img[0, 4:8], c) and np.array_equal(img[0, 12:16], c + 100) and valid[0].tolist() == [0] * 4 + [1] * 4 + [0] * 4 + [1] * 4
    assert valid[2].tolist() == [0] * 8 + [1] * 4 + [0] * 4
    with pytest.raises(KeyError):
        pack_detections([[(5, c)]], group)


# the detector's first stage (tag_oracle.quads_np) and the case set of tests/test_gpu_tag_quads.py
@pytest.fixture(scope="module")
def tag_quad_cases():
    from tests import tag_quad_cases
    return tag_quad_cases.build()


def test_tag_quad_case_set_hits_its_targets(tag_quad_cases):
    missed = [c["name"] for c in tag_quad_cases if not c["target"](c["oracle"])]
    assert not missed, missed


def test_quads_np_components_equal_opencv(tag_quad_cases):
    """The components of quads_np (scipy.ndimage.label) against cv2.connectedComponentsWithStats with 4-connectivity: count,
    areas, bounding boxes and centroids identical on the whole case set."""
    import cv2
    for c in tag_quad_cases:
        r = c["oracle"]
        n, lab, st, cen = cv2.connectedComponentsWithStats(r["dark"].astype(np.uint8), connectivity=4)
        assert n - 1 == r["n_all"], c["name"]
        bb = r["bbox"][1:]
        ours = np.column_stack([bb[:, 0], bb[:, 1], bb[:, 2] - bb[:, 0] + 1, bb[:, 3] - bb[:, 1] + 1, r["area"][1:]])
        order_cv = np.lexsort(st[1:].T[::-1])
        order_np = np.lexsort(ours.T[::-1])
        assert np.array_equal(st[1:][order_cv], ours[order_np]), c["name"]
        cen_np = np.column_stack([r["sx"][1:] / r["area"][1:], r["sy"][1:] / r["area"][1:]])
        assert np.array_equal(cen[1:][order_cv], cen_np[order_np]), c["name"]


def test_quads_np_far_points_equal_brute_force(tag_quad_cases):
    """The three farthest-point passes of quads_np (vectorised, segment maxima of packed keys) against a loop over every pixel of
    each component (boundary test per pixel, keys compared as (value, pixel index) pairs: the larger index wins a tie)."""
    F = np.float32
    checked = 0
    for c in tag_quad_cases:
        r = c["oracle"]
        lab, dark = r["labels"], r["dark"]
        hh, ww = dark.shape
        comps = [k for k in r["far"]][:40]
        for k in comps:
            ys, xs = np.nonzero(lab == k)
            px = []
            for y, x in zip(ys.tolist(), xs.tolist()):
                nb = [(y - 1, x), (y + 1, x), (y, x - 1), (y, x + 1)]
                if any(not (0 <= v < hh and 0 <= u < ww) or not dark[v, u] for v, u in nb):
                    px.append((y, x, y * ww + x))
            cx, cy = F(int(r["sx"][k]) / int(r["area"][k])), F(int(r["sy"][k]) / int(r["area"][k]))
            best = max(((F(F(F(x) - cx) * F(F(x) - cx)) + F(F(F(y) - cy) * F(F(y) - cy)), i) for y, x, i in px))
            alts = r["far"][k]
            assert best[1] in {a[0] for a in alts}, (c["name"], k)
            p0, sp, p2, sn, _ = alts[0]
            x0, y0 = p0 % ww, p0 // ww
            far2 = max(((x - x0) ** 2 + (y - y0) ** 2, i) for y, x, i in px)
            assert far2[1] == p2, (c["name"], k)
            x2, y2 = p2 % ww, p2 // ww
            d = [((x2 - x0) * (y - y0) - (y2 - y0) * (x - x0), i) for y, x, i in px]
            pos = max(((v, i) for v, i in d if v > 0), default=(0, 0))
            neg = max(((-v, i) for v, i in d if v < 0), default=(0, 0))
            assert (pos[1], neg[1]) == (sp, sn), (c["name"], k)
            checked += 1
    assert checked >= 200
