"""The covariance oracle (oracle/dpr_cov_oracle.py) pinned to independent code, calibrated statistically, and its
degenerate cases."""
import numpy as np
import pytest

from accurate_aprilgroup_tracking_b200 import synth
from oracle import dpr_cov_oracle, dpr_oracle, dpr_pin, lk_oracle

BAND = (0.15, 5.0)          # eigenvalues of the seed-to-seed scatter against sigma_level^2 H^-1 (see DESIGN.md section 2)


@pytest.fixture(scope="module")
def mdl():
    return dpr_pin.model()


@pytest.mark.parametrize("cam_name,i", [("vga", 0), ("vga", 7), ("1080p", 1), ("1080p", 5)])
def test_oracle_matches_independent_code(mdl, cam_name, i):
    """H = J^T J with J from cv2.projectPoints central differences and scipy's bilinear sampling (oracle/dpr_pin.py), c and n
    from the independent residual, at the start and at the refined pose."""
    cam = dpr_pin.CAMERAS[cam_name]
    truth, init, frame = dpr_pin.case(cam_name, i)
    pyr = lk_oracle.pyramid_cv(frame, 4)
    refined = dpr_oracle.refine(pyr, mdl, cam.mtx, init)["pose"]
    for pose in (init, refined):
        got = dpr_cov_oracle.covariance(pyr, mdl, cam.mtx, init, pose)
        r, ok = dpr_pin.independent_residuals(pyr, mdl, cam.mtx, init, pose)
        j = dpr_pin.independent_jacobian(pyr, mdl, cam.mtx, init, pose) * ok[:, None]
        h = j.T @ j
        scale = np.sqrt(np.outer(np.diag(h), np.diag(h)))
        assert got["n"] == int(ok.sum()) and got["ok"]
        assert abs(got["c"] - 0.5 * float(r @ r)) <= 1e-9 * got["c"]
        assert (np.abs(got["H"] - h) <= 2e-5 * scale).all(), np.abs(got["H"] - h).max() / scale.max()
        assert np.allclose(got["cov"] @ got["H"], got["s2"] * np.eye(6), atol=1e-9 * got["s2"])
        assert got["s2"] == pytest.approx(2 * got["c"] / (got["n"] - 6))


@pytest.mark.parametrize("cam_name", ["vga", "1080p"])
def test_statistical_calibration(mdl, cam_name):
    """4 poses x 40 noise seeds (the sweep of profiles/r03_pose_cov_calibration.log): the scatter of the refined pose
    against sigma_level^2 H^-1 - the pixel noise at the pyramid level the refinement reads - has every eigenvalue in [0.15, 5]."""
    cam = dpr_pin.CAMERAS[cam_name]
    for k, truth in enumerate(dpr_cov_oracle.calibration_poses(cam_name)):
        r = dpr_cov_oracle.calibration(cam, mdl, truth, dpr_cov_oracle.CALIBRATION_SEEDS, np.random.default_rng(k))
        print(f"{cam_name} pose {k}: eigenvalues {np.round(r['eig'], 2)}, residual sigma {r['sigma_res']:.1f}")
        assert BAND[0] <= r["eig"].min() and r["eig"].max() <= BAND[1], (k, r["eig"])


def test_degenerate_cases(mdl):
    cam = synth.CAMERA_1080P
    truth, init, frame = dpr_pin.case("1080p", 1)
    pyr = lk_oracle.pyramid_cv(frame, 4)
    # a pose that sees no tag: no valid sample
    far = init.copy()
    far[3] = 5.0
    got = dpr_cov_oracle.covariance(pyr, mdl, cam.mtx, far, far)
    assert got["n"] == 0 and not got["ok"] and np.isnan(got["cov"]).all() and np.isnan(got["s2"])
    # n_valid <= 6: the object pushed off the frame until a handful of samples remain
    ev = dpr_oracle.Evaluator(pyr, mdl, cam.mtx, init)
    for dx in np.linspace(0.0, 0.4, 4001):
        pose = init + np.array([0, 0, 0, dx, 0, 0])
        _, ok, _ = ev.residuals(dpr_oracle.rodrigues(pose[:3]), pose[3:])
        if 0 < ok.sum() <= 6:
            break
    else:
        pytest.fail("no pose with 1..6 valid samples found")
    got = dpr_cov_oracle.covariance(pyr, mdl, cam.mtx, init, pose)
    assert 0 < got["n"] <= 6 and not got["ok"] and np.isnan(got["cov"]).all() and np.isnan(got["s2"])
    # a flat frame: every sample valid, H = 0 -> not positive definite
    flat = [np.full_like(l, 128) for l in pyr]
    got = dpr_cov_oracle.covariance(flat, mdl, cam.mtx, init, init)
    assert got["n"] > 6 and not got["ok"] and np.isnan(got["cov"]).all()
