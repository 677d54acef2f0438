"""CPU oracle = executable specification of the covariance of a refined pose (agt_pose_covariance).

TEST INFRASTRUCTURE (see oracle/__init__.py).  Built on the dense-refinement oracle (oracle/dpr_oracle.py), whose
Evaluator.normal_equations is the cost function the refinement minimises; csrc/agt_dpr.cu:pose_cov_kernel is checked
against this file.

Specification (float64):

  cost function  fixed by the initial pose pose0 exactly as dpr_oracle.refine fixes it: pyramid level and active tags
                 decided at pose0 (dpr_oracle.Evaluator)
  one evaluation at `pose` (normally the refined pose):
                 J   n x 6 Jacobian of the valid residuals, [Y x g, g]: left perturbation R <- exp(w) R (radians), then
                     t <- t + dt (metres) - the refinement's tangent convention, rotation block first
                 H   = J^T J ;  c = 1/2 sum r^2 ;  n = #valid
                 s^2 = 2c / (n - 6)                  (residual variance, 6 parameters fitted)
                 Sigma = s^2 H^-1
                 ok  = n > 6 and H positive definite (Cholesky succeeds); otherwise s^2 (n <= 6) and Sigma are NaN

What Sigma is: the Gauss-Newton covariance of the estimate under independent residuals of one common variance s^2.  What
it is not: a bound on the error against the true pose.  The estimator's bias (DESIGN.md section 2) is not in it; the
residuals of neighbouring samples are correlated where samples are denser than pixels (VGA: Sigma too small) and
bilinear interpolation averages pixel noise where they are sparser (1080p: too large); on synthetic frames s^2 is
dominated by the mismatch between the sharp rendered cells and the blurred surface model, not by pixel noise.
"""
from __future__ import annotations

import math

import numpy as np

from oracle import dpr_oracle


def covariance(pyramid, model: dpr_oracle.Model, kmat: np.ndarray, pose0: np.ndarray, pose: np.ndarray) -> dict:
    """-> dict(H (6,6), c, n, s2, cov (6,6), ok) of the refinement's cost function (fixed by pose0) evaluated at pose."""
    ev = dpr_oracle.Evaluator(pyramid, model, kmat, np.asarray(pose0, dtype=np.float64))
    pose = np.asarray(pose, dtype=np.float64)
    hmat, _, c, n = ev.normal_equations(dpr_oracle.rodrigues(pose[:3]), pose[3:6])
    s2 = 2.0 * c / (n - 6) if n > 6 else math.nan
    ok = n > 6
    cov = np.full((6, 6), np.nan)
    if ok:
        try:
            low = np.linalg.cholesky(hmat)
        except np.linalg.LinAlgError:
            ok = False
        else:
            m = np.linalg.solve(low, np.eye(6))            # L^-1
            cov = s2 * (m.T @ m)
    return {"H": hmat, "c": c, "n": n, "s2": s2, "cov": cov, "ok": ok}


def tangent_offset(pose: np.ndarray, ref: np.ndarray) -> np.ndarray:
    """(w, dt) with R(pose) = exp(w) R(ref), t(pose) = t(ref) + dt: the refinement's tangent convention."""
    w = dpr_oracle.log_rotation(dpr_oracle.rodrigues(pose[:3]) @ dpr_oracle.rodrigues(ref[:3]).T)
    return np.concatenate([w, np.asarray(pose[3:6], dtype=np.float64) - ref[3:6]])


def level_noise_var(level: int, sigma: float) -> float:
    """Variance of the pixel noise at pyramid level `level` of frames with pixel noise sigma, quantised to 8 bits: cv2.pyrDown's
    separable [1 4 6 4 1]/16 filter scales a variance by (70/256)^2 per level and every level is rounded again (+1/12)."""
    var = sigma * sigma + 1.0 / 12.0
    for _ in range(level):
        var = var * (70.0 / 256.0) ** 2 + 1.0 / 12.0
    return var


def calibration(cam, model: dpr_oracle.Model, truth: np.ndarray, seeds, rng: np.random.Generator, sig_rot: float = 0.01,
                sig_trans: float = 0.0005) -> dict:
    """Seed-to-seed scatter of the refined pose against the predicted covariance at one true pose.

    Every seed renders the frame with its own pixel noise (synth.render, noise sigma synth.NOISE_SIGMA), the refinement starts
    from one start truth + N(0, sig_rot) / N(0, sig_trans) shared by all seeds and `covariance` is evaluated at its answer.
    The start is shared because it fixes the cost function: with a start per seed a tag near the 75 degree visibility limit
    is in the active set for some seeds and not for others, and the answers of the two cost functions differ by more than
    the noise moves either (seen as eigenvalues of 100 and more).  -> dict(eig: generalized
    eigenvalues of the scatter S against sigma_level^2 H^-1 (H averaged over the seeds; sigma_level^2 = level_noise_var, the
    pixel noise at the pyramid level the refinement reads), i.e. the eigenvalues of A^-1/2 S A^-1/2; level; nees: mean of d^T Sigma^-1 d over the seeds with d the offset from the mean answer and Sigma = s^2 H^-1;
    sigma_res: the residual sigma sqrt(s^2), mean; n: valid samples, mean; bias: |mean answer - truth| in rotation (rad) and
    translation (m) against the standard deviation s^2 H^-1 gives along the same axes)."""
    from scipy.linalg import eigh
    from accurate_aprilgroup_tracking_b200 import synth
    from oracle import lk_oracle
    offs, hs, covs, s2, ns = [], [], [], [], []
    init = truth + np.concatenate([rng.normal(0, sig_rot, 3), rng.normal(0, sig_trans, 3)])
    for seed in seeds:
        frame = synth.render(truth, cam, seed=int(seed), noise=True)
        pyr = lk_oracle.pyramid_cv(frame, 4)
        out = dpr_oracle.refine(pyr, model, cam.mtx, init)
        cv = covariance(pyr, model, cam.mtx, init, out["pose"])
        offs.append(tangent_offset(out["pose"], truth))
        hs.append(cv["H"]); covs.append(cv["cov"]); s2.append(cv["s2"]); ns.append(cv["n"])
    offs = np.array(offs)
    mean = offs.mean(axis=0)
    scatter = np.cov(offs.T)
    level = dpr_oracle.select_level(cam.fx, model.pitch, init[5], 4)
    predicted = level_noise_var(level, synth.NOISE_SIGMA) * np.linalg.inv(np.mean(hs, axis=0))
    eig = eigh(scatter, predicted, eigvals_only=True)
    d = offs - mean
    nees = float(np.mean([di @ np.linalg.solve(ci, di) for di, ci in zip(d, covs)]))
    sd = np.sqrt(np.diag(np.mean(covs, axis=0)))
    return {"eig": eig, "level": level, "nees": nees, "sigma_res": float(np.mean(np.sqrt(s2))), "n": float(np.mean(ns)),
            "bias_over_sd": np.abs(mean) / sd, "bias": mean}


CALIBRATION_POSES, CALIBRATION_SEEDS = 4, range(1000, 1040)


def calibration_poses(cam_name: str):
    """The true poses of the calibration sweep (tests/test_cpu_pose_cov.py, scripts/pose_cov_calibration.py)."""
    from accurate_aprilgroup_tracking_b200 import synth
    rng = np.random.default_rng(7100 if cam_name == "vga" else 7200)
    return [synth.random_pose(rng) for _ in range(CALIBRATION_POSES)]
