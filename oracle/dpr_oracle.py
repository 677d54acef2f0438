"""CPU oracle = executable specification of dense pose refinement (DPR).

TEST INFRASTRUCTURE (see oracle/__init__.py).  The mounted reference snapshot has
no dense-refinement code (README.md:20 only cites the DodecaPen paper as future
work), so there is no reference implementation to pin against: this file freezes
the semantics named by BASELINE.json north_star / SURVEY.md 9.4 and the CUDA
kernel (csrc/agt_dpr.cu) is checked against it.  What CAN be pinned is pinned to
independent code (oracle/dpr_pin.py, tests/golden/dpr_pin.npz, tests/test_cpu_dpr_pin.py):
  * the residual: cv2.projectPoints + scipy.ndimage.map_coordinates (bilinear) to 1e-9;
  * the answer: the loop below is Gauss-Newton with the Scharr gradient standing in for
    the derivative of the bilinear interpolant, so what it converges to is the pose where
    J^T r = 0 with that J.  scipy finds the same pose with its own solvers
    (least_squares(method="lm") to get near, then optimize.root(method="hybr") on
    g(p) = J^T r): 64 VGA + 64 1080p noisy renders agree to <= 1e-5 rad / 2 um.

Specification (float64 here; the kernel evaluates samples in float32 and
reduces/solves in float64):

  model    samples (S,4) = (x,y,z,O) in the group frame, tag-major, S = 12*G*G;
           tag_normals (12,3); tag_centres (12,3); pitch = metric sample spacing.
  frozen at the initial pose (R0,t0):
           tag k active  <=>  (R0 n_k) . (-c_k/|c_k|) > cos 75deg,  c_k = R0 t_k + t0
           level l = 0 if q < 2, 1 if q < 4, 2 if q < 8, else 3 (clamped to the
           levels available), q = fx * pitch / t0.z
  residual for sample i of an active tag at pose (R,t):
           Y = R x_i ; X = Y + t ; skip if X.z <= 1e-6
           u = fx X.x/X.z + cx ; v = fy X.y/X.z + cy            (pinhole)
           ul = u/2^l ; vl = v/2^l (pyrDown centres pixel i of level l+1 on pixel 2i of level l)
           x0 = floor(ul) ; y0 = floor(vl)
           valid <=> 1 <= x0 <= w_l-3 and 1 <= y0 <= h_l-3
           I  = bilinear(level_l u8)(ul,vl)
           G  = bilinear(Scharr_int16(level_l))(ul,vl) / 32 / 2^l   (per full-res pixel)
           r_i = I - O_i
           g  = (Gx fx/Z, Gy fy/Z, -(Gx fx X.x + Gy fy X.y)/Z^2)
           J_i = [ Y x g , g ]   (left perturbation R <- exp(w) R, then t)
  LM       H = sum J^T J, b = sum J^T r, c = 1/2 sum r^2, n = #valid
           lambda0 = 1e-3; solve (H + lambda diag H) d = -b (Cholesky, float64)
           trial = (exp(d_w) R, t + d_t); one evaluation per trial
           step length (Aitken): the Gauss-Newton map with the Scharr gradient contracts onto its fixed
           point linearly, and consecutive steps are collinear (cos 0.97..1.00 measured; ratio +0.25..+0.4
           at 1080p where the gradient overestimates the slope, -0.7 at VGA where it underestimates it and
           the iteration bounces across the solution).  With d the solve's step and d_prev the previous
           accepted one, in the metric of the current H: num = d^T H d_prev, den = d_prev^T H d_prev,
           if num^2 > 0.64 den (d^T H d):  alpha <- clamp(alpha / (1 - min(num/den, 0.75)), 0.25, 4)
           else                            alpha <- 1 + (alpha - 1)/2;          alpha = 1 without a d_prev.
           trial = (exp(alpha d_w) R, t + alpha d_t); one evaluation per trial
           (only while lambda <= lambda0, the undamped regime: a step solved with a larger lambda has alpha = 1 and is not
           remembered as d_prev - steps of different damping are not comparable)
           accept iff c_trial < c (1 + 1e-2) and c_trial <= c_0, the cost at the initial pose:
           lambda <- max(lambda/10, 1e-9), d_prev <- d;
           else lambda <- 10 lambda, alpha <- 1, d_prev forgotten.
           The slack is what makes the answer well defined: the Scharr gradient is not the exact
           derivative of the bilinear interpolant, so close to convergence the steps change the cost by
           ~1e-5 of itself in either direction (up to 2e-3 on far, ill-conditioned views, where a strict or a 1e-3 rule
           rejects every step towards the fixed point and the loop creeps to the evaluation cap: 1 frame in 4096 of
           the bench batch).  With a strict `c_trial < c` (round 1) accept/reject was
           decided by that noise and the loop stalled up to 3e-4 rad from the fixed point, at a place that
           depended on the solver; with the slack every such step is taken, rejections are left for steps
           that really overshoot, and the loop contracts onto J^T r = 0 (scipy's root finder lands within
           3e-6 rad of it; 8.3 evaluations on average at 1080p against 11.8 without the step length).
           The bound by c_0 keeps the slack from compounding on a poor start: a run that wanders (the slack accepts
           up to 1 % more per step) could otherwise end above the cost it started from.  Returning the lowest-cost
           accepted pose instead would not do: near convergence that pose is not the fixed point J^T r = 0.
           stop: |alpha d_w| < 5e-6 and |alpha d_t| < 1e-6 (accepted or rejected step), or 50 evaluations,
           or lambda > 1e6
  result   rvec = log(R), t, c, n, evaluations, status
           status: 1 converged, 2 evaluation cap, 3 lambda overflow, 0 no valid samples
  multi-hypothesis: independent runs; score = 2c/n; winner = the lowest index among the runs whose score is within 1e-4
           (relative) of the best one: runs that end in the same fixed point differ by ~1e-6 in score (their last
           steps), so an exact comparison would let that noise pick the index.
"""
from __future__ import annotations

import math
from dataclasses import dataclass
from typing import List, Optional, Sequence, Tuple

import cv2 as cv
import numpy as np

COS_VISIBLE = math.cos(math.radians(75.0))
LAMBDA0 = 1e-3
LAMBDA_MIN = 1e-9
LAMBDA_MAX = 1e6
MAX_EVALS = 50
TOL_ROT = 5e-6
TOL_TRANS = 1e-6
ACCEPT_SLACK = 1e-2
AITKEN_COS2 = 0.64          # use the ratio of consecutive steps only if they are collinear: cos^2 > 0.64
AITKEN_QMAX = 0.75
ALPHA_MIN, ALPHA_MAX = 0.25, 4.0
SELECT_TIE = 1e-4

ST_NONE, ST_CONVERGED, ST_MAX_EVALS, ST_LAMBDA = 0, 1, 2, 3


def rodrigues(r):
    r = np.asarray(r, dtype=np.float64).reshape(3)
    th = math.sqrt(float(r @ r))
    if th < 1e-12:
        k = np.array([[0, -r[2], r[1]], [r[2], 0, -r[0]], [-r[1], r[0], 0]])
        return np.eye(3) + k
    k = r / th
    kx = np.array([[0, -k[2], k[1]], [k[2], 0, -k[0]], [-k[1], k[0], 0]])
    return math.cos(th) * np.eye(3) + (1 - math.cos(th)) * np.outer(k, k) + math.sin(th) * kx


def log_rotation(m):
    return cv.Rodrigues(np.asarray(m, dtype=np.float64))[0].reshape(3)


@dataclass
class Model:
    samples: np.ndarray      # (S,4) float32
    sample_tag: np.ndarray   # (S,) uint8
    normals: np.ndarray      # (12,3) float32
    centres: np.ndarray      # (12,3) float32
    pitch: float


def select_level(fx: float, pitch: float, z: float, n_levels: int) -> int:
    q = fx * pitch / z
    lvl = 0 if q < 2 else 1 if q < 4 else 2 if q < 8 else 3
    return min(lvl, n_levels - 1)


def active_tags(model: Model, r0: np.ndarray, t0: np.ndarray) -> np.ndarray:
    c = model.centres.astype(np.float64) @ r0.T + t0
    n = model.normals.astype(np.float64) @ r0.T
    d = -np.sum(n * c, axis=1) / np.linalg.norm(c, axis=1)
    return d > COS_VISIBLE


class Evaluator:
    """Cost / normal equations of one frame at a fixed (active set, level)."""

    def __init__(self, pyramid: Sequence[np.ndarray], model: Model, kmat: np.ndarray, pose0: np.ndarray):
        self.fx, self.fy, self.cx, self.cy = kmat[0, 0], kmat[1, 1], kmat[0, 2], kmat[1, 2]
        r0 = rodrigues(pose0[:3])
        t0 = np.asarray(pose0[3:6], dtype=np.float64)
        self.level = select_level(self.fx, model.pitch, t0[2], len(pyramid))
        act = active_tags(model, r0, t0)
        self.active = act
        sel = act[model.sample_tag]
        s = model.samples[sel].astype(np.float64)
        self.x = s[:, :3]
        self.o = s[:, 3]
        lvl = pyramid[self.level]
        self.img = lvl.astype(np.float64)
        self.gx = cv.Scharr(lvl, cv.CV_16S, 1, 0).astype(np.float64)
        self.gy = cv.Scharr(lvl, cv.CV_16S, 0, 1).astype(np.float64)
        self.h, self.w = lvl.shape
        self.scale = 1.0 / (1 << self.level)

    def residuals(self, rmat, t, want_jac=True):
        y = self.x @ rmat.T
        xc = y + t
        z = xc[:, 2]
        ok = z > 1e-6
        zs = np.where(ok, z, 1.0)
        u = self.fx * xc[:, 0] / zs + self.cx
        v = self.fy * xc[:, 1] / zs + self.cy
        ul = u * self.scale
        vl = v * self.scale
        x0 = np.floor(ul)
        y0 = np.floor(vl)
        ok &= (x0 >= 1) & (x0 <= self.w - 3) & (y0 >= 1) & (y0 <= self.h - 3)
        xi = np.where(ok, x0, 1).astype(np.int64)
        yi = np.where(ok, y0, 1).astype(np.int64)
        a = ul - x0
        b = vl - y0
        w00, w01, w10, w11 = (1 - a) * (1 - b), a * (1 - b), (1 - a) * b, a * b

        def bil(p):
            return w00 * p[yi, xi] + w01 * p[yi, xi + 1] + w10 * p[yi + 1, xi] + w11 * p[yi + 1, xi + 1]

        r = np.where(ok, bil(self.img) - self.o, 0.0)
        if not want_jac:
            return r, ok, None
        gs = self.scale / 32.0
        gx = bil(self.gx) * gs
        gy = bil(self.gy) * gs
        g0 = gx * self.fx / zs
        g1 = gy * self.fy / zs
        g2 = -(g0 * xc[:, 0] + g1 * xc[:, 1]) / zs
        g = np.stack([g0, g1, g2], axis=1)
        jac = np.concatenate([np.cross(y, g), g], axis=1) * ok[:, None]
        return r, ok, jac

    def normal_equations(self, rmat, t):
        r, ok, jac = self.residuals(rmat, t)
        return jac.T @ jac, jac.T @ r, 0.5 * float(r @ r), int(ok.sum())


def refine(pyramid: Sequence[np.ndarray], model: Model, kmat: np.ndarray, pose0: np.ndarray,
           max_evals: int = MAX_EVALS):
    """-> dict(pose (6,), cost, n_valid, evals, status, level, active (12,) bool)."""
    ev = Evaluator(pyramid, model, kmat, pose0)
    rmat = rodrigues(pose0[:3])
    t = np.asarray(pose0[3:6], dtype=np.float64).copy()
    hmat, b, c, n = ev.normal_equations(rmat, t)
    evals = 1
    lam = LAMBDA0
    alpha = 1.0
    d_prev = None
    status = ST_MAX_EVALS
    c_start = c
    if n == 0:
        status = ST_NONE
    while status == ST_MAX_EVALS and evals < max_evals:
        a = hmat + lam * np.diag(np.diag(hmat))
        try:
            low = np.linalg.cholesky(a)
        except np.linalg.LinAlgError:
            lam *= 10.0
            if lam > LAMBDA_MAX:
                status = ST_LAMBDA
            continue
        d = -np.linalg.solve(low.T, np.linalg.solve(low, b))
        if lam > LAMBDA0:
            alpha, d_prev = 1.0, None              # damped steps are not comparable: no step-length adaptation
        elif d_prev is not None:
            hp = hmat @ d_prev
            num, den, dd = float(d @ hp), float(d_prev @ hp), float(d @ hmat @ d)
            if num * num > AITKEN_COS2 * den * dd:
                alpha = min(max(alpha / (1.0 - min(num / den, AITKEN_QMAX)), ALPHA_MIN), ALPHA_MAX)
            else:
                alpha = 1.0 + 0.5 * (alpha - 1.0)
        step = alpha * d
        r_try = rodrigues(step[:3]) @ rmat
        t_try = t + step[3:]
        h2, b2, c2, n2 = ev.normal_equations(r_try, t_try)
        evals += 1
        nw, nt = math.sqrt(float(step[:3] @ step[:3])), math.sqrt(float(step[3:] @ step[3:]))
        small = nw < TOL_ROT and nt < TOL_TRANS
        if n2 > 0 and c2 < c * (1.0 + ACCEPT_SLACK) and c2 <= c_start:
            rmat, t, hmat, b, c, n = r_try, t_try, h2, b2, c2, n2
            d_prev = d if lam <= LAMBDA0 else None
            lam = max(lam / 10.0, LAMBDA_MIN)
            if small:
                status = ST_CONVERGED
        else:
            lam *= 10.0
            alpha, d_prev = 1.0, None
            if small:
                status = ST_CONVERGED
            elif lam > LAMBDA_MAX:
                status = ST_LAMBDA
    return {"pose": np.concatenate([log_rotation(rmat), t]), "cost": c, "n_valid": n, "evals": evals,
            "status": status, "level": ev.level, "active": ev.active}


def refine_multi(pyramid, model, kmat, poses0: np.ndarray, max_evals: int = MAX_EVALS):
    """Multi-hypothesis selection (SURVEY.md 8a row A7): lowest index within SELECT_TIE of the lowest 2c/n."""
    runs = [refine(pyramid, model, kmat, p, max_evals) for p in poses0]
    return select(runs), runs


def select(runs) -> int:
    """Index of the winner among the results of refine() for the hypotheses of one frame (see refine_multi)."""
    score = np.array([2.0 * r["cost"] / r["n_valid"] if r["n_valid"] > 0 else np.inf for r in runs])
    if not np.isfinite(score).any():
        return 0
    return int(np.nonzero(score <= score.min() * (1.0 + SELECT_TIE))[0][0])
