"""CPU restatement of the reference's approximate-pose-estimation stage.

TEST INFRASTRUCTURE (see oracle/__init__.py).  Restates, with OpenCV underneath
exactly as the reference has it:

  * object points of a tag           transform_helper.py:41-96, detect_pose.py:405-437
  * the APE state machine            detect_pose.py:467-574
  * mean reprojection error gate     transform_helper.py:98-121
  * velocity / acceleration buffers  detect_pose.py:229-301
  * constant-acceleration predictor  detect_pose.py:303-349, transform_helper.py:123-259

Pinned against the unmodified reference by tests/test_oracle_ape.py (runs both
on the same seeded detections when /root/reference is mounted) and by the
golden vectors in tests/golden/ape_*.npz that ``make_golden.py`` generated from
the reference itself.

Quirks that are deliberately reproduced because a drop-in must show them:
cv2.solvePnP with useExtrinsicGuess=True writes its result INTO the guess
arrays (dtype preserved, so a float32 tvec guess yields a float32-rounded
tvec); ``extrinsic_guess`` aliases ``prev_transform`` after the first accepted
frame (detect_pose.py:551,569); the predictor composes the inverse-motion
"velocities" onto the previous pose (detect_pose.py:341); two float32 tvec
arrays are subtracted in float32; velocity buffers are not cleared on tracking
loss; exact zeros in a velocity raise ValueError (detect_pose.py:236-237), which
``step_given`` reports as an error flag.
"""
from __future__ import annotations

import copy
import math
from typing import List, Optional, Sequence, Tuple

import cv2 as cv
import numpy as np

MIN_TAGS = 2                 # detect_pose.py:494
MAX_MEAN_ERROR = 2.0         # detect_pose.py:539
DECISION_MARGIN_MIN = 50.0   # detect_pose.py:389
VEL_BUFFER = 2               # detect_pose.py:229


def tag_object_points(size: float, rvec_f32: np.ndarray, tvec_f32: np.ndarray) -> np.ndarray:
    """4 corners of one tag in the group frame; order (-,-),(-,+),(+,+),(+,-)
    (transform_helper.py:56-59); rotation from cv.Rodrigues of the float32 rvec
    (transform_helper.py:87); float64 result (transform_helper.py:90-94)."""
    h = size / 2.0
    base = np.array([-h, -h, 0.0, -h, h, 0.0, h, h, 0.0, h, -h, 0.0]).reshape(4, 3)
    rmat = cv.Rodrigues(rvec_f32)[0]
    return base @ rmat.T + tvec_f32.reshape(-1, 3)


def group_from_json(data: dict):
    """{tag_id: (size, tvec f32 (3,1), rvec f32 (3,1))} in JSON key order (detect_pose.py:122-139)."""
    out = {}
    for key, tag in data["tags"].items():
        out[int(key)] = (tag["size"],
                         np.array(tag["extrinsics"][:3], dtype=np.float32).reshape(3, 1),
                         np.array(tag["extrinsics"][-3:], dtype=np.float32).reshape(3, 1))
    return out


def filter_detections(dets, margins):
    """decision_margin < 50 is dropped (detect_pose.py:389-390)."""
    return [d for d, m in zip(dets, margins) if not (m < DECISION_MARGIN_MIN)]


def mean_reprojection_error(obj32, img32, rvec, tvec, mtx, dist):
    """Mean of per-point L2 pixel errors (transform_helper.py:106-119)."""
    proj, _ = cv.projectPoints(obj32, rvec, tvec, mtx, dist)
    proj = proj.reshape(-1, 2)
    return sum(np.linalg.norm(img32[i] - proj[i]) for i in range(len(proj))) / len(proj)


def euler_from_rotation(m):
    """transform_helper.py:239-259 (x,y,z with R = Rz Ry Rx)."""
    sy = math.sqrt(m[0, 0] * m[0, 0] + m[1, 0] * m[1, 0])
    if sy >= 1e-6:
        return np.array([math.atan2(m[2, 1], m[2, 2]), math.atan2(-m[2, 0], sy), math.atan2(m[1, 0], m[0, 0])])
    return np.array([math.atan2(-m[1, 2], m[1, 1]), math.atan2(-m[2, 0], sy), 0.0])


def rotation_from_euler(th):
    """transform_helper.py:215-236."""
    cx, sx, cy, sy, cz, sz = math.cos(th[0]), math.sin(th[0]), math.cos(th[1]), math.sin(th[1]), math.cos(th[2]), math.sin(th[2])
    rx = np.array([[1, 0, 0], [0, cx, -sx], [0, sx, cx]])
    ry = np.array([[cy, 0, sy], [0, 1, 0], [-sy, 0, cy]])
    rz = np.array([[cz, -sz, 0], [sz, cz, 0], [0, 0, 1]])
    return rz @ (ry @ rx)


def _homogeneous(rmat, tvec):
    return np.vstack((np.hstack((rmat, tvec)), np.array([0, 0, 0, 1])))     # transform_helper.py:134-138


class ApeOracle:
    """State machine of detect_pose.py:467-574 over lists of (tag_id, corners)."""

    def __init__(self, group: dict, mtx: np.ndarray, dist: Optional[np.ndarray], enhance_ape: bool = True):
        self.group = group
        self.mtx = mtx
        self.dist = dist
        self.enhance_ape = enhance_ape
        self.prev = (None, None)
        self.guess = (None, None)
        self.rot_vel: List[np.ndarray] = []
        self.tran_vel: List[np.ndarray] = []
        self.last_error = None      # mean reprojection error of the last solved frame
        self.last_accepted = False
        self.last_t64 = None

    # -- predictor --------------------------------------------------------
    def _velocities(self, curr, prev):
        rp = cv.Rodrigues(prev[0])[0]
        rc = cv.Rodrigues(curr[0])[0]
        tran = rc.T @ (prev[1] - curr[1])                 # detect_pose.py:279-280, transform_helper.py:184
        rot = rc.T @ rp                                   # detect_pose.py:283, transform_helper.py:207
        if not np.all(rot) or not np.all(tran):           # detect_pose.py:236-237
            raise ValueError("The rotational and translation velocities cannot be empty.")
        self.rot_vel.append(rot)
        self.tran_vel.append(tran)
        if len(self.rot_vel) > VEL_BUFFER:
            self.rot_vel.pop(0)
            self.tran_vel.pop(0)
        n = len(self.tran_vel)
        if n <= 1:
            return False, tran, rot, None, None
        tacc = self.rot_vel[n - 1].T @ (self.tran_vel[n - 2] - self.tran_vel[n - 1])   # detect_pose.py:293-296
        racc = self.rot_vel[n - 1].T @ self.rot_vel[n - 2]                              # detect_pose.py:297-299
        return True, tran, rot, tacc, racc

    def _predict(self, base, tran, tacc, rot, racc):
        half = rotation_from_euler(euler_from_rotation(racc) / 2)       # detect_pose.py:326-327
        rmat = cv.Rodrigues(base[0])[0]
        pred = _homogeneous(half, 0.5 * tacc) @ _homogeneous(rot, tran) @ _homogeneous(rmat, base[1])  # :334-341
        r_out = pred[0:3, 0:3]
        self.last_t64 = pred[0:3, 3].copy()                               # the predicted tvec before its float32 rounding
        t_out = np.array(pred[0:3, 3], dtype=np.float32).reshape(3, -1)  # transform_helper.py:158-159
        return cv.Rodrigues(r_out)[0], t_out

    # -- one frame ----------------------------------------------------------
    def step(self, dets: Sequence[Tuple[int, np.ndarray]]):
        """dets: accepted detections [(tag_id, corners (4,2))].  Mutates the state: solvePnP and the mean reprojection
        error (detect_pose.py:494-538), then ``step_given``."""
        self.last_error = None
        if len(dets) < MIN_TAGS:
            return self.step_given(len(dets), None, False, None)
        obj = np.array([tag_object_points(*self._sz_r_t(t)) for t, _ in dets], dtype=np.float32).reshape(-1, 3)
        img = np.array([np.asarray(c).reshape(1, 4, 2) for _, c in dets], dtype=np.float32).reshape(-1, 2)
        if self.guess[0] is None or not self.enhance_ape:
            ok, rvec, tvec = cv.solvePnP(obj, img, self.mtx, self.dist, flags=cv.SOLVEPNP_ITERATIVE)
        else:
            # (on copies of the guess arrays: step_given makes solvePnP's write into them, after it holds prev)
            ok, rvec, tvec = cv.solvePnP(obj, img, self.mtx, self.dist, self.guess[0].copy(), self.guess[1].copy(), True,
                                         flags=cv.SOLVEPNP_ITERATIVE)
        err = None
        if ok:
            err = mean_reprojection_error(obj, img, rvec, tvec, self.mtx, self.dist)
            self.last_error = float(err)
        return self.step_given(len(dets), (rvec, tvec), ok, err)

    def step_given(self, n_tags: int, pose, ok: bool, err) -> bool:
        """detect_pose.py:490-574 applied to a pose it is handed (what solvePnP, or the dense refinement, returned):
        n_tags accepted detections, pose (rvec, tvec) or 6 values, ok, err the mean reprojection error.  Mutates the
        state; sets ``last_accepted`` and returns the error flag: True where the reference raises ValueError on a
        zero entry in a velocity (detect_pose.py:236-237).  The state is then left as the reference held it when it
        raised: the guess arrays already overwritten, the velocities not appended, prev touched only through the
        aliased guess arrays; ``last_accepted`` is True (the pose passed the gate)."""
        held_prev = copy.deepcopy(self.prev)              # detect_pose.py:490
        self.last_accepted = False
        self.last_t64 = None
        if n_tags < MIN_TAGS:
            self.guess = (None, None)                     # detect_pose.py:573-574
            return False
        fresh = self.guess[0] is None or not self.enhance_ape
        if pose is not None and not isinstance(pose, tuple):
            pose = (np.asarray(pose, dtype=np.float64).reshape(6)[:3], np.asarray(pose, dtype=np.float64).reshape(6)[3:])
        if fresh:
            pose = (np.array(pose[0], dtype=np.float64).reshape(3, 1), np.array(pose[1], dtype=np.float64).reshape(3, 1))
        else:
            # solvePnP(useExtrinsicGuess=True) writes its result into the guess arrays, dtype preserved (a float32 tvec
            # after a prediction), and returns them; they are prev_transform's arrays too after a fresh solve
            self.guess[0][...] = np.asarray(pose[0]).reshape(self.guess[0].shape)
            self.guess[1][...] = np.asarray(pose[1]).reshape(self.guess[1].shape)
            pose = self.guess
        if not ok:
            return False                                   # detect_pose.py:533 (no else branch: state untouched)
        if not err < MAX_MEAN_ERROR:
            self.guess = (None, None)                      # detect_pose.py:570-572
            return False
        self.last_accepted = True
        if fresh:
            self.guess = pose                              # detect_pose.py:551
        else:
            try:
                good, tran, rot, tacc, racc = self._velocities(pose, held_prev)
            except ValueError:
                return True
            if good:
                self.guess = self._predict(held_prev, tran, tacc, rot, racc)   # detect_pose.py:558-566
        self.prev = pose                                   # detect_pose.py:569
        return False

    def state_record(self) -> np.ndarray:
        """The state as the device keeps it (AGT_STREAM_STATE_DOUBLES doubles, layout at the top of csrc/agt_ape.cu):
        has_prev, prev, has_guess, guess, guess aliases prev, guess tvec is float32, n_vel, rot/tran velocity slots
        (oldest first), prev tvec is float32 (slot 41), zeros beyond.  Without a guess its slots 8-15 are 0 (the device leaves them stale)."""
        s = np.zeros(64)
        if self.prev[0] is not None:
            s[0] = 1.0
            s[1:4], s[4:7] = np.ravel(self.prev[0]), np.ravel(self.prev[1])
        if self.guess[0] is not None:
            s[7] = 1.0
            s[8:11], s[11:14] = np.ravel(self.guess[0]), np.ravel(self.guess[1])
            s[14] = float(self.guess[0] is self.prev[0] and self.guess[1] is self.prev[1])
            s[15] = float(np.asarray(self.guess[1]).dtype == np.float32)
        if self.prev[0] is not None:
            s[41] = float(np.asarray(self.prev[1]).dtype == np.float32)
        s[16] = len(self.rot_vel)
        for k, (rot, tran) in enumerate(zip(self.rot_vel, self.tran_vel)):
            s[17 + 12 * k:26 + 12 * k] = np.ravel(rot)
            s[26 + 12 * k:29 + 12 * k] = np.ravel(tran)
        return s

    def _sz_r_t(self, tag_id):
        size, tvec, rvec = self.group[tag_id]
        return size, rvec, tvec

    def snapshot(self):
        def cp(t):
            return None if t[0] is None else (np.array(t[0], dtype=np.float64).reshape(3),
                                              np.array(t[1], dtype=np.float64).reshape(3))
        return {"prev": cp(self.prev), "guess": cp(self.guess), "n_vel": len(self.rot_vel)}
