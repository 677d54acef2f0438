"""``PoseDetector`` with the call surface of the reference class (detect_pose.py:28-714).

Same constructor, attributes (``prev_transform``, ``extrinsic_guess``, ``rot_velocities``,
``tran_velocities``, ``all_objpts``, ``extrinsics``, ``img``, ``draw_frame``) and per-frame
methods; the arithmetic the reference delegates to OpenCV on this path - solvePnP,
projectPoints - runs in libagt.so on the B200 (``cv_compat``), and the two stages the
reference names but does not yet contain can be switched on:

  ``use_lk``            inter-frame corner tracking (pyramidal LK, OpenCV-default semantics)
                        used when fewer than two tags are detected (SURVEY.md 3.4 / 9.2)
  ``use_dense_refine``  dense photometric refinement of every accepted pose before it becomes
                        ``prev_transform`` (SURVEY.md 9.4)
  ``pose_covariance``   with ``use_dense_refine``: after each frame ``self.pose_covariance`` holds the 6x6
                        covariance of the refined pose (rotation in radians first, then translation in
                        metres; ``HostContext.pose_covariance``), or None when the frame was not refined

Both default to False, which reproduces the reference's behaviour frame by frame,
including the in-place write of solvePnP into the guess arrays and the resulting
aliasing of ``extrinsic_guess`` and ``prev_transform``.  The frame ingest runs on the
device as well: ``process_frame`` is cv.undistort + crop (and keeps the gray image of the
result, computed in the same pass, for ``_detect_and_get_pose``), the gray conversion of
any other BGR frame is ``agt_bgr_to_gray`` - both bit-exact against cv2.  Tag detection uses the
host's ``apriltag`` module when there is one, exactly like the reference, and otherwise the device
detector behind the same surface (``apriltag_gpu``: quads from dark components, cornerSubPix, tag36h11
decoding; pinned to cv2.aruco in the tests).  Capture and drawing keep using ``cv2`` like the reference.

Cameras.  The reference passes (mtx, dist) to solvePnP / projectPoints even though the
frame it detects on has been undistorted and cropped by ``process_frame`` (detect_pose.py:
509-526 with :611-619); that is reproduced as it is.  Dense refinement reads pixels, so it
needs the camera the pixels were formed by: for a frame that came out of ``process_frame``
that is the new camera matrix of cv.getOptimalNewCameraMatrix with the principal point moved
by the crop offset and no distortion; for a frame handed in directly it is (mtx, no
distortion).  A distorted frame handed in directly cannot be refined and raises - it is
never skipped silently.
"""
import json
from copy import deepcopy
from pathlib import Path
from typing import Dict, List, Tuple

import numpy as np

from .. import cv_compat as agt_cv
from .. import synth
from .draw import Draw
from .transform_helper import TransformHelper

MIN_TAGS = 2               # detect_pose.py:494
MAX_MEAN_ERROR = 2         # detect_pose.py:539
MIN_DECISION_MARGIN = 50   # detect_pose.py:389


def bgr_to_gray(frame: np.ndarray) -> np.ndarray:
    """cv.cvtColor(frame, COLOR_BGR2GRAY) (detect_pose.py:602) in integer arithmetic:
    (B*3735 + G*19235 + R*9798 + 16384) >> 15, the fixed-point form OpenCV 4.x uses for 8-bit
    (checked bit-exact against cv2 in tests/test_cpu_host.py)."""
    f = frame.astype(np.uint32)
    return ((f[..., 0] * 3735 + f[..., 1] * 19235 + f[..., 2] * 9798 + 16384) >> 15).astype(np.uint8)


class PoseDetector(TransformHelper, Draw):
    DIRPATH = 'aprilgroup_tracking/aprilgroup_pose_estimation'
    JSON_FILE = 'april_group.json'

    def __init__(self, logger, mtx, dist, enhance_ape, use_lk: bool = False, use_dense_refine: bool = False,
                 surface_model=None, device: int = 0, pose_covariance: bool = False):
        TransformHelper.__init__(self, logger, mtx, dist)
        Draw.__init__(self, logger)
        self.logger = logger
        self.mtx = mtx
        self.dist = dist
        self.img = None
        self.draw_frame = None
        self.prev_transform = (None, None)
        self.extrinsic_guess = (None, None)
        self.rot_velocities: List[object] = []
        self.tran_velocities: List[object] = []
        self.enhance_ape = enhance_ape
        self.use_lk = use_lk
        self.use_dense_refine = use_dense_refine
        if pose_covariance and not use_dense_refine:
            raise ValueError("pose_covariance needs use_dense_refine: it is the covariance of the refined pose")
        self.want_pose_covariance = pose_covariance
        self.pose_covariance = None    # 6x6 covariance of the last frame's refined pose (want_pose_covariance)
        self._agt = agt_cv.default_context() if device == 0 else agt_cv.HostContext(device)   # raises without a B200
        self._gray = None
        self._prev_gray = None
        self._gray_mtx = None          # pinhole camera matrix of the pixels in self._gray (None: they are distorted)
        self._ingest = None            # (frame returned by process_frame, its gray image, its pinhole camera matrix)
        self._und_cache = {}           # (width, height) -> (new camera matrix, roi) of cv.getOptimalNewCameraMatrix
        self._prev_corners: List[Tuple[int, np.ndarray]] = []
        self._frame_corners: List[Tuple[int, np.ndarray]] = []
        try:
            import apriltag                      # the host's apriltag module, exactly as the reference (detect_pose.py:22)
        except ImportError:
            from .. import apriltag_gpu as apriltag      # not installed: the detector of csrc/agt_tags.cu behind the same surface
        self._apriltag = apriltag
        self.options = apriltag.DetectorOptions(families='tag36h11', border=1, nthreads=4, quad_decimate=1.0,
                                                quad_blur=0.0, refine_edges=True, refine_decode=False,
                                                refine_pose=True, debug=False, quad_contours=True)
        self.extrinsics = self.get_extrinsics()
        self.all_objpts = self.get_all_points(self.extrinsics)
        if use_dense_refine:
            model = surface_model if surface_model is not None else synth.surface_model() + (synth.model_pitch(),)
            self._agt.set_model(*model)

    # ------------------------------------------------------------------------------------
    # AprilGroup geometry (detect_pose.py:105-145, 185-227)
    # ------------------------------------------------------------------------------------
    def get_extrinsics(self) -> Dict:
        path = Path(self.DIRPATH) / self.JSON_FILE
        try:
            with open(path, "r") as fh:
                data = json.load(fh)
        except IOError as err:
            raise IOError("The filepath: {} does not exist.".format(path)) from err
        table: Dict = {}
        for key, tag in data['tags'].items():          # JSON key order defines the corner indexing
            tvec = np.array(tag['extrinsics'][:3], dtype=np.float32).reshape((3, 1))
            rvec = np.array(tag['extrinsics'][-3:], dtype=np.float32).reshape((3, 1))
            self.add_values_in_dict(table, int(key), [tag['size'], tvec, rvec])
        self.logger.info('Successfully Loaded AprilGroup Extrinsics!')
        return table

    def _tag_object_points(self, tag_id: int) -> np.ndarray:
        size, tvec, rvec = self.extrinsics[tag_id][0], self.extrinsics[tag_id][1], self.extrinsics[tag_id][2]
        return self.transform_marker_corners(self.get_initial_pts(size), (rvec, tvec))

    def get_all_points(self, extrinsics: Dict) -> np.ndarray:
        if not any(extrinsics):
            raise ValueError("The extrinsic matrix must be supplied.")
        pts = [self.transform_marker_corners(self.get_initial_pts(v[0]), (v[2], v[1])) for v in extrinsics.values()]
        self.logger.info('Successfully Obtained Aprilgroup Object Points!')
        return np.array(pts).reshape(-1, 3)

    # ------------------------------------------------------------------------------------
    # motion predictor (detect_pose.py:229-349)
    # ------------------------------------------------------------------------------------
    def _update_buffers(self, rot_vel: np.ndarray, tran_vel: np.ndarray, buf_size: int = 2) -> None:
        if not np.all(rot_vel) or not np.all(tran_vel):
            raise ValueError("The rotational and translation velocities cannot be empty.")
        self.rot_velocities.append(rot_vel)
        self.tran_velocities.append(tran_vel)
        if len(self.rot_velocities) > buf_size:
            del self.rot_velocities[0]
            del self.tran_velocities[0]

    def get_pose_vel_acc(self, curr_transform, prev_transform):
        prev_rmat = agt_cv.Rodrigues(prev_transform[0])[0]
        curr_rmat = agt_cv.Rodrigues(curr_transform[0])[0]
        tran_vel = self.get_relative_trans(curr_rmat, curr_transform[1], prev_transform[1])
        rot_vel = self.get_relative_rot(prev_rmat, curr_rmat)
        self._update_buffers(rot_vel, tran_vel)
        n = len(self.tran_velocities)
        if n <= 1:
            return False, tran_vel, rot_vel, 0.0, 0.0
        tran_acc = self.get_relative_trans(self.rot_velocities[n - 1], self.tran_velocities[n - 1], self.tran_velocities[n - 2])
        rot_acc = self.get_relative_rot(self.rot_velocities[n - 2], self.rot_velocities[n - 1])
        return True, tran_vel, rot_vel, tran_acc, rot_acc

    def apply_vel_acc(self, transformation, tran_vel, tran_acc, rot_vel, rot_acc):
        half_acc = self.euler_angles_to_rotation_matrix(self.rotation_matrix_to_euler_angles(rot_acc) / 2)
        rmat = agt_cv.Rodrigues(transformation[0])[0]
        pred = (self.get_extrinsic_matrix(half_acc, 0.5 * tran_acc)
                @ self.get_extrinsic_matrix(rot_vel, tran_vel)
                @ self.get_extrinsic_matrix(rmat, transformation[1]))
        rmat_pose, tvec_pose = self.get_rmat_tvec(pred)
        return agt_cv.Rodrigues(rmat_pose)[0], tvec_pose

    # ------------------------------------------------------------------------------------
    # detections (detect_pose.py:351-439)
    # ------------------------------------------------------------------------------------
    def _lists_from_detections(self, detections):
        """Filter + tag-id -> object-point mapping of detect_pose.py:385-437."""
        img_list, obj_list, ids = [], [], []
        self._frame_corners = []
        for det in detections:
            if det.decision_margin < MIN_DECISION_MARGIN:
                continue
            corners = np.asarray(det.corners)
            if self.img is not None:
                self.draw_corners(self.img, det)
            objpts = self._tag_object_points(det.tag_id)      # KeyError on unknown ids, like the reference
            img_list.append(corners.reshape(1, 4, 2))
            obj_list.append(objpts)
            ids.append(det.tag_id)
            self._frame_corners.append((det.tag_id, corners.reshape(4, 2).astype(np.float64)))
        return img_list, obj_list, ids

    def _obtain_detections(self, gray: np.ndarray):
        detector = self._apriltag.Detector(self.options)
        results, _ = detector.detect(gray, return_image=True)
        self.logger.info('Detected %d tags.', len(results))
        if not results or self.mtx is None:
            self._frame_corners = []
            return [], [], []
        return self._lists_from_detections(results)

    def _track_lost_tags(self, imgpoints_arr, objpoints_arr, tag_ids):
        """Stage 2: when < 2 tags are detected, follow the previous frame's accepted corners with
        pyramidal LK and re-admit every tag whose four corners were all tracked (status 1)."""
        if self._prev_gray is None or not self._prev_corners or self._gray.shape != self._prev_gray.shape:
            return imgpoints_arr, objpoints_arr, tag_ids
        have = set(tag_ids)
        todo = [(t, c) for t, c in self._prev_corners if t not in have]
        if not todo:
            return imgpoints_arr, objpoints_arr, tag_ids
        pts = np.concatenate([c for _, c in todo]).astype(np.float32)
        nxt, status, _ = self._agt.calcOpticalFlowPyrLK(self._prev_gray, self._gray, pts.reshape(-1, 1, 2), None)
        nxt, status = nxt.reshape(-1, 4, 2), status.reshape(-1, 4)
        for (tag_id, _), corners, st in zip(todo, nxt, status):
            if st.all():
                imgpoints_arr.append(corners.reshape(1, 4, 2).astype(np.float64))
                objpoints_arr.append(self._tag_object_points(tag_id))
                tag_ids.append(tag_id)
                self._frame_corners.append((tag_id, corners.astype(np.float64)))
        return imgpoints_arr, objpoints_arr, tag_ids

    # ------------------------------------------------------------------------------------
    # stage 1 (+3): detect_pose.py:441-574
    # ------------------------------------------------------------------------------------
    def _project_draw_points(self, transformation) -> None:
        imgpts, _ = agt_cv.projectPoints(self.all_objpts, transformation[0], transformation[1], self.mtx, self.dist)
        self.draw_squares_and_3d_pts(self.img, self.draw_frame, imgpts)

    def _estimate_pose(self, imgpoints_arr, objpoints_arr) -> None:
        held_prev = deepcopy(self.prev_transform)       # solvePnP overwrites the aliased guess arrays
        accepted = False
        if imgpoints_arr and objpoints_arr and len(imgpoints_arr) >= MIN_TAGS:
            obj = np.array(objpoints_arr, dtype=np.float32).reshape(-1, 3)
            img = np.array(imgpoints_arr, dtype=np.float32).reshape(-1, 2)
            fresh = self.extrinsic_guess[0] is None or not self.enhance_ape
            if fresh:
                ok, rvec, tvec = self._agt.solvePnP(obj, img, self.mtx, self.dist, flags=agt_cv.SOLVEPNP_ITERATIVE)
            else:
                ok, rvec, tvec = self._agt.solvePnP(obj, img, self.mtx, self.dist, self.extrinsic_guess[0],
                                                    self.extrinsic_guess[1], True, flags=agt_cv.SOLVEPNP_ITERATIVE)
            transformation = (rvec, tvec)
            if ok:
                mean_error = self.get_reprojection_error(obj, img, transformation)
                self.logger.info("Mean error: %s", mean_error)
                if mean_error < MAX_MEAN_ERROR:
                    accepted = True
                    if self.use_dense_refine and self._gray is not None:
                        self._refine_in_place(transformation)
                    self._project_draw_points(transformation)
                    if fresh:
                        self.extrinsic_guess = transformation
                    else:
                        good, tran_vel, rot_vel, tran_acc, rot_acc = self.get_pose_vel_acc(transformation, held_prev)
                        if good:
                            self.extrinsic_guess = self.apply_vel_acc(held_prev, tran_vel, tran_acc, rot_vel, rot_acc)
                    self.prev_transform = transformation
                else:
                    self.extrinsic_guess = (None, None)
        else:
            self.extrinsic_guess = (None, None)
        self._prev_corners = list(self._frame_corners) if accepted else []

    def _refine_in_place(self, transformation) -> None:
        """Stage 3: dense photometric refinement; the result replaces the PnP pose inside the same arrays."""
        if self._gray_mtx is None:
            raise ValueError("use_dense_refine: this frame carries lens distortion (dist != 0) and did not come out of "
                             "process_frame(); dense refinement needs undistorted pixels - pass frames through process_frame() "
                             "first, as the reference's capture loop does (detect_pose.py:678)")
        ok, rvec, tvec, _, _ = self._agt.refine_pose(self._gray, transformation[0], transformation[1], self._gray_mtx)
        if ok:
            if self.want_pose_covariance:
                init = np.concatenate([np.asarray(v, dtype=np.float64).reshape(3) for v in transformation])
                pose = np.concatenate([rvec.reshape(3), tvec.reshape(3)])
                self.pose_covariance = self._agt.pose_covariance(self._gray, init, pose, self._gray_mtx)["cov"][0, 0]
            transformation[0].reshape(-1)[:] = rvec.reshape(-1)
            transformation[1].reshape(-1)[:] = tvec.reshape(-1)

    # ------------------------------------------------------------------------------------
    # per-frame entry points (detect_pose.py:147-183, 576-619)
    # ------------------------------------------------------------------------------------
    def _has_distortion(self) -> bool:
        return self.dist is not None and bool(np.any(np.asarray(self.dist) != 0))

    def _set_gray(self, frame: np.ndarray) -> np.ndarray:
        """Gray image of the frame (detect_pose.py:602) and the pinhole camera its pixels were formed by."""
        if self._ingest is not None and frame is self._ingest[0]:
            gray, mtx = self._ingest[1], self._ingest[2]           # undistorted + converted in one pass by process_frame
        else:
            gray = self._agt.bgr_to_gray(frame) if frame.ndim == 3 else frame
            mtx = None if self._has_distortion() else self.mtx
        self._prev_gray, self._gray, self._gray_mtx = self._gray, gray, mtx
        return gray

    def _detect_and_get_pose(self, frame: np.ndarray) -> None:
        self.img = frame
        self.pose_covariance = None
        height, width = frame.shape[:2]
        self.draw_frame = np.zeros(shape=[height, width, 3], dtype=np.uint8)
        gray = self._set_gray(frame)
        imgpoints_arr, objpoints_arr, tag_ids = self._obtain_detections(gray)
        if self.use_lk and len(imgpoints_arr) < MIN_TAGS:
            imgpoints_arr, objpoints_arr, tag_ids = self._track_lost_tags(imgpoints_arr, objpoints_arr, tag_ids)
        self._estimate_pose(imgpoints_arr, objpoints_arr)

    def undistort_frame(self, frame: np.ndarray) -> np.ndarray:
        """detect_pose.py:147-183: cv.getOptimalNewCameraMatrix (host, 3x3 algebra, once per frame size), then cv.undistort +
        crop on the device; the gray image of the result comes out of the same pass and waits for _detect_and_get_pose."""
        height, width = frame.shape[:2]
        if (width, height) not in self._und_cache:
            import cv2 as cv
            self._und_cache[(width, height)] = cv.getOptimalNewCameraMatrix(self.mtx, self.dist, (width, height), 1, (width, height))
        new_mtx, roi = self._und_cache[(width, height)]
        out, gray = self._agt.undistort_frame(frame, self.mtx, self.dist, new_mtx, roi)
        pinhole = np.array(new_mtx, dtype=np.float64)
        pinhole[0, 2] -= roi[0]
        pinhole[1, 2] -= roi[1]
        self._ingest = (out, gray, pinhole)
        return out

    def process_frame(self, frame: np.ndarray) -> np.ndarray:
        return self.undistort_frame(frame) if self.dist is not None else frame

    def overlay_camera(self) -> None:
        """Capture/display loop of detect_pose.py:621-714 (camera + GUI: outside the accelerated path)."""
        import cv2 as cv
        cv.namedWindow('Camera')
        cap = cv.VideoCapture("/dev/video2", cv.CAP_V4L2)
        if not cap.isOpened():
            raise OSError("Error opening webcam, please check that the webcam is connected and the correct one is referenced.")
        cap.set(3, 1280)
        cap.set(4, 720)
        while True:
            ok, frame = cap.read()
            if not ok:
                break
            frame = self.process_frame(frame)
            self._detect_and_get_pose(frame)
            cv.imshow('Camera', self.img)
            cv.imshow('image', self.draw_frame)
            if cv.waitKey(1) == 27:
                cv.destroyAllWindows()
                break
