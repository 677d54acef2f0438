"""OpenCV-shaped host API over libagt.so (numpy in, numpy out, no torch needed).

These are the calls the reference's hot path makes into OpenCV, with the same
signatures, shapes, dtypes and mutation conventions (SURVEY.md 8b), executed by
the CUDA kernels through the ``*_host`` entry points of the C ABI:

  solvePnP              detect_pose.py:509-526   (SOLVEPNP_ITERATIVE only)
  projectPoints         detect_pose.py:455, transform_helper.py:106
  Rodrigues             detect_pose.py:275-276,330,344, transform_helper.py:87
  calcOpticalFlowPyrLK  (stage 2, absent from the snapshot; OpenCV defaults)
  pyrDown / Scharr / buildOpticalFlowPyramid   (pyramid the LK stage is defined on)
  refine_pose           (stage 3, dense photometric refinement)

No CPU fallback: constructing the context raises if libagt.so or a B200 is missing.
"""
from __future__ import annotations

import ctypes as C
import math
from typing import Optional, Tuple

import numpy as np

from . import _lib, synth

SOLVEPNP_ITERATIVE = 0
_F32P = C.POINTER(C.c_float)


class HostContext:
    """One libagt context driven with host (numpy) buffers."""

    def __init__(self, device: int = 0):
        self.lib = _lib.load()
        h = C.c_void_p()
        rc = self.lib.agt_create(int(device), C.byref(h))
        if rc != _lib.AGT_OK:
            msg = self.lib.agt_last_error(None)
            raise RuntimeError(f"agt_create failed ({rc}): {msg.decode() if msg else ''}")
        self.h = h
        self._cam_key = None
        self._model_set = False

    def close(self):
        if getattr(self, "h", None):
            self.lib.agt_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        _lib.check(self.h, rc)

    def launch_count(self) -> int:
        return int(self.lib.agt_launch_count(self.h))

    # -- configuration ----------------------------------------------------------------
    def use_camera(self, mtx, dist) -> None:
        k = np.ascontiguousarray(np.asarray(mtx, dtype=np.float64).reshape(9))
        d = None if dist is None else np.ascontiguousarray(np.asarray(dist, dtype=np.float64).reshape(-1))
        key = (k.tobytes(), None if d is None else d.tobytes())
        if key == self._cam_key:
            return
        if d is not None and d.size not in (4, 5):
            raise ValueError("distortion must hold 4 or 5 coefficients (k1 k2 p1 p2 [k3])")
        self._check(self.lib.agt_set_camera(self.h, k.ctypes.data_as(C.POINTER(C.c_double)),
                                            d.ctypes.data_as(C.POINTER(C.c_double)) if d is not None else None,
                                            0 if d is None else int(d.size)))
        self._cam_key = key

    def set_model(self, samples, sample_tag, normals, centres, pitch) -> None:
        s = np.ascontiguousarray(samples, dtype=np.float32)
        tg = np.ascontiguousarray(sample_tag, dtype=np.uint8)
        n = np.ascontiguousarray(normals, dtype=np.float32)
        c = np.ascontiguousarray(centres, dtype=np.float32)
        self._check(self.lib.agt_set_model(self.h, s.ctypes.data, tg.ctypes.data, int(s.shape[0]), n.ctypes.data, c.ctypes.data,
                                           int(n.shape[0]), float(pitch)))
        self._model_set = True

    # -- stage 1 ------------------------------------------------------------------------
    def solvePnP(self, objectPoints, imagePoints, cameraMatrix, distCoeffs, rvec=None, tvec=None,
                 useExtrinsicGuess=False, flags=SOLVEPNP_ITERATIVE):
        if flags != SOLVEPNP_ITERATIVE:
            raise ValueError("only SOLVEPNP_ITERATIVE is implemented (the flag the reference uses)")
        obj = np.ascontiguousarray(np.asarray(objectPoints, dtype=np.float32).reshape(-1, 3))
        img = np.ascontiguousarray(np.asarray(imagePoints, dtype=np.float32).reshape(-1, 2))
        if obj.shape[0] != img.shape[0]:
            raise ValueError("objectPoints and imagePoints differ in length")
        self.use_camera(cameraMatrix, distCoeffs)
        pose = np.zeros(6, dtype=np.float64)
        if useExtrinsicGuess:
            if rvec is None or tvec is None:
                raise ValueError("useExtrinsicGuess=True needs rvec and tvec")
            pose[:3] = np.asarray(rvec, dtype=np.float64).reshape(3)
            pose[3:] = np.asarray(tvec, dtype=np.float64).reshape(3)
        ok = C.c_int(0)
        err = C.c_float(0.0)
        self._check(self.lib.agt_solve_pnp_host(self.h, obj.ctypes.data, img.ctypes.data, int(obj.shape[0]),
                                                int(bool(useExtrinsicGuess)), pose.ctypes.data, C.byref(ok), C.byref(err)))
        self.last_reprojection_error = float(err.value)
        if useExtrinsicGuess and isinstance(rvec, np.ndarray) and isinstance(tvec, np.ndarray):
            # OpenCV writes the result into the caller's guess arrays and returns them (dtype preserved)
            rvec.reshape(-1)[:] = pose[:3]
            tvec.reshape(-1)[:] = pose[3:]
            return bool(ok.value), rvec, tvec
        return bool(ok.value), pose[:3].reshape(3, 1).copy(), pose[3:].reshape(3, 1).copy()

    def projectPoints(self, objectPoints, rvec, tvec, cameraMatrix, distCoeffs):
        src = np.asarray(objectPoints)
        obj = np.ascontiguousarray(src.astype(np.float32).reshape(-1, 3))
        self.use_camera(cameraMatrix, distCoeffs)
        pose = np.concatenate([np.asarray(rvec, dtype=np.float64).reshape(3), np.asarray(tvec, dtype=np.float64).reshape(3)])
        out = np.zeros((obj.shape[0], 2), dtype=np.float64)
        self._check(self.lib.agt_project_host(self.h, obj.ctypes.data, int(obj.shape[0]), pose.ctypes.data, out.ctypes.data))
        # cv.projectPoints returns the depth of objectPoints
        out_dtype = np.float32 if src.dtype == np.float32 else np.float64
        return out.astype(out_dtype).reshape(-1, 1, 2), None

    # -- stage 2 ------------------------------------------------------------------------
    @staticmethod
    def _levels_for(w: int, h: int, max_level: int, win=21) -> int:
        # cv::buildOpticalFlowPyramid stops before a level that is not larger than the window
        levels = 1
        while levels <= max_level:
            w, h = (w + 1) // 2, (h + 1) // 2
            if w <= win or h <= win:
                break
            levels += 1
        return levels

    def calcOpticalFlowPyrLK(self, prevImg, nextImg, prevPts, nextPts=None, winSize=(21, 21), maxLevel=3,
                             criteria=(3, 30, 0.01), flags=0, minEigThreshold=1e-4):
        if tuple(winSize) != (21, 21) or tuple(criteria) != (3, 30, 0.01) or flags != 0 or minEigThreshold != 1e-4:
            raise ValueError("only the OpenCV defaults (21x21, COUNT+EPS 30/0.01, flags 0, minEig 1e-4) are implemented")
        if maxLevel < 0 or maxLevel > _lib.AGT_MAX_LEVELS - 1:
            raise ValueError("maxLevel must be 0..3")
        a = np.ascontiguousarray(prevImg, dtype=np.uint8)
        b = np.ascontiguousarray(nextImg, dtype=np.uint8)
        if a.ndim != 2 or a.shape != b.shape:
            raise ValueError("prevImg/nextImg must be single-channel images of equal size")
        pts = np.ascontiguousarray(np.asarray(prevPts, dtype=np.float32).reshape(-1, 2))
        n = int(pts.shape[0])
        out = np.zeros((n, 2), np.float32)
        st = np.zeros(n, np.uint8)
        err = np.zeros(n, np.float32)
        h, w = a.shape
        levels = self._levels_for(w, h, maxLevel)
        self._check(self.lib.agt_lk_host(self.h, a.ctypes.data, b.ctypes.data, w, h, levels, pts.ctypes.data, n,
                                         out.ctypes.data, st.ctypes.data, err.ctypes.data))
        return out.reshape(-1, 1, 2), st.reshape(-1, 1), err.reshape(-1, 1)

    def pyramid(self, img, levels: int = 4):
        a = np.ascontiguousarray(img, dtype=np.uint8)
        h, w = a.shape
        outs = [a]
        ptrs = (C.c_void_p * levels)()
        for l in range(1, levels):
            w, h = (w + 1) // 2, (h + 1) // 2
            outs.append(np.zeros((h, w), np.uint8))
            ptrs[l] = outs[l].ctypes.data
        self._check(self.lib.agt_pyramid_host(self.h, a.ctypes.data, a.shape[1], a.shape[0], levels, ptrs))
        return outs

    def pyrDown(self, img):
        return self.pyramid(img, 2)[1]

    def Scharr(self, img):
        """-> (H,W,2) int16 interleaved (dx,dy)."""
        a = np.ascontiguousarray(img, dtype=np.uint8)
        out = np.zeros(a.shape + (2,), np.int16)
        self._check(self.lib.agt_scharr_host(self.h, a.ctypes.data, a.shape[1], a.shape[0], out.ctypes.data))
        return out

    def buildOpticalFlowPyramid(self, img, winSize=(21, 21), maxLevel=3, withDerivatives=True):
        a = np.ascontiguousarray(img, dtype=np.uint8)
        levels = self._levels_for(a.shape[1], a.shape[0], maxLevel, winSize[0])
        lv = self.pyramid(a, levels)
        out = []
        for l in lv:
            out.append(l)
            if withDerivatives:
                out.append(self.Scharr(l))
        return levels - 1, out

    # -- corner refinement (N3, first step) ---------------------------------------------
    def cornerSubPix(self, image, corners, winSize, zeroZone=(-1, -1), criteria=(3, 30, 0.001)):
        """cv.cornerSubPix(image, corners, winSize, zeroZone, criteria): corners [N,1,2] / [N,2] float32 are refined IN PLACE and
        returned, as OpenCV does.  Square windows of half-size 1..7, no zero zone, 8-bit single-channel images."""
        if tuple(zeroZone) != (-1, -1):
            raise ValueError("only zeroZone=(-1, -1) is implemented")
        if winSize[0] != winSize[1]:
            raise ValueError("only square windows are implemented")
        img = np.ascontiguousarray(image, dtype=np.uint8)
        if img.ndim != 2:
            raise ValueError("image must be single-channel")
        if not (isinstance(corners, np.ndarray) and corners.dtype == np.float32 and corners.flags.c_contiguous):
            raise ValueError("corners must be a C-contiguous float32 array (it is refined in place)")
        kind, count, eps = criteria
        max_iters = int(count) if (kind & 1) else 100
        eps = float(eps) if (kind & 2) else 0.0
        self._check(self.lib.agt_corner_subpix_host(self.h, C.c_void_p(img.ctypes.data), int(img.shape[1]), int(img.shape[0]),
                                                    C.c_void_p(corners.ctypes.data), int(corners.size // 2), int(winSize[0]),
                                                    max(1, max_iters), max(eps, 0.0)))
        return corners

    # -- tag detection (N3) --------------------------------------------------------------
    def set_tag_threshold(self, mode="auto"):
        """"auto" / "window" / "local": see Context.set_tag_threshold (a whole frame, which is what detect_tags takes, uses the
        local white level unless told otherwise)."""
        self._check(self.lib.agt_set_tag_threshold(self.h, {"auto": 0, "window": 1, "local": 2}[mode] if isinstance(mode, str) else int(mode)))

    def detect_tags(self, gray, max_tags: int = 64, max_hamming: int = 2, refine_win: int = 4):
        """-> list of (tag_id, corners (4,2) float64 in the reference's corner order, decision margin, hamming) of a gray frame."""
        img = np.ascontiguousarray(gray, dtype=np.uint8)
        if img.ndim != 2:
            raise ValueError("gray must be a single-channel image")
        if not getattr(self, "_tag_family", False):
            codes = np.ascontiguousarray(synth.TAG36H11_CODES, dtype=np.uint64)
            self._check(self.lib.agt_set_tag_family(self.h, codes.ctypes.data, int(codes.size)))
            self._tag_family = True
        n = C.c_int32(0)
        ids = np.zeros(max_tags, np.int32)
        corners = np.zeros((max_tags, 4, 2), np.float32)
        margin = np.zeros(max_tags, np.float32)
        ham = np.zeros(max_tags, np.uint8)
        self._check(self.lib.agt_detect_tags_host(self.h, C.c_void_p(img.ctypes.data), int(img.shape[1]), int(img.shape[0]), int(max_tags),
                                                  int(max_hamming), int(refine_win), C.byref(n), C.c_void_p(ids.ctypes.data),
                                                  C.c_void_p(corners.ctypes.data), C.c_void_p(margin.ctypes.data), C.c_void_p(ham.ctypes.data)))
        k = min(int(n.value), max_tags)
        order = np.argsort(ids[:k], kind="stable")
        return [(int(ids[i]), corners[i].astype(np.float64), float(margin[i]), int(ham[i])) for i in order]

    # -- frame ingest -------------------------------------------------------------------
    def undistort_gray(self, frame, cameraMatrix, distCoeffs, newCameraMatrix, roi):
        """cv.cvtColor(cv.undistort(frame, K, dist, None, newK)[y:y+h, x:x+w], COLOR_BGR2GRAY) in one device pass:
        the reference's undistort_frame (detect_pose.py:147-183) followed by the gray conversion (detect_pose.py:602),
        bit-exact for 8-bit frames.  frame [H,W,3] BGR or [H,W] gray; roi = (x, y, w, h) of getOptimalNewCameraMatrix."""
        src = np.ascontiguousarray(frame, dtype=np.uint8)
        if src.ndim not in (2, 3) or (src.ndim == 3 and src.shape[2] != 3):
            raise ValueError("frame must be [H,W] or [H,W,3] uint8")
        self.use_camera(cameraMatrix, distCoeffs)
        h, w = int(src.shape[0]), int(src.shape[1])
        x, y, rw, rh = (int(v) for v in roi)
        k = np.ascontiguousarray(newCameraMatrix, dtype=np.float64).reshape(9)
        key = (k.tobytes(), w, h, x, y, rw, rh, self._cam_key)
        if key != getattr(self, "_und_key", None):
            self._check(self.lib.agt_set_undistort(self.h, k.ctypes.data_as(C.POINTER(C.c_double)), w, h, x, y, rw, rh))
            self._und_key = key
        out = np.empty((rh, rw), dtype=np.uint8)
        self._check(self.lib.agt_undistort_to_gray_host(self.h, C.c_void_p(src.ctypes.data), w, h, 1 if src.ndim == 2 else 3,
                                                        C.c_void_p(out.ctypes.data)))
        return out

    def undistort_frame(self, frame, cameraMatrix, distCoeffs, newCameraMatrix, roi):
        """The reference's undistort_frame (detect_pose.py:147-183) with ONE upload of the frame: -> (cv.undistort(frame, K, dist,
        None, newK)[y:y+h, x:x+w], its cv.cvtColor(.., COLOR_BGR2GRAY)), both bit-exact for 8-bit frames.  The first is what
        process_frame returns (the reference draws on it and shows it), the second is what the tracking stages read."""
        src = np.ascontiguousarray(frame, dtype=np.uint8)
        if src.ndim not in (2, 3) or (src.ndim == 3 and src.shape[2] != 3):
            raise ValueError("frame must be [H,W] or [H,W,3] uint8")
        self.use_camera(cameraMatrix, distCoeffs)
        h, w = int(src.shape[0]), int(src.shape[1])
        x, y, rw, rh = (int(v) for v in roi)
        k = np.ascontiguousarray(newCameraMatrix, dtype=np.float64).reshape(9)
        key = (k.tobytes(), w, h, x, y, rw, rh, self._cam_key)
        if key != getattr(self, "_und_key", None):
            self._check(self.lib.agt_set_undistort(self.h, k.ctypes.data_as(C.POINTER(C.c_double)), w, h, x, y, rw, rh))
            self._und_key = key
        ch = 1 if src.ndim == 2 else 3
        out = np.empty((rh, rw) if ch == 1 else (rh, rw, 3), dtype=np.uint8)
        gray = np.empty((rh, rw), dtype=np.uint8)
        self._check(self.lib.agt_undistort_frame_host(self.h, C.c_void_p(src.ctypes.data), w, h, ch, C.c_void_p(out.ctypes.data),
                                                      C.c_void_p(gray.ctypes.data)))
        return out, gray

    def bgr_to_gray(self, frame):
        """cv.cvtColor(frame, cv.COLOR_BGR2GRAY) (detect_pose.py:602), bit-exact for 8-bit frames."""
        src = np.ascontiguousarray(frame, dtype=np.uint8)
        if src.ndim != 3 or src.shape[2] != 3:
            raise ValueError("frame must be [H,W,3] uint8")
        out = np.empty(src.shape[:2], dtype=np.uint8)
        self._check(self.lib.agt_bgr_to_gray_host(self.h, C.c_void_p(src.ctypes.data), int(src.shape[1]), int(src.shape[0]),
                                                  C.c_void_p(out.ctypes.data)))
        return out

    def set_roi_upload(self, enable: bool) -> None:
        self._check(self.lib.agt_set_roi_upload(self.h, int(bool(enable))))

    def set_upload_threads(self, threads: int) -> None:
        """Host threads that pack the rectangles of PAGEABLE frames into pinned staging (0: one 2-D copy per frame)."""
        self._check(self.lib.agt_set_upload_threads(self.h, int(threads)))

    def last_h2d_bytes(self) -> int:
        return int(self.lib.agt_last_h2d_bytes(self.h))

    # -- stage 3 ------------------------------------------------------------------------
    def refine_poses(self, frames, init, cameraMatrix, n_hyp: int = 1, levels: int = 4):
        """frames [B,H,W] u8 (host; pinned memory recommended), init [B,n_hyp,6] f64.
        -> dict(pose [B,n_hyp,6], cost, n_valid, evals, status, best [B] or None)."""
        if not self._model_set:
            raise RuntimeError("set_model() must be called before refine_poses()")
        self.use_camera(cameraMatrix, None)
        fr = frames if (isinstance(frames, np.ndarray) and frames.dtype == np.uint8 and frames.flags.c_contiguous) else \
            np.ascontiguousarray(frames, dtype=np.uint8)
        if fr.ndim == 2:
            fr = fr[None]
        b, h, w = fr.shape
        ini = np.ascontiguousarray(np.asarray(init, dtype=np.float64).reshape(b, n_hyp, 6))
        pose = np.zeros_like(ini)
        cost = np.zeros((b, n_hyp), np.float32)
        nv = np.zeros((b, n_hyp), np.int32)
        ev = np.zeros((b, n_hyp), np.int32)
        st = np.zeros((b, n_hyp), np.uint8)
        best = np.zeros(b, np.int32) if n_hyp > 1 else None
        self._check(self.lib.agt_refine_host(self.h, fr.ctypes.data, w, h, levels, b, ini.ctypes.data, n_hyp, pose.ctypes.data,
                                             cost.ctypes.data, nv.ctypes.data, ev.ctypes.data, st.ctypes.data,
                                             best.ctypes.data if best is not None else None))
        return {"pose": pose, "cost": cost, "n_valid": nv, "evals": ev, "status": st, "best": best}

    def pose_covariance(self, frames, init, pose, cameraMatrix, n_hyp: int = 1, levels: int = 4):
        """Covariance of refined poses (agt_pose_covariance_host): frames [B,H,W] u8 (host, whole frames are uploaded), init /
        pose [B,n_hyp,6] f64 - the refinement's start, which fixes its cost function, and the pose to evaluate at.
        -> dict(cov [B,n_hyp,6,6] = s^2 H^-1, info [B,n_hyp,6,6] = H, sigma2 [B,n_hyp] f32, n_valid [B,n_hyp] i32, ok [B,n_hyp] bool);
        rotation (radians) before translation (metres); cov is NaN where ok is False."""
        if not self._model_set:
            raise RuntimeError("set_model() must be called before pose_covariance()")
        self.use_camera(cameraMatrix, None)
        fr = np.ascontiguousarray(frames, dtype=np.uint8)
        if fr.ndim == 2:
            fr = fr[None]
        b, h, w = fr.shape
        ini = np.ascontiguousarray(np.asarray(init, dtype=np.float64).reshape(b, n_hyp, 6))
        ps = np.ascontiguousarray(np.asarray(pose, dtype=np.float64).reshape(b, n_hyp, 6))
        cov = np.zeros((b, n_hyp, 6, 6), np.float64)
        info = np.zeros((b, n_hyp, 6, 6), np.float64)
        s2 = np.zeros((b, n_hyp), np.float32)
        nv = np.zeros((b, n_hyp), np.int32)
        ok = np.zeros((b, n_hyp), np.uint8)
        self._check(self.lib.agt_pose_covariance_host(self.h, fr.ctypes.data, w, h, levels, b, ini.ctypes.data, ps.ctypes.data, n_hyp,
                                                      cov.ctypes.data, info.ctypes.data, s2.ctypes.data, nv.ctypes.data, ok.ctypes.data))
        return {"cov": cov, "info": info, "sigma2": s2, "n_valid": nv, "ok": ok.astype(bool)}

    def refine_pose(self, gray, rvec, tvec, cameraMatrix):
        """Single frame: -> (ok, rvec (3,1), tvec (3,1), cost, evals)."""
        init = np.concatenate([np.asarray(rvec, dtype=np.float64).reshape(3), np.asarray(tvec, dtype=np.float64).reshape(3)])
        r = self.refine_poses(np.asarray(gray)[None], init.reshape(1, 1, 6), cameraMatrix)
        ok = int(r["status"][0, 0]) != _lib.DPR_NONE
        p = r["pose"][0, 0]
        return ok, p[:3].reshape(3, 1).copy(), p[3:].reshape(3, 1).copy(), float(r["cost"][0, 0]), int(r["evals"][0, 0])


def pinned_frames(shape, dtype=np.uint8):
    """A numpy array in page-locked, device-mapped host memory (a camera ring buffer, a batch of frames): ``refine_poses`` reads
    the regions of interest of such frames in place over PCIe (3.9e5 poses/s on one B200 against 2.1e5 from a pageable array,
    which has to be packed into pinned staging by host threads first).  The array keeps its memory alive."""
    import torch
    return torch.empty(tuple(int(v) for v in shape), dtype=getattr(torch, np.dtype(dtype).name), pin_memory=True).numpy()


# -- Rodrigues is 3x3 host algebra (dozens of flops); it stays on the host like the rest of the predictor ----
def Rodrigues(src):
    """cv.Rodrigues for a (3,), (3,1), (1,3) vector or a (3,3) matrix -> (dst, None).
    The output depth follows the input depth as in OpenCV."""
    a = np.asarray(src)
    out_dtype = np.float32 if a.dtype == np.float32 else np.float64
    if a.shape == (3, 3):
        return synth.rotation_to_rvec(a.astype(np.float64)).reshape(3, 1).astype(out_dtype), None
    if a.size != 3:
        raise ValueError("Rodrigues expects a 3-vector or a 3x3 matrix")
    return synth.rodrigues(a.astype(np.float64).reshape(3)).astype(out_dtype), None


_default: Optional[HostContext] = None


def default_context() -> HostContext:
    global _default
    if _default is None:
        _default = HostContext(0)
    return _default


def solvePnP(*args, **kwargs):
    return default_context().solvePnP(*args, **kwargs)


def projectPoints(*args, **kwargs):
    return default_context().projectPoints(*args, **kwargs)


def calcOpticalFlowPyrLK(*args, **kwargs):
    return default_context().calcOpticalFlowPyrLK(*args, **kwargs)
