"""Batched device API over libagt.so: one ``AgtContext`` per GPU (one process per GPU).

torch is plumbing only here: it owns the device allocations (frames, pyramids,
points, poses) and the stream; every kernel that runs is hand-written CUDA
launched through the C ABI on ``torch.cuda.current_stream()``.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import List, Optional, Sequence, Tuple

import numpy as np

from . import _lib, synth


def _torch():
    import torch
    if not torch.cuda.is_available():
        raise RuntimeError("no CUDA device visible: the AprilGroup tracking path has no CPU fallback")
    return torch


@dataclass
class Pyramid:
    """Device pyramid batch: levels[l] is a uint8 tensor [B, h_l, pitch_l]."""
    levels: List["object"]
    widths: List[int]
    heights: List[int]
    desc: _lib.AgtPyramid
    batch: int

    @property
    def frames(self):
        """Level-0 view [B, H, W]."""
        return self.levels[0][:, :, : self.widths[0]]

    def level(self, l: int):
        return self.levels[l][:, :, : self.widths[l]]


class AgtContext:
    def __init__(self, device: int = 0, mtx: Optional[np.ndarray] = None, dist: Optional[np.ndarray] = None):
        self.lib = _lib.load()
        self.torch = _torch()
        self.device = int(device)
        self.tdev = self.torch.device("cuda", self.device)
        h = C.c_void_p()
        rc = self.lib.agt_create(self.device, C.byref(h))
        if rc != _lib.AGT_OK:
            msg = self.lib.agt_last_error(None)
            raise RuntimeError(f"agt_create failed ({rc}): {msg.decode() if msg else ''}")
        self.h = h
        self._model = None
        if mtx is not None:
            self.set_camera(mtx, dist)

    def close(self):
        if getattr(self, "h", None):
            self.lib.agt_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- plumbing -----------------------------------------------------------------
    def _check(self, rc, what=""):
        _lib.check(self.h, rc, what)

    def _use_current_stream(self):
        s = self.torch.cuda.current_stream(self.tdev).cuda_stream
        self._check(self.lib.agt_set_stream(self.h, C.c_void_p(s)))

    @staticmethod
    def _p(t):
        return C.c_void_p(t.data_ptr()) if t is not None else None

    def _dev(self, arr, dtype):
        t = self.torch
        if isinstance(arr, t.Tensor):
            return arr.to(device=self.tdev, dtype=dtype).contiguous()
        return t.as_tensor(np.ascontiguousarray(arr), dtype=dtype, device=self.tdev).contiguous()

    def launch_count(self) -> int:
        return int(self.lib.agt_launch_count(self.h))

    def sync(self):
        self.torch.cuda.synchronize(self.tdev)

    # -- configuration --------------------------------------------------------------
    def set_camera(self, mtx: np.ndarray, dist: Optional[np.ndarray] = None):
        k = np.ascontiguousarray(np.asarray(mtx, dtype=np.float64).reshape(9))
        if dist is None:
            d, nd = None, 0
        else:
            d = np.ascontiguousarray(np.asarray(dist, dtype=np.float64).reshape(-1))
            nd = int(d.size)
        self._check(self.lib.agt_set_camera(self.h, k.ctypes.data_as(C.POINTER(C.c_double)),
                                            d.ctypes.data_as(C.POINTER(C.c_double)) if d is not None else None, nd))
        self.mtx = np.asarray(mtx, dtype=np.float64).reshape(3, 3).copy()
        self.dist = None if dist is None else d.copy()
        self.config_epoch = getattr(self, "config_epoch", 0) + 1      # captured CUDA graphs hold the camera by value

    def set_model(self, samples: np.ndarray, sample_tag: np.ndarray, normals: np.ndarray, centres: np.ndarray, pitch: float):
        s = np.ascontiguousarray(samples, dtype=np.float32)
        tg = np.ascontiguousarray(sample_tag, dtype=np.uint8)
        n = np.ascontiguousarray(normals, dtype=np.float32)
        c = np.ascontiguousarray(centres, dtype=np.float32)
        self._check(self.lib.agt_set_model(self.h, s.ctypes.data, tg.ctypes.data, int(s.shape[0]), n.ctypes.data,
                                           c.ctypes.data, int(n.shape[0]), float(pitch)))
        self._model = (s, tg, n, c, float(pitch))
        self.config_epoch = getattr(self, "config_epoch", 0) + 1      # ... and the model's device pointers

    def set_synthetic_model(self):
        s, tg, n, c = synth.surface_model()
        self.set_model(s, tg, n, c, synth.model_pitch())

    # -- pyramids -------------------------------------------------------------------
    def alloc_pyramid(self, batch: int, width: int, height: int, levels: int = 4) -> Pyramid:
        t = self.torch
        desc = _lib.AgtPyramid()
        desc.levels = levels
        lv, ws, hs = [], [], []
        w, h = width, height
        for l in range(levels):
            pitch = (w + 15) // 16 * 16
            buf = t.empty((batch, h, pitch), dtype=t.uint8, device=self.tdev)
            lv.append(buf); ws.append(w); hs.append(h)
            desc.width[l], desc.height[l] = w, h
            desc.pitch[l], desc.frame_stride[l] = pitch, pitch * h
            desc.data[l] = buf.data_ptr()
            w, h = (w + 1) // 2, (h + 1) // 2
        return Pyramid(lv, ws, hs, desc, batch)

    def upload_frames(self, pyr: Pyramid, frames) -> None:
        """frames: [B,H,W] uint8 numpy array or tensor -> level 0."""
        t = self.torch
        src = frames if isinstance(frames, t.Tensor) else t.from_numpy(np.ascontiguousarray(frames))
        pyr.frames.copy_(src.to(self.tdev, non_blocking=True))

    def ingest_bgr(self, pyr: Pyramid, bgr) -> None:
        """bgr [B,H,W,3] uint8 (device tensor or numpy) -> level 0 of ``pyr`` as cv.cvtColor(BGR2GRAY) would give it."""
        t = self.torch
        src = self._dev(bgr, t.uint8)
        b, h, w = int(src.shape[0]), int(src.shape[1]), int(src.shape[2])
        self._use_current_stream()
        self._check(self.lib.agt_bgr_to_gray(self.h, self._p(src), w, h, 3 * w, 3 * w * h, self._p(pyr.levels[0]),
                                             pyr.desc.pitch[0], pyr.desc.frame_stride[0], b))

    def set_undistort(self, new_mtx, width: int, height: int, roi) -> None:
        """New camera matrix and crop (x, y, w, h) as cv.getOptimalNewCameraMatrix returns them (detect_pose.py:167-173)."""
        k = np.ascontiguousarray(new_mtx, dtype=np.float64).reshape(9)
        x, y, w, h = (int(v) for v in roi)
        self._check(self.lib.agt_set_undistort(self.h, k.ctypes.data_as(C.POINTER(C.c_double)), int(width), int(height), x, y, w, h))
        self._undistort_roi = (x, y, w, h)

    def ingest_undistort(self, pyr: Pyramid, frames) -> None:
        """frames [B,H,W,3] BGR or [B,H,W] gray, uint8 -> level 0 of ``pyr`` (roi_w x roi_h) as the reference's
        undistort_frame + BGR2GRAY would give it (detect_pose.py:147-183, 602)."""
        t = self.torch
        src = self._dev(frames, t.uint8)
        b, h, w = int(src.shape[0]), int(src.shape[1]), int(src.shape[2])
        ch = int(src.shape[3]) if src.dim() == 4 else 1
        self._use_current_stream()
        self._check(self.lib.agt_undistort_to_gray(self.h, self._p(src), w, h, ch, ch * w, ch * w * h, self._p(pyr.levels[0]),
                                                   pyr.desc.pitch[0], pyr.desc.frame_stride[0], b))

    def build_pyramid(self, pyr: Pyramid, batch: Optional[int] = None) -> None:
        self._use_current_stream()
        self._check(self.lib.agt_build_pyramid(self.h, C.byref(pyr.desc), int(pyr.batch if batch is None else batch)))

    def scharr(self, pyr: Pyramid, level: int = 0):
        """-> int16 tensor [B, h, w, 2] (dx, dy) of one level."""
        t = self.torch
        w, h = pyr.widths[level], pyr.heights[level]
        out = t.empty((pyr.batch, h, w, 2), dtype=t.int16, device=self.tdev)
        self._use_current_stream()
        self._check(self.lib.agt_scharr(self.h, self._p(pyr.levels[level]), w, h, pyr.desc.pitch[level],
                                        pyr.desc.frame_stride[level], self._p(out), pyr.batch))
        return out

    # -- K2 ---------------------------------------------------------------------------
    def lk(self, prev: Pyramid, nxt: Pyramid, prev_pts, n_tags=None):
        """prev_pts [B,P,2] float32 -> (next_pts [B,P,2] f32, status [B,P] u8, err [B,P] f32).
        n_tags [B] i32: frames with >= 2 detected tags are skipped (pipeline fallback rule)."""
        t = self.torch
        pts = self._dev(prev_pts, t.float32)
        b, p = int(pts.shape[0]), int(pts.shape[1])
        out = t.empty_like(pts)
        st = t.empty((b, p), dtype=t.uint8, device=self.tdev)
        err = t.empty((b, p), dtype=t.float32, device=self.tdev)
        self._use_current_stream()
        if n_tags is None:
            self._check(self.lib.agt_lk(self.h, C.byref(prev.desc), C.byref(nxt.desc), self._p(pts), self._p(out), self._p(st),
                                        self._p(err), b, p))
        else:
            self._check(self.lib.agt_lk_fallback(self.h, C.byref(prev.desc), C.byref(nxt.desc), self._p(pts), self._p(out),
                                                 self._p(st), self._p(err), self._p(n_tags), b, p))
        return out, st, err

    def corner_subpix(self, pyr: Pyramid, pts, valid=None, win: int = 5, max_iters: int = 30, eps: float = 1e-3):
        """cv.cornerSubPix on level 0 of every frame: pts [B,P,2] f32 -> refined [B,P,2] f32 (N3, first step)."""
        t = self.torch
        p = self._dev(pts, t.float32)
        b, n = int(p.shape[0]), int(p.shape[1])
        v = None if valid is None else self._dev(valid, t.uint8)
        out = t.empty_like(p)
        self._use_current_stream()
        self._check(self.lib.agt_corner_subpix(self.h, self._p(pyr.levels[0]), pyr.desc.width[0], pyr.desc.height[0], pyr.desc.pitch[0],
                                               pyr.desc.frame_stride[0], self._p(p), self._p(v) if v is not None else None, self._p(out),
                                               b, n, int(win), int(max_iters), float(eps)))
        return out

    def set_tag_family(self, codes=None):
        """The 36-bit code words of the tag family (default tag36h11, the reference's family: detect_pose.py:87)."""
        c = np.ascontiguousarray(synth.TAG36H11_CODES if codes is None else codes, dtype=np.uint64)
        self._check(self.lib.agt_set_tag_family(self.h, c.ctypes.data, int(c.size)))
        self._tag_family = int(c.size)

    TAG_THRESHOLDS = {"auto": 0, "window": 1, "local": 2}

    def set_tag_threshold(self, mode="auto"):
        """What the detector's threshold takes as white: "window" = the brightest pixel of a frame's search window, "local" = the
        brightest pixel of the 3 x 3 tiles of 32 x 32 pixels around the pixel (frames lit unevenly; the reference's apriltag
        library thresholds adaptively), "auto" = local for whole frames, window for search windows."""
        self._check(self.lib.agt_set_tag_threshold(self.h, self.TAG_THRESHOLDS[mode] if isinstance(mode, str) else int(mode)))

    def decode_tags(self, pyr: Pyramid, quads, valid=None, max_hamming: int = 2):
        """Identify the tag inside every quad: quads [B,Q,4,2] f32 (reference corner order, any rotation) ->
        dict(id [B,Q] i32 (-1: none), rotation u8, hamming u8, margin f32)."""
        t = self.torch
        if getattr(self, "_tag_family", 0) == 0:
            self.set_tag_family()
        q = self._dev(quads, t.float32)
        b, n = int(q.shape[0]), int(q.shape[1])
        v = None if valid is None else self._dev(valid, t.uint8)
        out = {"id": t.empty((b, n), dtype=t.int32, device=self.tdev), "rotation": t.empty((b, n), dtype=t.uint8, device=self.tdev),
               "hamming": t.empty((b, n), dtype=t.uint8, device=self.tdev), "margin": t.empty((b, n), dtype=t.float32, device=self.tdev)}
        self._use_current_stream()
        self._check(self.lib.agt_decode_tags(self.h, self._p(pyr.levels[0]), pyr.desc.width[0], pyr.desc.height[0], pyr.desc.pitch[0],
                                             pyr.desc.frame_stride[0], self._p(q), self._p(v) if v is not None else None, self._p(out["id"]),
                                             self._p(out["rotation"]), self._p(out["hamming"]), self._p(out["margin"]), b, n, int(max_hamming)))
        return out

    def track_rects(self, state, width: int, height: int, radius: float, margin: int = 48, out=None):
        """Search windows [B,4] i32 (x0,y0,x1,y1) of the detector from the stream states: around the predicted (else the last
        accepted) pose; the empty rectangle (= whole frame) for streams without one.  ``out``: preallocated [B,4] i32."""
        t = self.torch
        b = int(state.shape[0])
        rects = t.empty((b, 4), dtype=t.int32, device=self.tdev) if out is None else out
        self._use_current_stream()
        self._check(self.lib.agt_track_rects(self.h, self._p(state), float(radius), int(margin), int(width), int(height), self._p(rects), b))
        return rects

    def detect_tags(self, pyr: Pyramid, max_tags: int = 32, max_hamming: int = 2, refine_win: int = 4, rects=None):
        """Detect and identify the tags of every frame (level 0): -> dict(n [B] i32, id [B,T] i32, corners [B,T,4,2] f32 in the
        reference's corner order, margin [B,T] f32, hamming [B,T] u8); entries beyond n[b] are undefined.  ``rects`` [B,4] i32:
        search window per frame (empty = whole frame)."""
        t = self.torch
        if getattr(self, "_tag_family", 0) == 0:
            self.set_tag_family()
        b = pyr.batch
        out = {"n": t.empty(b, dtype=t.int32, device=self.tdev), "id": t.empty((b, max_tags), dtype=t.int32, device=self.tdev),
               "corners": t.empty((b, max_tags, 4, 2), dtype=t.float32, device=self.tdev),
               "margin": t.empty((b, max_tags), dtype=t.float32, device=self.tdev), "hamming": t.empty((b, max_tags), dtype=t.uint8, device=self.tdev)}
        self._use_current_stream()
        r = None if rects is None else self._dev(rects, t.int32)
        self._check(self.lib.agt_detect_tags_roi(self.h, self._p(pyr.levels[0]), pyr.desc.width[0], pyr.desc.height[0], pyr.desc.pitch[0],
                                                 pyr.desc.frame_stride[0], b, self._p(r) if r is not None else None,
                                                 int(r.shape[1]) if r is not None else 0, int(max_tags), int(max_hamming), int(refine_win),
                                                 self._p(out["n"]), self._p(out["id"]), self._p(out["corners"]), self._p(out["margin"]),
                                                 self._p(out["hamming"])))
        out["n"].clamp_(max=max_tags)
        return out

    def tag_quads(self, frames, width: Optional[int] = None, rects=None, max_quads: int = 64, refine_win: int = 4):
        """The detector's first stage alone (threshold, components, quadrilateral fit) -> dict(n_comp [B] i32 components of area
        >= 48 numbered, overflow [B] u8 (1: the global-memory union-find ran), n_quads [B] i32 (not clamped), quads
        [B,max_quads,4,2] f32 clockwise in frame coordinates, win [B,max_quads] u8 the corner-refinement window of each quad);
        slots beyond n_quads are undefined.  ``frames``: a Pyramid (level 0) or a uint8 tensor [B,H,pitch] on the device with
        the frame ``width`` <= pitch (any pitch: the row reads take 16, 4 or 1 pixels at a time depending on the alignment)."""
        t = self.torch
        if isinstance(frames, Pyramid):
            img, w, h, pitch, stride = frames.levels[0], frames.desc.width[0], frames.desc.height[0], frames.desc.pitch[0], frames.desc.frame_stride[0]
        else:
            if frames.dtype != t.uint8 or frames.dim() != 3 or not frames.is_cuda or frames.stride(2) != 1 or frames.stride(1) != frames.shape[2]:
                raise ValueError("tag_quads: frames must be a device uint8 tensor [B,H,pitch] with contiguous rows")
            img, h, pitch, stride = frames, int(frames.shape[1]), int(frames.shape[2]), int(frames.stride(0))
            w = pitch if width is None else int(width)
        b = int(img.shape[0])
        out = {"n_comp": t.empty(b, dtype=t.int32, device=self.tdev), "overflow": t.empty(b, dtype=t.uint8, device=self.tdev),
               "n_quads": t.empty(b, dtype=t.int32, device=self.tdev), "quads": t.empty((b, max_quads, 4, 2), dtype=t.float32, device=self.tdev),
               "win": t.empty((b, max_quads), dtype=t.uint8, device=self.tdev)}
        self._use_current_stream()
        r = None if rects is None else self._dev(rects, t.int32)
        self._check(self.lib.agt_tag_quads(self.h, self._p(img), int(w), int(h), int(pitch), int(stride), b, self._p(r) if r is not None else None,
                                           int(r.shape[1]) if r is not None else 0, int(max_quads), int(refine_win), self._p(out["n_comp"]),
                                           self._p(out["overflow"]), self._p(out["n_quads"]), self._p(out["quads"]), self._p(out["win"])))
        return out

    def pack_detections(self, det, group_ids, min_margin: float = 50.0, out=None):
        """A0 on the device: the dict ``detect_tags`` returns -> (img_pts [B,4T,2] f32, valid [B,4T] u8, n_tags [B] i32, n_unknown
        [B] i32) indexed by the tags' positions in ``group_ids`` (the group's ids in JSON key order); detections with
        margin < min_margin are dropped (detect_pose.py:389).  ``out`` = the same tuple of preallocated tensors."""
        t = self.torch
        g = self._dev(np.asarray(list(group_ids), dtype=np.int32), t.int32) if not hasattr(group_ids, "device") else group_ids
        b, mt, ng = int(det["id"].shape[0]), int(det["id"].shape[1]), int(g.numel())
        if out is None:
            out = (t.empty((b, 4 * ng, 2), dtype=t.float32, device=self.tdev), t.empty((b, 4 * ng), dtype=t.uint8, device=self.tdev),
                   t.empty(b, dtype=t.int32, device=self.tdev), t.empty(b, dtype=t.int32, device=self.tdev))
        self._use_current_stream()
        self._check(self.lib.agt_pack_detections(self.h, self._p(det["n"]), self._p(det["id"]), self._p(det["corners"]), self._p(det["margin"]),
                                                 mt, self._p(g), ng, float(min_margin), self._p(out[0]), self._p(out[1]), self._p(out[2]),
                                                 self._p(out[3]), b))
        return out

    def lk_rects(self, pyr: Pyramid, pts, valid=None, max_flow: int = 32):
        """Level-0 rectangle [B,4] i32 that tracking ``pts`` [B,P,2] can read while no corner moves more than max_flow px."""
        t = self.torch
        p = self._dev(pts, t.float32)
        b, n = int(p.shape[0]), int(p.shape[1])
        rects = t.empty((b, 4), dtype=t.int32, device=self.tdev)
        v = self._dev(valid, t.uint8) if valid is not None else None
        self._use_current_stream()
        self._check(self.lib.agt_lk_rects(self.h, C.byref(pyr.desc), self._p(p), self._p(v), n, int(max_flow), self._p(rects), 4, b))
        return rects

    def lk_roi(self, prev: Pyramid, nxt: Pyramid, prev_pts, rects_prev=None, n_tags=None, max_flow: int = 32, valid=None):
        """Tracking with the pyramid of the new frames built only where the corners can look, exact by construction:
        rectangles from prev_pts -> ROI pyramid of ``nxt`` (level 0 must hold the frames) -> LK; frames in which a corner
        looked outside what was built (``left_roi``) get complete pyramids and are tracked again, all on the device
        (the redo launches leave at once when nothing is flagged).  ``rects_prev``: rectangles ``prev`` was built under
        (None = complete).  -> (next_pts, status, err, rects, redo[B] u8); ``nxt`` is valid under ``rects`` except for
        the frames flagged in ``redo``, which are complete."""
        t = self.torch
        pts = self._dev(prev_pts, t.float32)
        b, p = int(pts.shape[0]), int(pts.shape[1])
        rects = self.lk_rects(nxt, pts, valid, max_flow)
        self.build_pyramid_roi(nxt, rects, b)
        out = t.empty_like(pts)
        st = t.empty((b, p), dtype=t.uint8, device=self.tdev)
        err = t.empty((b, p), dtype=t.float32, device=self.tdev)
        left = t.empty((b, p), dtype=t.uint8, device=self.tdev)
        redo = t.empty(b, dtype=t.uint8, device=self.tdev)
        self._use_current_stream()
        args = (self._p(pts), self._p(out), self._p(st), self._p(err), self._p(n_tags))
        self._check(self.lib.agt_lk_roi(self.h, C.byref(prev.desc), C.byref(nxt.desc), *args, self._p(rects_prev), self._p(rects), 4,
                                        None, self._p(left), b, p))
        self._check(self.lib.agt_any_flag(self.h, self._p(left), p, self._p(redo), b))
        self.build_pyramid_masked(nxt, redo, b)
        if rects_prev is not None:
            self.build_pyramid_masked(prev, redo, b)
        self._check(self.lib.agt_lk_roi(self.h, C.byref(prev.desc), C.byref(nxt.desc), *args, None, None, 0, self._p(redo), None, b, p))
        return out, st, err, rects, redo

    def lk_merge(self, tracked, status, prev_valid, img_pts, valid, n_tags, tracked_tags=None):
        """In place: re-admit fully tracked tags into img_pts/valid for frames with < 2 detected tags;
        tracked_tags [B] i32 (optional) receives the number of tags re-admitted per frame."""
        b, p = int(img_pts.shape[0]), int(img_pts.shape[1])
        self._use_current_stream()
        self._check(self.lib.agt_lk_merge(self.h, self._p(tracked), self._p(status), self._p(prev_valid), self._p(img_pts),
                                          self._p(valid), self._p(n_tags), self._p(tracked_tags), b, p))

    # -- K3 ---------------------------------------------------------------------------
    def pnp(self, obj_pts, img_pts, valid=None, guess=None, use_guess=None):
        """obj [P,3] f32 shared, img [B,P,2] f32, valid [B,P] u8, guess [B,6] f64, use_guess [B] u8
        -> (pose [B,6] f64, ok [B] u8, reproj_err [B] f32, iters [B] i32)."""
        t = self.torch
        obj = self._dev(obj_pts, t.float32)
        img = self._dev(img_pts, t.float32)
        b, p = int(img.shape[0]), int(img.shape[1])
        if obj.shape[0] != p:
            raise ValueError("obj_pts and img_pts disagree on the number of points")
        v = self._dev(valid, t.uint8) if valid is not None else None
        g = self._dev(guess, t.float64) if guess is not None else None
        ug = self._dev(use_guess, t.uint8) if use_guess is not None else (
            t.ones(b, dtype=t.uint8, device=self.tdev) if g is not None else None)
        pose = t.empty((b, 6), dtype=t.float64, device=self.tdev)
        ok = t.empty(b, dtype=t.uint8, device=self.tdev)
        err = t.empty(b, dtype=t.float32, device=self.tdev)
        iters = t.empty(b, dtype=t.int32, device=self.tdev)
        self._use_current_stream()
        self._check(self.lib.agt_pnp(self.h, self._p(obj), self._p(img), self._p(v), self._p(g), self._p(ug), self._p(pose),
                                     self._p(ok), self._p(err), self._p(iters), b, p))
        return pose, ok, err, iters

    def streams_front(self, obj, state, enhance_ape, img, valid, n_tags_in, tracked=None, lk_status=None, prev_valid=None,
                      want_gate=True):
        """agt_streams_front: lk_merge (when ``tracked`` is given) -> ape_prepare -> pnp -> accept_gate in one launch, on device tensors.
        ``img`` [B,P,2] f32 / ``valid`` [B,P] u8 are merged in place.  -> dict(pose, ok, err, iters, n_tags, tracked_tags, gate, status)."""
        t = self.torch
        b, p = int(img.shape[0]), int(img.shape[1])
        o = {"pose": t.empty((b, 6), dtype=t.float64, device=self.tdev), "ok": t.empty(b, dtype=t.uint8, device=self.tdev),
             "err": t.empty(b, dtype=t.float32, device=self.tdev), "iters": t.empty(b, dtype=t.int32, device=self.tdev),
             "n_tags": t.empty(b, dtype=t.int32, device=self.tdev),
             "tracked_tags": t.empty(b, dtype=t.int32, device=self.tdev) if tracked is not None else None,
             "gate": t.empty(b, dtype=t.uint8, device=self.tdev) if want_gate else None,
             "status": t.empty((b, 1), dtype=t.uint8, device=self.tdev) if want_gate else None}
        self._use_current_stream()
        self._check(self.lib.agt_streams_front(self.h, self._p(obj), self._p(tracked), self._p(lk_status), self._p(prev_valid), self._p(img),
                                               self._p(valid), self._p(n_tags_in), self._p(o["n_tags"]), self._p(o["tracked_tags"]),
                                               self._p(state), 1 if enhance_ape else 0, self._p(o["pose"]), self._p(o["ok"]), self._p(o["err"]),
                                               self._p(o["iters"]), self._p(o["gate"]), self._p(o["status"]), b, p))
        return o

    def project(self, obj_pts, poses):
        t = self.torch
        obj = self._dev(obj_pts, t.float32)
        ps = self._dev(poses, t.float64).reshape(-1, 6)
        out = t.empty((ps.shape[0], obj.shape[0], 2), dtype=t.float64, device=self.tdev)
        self._use_current_stream()
        self._check(self.lib.agt_project(self.h, self._p(obj), self._p(ps), self._p(out), int(ps.shape[0]), int(obj.shape[0])))
        return out

    # -- K0 ---------------------------------------------------------------------------
    def overlay_points(self, bgr, obj_pts, poses, frame_mask=None, radius: int = 5, color=(0, 0, 255), bounds=(1280, 720)):
        """The reference's pose overlay for a batch (detect_pose.py:441-465, draw.py:120-153): project `obj_pts` [P,3] with
        `poses` [B,6] and stamp a filled disc on every projection into `bgr` [B,H,W,3] uint8 (device tensor, in place).
        `bounds` is the (width, height) the reference tests the rounded centre against (hard-coded 1280 x 720 there);
        `frame_mask` [B] uint8 selects the frames that get an overlay (the accepted ones).  -> projections [B,P,2] f64."""
        t = self.torch
        if not (isinstance(bgr, t.Tensor) and bgr.is_cuda and bgr.dtype == t.uint8 and bgr.dim() == 4 and bgr.shape[3] == 3 and bgr.is_contiguous()):
            raise ValueError("bgr must be a contiguous uint8 CUDA tensor [B,H,W,3]")
        b, h, w = int(bgr.shape[0]), int(bgr.shape[1]), int(bgr.shape[2])
        proj = self.project(obj_pts, poses)
        m = None if frame_mask is None else self._dev(frame_mask, t.uint8)
        self._use_current_stream()
        self._check(self.lib.agt_draw_points(self.h, self._p(bgr), w, h, 3 * w, 3 * w * h, self._p(proj), self._p(m) if m is not None else None,
                                             b, int(proj.shape[1]), int(radius), int(bounds[0]), int(bounds[1]), int(color[0]), int(color[1]),
                                             int(color[2])))
        return proj

    def new_stream_state(self, n_streams: int):
        t = self.torch
        return t.zeros((n_streams, _lib.AGT_STREAM_STATE_DOUBLES), dtype=t.float64, device=self.tdev)

    def ape_prepare(self, state, enhance_ape: bool = True):
        t = self.torch
        b = int(state.shape[0])
        guess = t.empty((b, 6), dtype=t.float64, device=self.tdev)
        use = t.empty(b, dtype=t.uint8, device=self.tdev)
        self._use_current_stream()
        self._check(self.lib.agt_ape_prepare(self.h, self._p(state), self._p(guess), self._p(use), b, int(enhance_ape)))
        return guess, use

    def ape_update(self, state, n_tags, pose, ok, err, enhance_ape: bool = True):
        t = self.torch
        b = int(state.shape[0])
        nt = self._dev(n_tags, t.int32)
        acc = t.empty(b, dtype=t.uint8, device=self.tdev)
        flag = t.empty(b, dtype=t.uint8, device=self.tdev)
        self._use_current_stream()
        self._check(self.lib.agt_ape_update(self.h, self._p(state), self._p(nt), self._p(pose), self._p(ok), self._p(err),
                                            self._p(acc), self._p(flag), b, int(enhance_ape)))
        return acc, flag

    def accept_gate(self, ok, err, n_tags):
        """[B] u8: the reference's acceptance test of a solved frame (>= 2 tags, solvePnP ok, mean error < 2 px)."""
        t = self.torch
        b = int(ok.shape[0])
        gate = t.empty(b, dtype=t.uint8, device=self.tdev)
        self._use_current_stream()
        self._check(self.lib.agt_accept_gate(self.h, self._p(ok), self._p(err), self._p(n_tags), self._p(gate), b))
        return gate

    def ape_commit(self, state, n_tags, pose, ok, err, refined=None, img_pts=None, valid=None, prev_pts=None, prev_valid=None,
                   enhance_ape: bool = True):
        """ape_update with the refined pose where the refinement produced one, plus the hand-over of the frame's corners
        to the next LK step -> (accepted [B] u8, error_flag [B] u8, pose [B,6] f64 = each stream's prev_transform)."""
        t = self.torch
        b = int(state.shape[0])
        acc = t.empty(b, dtype=t.uint8, device=self.tdev)
        flag = t.empty(b, dtype=t.uint8, device=self.tdev)
        out = t.empty((b, 6), dtype=t.float64, device=self.tdev)
        rp = refined["pose"] if refined is not None else None
        rs = refined["status"] if refined is not None else None
        n_pts = int(img_pts.shape[1]) if img_pts is not None else 0
        self._use_current_stream()
        self._check(self.lib.agt_ape_commit(self.h, self._p(state), self._p(n_tags), self._p(pose), self._p(ok), self._p(err),
                                            self._p(rp), self._p(rs), self._p(img_pts), self._p(valid), self._p(prev_pts),
                                            self._p(prev_valid), n_pts, self._p(acc), self._p(flag), self._p(out), b,
                                            int(enhance_ape)))
        return acc, flag, out

    # -- K4 ---------------------------------------------------------------------------
    def refine(self, pyr: Pyramid, init, n_hyp: int = 1, batch: Optional[int] = None, mask=None, out=None, fused: bool = False):
        """init [B,H,6] f64 -> dict(pose [B,H,6], cost [B,H], n_valid, evals, status, left_roi).
        mask [B] u8: frames with 0 are skipped and none of their outputs is written; ``out`` (a previous result
        dict) receives the outputs in place, otherwise skipped frames read pose = init, everything else 0.
        fused: only level 0 of ``pyr`` holds the frames; every refinement builds the part of its level it reads
        inside the kernel (agt_refine_fused)."""
        t = self.torch
        b = int(pyr.batch if batch is None else batch)
        ini = self._dev(init, t.float64).reshape(b, n_hyp, 6)
        if out is None:
            fresh = t.zeros if mask is not None else t.empty
            out = {"pose": ini.clone() if mask is not None else t.empty_like(ini),
                   "cost": fresh((b, n_hyp), dtype=t.float32, device=self.tdev),
                   "n_valid": fresh((b, n_hyp), dtype=t.int32, device=self.tdev),
                   "evals": fresh((b, n_hyp), dtype=t.int32, device=self.tdev),
                   "status": fresh((b, n_hyp), dtype=t.uint8, device=self.tdev),
                   "left_roi": fresh((b, n_hyp), dtype=t.uint8, device=self.tdev)}
        msk = self._dev(mask, t.uint8) if mask is not None else None
        self._use_current_stream()
        fn = self.lib.agt_refine_fused if fused else self.lib.agt_refine
        self._check(fn(self.h, C.byref(pyr.desc), self._p(ini), n_hyp, self._p(msk), self._p(out["pose"]),
                       self._p(out["cost"]), self._p(out["n_valid"]), self._p(out["evals"]), self._p(out["status"]),
                       self._p(out["left_roi"]), b))
        return out

    def pose_covariance(self, pyr: Pyramid, init, pose, n_hyp: int = 1, mask=None, out=None):
        """Covariance of refined poses (agt_pose_covariance): the refinement's cost function, fixed by ``init`` [B,H,6] as
        ``refine`` fixes it, evaluated once at ``pose`` [B,H,6] (normally the refined pose) -> dict(cov [B,H,6,6] f64 =
        s^2 H^-1, info [B,H,6,6] f64 = H = J^T J, sigma2 [B,H] f32 = s^2 = 2c / (n_valid - 6), n_valid [B,H] i32, ok [B,H] u8).
        Tangent order: rotation (left perturbation R <- exp(w) R, radians), then translation (metres).  ok = 0 (cov NaN)
        when n_valid <= 6 or H is not positive definite.  mask [B] u8 / ``out`` as for ``refine``: frames with mask 0 are
        skipped and their outputs left as they are."""
        t = self.torch
        if n_hyp < 1:
            raise ValueError(f"pose_covariance: n_hyp must be at least 1 (got {n_hyp})")
        ini = self._dev(init, t.float64).reshape(-1, n_hyp, 6)
        b = int(ini.shape[0])
        if b > pyr.batch:
            raise ValueError(f"pose_covariance: {b} frames of poses for a pyramid of {pyr.batch}")
        ps = self._dev(pose, t.float64).reshape(b, n_hyp, 6)
        if out is None:
            fresh = t.zeros if mask is not None else t.empty
            out = {"cov": fresh((b, n_hyp, 6, 6), dtype=t.float64, device=self.tdev),
                   "info": fresh((b, n_hyp, 6, 6), dtype=t.float64, device=self.tdev),
                   "sigma2": fresh((b, n_hyp), dtype=t.float32, device=self.tdev),
                   "n_valid": fresh((b, n_hyp), dtype=t.int32, device=self.tdev),
                   "ok": fresh((b, n_hyp), dtype=t.uint8, device=self.tdev)}
        msk = self._dev(mask, t.uint8) if mask is not None else None
        self._use_current_stream()
        self._check(self.lib.agt_pose_covariance(self.h, C.byref(pyr.desc), self._p(ini), self._p(ps), n_hyp, self._p(msk),
                                                 self._p(out["cov"]), self._p(out.get("info")), self._p(out.get("sigma2")),
                                                 self._p(out.get("n_valid")), self._p(out["ok"]), b))
        return out

    def dpr_rects(self, pyr: Pyramid, init, n_hyp: int = 1, batch: Optional[int] = None):
        """Level-0 rectangle [B,4] i32 (x0,y0,x1,y1) each frame's refinements can read."""
        t = self.torch
        b = int(pyr.batch if batch is None else batch)
        ini = self._dev(init, t.float64).reshape(b, n_hyp, 6)
        rects = t.empty((b, 4), dtype=t.int32, device=self.tdev)
        self._use_current_stream()
        self._check(self.lib.agt_dpr_rects(self.h, C.byref(pyr.desc), self._p(ini), n_hyp, self._p(rects), b))
        return rects

    def build_pyramid_roi(self, pyr: Pyramid, rects, batch: Optional[int] = None) -> None:
        self._use_current_stream()
        self._check(self.lib.agt_build_pyramid_roi(self.h, C.byref(pyr.desc), self._p(rects), int(rects.shape[1]),
                                                   int(pyr.batch if batch is None else batch)))

    def build_pyramid_masked(self, pyr: Pyramid, mask, batch: Optional[int] = None) -> None:
        stride = int(mask.shape[1]) if mask.dim() > 1 else 1
        self._use_current_stream()
        self._check(self.lib.agt_build_pyramid_masked(self.h, C.byref(pyr.desc), self._p(mask), stride,
                                                      int(pyr.batch if batch is None else batch)))

    def refine_roi(self, pyr: Pyramid, init, n_hyp: int = 1, batch: Optional[int] = None):
        """Pyramid + refinement restricted to the region of interest, exact by construction:
        rectangles from the initial poses -> ROI pyramid -> refinement; frames whose refinement read outside
        their rectangle (``left_roi``) get the full pyramid and are refined again, all without leaving the device
        (the two redo launches exit immediately for frames that stayed inside)."""
        t = self.torch
        b = int(pyr.batch if batch is None else batch)
        ini = self._dev(init, t.float64).reshape(b, n_hyp, 6)
        rects = self.dpr_rects(pyr, ini, n_hyp, b)
        self.build_pyramid_roi(pyr, rects, b)
        res = self.refine(pyr, ini, n_hyp, b)
        redo = t.empty(b, dtype=t.uint8, device=self.tdev)
        self._check(self.lib.agt_any_flag(self.h, self._p(res["left_roi"]), n_hyp, self._p(redo), b))
        self.build_pyramid_masked(pyr, redo, b)
        self.refine(pyr, ini, n_hyp, b, mask=redo, out=res)
        res["redo"] = redo
        return res

    def refine_fused(self, pyr: Pyramid, init, n_hyp: int = 1, batch: Optional[int] = None, mask=None):
        """Refinement from level 0 alone (K1 fused into K4), exact by construction: every refinement builds the
        region of interest of its own pyramid level inside the kernel; frames whose refinement read outside that
        region (``left_roi``) get the full pyramid and are refined again, all without leaving the device.
        mask [B] u8: frames with 0 are skipped, as in ``refine``."""
        t = self.torch
        b = int(pyr.batch if batch is None else batch)
        ini = self._dev(init, t.float64).reshape(b, n_hyp, 6)
        res = self.refine(pyr, ini, n_hyp, b, mask=mask, fused=True)
        redo = t.empty(b, dtype=t.uint8, device=self.tdev)
        self._check(self.lib.agt_any_flag(self.h, self._p(res["left_roi"]), n_hyp, self._p(redo), b))
        self.build_pyramid_masked(pyr, redo, b)
        self.refine(pyr, ini, n_hyp, b, mask=redo, out=res)
        res["redo"] = redo
        return res

    def select_best(self, res):
        t = self.torch
        b, h = int(res["pose"].shape[0]), int(res["pose"].shape[1])
        best = t.empty(b, dtype=t.int32, device=self.tdev)
        bp = t.empty((b, 6), dtype=t.float64, device=self.tdev)
        self._use_current_stream()
        self._check(self.lib.agt_select_best(self.h, self._p(res["pose"]), self._p(res["cost"]), self._p(res["n_valid"]), h,
                                             self._p(best), self._p(bp), b))
        return best, bp

    # -- synthetic frames ---------------------------------------------------------------
    def render(self, pyr: Pyramid, poses, seeds, noise: bool = True, batch: Optional[int] = None, offset: int = 0) -> None:
        """Render the synthetic dodecahedron into level 0 of frames [offset, offset+batch)."""
        t = self.torch
        ps = self._dev(poses, t.float64).reshape(-1, 6)
        b = int(ps.shape[0] if batch is None else batch)
        if isinstance(seeds, t.Tensor):
            seeds = seeds.detach().cpu().numpy()
        sd32 = self._dev((np.asarray(seeds).astype(np.int64) & 0xFFFFFFFF).astype(np.uint32).view(np.int32), t.int32)
        if not hasattr(self, "_render_consts"):
            rk, tk = synth.group_transforms_f32()
            rt = np.concatenate([rk.reshape(12, 9), tk.reshape(12, 3)], axis=1)
            cells = synth.all_tag_cells().astype(np.uint8).reshape(12, 100)
            self._render_consts = (self._dev(rt, t.float64), self._dev(cells, t.uint8))
        rt, cells = self._render_consts
        base = pyr.levels[0].data_ptr() + offset * pyr.desc.frame_stride[0]
        self._use_current_stream()
        self._check(self.lib.agt_render(self.h, self._p(ps), self._p(sd32), C.c_void_p(base), pyr.widths[0], pyr.heights[0],
                                        pyr.desc.pitch[0], pyr.desc.frame_stride[0], self._p(rt), self._p(cells), 12,
                                        synth.INRADIUS, synth.CELL, int(noise), b))
