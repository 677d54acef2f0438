"""``BatchedPoseDetector``: the full hot path (APE -> LK -> dense refinement) for many camera
streams at once, one frame per stream per step, entirely on one GPU.

It is the batched counterpart of ``PoseDetector._detect_and_get_pose`` (detect_pose.py:576-609) with
the reference's per-stream state (detect_pose.py:74-78) kept in device memory.  Per step:

  K1  agt_build_pyramid    pyramid of the new frames (outside the captured sequence: ``ingest_next`` lets the caller run
                           it, with the frame ingest, on a side stream while the previous step refines)
  K2  agt_lk_fallback      streams with < 2 detected tags track the corners of the previous accepted frame
  --  agt_streams_front    ONE launch, a warp per stream: re-admit the tags whose four corners were tracked (agt_lk_merge: the
                           inlier set is LK status == 1), extrinsic guess from the predictor state (agt_ape_prepare,
                           detect_pose.py:508), K3 batched solvePnP + mean reprojection error (detect_pose.py:509-538), and the
                           2 px gate that masks the refinement (agt_accept_gate)
  K4  agt_refine           dense refinement of the poses that pass the gate
  K0  agt_ape_commit       accept / reset rules, velocity FIFOs, predictor (detect_pose.py:539-574) with the refined
                           pose, and the hand-over of the accepted frame's corners to the next LK step

Frames within a stream are sequential (the predictor needs poses t-1, t-2; LK needs frame t-1), so the
batch dimension is the number of streams; streams are pinned to GPUs by ``sharding.stream_owner``.
"""
from __future__ import annotations

from typing import Optional

import numpy as np

from . import synth
from .context import AgtContext


class BatchedPoseDetector:
    SLOTS = 3

    def __init__(self, ctx: AgtContext, n_streams: int, width: int, height: int, obj_pts: np.ndarray,
                 enhance_ape: bool = True, use_lk: bool = True, use_dense_refine: bool = True, levels: int = 4,
                 use_graphs: bool = True, tag_ids=None, pose_covariance: bool = False):
        """``obj_pts`` [4T,3]: the group's corners in JSON key order (``PoseDetector.all_objpts``); ``tag_ids``: the ids in the
        same order (``list(PoseDetector.extrinsics)``), default 0..T-1 - ``pack`` puts detections where their object points are.
        ``pose_covariance`` (with ``use_dense_refine``): one more launch per step after K4, masked by the same gate, puts the
        covariance of every refined pose (agt_pose_covariance) into the step's ``covariance`` [S,6,6] and ``covariance_ok`` [S]
        (0 where the frame was not refined or the covariance is undefined; ``covariance`` is not written for frames that were
        not refined)."""
        t = ctx.torch
        if obj_pts.shape[0] % 4:
            raise ValueError("obj_pts must hold four corners per tag")
        self.tag_pos = tag_positions(range(obj_pts.shape[0] // 4) if tag_ids is None else tag_ids)
        if len(self.tag_pos) * 4 != obj_pts.shape[0]:
            raise ValueError(f"{len(self.tag_pos)} tag ids for {obj_pts.shape[0] // 4} tags of object points")
        self.ctx, self.n, self.enhance_ape = ctx, int(n_streams), enhance_ape
        self.use_lk, self.use_dense_refine = use_lk, use_dense_refine
        if pose_covariance and not use_dense_refine:
            raise ValueError("pose_covariance needs use_dense_refine: it is the covariance of the refined pose")
        self.pose_covariance = bool(pose_covariance)
        self.n_pts = int(obj_pts.shape[0])
        self.obj = ctx._dev(obj_pts, t.float32)
        # three frame slots: a step reads the current and the previous one, the third is free to receive the next frame while
        # the step runs (double-buffered ingest)
        self.pyr = [ctx.alloc_pyramid(self.n, width, height, levels) for _ in range(self.SLOTS)]
        self.cur = 0
        self.state = ctx.new_stream_state(self.n)
        dev = ctx.tdev
        # static buffers: the per-step work is a fixed launch sequence, captured once per pyramid slot into a CUDA graph
        # (the three inputs of a step are views of ONE buffer, so that a caller who holds them packed - ``pack_inputs`` - pays one
        # copy per step instead of three)
        # One input buffer per frame slot: the inputs of the step after the coming one can be put in place (``detect_next``) while
        # the step in flight still reads its own.
        nb_img, nb_nt, nb_val = 8 * self.n * self.n_pts, 4 * self.n, self.n * self.n_pts
        self._in = []
        for _ in range(self.SLOTS):
            buf = t.zeros(nb_img + nb_nt + nb_val, dtype=t.uint8, device=dev)
            self._in.append((buf, buf[:nb_img].view(t.float32).view(self.n, self.n_pts, 2), buf[nb_img:nb_img + nb_nt].view(t.int32),
                             buf[nb_img + nb_nt:].view(self.n, self.n_pts)))
        self._rects_next = t.zeros((self.n, 4), dtype=t.int32, device=dev)      # search windows of the next frame (next_windows)
        self._det_done = None                                                     # event: the last detection issued has finished
        self.prev_pts = t.zeros((self.n, self.n_pts, 2), dtype=t.float32, device=dev)
        self.prev_valid = t.zeros((self.n, self.n_pts), dtype=t.uint8, device=dev)
        self.use_graphs = use_graphs
        self._graphs = [None] * self.SLOTS
        self._built = [False] * self.SLOTS        # the pyramid of the slot's current frame is already there
        self._outs = [None] * self.SLOTS
        self._steps = 0
        self.kernels_per_step = 0
        if use_dense_refine and ctx._model is None:
            ctx.set_synthetic_model()
        self._epoch = getattr(ctx, "config_epoch", 0)
        # the detector in front of the path (step_frames): the group's ids in JSON key order, and how many kept detections of the
        # last step carried an id outside the group
        self.group_ids = ctx._dev(np.array(sorted(self.tag_pos, key=self.tag_pos.get), dtype=np.int32), t.int32)
        self.n_unknown = t.zeros(self.n, dtype=t.int32, device=dev)
        self.radius = float(np.linalg.norm(np.asarray(obj_pts, dtype=np.float64), axis=1).max())      # bounding sphere of the group

    # the input buffers of the coming step
    @property
    def in_all(self):
        return self._in[self.cur][0]

    @property
    def in_img(self):
        return self._in[self.cur][1]

    @property
    def in_ntags(self):
        return self._in[self.cur][2]

    @property
    def in_valid(self):
        return self._in[self.cur][3]

    def pack(self, dets_per_stream):
        """Detections [(tag_id, corners (4,2)), ...] per stream -> the (img_pts, valid, n_tags) arrays ``step`` takes, indexed by
        the tags' positions in the group (KeyError for an id the group does not have)."""
        return pack_detections(dets_per_stream, self.tag_pos)

    def pack_inputs(self, img_pts, valid, n_tags, pin: bool = False):
        """(img_pts [S,P,2], valid [S,P], n_tags [S]) -> one uint8 tensor in the layout of the step's input buffer (host tensor,
        pinned on request, for numpy inputs; device tensor for device inputs): ``step(packed)`` then costs one copy."""
        t = self.ctx.torch
        parts = []
        for a, dt in ((img_pts, t.float32), (n_tags, t.int32), (valid, t.uint8)):
            x = a if isinstance(a, t.Tensor) else t.as_tensor(np.ascontiguousarray(a))
            parts.append(x.to(dt).contiguous().reshape(-1).view(t.uint8))
        packed = t.cat(parts)
        if packed.numel() != self.in_all.numel():
            raise ValueError("inputs do not have this detector's shape")
        return packed.pin_memory() if pin and not packed.is_cuda else packed

    def reset(self):
        """Forget all stream state (fresh streams); captured graphs stay valid because the buffers are reused."""
        self.state.zero_()
        self.prev_pts.zero_()
        self.prev_valid.zero_()
        self._built = [False] * self.SLOTS

    @property
    def frames(self):
        """Level-0 buffer [S,H,W] the caller fills (or renders into) before ``step``."""
        return self.pyr[self.cur].frames

    @property
    def next_frames(self):
        """Level-0 buffer of the step after the coming one: not read by the coming step, so the caller may fill it
        (on another stream, ordered after the previous step) while that step runs."""
        return self.pyr[(self.cur + 1) % self.SLOTS].frames

    def ingest_next(self, frames, build: bool = True) -> None:
        """Put the frame of the step after the coming one into its slot and build its pyramid (K1), on the current stream:
        neither is read by the coming step, so with a side stream (ordered after the previous step; the coming-but-one step
        ordered after it) the bandwidth-bound ingest runs under the latency-bound refinement of the step in flight."""
        slot = (self.cur + 1) % self.SLOTS
        self.ctx.upload_frames(self.pyr[slot], frames)
        if build:
            self.build_next()

    def build_next(self) -> None:
        """K1 of the frame in the next slot (the second half of ``ingest_next(frames, build=False)``: a caller that also runs
        ``detect_next``, which reads level 0 only, can put the two on different streams)."""
        slot = (self.cur + 1) % self.SLOTS
        self.ctx.build_pyramid(self.pyr[slot])
        self._built[slot] = True

    def _body(self, slot: int):
        """One frame of every stream: fixed launch sequence over static buffers (graph-capturable)."""
        ctx, t = self.ctx, self.ctx.torch
        cur, prv = self.pyr[slot], self.pyr[(slot - 1) % self.SLOTS]
        # The detections of the frame are merged in place in the static input buffers (every step fills them anew before its graph
        # runs); K2 only tracks frames with < 2 detected tags, and on the very first frame prev_valid is all zero, so nothing can be
        # re-admitted from the (not yet written) previous slot.
        _, img, ntags_in, val = self._in[slot]
        nxt = st = None
        if self.use_lk:
            nxt, st, _ = ctx.lk(prv, cur, self.prev_pts, n_tags=ntags_in)                                       # K2
        # merge + K0 (guess from the state records) + K3 + accept gate: the frame's warp does them all in one launch
        fr = ctx.streams_front(self.obj, self.state, self.enhance_ape, img, val, ntags_in, tracked=nxt, lk_status=st,
                               prev_valid=self.prev_valid if self.use_lk else None, want_gate=self.use_dense_refine)
        pose, ok, err, ntg, tracked_tags = fr["pose"], fr["ok"], fr["err"], fr["n_tags"], fr["tracked_tags"]
        refined = None
        if self.use_dense_refine:
            out = {k: t.empty((self.n, 1) + ((6,) if k == "pose" else ()), dtype=d, device=ctx.tdev)
                   for k, d in (("pose", t.float64), ("cost", t.float32), ("n_valid", t.int32), ("evals", t.int32),
                                ("left_roi", t.uint8))}
            out["status"] = fr["status"]                                          # masked frames keep status 0: pose unused
            refined = ctx.refine(cur, pose.reshape(self.n, 1, 6), 1, mask=fr["gate"], out=out)   # K4
        cov = None
        if self.pose_covariance:
            cov = {"cov": t.empty((self.n, 1, 6, 6), dtype=t.float64, device=ctx.tdev),
                   "ok": t.zeros((self.n, 1), dtype=t.uint8, device=ctx.tdev)}
            ctx.pose_covariance(cur, pose.reshape(self.n, 1, 6), refined["pose"], 1, mask=fr["gate"], out=cov)
        # K0 with the refined pose where there is one; the corners of the accepted frame feed the next LK step
        accepted, flag, pose_out = ctx.ape_commit(self.state, ntg, pose, ok, err, refined, img, val, self.prev_pts,
                                                  self.prev_valid, self.enhance_ape)
        res = {"pose": pose_out, "accepted": accepted, "error_flag": flag, "reproj_err": err,
               "n_tags": ntg, "tracked_tags": tracked_tags, "refine": refined}
        if cov is not None:
            res["covariance"], res["covariance_ok"] = cov["cov"].reshape(self.n, 6, 6), cov["ok"].reshape(self.n)
        return res

    def step_frames(self, frames=None, min_margin: float = 50.0, refine_win: int = 4, max_tags: int = 32, check_ids: bool = False,
                    track_window: bool = True, track_margin: int = 48):
        """Pixels in, poses out: ``_obtain_detections`` (detect_pose.py:351-439) on the device in front of ``step`` - agt_detect_tags
        on level 0 of the current slot, the decision-margin filter and the id -> position mapping by agt_pack_detections,
        straight into the static input buffers of the captured step; no detection ever visits the host.  ``check_ids`` reads
        ``n_unknown`` back and raises KeyError like the reference (detect_pose.py:408-415) when a kept detection carries an id
        the group does not have (a synchronisation: off by default, the count stays in ``self.n_unknown``).  ``track_window``: a
        stream that has a predicted or a last accepted pose is searched only around it (bounding sphere of the group + ``track_margin``
        pixels, agt_track_rects) - a few percent of a 1080p frame; streams without a pose are searched whole."""
        ctx = self.ctx
        slot = self.cur
        if frames is not None:
            ctx.upload_frames(self.pyr[slot], frames)
            self._built[slot] = False
        rects = None
        if track_window:
            # look where the object is expected: around the predicted / last accepted pose of each stream (whole frame without one)
            rects = ctx.track_rects(self.state, self.pyr[slot].desc.width[0], self.pyr[slot].desc.height[0], self.radius, track_margin)
        det = self._detect_into(slot, rects, min_margin, refine_win, max_tags)
        if check_ids and int(self.n_unknown.sum().item()):
            raise KeyError("a detected tag id is not in the group")
        out = self.step(None, None, None)
        out["detections"] = det
        return out

    def next_windows(self, track_margin: int = 64) -> None:
        """First half of the pipelined detector (``detect_next``): the search windows of the frame AFTER the coming one, from the
        stream states as they are now - call it on the stream the steps run on, before the coming step (whose commit moves the
        states).  The pose predicted for the coming frame stands in for the one after it, so the margin is wider than
        ``step_frames``' (the object moves twice as far)."""
        pyr = self.pyr[self.cur]
        self.ctx.track_rects(self.state, pyr.desc.width[0], pyr.desc.height[0], self.radius, track_margin, out=self._rects_next)

    def detect_next(self, min_margin: float = 50.0, refine_win: int = 4, max_tags: int = 32, track_window: bool = True) -> None:
        """Second half: detect the tags of the frame in the next slot (``ingest_next`` / ``next_frames`` put it there) inside the
        windows ``next_windows`` left, and pack them into that slot's input buffers - on the current stream, which the caller orders
        after ``next_windows`` and after the step that last read the slot.  Nothing the step in flight reads is touched, so the
        detector of frame f+1 runs under the PnP / refinement chain of frame f; the step for f+1 is then ``step(None)``."""
        slot = (self.cur + 1) % self.SLOTS
        self._detect_into(slot, self._rects_next if track_window else None, min_margin, refine_win, max_tags)

    def _detect_into(self, slot, rects, min_margin, refine_win, max_tags):
        """Detector + decision-margin filter + id mapping of the frame in ``slot`` into that slot's input buffers, on the current
        stream.  The detector's workspace belongs to the context, so two detections never overlap: each waits for the one issued
        before it, whatever streams they were issued on (``step_frames`` on the step's stream, ``detect_next`` on a side stream)."""
        t = self.ctx.torch
        cur = t.cuda.current_stream(self.ctx.tdev)
        if self._det_done is not None:
            cur.wait_event(self._det_done)
        else:
            self._det_done = t.cuda.Event()
        _, img, ntags_in, val = self._in[slot]
        det = self.ctx.detect_tags(self.pyr[slot], max_tags=max_tags, refine_win=refine_win, rects=rects)
        self.ctx.pack_detections(det, self.group_ids, min_margin, out=(img, val, ntags_in, self.n_unknown))
        self._det_done.record(cur)
        return det

    def step(self, img_pts, valid=None, n_tags=None, frames=None):
        """img_pts [S,P,2] f32, valid [S,P] u8 (corner-level; all four corners of a detected tag set),
        n_tags [S] i32 accepted detections - or ``step(packed)`` with the tensor ``pack_inputs`` made of them.  ``frames`` [S,H,W] u8 is copied into the current slot
        unless the caller wrote ``self.frames`` directly.  Returns a dict of device tensors (valid until the slot
        comes round again when CUDA graphs are in use: the graph of a slot reuses its output buffers)."""
        ctx, t = self.ctx, self.ctx.torch
        slot = self.cur
        if frames is not None:
            ctx.upload_frames(self.pyr[slot], frames)
            self._built[slot] = False
        if not self._built[slot]:
            ctx.build_pyramid(self.pyr[slot])                # K1 (unless ingest_next built this slot during the last step)
        self._built[slot] = False                            # the caller writes the next frame into it before it is used again
        if img_pts is not None and valid is None:            # the three inputs packed by ``pack_inputs``: one copy
            self.in_all.copy_(img_pts, non_blocking=True)
        elif img_pts is not None:                            # None: step_frames has filled the input buffers on the device
            self.in_img.copy_(ctx._dev(img_pts, t.float32))
            self.in_valid.copy_(ctx._dev(valid, t.uint8))
            self.in_ntags.copy_(ctx._dev(n_tags, t.int32))
        if self._epoch != getattr(ctx, "config_epoch", 0):
            # set_camera / set_model since the graphs were captured: they hold the camera by value and the model's pointers,
            # so replaying them would silently keep the old ones - drop them and capture again
            self._graphs = [None] * self.SLOTS
            self._outs = [None] * self.SLOTS
            self._epoch = getattr(ctx, "config_epoch", 0)
        if self.use_graphs and self._graphs[slot] is not None:
            self._graphs[slot].replay()
            out = self._outs[slot]
        elif self.use_graphs and self._steps >= 2:
            # two steps have run eagerly (lazy one-time setup is done): capture this slot and replay it
            g = t.cuda.CUDAGraph()
            t.cuda.synchronize(ctx.tdev)
            # captured on the caller's stream when that is not the default one, so that the kernel nodes take its priority: a
            # caller that runs the steps on a high-priority stream keeps the latency-bound chain ahead of the bandwidth-bound
            # ingest (copy + K1) it overlaps with
            cur = t.cuda.current_stream(ctx.tdev)
            with t.cuda.graph(g, stream=None if cur == t.cuda.default_stream(ctx.tdev) else cur):
                out = self._body(slot)
            g.replay()
            self._graphs[slot], self._outs[slot] = g, out
        else:
            l0 = ctx.launch_count()
            out = self._body(slot)
            self.kernels_per_step = ctx.launch_count() - l0     # what a graph replay launches, too
        self._steps += 1
        self.cur = (slot + 1) % self.SLOTS
        return out


class StreamGroups:
    """The streams of one GPU as G independent ``BatchedPoseDetector``s, each with its own context (its own camera and group, if
    the cameras differ), CUDA stream and ingest stream; the host drives the groups in turn from one thread.

    Streams are independent (the reference runs one ``PoseDetector`` per camera) and the kernels work frame by frame, so every
    stream gets exactly the arithmetic of the single batch: poses and accept decisions are bit-identical (tested).  What it is
    NOT is a way to more poses per second on one camera model: a frame-step is one dependent chain of latency-bound kernels whose
    length hardly depends on the batch (64 streams 0.33 ms, 32 streams 0.32 ms), so G groups of S/G streams in flight finish no
    sooner than one batch of S, and the ~0.1 ms of host work per group-step binds from G = 4 on (measured on B200, 64 streams x
    1080p, `bench.py --workload streams --stream-groups G`: 195 / 199 / 134 / 78 thousand poses/s at G = 1 / 2 / 4 / 8).  Use it
    for groups of cameras that differ (resolution, calibration, tag group), not for speed."""

    def __init__(self, contexts, n_streams: int, width: int, height: int, obj_pts: np.ndarray, **kw):
        if not contexts:
            raise ValueError("at least one context")
        g = len(contexts)
        if n_streams < g:
            raise ValueError(f"{n_streams} streams cannot fill {g} groups")
        t = contexts[0].torch
        self.torch, self.n, self.g = t, int(n_streams), g
        bounds = [round(k * n_streams / g) for k in range(g + 1)]
        self.slices = [slice(bounds[k], bounds[k + 1]) for k in range(g)]
        self.dets = [BatchedPoseDetector(c, sl.stop - sl.start, width, height, obj_pts, **kw) for c, sl in zip(contexts, self.slices)]
        dev = contexts[0].tdev
        self.mains = [t.cuda.Stream(dev) for _ in range(g)]
        self.sides = [t.cuda.Stream(dev) for _ in range(g)]
        self.landed = [t.cuda.Event() for _ in range(g)]
        self.stepped = [t.cuda.Event() for _ in range(g)]
        self._joined = t.cuda.Event()

    def reset(self):
        for d in self.dets:
            d.reset()

    def fork(self):
        """The groups' streams wait for what has been queued on the current stream (e.g. the frames of the first step)."""
        self._joined.record(self.torch.cuda.current_stream())
        for m, ev in zip(self.mains, self.stepped):
            m.wait_event(self._joined)
            ev.record(m)

    def join(self):
        """The current stream waits for every group."""
        cur = self.torch.cuda.current_stream()
        for m in self.mains:
            ev = self.torch.cuda.Event()
            ev.record(m)
            cur.wait_event(ev)

    def load(self, frames):
        """frames [S,H,W] -> the current slot of every group (on the current stream; call ``fork`` afterwards)."""
        for d, sl in zip(self.dets, self.slices):
            d.frames.copy_(frames[sl])

    def step(self, img_pts=None, valid=None, n_tags=None, next_frames=None, pose_out=None, accepted_out=None, **frames_kw):
        """One frame of every stream.  Detections as for ``BatchedPoseDetector.step`` ([S,...] arrays, sliced per group), or none
        at all: the detector runs on the device (``step_frames``).  ``next_frames`` [S,H,W]: the frames of the following step,
        ingested (copy + K1) on each group's side stream under the step in flight.  ``pose_out`` [S,6] / ``accepted_out`` [S]:
        receive the poses and the accept flags (on the groups' streams: ``join`` before reading them elsewhere).
        Returns the groups' output dicts (buffers of the captured graphs, valid on the group's stream until its slot comes round)."""
        t = self.torch
        outs = []
        for k, (d, sl) in enumerate(zip(self.dets, self.slices)):
            main, side = self.mains[k], self.sides[k]
            with t.cuda.stream(main):
                if next_frames is not None:
                    side.wait_event(self.stepped[k])                 # the free slot was last read by the previous step
                    with t.cuda.stream(side):
                        d.ingest_next(next_frames[sl])
                        self.landed[k].record(side)
                out = d.step_frames(**frames_kw) if img_pts is None else d.step(img_pts[sl], valid[sl], n_tags[sl])
                if pose_out is not None:
                    pose_out[sl].copy_(out["pose"])
                if accepted_out is not None:
                    accepted_out[sl].copy_(out["accepted"].reshape(-1))
                self.stepped[k].record(main)
                if next_frames is not None:
                    main.wait_event(self.landed[k])
            outs.append(out)
        return outs


def tag_positions(tag_ids) -> dict:
    """tag id -> position of the tag in the group, i.e. in the JSON key order that defines the corner index 4 * position + j
    (detect_pose.py:122, :202: ``extrinsics`` is filled, and ``all_objpts`` stacked, in that order).  ``tag_ids`` is that
    ordered sequence, e.g. ``list(PoseDetector.extrinsics)``."""
    pos = {}
    for k, tag in enumerate(tag_ids):
        tag = int(tag)
        if tag in pos:
            raise ValueError(f"tag id {tag} appears twice in the group")
        pos[tag] = k
    return pos


def pack_detections(dets_per_stream, tag_ids=None, n_tags_total: Optional[int] = None):
    """[(tag_id, corners (4,2)), ...] per stream -> (img_pts [S,4T,2] f32, valid [S,4T] u8, n_tags [S] i32).

    ``tag_ids``: the group's tag ids in JSON key order (see ``tag_positions``); a detection's corners go to the slots of its
    tag's POSITION in that order, which is where ``all_objpts`` holds its object points (detect_pose.py:405-437 looks the
    object points up by id, ``extrinsics[tag_id]``).  Default: ids 0..T-1 in order, the synthetic dodecahedron.  An id that is not
    in the group raises KeyError, as the reference does (detect_pose.py:408-415 catches ValueError only)."""
    if tag_ids is None:
        tag_ids = range(synth.NUM_TAGS if n_tags_total is None else n_tags_total)
    pos = tag_ids if isinstance(tag_ids, dict) else tag_positions(tag_ids)
    total = len(pos)
    if n_tags_total is not None and n_tags_total != total:
        raise ValueError(f"n_tags_total={n_tags_total} but the group has {total} tags")
    s = len(dets_per_stream)
    img = np.zeros((s, 4 * total, 2), np.float32)
    valid = np.zeros((s, 4 * total), np.uint8)
    n = np.zeros(s, np.int32)
    for i, dets in enumerate(dets_per_stream):
        for tag, corners in dets:
            k = pos[int(tag)]                      # KeyError for an id outside the group
            img[i, 4 * k:4 * k + 4] = np.asarray(corners, dtype=np.float32).reshape(4, 2)
            valid[i, 4 * k:4 * k + 4] = 1
        n[i] = int(valid[i].sum()) // 4            # a tag reported twice fills one slot
    return img, valid, n
