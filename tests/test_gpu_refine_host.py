"""agt_refine_host through each of its upload paths, against the device path (build_pyramid + refine) bit for bit.

How the frames of a call reach the GPU depends on where they live and on the frame width:
  GATHER  pinned, device-mapped frames (16-byte aligned, width % 16 == 0): a kernel reads the ROI rectangles over PCIe
  STAGED  pageable frames, upload threads > 0, width % 16 == 0: threads pack the rectangles into pinned staging
  COPIES  everything else with ROI upload on, and the redo of frames that left their rectangle: one 2-D copy per rectangle
  WHOLE   ROI upload off, width % 16 == 0: one copy per chunk
None of that may change a bit of the result, nor (among the ROI paths) the bytes moved."""
import numpy as np
import pytest

from accurate_aprilgroup_tracking_b200 import synth

pytestmark = pytest.mark.gpu
KEYS = ("pose", "cost", "n_valid", "evals", "status")
CHUNK = 1024                    # frames per chunk of agt_refine_host at these frame sizes (csrc/agt_api.cu)


@pytest.fixture()
def host(lib_built):
    """A fresh host context per test: what an earlier call left in a context must not matter, so each case starts clean."""
    from accurate_aprilgroup_tracking_b200 import cv_compat
    h = cv_compat.HostContext(0)
    s, tg, n, c = synth.surface_model()
    h.set_model(s, tg, n, c, synth.model_pitch())
    yield h
    h.close()


def _render(ctx, cam, n, seed, n_hyp=1):
    """n rendered frames of `cam` (device) and initial poses near the truth, some far enough off that their refinement
    leaves the predicted ROI and is redone from the whole frame."""
    rng = np.random.default_rng(seed)
    truth = np.array([synth.random_pose(rng) for _ in range(n)])
    pyr = ctx.alloc_pyramid(n, cam.width, cam.height, 1)
    ctx.render(pyr, truth, np.arange(n) + seed)
    init = truth + np.concatenate([rng.normal(0, 0.008, (n, 3)), rng.normal(0, 0.0004, (n, 3))], axis=1)
    init[3, 3] += 0.012             # 12 mm off: the LM run starts (and wanders) outside the predicted ROI
    init[7, :3] += 0.25
    init[n - 2, 3] -= 0.015
    init = np.repeat(init[:, None, :], n_hyp, axis=1)
    if n_hyp > 1:
        init[:, 1, :3] += 0.01
        init[:, 2, 3:] += 0.002
    return pyr.frames, init


def _device_path(ctx, cam, frames, init, roi=True):
    """build_pyramid + refine over the same frames per launch as agt_refine_host: chunks of CHUNK frames, then (ROI upload)
    the frames whose ROI refinement left its rectangle, all of them in one launch per chunk.  refine_impl picks its launch
    form from the job count, and the forms may differ in the last bits (test_gpu_dpr_forms.py: test_forms_agree), so the
    same bits need the same launches.  Frames that stay inside their rectangle get the same bits fused or not
    (test_fused_equals_unfused)."""
    t = ctx.torch
    n, n_hyp = init.shape[:2]

    def refine(idx, fused):
        p = ctx.alloc_pyramid(len(idx), cam.width, cam.height, 4)
        p.frames.copy_(frames[t.as_tensor(idx, device=frames.device)])
        ctx.build_pyramid(p)
        return ctx.refine(p, init[idx], n_hyp), (ctx.refine_fused(p, init[idx], n_hyp)["redo"] if fused else None)

    runs = [refine(np.arange(b0, min(b0 + CHUNK, n)), roi) for b0 in range(0, n, CHUNK)]
    out = {k: t.cat([r[k] for r, _ in runs]) for k in KEYS}
    if roi:
        ids = t.cat([redo for _, redo in runs]).nonzero().flatten().cpu().numpy()
        assert len(ids) > 0, "no frame leaves its ROI: the redo pass would go untested"
        for b0 in range(0, len(ids), CHUNK):
            part = ids[b0:b0 + CHUNK]
            r, _ = refine(part, False)
            for k in KEYS:
                out[k][t.as_tensor(part, device=frames.device)] = r[k]
    want = {k: v.cpu().numpy() for k, v in out.items()}
    if n_hyp > 1:
        want["best"] = ctx.select_best(out)[0].cpu().numpy()
    return want


def _assert_same(got, want, what):
    for k in want:
        assert np.array_equal(got[k].reshape(want[k].shape), want[k]), (what, k)


def _pinned(frames, offset=0):
    from accurate_aprilgroup_tracking_b200 import cv_compat
    flat = cv_compat.pinned_frames((frames.size + offset,))
    view = flat[offset:offset + frames.size].reshape(frames.shape)
    view[...] = frames
    return view


def test_every_upload_path_equals_device_path(host, ctxvga):
    cam = synth.CAMERA_VGA
    dframes, init = _render(ctxvga, cam, 40, 600)
    want = _device_path(ctxvga, cam, dframes, init)
    frames = dframes.cpu().numpy()
    h2d = {}
    _assert_same(host.refine_poses(_pinned(frames), init, cam.mtx), want, "gather")
    h2d["gather"] = host.last_h2d_bytes()
    _assert_same(host.refine_poses(frames, init, cam.mtx), want, "staged")
    h2d["staged"] = host.last_h2d_bytes()
    host.set_upload_threads(0)
    _assert_same(host.refine_poses(frames, init, cam.mtx), want, "copies")
    h2d["copies"] = host.last_h2d_bytes()
    assert len(set(h2d.values())) == 1, h2d
    host.set_roi_upload(False)
    _assert_same(host.refine_poses(frames, init, cam.mtx), _device_path(ctxvga, cam, dframes, init, roi=False), "whole")
    assert host.last_h2d_bytes() == init.nbytes + frames.nbytes > h2d["copies"]
    host.set_roi_upload(True)
    host.set_upload_threads(4)
    dframes3, init3 = _render(ctxvga, cam, 12, 640, n_hyp=3)
    want3 = _device_path(ctxvga, cam, dframes3, init3)
    frames3 = dframes3.cpu().numpy()
    _assert_same(host.refine_poses(frames3, init3, cam.mtx, n_hyp=3), want3, "staged, 3 hypotheses")
    _assert_same(host.refine_poses(_pinned(frames3), init3, cam.mtx, n_hyp=3), want3, "gather, 3 hypotheses")


def test_width_not_a_multiple_of_16(host, lib_built):
    from accurate_aprilgroup_tracking_b200.context import AgtContext
    cam = synth.Camera(632, 480, 600.0, 600.0, 316.0, 240.0)
    ctx = AgtContext(0, cam.mtx, None)
    try:
        ctx.set_synthetic_model()
        dframes, init = _render(ctx, cam, 24, 660)
        want, want_whole = _device_path(ctx, cam, dframes, init), _device_path(ctx, cam, dframes, init, roi=False)
        frames = dframes.cpu().numpy()
    finally:
        ctx.close()
    _assert_same(host.refine_poses(frames, init, cam.mtx), want, "roi")                      # per-rectangle copies
    _assert_same(host.refine_poses(_pinned(frames), init, cam.mtx), want, "roi, pinned")
    host.set_roi_upload(False)
    _assert_same(host.refine_poses(frames, init, cam.mtx), want_whole, "whole frames")        # per-frame copies (pitch != width)


def test_unaligned_pinned_frames_after_a_smaller_pageable_call(host, ctxvga):
    """Pinned frames whose base is not 16-byte aligned cannot take the gather kernel; they must take the per-rectangle
    copies even when an earlier call on the context packed (fewer) pageable frames through staging."""
    cam = synth.CAMERA_VGA
    dframes, init = _render(ctxvga, cam, 40, 680)
    want = _device_path(ctxvga, cam, dframes, init)
    frames = dframes.cpu().numpy()
    host.refine_poses(frames[:4], init[:4], cam.mtx)
    got = host.refine_poses(_pinned(frames, offset=1), init, cam.mtx)
    got_bytes = host.last_h2d_bytes()
    host.set_upload_threads(0)
    copies = host.refine_poses(frames, init, cam.mtx)
    _assert_same(got, {k: copies[k] for k in KEYS}, "unaligned pinned vs copies")
    assert got_bytes == host.last_h2d_bytes()
    _assert_same(got, want, "unaligned pinned")


def test_more_than_two_chunks(host, ctxvga):
    """2 x 1024 + 40 VGA frames are three chunks of the double-buffered upload: chunk 2 reuses the buffers (and the
    staging) of chunk 0 and has to wait for them."""
    cam = synth.CAMERA_VGA
    dframes, init = _render(ctxvga, cam, 2 * CHUNK + 40, 700)
    want = _device_path(ctxvga, cam, dframes, init)
    frames = dframes.cpu().numpy()
    _assert_same(host.refine_poses(_pinned(frames), init, cam.mtx), want, "gather")
    gather_bytes = host.last_h2d_bytes()
    _assert_same(host.refine_poses(frames, init, cam.mtx), want, "staged")
    assert host.last_h2d_bytes() == gather_bytes
