"""CPU oracle for tag identification and detection (SURVEY.md 8f row N3).

TEST INFRASTRUCTURE (see oracle/__init__.py).  The reference's detector is the un-vendored swatbotics `apriltag` C library
(detect_pose.py:86-95 tag36h11, :368-371 detect, :389-400 the `decision_margin < 50` filter and the corner order of
transform_helper.py:56-59); it is absent from the image.  What the image has is OpenCV's ArUco module with the same family
(cv2.aruco.DICT_APRILTAG_36h11, the table synth.TAG36H11_CODES was dumped from), so:

  `detect_cv`     cv2.aruco.ArucoDetector.detectMarkers - the oracle for WHICH tags are in a frame and where (its corners are
                  contour points, ~1 px from the true corners); ids and corner order converted to the reference's conventions
  `decode_np`     the frozen specification of the GPU identification step (csrc/agt_tags.cu): 8x8 cells (6x6 data + black border)
                  sampled through the quad's homography, threshold half way between the darkest and the brightest cell,
                  border check, dictionary match over the four rotations.  Pinned by the tests: on every tag cv2.aruco
                  finds, decode_np(aruco's corners) returns aruco's id; on the true corners it returns the true id, rotation 0.

Corner order everywhere: the reference's (-,-), (-,+), (+,+), (+,-) in tag coordinates with y up, i.e. bottom-left, top-left,
top-right, bottom-right of the tag as printed (transform_helper.py:56-59).
"""
from __future__ import annotations

import cv2 as cv
import numpy as np

from accurate_aprilgroup_tracking_b200 import synth

CELLS = 8                 # 6x6 data cells + one cell of black border on each side
SUB = (-0.25, 0.0, 0.25)  # sample offsets inside a cell, in cells
MAX_BORDER_ERRORS = 2
MAX_HAMMING = 2


def code_bits(code: int) -> np.ndarray:
    """(6,6) bits of a tag36h11 code word, row 0 = top row of the tag (synth.tag_cells)."""
    return np.array([(code >> (35 - i)) & 1 for i in range(36)], np.uint8).reshape(6, 6)


def detect_cv(gray: np.ndarray):
    """-> list of (tag_id, corners (4,2) f64 in the reference's order) from cv2.aruco (corners there: TL, TR, BR, BL)."""
    det = cv.aruco.ArucoDetector(cv.aruco.getPredefinedDictionary(cv.aruco.DICT_APRILTAG_36h11), cv.aruco.DetectorParameters())
    corners, ids, _ = det.detectMarkers(gray)
    out = []
    if ids is not None:
        for c, i in zip(corners, ids.ravel().tolist()):
            c = c.reshape(4, 2).astype(np.float64)
            out.append((int(i), np.stack([c[3], c[0], c[1], c[2]])))
    return out


def square_to_quad(q: np.ndarray):
    """Projective map of the unit square (s right, t down; (0,0) = top-left) onto the quad with corners in the reference's order
    (BL, TL, TR, BR) -> coefficients (a, b, c, d, e, f, g, h) of x = (a s + b t + c) / (g s + h t + 1), y = (d s + e t + f) / (...)."""
    (x3, y3), (x0, y0), (x1, y1), (x2, y2) = [tuple(map(float, p)) for p in q]       # TL=(0,0) TR=(1,0) BR=(1,1) BL=(0,1)
    dx1, dx2, sx = x1 - x2, x3 - x2, x0 - x1 + x2 - x3
    dy1, dy2, sy = y1 - y2, y3 - y2, y0 - y1 + y2 - y3
    den = dx1 * dy2 - dx2 * dy1
    g = (sx * dy2 - dx2 * sy) / den
    h = (dx1 * sy - sx * dy1) / den
    return (x1 - x0 + g * x1, x3 - x0 + h * x3, x0, y1 - y0 + g * y1, y3 - y0 + h * y3, y0, g, h)


def cell_means(gray: np.ndarray, quad: np.ndarray) -> np.ndarray:
    """(8,8) mean intensity of 3x3 bilinear samples per cell; NaN if a sample leaves the image."""
    a, b, c, d, e, f, g, h = square_to_quad(quad)
    hh, ww = gray.shape
    out = np.zeros((CELLS, CELLS))
    img = gray.astype(np.float64)
    for r in range(CELLS):
        for cc in range(CELLS):
            acc = 0.0
            for dt in SUB:
                for ds in SUB:
                    s, t = (cc + 0.5 + ds) / CELLS, (r + 0.5 + dt) / CELLS
                    w = g * s + h * t + 1.0
                    x, y = (a * s + b * t + c) / w, (d * s + e * t + f) / w
                    x0, y0 = int(np.floor(x)), int(np.floor(y))
                    if x0 < 0 or y0 < 0 or x0 + 1 >= ww or y0 + 1 >= hh:
                        return np.full((CELLS, CELLS), np.nan)
                    fx, fy = x - x0, y - y0
                    acc += ((1 - fx) * (1 - fy) * img[y0, x0] + fx * (1 - fy) * img[y0, x0 + 1]
                            + (1 - fx) * fy * img[y0 + 1, x0] + fx * fy * img[y0 + 1, x0 + 1])
            out[r, cc] = acc / 9.0
    return out


def decode_np(gray: np.ndarray, quad: np.ndarray, codes=None, max_hamming: int = MAX_HAMMING):
    """-> (tag_id or -1, rotation 0..3, hamming, margin).  rotation k: the quad's first corner is the tag's corner k (so the
    tag's corners in the reference's order are np.roll(quad, k, axis=0)); margin = mean |cell mean - threshold| (the
    analogue of apriltag's decision_margin, which the reference compares with 50, detect_pose.py:389)."""
    codes = synth.TAG36H11_CODES if codes is None else codes
    m = cell_means(gray, np.asarray(quad, dtype=np.float64))
    if np.isnan(m).any():
        return -1, 0, 255, 0.0
    thr = 0.5 * (m.min() + m.max())
    bits = (m > thr).astype(np.uint8)
    margin = float(np.abs(m - thr).mean())
    border = np.concatenate([bits[0], bits[-1], bits[1:-1, 0], bits[1:-1, -1]])
    if int(border.sum()) > MAX_BORDER_ERRORS:
        return -1, 0, 255, margin
    data = bits[1:-1, 1:-1]
    best = (-1, 0, 255)
    for rot in range(4):
        # the quad starts at tag corner `rot`: its sampled grid is the tag's grid turned by rot quarter turns
        grid = np.rot90(data, -rot)
        word = 0
        for v in grid.ravel():
            word = (word << 1) | int(v)
        for tag_id, code in enumerate(codes):
            hd = bin(word ^ int(code)).count("1")
            if hd < best[2]:
                best = (tag_id, rot, hd)
    if best[2] > max_hamming:
        return -1, 0, best[2], margin
    return best[0], best[1], best[2], margin


# ---------------------------------------------------------------------------------------------------------------------------
# quads_np: the frozen specification of the detector's first stage (csrc/agt_tags.cu, agt_tag_quads): threshold -> 4-connected
# dark components -> three farthest-point passes over the boundary pixels -> quadrilateral filter -> corner placement.  Plain
# numpy / scipy (the components by scipy.ndimage.label: independent of both union-finds of the device).
MAX_COMPONENTS = 4096         # component numbers per frame
RUNS_ENT_CAP = 4096           # non-empty 32-pixel items / runs the shared-memory union-find holds; beyond: the global-memory one
RUNS_RUN_CAP = 6144
MIN_AREA = 48                 # a component below this can never become a quad and takes no number
TILE = 32
F32 = np.float32


def frame_window(w: int, h: int, rect=None):
    """-> (x0, y0, ww, hh): the whole frame for None or an empty rectangle, else the rectangle clipped to the frame with its left
    edge rounded down to a multiple of 16."""
    if rect is not None:
        x0, y0, x1, y1 = max(int(rect[0]), 0) & ~15, max(int(rect[1]), 0), min(int(rect[2]), w), min(int(rect[3]), h)
        if x1 > x0 and y1 > y0:
            return x0, y0, x1 - x0, y1 - y0
    return 0, 0, w, h


def threshold_of(lo, hi):
    """Integer threshold for darkest lo and white level hi (arrays allowed); -1 (no dark pixel) without 40 levels of contrast."""
    lo, hi = np.asarray(lo, np.int64), np.asarray(hi, np.int64)
    return np.where(hi - lo < 40, -1, lo + (35 * (hi - lo)) // 100)


def threshold_map(img: np.ndarray, local: bool):
    """img = the window -> (lo, hi, per-pixel threshold [hh, ww] int64, tile maxima or None).  Local white level: hi of a pixel is
    the brightest pixel of the 3 x 3 tiles (32 rows x one 32-pixel item, clamped at the window's edges) around its tile."""
    hh, ww = img.shape
    lo, hi = int(img.min()), int(img.max())
    if not local:
        return lo, hi, np.full((hh, ww), int(threshold_of(lo, hi)), np.int64), None
    th, tw = -(-hh // TILE), -(-ww // TILE)
    pad = np.zeros((th * TILE, tw * TILE), np.uint8)
    pad[:hh, :ww] = img
    tiles = pad.reshape(th, TILE, tw, TILE).max(axis=(1, 3)).astype(np.int64)
    e = np.pad(tiles, 1, mode="edge")
    hi3 = np.max([e[1 + dy:1 + dy + th, 1 + dx:1 + dx + tw] for dy in (-1, 0, 1) for dx in (-1, 0, 1)], axis=0)
    thr = threshold_of(lo, hi3)
    return lo, hi, np.repeat(np.repeat(thr, TILE, axis=0), TILE, axis=1)[:hh, :ww], tiles


def item_counts(dark: np.ndarray):
    """-> (non-empty 32-pixel items, runs): a run is a maximal dark row segment inside one item."""
    hh, ww = dark.shape
    ch = -(-ww // 32)
    d = np.zeros((hh, ch * 32), bool)
    d[:, :ww] = dark
    d = d.reshape(hh, ch, 32)
    starts = d.copy()
    starts[:, :, 1:] &= ~d[:, :, :-1]
    return int(d.any(axis=2).sum()), int(starts.sum())


def _f32_sq_sum(a, b):
    """a*a + b*b in float32 as the device may evaluate it: plain, or contracted into an FMA either way round."""
    a64, b64 = a.astype(np.float64), b.astype(np.float64)
    plain = (a * a).astype(F32) + (b * b).astype(F32)
    return [plain.astype(F32), (a64 * a64 + (b * b).astype(F32)).astype(F32), (b64 * b64 + (a * a).astype(F32)).astype(F32)]


def _key(v, idx):
    return (np.maximum(np.asarray(v, F32), F32(0)).view(np.uint32).astype(np.uint64) << np.uint64(32)) | idx.astype(np.uint64)


def _seg_max(keys, seg_start):
    return np.maximum.reduceat(keys, seg_start) if len(keys) else keys


def quads_np(gray: np.ndarray, rect=None, local: bool = True, refine_win: int = 4):
    """One frame [h, w] uint8 -> dict with every intermediate of the first stage: window, lo / hi / threshold map, dark mask, labels
    (scipy, 4-connected), per-component statistics in window coordinates, item / run counts and the predicted union-find path,
    boundary mask, the farthest points of each pass with the device's tie rule (key = float key << 32 | pixel index: the larger
    index wins) and the tie counts, and the emitted quads (clockwise, half a pixel outwards from the centroid, frame
    coordinates; cwin = the corner-refinement window).  ``local``: the local white level (the detector's default on whole
    frames) or one white level per window.  Pass 0 keys are float32 distances from the float32 centroid; the device may
    contract a*a + b*b into an FMA, so each component gets the pass-0 winner of each evaluation order (`alts`, almost always one)
    and the quad that follows from each."""
    from scipy import ndimage

    h, w = gray.shape
    x0w, y0w, ww, hh = frame_window(w, h, rect)
    img = np.ascontiguousarray(gray[y0w:y0w + hh, x0w:x0w + ww])
    lo, hi, thr, tiles = threshold_map(img, local)
    dark = img.astype(np.int64) < thr
    n_items, n_runs = item_counts(dark)
    lab, n_all = ndimage.label(dark)                       # default structure: 4-connectivity
    flat = lab.ravel()
    yy, xx = np.divmod(np.arange(hh * ww, dtype=np.int64), ww)
    area = np.bincount(flat, minlength=n_all + 1)
    sx = np.bincount(flat, weights=xx, minlength=n_all + 1).astype(np.int64)
    sy = np.bincount(flat, weights=yy, minlength=n_all + 1).astype(np.int64)
    bbox = np.zeros((n_all + 1, 4), np.int64)              # x0, y0, x1, y1 (inclusive)
    for k, sl in enumerate(ndimage.find_objects(lab), 1):
        bbox[k] = sl[1].start, sl[0].start, sl[1].stop - 1, sl[0].stop - 1
    big = np.flatnonzero(area >= MIN_AREA)
    big = big[big > 0]
    # boundary: dark with a background 4-neighbour, or on the window's edge
    p = np.pad(dark, 1)
    boundary = dark & ~(p[:-2, 1:-1] & p[2:, 1:-1] & p[1:-1, :-2] & p[1:-1, 2:])
    bidx = np.flatnonzero(boundary.ravel() & (area[flat] >= MIN_AREA))
    blab = flat[bidx]
    order = np.argsort(blab, kind="stable")
    bidx, blab = bidx[order], blab[order]
    bx, by = xx[bidx], yy[bidx]
    seg_start = np.flatnonzero(np.r_[True, blab[1:] != blab[:-1]]) if len(blab) else np.zeros(0, np.int64)
    seg_lab = blab[seg_start]
    seg_of = np.repeat(np.arange(len(seg_start)), np.diff(np.r_[seg_start, len(blab)]))
    ties = {"pass0": 0, "pass1": 0, "pass2": 0, "pass0_orders": 0}

    def pick(keys):
        m = _seg_max(keys, seg_start)
        return (m & np.uint64(0xffffffff)).astype(np.int64), m

    def count_ties(vals):
        vmax = np.maximum.reduceat(vals, seg_start) if len(vals) else vals
        return int((np.bincount(seg_of, weights=(vals == vmax[seg_of]), minlength=len(seg_start)) > 1).sum())

    cx = (sx[blab].astype(np.float64) / area[blab]).astype(F32)
    cy = (sy[blab].astype(np.float64) / area[blab]).astype(F32)
    v0 = _f32_sq_sum(bx.astype(F32) - cx, by.astype(F32) - cy)
    picks0 = [pick(_key(v, bidx))[0] for v in v0]
    ties["pass0"] = count_ties(v0[0])
    ties["pass0_orders"] = int((np.stack(picks0).min(axis=0) != np.stack(picks0).max(axis=0)).sum()) if len(seg_start) else 0

    def passes12(p0):
        px0, py0 = p0 % ww, p0 // ww
        d1 = (bx - px0[seg_of]) ** 2 + (by - py0[seg_of]) ** 2
        assert d1.max(initial=0) < 1 << 24
        p2, k2 = pick(_key(d1.astype(F32), bidx))
        px2, py2 = p2 % ww, p2 // ww
        d = (px2 - px0)[seg_of] * (by - py0[seg_of]) - (py2 - py0)[seg_of] * (bx - px0[seg_of])
        assert np.abs(d).max(initial=0) < 1 << 24
        zero = np.zeros(len(d), np.uint64)
        sp, ksp = pick(np.where(d > 0, _key(np.abs(d).astype(F32), bidx), zero))
        sn, ksn = pick(np.where(d < 0, _key(np.abs(d).astype(F32), bidx), zero))
        return p2, k2, sp, ksp, sn, ksn, d1, d

    comps = {}
    for v, p0 in zip(range(3), picks0):
        k0 = pick(_key(v0[v], bidx))[1]
        p2, k2, sp, ksp, sn, ksn, d1, d = passes12(p0)
        if v == 0:
            ties["pass1"] = count_ties(d1)
            ties["pass2"] = count_ties(np.where(d > 0, d, 0)) + count_ties(np.where(d < 0, -d, 0))
        for s, c in enumerate(seg_lab):
            alt = (int(p0[s]), int(sp[s]), int(p2[s]), int(sn[s]), bool(k0[s] and k2[s] and ksp[s] and ksn[s]))
            comps.setdefault(int(c), [])
            if alt not in comps[int(c)]:
                comps[int(c)].append(alt)

    quads = []                                             # one entry per component with an emitted quad
    filters = {}                                           # component -> its values in the quad filter (None: cut by the window)
    for c, alts in comps.items():
        x0, y0, x1, y1 = bbox[c]
        filters[c] = None
        if x0 <= 0 or y0 <= 0 or x1 >= ww - 1 or y1 >= hh - 1:
            continue
        res = [_emit(alt, ww, x0w, y0w, int(area[c]), int(sx[c]), int(sy[c]), refine_win) for alt in alts]
        filters[c] = res[0][1]
        outs = [q for q, _ in res if q is not None]
        assert len(outs) in (0, len(alts)), "the evaluation orders of pass 0 disagree on whether a quad is emitted"
        if outs:
            quads.append({"comp": c, "alts": outs})
    return {"window": (x0w, y0w, ww, hh), "lo": lo, "hi": hi, "thr": thr, "tiles": tiles, "dark": dark, "labels": lab, "n_all": n_all,
            "area": area, "bbox": bbox, "sx": sx, "sy": sy, "n_comp": len(big), "numbered_exact": len(big) <= MAX_COMPONENTS,
            "n_items": n_items, "n_runs": n_runs, "overflow": n_items > RUNS_ENT_CAP or n_runs > RUNS_RUN_CAP, "boundary": boundary,
            "far": comps, "filters": filters, "ties": ties, "quads": quads, "n_quads": len(quads)}


def _emit(alt, ww, x0w, y0w, area, sx, sy, refine_win):
    """emit_quad of csrc/agt_tags.cu in float32 for one component's farthest points -> (dict(corners (4,2) f32 frame
    coordinates, pix (4,) window pixel indices in corner order, cwin) or None, dict of the filter's values)."""
    p0, sp, p2, sn, keys_ok = alt
    info = {"area": area, "qa": None, "smin": None, "smax": None}
    if not keys_ok:
        return None, info
    pix = [p0, sp, p2, sn]
    qx = [F32(p % ww) for p in pix]
    qy = [F32(p // ww) for p in pix]
    area2 = F32(0)
    for k in range(4):
        area2 = F32(area2 + F32(qx[k] * qy[(k + 1) & 3] - qx[(k + 1) & 3] * qy[k]))
    qa = F32(F32(0.5) * abs(area2))
    info["qa"] = float(qa)
    if qa < F32(64) or F32(area) < F32(F32(0.25) * qa) or F32(area) > F32(F32(1.15) * qa):
        return None, info
    smin, smax, mean_side = F32(1e30), F32(0), F32(0)
    for k in range(4):
        dx, dy = F32(qx[(k + 1) & 3] - qx[k]), F32(qy[(k + 1) & 3] - qy[k])
        ln = np.sqrt(F32(dx * dx + dy * dy), dtype=F32)
        smin, smax, mean_side = min(smin, ln), max(smax, ln), F32(mean_side + F32(F32(0.25) * ln))
    info["smin"], info["smax"] = float(smin), float(smax)
    if smin < F32(6) or smin < F32(F32(0.08) * smax):
        return None, info
    cw = area2 > 0
    cx, cy = F32(sx / area), F32(sy / area)
    corners = np.zeros((4, 2), F32)
    order = []
    for k in range(4):
        j = k if cw else (4 - k) & 3
        dx, dy = F32(qx[j] - cx), F32(qy[j] - cy)
        ln = max(np.sqrt(F32(dx * dx + dy * dy), dtype=F32), F32(1e-3))
        corners[k] = (F32(F32(x0w) + qx[j]) + F32(F32(F32(0.5) * dx) / ln), F32(F32(y0w) + qy[j]) + F32(F32(F32(0.5) * dy) / ln))
        order.append(pix[j])
    cwin = min(max(int(F32(F32(F32(0.5) * mean_side) / F32(8)) + F32(0.5)), 2), max(refine_win, 1))
    return {"corners": corners, "pix": order, "cwin": cwin}, info
