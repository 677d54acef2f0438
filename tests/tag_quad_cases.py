"""The case set of tests/test_gpu_tag_quads.py: frames aimed at the paths and edges of the detector's first stage
(csrc/agt_tags.cu, agt_tag_quads), each with the target it names, checked on the CPU by oracle/tag_oracle.quads_np.

A case is a dict: name, gray [h, w] uint8, pitch (the row pitch of the device buffer; 16-aligned rows take the sixteen-pixel
reads, pitch % 4 == 0 the four-pixel word loads, any other pitch byte loads), rect (None = whole frame), local (threshold
mode: the local white level or one white level per window), pyramid (True: the frame can go through a Pyramid and the end-to-end
checks) and target: a function of the quads_np result that says whether the case hits what it is for.
"""
from __future__ import annotations

import numpy as np

from accurate_aprilgroup_tracking_b200 import synth
from oracle import tag_oracle as T

BG, INK = 200, 20
SM_COUNT = 148                   # B200


def _frame(w, h, bg=BG):
    return np.full((h, w), bg, np.uint8)


def draw_tag(img, x, y, cell, tag_id, ink=INK, white=None):
    """A tag36h11 tag with its top-left corner at (x, y), cells of `cell` px: black border + 6 x 6 data (white = 1)."""
    white = int(img[y, x]) if white is None else white
    img[y:y + 8 * cell, x:x + 8 * cell] = ink
    bits = T.code_bits(int(synth.TAG36H11_CODES[tag_id]))
    for r in range(6):
        for c in range(6):
            if bits[r, c]:
                img[y + (r + 1) * cell:y + (r + 2) * cell, x + (c + 1) * cell:x + (c + 2) * cell] = white


def _case(name, gray, target, pitch=None, rect=None, local=False, offset=0):
    w = gray.shape[1]
    return {"name": name, "gray": gray, "pitch": w if pitch is None else pitch, "rect": rect, "local": local, "offset": offset,
            "pyramid": (pitch is None or pitch == w) and w % 16 == 0 and offset == 0, "target": target}


def init_rows(ww, hh, frame_wh, batch, windowed):
    """INIT_ROWS of ccl_init_kernel's sixteen-pixel form for a window of ww x hh of a frame of w x h in a batch (the grid of
    agt_tag_quads: min(pixels / 256, max(16, (8 with windows, else 32) x SMs / batch)) CTAs of 8 warps per frame)."""
    w, h = frame_wh
    nwarps = 8 * min((w * h + 255) // 256, max(16, (8 if windowed else 32) * SM_COUNT // batch))
    wch, rows = (ww + 511) >> 9, 16
    while rows > 1 and wch * (-(-hh // rows)) < nwarps:
        rows >>= 1
    return rows


def _rendered(seed, cam):
    pose = synth.trajectory(seed, 1)[0]
    return synth.render(pose, cam, seed=seed), pose


def _object_rows(pose, cam):
    pts = synth.project(synth.object_points(), pose, cam)
    return int(pts[:, 1].min()), int(pts[:, 1].max())


# ---------------------------------------------------------------------------------------------------------- case builders
def threshold_cases():
    out = []
    # pixels at thr - 1, thr and thr + 1 (one white level: lo 10, hi 200 -> thr 76), as squares and as stripes through squares
    g = _frame(256, 160)
    g[5, 5] = 10
    thr = int(T.threshold_of(10, BG))
    for k, v in enumerate((thr - 1, thr, thr + 1)):
        g[20:44, 20 + 40 * k:44 + 40 * k] = v
        g[80:120, 20 + 60 * k:60 + 60 * k] = 30
        g[80:120, 39 + 60 * k] = v                            # a one-pixel column at v: the square is one component or two
    out.append(_case("threshold: pixels at thr-1 / thr / thr+1", g,
                     lambda r, thr=thr: int(r["thr"][0, 0]) == thr and r["dark"][30, 30] and not r["dark"][30, 70] and not r["dark"][30, 110]
                     and r["labels"][100, 30] == r["labels"][100, 50] and r["labels"][100, 90] != r["labels"][100, 110])
               )
    # contrast of 39 and 40 levels
    for span in (39, 40):
        g = _frame(256, 160, 100 + span)
        g[30:60, 30:60] = 100
        g[80:130, 100:150] = 100
        out.append(_case(f"threshold: hi - lo = {span}", g,
                         lambda r, span=span: (r["hi"] - r["lo"] == span) and ((r["n_comp"] == 0) if span == 39 else (r["n_comp"] == 2 and r["n_quads"] == 2))))
    # local white level: a bright patch in each of the nine tiles around the tile of a mid-gray square (only the patch makes it dark)
    for layout in ("16", "4"):
        for dy in (-1, 0, 1):
            for dx in (-1, 0, 1):
                g = _frame(320, 224, 100)
                g[200, 10] = 30                               # darkest pixel
                g[100:121, 134:155] = 60                      # inside tile (3, 4); 60 < thr only with 250 among the 3 x 3 tiles' maxima
                ty, tx = 3 + dy, 4 + dx
                py, px = 32 * ty + 14, 32 * tx + 14
                if dy == 0 and dx == 0:
                    py, px = 98, 160 - 4                       # inside the square's own tile, outside the square
                g[py:py + 2, px:px + 2] = 250
                out.append(_case(f"local threshold: bright patch in tile ({dy:+d}, {dx:+d}), {layout}-byte reads", g,
                                 lambda r: bool(r["dark"][110, 144]) and r["n_quads"] == 1,
                                 pitch=320 if layout == "16" else 324, local=True))
        g = _frame(320, 224, 100)
        g[200, 10] = 30
        g[100:121, 134:155] = 60
        g[14:16, 300:302] = 250                               # far away: the square stays light
        out.append(_case(f"local threshold: no bright tile near, {layout}-byte reads", g, lambda r: not r["dark"][110, 144],
                         pitch=320 if layout == "16" else 324, local=True))
    return out


def _shapes(w, h, seed):
    """Squares, rings and a tag spread over a frame, some cut by the right / bottom edge of a partial item."""
    rng = np.random.default_rng(seed)
    g = _frame(w, h)
    draw_tag(g, 10, 10, 6, int(rng.integers(0, len(synth.TAG36H11_CODES))))
    for k in range(6):
        x, y, s = int(rng.integers(70, w - 30)), int(rng.integers(5, h - 30)), int(rng.integers(10, 26))
        g[y:y + s, x:x + s] = INK
        if k % 2:
            g[y + 3:y + s - 3, x + 3:x + s - 3] = BG
    g[h - 40:h - 18, w - 22:w - 1] = INK                       # ends 1 px before the right edge: inside the last item
    g[40:60, w - 12:w] = INK                                  # cut by the right edge
    return g


def read_form_cases():
    out = []
    for w, pitch in ((256, 256), (257, 272), (287, 288), (513, 528), (527, 528), (257, 257), (513, 516), (287, 300)):
        g = _shapes(w, 150, w * 7 + pitch)
        out.append(_case(f"read form: width {w} (mod 32 = {w % 32}), pitch {pitch}, height 150", g, lambda r: r["n_quads"] >= 3, pitch=pitch))
    # the 4-byte / byte forms at an odd base address as well
    g = _shapes(256, 150, 3)
    out.append(_case("read form: 16-aligned pitch, frame at an odd address", g, lambda r: r["n_quads"] >= 3, pitch=256, offset=1))
    # a small window: INIT_ROWS comes down to 1 (few rows per warp for a window this size)
    g = _shapes(512, 300, 11)
    out.append(_case("read form: 96-row window (INIT_ROWS 1)", g, lambda r: r["window"][3] == 96 and r["n_comp"] >= 1, rect=(0, 5, 512, 101)))
    return out


def labelling_cases():
    out = []
    # diagonal contacts only: a checkerboard of 20 px squares and single-pixel diagonal touches
    g = _frame(512, 256)
    yy, xx = np.mgrid[0:256, 0:512]
    g[((yy // 20) + (xx // 20)) % 2 == 0] = INK
    out.append(_case("labelling: checkerboard, diagonal contacts only", g,
                     lambda r: r["n_comp"] == int((((np.arange(13)[:, None] + np.arange(26)[None]) % 2) == 0).sum()) and r["n_quads"] > 64))
    # one-pixel 4-connected bridges across item boundaries; whole dark items
    g = _frame(512, 256)
    for k in range(4):
        x0 = 64 * k + 8
        g[20:44, x0:x0 + 23] = INK                             # ends at 32 k' - 1
        g[20:44, x0 + 26:x0 + 50] = INK
        g[30, x0 + 23:x0 + 26] = INK                           # the bridge crosses x = 32 k' - 1 | 32 k'
    for k in range(3):
        x = 32 * (k + 2) - 1 + (k % 2)                          # vertical bridge on a column at an item's first / last bit
        g[80:100, x - 10:x + 10] = INK
        g[100:110, x] = INK
        g[110:130, x - 10:x + 10] = INK
    g[150:230, 320:448] = INK                                  # whole dark items (m == 0xffffffff)
    g[160:220, 352:416] = BG
    g[170:210, 362:406] = INK
    out.append(_case("labelling: one-pixel bridges at item boundaries, whole dark items", g,
                     lambda r: r["labels"][30, 10] == r["labels"][30, 40] and r["labels"][85, 63] == r["labels"][125, 63]
                     and r["labels"][160, 330] != 0 and (r["dark"][150, 320:352]).all()))
    # combs and staircases whose arms meet only at the last row; a spiral
    g = _frame(640, 320)
    g[10:120, 20:300:4] = INK                                  # teeth 1 px wide, 4 px apart
    g[10:120, 21:300:4] = INK
    g[120, 20:300] = INK                                       # joined at the bottom row only
    for k in range(60):                                        # staircase: 4-connected steps down to the right, joined at the end
        g[150 + k:152 + k, 20 + 4 * k:26 + 4 * k] = INK
    sp = np.zeros((150, 150), bool)
    x0, y0, x1, y1 = 0, 0, 149, 149
    while x1 - x0 > 6 and y1 - y0 > 6:                          # a rectangular spiral of 2 px lines
        sp[y0:y0 + 2, x0:x1 + 1] = True; sp[y0:y1 + 1, x1 - 1:x1 + 1] = True
        sp[y1 - 1:y1 + 1, x0 + 4:x1 + 1] = True; sp[y0 + 4:y1 + 1, x0 + 4:x0 + 6] = True
        x0, y0, x1, y1 = x0 + 4, y0 + 4, x1 - 4, y1 - 4
        sp[y0:y0 + 2, x0:x0 + 2] = False
    g[160:310, 450:600][sp] = INK
    out.append(_case("labelling: comb, staircase and spiral joined at their last row", g,
                     lambda r: r["labels"][10, 20] == r["labels"][10, 296] and r["labels"][150, 20] == r["labels"][209, 256]))
    # a serpentine through hundreds of items
    g = _frame(1024, 300)
    for k in range(35):
        y = 10 + 8 * k
        g[y:y + 2, 10:1010] = INK
        x = 1008 if k % 2 == 0 else 10
        if k < 34:
            g[y:y + 10, x:x + 2] = INK
    out.append(_case("labelling: a serpentine through hundreds of items", g,
                     lambda r: r["labels"][10, 10] == r["labels"][10 + 8 * 34, 500] and r["n_items"] > 1000))
    # tags whose border touches a decoy through one-pixel bridges at item boundaries
    g = _frame(512, 256)
    for k, tid in enumerate((3, 7, 11)):
        x = 40 + 150 * k - (40 + 150 * k) % 32
        draw_tag(g, x, 60, 8, tid)
        g[90:110, x + 70:x + 90] = INK                          # decoy right of the tag, bridged at the item boundary
        g[100, x + 64:x + 70] = INK if k != 2 else BG
        g[200:215, x:x + 40] = INK
    out.append(_case("labelling: tags bridged to decoys", g, lambda r: r["labels"][100, 32] == r["labels"][100, 32 + 75] and r["n_quads"] >= 1))
    return out


def _spread(g, region, shape_fn, n, step):
    """n copies of shape_fn(g, y, x) on a grid of `step` inside region (y0, x0, y1, x1), in scan order."""
    y0, x0, y1, x1 = region
    k = 0
    for y in range(y0, y1 - step[0] + 1, step[0]):
        for x in range(x0, x1 - step[1] + 1, step[1]):
            if k == n:
                return k
            shape_fn(g, y, x)
            k += 1
    return k


def table_cap_cases():
    out = []
    # entries 4096 / 4097: single dark pixels in separate items, plus a square
    for extra in (0, 1):
        g = _frame(640, 480)
        g[420:450, 300:330] = INK
        base = T.item_counts(g < T.threshold_of(INK, BG))[0]
        need = 4096 - base + extra
        n = _spread(g, (2, 0, 418, 640), lambda g, y, x: g.__setitem__((y, x + 5), INK), need, (2, 32))
        assert n == need
        out.append(_case(f"table caps: {4096 + extra} non-empty items", g,
                         lambda r, e=extra: r["n_items"] == 4096 + e and r["n_runs"] <= T.RUNS_RUN_CAP and r["overflow"] == bool(e)))
    # runs 6144 / 6145: two runs per item (entries stay below the cap), one item with a third run
    for extra in (0, 1):
        g = _frame(640, 480)
        g[420:450, 300:330] = INK
        items, runs = T.item_counts(g < T.threshold_of(INK, BG))
        need = (6144 - runs) // 2
        n = _spread(g, (2, 0, 418, 640), lambda g, y, x: (g.__setitem__((y, x + 5), INK), g.__setitem__((y, x + 20), INK)), need, (2, 32))
        assert n == need
        if (6144 - runs) % 2:
            g[2, 5 + 12] = INK
        if extra:
            g[2, 5 + 28] = INK                                   # a third run in the first item: entries unchanged
        out.append(_case(f"table caps: {6144 + extra} runs", g,
                         lambda r, e=extra: r["n_runs"] == 6144 + e and r["n_items"] <= T.RUNS_ENT_CAP and r["overflow"] == bool(e)))
    return out


def filter_cases():
    out = []
    g = _frame(640, 320)
    g[10:16, 10:18] = INK                                      # area 48
    g[10:16, 30:38] = INK; g[10, 30] = BG                      # area 47
    # qa around 64: rings 2 px thick, sides 9 (qa 64) and 8 (qa 49); a diamond-ish ring in between
    for k, s in enumerate((8, 9, 10)):
        g[40:40 + s, 20 + 20 * k:20 + 20 * k + s] = INK
        g[42:40 + s - 2, 22 + 20 * k:20 + 20 * k + s - 2] = BG
    # area / qa around 1.15: filled squares of side 14 (1.160) and 15 (1.148); around 0.25: 1 px rings of side 17 (0.25) and 18
    for k, s in enumerate((14, 15)):
        g[70:70 + s, 20 + 30 * k:20 + 30 * k + s] = INK
    for k, s in enumerate((17, 18)):
        x = 100 + 30 * k
        g[70:70 + s, x:x + s] = INK
        g[71:70 + s - 1, x + 1:x + s - 1] = BG
    # smin around 6: rings 2 px thick of height 7 (smin 6) and 6 (smin 5); around 0.08 smax: height 7, widths 76 and 77
    for k, (wd, ht) in enumerate(((30, 7), (30, 6), (76, 7), (77, 7), (88, 8), (89, 8))):
        y, x = 110 + 20 * (k // 2), 20 + 100 * (k % 2)
        g[y:y + ht, x:x + wd] = INK
        g[y + 2:y + ht - 2, x + 2:x + wd - 2] = BG
    # components touching each edge of the window, and ones a pixel away from it
    g[0:20, 300:320] = INK; g[1:21, 330:350] = INK
    g[300:320, 300:320] = INK; g[299:319, 330:350] = INK
    g[150:170, 0:20] = INK; g[180:200, 1:21] = INK
    g[150:170, 620:640] = INK; g[180:200, 619:639] = INK
    def hits(r):
        info = r["filters"]
        qa = {v["qa"] for v in info.values() if v}
        ratio = [v["area"] / v["qa"] for v in info.values() if v and v["qa"] >= 64]
        return (47 in r["area"] and 48 in r["area"] and 64.0 in qa and 49.0 in qa and any(abs(x - 1.15) < 0.02 for x in ratio)
                and any(abs(x - 0.25) < 0.02 for x in ratio) and r["n_quads"] >= 8)
    out.append(_case("filters: area 47/48, qa 64, area/qa 0.25 and 1.15, smin 6 and 0.08 smax, window edges", g, hits))
    return out


def _diamond(r, flat=0):
    yy, xx = np.mgrid[-r:r + 1, -r - flat:r + flat + 1]
    return (np.abs(yy) + np.maximum(np.abs(xx) - flat, 0)) <= r


def tie_cases():
    g = _frame(640, 256)
    x = 10
    for s in (12, 16, 21, 25):                                  # squares: four corners tie in pass 0
        g[20:20 + s, x:x + s] = INK; x += s + 10
    x = 10
    for r, flat in ((8, 0), (11, 0), (9, 2), (12, 3), (10, 1)):  # diamonds, diamonds with a flat top: ties in passes 0, 1 and 2
        d = _diamond(r, flat)
        g[80:80 + d.shape[0], x:x + d.shape[1]][d] = INK; x += d.shape[1] + 8
    x = 10
    for s in (14, 20):                                          # octagons (squares with cut corners)
        m = np.ones((s, s), bool)
        c = s // 4
        for i in range(c):
            m[i, :c - i] = m[i, s - c + i:] = m[s - 1 - i, :c - i] = m[s - 1 - i, s - c + i:] = False
        g[160:160 + s, x:x + s][m] = INK; x += s + 10
    for k, (ht, half) in enumerate(((30, 10), (40, 12))):        # tall isosceles triangles: the two base corners tie in pass 1
        yy, xx = np.mgrid[0:ht + 1, -half:half + 1]
        g[200:201 + ht, 300 + 40 * k:301 + 40 * k + 2 * half][np.abs(xx) * ht <= yy * half] = INK
    return [_case("ties: squares, diamonds, flat-topped diamonds, octagons, triangles", g,
                  lambda r: r["ties"]["pass0"] > 0 and r["ties"]["pass1"] > 0 and r["ties"]["pass2"] > 0 and r["n_quads"] >= 4)]


def window_cases():
    cam = synth.CAMERA_1080P
    g, pose = _rendered(760, cam)
    pts = synth.project(synth.object_points(), pose, cam)
    x0, y0 = int(pts[:, 0].min()) - 61, int(pts[:, 1].min()) - 40
    x1, y1 = int(pts[:, 0].max()) + 60, int(pts[:, 1].max()) + 40
    out = [_case("window: whole frame (one white level)", g, lambda r: r["window"] == (0, 0, 1920, 1080) and r["n_quads"] >= 3)]
    out.append(_case("window: rect with x0 % 16 != 0", g, lambda r, x0=x0: x0 % 16 != 0 and r["window"][0] == x0 & ~15 and r["n_quads"] >= 3,
                     rect=(x0, y0, x1, y1)))
    out.append(_case("window: rect clipped by the frame", g, lambda r: r["window"][0] == 0 and r["window"][3] < 1080 and r["n_comp"] >= 1,
                     rect=(-50, y0, (x0 + x1) // 2, 1200)))
    out.append(_case("window: empty rect = whole frame", g, lambda r: r["window"] == (0, 0, 1920, 1080), rect=(500, 300, 400, 900)))
    return out


def max_component_cases():
    out = []
    for path in ("shared", "global"):
        for total in (4096, 4097):
            g = _frame(1024, 512)
            draw_tag(g, 480, 420, 8, 5)                        # below everything else: numbered last in scan order
            if path == "global":
                g[300:330, 40:1000:2] = INK                      # one comb of ~14 000 runs: over the run table
                g[330, 40:1000] = INK
            base = T.quads_np(g, local=False)["n_all"]
            n = total - base
            # specks two to an item (one run each), in the rows above the tag
            k = _spread(g, (2, 0, 290, 1024), lambda g, y, x: (g.__setitem__((y, x + 5), INK), g.__setitem__((y, x + 20), INK)), n // 2, (2, 32))
            assert k == n // 2
            if n % 2:
                g[294, 500] = INK
            out.append(_case(f"MAX_COMPONENTS: {total} components in total, {path} union-find", g,
                             lambda r, t=total, p=path: r["n_all"] == t and r["overflow"] == (p == "global") and r["n_quads"] >= 1))
    # about 5 000 one-pixel specks above a rendered object, on either path
    cam = synth.CAMERA_1080P
    for path, per_item in (("shared", 2), ("global", 3)):
        g, pose = _rendered(701, cam)
        top, _ = _object_rows(pose, cam)
        lo = int(g.min())
        n = 0
        for y in range(2, top - 20, 2):
            for x in range(0, 1920, 32):
                for j in range(per_item):
                    if n < (4800 if per_item == 2 else 6200):
                        g[y, x + 3 + 10 * j] = lo; n += 1
        out.append(_case(f"MAX_COMPONENTS: {n} specks above a rendered object, {path} union-find", g,
                         lambda r, p=path: r["n_all"] > 4096 and r["overflow"] == (p == "global") and r["n_quads"] >= 3, local=True))
    return out


def rendered_cases():
    out = []
    for cam, name in ((synth.CAMERA_1080P, "1080p"), (synth.CAMERA_VGA, "VGA")):
        for seed in (700, 702):
            g, _ = _rendered(seed, cam)
            out.append(_case(f"rendered {name} seed {seed}", g, lambda r: r["n_quads"] >= 2, local=True))
    g, _ = _rendered(700, synth.CAMERA_1080P)
    out.append(_case("read form: rendered 1080p cropped to 1916 (word loads)", np.ascontiguousarray(g[:, :1916]), lambda r: r["n_quads"] >= 2,
                     pitch=1916, local=True))
    out.append(_case("read form: rendered 1080p cropped to 1915 (byte loads)", np.ascontiguousarray(g[:, :1915]), lambda r: r["n_quads"] >= 2,
                     pitch=1915, local=True))
    return out


def build():
    cases = (threshold_cases() + read_form_cases() + labelling_cases() + table_cap_cases() + filter_cases() + tie_cases() + window_cases()
             + max_component_cases() + rendered_cases())
    for c in cases:
        c["oracle"] = T.quads_np(c["gray"], c["rect"], c["local"])
    return cases
