"""The detector's first stage (csrc/agt_tags.cu, agt_tag_quads: threshold -> components -> farthest points -> quads) against
oracle/tag_oracle.quads_np, pixel for pixel, on the case set of tests/tag_quad_cases.py, in every path the stage can take.

Each case runs at two positions of a batch of 3 (separate launches of comp_far_kernel and quad_emit_kernel) and of a batch of
9 (quad_fit_cluster_kernel); a few also at batches of 7 and 8, either side of the switch.  The other frames of a batch are
flat (no contrast: no dark pixel).  Per case and form: the number of components numbered, the union-find path, the number of
quads, the quads as a set (slot order is atomic) - corners within 1e-4 px of the oracle's, which places them from the
oracle's farthest pixels (the device's tie rule: the larger pixel index wins), and the same refinement window - and the same
bytes at every position and in every form.  End to end: agt_detect_tags without refinement equals decode_np on the stage's
quads, and with refinement equals agt_corner_subpix (grouped by window) followed by agt_decode_tags, bit for bit."""
from __future__ import annotations

import re
import time

import numpy as np
import pytest

from oracle import tag_oracle as T
from tests import tag_quad_cases as C

pytestmark = pytest.mark.gpu

MAX_QUADS = 4096                 # the detector's slots for max_tags = 1024
FORMS = ((3, (0, 2)), (9, (1, 7)))
STRADDLE = ((7, (6,)), (8, (0, 5)))
LARGE = ((64, (0, 63)),)           # window cases: fewer CTAs per frame, INIT_ROWS up to 16
FILL = 128
REFINE_WIN = 4
SUBPIX_ITERS, SUBPIX_EPS = 10, 1e-3      # the detector's corner refinement
REPORT = []


@pytest.fixture(scope="module")
def cases():
    return C.build()


def _frames(ctx, case, batch, positions):
    """A device buffer [batch, h, pitch] (at an odd address if the case says so) with the case at `positions`, flat elsewhere."""
    torch = ctx.torch
    g = case["gray"]
    h, w = g.shape
    pitch, off = case["pitch"], case["offset"]
    buf = torch.full((off + batch * h * pitch,), FILL, dtype=torch.uint8, device=ctx.tdev)
    frames = buf[off:].view(batch, h, pitch)
    host = np.full((h, pitch), FILL, np.uint8)
    host[:, :w] = g
    for p in positions:
        frames[p].copy_(torch.from_numpy(host))
    return frames


def _rects(case, batch, positions):
    if case["rect"] is None:
        return None
    r = np.zeros((batch, 4), np.int32)
    r[list(positions)] = case["rect"]
    return r


def _run(ctx, case, batch, positions, profile=False):
    ctx.set_tag_threshold("local" if case["local"] else "window")
    frames = _frames(ctx, case, batch, positions)
    rects = _rects(case, batch, positions)
    names = set()
    if profile:
        from torch.profiler import ProfilerActivity, profile as tprofile
        with tprofile(activities=[ProfilerActivity.CUDA]) as prof:
            # a moment between opening the trace and the first launch: late in a long GPU session the window's first kernel
            # (tile_max_kernel) was missing from the trace while its results were there
            time.sleep(0.01)
            out = ctx.tag_quads(frames, width=case["gray"].shape[1], rects=rects, max_quads=MAX_QUADS, refine_win=REFINE_WIN)
            ctx.sync()
        names = {e.name for e in prof.events() if "_kernel" in e.name}
    else:
        out = ctx.tag_quads(frames, width=case["gray"].shape[1], rects=rects, max_quads=MAX_QUADS, refine_win=REFINE_WIN)
    ctx.set_tag_threshold("auto")
    return {k: v.cpu().numpy() for k, v in out.items()}, names


def _sorted_quads(out, p):
    n = min(int(out["n_quads"][p]), MAX_QUADS)
    q, wn = out["quads"][p, :n], out["win"][p, :n]
    order = sorted(range(n), key=lambda k: q[k].tobytes() + bytes([wn[k]]))
    return q[order], wn[order]


def _match(case, out, p):
    """-> list of problems of frame p against the oracle (empty: identical)."""
    r = case["oracle"]
    bad = []
    if int(out["n_comp"][p]) != r["n_comp"]:
        bad.append(f"n_comp {out['n_comp'][p]} != {r['n_comp']}")
    if bool(out["overflow"][p]) != r["overflow"]:
        bad.append(f"overflow {out['overflow'][p]} != {r['overflow']}")
    if int(out["n_quads"][p]) != r["n_quads"]:
        bad.append(f"n_quads {out['n_quads'][p]} != {r['n_quads']}")
    q, wn = _sorted_quads(out, p)
    left = list(range(len(r["quads"])))
    for k in range(len(q)):
        hit = None
        for j in left:
            for alt in r["quads"][j]["alts"]:
                if np.abs(q[k] - alt["corners"]).max() <= 1e-4 and wn[k] == alt["cwin"]:
                    hit = j
            if hit is not None:
                break
        if hit is None:
            bad.append(f"quad {q[k].ravel().tolist()} win {wn[k]} is not the oracle's")
        else:
            left.remove(hit)
    if left and len(q) == r["n_quads"]:
        bad.append(f"{len(left)} oracle quads not emitted")
    return bad


@pytest.fixture(scope="module")
def runs(ctx1080, cases):
    res = {}
    for ci, case in enumerate(cases):
        for batch, positions in FORMS:
            res[(ci, batch)] = _run(ctx1080, case, batch, positions, profile=(ci == 0))
        if case["pyramid"] and case["name"].startswith(("rendered", "MAX_COMPONENTS")):
            for batch, positions in STRADDLE:
                res[(ci, batch)] = _run(ctx1080, case, batch, positions, profile=True)
        if case["name"].startswith("window"):
            for batch, positions in LARGE:
                res[(ci, batch)] = _run(ctx1080, case, batch, positions)
    return res


def test_stage_matches_oracle(cases, runs):
    failures = []
    for (ci, batch), (out, _) in runs.items():
        case = cases[ci]
        positions = dict(FORMS + STRADDLE + LARGE)[batch]
        for p in positions:
            bad = _match(case, out, p)
            if bad:
                failures.append(f"{case['name']} [batch {batch}, position {p}]: " + "; ".join(bad[:4]))
        for p in set(range(batch)) - set(positions):
            assert out["n_comp"][p] == 0 and out["n_quads"][p] == 0 and out["overflow"][p] == 0
    for ci, case in enumerate(cases):
        r = case["oracle"]
        REPORT.append(f"{case['name']}: components {r['n_all']} ({r['n_comp']} of area >= 48), items {r['n_items']}, runs {r['n_runs']}, "
                      f"{'global' if r['overflow'] else 'shared'}-memory union-find, quads {r['n_quads']}, ties pass0/1/2 "
                      f"{r['ties']['pass0']}/{r['ties']['pass1']}/{r['ties']['pass2']}, pass-0 evaluation orders disagree "
                      f"{r['ties']['pass0_orders']}; device {'matches' if not any(f.startswith(case['name'] + ' [') for f in failures) else 'DIFFERS'}")
    assert not failures, "\n".join(failures)


def test_forms_and_positions_bit_identical(cases, runs):
    for ci, case in enumerate(cases):
        ref = None
        for (cj, batch), (out, _) in runs.items():
            if cj != ci:
                continue
            for p in dict(FORMS + STRADDLE + LARGE)[batch]:
                q, wn = _sorted_quads(out, p)
                key = (q.tobytes(), wn.tobytes(), int(out["n_comp"][p]), int(out["n_quads"][p]), int(out["overflow"][p]))
                ref = key if ref is None else ref
                assert key == ref, (case["name"], batch, p)


def test_every_path_ran(cases, runs):
    names = set()
    for _, (_, n) in runs.items():
        names |= n
    kern = lambda k: any(k in s for s in names)
    by_batch = {b: set() for b in (3, 7, 8, 9, 64)}
    for (ci, batch), (_, n) in runs.items():
        by_batch[batch] |= n
    short = lambda n: sorted({m for s in n for m in re.findall(r"\w+_kernel", s)})
    REPORT.append("kernels in the profiler traces: " + ", ".join(short(names)))
    for b, n in by_batch.items():
        REPORT.append(f"  batch {b}: " + ", ".join(k for k in short(n) if "far" in k or "quad_" in k))
    assert kern("comp_far_kernel") and kern("quad_emit_kernel") and kern("quad_fit_cluster_kernel") and kern("tile_max_kernel")
    assert any("quad_fit_cluster_kernel" in s for s in by_batch[8]) and not any("quad_fit_cluster_kernel" in s for s in by_batch[7])
    assert any("comp_far_kernel" in s for s in by_batch[7]) and not any("comp_far_kernel" in s for s in by_batch[8])
    over = {bool(cases[ci]["oracle"]["overflow"]) for (ci, _), (out, _) in runs.items()}
    assert over == {True, False}
    layouts = {("16" if c["pitch"] % 16 == 0 and c["offset"] == 0 else "4" if c["pitch"] % 4 == 0 and c["offset"] == 0 else "1") for c in cases}
    assert layouts == {"16", "4", "1"}
    rows = {C.init_rows(c["oracle"]["window"][2], c["oracle"]["window"][3], c["gray"].shape[::-1], batch, c["rect"] is not None)
            for (ci, batch) in runs for c in [cases[ci]] if c["pitch"] % 16 == 0 and c["offset"] == 0}
    REPORT.append(f"INIT_ROWS of the sixteen-pixel threshold pass over the runs: {sorted(rows)}")
    assert 1 in rows and 16 in rows


def _tags(det, p):
    n = int(det["n"][p])
    return sorted((int(det["id"][p, j]), det["corners"][p, j].tobytes()) for j in range(n))


def test_detect_tags_end_to_end(ctx1080, cases, runs):
    """refine_win 0: the tags are decode_np of the stage's quads; refine_win 4: agt_corner_subpix on the stage's quads, grouped by
    their window, then agt_decode_tags - bit for bit.  Speckled frames: every tag quads_np + decode_np find is found."""
    ctx = ctx1080
    torch = ctx.torch
    n_tags = 0
    for ci, case in enumerate(cases):
        if not case["pyramid"]:
            continue
        g = case["gray"]
        h, w = g.shape
        out = runs[(ci, 3)][0]
        pyr = ctx.alloc_pyramid(3, w, h, 1)
        ctx.upload_frames(pyr, np.stack([g, np.full_like(g, FILL), g]))
        ctx.set_tag_threshold("local" if case["local"] else "window")
        try:
            rects = _rects(case, 3, (0, 2))
            d0 = {k: v.cpu().numpy() for k, v in ctx.detect_tags(pyr, max_tags=1024, refine_win=0, rects=rects).items()}
            d4 = {k: v.cpu().numpy() for k, v in ctx.detect_tags(pyr, max_tags=1024, refine_win=REFINE_WIN, rects=rects).items()}
        finally:
            ctx.set_tag_threshold("auto")
        nq = min(int(out["n_quads"][0]), MAX_QUADS)
        quads, wins = out["quads"][0, :nq], out["win"][0, :nq]
        want = []
        for q in quads:
            tid, rot, _, _ = T.decode_np(g, q.astype(np.float64))
            if tid >= 0:
                want.append((tid, np.roll(q, rot, axis=0).astype(np.float32).tobytes()))
        assert _tags(d0, 0) == sorted(want) == _tags(d0, 2), case["name"]
        n_tags += len(want)
        if case["name"].startswith("MAX_COMPONENTS"):
            oracle_ids = {T.decode_np(g, qd["alts"][0]["corners"].astype(np.float64))[0] for qd in case["oracle"]["quads"]} - {-1}
            assert oracle_ids and oracle_ids <= {i for i, _ in _tags(d4, 0)}, case["name"]
        # refinement: the stage's quads through agt_corner_subpix window by window, then agt_decode_tags
        if nq == 0:
            assert int(d4["n"][0]) == 0
            continue
        pts = torch.tensor(np.ascontiguousarray(quads.reshape(1, -1, 2)), device=ctx.tdev)
        refined = quads.reshape(-1, 2).copy()
        for cw in np.unique(wins):
            valid = np.repeat(wins == cw, 4).astype(np.uint8)[None]
            r = ctx.corner_subpix(pyr, pts, valid=valid, win=int(cw), max_iters=SUBPIX_ITERS, eps=SUBPIX_EPS).cpu().numpy()[0]
            refined[valid[0] == 1] = r[valid[0] == 1]
        refined = refined.reshape(1, nq, 4, 2)
        dec = {k: v.cpu().numpy() for k, v in ctx.decode_tags(pyr, np.concatenate([refined, refined, refined])).items()}
        want4 = sorted((int(dec["id"][0, k]), np.roll(refined[0, k], int(dec["rotation"][0, k]), axis=0).tobytes())
                       for k in range(nq) if dec["id"][0, k] >= 0)
        assert _tags(d4, 0) == want4, case["name"]
    REPORT.append(f"end to end: {n_tags} tags decoded from the stage's quads on the frames that fit a pyramid")
    assert n_tags >= 20


def test_zz_report():
    print("\n" + "\n".join(REPORT))
