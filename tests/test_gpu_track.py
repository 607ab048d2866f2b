"""GPU parity: camshift.Tracker + getWhitebalance through the C ABI vs the CPU oracle."""
import math

import numpy as np
import pytest

import oracle
from headtrackr_b200 import synth

pytestmark = pytest.mark.gpu


def face_rect(blob, f):
    res = oracle.detect(f, blob)
    best = max(res, key=lambda r: r[4])          # no confidence ties in these frames
    return [int(math.floor(v)) for v in best[:4]]


@pytest.mark.parametrize("W,H,idx,calc", [(320, 240, 0, True), (320, 240, 1, False), (640, 480, 3, False),
                                          (640, 480, 2, True)])
def test_track_matches_oracle(ctx, blob, W, H, idx, calc):
    f = synth.frame(idx, W, H)
    rect = face_rect(blob, f)
    ot = oracle.CamshiftTracker(calc_angles=calc)
    ot.init_tracker(f, *rect)
    ctx.track_init(f, [rect], calc_angles=calc)
    assert np.array_equal(ctx.debug_model_hist(0), np.frombuffer(bytes(ot.t.model_hist), np.uint32))
    for call in range(5):
        ot.track(f)
        objs, wins = ctx.track(f)
        want = ot.track_obj()
        got = objs[0]
        assert (got["x"], got["y"], got["width"], got["height"]) == (want["x"], want["y"], want["width"], want["height"]), call
        assert abs(got["angle"] - want["angle"]) <= 1e-4          # north_star tolerance for the angle
        assert wins[0] == ot.search_window()
    assert want["width"] > 0 and want["height"] > 0


def test_n_calls_equals_repeated_calls(ctx, blob):
    f = synth.frame(3, 640, 480)
    rect = face_rect(blob, f)
    ot = oracle.CamshiftTracker(calc_angles=False)
    ot.init_tracker(f, *rect)
    for _ in range(30):
        ot.track(f)
    ctx.track_init(f, [rect], calc_angles=False)
    objs, wins = ctx.track(f, n_calls=30)
    want = ot.track_obj()
    assert (objs[0]["x"], objs[0]["y"], objs[0]["width"], objs[0]["height"]) == (want["x"], want["y"], want["width"], want["height"])
    assert wins[0] == ot.search_window()


def test_lost_face_degenerates_like_reference(ctx, blob):
    """Model colours absent from the frame -> all weights 0 -> NaN moments -> width == height == 0 (src/main.js:230)."""
    f = synth.frame(0, 320, 240)
    rect = face_rect(blob, f)
    g = synth.frame(0, 320, 240, kind="constant")
    ot = oracle.CamshiftTracker(calc_angles=False)
    ot.init_tracker(f, *rect)
    ot.track(g)
    ctx.track_init(f, [rect], calc_angles=False)
    objs, wins = ctx.track(g)
    want = ot.track_obj()
    assert (objs[0]["x"], objs[0]["y"], objs[0]["width"], objs[0]["height"]) == (want["x"], want["y"], want["width"], want["height"])
    assert wins[0] == ot.search_window()


def test_rect_outside_canvas(ctx, blob):
    f = synth.frame(1, 320, 240)
    rect = [300, 220, 60, 50]
    ot = oracle.CamshiftTracker(calc_angles=True)
    ot.init_tracker(f, *rect)
    ctx.track_init(f, [rect], calc_angles=True)
    assert np.array_equal(ctx.debug_model_hist(0), np.frombuffer(bytes(ot.t.model_hist), np.uint32))
    ot.track(f)
    objs, wins = ctx.track(f)
    want = ot.track_obj()
    assert (objs[0]["x"], objs[0]["y"], objs[0]["width"], objs[0]["height"]) == (want["x"], want["y"], want["width"], want["height"])


def test_batched_streams_and_slots(ctx, blob):
    frames = synth.batch(4, 320, 240, start=0)
    rects = [face_rect(blob, frames[i]) for i in range(4)]
    slots = [7, 2, 5, 0]
    ctx.track_init(frames, rects, slots=slots, calc_angles=False)
    objs, wins = ctx.track(frames, slots=slots, n_calls=3)
    for i in range(4):
        ot = oracle.CamshiftTracker(calc_angles=False)
        ot.init_tracker(frames[i], *rects[i])
        for _ in range(3):
            ot.track(frames[i])
        want = ot.track_obj()
        assert (objs[i]["x"], objs[i]["y"], objs[i]["width"], objs[i]["height"]) == (want["x"], want["y"], want["width"], want["height"])
        assert wins[i] == ot.search_window()


def test_track_init_from_detect(ctx, blob):
    frames = synth.batch(3, 640, 480, start=0)
    rects, counts = ctx.detect_raw(frames, 5, 1)
    found = ctx.track_init_from_detect(frames, rects, counts, calc_angles=False)
    objs, wins = ctx.track(frames, n_calls=2)
    for i in range(3):
        res = oracle.detect(frames[i], blob)
        cand = None
        for r in res:                                  # src/facetrackr.js:157-165
            if cand is None or r[4] > cand[4]:
                cand = r
        assert found[i] == int(cand is not None and cand[4] > -10)
        ot = oracle.CamshiftTracker(calc_angles=False)
        ot.init_tracker(frames[i], *[int(math.floor(v)) for v in cand[:4]])
        ot.track(frames[i]); ot.track(frames[i])
        want = ot.track_obj()
        assert (objs[i]["x"], objs[i]["y"], objs[i]["width"], objs[i]["height"]) == (want["x"], want["y"], want["width"], want["height"])


def test_uninitialised_slot_is_an_error(ctx):
    from headtrackr_b200._lib import HtError, HT_ERR_STATE
    f = synth.frame(0, 320, 240)
    with pytest.raises(HtError) as e:
        ctx.track(f, slots=[15])
    assert e.value.code == HT_ERR_STATE


def test_backprojection_and_whitebalance(ctx, blob):
    f = synth.frame(2, 320, 240)
    rect = face_rect(blob, f)
    ot = oracle.CamshiftTracker(calc_angles=False)
    ot.init_tracker(f, *rect)
    ctx.track_init(f, [rect], calc_angles=False)
    assert np.array_equal(ctx.backprojection(f, 0), ot.backprojection_img(f))
    frames = synth.batch(3, 320, 240, start=5)
    wb = ctx.whitebalance(frames)
    for i in range(3):
        assert wb[i] == oracle.whitebalance(frames[i])


def test_detect_track_host_and_device(ctx, blob):
    """ht_detect_track (chunk-pipelined host path and device path) == detect -> pick -> init -> n x track."""
    import torch
    frames = synth.batch(5, 640, 480, start=60)
    frames[4] = synth.frame(0, 640, 480, kind="constant")        # a frame without any face
    ref_objs = []
    for i in range(5):
        res = oracle.detect(frames[i], blob)
        cand = None
        for r in res:
            if cand is None or r[4] > cand[4]:
                cand = r
        if cand is None or not cand[4] > -10:
            ref_objs.append(None)
            continue
        ot = oracle.CamshiftTracker(calc_angles=False)
        ot.init_tracker(frames[i], *[int(math.floor(v)) for v in cand[:4]])
        for _ in range(4):
            ot.track(frames[i])
        ref_objs.append((ot.track_obj(), ot.search_window(), res))
    for src in (frames, torch.from_numpy(frames).cuda()):
        dets, found, objs, wins = ctx.detect_track(src, 5, 1, calc_angles=False, n_calls=4)
        for i in range(5):
            if ref_objs[i] is None:
                assert found[i] == 0 and dets[i] == [] and objs[i]["width"] == 0
                continue
            want, win, res = ref_objs[i]
            assert found[i] == 1
            assert [(d["x"], d["y"], d["width"], d["height"], d["confidence"], d["neighbors"]) for d in dets[i]] == res
            assert (objs[i]["x"], objs[i]["y"], objs[i]["width"], objs[i]["height"]) == (want["x"], want["y"], want["width"], want["height"])
            assert wins[i] == win


def test_track_odd_width_scalar_path(ctx, blob):
    """W % 4 != 0 takes the scalar bin-plane path of k_track."""
    f = synth.frame(2, 333, 251)
    rect = face_rect(blob, f)
    ot = oracle.CamshiftTracker(calc_angles=True)
    ot.init_tracker(f, *rect)
    ctx.track_init(f, [rect], calc_angles=True)
    for _ in range(3):
        ot.track(f)
        objs, wins = ctx.track(f)
    want = ot.track_obj()
    assert (objs[0]["x"], objs[0]["y"], objs[0]["width"], objs[0]["height"]) == (want["x"], want["y"], want["width"], want["height"])
    assert abs(objs[0]["angle"] - want["angle"]) <= 1e-4 and wins[0] == ot.search_window()


@pytest.mark.parametrize("env", [{}, {"HT_TRACK_HEAVY": "8"}, {"HT_TRACK_HEAVY": "4,4"},
                                 {"HT_TRACK_LPT": "0"}, {"HT_TRACK_MEMO": "0"}])
def test_scheduled_launch_orders_do_not_change_results(blob, env, monkeypatch):
    """>= 128 streams: k_track runs the streams longest-window-first (optionally the largest ones on a bigger cluster
    on a second stream).  The schedule must not change any stream's result."""
    from headtrackr_b200 import Context
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    W, H, U, N = 320, 240, 16, 144
    uniq = synth.batch(U, W, H, start=900)
    want = [oracle.detect_track(uniq[i], blob, n_calls=6) for i in range(U)]
    frames = np.stack([uniq[i % U] for i in range(N)])
    c = Context(max_width=W, max_height=H, max_frames=N)
    try:
        for _ in range(2):
            dets, found, objs, wins = c.detect_track(frames, 5, 1, calc_angles=False, n_calls=6)
            for i in range(N):
                n_det, fnd, obj = want[i % U]
                assert len(dets[i]) == n_det and found[i] == fnd
                if fnd:
                    assert (objs[i]["x"], objs[i]["y"], objs[i]["width"], objs[i]["height"]) == \
                        (obj["x"], obj["y"], obj["width"], obj["height"])
    finally:
        c.close()


def test_window_memo_does_not_change_results(ctx, blob):
    """30 track() calls on one frame: with the window memo the kernel sums far fewer passes, and every output is
    identical to the strict run and to the oracle."""
    frames = synth.batch(6, 640, 480, start=56)
    want = [oracle.detect_track(frames[i], blob, n_calls=30) for i in range(6)]
    runs = {}
    try:
        for memo in (False, True):
            ctx.set_track_memo(memo)
            ctx.debug_track_stats(reset=True)
            dets, found, objs, wins = ctx.detect_track(frames, 5, 1, calc_angles=False, n_calls=30)
            runs[memo] = (found, objs, wins, ctx.debug_track_stats(reset=True))
    finally:
        ctx.set_track_memo(True)
    assert runs[False][:3] == runs[True][:3]
    strict, memo = runs[False][3], runs[True][3]
    assert strict["memo_hits"] == 0 and memo["memo_hits"] > 0
    assert memo["passes"] + memo["memo_hits"] == strict["passes"] and memo["calls"] == strict["calls"]
    for i in range(6):
        n_det, fnd, obj = want[i]
        assert runs[True][0][i] == fnd
        if fnd:
            o = runs[True][1][i]
            assert (o["x"], o["y"], o["width"], o["height"]) == (obj["x"], obj["y"], obj["width"], obj["height"])


@pytest.mark.parametrize("W,H", [(320, 240), (333, 251)])
def test_zero_weight_marking_changes_nothing(blob, W, H, monkeypatch):
    """k_bins_mask rewrites the plane entries of colours absent from the model histogram to the table's +0.0 entry and
    k_track skips all-zero row segments (src/camshift.js:314-330: such pixels have weight exactly 0): every output equals
    the unmarked run's and the oracle's - also for odd frame sizes (unaligned planes take the scalar path)."""
    import os
    from headtrackr_b200.context import Context
    frames = synth.batch(3, W, H, start=2)
    rects = [face_rect(blob, frames[i]) for i in range(3)]
    results = {}
    for tag, env in (("marked", "1,0"), ("unmarked", "0")):
        monkeypatch.setenv("HT_TRACK_MASK", env)
        c = Context(max_width=W, max_height=H, max_frames=3, max_raw_per_frame=4096)
        try:
            c.set_track_memo(False)
            c.track_init(frames, rects, calc_angles=True)
            results[tag] = c.track(frames, n_calls=12)
        finally:
            c.close()
    assert results["marked"] == results["unmarked"]
    objs, wins = results["marked"]
    for i in range(3):
        ot = oracle.CamshiftTracker(calc_angles=True)
        ot.init_tracker(frames[i], *rects[i])
        for _ in range(12):
            ot.track(frames[i])
        w = ot.track_obj()
        assert (objs[i]["x"], objs[i]["y"], objs[i]["width"], objs[i]["height"]) == (w["x"], w["y"], w["width"], w["height"])
        assert abs(objs[i]["angle"] - w["angle"]) <= 1e-4
        assert wins[i] == ot.search_window()
