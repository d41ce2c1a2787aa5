"""GPU tests of REPP on the device (csrc/repp.cu tscd_repp_prep / _tubelets / _emit after tscd_repp_link): the predictions must
equal the oracle's (the reference's REPP loops, tests/golden/repp.json pins it) -- same tubelets, track ids, order, boxes and
scores bit for bit -- and the packed path from the stage's detections must equal evalglue.repp_predictions followed by
REPPB200.__call__."""
import copy
import json
import os
import sys

import numpy as np
import pytest
import torch

from conftest import GOLDEN, ROOT

pytestmark = pytest.mark.gpu

G = json.load(open(os.path.join(GOLDEN, "repp.json")))
CFG = G["cases"][0]["cfg"]          # logreg, clf_mode dot, re-coordination on, no unmatched


def _oracle(cfg, video):
    from oracle import repp_oracle
    return repp_oracle.REPPOracle(logreg=G["logreg"], **cfg)(copy.deepcopy(video))


def _ours(cfg, video):
    from tscd_b200.repp import REPPB200
    return REPPB200(logreg=G["logreg"], **cfg)(copy.deepcopy(video))


def _track(T, nobj, seed, ih=480, iw=854, step=0.3, reps=3):
    """Dicts typed as Predictor.to_repp_heavy types them: float32 coordinates, the int 0 where a box is clipped at the left / top."""
    rng = np.random.default_rng(seed)
    pos = rng.uniform([-40, -40], [iw - 150, ih - 150], size=(nobj, 2))
    vel = rng.normal(0, 4, size=(nobj, 2))
    size = rng.uniform(25, 140, size=(nobj, 2))
    cls = rng.integers(0, 30, size=nobj)
    video = {}
    for t in range(T):
        dets = []
        for o in range(nobj):
            for rep in range(int(rng.integers(0, reps))):
                xy = pos[o] + vel[o] * t * step + rng.normal(0, 2.5, 2)
                wh = size[o] * (1 + rng.normal(0, 0.05, 2))
                x_min = 0 if xy[0] <= 0 else np.float32(xy[0])
                y_min = 0 if xy[1] <= 0 else np.float32(xy[1])
                w_, h_ = np.float32(wh[0]), np.float32(wh[1])
                c = [np.float32((x_min + w_ / 2) / max(iw, ih)), np.float32((y_min + (iw - ih) // 2 + h_ / 2) / max(iw, ih))]
                sc = np.array([rng.uniform(0.05, 0.95), rng.uniform(0.02, 0.9), cls[o] if rep == 0 else int(rng.integers(0, 30))],
                              dtype=np.float32)
                dets.append({"image_id": f"v/{t:06d}", "bbox": [x_min, y_min, w_, h_], "bbox_center": c, "scores": sc})
        video[str(t)] = dets
    return video


def _assert_same(got, want, least=1):
    assert len(got) == len(want) >= least
    for a, b in zip(got, want):
        assert a == b, (a, b)


# ---- dict input ------------------------------------------------------------------------------------------------------------
VARIANTS = [dict(), dict(add_unmatched=True), dict(recoordinate=False), dict(recoordinate=False, add_unmatched=True),
            dict(min_pred_score=0.0, add_unmatched=True), dict(min_pred_score=0.0),
            dict(clf_mode="max"), dict(clf_mode="dot_plus", clf_thr=0.5), dict(clf_mode="raw", add_unmatched=True),
            dict(distance_func="def"), dict(distance_func="def", add_unmatched=True, recoordinate_std=0.9)]


@pytest.mark.parametrize("var", VARIANTS, ids=[",".join(f"{k}={v}" for k, v in v.items()) or "default" for v in VARIANTS])
def test_configurations_vs_oracle(var):
    cfg = dict(CFG, **var)
    video = _track(40, 30, seed=11)
    _assert_same(_ours(cfg, video), _oracle(cfg, video), least=300)


def test_one_object_through_300_frames_and_mixed_dtypes():
    """One object in every frame of a 300-frame video (one 300-member tubelet), one object that moves across the left edge
    (members with the int 0: a float64 tubelet next to float32 ones), one box covering the whole image in every frame (all-int
    coordinates: an int64 tubelet), and unmatched clutter."""
    rng = np.random.default_rng(3)
    ih, iw, T = 480, 854, 300
    video = {}
    for t in range(T):
        dets = []
        x, y = 300 + 0.5 * t + rng.normal(0, 1), 200 + 0.2 * t + rng.normal(0, 1)
        dets.append({"image_id": t, "bbox": [np.float32(x), np.float32(y), np.float32(80 + rng.normal(0, 1)), np.float32(60)],
                     "bbox_center": [np.float32((x + 40) / iw), np.float32((y + 187 + 30) / iw)],
                     "scores": np.array([0.9, 0.8, 7], dtype=np.float32)})
        xl = 30 - 0.3 * t + rng.normal(0, 1)
        dets.append({"image_id": t, "bbox": [0 if xl <= 0 else np.float32(xl), np.float32(100), np.float32(50), np.float32(50)],
                     "bbox_center": [np.float32((max(0, xl) + 25) / iw), np.float32((100 + 187 + 25) / iw)],
                     "scores": np.array([0.7, 0.6, 3], dtype=np.float32)})
        if t % 50 < 40:
            dets.append({"image_id": t, "bbox": [0, 0, iw, ih], "bbox_center": [np.float32(0.5), np.float32(0.5)],
                         "scores": np.array([0.5, 0.5, 12], dtype=np.float32)})
        for _ in range(int(rng.integers(0, 3))):
            xy = rng.uniform(0, 700, 2)
            dets.append({"image_id": t, "bbox": [np.float32(xy[0]), np.float32(xy[1] / 2), np.float32(20), np.float32(20)],
                         "bbox_center": [np.float32(xy[0] / iw), np.float32(xy[1] / iw)],
                         "scores": np.array([0.3, 0.4, int(rng.integers(0, 30))], dtype=np.float32)})
        video[str(t)] = dets
    for var in (dict(), dict(add_unmatched=True, min_pred_score=0.0), dict(distance_func="def", add_unmatched=True)):
        cfg = dict(CFG, **var)
        want = _oracle(cfg, video)
        assert max(p["track_id"] for p in want) >= 2
        assert max(sum(p["track_id"] == t for p in want) for t in range(3)) >= T    # the long tubelet
        _assert_same(_ours(cfg, video), want, least=T)


def test_keys_out_of_numeric_order():
    """Linking follows the sorted frames, tubelet members and singletons index the dict in insertion order (REPP.py:141, :240):
    with equal detection counts the result is the oracle's; where an index falls outside its frame both raise IndexError."""
    rng = np.random.default_rng(7)
    base = _track(12, 6, seed=5, reps=2)
    order = [str(k) for k in rng.permutation(12)]
    cfg = dict(CFG, add_unmatched=True, min_tubelet_score=0.0)
    pad = {"image_id": "pad", "bbox": [np.float32(700), np.float32(400), np.float32(30), np.float32(30)],
           "bbox_center": [np.float32(0.84), np.float32(0.7)], "scores": np.array([0.5, 0.5, 2], dtype=np.float32)}
    same = {k: (base[k] + [copy.deepcopy(pad) for _ in range(8)])[:8] for k in order}
    _assert_same(_ours(cfg, same), _oracle(cfg, same), least=20)
    uneven = {k: base[k] for k in order}
    try:
        want = _oracle(cfg, uneven)
    except IndexError:
        with pytest.raises(IndexError):
            _ours(cfg, uneven)
    else:
        _assert_same(_ours(cfg, uneven), want)
    # a sorted dict given as is: the same answer as before
    _assert_same(_ours(cfg, base), _oracle(cfg, base))


def test_bench_video_vs_oracle():
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    from bench_repp import synth
    video = synth(300, 45)
    _assert_same(_ours(CFG, video), _oracle(CFG, video), least=10000)


def test_edge_videos():
    one = _track(1, 10, seed=2)
    assert _ours(CFG, one) == _oracle(CFG, one) == []
    # objects far apart and jumping: no frame pair links
    far = {str(t): [{"image_id": t, "bbox": [np.float32(10 + 400 * (t % 2)), np.float32(10), np.float32(20), np.float32(20)],
                     "bbox_center": [np.float32((20 + 400 * (t % 2)) / 854), np.float32(0.1)],
                     "scores": np.array([0.9, 0.9, 1], dtype=np.float32)}]
           for t in range(6)}
    cfg = dict(CFG, add_unmatched=True)
    want = _oracle(cfg, far)
    assert len(want) == 5 and len({p["track_id"] for p in want}) == 5
    _assert_same(_ours(cfg, far), want)


def test_more_than_4096_detections_in_a_frame_raises():
    big = {"0": [{"image_id": 0, "bbox": [np.float32(i % 800), np.float32(i // 800), np.float32(10), np.float32(10)],
                  "bbox_center": [np.float32(0.1), np.float32(0.1)], "scores": np.array([0.9, 0.9, 1], dtype=np.float32)}
                 for i in range(4097)],
           "1": [{"image_id": 1, "bbox": [np.float32(5), np.float32(5), np.float32(10), np.float32(10)],
                  "bbox_center": [np.float32(0.1), np.float32(0.1)], "scores": np.array([0.9, 0.9, 1], dtype=np.float32)}]}
    with pytest.raises(RuntimeError):
        _ours(CFG, big)


# ---- packed input (the stage's detections) ----------------------------------------------------------------------------------
def _stage_rows(F, cap, ih, iw, ratio, seed, counts=None):
    """Stage rows [F, cap, 7] (x1, y1, x2, y2 in network-input units, obj, cls_score, cls) of objects moving through the frames;
    some boxes clipped at the left, top, right, bottom, on both sides of one axis and on all four sides."""
    rng = np.random.default_rng(seed)
    nobj = 14
    pos = rng.uniform([30, 30], [iw - 200, ih - 200], size=(nobj, 2))
    vel = rng.normal(0, 3, size=(nobj, 2))
    size = rng.uniform(30, 140, size=(nobj, 2))
    cls = rng.integers(0, 30, size=nobj)
    rows = np.zeros((F, cap, 7), dtype=np.float32)
    n_f = []
    for f in range(F):
        boxes = []
        for o in range(nobj):
            if rng.uniform() < 0.15:
                continue
            x1, y1 = pos[o] + vel[o] * f + rng.normal(0, 2, 2)
            w, h = size[o] * (1 + rng.normal(0, 0.04, 2))
            x2, y2 = x1 + w, y1 + h
            if o == 0:
                x1 -= 200                                  # left
            elif o == 1:
                y1 -= 200                                  # top
            elif o == 2:
                x2 = iw + 10 + f                           # right
            elif o == 3:
                y2 = ih + 3                                # bottom
            elif o == 4:
                x1, x2 = -5.0, iw + 5.0                    # both sides of x
            elif o == 5:
                x1, y1, x2, y2 = -1.0, -1.0, iw + 1.0, ih + 1.0   # the whole image
            elif o == 6 and ratio == 1.0:
                x1, x2 = 0.0, float(iw)                    # exactly on the bounds
            c = cls[o] if rng.uniform() < 0.9 else rng.integers(0, 30)
            boxes.append([x1 * ratio, y1 * ratio, x2 * ratio, y2 * ratio, rng.uniform(0.05, 0.95), rng.uniform(0.01, 0.9), c])
        rng.shuffle(boxes)
        n = len(boxes) if counts is None else min(counts[f], len(boxes))
        rows[f, :n] = np.asarray(boxes[:n], dtype=np.float32).reshape(-1, 7)
        n_f.append(n)
    return rows, n_f


def _packed_case(rows, n_f, ratio, det_cand, img_sizes, cfg):
    from tscd_b200 import evalglue
    from tscd_b200.repp import REPPB200
    F = rows.shape[0]
    ids = [f"clip/{f:06d}" for f in range(F)]
    packed, offsets = evalglue.pack_detections(torch.from_numpy(rows).cuda().contiguous(),
                                               torch.tensor(n_f, dtype=torch.int32).cuda(), torch.full((F,), ratio))
    post = REPPB200(logreg=G["logreg"], **cfg)
    got = post.from_detections(packed, offsets, det_cand, img_sizes, ids).predictions()
    table, off = evalglue.to_host(packed, offsets)
    video = {str(f): p for f, p in enumerate(evalglue.repp_predictions(table, off, det_cand, img_sizes, ids))}
    want = post(copy.deepcopy(video))
    _assert_same(got, want, least=0)
    if F > 1:
        _assert_same(got, _oracle(cfg, video), least=0)
    return got


@pytest.mark.parametrize("ih,iw,ratio", [(480, 854, 1.0), (720, 540, 0.8), (576, 576, 1.25)])
def test_packed_path_matches_dicts(ih, iw, ratio):
    F, cap = 24, 16
    counts = [16] * F
    counts[5] = 0                                          # an empty frame
    rows, n_f = _stage_rows(F, cap, ih, iw, ratio, seed=ih + iw, counts=counts)
    det_cand = list(n_f)
    det_cand[9] = 0                                        # rows present, but the frame has no output
    sizes = [(ih, iw)] * F
    for var in (dict(), dict(add_unmatched=True), dict(add_unmatched=True, recoordinate=False), dict(min_pred_score=0.0),
                dict(distance_func="def", add_unmatched=True), dict(min_tubelet_score=0.2)):
        got = _packed_case(rows, n_f, ratio, det_cand, sizes, dict(CFG, **var))
        assert len(got) > 40


def test_packed_path_edge_videos():
    rows, n_f = _stage_rows(1, 16, 480, 854, 1.0, seed=1)
    assert _packed_case(rows, n_f, 1.0, n_f, [(480, 854)], CFG) == []
    rows, n_f = _stage_rows(5, 16, 480, 854, 1.0, seed=1)
    assert _packed_case(rows, n_f, 1.0, [0] * 5, [(480, 854)] * 5, dict(CFG, add_unmatched=True)) == []
    # no links: every frame's boxes far from the next frame's
    rows = np.zeros((6, 2, 7), dtype=np.float32)
    for f in range(6):
        x = 10 + 500 * (f % 2)
        rows[f, 0] = [x, 10 + 40 * f, x + 30, 40 + 40 * f, 0.9, 0.9, 4]
    got = _packed_case(rows, [1] * 6, 1.0, [1] * 6, [(480, 854)] * 6, dict(CFG, add_unmatched=True))
    assert len(got) == 5 and [p["track_id"] for p in got] == list(range(5))
