"""VideoStream (tscd_b200/video.py) and tscd_video_pack on the GPU.  The bar is byte equality: every video's table equals
evalglue.pack_detections over the frame-ordered detections of the device path (ingest_frames + one clip per forward_clips call,
CAFM memory carried with resume), and tscd_video_pack equals tscd_pack_detections.

Videos are seeded synthetic head outputs (as in test_gpu_frame_store.py) written into the stream's pinned staging buffers; clips
come from clips.demo_clips with a seeded rng."""
import random

import pytest
import torch

import oracle

pytestmark = pytest.mark.gpu

HW = [(24, 24), (12, 12), (6, 6)]
A = sum(h * w for h, w in HW)
D = 256


def _sel_cfg(kind):
    from tscd_b200 import selection
    if kind == "A":
        return selection.SelectionConfig(mode="A", pre_k=750, top_k=30, nms_thresh=0.75)
    if kind == "ovis_l":
        return selection.SelectionConfig(mode="B", minimal_limit=50, maximal_limit=500, use_pre_nms=False)
    if kind == "vid_l":
        return selection.SelectionConfig(mode="B", minimal_limit=50, maximal_limit=0, use_pre_nms=False)
    if kind == "wide":
        return selection.SelectionConfig(mode="B", minimal_limit=50, maximal_limit=0, use_pre_nms=False, max_proposals=2048)
    if kind == "small":                   # a 64-proposal tier that a dense frame overflows
        return selection.SelectionConfig(mode="B", minimal_limit=20, maximal_limit=0, use_pre_nms=False, max_proposals=64)
    raise ValueError(kind)


def _stage(C, kind):
    from tscd_b200 import stage, weights
    return stage.AggregationStage(stage.StageConfig(num_classes=C, selection=_sel_cfg(kind)), weights.random_state_dict(C, D, seed=11))


def _video(n, C, seed, obj_mean, n_obj=40):
    from tscd_b200 import ops
    head, feats = oracle.synth_head_outputs(n, HW, C, dim=D, seed=seed, clustered=True, obj_mean=obj_mean, n_obj=n_obj)
    logit = torch.logit(head[:, :, 4:].clamp(1e-6, 1 - 1e-6))
    rows = torch.zeros(n, A, ops.row_pitch(C), dtype=torch.float16)
    rows[:, :, :4] = head[:, :, :4].half()
    rows[:, :, 4:5 + C] = logit.half()
    objp = torch.zeros(n, (A + 7) // 8 * 8, dtype=torch.float16)
    objp[:, :A] = rows[:, :, 4]
    return dict(rows=rows, objp=objp, feats=[f.half().contiguous() for f in feats])


def _write(buf, v, f0):
    """A video's frames into a buffer set at frame f0 (what a producer does)."""
    n = v["rows"].shape[0]
    buf["rows"][0][f0:f0 + n].copy_(v["rows"])
    buf["objp"][0][f0:f0 + n, :v["objp"].shape[1]].copy_(v["objp"])
    for k, f in zip(("f_cls", "f_reg", "f_edge"), v["feats"]):
        s = 0
        for (h, w), t in zip(HW, buf[k]):
            t[f0:f0 + n].permute(0, 2, 3, 1).copy_(f[:, s:s + h * w].reshape(n, h, w, D))
            s += h * w


def _views(v, C):
    from tscd_b200 import ops
    an = ops.AnchorSpec(HW)
    d = {k: (x.cuda() if isinstance(x, torch.Tensor) else [t.cuda() for t in x]) for k, x in v.items()}
    return d, ops.HeadViews.from_rows(d["rows"], d["objp"], an, C), tuple(ops.view_rowmajor(f, an) for f in d["feats"])


def _te(paths):
    from tscd_b200 import clips
    return torch.cat([clips.time_embedding(p) for p in paths], 0).cuda()


def _item(n, L, G, first, seed, ratio=1.0):
    from tscd_b200 import clips
    cl, pa = clips.demo_clips(n, L, G, rng=random.Random(seed))
    ratios = [ratio * (1 + 0.05 * (f % 3)) for f in range(n)]
    return dict(first_frame=first, num_frames=n, clips=cl, paths=pa, ratios=ratios)


def _reference(st, C, v, item):
    """Device path: ingest_frames, one clip per forward_clips call with resume, frame-ordered rows -> pack_detections."""
    from tscd_b200 import evalglue, frames, stage
    from tscd_b200.video import local_frames
    n = item["num_frames"]
    kmax = st.cfg.selection.max_keep(A)
    store = frames.FrameStore(n, kmax, C)
    keep, head, feats = _views(v, C)
    st.ingest_frames(store, head, feats, torch.float16, list(range(n)))
    pool = stage.CAFMState(1, kmax)
    L = len(item["paths"][0])
    outs = [st.forward_clips(store, [c], L, _te([p]), state=pool, resume=[int(i > 0)], state_slots=[0])
            for i, (c, p) in enumerate(zip(item["clips"], item["paths"]))]
    where = local_frames(item["clips"], item["paths"], n)
    rows = torch.stack([outs[c]["det_rows"][l] for c, l in where]).contiguous()
    cnt = torch.stack([outs[c]["det_count"][l] for c, l in where]).contiguous()
    cand = [int(outs[c]["det_cand"][l]) for c, l in where]
    for o in outs:
        assert int(o["status"].item()) == 0
    packed, off = evalglue.pack_detections(rows, cnt, torch.tensor(item["ratios"]))
    orows = torch.stack([outs[c]["ori_rows"][l] for c, l in where]).contiguous()
    ocnt = torch.stack([outs[c]["ori_count"][l] for c, l in where]).contiguous()
    opacked, ooff = evalglue.pack_detections(orows, ocnt, torch.tensor(item["ratios"]))
    torch.cuda.synchronize()
    off, ooff = off.cpu(), ooff.cpu()
    _ORI[id(item)] = (opacked[:int(ooff[-1])].cpu(), ooff)
    return packed[:int(off[-1])].cpu(), off, cand


_ORI = {}          # still-detector tables of the last _reference calls, by item


def _assert_ori(got, item):
    packed, off = _ORI[id(item)]
    assert torch.equal(got["ori_offsets"], off.to(torch.int32)) and int(off[-1]) > 0
    assert torch.equal(got["ori_packed"].view(torch.int32), packed.view(torch.int32))


def _assert_table(got, want):
    packed, off, cand = want
    assert torch.equal(got["offsets"], off.to(torch.int32))
    assert got["packed"].shape == packed.shape and torch.equal(got["packed"].view(torch.int32), packed.view(torch.int32))
    assert got["det_cand"].tolist() == cand


@pytest.fixture(autouse=True)
def _collect():
    yield
    import gc
    gc.collect()
    torch.cuda.synchronize()


def test_video_pack_matches_pack_detections():
    """Random padded rows of three calls (frames with 0 rows and at cap, rows no frame maps to), two videos, scales != 1."""
    from tscd_b200 import evalglue, ops
    g = torch.Generator().manual_seed(3)
    cap = 6
    calls = []
    for n in (6, 4, 8):
        rows = (torch.rand(n, cap, 7, generator=g) * 100).cuda()
        cnt = torch.randint(0, cap + 1, (n,), generator=g, dtype=torch.int32)
        cnt[0], cnt[-1] = 0, cap
        cand = (cnt > 0).to(torch.int32) * torch.randint(0, 2, (n,), generator=g, dtype=torch.int32) + cnt
        calls.append((rows, cnt.cuda(), cand.cuda()))
    videos = [[(0, 0), (0, 3), (1, 2), (2, 7), (2, 0)], [(1, 1), (2, 5), (0, 5), (1, 3)]]      # (call, row); others unmapped
    scales = [float(x) for x in torch.rand(9, generator=g) * 2 + 0.5]
    fmap = torch.tensor([(c, r, f) for vid in videos for f, (c, r) in enumerate(vid)], dtype=torch.int32).cuda()
    status = torch.zeros(1, dtype=torch.int32, device="cuda")
    out = ops.video_pack(calls, fmap, torch.tensor(scales).cuda(), status)
    torch.cuda.synchronize()
    assert int(status.item()) == 0
    off = out["offsets"].cpu()
    f0 = 0
    for vid in videos:
        rows = torch.stack([calls[c][0][r] for c, r in vid]).contiguous()
        cnt = torch.stack([calls[c][1][r] for c, r in vid]).contiguous()
        want_p, want_o = evalglue.pack_detections(rows, cnt, torch.tensor(scales[f0:f0 + len(vid)]))
        want_o = want_o.cpu()
        o = off[f0:f0 + len(vid) + 1]
        assert torch.equal(o - o[0], want_o)
        n = int(want_o[-1])
        assert torch.equal(out["packed"][int(o[0]):int(o[0]) + n].cpu().view(torch.int32), want_p[:n].cpu().view(torch.int32))
        assert out["det_cand"][f0:f0 + len(vid)].tolist() == [int(calls[c][2][r]) for c, r in vid]
        f0 += len(vid)
    bad = torch.tensor([[0, 0, 0], [3, 0, 1], [1, 9, 2]], dtype=torch.int32).cuda()
    out = ops.video_pack(calls, bad, None, status)
    torch.cuda.synchronize()
    from tscd_b200 import _lib
    assert int(status.item()) == _lib.TSCD_ERR_INVALID_ARG and out["offsets"].tolist()[1:] == [int(calls[0][1][0])] * 3


CASES = {
    # kind, C, L, G, video lengths, objectness means per frame (None: -3), n_obj
    "ovis_a": ("A", 25, 8, 24, [20, 8, 13], None, 40),
    "ovis_l": ("ovis_l", 25, 8, 24, [17, 10], [-9.0, -5.0, -3.0, -7.0], 12),
    "vid_l": ("vid_l", 30, 1, 31, [12, 7], [-9.0, -8.0, -10.0], 10),
    "wide": ("wide", 30, 2, 6, [9], [-9.0, 3.0, -8.0, -6.0, -9.5, -4.0], 10),
}


def _case_videos(name, seed0=0):
    kind, C, L, G, lens, means, n_obj = CASES[name]
    vids, items, f0 = [], [], 0
    for i, n in enumerate(lens):
        m = -3.0 if means is None else (means * n)[:n]
        vids.append(_video(n, C, seed=seed0 + 10 + i, obj_mean=m, n_obj=n_obj))
        items.append(_item(n, L, G, f0, seed=seed0 + i, ratio=1.0 + 0.25 * i))
        f0 += n
    return vids, items


@pytest.mark.parametrize("name", list(CASES))
def test_stream_matches_device_path(name):
    """Lengths not a multiple of L, a single-clip video (n = L), videos shorter than L + G; two clips per slot chained in one
    call; the still-detector tables (ori=True) as well.  (Frames without rows are covered by
    test_video_pack_matches_pack_detections.)"""
    from tscd_b200.video import VideoStream
    kind, C = CASES[name][:2]
    st = _stage(C, kind)
    vids, items = _case_videos(name)
    vs = VideoStream(st, HW, max_frames=sum(CASES[name][4]), slots=len(vids), clips_per_slot=2, depth=1, ingest_chunk=8, ori=True)
    for v, it in zip(vids, items):
        _write(vs.staging(0), v, it["first_frame"])
    got = vs.collect(vs.submit(0, items))
    total = 0
    for v, it, g in zip(vids, items, got):
        want = _reference(st, C, v, it)
        _assert_table(g, want)
        _assert_ori(g, it)
        total += int(want[1][-1])
    assert total > 0
    if name == "wide":
        assert int(vs.store.count.max()) > 512


def test_stream_matches_forward_host():
    """Default tier, stateful forward_host one clip per call: the same detections as the stream's table."""
    from tscd_b200 import evalglue, ops, stage
    from tscd_b200.video import VideoStream, local_frames
    C, L, G = 25, 8, 24
    st = _stage(C, "A")
    v = _video(20, C, seed=77, obj_mean=-3.0)
    it = _item(20, L, G, 0, seed=5)
    vs = VideoStream(st, HW, max_frames=20, slots=1, clips_per_slot=1, depth=1)
    _write(vs.staging(0), v, 0)
    got = vs.collect(vs.submit(0, [it]))[0]
    pool = stage.CAFMState(1, st.cfg.selection.max_keep(A))
    res = []
    F = len(it["clips"][0])
    for i, (c, p) in enumerate(zip(it["clips"], it["paths"])):
        idx = torch.tensor(c)
        clip = dict(rows=v["rows"][idx], objp=v["objp"][idx], feats=[f[idx] for f in v["feats"]])
        host = dict(rows=[clip["rows"].pin_memory()], objp=[clip["objp"].pin_memory()])
        for k, f in zip(("f_cls", "f_reg", "f_edge"), clip["feats"]):
            lv, s = [], 0
            for h, w in HW:
                t = torch.empty(F, h, w, D, dtype=torch.float16, pin_memory=True)
                t.copy_(f[:, s:s + h * w].reshape(F, h, w, D))
                lv.append(t.permute(0, 3, 1, 2))
                s += h * w
            host[k] = lv
        r, _, _, _ = st.forward_host(host, HW, _te([p]).cpu(), 1, F, L, state=pool, resume=[int(i > 0)], state_slots=[0])
        res.append(r)
    where = local_frames(it["clips"], it["paths"], 20)
    dets = [res[c][l] for c, l in where]
    cap = max([1] + [d.shape[0] for d in dets if d is not None])
    rows = torch.zeros(20, cap, 7)
    cnt = torch.zeros(20, dtype=torch.int32)
    for f, d in enumerate(dets):
        if d is not None:
            rows[f, :d.shape[0]] = d
            cnt[f] = d.shape[0]
    packed, off = evalglue.pack_detections(rows.cuda(), cnt.cuda(), torch.tensor(it["ratios"]))
    off = off.cpu()
    assert torch.equal(got["offsets"], off) and int(off[-1]) > 0
    assert torch.equal(got["packed"].view(torch.int32), packed[:int(off[-1])].cpu().view(torch.int32))
    assert [int(d is not None) for d in dets] == [int(x > 0) for x in got["det_cand"].tolist()]


def test_groups_in_flight_reuse_sets_and_equal_depth_one():
    """depth 2: groups on sets 0, 1, 0, 1 (store ranges, pool slots and buffers reused) give the tables of depth 1; a second
    pass over the same workload captures no new plan (plan_builds stops growing)."""
    from tscd_b200.video import VideoStream
    C = 25
    st = _stage(C, "A")
    vids, items = _case_videos("ovis_a", seed0=100)
    groups = [[0, 1], [2], [1, 2], [0]]

    def run(depth):
        vs = VideoStream(st, HW, max_frames=41, slots=2, clips_per_slot=2, depth=depth, ingest_chunk=16)
        out, pending = [], []
        for gi, g in enumerate(groups):
            s = gi % depth
            if pending and len(pending) == depth:
                out.append(vs.collect(pending.pop(0)))
            f0, its = 0, []
            for v in g:
                _write(vs.staging(s), vids[v], f0)
                its.append(dict(items[v], first_frame=f0))
                f0 += items[v]["num_frames"]
            pending.append(vs.submit(s, its))
        out += [vs.collect(t) for t in pending]
        if depth == 2:                           # the same workload again: every plan is cached
            warm = vs.plan_builds
            pending = []
            for gi, g in enumerate(groups):
                if len(pending) == 2:
                    vs.collect(pending.pop(0))
                f0, its = 0, []
                for v in g:
                    _write(vs.staging(gi % 2), vids[v], f0)
                    its.append(dict(items[v], first_frame=f0))
                    f0 += items[v]["num_frames"]
                pending.append(vs.submit(gi % 2, its))
            for t in pending:
                vs.collect(t)
            vs_builds.append((warm, vs.plan_builds))
        return out

    vs_builds = []

    a, b = run(2), run(1)
    assert vs_builds[0][0] > 0 and vs_builds[0][1] == vs_builds[0][0], vs_builds      # depth 2: the second pass builds nothing
    for ga, gb in zip(a, b):
        for x, y in zip(ga, gb):
            assert torch.equal(x["offsets"], y["offsets"]) and torch.equal(x["packed"].view(torch.int32), y["packed"].view(torch.int32))
    want = _reference(st, C, vids[2], items[2])
    _assert_table(a[2][1], want)


def test_repp_post():
    import json
    import os
    from conftest import GOLDEN
    from tscd_b200.repp import REPPB200
    from tscd_b200.video import VideoStream
    G_ = json.load(open(os.path.join(GOLDEN, "repp.json")))
    post = REPPB200(logreg=G_["logreg"], **G_["cases"][0]["cfg"])
    C = 25
    st = _stage(C, "A")                                   # <= 750 detections per frame (REPP links up to 4096)
    vids, items = _case_videos("ovis_a")
    for it in items:
        it["img_sizes"] = [(480, 640)] * it["num_frames"]
        it["image_ids"] = [f"v/{f:06d}" for f in range(it["num_frames"])]
    vs = VideoStream(st, HW, max_frames=41, slots=3, clips_per_slot=4, depth=1, post=post)
    for v, it in zip(vids, items):
        _write(vs.staging(0), v, it["first_frame"])
    got = vs.collect(vs.submit(0, items))
    for g, it in zip(got, items):
        want = post.from_detections(g["packed"].cuda(), g["offsets"].cuda(), g["det_cand"].tolist(), it["img_sizes"], it["image_ids"])
        assert g["repp"].predictions() == want.predictions()


def test_capacity_error_names_video_and_stream_recovers():
    """A frame that overflows a 64-proposal tier: collect raises naming the video and its frames; the next group runs right."""
    from tscd_b200.video import VideoStream
    C, L, G = 25, 2, 4
    st = _stage(C, "small")
    good = _video(8, C, seed=90, obj_mean=-13.0, n_obj=2)
    bad = _video(8, C, seed=91, obj_mean=[-13.0, -13.0, -13.0, 2.0, -13.0, -13.0, -13.0, -13.0], n_obj=2)
    vs = VideoStream(st, HW, max_frames=16, slots=2, clips_per_slot=2, depth=1, ingest_chunk=4)
    it0, it1 = _item(8, L, G, 0, seed=1), _item(8, L, G, 8, seed=2)
    _write(vs.staging(0), good, 0)
    _write(vs.staging(0), bad, 8)
    t = vs.submit(0, [it0, it1])
    with pytest.raises(RuntimeError, match=r"video 1, frames 0\.\.3: .*capacity exceeded.*wide-tier"):
        vs.collect(t)
    _write(vs.staging(0), good, 8)
    got = vs.collect(vs.submit(0, [it0, dict(it1, clips=it0["clips"], paths=it0["paths"])]))
    want = _reference(st, C, good, it0)
    _assert_table(got[0], want)
    _assert_table(got[1], want)


@pytest.mark.parametrize("kind", ["A", "ovis_l"])
def test_captured_ingest_equals_eager_ingest(kind):
    """The stream's captured ingest chunks (replayed into the store range of buffer set 1) give the store bytes, counts and
    status of eager ingest_host_frames of the same pinned frames."""
    from tscd_b200 import frames
    from tscd_b200.video import VideoStream
    C, L, G = 25, 2, 4
    st = _stage(C, kind)
    v = _video(12, C, seed=30, obj_mean=-3.0 if kind == "A" else [-9.0, -5.0, -3.0, -7.0] * 3, n_obj=40 if kind == "A" else 12)
    vs = VideoStream(st, HW, max_frames=12, slots=1, depth=2, ingest_chunk=5)
    it = _item(12, L, G, 0, seed=3)
    for s_ in (0, 1):
        _write(vs.staging(s_), v, 0)
    vs.collect(vs.submit(0, [it]))
    t = vs.submit(1, [it])                            # second group: the chunks of set 1 replay their graphs
    vs.collect(t)
    assert [x[1:3] for x in t["ingest"]] == [(0, 5), (5, 10), (10, 12)]
    assert all(int(x[3].item()) == 0 for x in t["ingest"])
    kmax = st.cfg.selection.max_keep(A)
    ref = frames.FrameStore(12, kmax, C)
    sel, _ = st.ingest_host_frames(ref, vs.staging(1), HW, list(range(12)))
    torch.cuda.synchronize()
    assert int(sel["status"].item()) == 0
    got = slice(12, 24)
    assert torch.equal(vs.store.count[got], ref.count) and torch.equal(vs.store.status[got], ref.status)
    for f, c in enumerate(ref.count.tolist()):
        for k in ("bank_cls", "bank_reg", "bank_edge", "bank_score", "sel_idx", "sel_rows"):
            assert torch.equal(getattr(vs.store, k)[12 + f, :c], getattr(ref, k)[f, :c]), (f, k)
