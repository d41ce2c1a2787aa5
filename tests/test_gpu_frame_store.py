"""Frame store (tscd_b200.frames): K1-K3 once per video frame (AggregationStage.ingest_frames) + clips assembled on the device
(forward_clips = tscd_clip_assemble + forward_from_bank) against the existing path, forward() on clip tensors materialised
with index_select of the per-frame tensors.  The bar is bit-identical: detections, sel_count, row_off, every bank row,
sel_idx and the local frames' sel_rows compare with torch.equal.

Videos are seeded synthetic head outputs (oracle.synth_head_outputs, logits in the fused-row layout the drop-in head emits);
clips come from clips.demo_clips / clips.dataset_clips with a seeded rng, so global frames are drawn from the whole video."""
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
    if kind == "A":                       # OVIS headline selection: top-750 -> NMS 0.75 -> 30
        return selection.SelectionConfig(mode="A", pre_k=750, top_k=30, nms_thresh=0.75)
    if kind == "ovis_l":                  # exps/TSCD_OVIS/ovis_tscd_large.py
        return selection.SelectionConfig(mode="B", minimal_limit=50, maximal_limit=500, use_pre_nms=False)
    if kind == "vid_l":                   # exps/TSCD_VID/vid_tscd_large.py: no maximal_limit
        return selection.SelectionConfig(mode="B", minimal_limit=50, maximal_limit=0, use_pre_nms=False)
    if kind == "wide":
        return selection.SelectionConfig(mode="B", minimal_limit=50, maximal_limit=0, use_pre_nms=False, max_proposals=2048)
    raise ValueError(kind)


def _stage(C, kind):
    from tscd_b200 import stage, weights
    return stage.AggregationStage(stage.StageConfig(num_classes=C, selection=_sel_cfg(kind)), weights.random_state_dict(C, D, seed=11))


def _video(n, C, seed, obj_mean, n_obj=40):
    """One video of n frames on the device: fused head rows (raw logits) + objectness plane, three row-major feature planes."""
    from tscd_b200 import ops
    head, feats = oracle.synth_head_outputs(n, HW, C, dim=D, seed=seed, clustered=True, obj_mean=obj_mean, n_obj=n_obj)
    logit = torch.logit(head[:, :, 4:].clamp(1e-6, 1 - 1e-6))
    rows = torch.zeros(n, A, ops.row_pitch(C), dtype=torch.float16)
    rows[:, :, :4] = head[:, :, :4].half()
    rows[:, :, 4:5 + C] = logit.half()
    objp = torch.zeros(n, (A + 7) // 8 * 8, dtype=torch.float16)
    objp[:, :A] = rows[:, :, 4]
    return dict(rows=rows.cuda(), objp=objp.cuda(), feats=[f.half().cuda().contiguous() for f in feats])


def _pick(v, idx):
    """Clip tensors materialised from per-frame tensors with index_select (the caller keeps the dict alive while the views are
    in use: tscd_view holds raw pointers)."""
    return {k: ([t.index_select(0, idx) for t in x] if isinstance(x, list) else x.index_select(0, idx)) for k, x in v.items()}


def _views(v, C, edge=None):
    from tscd_b200 import ops
    an = ops.AnchorSpec(HW)
    head = ops.HeadViews.from_rows(v["rows"], v["objp"], an, C)
    feats = [ops.view_rowmajor(f, an) for f in v["feats"]]
    if edge is not None:
        feats[2] = edge
    return head, tuple(feats)


@pytest.fixture(autouse=True)
def _collect():
    """Leave no cyclic garbage holding device objects behind for later tests (it could be collected inside their graph capture)."""
    yield
    import gc
    gc.collect()
    torch.cuda.synchronize()


def _edge_block(seed=5):
    from tscd_b200 import ops
    g = torch.Generator().manual_seed(seed)
    w3 = [torch.randn(256, 256, 3, 3, generator=g) * 0.02 for _ in range(3)]
    b3 = [torch.randn(256, generator=g) * 0.1 for _ in range(3)]
    w1 = [torch.randn(768, 768, 1, 1, generator=g) * 0.03 for _ in range(3)]
    b1 = [torch.randn(768, generator=g) * 0.1 for _ in range(3)]
    return ops.EdgeBlock(w3, b3, w1, b1, dtype=torch.float16)


def _te(paths):
    from tscd_b200 import clips
    return torch.cat([clips.time_embedding(p) for p in paths], 0).cuda()


def _same(a, b):
    return len(a) == len(b) and all((x is None) == (y is None) and (x is None or torch.equal(x.cpu(), y.cpu())) for x, y in zip(a, b))


def _assert_identical(st, ref, got, B, F, L):
    sr, sg = ref["sel"], got["sel"]
    assert torch.equal(sr["sel_count"], sg["sel_count"]) and torch.equal(sr["row_off"], sg["row_off"])
    n = int(sr["row_off"][-1])
    for k in ("bank_cls", "bank_reg", "bank_edge", "bank_score"):
        assert torch.equal(sr[k][:n], sg[k][:n]), k
    cnt = sr["sel_count"].tolist()
    for f in range(B * F):
        assert torch.equal(sr["sel_idx"][f, :cnt[f]], sg["sel_idx"][f, :cnt[f]]), f
        if f % F < L:
            assert torch.equal(sr["sel_rows"][f, :cnt[f]], sg["sel_rows"][f, :cnt[f]]), f
    r_ref, r_got = st.to_lists(ref, B, L), st.to_lists(got, B, L)
    assert _same(r_ref[0], r_got[0]) and _same(r_ref[1], r_got[1])
    assert sum(len(r) for r in r_ref[0] if r is not None) > 0
    return cnt


def _run_both(st, C, v, clip_list, paths, L, edge=None, store=None, base=0, chunk=16):
    """forward() on index_select-ed clip tensors vs ingest_frames (once per frame) + forward_clips, chunk clips per call."""
    from tscd_b200 import frames
    n = v["rows"].shape[0]
    kmax = st.cfg.selection.max_keep(A)
    if store is None:
        store = frames.FrameStore(base + n, kmax, C)
        st.ingest_frames(store, *_views(v, C, edge), torch.float16, list(range(base, base + n)))
    F = len(clip_list[0])
    counts = []
    for c0 in range(0, len(clip_list), chunk):
        cl, pa = clip_list[c0:c0 + chunk], paths[c0:c0 + chunk]
        B = len(cl)
        idx = torch.tensor([f for c in cl for f in c], dtype=torch.long, device="cuda")
        te = _te(pa)
        clip_v = _pick(v, idx)
        ref = st.forward(*_views(clip_v, C, edge), torch.float16, te, B, F, L)
        got = st.forward_clips(store, [[base + f for f in c] for c in cl], L, te)
        torch.cuda.synchronize()
        assert int(ref["status"].item()) == 0
        counts += _assert_identical(st, ref, got, B, F, L)
    return store, counts


def test_mode_a_ovis_headline_with_edge_block():
    """Mode A, C 25, 8 local + 24 global, fused rows, the edge block evaluated at the kept proposals."""
    from tscd_b200 import clips
    C, L, G = 25, 8, 24
    st = _stage(C, "A")
    v = _video(44, C, seed=1, obj_mean=-3.0)
    cl, pa = clips.demo_clips(44, L, G, rng=random.Random(7))
    assert len(cl) == 6                                   # 5 full clips + a padded tail clip
    _run_both(st, C, v, cl, pa, L, edge=_edge_block())


def test_mode_b_ovis_l():
    """Mode B, minimal_limit 50 / maximal_limit 500 (ragged 50..500 proposals per frame)."""
    from tscd_b200 import clips
    C, L, G = 25, 8, 24
    st = _stage(C, "ovis_l")
    v = _video(40, C, seed=2, obj_mean=[-9.0, -5.0, -3.0, -7.0] * 10, n_obj=12)
    cl, pa = clips.demo_clips(40, L, G, rng=random.Random(8))
    _, counts = _run_both(st, C, v, cl, pa, L)
    assert min(counts) >= 50 and max(counts) > 150


def test_mode_b_vid_l():
    """Mode B, C 30, 1 local + 31 global, minimal_limit 50 and no maximal_limit (kmax 512)."""
    from tscd_b200 import clips
    C, L, G = 30, 1, 31
    st = _stage(C, "vid_l")
    v = _video(36, C, seed=3, obj_mean=[-9.0, -8.0, -10.0] * 12, n_obj=10)
    cl, pa = clips.demo_clips(36, L, G, rng=random.Random(9))
    assert len(cl) == 36
    _, counts = _run_both(st, C, v, cl, pa, L, chunk=12)
    assert max(counts) > 50


def test_repeated_slots_tail_clip_and_short_video():
    """A padded tail clip (demo_clips) and an OVIS short video padded with its last frame (dataset_clips): slots repeat inside a
    clip.  The short video sits in the upper slots of a larger store (slots 27..46)."""
    from tscd_b200 import clips
    C, L, G = 25, 8, 24
    st = _stage(C, "A")
    v = _video(27, C, seed=4, obj_mean=-3.0)
    cl, pa = clips.demo_clips(27, L, G, rng=random.Random(3))    # 27 <= L + G: gframe shrinks, tail padded
    assert any(len(set(c)) < len(c) for c in cl)
    store, _ = _run_both(st, C, v, cl, pa, L, chunk=2)
    short = _video(20, C, seed=5, obj_mean=-3.0)
    cs = clips.dataset_clips([list(range(20))], L, G, mode="random", dataset="ovis", rng=random.Random(4))
    assert cs and all(len(c) == L + G and len(set(c)) < len(c) for c in cs)
    from tscd_b200 import frames
    big = frames.FrameStore(27 + 20, store.kmax, C)
    st.ingest_frames(big, *_views(short, C), torch.float16, torch.arange(27, 47, dtype=torch.int32, device="cuda"))
    _run_both(st, C, short, cs, [list(range(i * L, (i + 1) * L)) for i in range(len(cs))], L, store=big, base=27)


def test_wide_tier():
    """max_proposals 2048 with frames of more than 512 proposals, against the wide-tier forward."""
    from tscd_b200 import clips
    C, L, G = 30, 2, 6
    st = _stage(C, "wide")
    means = [-9.0, 3.0, -8.0, -6.0, -9.5, -4.0] * 3
    v = _video(18, C, seed=6, obj_mean=means, n_obj=10)
    cl, pa = clips.demo_clips(18, L, G, rng=random.Random(5))
    store, counts = _run_both(st, C, v, cl, pa, L)
    assert store.kmax == A and max(counts) > 512


def test_clip_scheduler_with_cafm_pool():
    """Several videos through ClipScheduler with a CAFMState pool (resume, state_slots) == the same schedule on forward."""
    from tscd_b200 import clips, frames, stage
    C, L, G = 25, 2, 4
    st = _stage(C, "A")
    lens = [13, 8, 17, 10]
    vids = [_video(n, C, seed=20 + i, obj_mean=-3.0) for i, n in enumerate(lens)]
    base = [sum(lens[:i]) for i in range(len(lens))]
    rng = random.Random(11)
    per_video = []
    for n in lens:
        cl, pa = clips.demo_clips(n, L, G, rng=rng)
        per_video.append(list(zip(cl, pa)))
    kmax = st.cfg.selection.max_keep(A)
    store = frames.FrameStore(sum(lens), kmax, C)
    for i, v in enumerate(vids):                      # every frame of a video before any of its clips
        st.ingest_frames(store, *_views(v, C), torch.float16, list(range(base[i], base[i] + lens[i])))
    pool_ref, pool_new = stage.CAFMState(3, kmax), stage.CAFMState(3, kmax)
    allv = dict(rows=torch.cat([v["rows"] for v in vids]), objp=torch.cat([v["objp"] for v in vids]),
                feats=[torch.cat([v["feats"][k] for v in vids]) for k in range(3)])
    n_batches = 0
    for batch in clips.ClipScheduler(per_video, world=1, slots=3).batches(0):
        B = len(batch)
        slots = [c.slot for c in batch]
        resume = [c.resume for c in batch]
        idx = torch.tensor([base[c.video] + f for c in batch for f in c.frames], dtype=torch.long, device="cuda")
        te = _te([c.frame_numbers for c in batch])
        clip_v = _pick(allv, idx)
        ref = st.forward(*_views(clip_v, C), torch.float16, te, B, L + G, L, state=pool_ref,
                         resume=torch.tensor(resume, dtype=torch.int32, device="cuda"), state_slots=slots)
        got = st.forward_clips(store, [[base[c.video] + f for f in c.frames] for c in batch], L, te, state=pool_new,
                               resume=resume, state_slots=slots)
        torch.cuda.synchronize()
        _assert_identical(st, ref, got, B, L + G, L)
        n_batches += 1
    assert n_batches >= 5
    assert torch.equal(pool_ref.flat.view(torch.int32), pool_new.flat.view(torch.int32))


def _host_planes(v):
    """Pinned host copies in forward_host's fused layout: rows / objp + per-level channels_last feature planes."""
    host = dict(rows=[v["rows"].cpu().pin_memory()], objp=[v["objp"].cpu().pin_memory()])
    n = v["rows"].shape[0]
    for k, f in zip(("f_cls", "f_reg", "f_edge"), v["feats"]):
        lv, s = [], 0
        for h, w in HW:
            t = torch.empty(n, h, w, D, dtype=torch.float16, pin_memory=True)
            t.copy_(f[:, s:s + h * w].reshape(n, h, w, D))
            lv.append(t.permute(0, 3, 1, 2))            # [n, 256, h, w], channels_last strides
            s += h * w
        host[k] = lv
    return host


@pytest.mark.parametrize("kind", ["A", "ovis_l"])
def test_host_ingest_equals_device_ingest(kind):
    """Pinned host frames (objectness copied; mode A reads the survivors' rows in place, mode B copies them; feature rows read
    in place) give the same store contents as device ingest, bit for bit."""
    from tscd_b200 import frames
    C = 25
    st = _stage(C, kind)
    v = _video(12, C, seed=30, obj_mean=-3.0 if kind == "A" else [-9.0, -5.0, -3.0, -7.0] * 3, n_obj=40 if kind == "A" else 12)
    kmax = st.cfg.selection.max_keep(A)
    dev_store, host_store = frames.FrameStore(16, kmax, C), frames.FrameStore(16, kmax, C)
    slots = [3, 15, 0, 7, 1, 2, 9, 4, 13, 5, 6, 8]
    st.ingest_frames(dev_store, *_views(v, C), torch.float16, slots)
    _, h2d = st.ingest_host_frames(host_store, _host_planes(v), HW, slots)
    torch.cuda.synchronize()
    assert h2d == v["objp"].numel() * 2 + (0 if kind == "A" else v["rows"].numel() * 2)
    assert torch.equal(dev_store.count, host_store.count) and torch.equal(dev_store.status, host_store.status)
    cnt = dev_store.count.tolist()
    assert sorted(s for s, c in enumerate(cnt) if c >= 0) == sorted(slots) and max(cnt) > 0
    for s, c in enumerate(cnt):
        for k in ("bank_cls", "bank_reg", "bank_edge", "bank_score", "sel_idx", "sel_rows"):
            assert torch.equal(getattr(dev_store, k)[s, :max(c, 0)], getattr(host_store, k)[s, :max(c, 0)]), (s, k)


def test_captured_forward_clips_refill_and_replay():
    """forward_clips captured with capture_fn on a device clip_slots tensor: refill the slots (and time embedding), replay, and
    the result equals an eager call on the new slots."""
    from tscd_b200 import clips, frames
    C, L, G = 25, 8, 24
    st = _stage(C, "A")
    v = _video(40, C, seed=40, obj_mean=-3.0)
    kmax = st.cfg.selection.max_keep(A)
    store = frames.FrameStore(40, kmax, C)
    st.ingest_frames(store, *_views(v, C), torch.float16, torch.arange(40, dtype=torch.int32, device="cuda"))
    c1, p1 = clips.demo_clips(40, L, G, rng=random.Random(1))
    c2, p2 = clips.demo_clips(40, L, G, rng=random.Random(2))
    B = 4
    slots = torch.tensor(c1[:B], dtype=torch.int32, device="cuda")
    te = _te(p1[:B])
    graph, out = st.capture_fn(lambda: st.forward_clips(store, slots, L, te))
    slots.copy_(torch.tensor(c2[1:B + 1], dtype=torch.int32))
    te.copy_(_te(p2[1:B + 1]))
    graph.replay()
    torch.cuda.synchronize()
    eager = st.forward_clips(store, c2[1:B + 1], L, _te(p2[1:B + 1]))
    torch.cuda.synchronize()
    _assert_identical(st, eager, out, B, L + G, L)
    del graph


def test_never_written_slot_raises():
    """A clip that references a slot never written (count -1) -- or one outside the store, given on the device -- raises from
    to_lists and names the cause; nothing is read from the slot."""
    from tscd_b200 import frames
    C, L = 25, 2
    st = _stage(C, "A")
    v = _video(8, C, seed=50, obj_mean=-3.0)
    store = frames.FrameStore(10, st.cfg.selection.max_keep(A), C)
    st.ingest_frames(store, *_views(v, C), torch.float16, list(range(8)))
    te = _te([[0, 1]])
    ok = st.forward_clips(store, [[0, 1, 2, 3, 4, 5]], L, te)
    st.to_lists(ok, 1, L)
    bad = st.forward_clips(store, [[0, 1, 2, 9, 4, 5]], L, te)           # slot 9: never written
    with pytest.raises(RuntimeError, match="never written"):
        st.to_lists(bad, 1, L)
    off = st.forward_clips(store, torch.tensor([[0, 1, 2, 3, 4, 77]], dtype=torch.int32, device="cuda"), L, te)
    with pytest.raises(RuntimeError, match="outside the FrameStore"):
        st.to_lists(off, 1, L)
    with pytest.raises(RuntimeError, match="outside"):                    # host-side slots are checked before any launch
        st.forward_clips(store, [[0, 1, 2, 3, 4, 77]], L, te)


def test_captured_ingest_equals_eager_ingest():
    """ingest_frames with frame_slots as an int32 device tensor, captured with capture_fn: refill the slot tensor, replay, and
    the store equals an eager ingest into the same slots (mode B, ragged counts)."""
    from tscd_b200 import frames
    C = 25
    st = _stage(C, "ovis_l")
    v = _video(10, C, seed=60, obj_mean=[-9.0, -5.0, -3.0, -7.0, -6.0] * 2, n_obj=12)
    kmax = st.cfg.selection.max_keep(A)
    cap, ref = frames.FrameStore(24, kmax, C), frames.FrameStore(24, kmax, C)
    slots = torch.arange(10, dtype=torch.int32, device="cuda")
    head, feats = _views(v, C)
    graph, _ = st.capture_fn(lambda: st.ingest_frames(cap, head, feats, torch.float16, slots))
    new = [23, 4, 17, 0, 9, 12, 5, 20, 1, 14]
    slots.copy_(torch.tensor(new, dtype=torch.int32))
    graph.replay()
    st.ingest_frames(ref, head, feats, torch.float16, new)
    torch.cuda.synchronize()
    cnt = ref.count.tolist()
    assert all(cnt[s] >= 50 for s in new)
    # the capture's warm-up and first replay wrote slots 0..9 as well: compare the slots of the replay
    assert torch.equal(cap.count[new], ref.count[new]) and torch.equal(cap.status[new], ref.status[new])
    for s in new:
        for k in ("bank_cls", "bank_reg", "bank_edge", "bank_score", "sel_idx", "sel_rows"):
            assert torch.equal(getattr(cap, k)[s, :cnt[s]], getattr(ref, k)[s, :cnt[s]]), (s, k)
    del graph


def test_ingest_status_and_bad_device_slot():
    """A capacity flag of an ingest call reaches every slot the call writes, whatever else the call reports: a device slot outside
    the store goes to the separate slot_error word and does not overwrite it.  The clips that use those slots raise."""
    from tscd_b200 import frames, selection, stage, weights
    C = 25
    cfg = stage.StageConfig(num_classes=C, selection=selection.SelectionConfig(mode="B", minimal_limit=20, maximal_limit=0,
                                                                               use_pre_nms=False, max_proposals=64))
    st = stage.AggregationStage(cfg, weights.random_state_dict(C, D, seed=11))
    v = _video(6, C, seed=70, obj_mean=[-9.0, 2.0, -9.0, -9.0, -9.0, -9.0], n_obj=4)    # frame 1 keeps far more than 64
    store = frames.FrameStore(8, st.cfg.selection.max_keep(A), C)
    sel = st.ingest_frames(store, *_views(v, C), torch.float16, torch.tensor([0, 1, 2, 3, 99, 5], dtype=torch.int32, device="cuda"))
    torch.cuda.synchronize()
    from tscd_b200 import _lib
    assert int(sel["status"].item()) == _lib.TSCD_ERR_CAPACITY and int(sel["slot_error"].item()) == _lib.TSCD_ERR_FRAME_SLOT
    assert store.status.tolist() == [_lib.TSCD_ERR_CAPACITY] * 4 + [0, _lib.TSCD_ERR_CAPACITY, 0, 0]
    assert store.count.tolist()[4] == -1 and store.count.tolist()[6:] == [-1, -1]
    with pytest.raises(RuntimeError, match="capacity exceeded"):
        st.to_lists(st.forward_clips(store, [[0, 2, 3]], 1, _te([[0]])), 1, 1)
    with pytest.raises(RuntimeError, match="never written"):
        st.to_lists(st.forward_clips(store, [[4, 2, 3]], 1, _te([[0]])), 1, 1)


def test_forward_clips_on_an_empty_store_raises():
    from tscd_b200 import frames
    C = 25
    st = _stage(C, "A")
    store = frames.FrameStore(4, st.cfg.selection.max_keep(A), C)
    with pytest.raises(RuntimeError, match="holds no frames yet"):
        st.forward_clips(store, [[0, 1]], 1, _te([[0]]))
