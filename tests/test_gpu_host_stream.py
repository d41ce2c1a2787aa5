"""Streaming videos through the host-buffer path with CAFM memory (forward_host(state=pool, resume=, state_slots=)).

  * the kernel-side slot map gives exactly what copying the slots out and back (CAFMState.select / update_from) gives:
    detections and the whole pool, untouched slots included, bit for bit;
  * clips of several videos scheduled by clips.ClipScheduler and streamed through forward_host -- synchronously or with
    several calls in flight, consecutive clips of one video submitted before the previous call is collected -- return exactly
    the detections of the device-path procedure of test_gpu_clip_schedule.py (forward on select()-ed sub-states);
  * the memory is really carried (resume 0 changes resumed clips), and stateless host plans never share memory."""
import pytest
import torch

pytestmark = pytest.mark.gpu

F, C, D = 8, 7, 256
HW = [(24, 24), (12, 12), (6, 6)]
N_CLIPS = [3, 1, 4, 2, 2]          # clips per video


def _sel(mode):
    from tscd_b200 import selection
    if mode == "A":                 # kmax 12: fast chain
        return selection.SelectionConfig(mode="A", pre_k=200, top_k=12, nms_thresh=0.75)
    return selection.SelectionConfig(mode="B", minimal_limit=12, maximal_limit=40, use_pre_nms=False)   # kmax 40: wide chain


def _stage(mode):
    from tscd_b200 import stage, weights
    return stage.AggregationStage(stage.StageConfig(num_classes=C, selection=_sel(mode)), weights.random_state_dict(C, D, seed=5))


def _clip(seed):
    """Head logits (per level) and feature planes of one clip of F frames, on the device."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    out = dict(reg=[], obj=[], cls=[], f_cls=[], f_reg=[], f_edge=[])
    for (h, w) in HW:
        xy = torch.rand(F, 2, h, w, generator=g, device="cuda") * 2 - 0.5
        wh = torch.randn(F, 2, h, w, generator=g, device="cuda") * 0.7 + 1.0
        out["reg"].append(torch.cat([xy, wh], 1).half())
        out["obj"].append((torch.randn(F, 1, h, w, generator=g, device="cuda") * 2 - 3).half())
        out["cls"].append((torch.randn(F, C, h, w, generator=g, device="cuda") * 2 - 3).half())
        for k in ("f_cls", "f_reg", "f_edge"):
            out[k].append(torch.randn(F, D, h, w, generator=g, device="cuda").half().contiguous(memory_format=torch.channels_last))
    return out


def _batch(clips):
    return {k: [torch.cat([c[k][l] for c in clips], 0) for l in range(3)] for k in clips[0]}


def _forward(st, dev, B, Lf, te, **kw):
    from tscd_b200 import ops
    an = ops.AnchorSpec(HW)
    head = ops.HeadViews.from_levels(dev["reg"], dev["obj"], dev["cls"], an)
    feats = tuple(ops.view_levels(dev[k]) for k in ("f_cls", "f_reg", "f_edge"))
    out = st.forward(head, feats, torch.float16, te.cuda(), B, F, Lf, **kw)
    torch.cuda.synchronize()
    return st.to_lists(out, B, Lf)


def _same(a, b):
    for x, y in zip(a, b):
        if (x is None) != (y is None) or (x is not None and not torch.equal(x.cpu(), y.cpu())):
            return False
    return len(a) == len(b)


@pytest.mark.parametrize("mode", ["A", "B"])
def test_slot_map_equals_select_update(mode):
    """forward(state=pool, state_slots=perm) on a 5-slot pool with B = 3 == select -> forward -> update_from."""
    from tscd_b200 import ops, stage, weights
    Lf = 3
    st = _stage(mode)
    kmax = st.cfg.selection.max_keep(ops.AnchorSpec(HW).num_anchors)
    te5 = torch.cat([weights.timing_signal_1d(torch.arange(Lf), 256)] * 5, 0)
    pool = stage.CAFMState(5, kmax, D)
    _forward(st, _batch([_clip(100 + i) for i in range(5)]), 5, Lf, te5, state=pool)   # fill every slot with a memory
    pool2 = stage.CAFMState(5, kmax, D)
    pool2.flat.copy_(pool.flat)
    perm, resume = [3, 0, 4], torch.tensor([1, 0, 1], dtype=torch.int32, device="cuda")
    dev = _batch([_clip(200 + i) for i in range(3)])
    te3 = torch.cat([weights.timing_signal_1d(torch.arange(Lf, 2 * Lf), 256)] * 3, 0)
    got = _forward(st, dev, 3, Lf, te3, state=pool, resume=resume, state_slots=perm)
    sub = pool2.select(perm)
    want = _forward(st, dev, 3, Lf, te3, state=sub, resume=resume)
    pool2.update_from(sub, perm)
    torch.cuda.synchronize()
    assert _same(got[0], want[0]) and _same(got[1], want[1])
    assert sum(len(r) for r in got[0] if r is not None) > 0
    assert torch.equal(pool.flat.view(torch.int32), pool2.flat.view(torch.int32))
    # a device tensor slot map (the form graph capture uses) gives the same again
    pool3 = stage.CAFMState(5, kmax, D)
    pool3.flat.copy_(pool2.flat)
    sub2 = stage.CAFMState(5, kmax, D)
    sub2.flat.copy_(pool2.flat)
    a = _forward(st, dev, 3, Lf, te3, state=pool3, resume=resume, state_slots=torch.tensor(perm, dtype=torch.int32, device="cuda"))
    b = _forward(st, dev, 3, Lf, te3, state=sub2, resume=resume, state_slots=perm)
    assert _same(a[0], b[0]) and torch.equal(pool3.flat.view(torch.int32), sub2.flat.view(torch.int32))


_DATA = {}


def _videos():
    if not _DATA:
        for v, n in enumerate(N_CLIPS):
            for c in range(n):
                _DATA[(v, c)] = _clip(1000 + 10 * v + c)
    return _DATA


def _schedule(Lf):
    from tscd_b200 import clips
    per_video = [[([v, c], list(range(c * Lf, (c + 1) * Lf))) for c in range(n)] for v, n in enumerate(N_CLIPS)]
    return list(clips.ClipScheduler(per_video, world=1, slots=3).batches(0))


def _reference(st, Lf, batches):
    """The device-path procedure of test_gpu_clip_schedule.py: forward on select()-ed slots, written back with update_from."""
    from tscd_b200 import clips, ops, stage
    data = _videos()
    kmax = st.cfg.selection.max_keep(ops.AnchorSpec(HW).num_anchors)
    pool = stage.CAFMState(3, kmax, D)
    want = {}
    for batch in batches:
        slots = [c.slot for c in batch]
        sub = pool.select(slots)
        te = torch.cat([clips.time_embedding(c.frame_numbers) for c in batch], 0)
        res, ori = _forward(st, _batch([data[(c.video, c.clip)] for c in batch]), len(batch), Lf, te, state=sub,
                            resume=torch.tensor([c.resume for c in batch], dtype=torch.int32, device="cuda"))
        pool.update_from(sub, slots)
        for i, c in enumerate(batch):
            want[(c.video, c.clip)] = (res[i * Lf:(i + 1) * Lf], ori[i * Lf:(i + 1) * Lf])
    return want


def _prestage(batches, Lf):
    """Pinned staging buffers of every call (fused head rows + feature planes) and its time embedding, filled up front so
    that the streaming loop itself does no device work between submits."""
    from tscd_b200 import clips, ops
    data = _videos()
    an = ops.AnchorSpec(HW)
    staged = []
    for batch in batches:
        dev = _batch([data[(c.video, c.clip)] for c in batch])
        packed = ops.pack_head(ops.HeadViews.from_levels(dev["reg"], dev["obj"], dev["cls"], an))
        torch.cuda.synchronize()
        h = {k: [torch.empty(t.shape, dtype=t.dtype, pin_memory=True, memory_format=torch.channels_last).copy_(t) for t in dev[k]]
             for k in ("f_cls", "f_reg", "f_edge")}
        h["rows"], h["objp"] = [packed._keep[0].cpu().pin_memory()], [packed._keep[1].cpu().pin_memory()]
        te = torch.cat([clips.time_embedding(c.frame_numbers) for c in batch], 0).pin_memory()
        staged.append((batch, h, te))
    return staged


def _stream(st, Lf, staged, depth, graph, pool, force_resume0=False):
    """The streaming loop of INTEGRATION.md with `depth` calls in flight.  A first pass builds (captures) every call's plan --
    a build synchronises the device -- then the pool is cleared and the pass that is returned runs with no device
    synchronisation between submits: with depth > 1 consecutive clips of one video really are on the GPU together, and only
    the ordering of the pool accesses keeps them apart."""
    def run():
        inflight, got = [], {}

        def collect():
            batch, ticket = inflight.pop(0)
            res, ori, _, _ = st.forward_host_collect(ticket)
            for i, c in enumerate(batch):
                got[(c.video, c.clip)] = (res[i * Lf:(i + 1) * Lf], ori[i * Lf:(i + 1) * Lf])

        for i, (batch, h, te) in enumerate(staged):
            if len(inflight) == depth:
                collect()
            kw = {}
            if pool is not None:
                kw = dict(state=pool, resume=[0 if force_resume0 else c.resume for c in batch], state_slots=[c.slot for c in batch])
            inflight.append((batch, st.forward_host_submit(h, HW, te, len(batch), F, Lf, chunk_clips=2, graph=graph,
                                                           slot=i % depth, **kw)))
        while inflight:
            collect()
        return got

    run()
    if pool is not None:
        pool.flat.zero_()
    torch.cuda.synchronize()
    builds = getattr(st, "host_plan_builds", 0)
    got = run()
    assert st.host_plan_builds == builds            # no plan was built (no device synchronisation) in the returned pass
    return got


@pytest.mark.parametrize("depth", [1, 3])
@pytest.mark.parametrize("graph", [True, False])
@pytest.mark.parametrize("mode", ["A", "B"])
@pytest.mark.parametrize("Lf", [1, 3])
def test_streaming_equals_device_schedule(Lf, mode, graph, depth):
    from tscd_b200 import ops, stage
    st = _stage(mode)
    batches = _schedule(Lf)
    assert any(len(b) < 3 for b in batches) and any(c.resume for b in batches for c in b)
    want = _reference(st, Lf, batches)
    pool = stage.CAFMState(3, st.cfg.selection.max_keep(ops.AnchorSpec(HW).num_anchors), D)
    staged = _prestage(batches, Lf)
    got = _stream(st, Lf, staged, depth, graph, pool)
    assert set(got) == set(want)
    n_det = 0
    for k in want:
        assert _same(got[k][0], want[k][0]) and _same(got[k][1], want[k][1]), k
        n_det += sum(len(r) for r in got[k][0] if r is not None)
    assert n_det > 0
    assert pool._host_in_flight == 0
    # the plan keeps its pool alive (its graph holds the pool's pointers); the device path refuses the pool while a host call
    # on it is in flight (checked before any launch)
    batch, h, te = staged[-1]
    slots = [c.slot for c in batch]
    ticket = st.forward_host_submit(h, HW, te, len(batch), F, Lf, chunk_clips=2, graph=graph, state=pool,
                                    resume=[0] * len(batch), state_slots=slots)
    if graph:
        assert any(x is pool for x in ticket["_keep"])
    with pytest.raises(RuntimeError, match="in flight"):
        st.forward_from_bank(None, len(batch), F, Lf, pool.kmax, None, state=pool, state_slots=slots)
    st.forward_host_collect(ticket)
    assert pool._host_in_flight == 0


@pytest.mark.parametrize("graph", [True, False])
def test_all_calls_in_flight_keep_pool_order(graph):
    """Every call of the stream submitted before the first is collected, with long CAFM phases (mode B wide chain over 8
    local frames per clip): each call's cost kernel and chain must wait for the previous call's on the pool, otherwise a
    resumed clip reads a memory its predecessor has not written yet."""
    from tscd_b200 import ops, stage
    Lf = F
    st = _stage("B")
    batches = _schedule(Lf)
    want = _reference(st, Lf, batches)
    pool = stage.CAFMState(3, st.cfg.selection.max_keep(ops.AnchorSpec(HW).num_anchors), D)
    got = _stream(st, Lf, _prestage(batches, Lf), len(batches), graph, pool)
    for k in want:
        assert _same(got[k][0], want[k][0]) and _same(got[k][1], want[k][1]), k


@pytest.mark.parametrize("mode,Lf", [("A", 1), ("B", 3)])
def test_memory_is_used(mode, Lf):
    """Resume 0 on the same stream changes resumed clips; resume 0 through the pool equals the stateless host call."""
    from tscd_b200 import ops, stage
    st = _stage(mode)
    batches = _schedule(Lf)
    kmax = st.cfg.selection.max_keep(ops.AnchorSpec(HW).num_anchors)
    staged = _prestage(batches, Lf)
    stateful = _stream(st, Lf, staged, 1, True, stage.CAFMState(3, kmax, D))
    zero = _stream(st, Lf, staged, 1, True, stage.CAFMState(3, kmax, D), force_resume0=True)
    stateless = _stream(st, Lf, staged, 1, True, None)
    resumed = [(c.video, c.clip) for b in batches for c in b if c.resume]
    changed = [k for k in resumed if not _same(stateful[k][0], zero[k][0])]
    assert changed, "no resumed clip depends on the carried memory"
    for k in changed:
        assert not _same(stateful[k][0], stateless[k][0])
    for k in zero:
        assert _same(zero[k][0], stateless[k][0]) and _same(zero[k][1], stateless[k][1]), k
    first = [(c.video, c.clip) for b in batches for c in b if not c.resume]
    for k in first:
        assert _same(stateful[k][0], stateless[k][0]), k


def test_stateless_plans_are_isolated():
    """Seven stateless plans (distinct staging buffers) in mode B (kmax 40: the wide chain keeps its memory between frames);
    two in flight on different slots return their synchronous results, and no two cached plans share CAFM memory."""
    from tscd_b200 import ops, weights
    Lf, B = 3, 3
    st = _stage("B")
    an = ops.AnchorSpec(HW)
    te = torch.cat([weights.timing_signal_1d(torch.arange(Lf), 256)] * B, 0).pin_memory()
    hosts = []
    for j in range(7):
        dev = _batch([_clip(3000 + 10 * j + i) for i in range(B)])
        packed = ops.pack_head(ops.HeadViews.from_levels(dev["reg"], dev["obj"], dev["cls"], an))
        torch.cuda.synchronize()
        h = {k: [torch.empty(t.shape, dtype=t.dtype, pin_memory=True, memory_format=torch.channels_last).copy_(t) for t in dev[k]]
             for k in ("f_cls", "f_reg", "f_edge")}
        h["rows"], h["objp"] = [packed._keep[0].cpu().pin_memory()], [packed._keep[1].cpu().pin_memory()]
        hosts.append(h)
    want = [st.forward_host(h, HW, te, B, F, Lf, chunk_clips=2) for h in hosts]

    def check_distinct():
        ptrs = [s.flat.data_ptr() for p in st._host_plans.values() for s in p["states"]]
        assert len(ptrs) == len(set(ptrs))
        return len(ptrs)

    assert len(st._host_plans) >= 7 and check_distinct() >= 14
    for _ in range(2):
        for j in range(1, 7):
            t0 = st.forward_host_submit(hosts[0], HW, te, B, F, Lf, chunk_clips=2, slot=0)
            t1 = st.forward_host_submit(hosts[j], HW, te, B, F, Lf, chunk_clips=2, slot=1)
            for ticket, w in ((t0, want[0]), (t1, want[j])):
                res, ori, _, _ = st.forward_host_collect(ticket)
                assert _same(res, w[0]) and _same(ori, w[1])
        check_distinct()
    assert sum(len(r) for r in want[0][0] if r is not None) > 0
