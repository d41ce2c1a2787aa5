"""Whole videos from pinned host memory: every frame crosses PCIe once, a video's clips run chained, and the detections come
back as one packed table per video.

    stream = VideoStream(stage, hw, max_frames=600, slots=8, clips_per_slot=4)
    buf = stream.staging(0)                  # pinned, fused-row layout: the producer writes frames here in place
    ...                                      # (tower D2H, decoder): frames [first_frame, first_frame + num_frames) per video
    ticket = stream.submit(0, [dict(first_frame=0, num_frames=n, clips=cl, paths=pa, ratios=r), ...])
    tables = stream.collect(ticket)          # per video: packed [n, 12], offsets [frames + 1], det_cand [frames]

A group (one submit) runs, for the videos it names:
  * ingest: AggregationStage.ingest_host_frames of every video frame, `ingest_chunk` frames per call, into the group's range of
    one FrameStore (K1-K3 once per frame; the objectness plane is copied, the survivors' rows and the kept feature rows are read
    in place), on the stream's i/o stream;
  * clip calls: the videos' clips (clips.demo_clips output) scheduled by clips.ClipScheduler, `slots` videos at a time with up
    to `clips_per_slot` consecutive clips of each chained in one forward_clips call, CAFM memory in the group's CAFMState slots,
    on the compute stream;
  * pack: tscd_video_pack gathers every video frame's detections from the calls, leaves out the padded tail frames demo_clips
    appends, and writes each video's evalglue.pack_detections table (scaled by its resize ratios) back to back;
  * read-back: the status words of every ingest chunk and clip call, the offsets and the candidate counts in one copy queued
    with the group; collect() then copies exactly the valid rows on a copy stream that waits for this group only.
With `depth` buffer sets the ingest of one group overlaps the clip calls of the previous one; buffer sets, store ranges and pool
slots are reused only after the group that used them has finished (events, no host sync).

Errors.  Host-side argument errors are raised by submit() before any launch.  A capacity flag (a frame with more proposals than
the stage's tier holds) is raised by collect(), naming the video and the frames of the ingest call, or the clips of the call,
it came from.  The stream stays usable: every video starts with resume 0 in its group, so the pool slots of the affected videos
begin afresh on the next submit.  The stream runs the stage's own tier; VID TSCD-L frames above 512 proposals need a wide-tier
stage (SelectionConfig(max_proposals=2048)).

Plans.  Every ingest chunk is a captured ingest_host_frames (one CUDA graph per buffer set, chunk start and chunk size, device slot
tensor), and every clip call a captured forward_clips (one graph per B, F, L and chain flags; clip slots, resume flags, state slots
and time embedding are refilled before each replay, the call's detections copied out after it).  The `max_plans` most recently
used plans are kept; `plan_builds` counts the captures, and stops growing once a repeated workload is warm.

Streams.  submit() orders the group after the work queued so far on the caller's current stream (a producer's copies into the
staging buffers); collect() orders the caller's current stream after the group before it hands out device tensors."""
from collections import OrderedDict
from typing import List, Optional, Sequence

import numpy as np
import torch

from . import _lib as L
from . import clips as _clips
from . import frames as _frames
from . import ops
from . import selection as _selection
from .stage import AggregationStage, CAFMState, _no_gc_during_capture


def local_frames(clip_list: Sequence[Sequence[int]], paths: Sequence[Sequence[int]], num_frames: int):
    """For every frame 0..num_frames-1 of a video, the (clip, local index) whose detections are the frame's: the first local
    occurrence in clip order.  The copies of the last frame demo_clips pads the tail clip with come later and are left out (as
    tools/tscd_demo.py trims them).  Raises when a frame is not a local frame of any clip."""
    where = [None] * num_frames
    for c, (cl, pa) in enumerate(zip(clip_list, paths)):
        for l in range(len(pa)):
            f = int(cl[l])
            if 0 <= f < num_frames and where[f] is None:
                where[f] = (c, l)
    missing = [f for f, w in enumerate(where) if w is None]
    if missing:
        raise RuntimeError(f"frames {missing[:8]} of the video are not a local frame of any clip; the clips must cover the "
                           "video (clips.demo_clips)")
    return where


def check_video(i: int, v: dict, max_frames: int, post=None):
    """Host-side checks of one video item of a submit (no device work).  Returns (F, L)."""
    for k in ("first_frame", "num_frames", "clips", "paths", "ratios"):
        if k not in v:
            raise RuntimeError(f"video {i}: missing '{k}' (items hold first_frame, num_frames, clips, paths, ratios)")
    f0, n = int(v["first_frame"]), int(v["num_frames"])
    if n < 1 or f0 < 0:
        raise RuntimeError(f"video {i}: first_frame {f0} / num_frames {n}: need first_frame >= 0 and num_frames >= 1")
    if f0 + n > max_frames:
        raise RuntimeError(f"video {i}: frames [{f0}, {f0 + n}) exceed the {max_frames} frames of a buffer set (max_frames)")
    cl, pa = v["clips"], v["paths"]
    if len(cl) == 0 or len(cl) != len(pa):
        raise RuntimeError(f"video {i}: {len(cl)} clips and {len(pa)} path sequences; pass clips.demo_clips output")
    F, Lf = len(cl[0]), len(pa[0])
    for c, (x, p) in enumerate(zip(cl, pa)):
        if len(x) != F or len(p) != Lf or not 1 <= Lf <= F:
            raise RuntimeError(f"video {i}, clip {c}: {len(x)} frames / {len(p)} local frames; every clip of a video has the same "
                               f"F = {F} frames and L = {Lf} local frames")
        bad = [int(f) for f in x if not 0 <= int(f) < n]
        if bad:
            raise RuntimeError(f"video {i}, clip {c}: frame {bad[0]} outside the video's {n} frames (clip frames are relative to "
                               "the video)")
    if len(v["ratios"]) != n:
        raise RuntimeError(f"video {i}: {len(v['ratios'])} ratios for {n} frames (one resize ratio per frame)")
    if post is not None:
        for k in ("img_sizes", "image_ids"):
            if k not in v or len(v[k]) != n:
                raise RuntimeError(f"video {i}: REPP needs '{k}' with one entry per frame ({n})")
    return F, Lf


def check_group(videos: List[dict], slots: int, max_frames: int, post=None):
    """Host-side checks of one submit (no device work).  Returns ([(F, L)] per video, [local_frames] per video)."""
    if not videos:
        raise RuntimeError("VideoStream.submit: no videos")
    if len(videos) > slots:
        raise RuntimeError(f"VideoStream.submit: {len(videos)} videos for {slots} pool slots; a group holds at most `slots` videos")
    shapes = [check_video(v, item, max_frames, post) for v, item in enumerate(videos)]
    spans = sorted((int(x["first_frame"]), int(x["first_frame"]) + int(x["num_frames"]), v) for v, x in enumerate(videos))
    for (a0, a1, va), (b0, b1, vb) in zip(spans, spans[1:]):
        if b0 < a1:
            raise RuntimeError(f"VideoStream.submit: videos {va} and {vb} overlap in the buffer set ([{a0}, {a1}) and [{b0}, {b1}))")
    return shapes, [local_frames(x["clips"], x["paths"], int(x["num_frames"])) for x in videos]


def check_staging(host: dict, max_frames: int, A: int, row_w: int, hw):
    """A buffer set must be pinned and in the fused-row layout ingest_host_frames reads."""
    if "rows" not in host or "objp" not in host:
        raise RuntimeError("VideoStream: staging buffers must be in the fused-row layout (host['rows'], host['objp'])")
    for k in ("rows", "objp", "f_cls", "f_reg", "f_edge"):
        if k not in host:
            raise RuntimeError(f"VideoStream: staging buffers lack '{k}'")
        for t in host[k]:
            if t.device.type != "cpu" or not t.is_pinned():
                raise RuntimeError(f"VideoStream: staging['{k}'] must be pinned CPU tensors (cudaHostAlloc) so the GPU can read "
                                   "them in place")
            if t.shape[0] < max_frames:
                raise RuntimeError(f"VideoStream: staging['{k}'] holds {t.shape[0]} frames, max_frames is {max_frames}")
    r = host["rows"][0]
    if r.dim() != 3 or r.shape[1] != A or r.shape[2] != row_w:
        raise RuntimeError(f"VideoStream: staging['rows'] must be [frames, {A}, {row_w}], got {tuple(r.shape)}")
    for k in ("f_cls", "f_reg", "f_edge"):
        if len(host[k]) != len(hw) or any(t.shape[2:] != tuple(s) for t, s in zip(host[k], hw)):
            raise RuntimeError(f"VideoStream: staging['{k}'] must hold one [frames, 256, H, W] plane per level {list(hw)}")


class VideoStream:
    """Streams groups of whole videos from pinned host memory through one AggregationStage (see the module docstring).

    stage: the AggregationStage (its tier is used as is); hw / strides: the input's feature-map sizes; max_frames: frames of one
    buffer set; slots: videos of one group (CAFMState pool slots per group); clips_per_slot: consecutive clips of a video chained
    in one call; depth: buffer sets (groups in flight); ingest_chunk: frames per ingest call; post: optional REPPB200, run per
    video by collect(); ori: also pack the still-detector rows (ori_rows); buffers: optional caller-allocated buffer sets (a list
    of `depth` dicts in the fused-row layout, pinned) instead of the stream's own."""

    def __init__(self, stage: AggregationStage, hw, max_frames: int, slots: int, clips_per_slot: int = 1, depth: int = 2,
                 ingest_chunk: int = 64, strides=(8, 16, 32), post=None, ori: bool = False, buffers: Optional[List[dict]] = None,
                 max_plans: int = 64):
        if max_frames < 1 or slots < 1 or clips_per_slot < 1 or depth < 1 or ingest_chunk < 1:
            raise RuntimeError("VideoStream: max_frames, slots, clips_per_slot, depth and ingest_chunk must be positive")
        cfg = stage.cfg
        self.stage, self.hw, self.strides = stage, [tuple(x) for x in hw], tuple(strides)
        self.max_frames, self.slots, self.clips_per_slot, self.depth, self.ingest_chunk = max_frames, slots, clips_per_slot, depth, ingest_chunk
        self.post, self.ori = post, ori
        an = ops.AnchorSpec(self.hw, self.strides)
        self.A = an.num_anchors
        self.kmax = cfg.selection.max_keep(self.A)
        self.wide = _selection.is_wide(cfg.selection.max_proposals)
        dev = stage.device
        row_w = ops.row_pitch(cfg.num_classes)
        if buffers is None:
            buffers = [self._alloc(row_w, cfg.dtype) for _ in range(depth)]
        if len(buffers) != depth:
            raise RuntimeError(f"VideoStream: {len(buffers)} buffer sets for depth {depth}")
        for b in buffers:
            check_staging(b, max_frames, self.A, row_w, self.hw)
        self.buffers = buffers
        self.store = _frames.FrameStore(depth * max_frames, self.kmax, cfg.num_classes, cfg.dim, cfg.dtype, dev)
        self.pool = CAFMState(depth * slots, self.kmax, cfg.dim, dev)
        self._store_slots = torch.arange(depth * max_frames, dtype=torch.int32, device=dev)
        self.io = torch.cuda.Stream(device=dev, priority=-1)
        self.compute = torch.cuda.Stream(device=dev)
        self._d2h = torch.cuda.Stream(device=dev)
        self._free = [None] * depth          # per buffer set: event after the last work of the group that used it
        self._busy = [None] * depth          # per buffer set: the uncollected ticket
        # CUDA-graph plans: ingest chunks keyed on (buffer set, chunk start, chunk size), clip calls on (B, F, L, chain flags);
        # the most recently used `max_plans` are kept (a plan a group in flight uses stays alive through its ticket)
        self._plans = OrderedDict()
        self.max_plans = max_plans
        self.plan_builds = 0                 # captures so far: stops growing once a repeated workload is warm
        self._scratch_pool = None            # clip-plan warm-up runs on a throwaway pool of the real pool's shape

    def _alloc(self, row_w: int, dtype: torch.dtype) -> dict:
        n, A = self.max_frames, self.A
        # uninitialised: the producer writes every frame a group names before submitting it
        host = dict(rows=[torch.empty(n, A, row_w, dtype=torch.float16, pin_memory=True)],
                    objp=[torch.empty(n, (A + 7) // 8 * 8, dtype=torch.float16, pin_memory=True)])
        for k in ("f_cls", "f_reg", "f_edge"):
            host[k] = [torch.empty(n, 256, h, w, dtype=dtype, pin_memory=True, memory_format=torch.channels_last) for h, w in self.hw]
        return host

    def staging(self, i: int) -> dict:
        """Buffer set i (pinned, fused-row layout): rows [max_frames, A, 32|64], objp [max_frames, >=A], per-level channels_last
        f_cls / f_reg / f_edge [max_frames, 256, H, W].  Write a group's frames here before submit(i, ...); a set whose group is
        in flight must be collected first."""
        if self._busy[i] is not None:
            raise RuntimeError(f"VideoStream.staging({i}): buffer set {i} still has a group in flight; collect it first")
        return self.buffers[i]

    # ------------------------------------------------------------------------------------------------------
    def _capture(self, after: torch.cuda.Stream, warm, fn):
        """warm() once eagerly (lazy module loading, per-stream stage state), then fn() captured into a CUDA graph, both on a
        high-priority stream that first waits for `after`.  Returns (graph, what fn returned)."""
        s = torch.cuda.Stream(device=self.stage.device, priority=-1)
        s.wait_stream(after)
        with torch.cuda.stream(s):
            warm()
        g = torch.cuda.CUDAGraph()
        with _no_gc_during_capture(), torch.cuda.graph(g, stream=s):
            out = fn()
        self.plan_builds += 1
        return g, out

    def _plan(self, key, build):
        plan = self._plans.pop(key, None)
        if plan is None:
            plan = build()
        self._plans[key] = plan                  # most recently used last
        while len(self._plans) > self.max_plans:
            self._plans.popitem(last=False)
        return plan

    def _ingest_plan(self, i: int, c0: int, c1: int):
        """Captured ingest_host_frames of frames [c0, c1) of buffer set i into their store slots (a device slot tensor)."""
        def build():
            sub = {k: [t[c0:c1] for t in self.buffers[i][k]] for k in ("rows", "objp", "f_cls", "f_reg", "f_edge")}
            slots = self._store_slots[i * self.max_frames + c0:i * self.max_frames + c1]
            fn = lambda: self.stage.ingest_host_frames(self.store, sub, self.hw, slots, self.strides)   # noqa: E731
            g, (sel, h2d) = self._capture(self.io, fn, fn)
            return dict(graph=g, status=sel["status"], h2d=h2d, sel=sel, sub=sub)
        return self._plan(("ingest", i, c0, c1), build)

    def _clip_plan(self, B: int, F: int, Lf: int, chain: tuple, fill):
        """Captured forward_clips of B clips of F frames, chain flags `chain`, on device input tensors refilled per replay
        (clip slots, resume flags, state slots, time embedding).  `fill(inp)` writes this batch's inputs (before the build too:
        the warm-up runs the real batch, on a throwaway pool)."""
        def build():
            dev = self.stage.device
            inp = dict(slots=torch.zeros(B, F, dtype=torch.int32, device=dev), resume=torch.zeros(B, dtype=torch.int32, device=dev),
                       state_slots=torch.zeros(B, dtype=torch.int32, device=dev),
                       te=torch.zeros(B * Lf, self.stage.cfg.dim, dtype=torch.float32, device=dev))
            fill(inp)
            if self._scratch_pool is None:
                self._scratch_pool = CAFMState(self.pool.slots, self.pool.kmax, self.pool.dim, dev)
            ch = list(chain) if any(chain) else None

            def run(pool):
                return self.stage.forward_clips(self.store, inp["slots"], Lf, inp["te"], state=pool, resume=inp["resume"],
                                                state_slots=inp["state_slots"], chain=ch)
            g, out = self._capture(self.compute, lambda: run(self._scratch_pool), lambda: run(self.pool))
            return dict(graph=g, inp=inp, out=out, built=True)
        plan = self._plan(("clip", B, F, Lf, chain), build)
        if not plan.pop("built", False):
            fill(plan["inp"])
        return plan

    # ------------------------------------------------------------------------------------------------------
    def submit(self, i: int, videos: List[dict]):
        """Launches the group of `videos` held in buffer set i; returns the ticket for collect() without waiting.  The group's
        work is ordered after everything already queued on the caller's current stream (a producer's copies into staging(i))."""
        if not 0 <= i < self.depth:
            raise RuntimeError(f"VideoStream.submit: buffer set {i} outside [0, {self.depth})")
        if self._busy[i] is not None:
            raise RuntimeError(f"VideoStream.submit: buffer set {i} still has a group in flight; collect it first")
        shapes, where = check_group(videos, self.slots, self.max_frames, self.post)
        dev, sbase, pbase = self.stage.device, i * self.max_frames, i * self.slots
        caller = torch.cuda.current_stream()
        ticket = dict(set=i, videos=videos, ingest=[], calls=[], plans=[])

        # ---- ingest (i/o stream): every frame once, in captured chunks per video ----
        self.io.wait_stream(caller)
        if self._free[i] is not None:
            self.io.wait_event(self._free[i])
        ev = {k: torch.cuda.Event(enable_timing=True) for k in ("ingest0", "ingested", "calls", "done")}
        h2d, chunks = 0, []
        for v, x in enumerate(videos):
            f0, n = int(x["first_frame"]), int(x["num_frames"])
            for c0 in range(f0, f0 + n, self.ingest_chunk):
                chunks.append((v, f0, c0, min(c0 + self.ingest_chunk, f0 + n)))
        plans = [self._ingest_plan(i, c0, c1) for _, _, c0, c1 in chunks]      # (builds, if any, before the timed window)
        with torch.cuda.stream(self.io):
            ev["ingest0"].record(self.io)
            for (v, f0, c0, c1), p in zip(chunks, plans):
                p["graph"].replay()
                h2d += p["h2d"]
                ticket["ingest"].append((v, c0 - f0, c1 - f0, p["status"]))
            ev["ingested"].record(self.io)
        ticket["plans"] += plans
        ticket["h2d"] = h2d

        # ---- clip calls (compute stream): captured forward_clips, inputs refilled, outputs copied out per replay ----
        cs = self.compute
        pos = {}                                   # (video, clip) -> (call, batch position)
        cs.wait_event(ev["ingested"])
        for (F, Lf) in sorted(set(shapes)):
            vids = [v for v in range(len(videos)) if shapes[v] == (F, Lf)]
            per_video = [list(zip(videos[v]["clips"], videos[v]["paths"])) for v in vids]
            for batch in _clips.ClipScheduler(per_video, world=1, slots=self.slots, clips_per_slot=self.clips_per_slot).batches(0):
                B = len(batch)
                ints = torch.empty(B * F + 2 * B, dtype=torch.int32, pin_memory=True)
                a = ints.numpy()
                a[:B * F] = [sbase + int(videos[vids[c.video]]["first_frame"]) + int(f) for c in batch for f in c.frames]
                a[B * F:B * F + B] = [c.resume for c in batch]
                a[B * F + B:] = [pbase + c.slot for c in batch]
                te = torch.cat([_clips.time_embedding(c.frame_numbers) for c in batch], 0).pin_memory()

                def fill(inp, ints=ints, te=te, B=B, F=F):
                    with torch.cuda.stream(cs):        # pinned sources: the caching host allocator keeps them until copied
                        inp["slots"].view(-1).copy_(ints[:B * F], non_blocking=True)
                        inp["resume"].copy_(ints[B * F:B * F + B], non_blocking=True)
                        inp["state_slots"].copy_(ints[B * F + B:], non_blocking=True)
                        inp["te"].copy_(te, non_blocking=True)
                plan = self._clip_plan(B, F, Lf, tuple(c.chain for c in batch), fill)
                with torch.cuda.stream(cs):
                    plan["graph"].replay()
                    o = plan["out"]                    # the next replay of this plan overwrites it: keep this call's results
                    keep = {k: o[k].clone() for k in ("det_rows", "det_count", "det_cand", "status")}
                    if self.ori:
                        keep.update({k: o[k].clone() for k in ("ori_rows", "ori_count")})
                for b, c in enumerate(batch):
                    pos[(vids[c.video], c.clip)] = (len(ticket["calls"]), b * Lf)
                ticket["calls"].append(dict(out=keep, clips=[(vids[c.video], c.clip) for c in batch]))
                ticket["plans"].append(plan)

        # ---- pack every video's frames in order + the one header read-back ----
        with torch.cuda.stream(cs):
            ev["calls"].record(cs)
            fmap, scale = [], []
            for v, x in enumerate(videos):
                for f, (c, l) in enumerate(where[v]):
                    call, r = pos[(v, c)]
                    fmap.append((call, r + l, f))
                scale += [float(r_) for r_ in x["ratios"]]
            nf = len(fmap)
            fmap_d = torch.tensor(fmap, dtype=torch.int32).pin_memory().to(dev, non_blocking=True)
            scale_d = torch.tensor(scale, dtype=torch.float32).pin_memory().to(dev, non_blocking=True)
            pack_status = torch.zeros(1, dtype=torch.int32, device=dev)
            outs = [c["out"] for c in ticket["calls"]]
            det = ops.video_pack([(o["det_rows"], o["det_count"], o["det_cand"]) for o in outs], fmap_d, scale_d, pack_status)
            parts = [t[3] for t in ticket["ingest"]] + [o["status"] for o in outs] + [pack_status, det["offsets"], det["det_cand"]]
            ori = None
            if self.ori:
                ori = ops.video_pack([(o["ori_rows"], o["ori_count"], None) for o in outs], fmap_d, scale_d, pack_status)
                parts.append(ori["offsets"])
            header = torch.cat(parts)
            header_h = torch.empty(header.shape, dtype=torch.int32, pin_memory=True)
            header_h.copy_(header, non_blocking=True)
            ev["done"].record(cs)
        self._free[i] = ev["done"]
        self._busy[i] = ticket
        ticket.update(done=ev["done"], events=ev, header=header_h, det=det, ori=ori, nf=nf, _keep=(header, fmap_d, scale_d))
        return ticket

    # ------------------------------------------------------------------------------------------------------
    def _raise_status(self, ticket, hdr):
        n_ing, n_calls = len(ticket["ingest"]), len(ticket["calls"])
        tier = ("" if self.wide else f"; frames of more than {self.kmax} proposals need a wide-tier stage "
                "(SelectionConfig(max_proposals=2048): VID TSCD-L frames above 512)")
        for k, (v, a, b, _) in enumerate(ticket["ingest"]):
            if hdr[k] != 0:
                raise RuntimeError(f"VideoStream: video {v}, frames {a}..{b - 1}: ingest reported error {hdr[k]} (capacity exceeded: "
                                   f"a frame holds more proposals than the per-frame capacity of {self.kmax}){tier}")
        for k, c in enumerate(ticket["calls"]):
            s = hdr[n_ing + k]
            if s != 0:
                what = "capacity exceeded" if s == L.TSCD_ERR_CAPACITY else "stage error"
                clips = ", ".join(f"video {v} clip {c_}" for v, c_ in c["clips"])
                raise RuntimeError(f"VideoStream: clip call {k} ({clips}) reported error {s} ({what}){tier}")
        if hdr[n_ing + n_calls] != 0:
            raise RuntimeError(f"VideoStream: tscd_video_pack reported error {hdr[n_ing + n_calls]} (frame map outside the calls)")

    def _readback(self, ticket, rows: torch.Tensor) -> torch.Tensor:
        """The valid rows into fresh pinned host memory, on a copy stream that waits for this group only (the compute stream
        may already run the next group's clip calls)."""
        h = torch.empty(rows.shape, dtype=rows.dtype, pin_memory=True)
        with torch.cuda.stream(self._d2h):
            self._d2h.wait_event(ticket["done"])
            h.copy_(rows, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(self._d2h)
        ev.synchronize()
        return h

    def collect(self, ticket, timing: Optional[dict] = None) -> List[dict]:
        """Waits for a submitted group; returns per video a dict: 'packed' (host [n, 12], evalglue.pack_detections rows of the
        video's frames in order, scaled by its ratios), 'offsets' (host int32 [frames + 1]), 'det_cand' (host int32 [frames],
        0 = the reference's None), 'packed_dev' / 'offsets_dev' (the same on the device), with ori=True 'ori_packed' /
        'ori_offsets', and with post= 'repp' (post.from_detections of the device table).  Raises on a capacity flag (see the
        module docstring); the stream stays usable."""
        import time as _time
        t0 = _time.perf_counter()
        ticket["done"].synchronize()
        t1 = _time.perf_counter()
        i = ticket["set"]
        if self._busy[i] is ticket:
            self._busy[i] = None
        hdr = ticket["header"].tolist()
        self._raise_status(ticket, hdr)
        nf = ticket["nf"]
        base = len(ticket["ingest"]) + len(ticket["calls"]) + 1
        off = hdr[base:base + nf + 1]
        cand = hdr[base + nf + 1:base + 2 * nf + 1]
        det = ticket["det"]
        table = self._readback(ticket, det["packed"][:off[-1]])
        ori_table = ori_off = None
        if ticket["ori"] is not None:
            ori_off = hdr[base + 2 * nf + 1:base + 3 * nf + 2]
            ori_table = self._readback(ticket, ticket["ori"]["packed"][:ori_off[-1]])
        t2 = _time.perf_counter()
        # the device tables are handed to the caller's stream: order it after the group, and keep the memory (allocated on the
        # compute stream) until the caller's work on it has run
        caller = torch.cuda.current_stream()
        caller.wait_event(ticket["done"])
        for t in (det["packed"], det["offsets"]):
            t.record_stream(caller)
        res, f0 = [], 0
        for x in ticket["videos"]:
            n = int(x["num_frames"])
            o = off[f0:f0 + n + 1]
            r = dict(packed=table[o[0]:o[-1]], offsets=torch.tensor([a - o[0] for a in o], dtype=torch.int32),
                     det_cand=torch.tensor(cand[f0:f0 + n], dtype=torch.int32),
                     packed_dev=det["packed"][o[0]:o[-1]], offsets_dev=det["offsets"][f0:f0 + n + 1] - o[0])
            if ori_table is not None:
                oo = ori_off[f0:f0 + n + 1]
                r.update(ori_packed=ori_table[oo[0]:oo[-1]], ori_offsets=torch.tensor([a - oo[0] for a in oo], dtype=torch.int32))
            if self.post is not None:
                # (at least one row: from_detections sizes its workspaces by the table's rows)
                r["repp"] = self.post.from_detections(det["packed"][o[0]:max(o[-1], o[0] + 1)], r["offsets_dev"], cand[f0:f0 + n],
                                                      x["img_sizes"], x["image_ids"])
            res.append(r)
            f0 += n
        if timing is not None:
            ev = ticket["events"]
            # device phases: ingest (i/o stream), clip calls (from the end of the ingest), pack + header copy
            timing.update(ingest=ev["ingest0"].elapsed_time(ev["ingested"]), calls=ev["ingested"].elapsed_time(ev["calls"]),
                          pack=ev["calls"].elapsed_time(ev["done"]))
            timing.update(wait=1e3 * (t1 - t0), readback=1e3 * (t2 - t1), unpack=1e3 * (_time.perf_counter() - t2),
                          h2d=ticket["h2d"], d2h=ticket["header"].numel() * 4 + table.numel() * 4 +
                          (0 if ori_table is None else ori_table.numel() * 4))
        return res
