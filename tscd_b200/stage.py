"""The TSCD aggregation stage as one host-side object: everything in TSCDHead.forward after the decoupled-head
convolutions (yolox/models/tscd_head.py:374-733), for a BATCH of clips, on hand-written sm_100a kernels.

Host code is plumbing only (buffer allocation through torch, C-ABI calls on the current stream).  All
data-dependent sizes stay on the device until the single read-back that turns the padded detection tensors
into the reference's `list[Tensor[n,7] | None]` containers.  There is no CPU / PyTorch fallback: if
libtscd_b200.so is missing `tscd_b200._lib.lib()` raises.
"""
import math
from dataclasses import dataclass, field
from typing import Dict, List, Optional

import numpy as np
import torch

from . import _lib as L
from . import aggregate, ops
from . import frames as _frames
from . import selection as _selection
from .selection import SelectionConfig


def _r128(x: int) -> int:
    return (x + 127) // 128 * 128


class _no_gc_during_capture:
    """Keeps Python's cyclic garbage collector from running inside a CUDA-graph capture.  torch.cuda.graph collects once on
    entry, but a collection triggered during the capture can free cyclic garbage of earlier calls (host plans, pinned staging
    buffers, graphs) whose destructors make CUDA calls that are illegal while a stream is capturing, which aborts the process."""

    def __enter__(self):
        import gc
        self.was = gc.isenabled()
        gc.disable()

    def __exit__(self, *exc):
        import gc
        if self.was:
            gc.enable()
        return False


@dataclass
class StageConfig:
    num_classes: int
    selection: SelectionConfig = field(default_factory=SelectionConfig)
    dim: int = 256                    # int(256 * width); the kernels are specialised for 256 (TSCD-L)
    heads: int = 4
    sim_thresh: float = 0.75          # TSCDHead ctor `sim_thresh`
    conf_sim_thresh: float = 0.99     # kwargs['conf_sim_thresh'] (post_trans.py:693)
    final_nms_thresh: float = 0.5     # forward(..., nms_thresh=0.5)
    final_conf_thresh: float = 0.001  # post_process.py:10 default (not overridable in the reference)
    dtype: torch.dtype = torch.float16  # tensor-core operand type (fp16 = the reference's eval dtype; bf16 also supported)


def validate_config(cfg: StageConfig):
    """Capacity limits of the kernels, checked when the stage is CONSTRUCTED (not at the first forward): a configuration
    that cannot fit is rejected here with the limit it breaks."""
    sel = cfg.selection
    sel.validate()
    kmax = sel.top_k if sel.mode == "A" else sel.max_proposals
    if sel.mode == "B" and sel.maximal_limit:
        kmax = max(sel.maximal_limit, sel.minimal_limit)
    if _selection.is_wide(sel.max_proposals):
        if kmax * cfg.num_classes > ops.NMS_WIDE_CAP:
            raise RuntimeError(
                f"final per-class NMS (wide tier, max_proposals = {sel.max_proposals} > {_selection.DEFAULT_TIER_MAX}): up to {kmax} "
                f"proposals x {cfg.num_classes} classes = {kmax * cfg.num_classes} candidate rows per frame exceed the NMS capacity "
                f"of {ops.NMS_WIDE_CAP}; lower max_proposals / maximal_limit to <= {ops.NMS_WIDE_CAP // cfg.num_classes}")
    elif kmax * cfg.num_classes > ops.NMS_MAX_CAP:
        raise RuntimeError(
            f"final per-class NMS: up to {kmax} proposals x {cfg.num_classes} classes = {kmax * cfg.num_classes} candidate rows per "
            f"frame (post_process.py:36-46) exceed the NMS capacity of {ops.NMS_MAX_CAP}; lower max_proposals / maximal_limit "
            f"to <= {ops.NMS_MAX_CAP // cfg.num_classes}")
    if cfg.num_classes > 255:
        raise RuntimeError("more than 255 classes are not supported (8-bit class ids in the selection kernels)")


MAX_KEYS_PER_CLIP = _frames.MAX_KEYS_PER_CLIP     # attention kernels: keys of one clip (csrc/attn.cu, 16-bit key index in row_meta)


def check_state_args(B: int, kmax: int, state=None, resume=None, state_slots=None, host: bool = False):
    """Validates the CAFM-memory arguments of one call of B clips (no device work; raises RuntimeError).

    state: a CAFMState; resume: [B] flags; state_slots: [B] slot of every clip in `state` (a list / array, or an int32 device
    tensor, whose values are then not read back: capture-safe).  Without state_slots the state holds exactly B slots (clip b
    uses slot b).  host=True: the forward_host rules -- state, resume and state_slots go together.  host=False: the device
    path, which refuses a pool that still has forward_host calls in flight (their CAFM phases are ordered on the device
    only among themselves)."""
    where = "forward_host" if host else "forward"
    if state is None:
        if state_slots is not None or (host and resume is not None):
            raise RuntimeError(f"{where}: resume / state_slots were given without state; pass the CAFMState pool they refer to")
        return
    if host and (resume is None or state_slots is None):
        raise RuntimeError(f"{where}: state needs resume and state_slots (one resume flag and one state slot per clip)")
    if state.kmax != kmax:
        raise RuntimeError(f"{where}: the CAFMState holds {state.kmax} rows per slot, this configuration needs kmax = {kmax} "
                           f"(SelectionConfig.max_keep); allocate CAFMState(slots, {kmax})")
    for name, v in (("resume", resume), ("state_slots", state_slots)):
        if host and isinstance(v, torch.Tensor) and v.device.type != "cpu":
            raise RuntimeError(f"{where}: {name} must be host-side (a list, NumPy array or CPU tensor); it is copied with the call")
        if v is not None and len(v) != B:
            raise RuntimeError(f"{where}: {name} has {len(v)} entries for {B} clips")
    if state_slots is not None:
        if isinstance(state_slots, torch.Tensor) and state_slots.is_cuda:
            if state_slots.dtype != torch.int32 or state_slots.dim() != 1:
                raise RuntimeError(f"{where}: a device state_slots tensor must be 1-D int32")
        else:
            sl = np.asarray(state_slots.cpu() if isinstance(state_slots, torch.Tensor) else state_slots).reshape(-1)
            bad = [int(x) for x in sl if not 0 <= int(x) < state.slots]
            if bad:
                raise RuntimeError(f"{where}: state slot(s) {bad} outside [0, {state.slots}) of the CAFMState pool")
            if len(set(int(x) for x in sl)) != len(sl):
                raise RuntimeError(f"{where}: duplicate state slot in one call ({sorted(int(x) for x in sl)}); the clips of a "
                                   "call run concurrently and need distinct slots")
    if not host and state._host_in_flight:
        raise RuntimeError(f"{where}: the CAFMState pool still has {state._host_in_flight} forward_host call(s) in flight; "
                           "collect them (forward_host_collect) before using the pool on the device path")


class StageWeights:
    """Device copies of the aggregation-stage parameters (reference state_dict key names, SURVEY App. B)."""

    def __init__(self, sd: Dict[str, torch.Tensor], cfg: StageConfig, device="cuda"):
        dt = cfg.dtype

        def w16(name):
            return sd[name].detach().to(device=device, dtype=dt).contiguous()

        def f32(name):
            return sd[name].detach().to(device=device, dtype=torch.float32).contiguous()

        self.agg = aggregate.MCAWeights(sd, "agg.", dt, device)
        self.agg_iou = aggregate.MCAWeights(sd, "agg_iou.", dt, device)
        m = "local_reg_matcher."
        lay = m + "transformer_aware_cross_attention_layers.0."
        self.ape_w, self.ape_b = w16(m + "absolute_position_embedding.weight"), f32(m + "absolute_position_embedding.bias")
        self.cafm_wk = w16(lay + "multihead_attn.k_reg.weight")
        self.cafm_wv = w16(lay + "multihead_attn.v_reg.weight")
        self.cafm_wq_t = f32(lay + "multihead_attn.q_reg.weight").t().contiguous()     # [in, out] (generic chain)
        self.cafm_wq16 = w16(lay + "multihead_attn.q_reg.weight")                       # [out, in] (fast chain, kmax <= 32)
        self.se_w1, self.se_w2 = f32(lay + "CA.fc.0.weight"), f32(lay + "CA.fc.2.weight")
        self.cafm_ln_w, self.cafm_ln_b = f32(lay + "norm.weight"), f32(lay + "norm.bias")
        self.cafm_dec_w, self.cafm_dec_b = f32(m + "decoder_norm.weight"), f32(m + "decoder_norm.bias")
        self.fc_w, self.fc_b = w16("fc_reg_matcher.weight"), f32("fc_reg_matcher.bias")
        t = "task_aligned.transformer_cross_attention_layers.0."
        self.ta_wq = w16(t + "multihead_attn.q_reg.weight")
        self.ta_wkv = torch.cat([w16(t + "multihead_attn.k_reg.weight"), w16(t + "multihead_attn.v_reg.weight")], 0).contiguous()
        self.ta_ln_w, self.ta_ln_b = f32(t + "norm.weight"), f32(t + "norm.bias")
        self.ta_dec_w, self.ta_dec_b = f32("task_aligned.decoder_norm.weight"), f32("task_aligned.decoder_norm.bias")
        self.cls_w, self.cls_b = w16("cls_pred.weight"), f32("cls_pred.bias")
        self.obj_w, self.obj_b = w16("matcher_obj_pred.weight"), f32("matcher_obj_pred.bias")
        self.obj_w32 = self.obj_w.float().reshape(-1).contiguous()       # the 16-bit weight values, fp32 storage (fused head)
        self.reg_w, self.reg_b = w16("matcher_reg_pred.weight"), f32("matcher_reg_pred.bias")


class CAFMState:
    """Caller-owned CAFM memory (tscd_matching.py:708-715) for `slots` concurrent video streams.  All fields are views of ONE
    flat fp32 buffer (`flat`; `n` is its first `slots` words viewed as int32), so handing the memory to another rank in the
    long-clip mode is a single message."""

    def widened(self, kmax: int) -> "CAFMState":
        """Copy of this state with a larger row capacity `kmax` (rows beyond the old capacity are zero; the chain only reads
        the first n).  The drop-in head moves a video's memory to the wide tier with it."""
        if kmax < self.kmax:
            raise RuntimeError(f"CAFMState.widened: kmax {kmax} < current {self.kmax}")
        big = CAFMState(self.slots, kmax, self.dim, self.flat.device)
        for f in self._FIELDS:
            src, dst = getattr(self, f), getattr(big, f)
            if f in ("n", "time"):
                dst.copy_(src)
            else:
                dst[:, :self.kmax].copy_(src)
        return big

    def __init__(self, slots: int, kmax: int, dim: int = 256, device="cuda"):
        self.slots, self.kmax, self.dim = slots, kmax, dim
        self._host_in_flight = 0           # submitted, not yet collected stateful forward_host calls on this pool
        self._host_cafm_done = None        # CAFM-done event of the most recently submitted of them (ordering of pool accesses)
        self._host_order_stream = None     # stream on which those calls' gates are recorded (created by the first of them)
        sizes = [("n", slots), ("out", slots * kmax * dim), ("edge", slots * kmax * dim), ("reg", slots * kmax * 4 * dim),
                 ("cls", slots * kmax * 4 * dim), ("nreg", slots * kmax), ("ncls", slots * kmax), ("time", slots * dim)]
        total = sum(((n + 3) // 4) * 4 for _, n in sizes)            # every field 16-byte aligned
        self.flat = torch.zeros(total, dtype=torch.float32, device=device)
        off, views = 0, {}
        for name, n in sizes:
            views[name] = self.flat[off:off + n]
            off += ((n + 3) // 4) * 4
        self.n = views["n"].view(torch.int32)
        self.out, self.edge = views["out"].view(slots, kmax, dim), views["edge"].view(slots, kmax, dim)
        self.reg, self.cls = views["reg"].view(slots, kmax, 4 * dim), views["cls"].view(slots, kmax, 4 * dim)
        self.nreg, self.ncls, self.time = views["nreg"].view(slots, kmax), views["ncls"].view(slots, kmax), views["time"].view(slots, dim)

    _FIELDS = ("n", "out", "edge", "reg", "cls", "nreg", "ncls", "time")

    def select(self, slot_ids) -> "CAFMState":
        """Copy of the given slots as a dense state (batch position i <- slot slot_ids[i]): for batches that run only some of
        the concurrent video streams (tscd_b200.clips.ClipScheduler near the end of a rank's work list)."""
        sub = CAFMState(len(slot_ids), self.kmax, self.dim, self.flat.device)
        idx = torch.as_tensor(list(slot_ids), dtype=torch.long, device=self.flat.device)
        for f in self._FIELDS:
            getattr(sub, f).copy_(getattr(self, f).index_select(0, idx))
        return sub

    def update_from(self, sub: "CAFMState", slot_ids):
        """Write a dense sub-state back into its slots (inverse of select)."""
        idx = torch.as_tensor(list(slot_ids), dtype=torch.long, device=self.flat.device)
        for f in self._FIELDS:
            getattr(self, f).index_copy_(0, idx, getattr(sub, f))


class AggregationStage:
    """forward(): head outputs + feature planes of B clips x F frames -> refined detections of the B x L local frames."""

    def __init__(self, cfg: StageConfig, state_dict: Dict[str, torch.Tensor], device="cuda"):
        if cfg.dim != 256 or cfg.heads != 4:
            raise RuntimeError("tscd_b200 kernels are specialised for TSCD-L (dim 256, 4 heads)")
        L.lib()  # fail loudly if the CUDA library is missing
        validate_config(cfg)
        self.cfg = cfg
        self.w = StageWeights(state_dict, cfg, device)
        self.device = device
        self._side = {}
        self._part_streams = []
        self._default_state = {}
        self._zero_resume = {}
        self.serialize = False     # True: run the classification branch on the launching stream (per-kernel profiling passes)

    def _side_stream(self):
        """Side stream of the classification branch, one per launching stream (concurrent sub-batches must not share it)."""
        key = torch.cuda.current_stream().cuda_stream
        if key not in self._side:
            self._side[key] = torch.cuda.Stream(device=self.device)
        return self._side[key]

    # ------------------------------------------------------------------------------------------------------
    def forward_concurrent(self, parts, feat_dtype, F: int, Lf: int):
        """Run independent sub-batches of clips concurrently, each on its own stream (plus its own side stream).

        Clips are independent units of work, and most kernels of the stage are latency-bound with modest grids (one
        CTA per clip / frame), so two or more sub-batches in flight fill the SMs that a single launch sequence leaves
        idle: the front end (select / NMS / gather) of one sub-batch overlaps the attention / CAFM tail of another.
        parts: list of (head_views, feats, time_embedding, n_clips).  Returns the list of forward() outputs; all streams
        are joined into the current stream before returning (CUDA-graph capturable)."""
        main = torch.cuda.current_stream()
        while len(self._part_streams) < len(parts):
            self._part_streams.append(torch.cuda.Stream(device=self.device))
        fork = torch.cuda.Event()
        fork.record(main)
        outs, joins = [], []
        for i, (head, feats, te, nb) in enumerate(parts):
            st = self._part_streams[i]
            with torch.cuda.stream(st):
                st.wait_event(fork)
                outs.append(self.forward(head, feats, feat_dtype, te, nb, F, Lf))
                ev = torch.cuda.Event()
                ev.record(st)
                joins.append(ev)
        for ev in joins:
            main.wait_event(ev)
        return outs

    # ------------------------------------------------------------------------------------------------------
    def forward(self, head: ops.HeadViews, feats, feat_dtype, time_embedding: torch.Tensor, B: int, F: int, Lf: int,
                state: Optional[CAFMState] = None, resume: Optional[torch.Tensor] = None, trace: Optional[dict] = None,
                state_slots=None):
        """state_slots (optional, with `state`): [B] slot of every clip in `state` (list, or int32 device tensor -- the latter
        under CUDA-graph capture); the kernels then read and write those slots in place, so `state` may be a pool with more
        slots than clips (one per concurrent video).  Without it `state` holds exactly B slots, clip b in slot b."""
        cfg, w, dev, dt = self.cfg, self.w, self.device, self.cfg.dtype
        C = cfg.num_classes
        D = cfg.dim
        assert head.num_frames == B * F and 1 <= Lf <= F
        A = head.anchors.num_anchors
        kmax = cfg.selection.max_keep(A)
        _frames.check_keys_per_clip(F, kmax)
        check_state_args(B, kmax, state, resume, state_slots)
        status = torch.zeros(1, dtype=torch.int32, device=dev)

        # ---- K1-K3: selection + bank (operand arrays are read in 128-row TMA boxes: capacity padded) ------
        row_cap = _r128(B * F * kmax) + 128
        sel = _selection.select_and_gather(head, feats, feat_dtype, D, cfg.selection, bank_dtype=dt, status=status,
                                           bank_rows=row_cap)
        return self.forward_from_bank(sel, B, F, Lf, kmax, time_embedding, state=state, resume=resume, trace=trace,
                                      status=status, state_slots=state_slots)

    # ------------------------------------------------------------------------------------------------------
    def _store_kmax(self, store: _frames.FrameStore, A: Optional[int] = None) -> int:
        """kmax of this stage for the frames of `store`: A = anchors per frame of the frames at hand (ingest_frames), else those
        of the frames ingested so far (forward_clips)."""
        if A is None:
            if store.num_anchors is None:
                raise RuntimeError("forward_clips: the FrameStore holds no frames yet; ingest_frames the frames of the clips first")
            A = store.num_anchors
        elif store.num_anchors not in (None, A):
            raise RuntimeError(f"ingest_frames: the FrameStore holds frames of {store.num_anchors} anchors, these frames have {A}; "
                               "one store holds frames of one input size")
        return self.cfg.selection.max_keep(A)

    def ingest_frames(self, store: _frames.FrameStore, head: ops.HeadViews, feats, feat_dtype, frame_slots):
        """K1-K3 (selection, pre-NMS, bank gather, edge rows) ONCE for N video frames, written into the slots `frame_slots` of
        `store` (tscd_frame_scatter).  head / feats: the N frames in any layout forward() accepts (fused rows, per level,
        row-major, or an EdgeBlock as feats[2]).  frame_slots: [N] distinct slots (a list, or an int32 device tensor -- then
        nothing is read back and the call can be captured into a CUDA graph).  Returns the K1-K3 output of the N frames: its
        'status' is the flag every written slot carries (a capacity error shows up in the clips that use these frames), and
        'slot_error' ([1] int32, device) is TSCD_ERR_FRAME_SLOT when a device-tensor slot lay outside the store -- such a frame is
        not written, and nothing else reports it (host-side slots are checked before any launch).
        Capacity flags are per call, not per frame: ingesting a video in several calls narrows which clips an overflow stops."""
        cfg, dev, dt = self.cfg, self.device, self.cfg.dtype
        A, N = head.anchors.num_anchors, head.num_frames
        kmax = self._store_kmax(store, A)
        _frames.check_clip_args(store, frame_slots, kmax, cfg.num_classes, cfg.dim, dt, num_frames=N)
        store.num_anchors = A
        slots = self._slot_tensor(frame_slots)
        status = torch.zeros(1, dtype=torch.int32, device=dev)
        sel = _selection.select_and_gather(head, feats, feat_dtype, cfg.dim, cfg.selection, bank_dtype=dt, status=status,
                                           bank_rows=_r128(N * kmax) + 128)
        sel["slot_error"] = torch.zeros(1, dtype=torch.int32, device=dev)
        ops.frame_scatter(store, slots, sel, status, sel["slot_error"])
        return sel

    def ingest_host_frames(self, store: _frames.FrameStore, host: dict, hw, frame_slots, strides=(8, 16, 32)):
        """ingest_frames for N frames in PINNED HOST memory, in the fused-row layout forward_host reads: host['rows'] = [rows
        [N, A, 32|64] fp16], host['objp'] = [objectness plane [N, >=A]], host['f_cls' / 'f_reg' / 'f_edge'] = per-level
        [N, 256, H, W] channels_last planes.  As in forward_host, the objectness plane is copied; in mode A, K1 / K3 read the
        survivors' rows in place, mode B copies the rows; K3 reads the kept proposals' feature rows in place (UVA).  So each
        frame crosses PCIe once however many clips use it.  Eager launches, no host sync.  Returns (K1-K3 output, bytes
        copied host->device); the bytes read in place follow from the counts (tools/bench_frame_store.py)."""
        an = ops.AnchorSpec(hw, strides)
        if "rows" not in host:
            raise RuntimeError("ingest_host_frames: host frames must be in the fused-row layout (host['rows'], host['objp'])")
        for k in ("rows", "objp", "f_cls", "f_reg", "f_edge"):
            for t in host[k]:
                if t.device.type != "cpu" or not t.is_pinned():
                    raise RuntimeError(f"ingest_host_frames: host['{k}'] must be pinned CPU tensors (cudaHostAlloc) so the GPU can "
                                       "read them in place; there is no pageable-memory / CPU path")
        rows_in_place = self.cfg.selection.mode == "A"
        copied = ("objp",) if rows_in_place else ("objp", "rows")
        dbuf = {k: host[k][0].to(self.device, non_blocking=True) for k in copied}
        h2d = sum(host[k][0].numel() * host[k][0].element_size() for k in copied)
        head = ops.HeadViews.from_rows(host["rows"][0] if rows_in_place else dbuf["rows"], dbuf["objp"], an, self.cfg.num_classes)
        feats = tuple(ops.view_levels(host[k]) for k in ("f_cls", "f_reg", "f_edge"))
        return self.ingest_frames(store, head, feats, host["f_cls"][0].dtype, frame_slots), h2d

    def forward_clips(self, store: _frames.FrameStore, clip_slots, Lf: int, time_embedding: torch.Tensor,
                      state: Optional[CAFMState] = None, resume=None, state_slots=None):
        """The stage for B clips whose frames are in `store` (ingest_frames): clip_slots [B, F] holds the slot of every frame of
        every clip, local frames first (a slot may repeat, within a clip too).  tscd_clip_assemble rebuilds the packed clip bank
        K1-K3 would have produced for those frames, then forward_from_bank runs the rest; the result is the dict forward()
        returns (to_lists works unchanged), bit for bit.  clip_slots as an int32 device tensor: nothing is read back, and the
        call can be captured (capture_fn) and replayed with refilled slots.  state / resume / state_slots: as in forward()."""
        cfg, dt = self.cfg, self.cfg.dtype
        kmax = self._store_kmax(store)
        _frames.check_clip_args(store, clip_slots, kmax, cfg.num_classes, cfg.dim, dt, L=Lf)
        slots = self._slot_tensor(clip_slots)
        B, F = slots.shape
        check_state_args(B, kmax, state, resume, state_slots)
        status = torch.zeros(1, dtype=torch.int32, device=self.device)
        sel = ops.clip_assemble(store, slots, B, F, Lf, _r128(B * F * kmax) + 128, status)
        return self._from_bank(sel, B, F, Lf, kmax, time_embedding, state, resume, status=status, state_slots=state_slots)

    def _slot_tensor(self, slots) -> torch.Tensor:
        if isinstance(slots, torch.Tensor) and slots.is_cuda:
            return slots
        return torch.tensor(np.asarray(slots.cpu() if isinstance(slots, torch.Tensor) else slots, dtype=np.int32),
                            dtype=torch.int32, device=self.device)

    # ------------------------------------------------------------------------------------------------------
    def forward_host(self, host: dict, hw, time_embedding: torch.Tensor, B: int, F: int, Lf: int, chunk_clips: int = 8,
                     strides=(8, 16, 32), zero_copy_logits: bool = False, graph: bool = True, lanes: int = 4,
                     state: Optional[CAFMState] = None, resume=None, state_slots=None):
        """The stage for callers whose boundary tensors live in (pinned) HOST memory -> detections on the host.

        `host` holds per-level lists of pinned CPU tensors: the feature planes f_cls, f_reg, f_edge ([B*F, 256, H, W],
        channels_last) and the head logits either in the fused layout the drop-in head emits -- rows [B*F, A, 32|64] +
        objp [B*F, >=A] (include/tscd_b200.h tscd_pack_head) -- or per level (reg, obj, cls: [B*F, ch, H, W]).  Only what
        the kernels consume crosses PCIe:
          * fused layout, mode A: the 2-byte objectness plane is copied host->device on a copy stream (13.6 KB per frame),
            one chunk of clips ahead of compute; K1 / K3 fetch the ~pre_k survivors' 64-byte rows IN PLACE from the pinned
            tensor (cp.async / vector loads over PCIe; tools/zc_probe.cu measures 380 M rows/s = 24 GB/s for this pattern);
            per-level layouts: the whole logits (~0.4 MB per frame) are copied;
          * the 256-channel feature planes (10.4 MB per frame) are NOT copied: K3 gathers the kept proposals' rows straight
            out of the pinned host tensors (3 x 512 B per kept proposal), exactly the rows find_feature_score
            (tscd_head.py:976-1006) indexes;
          * detections come back as two padded tensors + counts in ONE device->host copy per chunk.
        graph=True: the whole call (copies, every chunk's ~130 launches on two streams, read-backs) is captured ONCE per set
        of host buffers into a CUDA graph and replayed afterwards -- callers that reuse their pinned staging buffers pay one
        cudaGraphLaunch per call instead of ~1.4 ms of launch overhead per chunk.  (The graph reads the buffers at their
        addresses: new tensors -> new capture; the eight most recent plans are kept.)
        forward_host = forward_host_submit + forward_host_collect; callers that stream clips keep two calls in flight (two
        `slot`s: separate staging / output buffers and graphs) so that the PCIe phases of one call overlap the compute tail and the
        host-side unpacking of the previous one.
        CAFM memory: without `state` every clip starts a new video (resume 0; the plan's own scratch memory).  With `state` (a
        caller-owned CAFMState pool of any number of slots >= B, kmax = SelectionConfig.max_keep), `resume` ([B] flags) and
        `state_slots` ([B] distinct slots of the pool) the call continues the videos held in those slots, exactly like
        forward(state=, resume=, state_slots=): a video's clips can be streamed through successive calls.  The flags and the
        slot map are copied per call, so one captured plan serves every slot map.
        Returns (result, result_ori, h2d_bytes, d2h_bytes) with fresh host tensors in the reference's list layout."""
        return self.forward_host_collect(self.forward_host_submit(host, hw, time_embedding, B, F, Lf, chunk_clips, strides,
                                                                  zero_copy_logits, graph, lanes, state=state, resume=resume,
                                                                  state_slots=state_slots))

    def forward_host_submit(self, host: dict, hw, time_embedding: torch.Tensor, B: int, F: int, Lf: int, chunk_clips: int = 8,
                            strides=(8, 16, 32), zero_copy_logits: bool = False, graph: bool = True, lanes: int = 4, slot: int = 0,
                            state: Optional[CAFMState] = None, resume=None, state_slots=None):
        """Launches one forward_host call without waiting for it; returns the ticket for forward_host_collect.  Calls submitted with
        different `slot`s own separate buffers and may be in flight together; a slot must be collected before it is reused.
        (`slot` is the in-flight buffer set; `state_slots` are CAFM memory slots of `state`, see forward_host.)
        Stateful calls on one pool access it in submission order: each call's CAFM phases (matching costs + chain) wait for
        those of the call submitted before it on the same pool, while its copies, selection and attention overlap them."""
        if _selection.is_wide(self.cfg.selection.max_proposals):
            raise RuntimeError(f"forward_host: the host-buffer path supports the default tier only (max_proposals <= "
                               f"{_selection.DEFAULT_TIER_MAX}); use forward() for max_proposals = {self.cfg.selection.max_proposals}")
        check_state_args(B, self.cfg.selection.max_keep(ops.AnchorSpec(hw, strides).num_anchors), state, resume, state_slots,
                         host=True)
        fused = "rows" in host
        head_keys = ("rows", "objp") if fused else ("reg", "obj", "cls")
        for k in head_keys + ("f_cls", "f_reg", "f_edge"):
            for t in host[k]:
                if t.device.type != "cpu" or not t.is_pinned():
                    raise RuntimeError(f"forward_host: host['{k}'] must be pinned CPU tensors (cudaHostAlloc) so the GPU can "
                                       "read them in place; there is no pageable-memory / CPU path")
        key = (tuple((k, t.data_ptr(), tuple(t.shape), t.stride(), t.dtype) for k in head_keys + ("f_cls", "f_reg", "f_edge") for t in host[k]),
               tuple(tuple(x) for x in hw), tuple(strides), B, F, Lf, chunk_clips, zero_copy_logits, graph, lanes,
               tuple(time_embedding.shape), slot,
               None if state is None else (state.flat.data_ptr(), state.slots, state.kmax, state.dim))   # the graph holds the pool's field pointers
        plans = self.__dict__.setdefault("_host_plans", {})
        plan = plans.pop(key, None)
        if plan is None:
            plan = self._build_host_plan(host, hw, time_embedding, B, F, Lf, chunk_clips, strides, zero_copy_logits, graph, fused, lanes,
                                         state)
            self.host_plan_builds = getattr(self, "host_plan_builds", 0) + 1      # diagnostics: a caller that keeps missing the plan cache pays a capture per call
        plans[key] = plan                                      # most recently used last
        while len(plans) > 8:
            idle = next((k for k, v in plans.items() if not v.get("busy") and v is not plan), None)
            if idle is None:
                break
            plans.pop(idle)
        if plan.get("busy"):
            raise RuntimeError("forward_host_submit: this slot still has a call in flight (collect it first or use another slot)")
        # plain single-threaded memcpy: torch's copy_ / clone of more than 32 K elements open an OpenMP region, and waking (then
        # spinning) the whole intra-op pool once per call starves this thread on CPU-quota-limited containers (measured: 8 ms here
        # and 28 ms in the unpack instead of 0.2 / 0.5 ms, intermittently, depending on the box)
        np.copyto(plan["te_pin"].numpy(), time_embedding.detach().cpu().numpy())
        if state is not None:
            np.copyto(plan["resume_pin"].numpy(), np.asarray(resume, dtype=np.int64).reshape(-1), casting="unsafe")
            np.copyto(plan["slots_pin"].numpy(), np.asarray(state_slots, dtype=np.int64).reshape(-1), casting="unsafe")
            # ordering of the pool's accesses: this call's CAFM phases (graph: event-wait nodes on `gate`) start after the
            # previous call's on the same pool have finished (its `cafm_done`).  One ordering stream per pool: calls on other
            # pools do not wait for this one.
            if state._host_order_stream is None:
                state._host_order_stream = torch.cuda.Stream(device=self.device)
            order = state._host_order_stream
            if state._host_cafm_done is not None:
                order.wait_event(state._host_cafm_done)
            plan["gate"].record(order)
        if plan["graph"] is not None:
            with torch.cuda.stream(plan["launch"]):            # one launch stream per plan: calls of different slots run concurrently
                plan["graph"].replay()
                plan["done"].record()
        else:
            plan["issue"](state)
            plan["done"].record()
        if state is not None:                                  # launched: from here on this call is the pool's last one
            state._host_cafm_done = plan["cafm_done"]
            state._host_in_flight += 1
        plan["busy"] = True
        plan["pool"] = state
        return plan

    def forward_host_collect(self, plan, timing: Optional[dict] = None):
        """Waits for a submitted call and returns (result, result_ori, h2d_bytes, d2h_bytes).  `timing` (optional dict) receives
        the host-side split of this call in ms: 'wait' (event synchronise) and 'unpack' (detections -> reference list layout)."""
        import time as _time
        t0 = _time.perf_counter()
        plan["done"].synchronize()
        t1 = _time.perf_counter()
        plan["busy"] = False
        if plan.get("pool") is not None:
            plan["pool"]._host_in_flight -= 1
            plan["pool"] = None
        result, result_ori, d2h = [], [], 0
        h2d = plan["h2d"]
        for nc, pk in plan["pend"]:
            r, o, nb, zb = self._unpack_host(pk, nc * plan["Lf"])
            result += r
            result_ori += o
            d2h += nb
            h2d += zb
        if timing is not None:
            timing["wait"] = 1e3 * (t1 - t0)
            timing["unpack"] = 1e3 * (_time.perf_counter() - t1)
        return result, result_ori, h2d, d2h

    def _build_host_plan(self, host, hw, time_embedding, B, F, Lf, chunk_clips, strides, zero_copy_logits, graph, fused, n_lanes,
                         pool=None):
        """Staging buffers + the launch sequence of one forward_host call (optionally captured into a CUDA graph).
        pool: the caller's CAFMState (stateful plan) or None (the plan owns one scratch CAFMState per chunk: resume 0)."""
        dev = self.device
        an = ops.AnchorSpec(hw, strides)
        feat_dtype = host["f_cls"][0].dtype
        head_keys = ("rows", "objp") if fused else ("reg", "obj", "cls")
        # Mode A only touches the objectness plane plus the class / regression rows of the ~pre_k survivors.
        #  * fused layout: the objectness plane is copied and K1 / K3 read the survivors' 64-byte rows in place (measured,
        #    profiles/zc_probe_r2.txt: 24 GB/s for 750-of-6804 row sets vs 55 GB/s for the copy engine moving all 435 KB);
        #  * per-level layouts: zero_copy_logits=True copies just `obj` and reads the separate class / regression rows in
        #    place.  Measured slower (40 k clip-frames/s vs 93 k): two unaligned bursts per survivor -> off by default.
        zc = (not fused) and zero_copy_logits and self.cfg.selection.mode == "A" and all(t.stride(1) == 1 for t in host["cls"]) \
            and all(t.stride(1) == 1 for t in host["reg"])
        rows_in_place = fused and self.cfg.selection.mode == "A"
        copied = (("objp",) if rows_in_place else ("objp", "rows")) if fused else (("obj",) if zc else ("reg", "obj", "cls"))
        dbuf = {k: [torch.empty_strided(t.shape, t.stride(), dtype=t.dtype, device=dev) for t in host[k]] for k in copied}
        te_pin = torch.empty(time_embedding.shape, dtype=time_embedding.dtype, pin_memory=True)
        te_pin.copy_(time_embedding)
        cp = torch.cuda.Stream(device=dev)
        io = torch.cuda.Stream(device=dev, priority=-1)
        aux = [torch.cuda.Stream(device=dev, priority=-1) for _ in range(max(0, n_lanes - 1))]
        chunks = [(c0, min(chunk_clips, B - c0)) for c0 in range(0, B, chunk_clips)]
        plan = {"te_pin": te_pin, "graph": None, "pend": None, "h2d": 0, "_keep": (dbuf, host, cp, aux, io), "Lf": Lf, "busy": False,
                "done": torch.cuda.Event(), "launch": torch.cuda.Stream(device=dev, priority=-1)}
        fused_row_bytes = host["rows"][0].shape[2] * 2 if fused else None
        kmax = self.cfg.selection.max_keep(an.num_anchors)
        if pool is None:
            # stateless: CAFM memory owned by the plan, one state per chunk (chunks run concurrently); never read (resume 0)
            plan["states"] = [CAFMState(nc, kmax, self.cfg.dim, dev) for _, nc in chunks]
        else:
            # stateful: per-call resume flags and slot map, filled by forward_host_submit and copied with the call; external
            # events so that the ordering also holds between graph replays (event record / wait nodes)
            plan["resume_pin"] = torch.zeros(B, dtype=torch.int32, pin_memory=True)
            plan["slots_pin"] = torch.arange(B, dtype=torch.int32).pin_memory()
            plan["gate"], plan["cafm_done"] = torch.cuda.Event(external=True), torch.cuda.Event(external=True)
            plan["cafm_join"] = torch.cuda.Stream(device=dev)
            plan["_keep"] += (pool,)          # the graph holds the pool's pointers: its memory must not go to another pool
            for ev in (plan["gate"], plan["cafm_done"]):   # created (recorded once) before capture: waits on an unrecorded event are no-ops
                ev.record(torch.cuda.current_stream())

        def issue(st=None):
            main = torch.cuda.current_stream()
            cp.wait_stream(main)                               # earlier work on this stream is done with the staging buffers
            events, h2d = [], 0
            with torch.cuda.stream(cp):
                te_dev = te_pin.to(dev, non_blocking=True)
                h2d += te_pin.numel() * te_pin.element_size()
                if st is not None:
                    resume_dev = plan["resume_pin"].to(dev, non_blocking=True)
                    slots_dev = plan["slots_pin"].to(dev, non_blocking=True)
                    h2d += 2 * 4 * B
                for (c0, nc) in chunks:
                    f0, f1 = c0 * F, (c0 + nc) * F
                    for k in copied:
                        for l, t in enumerate(host[k]):
                            dbuf[k][l][f0:f1].copy_(t[f0:f1], non_blocking=True)
                            h2d += (f1 - f0) * t[0].numel() * t.element_size()
                    ev = torch.cuda.Event()
                    ev.record(cp)
                    events.append(ev)
            te_dev.record_stream(main)
            # Software pipeline over chunks of clips: ONE i/o lane runs K1 -> K2 -> K3 of every chunk back to back -- these are
            # the PCIe-bound kernels (survivor rows and kept feature rows are read in place), so the link never idles --
            # while the tensor-core / latency-bound tail of the previous chunks runs on the compute lanes.  (Chunks that walk
            # through all phases in lockstep on parallel lanes leave the link idle during every compute phase.)
            cfg_sel = self.cfg.selection
            if _r128(F * kmax) > MAX_KEYS_PER_CLIP:
                raise RuntimeError(f"{F} frames x {kmax} proposals per frame exceed the attention kernels' capacity of {MAX_KEYS_PER_CLIP} keys per clip")
            lanes = ([main] + aux)[:max(1, min(len(chunks), n_lanes))]
            io.wait_stream(main)
            for a_ in lanes[1:]:
                a_.wait_stream(main)
            banks = []
            with torch.cuda.stream(io):
                for (c0, nc), ev in zip(chunks, events):
                    f0, f1 = c0 * F, (c0 + nc) * F
                    io.wait_event(ev)
                    if fused:
                        rows_src = host["rows"][0] if rows_in_place else dbuf["rows"][0]
                        head = ops.HeadViews.from_rows(rows_src[f0:f1], dbuf["objp"][0][f0:f1], an, self.cfg.num_classes)
                    else:
                        src = {k: (dbuf[k] if k in copied else host[k]) for k in ("reg", "obj", "cls")}
                        head = ops.HeadViews.from_levels([t[f0:f1] for t in src["reg"]], [t[f0:f1] for t in src["obj"]],
                                                         [t[f0:f1] for t in src["cls"]], an)
                    feats = tuple(ops.view_levels([t[f0:f1] for t in host[k]]) for k in ("f_cls", "f_reg", "f_edge"))
                    status = torch.zeros(1, dtype=torch.int32, device=dev)
                    sel = _selection.select_and_gather(head, feats, feat_dtype, self.cfg.dim, cfg_sel, bank_dtype=self.cfg.dtype,
                                                       status=status, bank_rows=_r128(nc * F * kmax) + 128)
                    evb = torch.cuda.Event()
                    evb.record(io)
                    banks.append((sel, status, evb))
            pend, cafm_evs = [], []
            for ci, ((c0, nc), (sel, status, evb)) in enumerate(zip(chunks, banks)):
                lane_s = lanes[ci % len(lanes)]
                with torch.cuda.stream(lane_s):
                    lane_s.wait_event(evb)
                    if lane_s is not main:
                        for t in (te_dev,) if st is None else (te_dev, resume_dev, slots_dev):
                            t.record_stream(lane_s)
                    te_c = te_dev[c0 * Lf:(c0 + nc) * Lf]
                    if st is None:
                        out = self._from_bank(sel, nc, F, Lf, kmax, te_c, plan["states"][ci], None, status=status)
                    else:                      # chunk c0..c0+nc: its slice of the flags and of the slot map
                        ev_c = torch.cuda.Event()
                        out = self._from_bank(sel, nc, F, Lf, kmax, te_c, st, resume_dev[c0:c0 + nc], status=status,
                                              state_slots=slots_dev[c0:c0 + nc], cafm_gate=plan["gate"],
                                              after_cafm=lambda _s, e=ev_c: e.record())
                        cafm_evs.append(ev_c)
                    reuse = plan["pend"][len(pend)][1] if plan["pend"] is not None else None
                    pend.append((nc, self._pack_to_host(out, zc or rows_in_place, fused_row_bytes, reuse)))
            if st is not None:                 # every chunk's chain is done with the pool -> the next call on it may start its CAFM
                ordst = plan["cafm_join"]
                for e in cafm_evs:
                    ordst.wait_event(e)
                plan["cafm_done"].record(ordst)
                main.wait_stream(ordst)
                for t in (resume_dev, slots_dev):
                    t.record_stream(main)
            main.wait_stream(io)
            for a_ in lanes[1:]:
                main.wait_stream(a_)
            # the banks were allocated on the i/o lane and are read on the compute lanes: keep them until the call has synchronised
            plan["_banks"] = banks
            plan["pend"], plan["h2d"] = pend, h2d

        plan["issue"] = issue
        if graph:
            # warm up (lazy module loading, per-stream stage state) and capture on one high-priority stream, like capture_fn
            # (a stateful plan warms up on a throwaway pool of the same shape -- resume_pin is still 0 -- so that the real pool is
            # advanced by the replays only, and is captured against the real pool)
            hp = torch.cuda.Stream(device=dev, priority=-1)
            hp.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(hp):
                issue(None if pool is None else CAFMState(pool.slots, pool.kmax, pool.dim, dev))
            torch.cuda.current_stream().wait_stream(hp)
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with _no_gc_during_capture(), torch.cuda.graph(g, stream=hp):
                issue(pool)
            plan["graph"] = g
        return plan

    @staticmethod
    def _pack_to_host(out, zero_copy_logits=False, fused_row_bytes=None, reuse=None):
        """Device-side compaction of the padded detections (tscd_pack_rows: packed [sum n, 7] + offsets) and the asynchronous D2H
        of tables, counts and status (one pinned buffer each; `reuse` = the dict a previous call returned: its pinned buffers
        are written again -- no host allocation, as required under graph capture)."""
        pk = {}

        def pinned(name, src):
            h = reuse[name] if reuse is not None else torch.empty(src.shape, dtype=src.dtype, pin_memory=True)
            h.copy_(src, non_blocking=True)
            pk[name] = h

        if zero_copy_logits:         # bytes K1 / K3 read in place: survivors' class + regression rows, kept rows again
            pinned("cand_count", out["sel"]["cand"]["count"])
            pk["_logit_row_bytes"] = fused_row_bytes or (out["sel"]["sel_rows"].shape[2] - 7 + 4 + 1) * 2
        for name in ("det", "ori"):
            rows, cnt = out[name + "_rows"], out[name + "_count"]
            nf, cap, _ = rows.shape
            packed = torch.empty(nf * cap, 7, dtype=torch.float32, device=rows.device)
            offsets = torch.empty(nf + 1, dtype=torch.int32, device=rows.device)
            ops.call("tscd_pack_rows", L.PackRowsArgs, num_frames=nf, cap=cap, rows=rows, count=cnt, offsets=offsets, packed=packed)
            pinned(name + "_packed", packed)
            pinned(name + "_offsets", offsets)
        for k in ("det_cand", "status"):
            pinned(k, out[k])
        pinned("sel_count", out["sel"]["sel_count"])
        pk["_row_bytes"] = 3 * out["sel"]["bank_cls"].shape[1] * 2
        return pk

    @staticmethod
    def _unpack_host(pk, nlf):
        """Pinned read-back buffers of one chunk -> the reference's list layout.  The buffers belong to the plan (a graph
        replay overwrites them), so the valid rows are copied out: ONE contiguous clone per output, split into per-frame views
        (fresh tensors, as the callers mutate them in place -- ovis_evaluator_v2.py:268-271)."""
        st = int(pk["status"][0])
        if st != 0:
            raise RuntimeError(f"tscd_b200 stage reported error {st} (capacity exceeded: a frame holds more proposals than "
                               "SelectionConfig.max_proposals)")
        zc_bytes = int(pk["sel_count"].sum()) * pk["_row_bytes"]          # zero-copy reads of the feature rows
        if "cand_count" in pk:
            zc_bytes += (int(pk["cand_count"].sum()) + int(pk["sel_count"].sum())) * pk["_logit_row_bytes"]
        det_c = pk["det_cand"][:nlf].tolist()
        lists, nb = [], 0
        for name in ("det", "ori"):
            off = pk[name + "_offsets"][:nlf + 1].tolist()
            table = torch.from_numpy(pk[name + "_packed"][:off[-1]].numpy().copy())     # single-threaded copy (see forward_host_submit)
            parts = table.split([off[i + 1] - off[i] for i in range(nlf)])
            lists.append([p_ if c else None for p_, c in zip(parts, det_c)])     # post_process.py:54-55: no candidates -> None
            nb += pk[name + "_packed"].numel() * 4 + pk[name + "_offsets"].numel() * 4
        result, result_ori = lists
        nb += sum(pk[k].numel() * pk[k].element_size() for k in ("det_cand", "status", "sel_count"))
        return result, result_ori, nb, zc_bytes

    # ------------------------------------------------------------------------------------------------------
    def capture(self, head: ops.HeadViews, feats, feat_dtype, time_embedding: torch.Tensor, B: int, F: int, Lf: int,
                state: Optional["CAFMState"] = None, resume: Optional[torch.Tensor] = None, warmup: int = 2, state_slots=None):
        """Capture one forward() over FIXED input buffers into a CUDA graph (the stage has no host sync, so the whole
        launch sequence -- ~130 kernels on two streams -- replays from one cudaGraphLaunch).  Returns (graph, out):
        refill the input tensors in place, call graph.replay(), read `out` (same dict forward() returns).
        state_slots: as in forward(); a list is copied to a device tensor once, refill that (out["state_slots"]) to remap."""
        A = head.anchors.num_anchors
        kmax = self.cfg.selection.max_keep(A)
        check_state_args(B, kmax, state, resume, state_slots)
        if state is None:
            state = CAFMState(B, kmax, self.cfg.dim, self.device)
        if resume is None:
            resume = torch.zeros(B, dtype=torch.int32, device=self.device)
        if state_slots is not None and not (isinstance(state_slots, torch.Tensor) and state_slots.is_cuda):
            state_slots = torch.tensor([int(x) for x in state_slots], dtype=torch.int32, device=self.device)
        te = time_embedding.to(self.device)
        s = torch.cuda.Stream(device=self.device)
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):                     # warm-up on a side stream (lazy module loading, attribute setting)
            for _ in range(warmup):
                self.forward(head, feats, feat_dtype, te, B, F, Lf, state=state, resume=resume, state_slots=state_slots)
        torch.cuda.current_stream().wait_stream(s)
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with _no_gc_during_capture(), torch.cuda.graph(graph):
            out = self.forward(head, feats, feat_dtype, te, B, F, Lf, state=state, resume=resume, state_slots=state_slots)
        if state_slots is not None:
            out["state_slots"] = state_slots
        return graph, out

    # ------------------------------------------------------------------------------------------------------
    def capture_fn(self, fn, warmup: int = 2):
        """Capture an arbitrary launch sequence of this stage (e.g. forward_concurrent over fixed input buffers) into a
        CUDA graph.  Returns (graph, value returned by fn during capture)."""
        # warm up and capture on the SAME high-priority stream (lazy per-stream state -- side streams, default CAFM memory --
        # is then created before the capture starts).  High priority: the stage's own side streams (classification branch)
        # have default priority, so whenever both have blocks pending the critical path (agg_iou -> CAFM -> TaskAligned)
        # is scheduled first.
        hp = torch.cuda.Stream(device=self.device, priority=-1)
        hp.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(hp):
            for _ in range(warmup):
                fn()
        torch.cuda.current_stream().wait_stream(hp)
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with _no_gc_during_capture(), torch.cuda.graph(graph, stream=hp):
            out = fn()
        return graph, out

    # ------------------------------------------------------------------------------------------------------
    def forward_from_bank(self, sel, B: int, F: int, Lf: int, kmax: int, time_embedding, state=None, resume=None,
                          trace=None, status=None, before_cafm=None, after_cafm=None, state_slots=None):
        """Everything after K1-K3.  `sel` holds the packed clip bank (bank_cls/reg/edge/score with >= _r128(B*F*kmax)+128
        rows), sel_count [B*F], row_off [B*F+1] and sel_rows [B*F,kmax,7+C] (only local frames' rows are read).
        `before_cafm(state)` / `after_cafm(state)` let a caller hand the CAFM memory from rank to rank.
        state_slots: see forward()."""
        check_state_args(B, kmax, state, resume, state_slots)
        return self._from_bank(sel, B, F, Lf, kmax, time_embedding, state, resume, trace, status, before_cafm, after_cafm,
                               state_slots)

    def _from_bank(self, sel, B, F, Lf, kmax, time_embedding, state, resume, trace=None, status=None, before_cafm=None,
                   after_cafm=None, state_slots=None, cafm_gate=None):
        """forward_from_bank without the argument checks.  cafm_gate: event the CAFM memory accesses wait for (host path)."""
        cfg, w, dev, dt = self.cfg, self.w, self.device, self.cfg.dtype
        C, D = cfg.num_classes, cfg.dim
        if status is None:
            status = torch.zeros(1, dtype=torch.int32, device=dev)
        row_cap = sel["bank_cls"].shape[0]
        assert row_cap >= _r128(B * F * kmax) + 128
        loc_cap = _r128(B * Lf * kmax)
        nk_pitch = _r128(F * kmax)
        bank_cls, bank_reg, bank_edge, bank_score = sel["bank_cls"], sel["bank_reg"], sel["bank_edge"], sel["bank_score"]
        lay = aggregate.make_layout(sel["sel_count"], B, F, Lf, row_cap, loc_cap, nk_pitch, dt, row_off=sel["row_off"])
        n_rows_dev, n_loc_dev = lay.row_off[-1:], lay.lrow_off[-1:]

        # ---- K4: agg_iou (reg / obj refinement, feeds the CAFM recurrence) on the main stream; agg (cls refinement)
        #      + cls_pred on a side stream that starts when the recurrence does: the chain occupies one SM per clip,
        #      the independent classification branch fills the rest of the GPU --------------------------------
        main = torch.cuda.current_stream()
        side = main if self.serialize else self._side_stream()
        # agg_iou's cls output feeds the CAFM matching only.  Frames of <= 32 proposals match on the 16-bit GEMM outputs
        # (tensor-core cost kernel, csrc/cafm.cu cafm_cost16_kernel): no fp32 copy is written at all
        emb16 = kmax <= 32 and trace is None
        (iou_cls16, iou_cls32), (iou_reg16, iou_reg32) = aggregate.mca_forward(
            lay, w.agg_iou, bank_cls, bank_reg, bank_score, n_rows_dev, n_loc_dev, need_reg=True,
            sim_thresh=cfg.sim_thresh, conf_sim_thresh=cfg.conf_sim_thresh, cls_out=(True, not emb16), tag="agg_iou")
        ev_fork = torch.cuda.Event()
        ev_fork.record(main)
        with torch.cuda.stream(side):
            side.wait_event(ev_fork)
            (agg_cls16, agg_cls32), _ = aggregate.mca_forward(lay, w.agg, bank_cls, bank_reg, bank_score, n_rows_dev,
                                                              n_loc_dev, need_reg=False, sim_thresh=cfg.sim_thresh,
                                                              conf_sim_thresh=cfg.conf_sim_thresh,
                                                              cls_out=(True, trace is not None), tag="agg")
            _, cls_logits = ops.linear(agg_cls16, w.cls_w, w.cls_b, m_dev=n_loc_dev, want16=False, want32=True, tag="cls_pred")
            ev_join = torch.cuda.Event()
            ev_join.record(side)
        if not torch.cuda.is_current_stream_capturing():
            for t in (cls_logits, agg_cls32):
                if t is not None:
                    t.record_stream(main)

        # ---- K5: CAFM --------------------------------------------------------------------------------
        # Default memory: one CAFMState per (clips, kmax) owned by the stage object, like the reference keeps its memory on
        # the module (tscd_matching.py:708-715).  With resume = 0 the chain never reads it, so nothing is cleared per call.
        if state is None:
            key = (B, kmax, torch.cuda.current_stream().cuda_stream)     # one per launching stream (concurrent sub-batches)
            if key not in self._default_state:
                self._default_state[key] = CAFMState(B, kmax, D, dev)
            state = self._default_state[key]
        if resume is None:
            if B not in self._zero_resume:
                self._zero_resume[B] = torch.zeros(B, dtype=torch.int32, device=dev)
            resume = self._zero_resume[B]
        elif not isinstance(resume, torch.Tensor):
            resume = torch.tensor([int(x) for x in resume], dtype=torch.int32, device=dev)
        if state_slots is not None and not (isinstance(state_slots, torch.Tensor) and state_slots.is_cuda):
            state_slots = torch.tensor([int(x) for x in state_slots], dtype=torch.int32, device=dev)
        if before_cafm is not None:
            before_cafm(state)
        cafm16, cafm32, perm, te32 = self.run_cafm(lay, bank_reg, bank_edge, iou_reg16 if kmax <= 32 else iou_reg32,
                                                   iou_cls16 if kmax <= 32 else iou_cls32, time_embedding, kmax,
                                                   state, resume, status, want_debug=trace is not None, debug=trace,
                                                   emb16=None if kmax <= 32 else (iou_reg16, iou_cls16),
                                                   state_slots=state_slots, gate=cafm_gate)
        if after_cafm is not None:
            after_cafm(state)
        f32z = lambda *s: torch.empty(*s, dtype=torch.float32, device=dev)  # noqa: E731  (fully written before read)

        # ---- fc_reg_matcher, TaskAligned, prediction heads ---------------------------------------------
        matched16, matched32 = ops.linear(cafm16, w.fc_w, w.fc_b, m_dev=n_loc_dev, want16=True, want32=trace is not None, tag="fc_reg_matcher")
        _, reg_deltas = ops.linear(matched16, w.reg_w, w.reg_b, m_dev=n_loc_dev, want16=False, want32=True, tag="reg_pred")
        # TaskAligned attention on 16-bit q/k/v: frames of <= 32 rows in one mma.sync tile (csrc/tail.cu frame_attention16_kernel),
        # larger frames on the flash kernel (csrc/frame_flash.cu)
        tq, _ = ops.linear(iou_reg16, w.ta_wq, m_dev=n_loc_dev, want16=True, want32=False, tag="ta_q")
        tkv, _ = ops.linear(matched16, w.ta_wkv, m_dev=n_loc_dev, want16=True, want32=False, tag="ta_kv")
        att = f32z(loc_cap, 4 * D)
        if kmax <= 32:
            ops.call("tscd_frame_attention", L.FrameAttentionArgs, num_frames=B * Lf, heads=8, head_dim=(4 * D) // 8,
                     in_dtype=dt, lrow_off=lay.lrow_off, q=tq, ldq=tq.stride(0), k=tkv, ldk=tkv.stride(0),
                     v=tkv[:, 4 * D:], ldv=tkv.stride(0), out=att, ldo=att.stride(0))
        else:
            ops.call("tscd_frame_flash", L.FrameFlashArgs, tag="task_aligned", num_items=B * Lf, heads=8, head_dim=(4 * D) // 8, dtype=dt,
                     max_q=kmax, q_beg=lay.lrow_off, q_end=lay.lrow_off[1:], kv_beg=lay.lrow_off, kv_end=lay.lrow_off[1:],
                     q=tq, ldq=tq.stride(0), k=tkv, ldk=tkv.stride(0), v=tkv[:, 4 * D:], ldv=tkv.stride(0), out=att, ldo=att.stride(0))
        # LN(LN(x + attn)) with the 1-output objectness head (matcher_obj_pred) fused: the LayerNorm output row is in
        # registers, so the refined features are only materialised for tracing
        objref32 = f32z(loc_cap, 4 * D) if trace is not None else None
        obj_logits = f32z(loc_cap, 1)
        ops.call("tscd_residual_ln2", L.ResidualLn2Args, rows_cap=loc_cap, dim=4 * D, n_rows=n_loc_dev, x=iou_reg32, r=att,
                 w_a=w.ta_ln_w, b_a=w.ta_ln_b, w_b=w.ta_dec_w, b_b=w.ta_dec_b, out_dtype=dt, out16=None, out32=objref32,
                 head_w=w.obj_w32, head_b=w.obj_b, head_out=obj_logits)
        main.wait_event(ev_join)                 # classification branch joins here

        # ---- final per-class expansion + NMS ---------------------------------------------------------------
        nlf = B * Lf
        rcap, ocap = kmax * C, kmax
        i32 = lambda *s: torch.empty(*s, dtype=torch.int32, device=dev)  # noqa: E731
        r = dict(box=f32z(nlf, rcap, 4), score=f32z(nlf, rcap), cls=i32(nlf, rcap), obj=f32z(nlf, rcap),
                 cscore=f32z(nlf, rcap), count=i32(nlf))
        o = dict(box=f32z(nlf, ocap, 4), score=f32z(nlf, ocap), cls=i32(nlf, ocap), obj=f32z(nlf, ocap),
                 cscore=f32z(nlf, ocap), count=i32(nlf))
        ops.call("tscd_final_expand", L.FinalExpandArgs, B=B, F=F, L=Lf, num_classes=C, max_keep=kmax,
                 conf_thre=cfg.final_conf_thresh, xform_clip=math.log(736.0 / 32), sel_count=sel["sel_count"],
                 sel_rows=sel["sel_rows"], lrow_off=lay.lrow_off, cls_logits=cls_logits, ld_cls=cls_logits.stride(0),
                 obj_logits=obj_logits, ld_obj=obj_logits.stride(0), reg_deltas=reg_deltas, ld_reg=reg_deltas.stride(0),
                 r_box=r["box"], r_score=r["score"], r_cls=r["cls"], r_obj=r["obj"], r_cscore=r["cscore"], r_count=r["count"],
                 o_box=o["box"], o_score=o["score"], o_cls=o["cls"], o_obj=o["obj"], o_cscore=o["cscore"], o_count=o["count"])
        out = {}
        for name, c, cap in (("det", r, rcap), ("ori", o, ocap)):
            keep, kc, _ = ops.nms(c["box"], c["score"], c["cls"], c["count"], cfg.final_nms_thresh, max_keep=cap, status=status,
                                  tag="final_" + name, wide=_selection.is_wide(cfg.selection.max_proposals))
            rows = f32z(nlf, cap, 7)
            ops.call("tscd_final_rows", L.FinalRowsArgs, num_frames=nlf, cand_cap=cap, keep_cap=cap, box=c["box"],
                     obj=c["obj"], cscore=c["cscore"], cls=c["cls"], keep=keep, keep_count=kc, rows=rows)
            out[name + "_rows"], out[name + "_count"], out[name + "_cand"] = rows, kc, c["count"]
        out.update(status=status, sel=sel, layout=lay, state=state)
        if trace is not None:
            trace.update(agg_cls=agg_cls32, iou_cls=iou_cls32, iou_reg=iou_reg32, cafm=cafm32, perm=perm, matched=matched32,
                         obj_ref=objref32, cls_logits=cls_logits, obj_logits=obj_logits, reg_deltas=reg_deltas,
                         time_emb=te32, att=att)
        return out

    # ------------------------------------------------------------------------------------------------------
    def run_cafm(self, lay: ops.AttnLayoutT, bank_reg, bank_edge, emb_reg32, emb_cls32, time_embedding, kmax: int,
                 state: CAFMState, resume: torch.Tensor, status: torch.Tensor, want_debug=False, debug: Optional[dict] = None,
                 emb16=None, state_slots: Optional[torch.Tensor] = None, gate=None):
        """CAFM (AwarePositionRegMatcher.forward, tscd_matching.py:722-888) for all clips of the batch.
        state_slots ([B] int32 device tensor, optional): clip b uses slot state_slots[b] of `state` (kernel-side slot map).
        gate (optional event): the current stream waits for it right before the first kernel that touches `state`.
        emb16 (wide frames): 16-bit copies of the fp32 matching embeddings -> tensor-core cost kernel.
        emb_reg32 / emb_cls32 [loc_cap,1024] are the agg_iou outputs used for matching only: fp32, or -- frames of <= 32
        proposals -- the 16-bit GEMM outputs (fp32 tensors are rounded to the operand type then)."""
        w, dev, dt, D = self.w, self.device, self.cfg.dtype, self.cfg.dim
        if kmax <= 32 and emb_reg32.dtype == torch.float32:
            emb_reg32, emb_cls32 = emb_reg32.to(dt), emb_cls32.to(dt)
        emb_dtype = emb_reg32.dtype
        assert emb_cls32.dtype == emb_dtype and (emb_dtype == torch.float32 or kmax <= 32)
        B, F, Lf, loc_cap = lay.B, lay.F, lay.L, lay.loc_cap
        n_loc_dev = lay.lrow_off[-1:]
        te16 = time_embedding.to(device=dev, dtype=dt).contiguous()
        assert te16.shape == (B * Lf, 256)
        assert (state.slots == B if state_slots is None else state.slots >= B) and state.kmax == kmax
        _, te32 = ops.linear(te16, w.ape_w, w.ape_b, want16=False, want32=True, tag="time_emb")
        f32z = lambda *s: torch.empty(*s, dtype=torch.float32, device=dev)  # noqa: E731  (fully written before read)
        fast = kmax <= 32            # every frame's working set fits the shared-memory / mma.sync chain (csrc/cafm.cu)
        feat = edge = kin = None
        if not fast:
            feat, edge, kin = f32z(loc_cap, D), f32z(loc_cap, D), f32z(loc_cap, D)
        feat16 = torch.empty(loc_cap, D, dtype=dt, device=dev)
        kin16 = torch.empty(loc_cap, D, dtype=dt, device=dev)
        norm_reg, norm_cls = f32z(loc_cap), f32z(loc_cap)
        ops.call("tscd_cafm_prep", L.CafmPrepArgs, B=B, F=F, L=Lf, D=D, bank_dtype=dt, row_off=lay.row_off,
                 lrow_off=lay.lrow_off, bank_reg=bank_reg, bank_edge=bank_edge, time_emb=te32, se_w1=w.se_w1,
                 se_w2=w.se_w2, emb_reg=emb_reg32, emb_cls=emb_cls32, feat=feat, edge=edge, feat16=feat16,
                 kin16=kin16, kin=kin, norm_reg=norm_reg, norm_cls=norm_cls, emb_dtype=emb_dtype)
        kproj16, kproj = ops.linear(kin16, w.cafm_wk, m_dev=n_loc_dev, want16=True, want32=False, tag="cafm_k")
        vproj16, vproj = ops.linear(feat16, w.cafm_wv, m_dev=n_loc_dev, want16=True, want32=False, tag="cafm_v")
        cafm16 = torch.empty(loc_cap, D, dtype=dt, device=dev)
        cafm32 = f32z(loc_cap, D) if want_debug else None
        perm = torch.empty(loc_cap, dtype=torch.int32, device=dev) if want_debug else None
        cost_full = f32z(B * Lf, kmax, kmax)
        ref_n = torch.empty(B * Lf, dtype=torch.int32, device=dev)
        if gate is not None:
            torch.cuda.current_stream().wait_event(gate)
        ops.call("tscd_cafm_cost", L.CafmCostArgs, slot=state_slots, B=B, L=Lf, D=D, kmax=kmax, lrow_off=lay.lrow_off, resume=resume,
                 st_n=state.n, emb_reg=emb_reg32, emb_cls=emb_cls32, norm_reg=norm_reg, norm_cls=norm_cls,
                 st_reg=state.reg, st_cls=state.cls, st_nreg=state.nreg, st_ncls=state.ncls, cost=cost_full, ref_n=ref_n,
                 emb_dtype=emb_dtype, emb_reg16=None if emb16 is None else emb16[0], emb_cls16=None if emb16 is None else emb16[1],
                 emb16_dtype=dt)
        lap_col = torch.empty(B * Lf, kmax, dtype=torch.int32, device=dev)
        lap_row = torch.empty(B * Lf, kmax, dtype=torch.int32, device=dev)
        ops.call("tscd_cafm_lap", L.CafmLapArgs, num_frames=B * Lf, kmax=kmax, lrow_off=lay.lrow_off, ref_n=ref_n, cost=cost_full,
                 lap_col=lap_col, lap_row=lap_row)
        chain_kw = dict(B=B, F=F, L=Lf, D=D, kmax=kmax, out_dtype=dt, row_off=lay.row_off,
                        lrow_off=lay.lrow_off, resume=resume, feat=feat, edge=edge, kin=kin, kproj=None, vproj=None,
                        kproj16=kproj16 if fast else None, vproj16=vproj16 if fast else None, wq16=w.cafm_wq16 if fast else None,
                        bank_reg=bank_reg if fast else None, bank_edge=bank_edge if fast else None, time_emb=te32, emb_reg=emb_reg32,
                        emb_cls=emb_cls32, norm_reg=norm_reg, norm_cls=norm_cls,
                        wq_t=None, se_w1=w.se_w1, se_w2=w.se_w2, ln_w=w.cafm_ln_w, ln_b=w.cafm_ln_b,
                        dec_w=w.cafm_dec_w, dec_b=w.cafm_dec_b, st_n=state.n, st_out=state.out, st_edge=state.edge,
                        st_reg=state.reg, st_cls=state.cls, st_nreg=state.nreg, st_ncls=state.ncls, st_time=state.time,
                        sc_qin=None, sc_q=None, sc_k=None, ref_n=ref_n, lap_col=lap_col, lap_row=lap_row,
                        out16=cafm16, out32=cafm32, perm=perm, status=status, emb_dtype=emb_dtype, slot=state_slots)
        if fast:
            ops.call("tscd_cafm_chain", L.CafmChainArgs, **chain_kw)
        else:
            self._cafm_wide(chain_kw, kproj16, vproj16, B, Lf, kmax, D)
        if debug is not None:        # matching tables of every local frame (tests: LSAP exactness on the device's own costs)
            debug.update(cafm_cost=cost_full, cafm_ref_n=ref_n, cafm_lap_col=lap_col, cafm_lap_row=lap_row)
        return cafm16, cafm32, perm, te32

    # ------------------------------------------------------------------------------------------------------
    def _cafm_wide(self, chain_kw, kproj16, vproj16, B: int, Lf: int, kmax: int, D: int):
        """CAFM recurrence for frames of more than 32 proposals (mode B: 50..500 per frame): per local frame a short sequence
        of batch-wide launches over all clips -- permutation + SE-gated query rows, q projection on the tcgen05 GEMM, the
        n x n cosine attention on the mma.sync flash kernel, LayerNorms + state update (csrc/cafm.cu "wide chain")."""
        import ctypes as C
        w, dev, dt = self.w, self.device, self.cfg.dtype
        base = L.CafmChainArgs()
        for k_, v_ in chain_kw.items():
            if isinstance(v_, torch.Tensor) or v_ is None:
                v_ = ops._p(v_)
            elif isinstance(v_, torch.dtype):
                v_ = ops._DT[v_]
            setattr(base, k_, v_)
        rows = _r128(B * kmax)
        i32 = lambda *s_: torch.empty(*s_, dtype=torch.int32, device=dev)  # noqa: E731
        qin16 = torch.empty(rows, D, dtype=dt, device=dev)
        attn = torch.empty(rows, D, dtype=torch.float32, device=dev)
        rng = [i32(B) for _ in range(4)]
        scratch = dict(ctl=i32(B, 8), perm_s=i32(B, kmax), prow_s=i32(B, kmax), ord_prev=i32(B, kmax), n_prev=i32(B), last_l0=i32(B))
        wa = L.CafmWideArgs()
        wa.base = base
        wa.qin16, wa.attn = ops._p(qin16), ops._p(attn)
        wa.q_beg, wa.q_end, wa.kv_beg, wa.kv_end = (ops._p(t) for t in rng)
        for k_, v_ in scratch.items():
            setattr(wa, k_, ops._p(v_))

        def phase(p_, f_):
            with L.timed("tscd_cafm_wide", f"phase{p_}"):
                L.check(L.lib().tscd_cafm_wide(C.byref(wa), p_, f_, ops._stream()), "tscd_cafm_wide_p1" if p_ == 1 else "tscd_cafm_wide")

        phase(0, 0)
        for f in range(Lf):
            phase(1, f)
            q16, _ = ops.linear(qin16, w.cafm_wq16, want16=True, want32=False, tag="cafm_q")
            ops.call("tscd_frame_flash", L.FrameFlashArgs, tag="cafm", num_items=B, heads=8, head_dim=D // 8, dtype=dt, max_q=kmax,
                     q_beg=rng[0], q_end=rng[1], kv_beg=rng[2], kv_end=rng[3], q=q16, ldq=q16.stride(0), k=kproj16,
                     ldk=kproj16.stride(0), v=vproj16, ldv=vproj16.stride(0), out=attn, ldo=attn.stride(0))
            phase(2, f)
        phase(3, 0)

    # ------------------------------------------------------------------------------------------------------
    @staticmethod
    def to_lists(out, B: int, Lf: int):
        """One device->host read; returns (result, result_ori) with the reference's container types
        (post_process.py:12-13,85): per local frame a fresh Tensor[n,7] or None."""
        st = int(out["status"].item())
        if st == L.TSCD_ERR_FRAME_SLOT:
            raise RuntimeError(f"tscd_b200 stage reported error {st} (a clip references a frame-store slot that was never written "
                               "or lies outside the FrameStore: ingest_frames every frame of the clips before forward_clips)")
        if st != 0:
            raise RuntimeError(f"tscd_b200 stage reported error {st} (capacity exceeded: a frame holds more proposals than "
                               f"the per-frame capacity of {out['sel']['sel_rows'].shape[1]} -- raise SelectionConfig.max_proposals "
                               f"(<= {_selection.MAX_PROPOSALS}) or set maximal_limit)")
        det_n, ori_n = out["det_count"].cpu().tolist(), out["ori_count"].cpu().tolist()
        det_c = out["det_cand"].cpu().tolist()
        result, result_ori = [], []
        for i in range(B * Lf):
            if det_c[i] == 0:                      # post_process.py:54-55: `continue` skips both outputs
                result.append(None)
                result_ori.append(None)
                continue
            result.append(out["det_rows"][i, :det_n[i]].clone())
            result_ori.append(out["ori_rows"][i, :ori_n[i]].clone())
        return result, result_ori
