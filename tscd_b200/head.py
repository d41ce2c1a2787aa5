"""Drop-in head for the reference's own tools: `TSCDHeadB200` keeps TSCDHead's constructor, parameter names
(strict `load_state_dict` of reference checkpoints works, SURVEY App. B) and forward signature / return types,
reuses the reference's conv towers unchanged (PyTorch/cuDNN, out of scope) and replaces ONLY the inference
tail (yolox/models/tscd_head.py:374-733) by the sm_100a kernels of this package.

The reference package (`yolox`) is not vendored: the class is created on demand by `make_head_class()` when
`yolox.models.tscd_head.TSCDHead` is importable (i.e. inside a reference checkout), see INTEGRATION.md.
Training mode and configurations the kernels do not cover raise loudly; there is no silent fallback."""
from typing import List

import torch

from . import ops
from .selection import DEFAULT_TIER_MAX, MAX_PROPOSALS, SelectionConfig
from .stage import MAX_KEYS_PER_CLIP, AggregationStage, CAFMState, StageConfig, validate_config
from .weights import timing_signal_1d  # noqa: F401  (re-exported for callers that build time embeddings)

_CONV_PREFIXES = ("stems", "cls_convs", "reg_convs", "edge_enhance", "cls_preds", "reg_preds", "obj_preds")


def stage_config_from_head(head) -> StageConfig:
    """Translate TSCDHead's ctor arguments / kwargs (SURVEY section 8b) into a StageConfig; reject what is unsupported."""
    kw = head.kwargs
    if kw.get("agg_type", "localagg") != "mca" or not kw.get("decouple_reg", False) or not kw.get("reconf", False) \
            or not kw.get("ota_mode", False):
        raise RuntimeError("TSCDHeadB200 supports the TSCD configuration only: agg_type='mca', decouple_reg, reconf, ota_mode")
    if kw.get("local_mask", False) or head.use_mask or not head.ave:
        raise RuntimeError("TSCDHeadB200: local_mask / use_mask / ave=False are not implemented (not used by the TSCD exps)")
    # max_proposals: per-frame capacity of the proposal list.  The reference's list is unbounded when no maximal_limit is set
    # (VID TSCD-L, exps/TSCD_VID/vid_tscd_large.py:39-42); the default tier holds at most 512 (fewer when 512 x classes would
    # exceed the final NMS's 16384 candidate rows), and forward() reruns a call that overflows it on the wide tier
    # (wide_capacity).  kwargs['max_proposals'] overrides the default and turns that escalation off: overflow then raises.
    cap = min(DEFAULT_TIER_MAX, ops.NMS_MAX_CAP // max(1, head.num_classes))
    sel = SelectionConfig(mode="B", nms_thresh=head.nms_thresh, conf_thresh=0.001,
                          minimal_limit=kw.get("minimal_limit", 0), maximal_limit=kw.get("maximal_limit", 0),
                          use_pre_nms=kw.get("use_pre_nms", True), max_proposals=int(kw.get("max_proposals", cap)))
    cfg = StageConfig(num_classes=head.num_classes, selection=sel, dim=head.width, heads=4, sim_thresh=head.sim_thresh,
                      conf_sim_thresh=kw.get("conf_sim_thresh", 0.99))
    validate_config(cfg)             # capacity problems surface when the head is built, not at the first forward
    return cfg


def wide_capacity(num_frames: int, num_classes: int) -> int:
    """Per-frame capacity of the wide tier for clips of `num_frames` frames: the attention kernels hold 65536 keys per clip and
    the final NMS 65536 candidate rows (proposals x classes) per frame."""
    return min(MAX_PROPOSALS, MAX_KEYS_PER_CLIP // max(1, num_frames), ops.NMS_WIDE_CAP // max(1, num_classes))


def make_head_class():
    """Returns class TSCDHeadB200(TSCDHead).  Requires the reference's `yolox` package on sys.path."""
    from yolox.models.tscd_head import TSCDHead  # reference checkout

    class TSCDHeadB200(TSCDHead):
        def __init__(self, *args, **kwargs):
            super().__init__(*args, **kwargs)
            self._b200_stage = None
            self._b200_state = None
            self._b200_key = None
            self._b200_wide = {}              # wide-tier stages by capacity (built on the first overflow)
            self._b200_on_wide = False        # this video's resume=True calls stay on the wide tier
            stage_config_from_head(self)      # reject unsupported / over-capacity configurations at construction
            # model.load_state_dict(ckpt) recurses through _load_from_state_dict and never calls a child's load_state_dict:
            # the post-hook fires for this module either way
            self.register_load_state_dict_post_hook(lambda module, incompatible: module._b200_invalidate())

        def _b200_invalidate(self):
            self._b200_stage = None           # weights changed / moved: rebuild the 16-bit device copies lazily
            self._b200_state = None
            self._b200_edge = None
            self._b200_wide = {}
            self._b200_on_wide = False

        def _apply(self, fn, *a, **k):        # .half() / .to() / .cuda() / .float()
            self._b200_invalidate()
            return super()._apply(fn, *a, **k)

        def _stage(self):
            # the snapshot is keyed on the parameters' identity and in-place version counters, so optimiser steps or manual
            # edits of the weights are picked up as well
            params = [p for n, p in self.named_parameters() if not n.startswith(_CONV_PREFIXES)]
            key = (params[0].device, tuple((p.data_ptr(), p._version) for p in params))
            if self._b200_stage is None or self._b200_key != key:
                sd = {k: v for k, v in self.state_dict().items() if not k.startswith(_CONV_PREFIXES)}
                self._b200_stage = AggregationStage(stage_config_from_head(self), sd, device=params[0].device)
                self._b200_key = key
                self._b200_state = None
                self._b200_wide = {}
                self._b200_on_wide = False
            return self._b200_stage

        def _wide_stage(self, cap):
            """Stage of the wide tier (same weights as _stage(), per-frame capacity `cap`)."""
            if cap not in self._b200_wide:
                st = self._b200_stage
                cfg = stage_config_from_head(self)
                cfg.selection.max_proposals = cap
                validate_config(cfg)
                sd = {k: v for k, v in self.state_dict().items() if not k.startswith(_CONV_PREFIXES)}
                self._b200_wide[cap] = AggregationStage(cfg, sd, device=st.device)
            return self._b200_wide[cap]

        def _edge_block(self, dtype):
            """16-bit copies of the per-level WaveletsHFBlock weights for the selected-anchor evaluation (ops.EdgeBlock)."""
            params = list(self.edge_enhance_reg.parameters())
            key = (params[0].device, dtype, tuple((p.data_ptr(), p._version) for p in params))
            if getattr(self, "_b200_edge", None) is None or self._b200_edge[0] != key:
                self._b200_edge = (key, ops.EdgeBlock.from_modules(self.edge_enhance_reg, dtype=dtype, device=params[0].device))
            return self._b200_edge[1]

        def forward(self, xin, labels=None, imgs=None, time_embedding=None, nms_thresh=0.5, lframe=0, gframe=32,
                    resume=False):
            if self.training:
                raise RuntimeError("TSCDHeadB200 is inference-only (the training branches are out of scope)")
            if imgs.shape[0] == 1:
                return super().forward(xin, labels, imgs, time_embedding, nms_thresh, lframe, gframe, resume)
            # ---- conv towers: the reference's own modules, channels_last so an anchor's 256 channels are contiguous ----
            # kwargs['b200_pred_gemm'] (fp16 only): the 1x1 prediction convs run as tcgen05 GEMMs that write the fused layout
            # directly (ops.pred_heads) instead of cuDNN convs + tscd_pack_head; logits then differ from cuDNN's in the last bits
            pred_gemm = bool(self.kwargs.get("b200_pred_gemm", False)) and xin[0].dtype == torch.float16 and self.num_classes <= 59
            # SURVEY 8f-2: the wavelet edge block (edge_enhance_reg, tscd_head.py:367) is evaluated at the kept proposals only
            # (csrc/edge.cu) instead of densely over every level; kwargs['b200_dense_edge'] keeps the reference's dense modules
            dense_edge = bool(self.kwargs.get("b200_dense_edge", False))
            reg_o, obj_o, cls_o, f_cls, f_reg, f_edge, reg_f, cls_f = [], [], [], [], [], [], [], []
            for k, x in enumerate(xin):
                x = self.stems[k](x.contiguous(memory_format=torch.channels_last))
                reg_feat, cls_feat = self.reg_convs[k](x), self.cls_convs[k](x)
                vid_cls = self.cls_convs2[k](x) if self.kwargs.get("vid_cls", True) else cls_feat
                vid_reg = self.reg_convs2[k](x) if self.kwargs.get("vid_reg", True) else reg_feat
                if pred_gemm:
                    reg_f.append(reg_feat.contiguous(memory_format=torch.channels_last))
                    cls_f.append(cls_feat.contiguous(memory_format=torch.channels_last))
                else:
                    reg_o.append(self.reg_preds[k](reg_feat)); obj_o.append(self.obj_preds[k](reg_feat))
                    cls_o.append(self.cls_preds[k](cls_feat))
                f_cls.append(vid_cls); f_reg.append(vid_reg)
                if dense_edge:
                    f_edge.append(self.edge_enhance_reg[k](vid_reg))
            hw = [tuple(t.shape[-2:]) for t in f_cls]
            an = ops.AnchorSpec(hw, tuple(self.strides))
            if pred_gemm:
                wro = [torch.cat([self.reg_preds[k].weight, self.obj_preds[k].weight], 0).flatten(1).contiguous() for k in range(len(xin))]
                bro = [torch.cat([self.reg_preds[k].bias, self.obj_preds[k].bias], 0).float().contiguous() for k in range(len(xin))]
                wc = [self.cls_preds[k].weight.flatten(1).contiguous() for k in range(len(xin))]
                bc = [self.cls_preds[k].bias.float().contiguous() for k in range(len(xin))]
                head = ops.pred_heads(reg_f, cls_f, wro, bro, wc, bc, an, self.num_classes)
            else:
                head = ops.HeadViews.from_levels(reg_o, obj_o, cls_o, an)
            if not pred_gemm and reg_o[0].dtype == torch.float16 and self.num_classes <= 59:
                # conv-tower seam (SURVEY 8f-2): instead of the reference's flatten / cat / permute copies into [F, A, 5+C]
                # (tscd_head.py:374-376), ONE pass writes the fused layout -- a 64 / 128-byte row [reg4|obj|cls C] per anchor
                # plus the dense objectness plane -- that the row kernels of K1 / K3 consume (csrc/select_rows.cu); sigmoid
                # and decode stay fused in those kernels, values are copied bit for bit
                head = ops.pack_head(head)
            st = self._stage()
            feats = (ops.view_levels(f_cls), ops.view_levels(f_reg),
                     ops.view_levels(f_edge) if dense_edge else self._edge_block(st.cfg.dtype))
            F = imgs.shape[0]
            # Tiers: a call runs on the default tier (<= 512 proposals per frame) unless the video is already on the wide tier.
            # A default-tier call whose frames overflow is rerun on the wide tier from the CAFM memory it started with (the
            # overflowing run may have written the memory), and the video's following resume=True calls stay there; the next
            # resume=False call starts again on the default tier.  An explicit kwargs['max_proposals'] never escalates.
            wide_cap = wide_capacity(F, self.num_classes)
            can_widen = "max_proposals" not in self.kwargs and self.kwargs.get("maximal_limit", 0) == 0 \
                and wide_cap > st.cfg.selection.max_proposals
            if not resume:
                self._b200_on_wide = False
            on_wide = self._b200_on_wide and can_widen
            run = self._wide_stage(wide_cap) if on_wide else st
            run.cfg.final_nms_thresh = nms_thresh
            kmax = run.cfg.selection.max_keep(an.num_anchors)
            if self._b200_state is not None and resume and self._b200_state.kmax < kmax:
                self._b200_state = self._b200_state.widened(kmax)
            elif self._b200_state is None or self._b200_state.kmax != kmax:
                self._b200_state = CAFMState(1, kmax, st.cfg.dim, imgs.device)
            res = torch.tensor([int(bool(resume))], dtype=torch.int32, device=imgs.device)
            te = time_embedding[:lframe].float()
            snapshot = self._b200_state.flat.clone() if (resume and can_widen and not on_wide) else None
            out = run.forward(head, feats, f_cls[0].dtype, te, 1, F, lframe, state=self._b200_state, resume=res)
            if can_widen and not on_wide and int(out["status"].item()) != 0:
                if snapshot is not None:
                    self._b200_state.flat.copy_(snapshot)
                run = self._wide_stage(wide_cap)
                run.cfg.final_nms_thresh = nms_thresh
                self._b200_state = self._b200_state.widened(run.cfg.selection.max_keep(an.num_anchors))
                self._b200_on_wide = True
                out = run.forward(head, feats, f_cls[0].dtype, te, 1, F, lframe, state=self._b200_state, resume=res)
            result, result_ori = run.to_lists(out, 1, lframe)
            if int(out["sel"]["sel_count"].sum().item()) == 0:
                # no proposal in any frame: the reference returns its F-length pred_result twice (tscd_head.py:439-440)
                return [None] * F, [None] * F
            dt = xin[0].dtype
            return ([None if r is None else r.to(dt) for r in result], [None if r is None else r.to(dt) for r in result_ori])

    return TSCDHeadB200
