"""Proposal selection + bank gather (K1-K3) as one host-side call, sync-free.

Mirrors TSCDHead.postprocess_widx / postpro_woclass + find_feature_score (tscd_head.py:1546-1693,
post_process.py:464-521, tscd_head.py:976-1006) but for a whole batch of frames at once and with all
data-dependent sizes left on the device."""
from dataclasses import dataclass
from typing import Optional

import torch

from . import ops

DEFAULT_TIER_MAX = 512     # max_proposals up to here: the default tier (csrc/cafm.cu kChainMax; 16384-row final NMS)
MAX_PROPOSALS = 2048       # wide tier limit (include/tscd_b200.h TSCD_MAX_PROPOSALS)


def is_wide(max_proposals: int) -> bool:
    """Wide tier: more than DEFAULT_TIER_MAX proposals per frame (CTA LSAP, global-memory final-NMS merge)."""
    return max_proposals > DEFAULT_TIER_MAX


@dataclass
class SelectionConfig:
    mode: str = "B"                 # "A" = postpro_woclass (top-P objectness -> NMS -> first K); "B" = postprocess_widx
    pre_k: int = 750                # mode A: P   (Prenum)
    top_k: int = 30                 # mode A: K   (Afternum)
    nms_thresh: float = 0.75        # pre-NMS IoU threshold (TSCDHead pre_nms)
    conf_thresh: float = 0.001      # mode B
    minimal_limit: int = 0          # mode B
    maximal_limit: int = 0          # mode B
    use_pre_nms: bool = True        # mode B (False in both shipped -L exps)
    # Mode B without a maximal_limit (VID TSCD-L, exps/TSCD_VID/vid_tscd_large.py:39-42) keeps EVERY anchor at or above
    # conf_thresh: the reference's per-frame list is unbounded (up to all A = 6804 anchors), the kernels' buffers are not.
    # max_proposals is the explicit per-frame capacity of the proposal list (bank pitch, CAFM state / cost tables);
    # a frame that would keep more sets the stage's status flag and forward raises -- never a silent truncation.
    # up to 512: the default tier; 513 .. MAX_PROPOSALS (2048): the wide tier (stage.validate_config states its limits)
    max_proposals: int = 512

    def validate(self, chain_capacity: int = MAX_PROPOSALS):
        if self.mode not in ("A", "B"):
            raise RuntimeError(f"selection mode {self.mode!r}: expected 'A' (postpro_woclass) or 'B' (postprocess_widx)")
        if not 1 <= self.max_proposals <= chain_capacity:
            raise RuntimeError(f"max_proposals = {self.max_proposals}: the CAFM chain holds at most {chain_capacity} proposals per frame")
        if self.mode == "A":
            if self.top_k > self.max_proposals:
                raise RuntimeError(f"top_k = {self.top_k} exceeds max_proposals = {self.max_proposals}")
            if self.pre_k > 8192:
                raise RuntimeError(f"pre_k = {self.pre_k}: the selection kernel sorts at most 8192 survivors per frame")
        else:
            if max(self.maximal_limit, self.minimal_limit) > self.max_proposals:
                raise RuntimeError(f"minimal_limit / maximal_limit = {self.minimal_limit} / {self.maximal_limit} exceed "
                                   f"max_proposals = {self.max_proposals} (per-frame capacity of the aggregation kernels)")

    def max_keep(self, num_anchors: int) -> int:
        """Per-frame capacity of the kept-proposal list (pitch of sel_rows / sel_idx, CAFM kmax)."""
        if self.mode == "A":
            return min(self.top_k, self.pre_k, num_anchors)
        cap = self.maximal_limit if self.maximal_limit else num_anchors
        if self.minimal_limit:
            cap = max(cap, min(self.minimal_limit, num_anchors))
        return min(cap, self.max_proposals)

    def cand_cap(self, num_anchors: int) -> int:
        """Per-frame capacity of the candidate list K1 emits (input of the pre-NMS when there is one)."""
        if self.mode == "A":
            return min(self.pre_k, num_anchors)
        if not self.use_pre_nms:
            return self.max_keep(num_anchors)          # the candidates ARE the proposals
        cap = self.maximal_limit if self.maximal_limit else num_anchors
        if self.minimal_limit:
            cap = max(cap, min(self.minimal_limit, num_anchors))
        return cap


def select_and_gather(head: ops.HeadViews, feats, feat_dtype, feat_dim, cfg: SelectionConfig,
                      bank_dtype=torch.float16, status: Optional[torch.Tensor] = None, bank_rows: Optional[int] = None):
    """Runs K1 (+K2) + K3.  Returns the dict of ops.gather plus the candidate dict under 'cand'."""
    picked = select_candidates(head, cfg, status)
    return gather_bank(head, feats, feat_dtype, feat_dim, cfg, picked, bank_dtype=bank_dtype, bank_rows=bank_rows)


def select_candidates(head: ops.HeadViews, cfg: SelectionConfig, status: Optional[torch.Tensor] = None):
    """K1 (+K2): candidate lists and, where the configuration has a pre-NMS, the kept positions.  Returns (cand, keep, keep_count,
    status, max_keep) for gather_bank (forward_host runs the two halves on different lanes)."""
    A = head.anchors.num_anchors
    if status is None:
        status = torch.zeros(1, dtype=torch.int32, device=ops._dev(head))
    cand_cap = cfg.cand_cap(A)
    if cand_cap > ops.NMS_MAX_CAP:
        raise RuntimeError(f"mode B pre-NMS over {cand_cap} candidates per frame exceeds the NMS capacity of {ops.NMS_MAX_CAP}; "
                           "set maximal_limit or use_pre_nms=False")
    max_keep = cfg.max_keep(A)
    # mode A over the fused-row layout: K1 skips its objectness sort (K2 orders by score anyway; the objectness order only
    # breaks score ties and travels as a rank key) whenever K2 runs its top-K kernel
    unsorted = cfg.mode == "A" and head.fused and head.num_frames > 0 and 64 < cand_cap <= ops.NMS_SMEM_CAP and 4 * max_keep < cand_cap \
        and min(cfg.pre_k, A) <= cand_cap and A <= 65535
    cand = ops.select(head, cfg.mode, pre_k=cfg.pre_k, conf_thresh=cfg.conf_thresh,
                      minimal_limit=cfg.minimal_limit, maximal_limit=cfg.maximal_limit, cand_cap=cand_cap, status=status,
                      unsorted=unsorted)
    keep = keep_count = None
    if cfg.mode == "A" or cfg.use_pre_nms:
        # mode A: the first top_k survivors ARE the semantics; mode B: max_keep is a buffer capacity, overflow is an error
        keep, keep_count, status = ops.nms(cand["box"], cand["score"], cand["cls"], cand["count"], cfg.nms_thresh,
                                           max_keep=max_keep, status=status, strict_keep=cfg.mode == "B", tag="pre",
                                           rank=cand.get("rank"))
    return cand, keep, keep_count, status, max_keep


def gather_bank(head: ops.HeadViews, feats, feat_dtype, feat_dim, cfg: SelectionConfig, picked, bank_dtype=torch.float16,
                bank_rows: Optional[int] = None):
    """K3 (+ the selected-anchor edge block) on the output of select_candidates."""
    cand, keep, keep_count, status, max_keep = picked
    out = ops.gather(head, feats, feat_dtype, feat_dim, cand, keep, keep_count, max_keep=max_keep,
                     bank_dtype=bank_dtype, bank_rows=bank_rows)
    if isinstance(feats[2], ops.EdgeBlock):
        # SURVEY 8f-2: the wavelet edge block is evaluated at the kept proposals only (the dense maps are never built)
        ops.edge_rows(feats[2], feats[1], feat_dtype, head.anchors, out, head.num_frames, status=status)
    out["cand"] = cand
    out["status"] = status
    return out


def to_lists(sel):
    """Host-side view in the reference's container types: (rows list F x [n,7+C] or None, idx list F x int64[n]).
    This is the only place that synchronises."""
    counts = sel["sel_count"].cpu().tolist()
    rows, idxs = [], []
    for f, n in enumerate(counts):
        if n == 0:
            rows.append(None)
            idxs.append(None)
        else:
            rows.append(sel["sel_rows"][f, :n].clone())
            idxs.append(sel["sel_idx"][f, :n].to(torch.int64))
    return rows, idxs
