"""Host orchestration of the MCA (global->local cross-attention) aggregation modules.

Reference: MCA_tscd_g2l_reg.forward (post_trans.py:1127-1162) + Attention_mca_g2l.forward (:601-714), used
twice by TSCDHead (`agg`, `agg_iou`; tscd_head.py:104,113,480,491).  Differences in *how*, not *what*:
the q/kv projections of both modules run as one GEMM per branch over the whole bank (the reference
re-projects the global bank once per local frame and module), and the per-local-frame loop is one masked
attention launch."""
from typing import Dict, Optional

import torch

import os

# attn_pv statistics with BF16 operands: single pass with this upper bound of the logits (scale 25 x cosine <= 1 x class score <= 1)
# instead of a first pass for the row maxima (include/tscd_b200.h tscd_attn_pv_args.max_logit; fp16 operands always run two passes:
# an online softmax with a per-tile exchange of the row maxima between the four column-quarter warps was measured SLOWER, 174 vs 113 us)
SINGLE_PASS_MAX_LOGIT = float(os.environ.get("TSCD_ATTN_MAX_LOGIT", "25.0"))

from . import ops

# q|k|v projections with the normalise / scale / transpose step fused into the GEMM epilogue (tscd_qkv_project) instead of
# tscd_linear + tscd_attn_prep; the unfused pair is kept for the MSA path and as a cross-check
FUSED_QKV = True


class MCAWeights:
    """16-bit device copies of one module's weights, q/kv fused as [Wq; Wkv] per branch."""

    def __init__(self, sd: Dict[str, torch.Tensor], prefix: str, dtype=torch.float16, device="cuda"):
        def w(name):
            return sd[prefix + name].detach().to(device=device, dtype=dtype).contiguous()

        def b(name):
            return sd[prefix + name].detach().to(device=device, dtype=torch.float32).contiguous()

        self.qkv_cls = torch.cat([w("mca.q_cls_local.weight"), w("mca.kv_cls.weight")], 0).contiguous()   # [768,256]
        self.qkv_reg = torch.cat([w("mca.q_reg_local.weight"), w("mca.kv_reg.weight")], 0).contiguous()
        self.lin_w, self.lin_b = w("mca.linear.weight"), b("mca.linear.bias")
        self.has_reg = (prefix + "mca.linear_reg.weight") in sd
        if self.has_reg:
            self.linreg_w, self.linreg_b = w("mca.linear_reg.weight"), b("mca.linear_reg.bias")
            self.obj_w, self.obj_b = w("linear_obj.weight"), b("linear_obj.bias")
        self.out_w, self.out_b = w("linear.weight"), b("linear.bias")


def make_layout(sel_count: torch.Tensor, B: int, F: int, L: int, row_cap: int, loc_cap: int, nk_pitch: int,
                dtype=torch.float16, row_off: Optional[torch.Tensor] = None) -> ops.AttnLayoutT:
    """Device-side prefix offsets from per-frame counts (torch ops on the current stream; no sync)."""
    if row_off is None:
        cnt = sel_count.view(B, F).to(torch.int32)
        row_off = torch.zeros(B * F + 1, dtype=torch.int32, device=sel_count.device)
        row_off[1:] = torch.cumsum(cnt.reshape(-1), 0)
    lrow_off = torch.empty(B * L + 1, dtype=torch.int32, device=sel_count.device)
    assert sel_count.dtype == torch.int32 and sel_count.is_contiguous()
    ops.call("tscd_local_offsets", ops.L.LocalOffsetsArgs, B=B, F=F, L=L, sel_count=sel_count, lrow_off=lrow_off)
    return ops.AttnLayoutT(B, F, L, row_off, lrow_off, row_cap, loc_cap, nk_pitch, dtype)


def mca_forward(lay: ops.AttnLayoutT, w: MCAWeights, bank_cls, bank_reg, bank_score, n_rows_dev, n_loc_dev,
                need_reg=True, sim_thresh=0.75, conf_sim_thresh=0.99, debug=None, cls_out=(True, True), obj_out=(True, True),
                tag="mca"):
    """One MCA module.  bank_* [row_cap,256] 16-bit, bank_score [row_cap] fp32; n_rows_dev / n_loc_dev are int32
    device scalars (total bank rows / total local rows).  Returns (trans_cls [loc_cap,1024], trans_obj or None), each a
    (16-bit, fp32) pair; cls_out / obj_out = (want16, want32) select which copies the output GEMMs write."""
    dev, dt = bank_cls.device, lay.dtype
    tmp_c = torch.empty(lay.loc_cap, 512, dtype=dt, device=dev)      # [attn@v | x_ori]
    tmp_r = torch.empty(lay.loc_cap, 512, dtype=dt, device=dev)
    qkv_c = qkv_r = None
    if FUSED_QKV:
        # without need_reg nothing reads the reg branch's V^T or x_ori (only attn_pv's reg-value product and linear_reg do)
        bufs = ops.qkv_project_fused(lay, bank_cls, bank_reg, w.qkv_cls, w.qkv_reg, bank_score, n_rows_dev,
                                     xori_cls=tmp_c[:, 256:], xori_reg=tmp_r[:, 256:] if need_reg else None, tag=tag,
                                     need_reg=need_reg)
    else:
        qkv_c, _ = ops.linear(bank_cls, w.qkv_cls, m_dev=n_rows_dev)
        qkv_r, _ = ops.linear(bank_reg, w.qkv_reg, m_dev=n_rows_dev)
        bufs = ops.attn_prep(lay, qkv_c, qkv_r, bank_score, xori_cls=tmp_c[:, 256:], xori_reg=tmp_r[:, 256:])
    stats = torch.empty(lay.loc_cap, 16, dtype=torch.float32, device=dev)
    ops.attn_pv(lay, bufs, tmp_c[:, :256], tmp_r[:, :256], stats, need_reg=need_reg, tag=tag, max_logit=SINGLE_PASS_MAX_LOGIT)
    cat_c = torch.empty(lay.loc_cap, 768, dtype=dt, device=dev)      # [round2 @ V | linear(x)]
    ops.linear(tmp_c, w.lin_w, w.lin_b, m_dev=n_loc_dev, out16=cat_c[:, 256:], want16=False, tag=tag + ".mca_linear")
    # with a reg output to follow, the cls launch keeps its weights (sim_mask * exp(mean attention)) for the obj launch
    w_keep = torch.empty(lay.loc_cap, lay.nk_pitch, dtype=dt, device=dev) if need_reg else None
    ops.attn_round2(lay, bufs, bufs["vt_cls"], stats, cat_c[:, :256], use_obj_mask=False, sim_thresh=sim_thresh,
                    conf_sim_thresh=conf_sim_thresh, w_out=w_keep, tag=tag + ".cls")
    trans_cls16, trans_cls32 = ops.linear(cat_c, w.out_w, w.out_b, m_dev=n_loc_dev, want16=cls_out[0], want32=cls_out[1],
                                          tag=tag + ".linear")
    trans_obj16 = trans_obj32 = None
    cat_r = None
    if need_reg:
        cat_r = torch.empty(lay.loc_cap, 768, dtype=dt, device=dev)
        ops.linear(tmp_r, w.linreg_w, w.linreg_b, m_dev=n_loc_dev, out16=cat_r[:, 256:], want16=False, tag=tag + ".mca_linear_reg")
        ops.attn_round2(lay, bufs, bufs["vt_reg"], stats, cat_r[:, :256], use_obj_mask=True, sim_thresh=sim_thresh,
                        conf_sim_thresh=conf_sim_thresh, w_in=w_keep, tag=tag + ".obj")
        trans_obj16, trans_obj32 = ops.linear(cat_r, w.obj_w, w.obj_b, m_dev=n_loc_dev, want16=obj_out[0], want32=obj_out[1],
                                              tag=tag + ".linear_obj")
    if debug is not None:
        debug.update(qkv_c=qkv_c, qkv_r=qkv_r, bufs=bufs, tmp_c=tmp_c, tmp_r=tmp_r, stats=stats, cat_c=cat_c, cat_r=cat_r)
    return (trans_cls16, trans_cls32), (trans_obj16, trans_obj32)


# ----------------------------------------------------------------------------------------------- gen-1 MSA
class MSAWeights:
    """MSA_yolov parameters (post_trans.py:1227-1236): msa.qkv_cls / msa.qkv_reg, linear1, linear2."""

    def __init__(self, sd: Dict[str, torch.Tensor], prefix: str, dtype=torch.float16, device="cuda"):
        w = lambda n: sd[prefix + n].detach().to(device=device, dtype=dtype).contiguous()          # noqa: E731
        b = lambda n: sd[prefix + n].detach().to(device=device, dtype=torch.float32).contiguous()  # noqa: E731
        self.qkv_cls, self.qkv_reg = w("msa.qkv_cls.weight"), w("msa.qkv_reg.weight")               # [768,256]: q|k|v
        self.l1_w, self.l1_b = w("linear1.weight"), b("linear1.bias")
        self.l2_w, self.l2_b = w("linear2.weight"), b("linear2.bias")


def msa_forward(lay: ops.AttnLayoutT, w: MSAWeights, bank_cls, bank_reg, bank_score, n_rows_dev,
                sim_thresh=0.75, conf_sim_thresh=0.99):
    """MSA_yolov.forward (post_trans.py:1256-1269; gen-1 self-attention over ALL proposals of a clip, reconf off).
    `lay` must be a self-attention layout (L == F, lrow_off is row_off).  Returns (out16, out32) [row_cap, 1024]."""
    assert lay.self_attn and lay.L == lay.F
    dev, dt, cap = bank_cls.device, lay.dtype, lay.row_cap
    qkv_c, _ = ops.linear(bank_cls, w.qkv_cls, m_dev=n_rows_dev, tag="msa.qkv_cls")
    qkv_r, _ = ops.linear(bank_reg, w.qkv_reg, m_dev=n_rows_dev, tag="msa.qkv_reg")
    tmp_c = torch.empty(cap, 512, dtype=dt, device=dev)                  # [attn@v | v]
    tmp_r = torch.empty(cap, 512, dtype=dt, device=dev)
    bufs = ops.attn_prep(lay, qkv_c, qkv_r, bank_score, xori_cls=tmp_c[:, 256:], xori_reg=tmp_r[:, 256:])
    stats = torch.empty(cap, 16, dtype=torch.float32, device=dev)
    ops.attn_pv(lay, bufs, tmp_c[:, :256], tmp_r[:, :256], stats, need_reg=False, tag="msa", max_logit=SINGLE_PASS_MAX_LOGIT)
    cat = torch.empty(cap, 1024, dtype=dt, device=dev)                   # [round2 @ tc | tc]
    ops.linear(tmp_c, w.l1_w, w.l1_b, m_dev=n_rows_dev, out16=cat[:, 512:], want16=False, tag="msa.linear1")
    tct = torch.empty(lay.B * 512, lay.nk_pitch, dtype=dt, device=dev)
    ops.call("tscd_transpose_clip", ops.L.TransposeArgs, lay=lay.to_c(), width=512, x=cat[:, 512:], ld_x=cat.stride(0), xt=tct)
    # round 2 aggregates linear1's output, 256 columns per launch; V^T rows of clip b start at b*512 (+256)
    for half in range(2):
        vt = tct.view(lay.B, 512, lay.nk_pitch)[:, half * 256:(half + 1) * 256]
        vt = vt.contiguous().view(lay.B * 256, lay.nk_pitch)
        ops.attn_round2(lay, bufs, vt, stats, cat[:, half * 256:(half + 1) * 256], use_obj_mask=False,
                        sim_thresh=sim_thresh, conf_sim_thresh=conf_sim_thresh, tag=f"msa.half{half}")
    return ops.linear(cat, w.l2_w, w.l2_b, m_dev=n_rows_dev, want16=True, want32=True, tag="msa.linear2")
