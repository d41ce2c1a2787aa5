"""Thin Python wrappers: torch tensors in, C-ABI calls (raw pointers) out.  PyTorch is used for device
memory and streams only."""
import ctypes as C
from dataclasses import dataclass
from typing import List, Optional, Sequence

import torch

from . import _lib as L

_DT = {torch.float32: L.TSCD_F32, torch.float16: L.TSCD_F16, torch.bfloat16: L.TSCD_BF16}


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _p(t: Optional[torch.Tensor]):
    return C.c_void_p(0 if t is None else t.data_ptr())


@dataclass
class AnchorSpec:
    """Level-major, row-major anchor geometry (tscd_head.py:374-376, 755-766)."""
    hw: Sequence[Sequence[int]]
    strides: Sequence[int] = (8, 16, 32)

    @property
    def num_anchors(self):
        return sum(h * w for h, w in self.hw)

    def to_c(self) -> L.Anchors:
        a = L.Anchors()
        a.num_levels = len(self.hw)
        start = 0
        for i, ((h, w), s) in enumerate(zip(self.hw, self.strides)):
            a.level_h[i], a.level_w[i], a.level_stride[i], a.level_start[i] = h, w, s, start
            start += h * w
        a.level_start[len(self.hw)] = start
        return a


def view_rowmajor(t: torch.Tensor, anchors: AnchorSpec, col: int = 0) -> L.View:
    """View of columns [col, col+ch) of a contiguous [F, A, W] tensor."""
    assert t.is_contiguous() and t.dim() == 3
    Fn, A, W = t.shape
    v = L.View()
    es = t.element_size()
    start = 0
    for i, (h, w) in enumerate(anchors.hw):
        v.ptr[i] = t.data_ptr() + (start * W + col) * es
        v.frame_stride[i], v.anchor_stride[i], v.chan_stride[i] = A * W, W, 1
        start += h * w
    return v


def view_levels(ts: List[torch.Tensor]) -> L.View:
    """View of per-level conv outputs [F, ch, H, W] in NCHW or channels_last memory format."""
    v = L.View()
    for i, t in enumerate(ts):
        assert t.dim() == 4
        Fn, ch, H, W = t.shape
        sF, sC, sH, sW = t.stride()
        assert sH == W * sW, "rows of a level must be dense in the anchor dimension"
        v.ptr[i] = t.data_ptr()
        v.frame_stride[i], v.anchor_stride[i], v.chan_stride[i] = sF, sW, sC
    return v


@dataclass
class HeadViews:
    anchors: AnchorSpec
    reg: L.View
    obj: L.View
    cls: L.View
    dtype: torch.dtype
    num_frames: int
    num_classes: int
    apply_sigmoid: bool
    apply_decode: bool
    _keep: tuple = ()  # keeps the tensors alive
    fused: bool = False  # the fused-row layout (from_rows): the row kernels of csrc/select_rows.cu apply

    @staticmethod
    def from_fused(t: torch.Tensor, anchors: AnchorSpec, apply_sigmoid: bool, apply_decode: bool):
        """[F, A, 5+C] tensor: seam S2 (sigmoid applied, not decoded) or S3 (decoded cxcywh)."""
        t = t.contiguous()
        return HeadViews(anchors, view_rowmajor(t, anchors, 0), view_rowmajor(t, anchors, 4),
                         view_rowmajor(t, anchors, 5), t.dtype, t.shape[0], t.shape[2] - 5, apply_sigmoid,
                         apply_decode, (t,))

    @staticmethod
    def from_rows(rows: torch.Tensor, obj: torch.Tensor, anchors: AnchorSpec, num_classes: int, apply_sigmoid: bool = True,
                  apply_decode: bool = True):
        """The FUSED head layout (include/tscd_b200.h tscd_pack_head): rows [F, A, 32|64] fp16 = [reg4|obj|cls C|pad] plus the
        dense objectness plane obj [F, >=A].  Either tensor may live in pinned host memory (forward_host reads the rows
        in place)."""
        assert rows.dim() == 3 and rows.is_contiguous() and rows.dtype == torch.float16 and rows.shape[2] in (32, 64)
        assert obj.dim() == 2 and obj.stride(1) == 1 and obj.dtype == torch.float16 and obj.shape[0] == rows.shape[0]
        assert rows.shape[1] == anchors.num_anchors and obj.shape[1] >= anchors.num_anchors and 5 + num_classes <= rows.shape[2]
        ov = L.View()
        start = 0
        for i, (h, w) in enumerate(anchors.hw):
            ov.ptr[i] = obj.data_ptr() + start * 2
            ov.frame_stride[i], ov.anchor_stride[i], ov.chan_stride[i] = obj.stride(0), 1, 1
            start += h * w
        return HeadViews(anchors, view_rowmajor(rows, anchors, 0), ov, view_rowmajor(rows, anchors, 5), rows.dtype,
                         rows.shape[0], num_classes, apply_sigmoid, apply_decode, (rows, obj), True)

    @staticmethod
    def from_level_rows(rows: List[torch.Tensor], obj: torch.Tensor, anchors: AnchorSpec, num_classes: int, apply_sigmoid: bool = True,
                        apply_decode: bool = True):
        """Fused rows kept per FPN level: rows[l] is [F, H_l*W_l, 32|64] (what pred_heads writes), obj the dense [F, >=A] plane."""
        ov, rv, cv = L.View(), L.View(), L.View()
        start = 0
        for i, ((h, w), t) in enumerate(zip(anchors.hw, rows)):
            assert t.dim() == 3 and t.is_contiguous() and t.dtype == torch.float16 and t.shape[1] == h * w and t.shape[2] in (32, 64)
            rp = t.shape[2]
            ov.ptr[i] = obj.data_ptr() + start * 2
            ov.frame_stride[i], ov.anchor_stride[i], ov.chan_stride[i] = obj.stride(0), 1, 1
            rv.ptr[i], cv.ptr[i] = t.data_ptr(), t.data_ptr() + 5 * 2
            for v in (rv, cv):
                v.frame_stride[i], v.anchor_stride[i], v.chan_stride[i] = h * w * rp, rp, 1
            start += h * w
        return HeadViews(anchors, rv, ov, cv, torch.float16, rows[0].shape[0], num_classes, apply_sigmoid, apply_decode,
                         (tuple(rows), obj), True)

    @staticmethod
    def from_levels(reg: List[torch.Tensor], obj: List[torch.Tensor], cls: List[torch.Tensor], anchors: AnchorSpec):
        """Seam S1: raw per-level conv outputs (logits), sigmoid + decode fused into the kernels."""
        return HeadViews(anchors, view_levels(reg), view_levels(obj), view_levels(cls), cls[0].dtype,
                         cls[0].shape[0], cls[0].shape[1], True, True, (tuple(reg), tuple(obj), tuple(cls)))


def _dev(head: "HeadViews"):
    """Device of the head tensors (outputs are allocated next to their inputs, not on the current device).  Pinned host
    tensors (forward_host's zero-copy views) fall back to the current CUDA device."""
    for group in head._keep:
        for t in (group if isinstance(group, (tuple, list)) else (group,)):
            if isinstance(t, torch.Tensor) and t.is_cuda:
                return t.device
    return torch.device("cuda", torch.cuda.current_device())


def select(head: HeadViews, mode: str, pre_k: int = 750, conf_thresh: float = 0.001, minimal_limit: int = 0,
           maximal_limit: int = 0, cand_cap: Optional[int] = None, status: Optional[torch.Tensor] = None, unsorted: bool = False):
    """K1.  Returns dict(idx,box,score,cls,count) of device tensors [F,cap(,4)] / [F].  `status` ([1] int32) receives
    TSCD_ERR_CAPACITY when a mode-B frame selects more than cand_cap anchors.
    unsorted (mode A, fused-row layout only): skip the objectness sort -- candidates come in ascending anchor order and
    out['rank'] carries the order for ops.nms(rank=...) (same keep list, see include/tscd_b200.h cand_rank)."""
    dev = _dev(head)
    Fn, A = head.num_frames, head.anchors.num_anchors
    if cand_cap is None:
        cand_cap = min(pre_k, A) if mode == "A" else (maximal_limit if maximal_limit else A)
        if mode == "B" and minimal_limit:
            cand_cap = max(cand_cap, min(minimal_limit, A))
    out = dict(idx=torch.empty(Fn, cand_cap, dtype=torch.int32, device=dev),
               box=torch.empty(Fn, cand_cap, 4, dtype=torch.float32, device=dev),
               score=torch.empty(Fn, cand_cap, dtype=torch.float32, device=dev),
               cls=torch.empty(Fn, cand_cap, dtype=torch.int32, device=dev),
               count=torch.empty(Fn, dtype=torch.int32, device=dev), cap=cand_cap)
    a = L.SelectArgs()
    a.mode = 0 if mode == "A" else 1
    a.num_frames, a.num_classes, a.head_dtype = Fn, head.num_classes, _DT[head.dtype]
    a.apply_sigmoid, a.apply_decode = int(head.apply_sigmoid), int(head.apply_decode)
    a.pre_k, a.conf_thresh = pre_k, conf_thresh
    a.minimal_limit, a.maximal_limit, a.cand_cap = minimal_limit, maximal_limit, cand_cap
    a.anchors, a.reg, a.obj, a.cls = head.anchors.to_c(), head.reg, head.obj, head.cls
    a.cand_idx, a.cand_box, a.cand_score = _p(out["idx"]), _p(out["box"]), _p(out["score"])
    a.cand_cls, a.cand_count = _p(out["cls"]), _p(out["count"])
    a.status = _p(status)
    if unsorted:
        if not (mode == "A" and head.fused and Fn > 0):
            raise RuntimeError("ops.select(unsorted=True) needs mode A over the fused-row head layout")
        out["rank"] = torch.empty(Fn, cand_cap, dtype=torch.int32, device=dev)
        a.cand_rank = _p(out["rank"])
    class_contiguous = all(head.cls.chan_stride[i] == 1 for i in range(len(head.anchors.hw)))
    if mode == "A" and not class_contiguous:   # workspace of the streaming class-max kernel (K1 = two kernels for NCHW planes)
        pitch = (A + 15) // 16 * 16
        ws_conf = torch.empty(Fn, pitch, dtype=head.dtype, device=dev)
        ws_cls = torch.empty(Fn, pitch, dtype=torch.uint8, device=dev)
        a.ws_conf, a.ws_cls, a.ws_pitch = _p(ws_conf), _p(ws_cls), pitch
        out["_ws"] = (ws_conf, ws_cls)
        L.launch_count += 1
    with L.timed("tscd_select"):
        L.check(L.lib().tscd_select(C.byref(a), _stream()), "tscd_select")
    return out


def row_pitch(num_classes: int) -> int:
    """Elements per fused head row: 32 (64 bytes) up to 27 classes, 64 (128 bytes) up to 59."""
    if 5 + num_classes <= 32:
        return 32
    if 5 + num_classes <= 64:
        return 64
    raise RuntimeError(f"fused head rows hold at most 59 classes, got {num_classes}")


def pack_head(head: HeadViews, rows: Optional[torch.Tensor] = None, obj: Optional[torch.Tensor] = None) -> HeadViews:
    """tscd_pack_head: any strided fp16 head layout (per-level conv outputs) -> the fused-row layout, one pass."""
    if head.dtype != torch.float16:
        raise RuntimeError("tscd_pack_head: fp16 head outputs only (the fused rows are 16-bit)")
    dev = _dev(head)
    Fn, A = head.num_frames, head.anchors.num_anchors
    rp = row_pitch(head.num_classes)
    if rows is None:
        rows = torch.empty(Fn, A, rp, dtype=torch.float16, device=dev)
    if obj is None:
        obj = torch.empty(Fn, (A + 7) // 8 * 8, dtype=torch.float16, device=dev)     # 16-byte aligned frames
    call("tscd_pack_head", L.PackHeadArgs, num_frames=Fn, num_classes=head.num_classes, head_dtype=head.dtype, row_pitch=rp,
         obj_pitch=obj.stride(0), anchors=head.anchors.to_c(), reg=head.reg, obj=head.obj, cls=head.cls, rows=rows,
         obj_plane=obj)
    return HeadViews.from_rows(rows, obj, head.anchors, head.num_classes, head.apply_sigmoid, head.apply_decode)


def pred_heads(reg_feats: List[torch.Tensor], cls_feats: List[torch.Tensor], w_regobj: List[torch.Tensor], b_regobj: List[torch.Tensor],
               w_cls: List[torch.Tensor], b_cls: List[torch.Tensor], anchors: AnchorSpec, num_classes: int) -> HeadViews:
    """The 1x1 prediction convolutions of the decoupled head (reg_preds / obj_preds on reg_feat, cls_preds on cls_feat,
    tscd_head.py:327-329) as tcgen05 GEMMs that write the FUSED head layout directly (SURVEY 8f-2: the pred convs folded into the
    seam): per level  rows[:, 0:5] = reg_feat @ [W_reg; W_obj]^T + b,  rows[:, 5:5+C] = cls_feat @ W_cls^T + b  over the
    channels_last feature maps viewed as [F*H*W, 256] matrices, then the objectness column into the dense plane.
    reg_feats / cls_feats: per level [F, 256, H, W] fp16 channels_last; w_regobj[l] [5, 256] / w_cls[l] [C, 256] fp16; biases fp32."""
    Fn = reg_feats[0].shape[0]
    dev = reg_feats[0].device
    rp = row_pitch(num_classes)
    A = anchors.num_anchors
    objp = torch.empty(Fn, (A + 7) // 8 * 8, dtype=torch.float16, device=dev)
    rows, start = [], 0
    for l, ((h, w), rf, cf) in enumerate(zip(anchors.hw, reg_feats, cls_feats)):
        assert rf.dtype == torch.float16 and rf.is_contiguous(memory_format=torch.channels_last) and cf.is_contiguous(memory_format=torch.channels_last)
        K = rf.shape[1]
        xr = rf.permute(0, 2, 3, 1).reshape(Fn * h * w, K)          # views: channels_last memory is [F, H, W, C]
        xc = cf.permute(0, 2, 3, 1).reshape(Fn * h * w, K)
        r = torch.zeros(Fn * h * w, rp, dtype=torch.float16, device=dev)
        linear(xr, w_regobj[l], b_regobj[l], out16=r[:, 0:5], want32=False, tag="pred_regobj")
        linear(xc, w_cls[l], b_cls[l], out16=r[:, 5:5 + num_classes], want32=False, tag="pred_cls")
        r = r.view(Fn, h * w, rp)
        objp[:, start:start + h * w].copy_(r[:, :, 4])
        rows.append(r)
        start += h * w
    return HeadViews.from_level_rows(rows, objp, anchors, num_classes)


NMS_SMEM_CAP = 4096       # csrc/nms.cuh kNmsCap: larger candidate lists take the workspace path (csrc/nms_large.cu)
NMS_MAX_CAP = 16384       # kNmsLargeCap: per-frame merge in shared memory (the default tier's final-NMS limit)
NMS_WIDE_CAP = 65536      # kNmsWideCap: merge through global memory (the wide tier's final-NMS limit)


def nms(box: torch.Tensor, score: torch.Tensor, cls: torch.Tensor, count: torch.Tensor, iou_thresh: float,
        max_keep: Optional[int] = None, status: Optional[torch.Tensor] = None, strict_keep: bool = False, tag=None,
        rank: Optional[torch.Tensor] = None, wide: bool = False):
    """K2.  box [F,cap,4] f32, score [F,cap] f32, cls [F,cap] i32, count [F] i32 -> (keep [F,max_keep], keep_count [F]).
    strict_keep: more than max_keep survivors in a frame is a capacity error (status) instead of a truncation.
    wide: the caller is a wide-tier stage (SelectionConfig.max_proposals > 512) and accepts up to NMS_WIDE_CAP candidates per
    frame (global-memory merge); otherwise the limit is NMS_MAX_CAP."""
    Fn, cap = score.shape
    limit = NMS_WIDE_CAP if wide else NMS_MAX_CAP
    if cap > limit:
        raise RuntimeError(f"tscd_nms: {cap} candidates per frame exceed the kernel capacity of {limit}")
    max_keep = cap if max_keep is None else max_keep
    keep = torch.empty(Fn, max_keep, dtype=torch.int32, device=score.device)
    keep_count = torch.empty(Fn, dtype=torch.int32, device=score.device)
    if status is None:
        status = torch.zeros(1, dtype=torch.int32, device=score.device)
    a = L.NmsArgs()
    a.num_frames, a.cand_cap, a.max_keep, a.iou_thresh = Fn, cap, max_keep, iou_thresh
    a.box, a.score, a.cls, a.count = _p(box), _p(score), _p(cls), _p(count)
    a.keep, a.keep_count, a.status = _p(keep), _p(keep_count), _p(status)
    a.strict_keep = int(strict_keep)
    a.rank = _p(rank)
    ws = None
    if cap > NMS_SMEM_CAP:
        a.ws_bytes = L.lib().tscd_nms_workspace_bytes(Fn, cap)
        ws = torch.empty(a.ws_bytes, dtype=torch.uint8, device=score.device)
        a.ws = _p(ws)
    with L.timed("tscd_nms", tag):
        L.check(L.lib().tscd_nms(C.byref(a), _stream()), "tscd_nms_large" if ws is not None else "tscd_nms")
    if ws is not None and not torch.cuda.is_current_stream_capturing():
        ws.record_stream(torch.cuda.current_stream())
    return keep, keep_count, status


def gather(head: HeadViews, feats, feat_dtype: torch.dtype, feat_dim: int, cand, keep=None, keep_count=None,
           max_keep: Optional[int] = None, bank_dtype: torch.dtype = torch.float16, bank_rows: Optional[int] = None):
    """K3.  feats = (view_cls, view_reg, view_edge).  Returns dict with sel_count,row_off,sel_idx,sel_rows,bank_*."""
    dev = cand["idx"].device
    Fn, Cn = head.num_frames, head.num_classes
    use_keep = keep is not None
    max_keep = (keep.shape[1] if use_keep else cand["cap"]) if max_keep is None else max_keep
    rows_cap = Fn * max_keep if bank_rows is None else bank_rows
    out = dict(sel_count=torch.empty(Fn, dtype=torch.int32, device=dev),
               row_off=torch.empty(Fn + 1, dtype=torch.int32, device=dev),
               sel_idx=torch.empty(Fn, max_keep, dtype=torch.int32, device=dev),
               sel_rows=torch.empty(Fn, max_keep, 7 + Cn, dtype=torch.float32, device=dev),
               # rows past the packed count are never consumed (every kernel is bounded by the device-side counts)
               bank_cls=torch.empty(rows_cap, feat_dim, dtype=bank_dtype, device=dev),
               bank_reg=torch.empty(rows_cap, feat_dim, dtype=bank_dtype, device=dev),
               bank_edge=torch.empty(rows_cap, feat_dim, dtype=bank_dtype, device=dev),
               bank_score=torch.empty(rows_cap, dtype=torch.float32, device=dev),
               bank_fg=torch.empty(rows_cap, dtype=torch.float32, device=dev),
               bank_box=torch.empty(rows_cap, 4, dtype=torch.float32, device=dev), max_keep=max_keep)
    a = L.GatherArgs()
    a.num_frames, a.num_classes, a.head_dtype = Fn, Cn, _DT[head.dtype]
    a.apply_sigmoid, a.apply_decode = int(head.apply_sigmoid), int(head.apply_decode)
    a.cand_cap, a.max_keep, a.use_keep = cand["cap"], max_keep, int(use_keep)
    a.feat_dim, a.feat_dtype, a.bank_dtype = feat_dim, _DT[feat_dtype], _DT[bank_dtype]
    a.anchors, a.reg, a.obj, a.cls = head.anchors.to_c(), head.reg, head.obj, head.cls
    a.feat_cls, a.feat_reg = feats[0], feats[1]
    a.feat_edge = feats[2] if isinstance(feats[2], L.View) else L.View()   # EdgeBlock: rows computed afterwards (edge_rows)
    a.cand_idx, a.cand_count = _p(cand["idx"]), _p(cand["count"])
    a.keep, a.keep_count = _p(keep), _p(keep_count)
    for k in ("sel_count", "row_off", "sel_idx", "sel_rows", "bank_cls", "bank_reg", "bank_edge", "bank_score",
              "bank_fg", "bank_box"):
        setattr(a, k, _p(out[k]))
    with L.timed("tscd_gather"):
        L.check(L.lib().tscd_gather(C.byref(a), _stream()), "tscd_gather")
    return out


class EdgeBlock:
    """Weights of the head's per-level WaveletsHFBlock modules (edge_enhance_reg, tscd_head.py:206; surrounding_extraction.py:
    215-233) laid out for the selected-anchor evaluation (csrc/edge.cu): pass it as the third element of `feats` instead of a
    view of densely computed edge maps.  w3[l] [256, 9*256] is filter2's 3x3 kernel tap-major ((ky, kx), input channel), w1[l]
    [768, 768] filter1's 1x1 kernel; 16-bit operands in the stage's operand dtype, fp32 biases."""

    def __init__(self, w3: List[torch.Tensor], b3: List[torch.Tensor], w1: List[torch.Tensor], b1: List[torch.Tensor],
                 dtype: torch.dtype = torch.float16, device="cuda"):
        assert dtype in (torch.float16, torch.bfloat16)
        self.dtype = dtype
        self.w3, self.b3, self.w1, self.b1 = [], [], [], []
        for k in range(len(w3)):
            co, ci, kh, kw = w3[k].shape
            if (co, ci, kh, kw) != (256, 256, 3, 3) or tuple(w1[k].shape[:2]) != (768, 768):
                raise RuntimeError("EdgeBlock: the kernels are specialised for WaveletsHFBlock(256)")
            self.w3.append(w3[k].detach().permute(0, 2, 3, 1).reshape(co, kh * kw * ci).to(device=device, dtype=dtype).contiguous())
            self.w1.append(w1[k].detach().reshape(768, 768).to(device=device, dtype=dtype).contiguous())
            self.b3.append(b3[k].detach().to(device=device, dtype=torch.float32).contiguous())
            self.b1.append(b1[k].detach().to(device=device, dtype=torch.float32).contiguous())

    @staticmethod
    def from_modules(blocks, dtype: torch.dtype = torch.float16, device="cuda") -> "EdgeBlock":
        """blocks: the head's nn.ModuleList edge_enhance_reg (filter1 = Conv2d(768,768,1)+ReLU, filter2 = Conv2d(256,256,3,p=1)+ReLU)."""
        blocks = [b if hasattr(b, "filter2") else b[0] for b in blocks]      # the head wraps each block in nn.Sequential (:206-212)
        return EdgeBlock([b.filter2[0].weight for b in blocks], [b.filter2[0].bias for b in blocks],
                         [b.filter1[0].weight for b in blocks], [b.filter1[0].bias for b in blocks], dtype, device)


def edge_rows(block: EdgeBlock, feat_reg: L.View, feat_dtype: torch.dtype, anchors: AnchorSpec, gathered: dict, num_frames: int,
              status: Optional[torch.Tensor] = None):
    """Fills gathered['bank_edge'] with WaveletsHFBlock(feat_reg) at the kept proposals: patch / Haar rows per level
    (tscd_edge_patches), two tcgen05 GEMMs per level with the device-side row count, combine (tscd_edge_combine)."""
    bank = gathered["bank_edge"]
    dev, dt = bank.device, bank.dtype
    if dt != block.dtype:
        raise RuntimeError(f"EdgeBlock weights are {block.dtype}, the bank is {dt}")
    if len(block.w3) != len(anchors.hw):
        raise RuntimeError("EdgeBlock: one weight set per pyramid level expected")
    max_keep = gathered["max_keep"]
    rows = num_frames * max_keep
    seg_cap = [((min(rows, num_frames * h * w) + 127) // 128) * 128 for h, w in anchors.hw]
    seg_base = [sum(seg_cap[:l]) for l in range(len(seg_cap))]
    slots = sum(seg_cap)
    patches = torch.empty(slots, 9 * 256, dtype=dt, device=dev)
    hf = torch.empty(slots, 3 * 256, dtype=dt, device=dev)
    content = torch.empty(slots, 256, dtype=dt, device=dev)
    hf_out = torch.empty(slots, 3 * 256, dtype=dt, device=dev)
    level_count = torch.empty(L.MAX_LEVELS, dtype=torch.int32, device=dev)
    slot = torch.empty(bank.shape[0], dtype=torch.int32, device=dev)
    a = L.EdgePatchesArgs()
    a.num_frames, a.max_keep, a.feat_dtype, a.op_dtype = num_frames, max_keep, _DT[feat_dtype], _DT[dt]
    a.anchors, a.feat_reg = anchors.to_c(), feat_reg
    a.sel_idx, a.sel_count, a.row_off = _p(gathered["sel_idx"]), _p(gathered["sel_count"]), _p(gathered["row_off"])
    for l in range(len(seg_cap)):
        a.seg_base[l], a.seg_cap[l] = seg_base[l], seg_cap[l]
    a.level_count, a.slot, a.patches, a.hf, a.status = _p(level_count), _p(slot), _p(patches), _p(hf), _p(status)
    with L.timed("tscd_edge_patches"):
        L.check(L.lib().tscd_edge_patches(C.byref(a), _stream()), "tscd_edge_patches")
    for l in range(len(seg_cap)):
        s0, s1 = seg_base[l], seg_base[l] + seg_cap[l]
        linear(patches[s0:s1], block.w3[l], block.b3[l], m_dev=level_count[l:l + 1], out16=content[s0:s1], tag="edge_f2")
        linear(hf[s0:s1], block.w1[l], block.b1[l], m_dev=level_count[l:l + 1], out16=hf_out[s0:s1], tag="edge_f1")
    c = L.EdgeCombineArgs()
    c.rows_cap, c.op_dtype = bank.shape[0], _DT[dt]
    c.total_rows, c.slot = _p(gathered["row_off"][num_frames:]), _p(slot)
    c.content, c.hf_out, c.bank_edge = _p(content), _p(hf_out), _p(bank)
    with L.timed("tscd_edge_combine"):
        L.check(L.lib().tscd_edge_combine(C.byref(c), _stream()), "tscd_edge_combine")
    return bank


def linear(x: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor] = None, m_dev: Optional[torch.Tensor] = None,
           out16: Optional[torch.Tensor] = None, out32: Optional[torch.Tensor] = None, want16=True, want32=False, tag=None):
    """y = x @ w.T + bias on the tcgen05 GEMM.  x [M,K] (row pitch may exceed K), w [N,K]; both fp16 or bf16.
    Outputs may be column slices of wider buffers (stride(0) is the pitch)."""
    assert x.dtype == w.dtype and x.dtype in (torch.float16, torch.bfloat16)
    assert x.stride(1) == 1 and w.stride(1) == 1
    M, K = x.shape
    N = w.shape[0]
    if out16 is None and want16:
        out16 = torch.empty(M, N, dtype=x.dtype, device=x.device)
    if out32 is None and want32:
        out32 = torch.empty(M, N, dtype=torch.float32, device=x.device)
    a = L.LinearArgs()
    a.M, a.N, a.K, a.dtype = M, N, K, _DT[x.dtype]
    a.x, a.ldx, a.w, a.ldw = _p(x), x.stride(0), _p(w), w.stride(0)
    a.bias = _p(bias)
    a.m_dev = _p(m_dev)
    a.out16, a.ld16 = _p(out16), (0 if out16 is None else out16.stride(0))
    a.out32, a.ld32 = _p(out32), (0 if out32 is None else out32.stride(0))
    if bias is not None:
        assert bias.dtype == torch.float32 and bias.is_contiguous()
    if L.profile is not None:
        L.profile.setdefault("linear", []).append((M, N, K, m_dev, tag, out16 is not None, out32 is not None))
    with L.timed("tscd_linear", tag):
        L.check(L.lib().tscd_linear(C.byref(a), _stream()), "tscd_linear")
    return out16, out32


# ----------------------------------------------------------------------------------------------- K4 attention
@dataclass
class AttnLayoutT:
    """Batch layout shared by the attention kernels (device offsets, no host sync)."""
    B: int
    F: int
    L: int
    row_off: torch.Tensor      # int32 [B*F+1]
    lrow_off: torch.Tensor     # int32 [B*L+1]
    row_cap: int
    loc_cap: int
    nk_pitch: int
    dtype: torch.dtype
    self_attn: bool = False

    def to_c(self) -> L.AttnLayout:
        a = L.AttnLayout()
        a.B, a.F, a.L, a.self_attn, a.dtype = self.B, self.F, self.L, int(self.self_attn), _DT[self.dtype]
        a.row_cap, a.nk_pitch = self.row_cap, self.nk_pitch
        a.row_off, a.lrow_off = _p(self.row_off), _p(self.lrow_off)
        return a


def attn_prep(lay: AttnLayoutT, qkv_cls, qkv_reg, key_score, xori_cls=None, xori_reg=None, scale=25.0, bufs=None):
    """Normalise / scale / transpose.  qkv_* are [row_cap, >=768] views (q|k|v).  Returns dict of operand buffers."""
    dev, dt = qkv_cls.device, lay.dtype
    if bufs is None:
        bufs = {}
        # no zero fill: invalid keys are masked by select (never multiplied) and the prep kernel itself zero-fills
        # the V^T padding that the P@V / W@V products read
        for n in ("qn_cls", "kn_cls", "vn_cls", "qn_reg", "kn_reg", "vn_reg"):
            bufs[n] = torch.empty(lay.row_cap, 256, dtype=dt, device=dev)
        for n in ("vt_cls", "vt_reg"):
            bufs[n] = torch.empty(lay.B * 256, lay.nk_pitch, dtype=dt, device=dev)
        bufs["row_frame"] = torch.empty(lay.row_cap, dtype=torch.int32, device=dev)
    a = L.AttnPrepArgs()
    a.lay, a.scale = lay.to_c(), scale
    assert qkv_cls.stride(1) == 1 and qkv_cls.stride(0) == qkv_reg.stride(0)
    a.qkv_cls, a.qkv_reg, a.ld_qkv, a.key_score = _p(qkv_cls), _p(qkv_reg), qkv_cls.stride(0), _p(key_score)
    for n in ("qn_cls", "kn_cls", "vn_cls", "qn_reg", "kn_reg", "vn_reg", "vt_cls", "vt_reg", "row_frame"):
        setattr(a, n, _p(bufs[n]))
    a.xori_cls, a.xori_reg = _p(xori_cls), _p(xori_reg)
    a.ld_xori = 0 if xori_cls is None else xori_cls.stride(0)
    with L.timed("tscd_attn_prep"):
        L.check(L.lib().tscd_attn_prep(C.byref(a), _stream()), "tscd_attn_prep")
    return bufs


def qkv_project_fused(lay: AttnLayoutT, bank_cls, bank_reg, w_cls, w_reg, key_score, n_rows_dev, xori_cls=None, xori_reg=None,
                      scale=25.0, tag=None, bufs=None, need_reg=True):
    """tscd_attn_rowmeta + 2 x tscd_qkv_project: the q|k|v projections of both branches with the normalise / scale /
    transpose step of tscd_attn_prep fused into the GEMM epilogue.  Returns the same operand dict as attn_prep (plus
    row_meta); `bufs` may supply that dict's buffers.  need_reg=False: a module whose attention never reads the reg
    branch's V^T (attn_pv / mca_forward with need_reg=False): no vt_reg is allocated or computed; pass xori_reg=None too."""
    dev, dt = bank_cls.device, lay.dtype
    if bufs is None:
        bufs = {}
        for n in ("qn_cls", "kn_cls", "vn_cls", "qn_reg", "kn_reg", "vn_reg"):
            bufs[n] = torch.empty(lay.row_cap, 256, dtype=dt, device=dev)
        for n in ("vt_cls", "vt_reg")[:2 if need_reg else 1]:
            bufs[n] = torch.empty(lay.B * 256, lay.nk_pitch, dtype=dt, device=dev)
        bufs["row_frame"] = torch.empty(lay.row_cap, dtype=torch.int32, device=dev)
        bufs["row_meta"] = torch.empty(lay.row_cap, dtype=torch.int32, device=dev)
    call("tscd_attn_rowmeta", L.AttnRowmetaArgs, lay=lay.to_c(), row_frame=bufs["row_frame"], row_meta=bufs["row_meta"],
         vt_cls=bufs["vt_cls"], vt_reg=bufs.get("vt_reg"))
    for br, bank, w, ks, xo in (("cls", bank_cls, w_cls, key_score, xori_cls), ("reg", bank_reg, w_reg, None, xori_reg)):
        assert bank.shape[0] >= lay.row_cap and bank.stride(1) == 1 and w.shape == (768, 256) and w.is_contiguous()
        call("tscd_qkv_project", L.QkvProjectArgs, tag=None if tag is None else f"{tag}.{br}", lay=lay.to_c(), rows=lay.row_cap, m_dev=n_rows_dev, x=bank, ldx=bank.stride(0),
             w=w, row_meta=bufs["row_meta"], key_score=ks, scale=scale, qn=bufs["qn_" + br], kn=bufs["kn_" + br],
             vn=bufs["vn_" + br], vt=bufs.get("vt_" + br), xori=xo, ld_xori=0 if xo is None else xo.stride(0))
    return bufs


def attn_pv(lay: AttnLayoutT, bufs, x_cls, x_reg, stats, need_reg=True, tag=None, max_logit: float = 0.0):
    """max_logit > 0: single-pass mode (include/tscd_b200.h tscd_attn_pv_args.max_logit)."""
    a = L.AttnPvArgs()
    a.max_logit = max_logit
    a.lay = lay.to_c()
    for n in ("qn_cls", "kn_cls", "qn_reg", "kn_reg", "vt_cls", "vt_reg", "row_frame"):
        setattr(a, n, _p(bufs.get(n)))
    a.need_reg = int(need_reg)
    a.x_cls, a.x_reg, a.ld_x, a.stats = _p(x_cls), _p(x_reg), x_cls.stride(0), _p(stats)
    with L.timed("tscd_attn_pv", tag):
        L.check(L.lib().tscd_attn_pv(C.byref(a), _stream()), "tscd_attn_pv")


def attn_round2(lay: AttnLayoutT, bufs, vt, stats, out, use_obj_mask, sim_thresh=0.75, conf_sim_thresh=0.99, w_out=None, w_in=None,
                tag=None):
    a = L.AttnRound2Args()
    a.lay = lay.to_c()
    for n in ("qn_cls", "kn_cls", "qn_reg", "kn_reg", "vn_cls", "vn_reg", "row_frame"):
        setattr(a, n, _p(bufs[n]))
    a.vt, a.stats, a.use_obj_mask = _p(vt), _p(stats), int(use_obj_mask)
    a.sim_thresh, a.conf_sim_thresh = sim_thresh, conf_sim_thresh
    a.out, a.ld_out = _p(out), out.stride(0)
    a.w_out, a.w_in = _p(w_out), _p(w_in)
    for t in (w_out, w_in):
        assert t is None or (t.dtype == lay.dtype and t.stride(0) == lay.nk_pitch and t.stride(1) == 1)
    with L.timed("tscd_attn_round2", tag):
        L.check(L.lib().tscd_attn_round2(C.byref(a), _stream()), "tscd_attn_round2")


# ----------------------------------------------------------------------------------------------- generic call helper
def call(name: str, struct_cls, tag=None, **kw):
    """Fill a ctypes argument struct from keyword arguments (tensors -> data_ptr) and call the C-ABI entry point."""
    a = struct_cls()
    for k, v in kw.items():
        if isinstance(v, C.Structure):
            pass
        elif isinstance(v, torch.Tensor) or v is None:
            v = _p(v)
        elif isinstance(v, torch.dtype):
            v = _DT[v]
        setattr(a, k, v)
    missing = {f[0] for f in struct_cls._fields_} - set(kw)
    assert not missing, f"{name}: missing {missing}"
    with L.timed(name, tag):
        L.check(getattr(L.lib(), name)(C.byref(a), _stream()), name)


# ----------------------------------------------------------------------------------------------- frame store
def frame_scatter(store, frame_slots: torch.Tensor, sel: dict, status: torch.Tensor, slot_error: Optional[torch.Tensor] = None):
    """tscd_frame_scatter: the K1-K3 output `sel` of N frames (ops.gather dict, max_keep == store.kmax) -> store slots
    frame_slots [N] (int32 device tensor).  `status` (the K1-K3 flag) is copied into every slot written; `slot_error` ([1],
    optional) receives TSCD_ERR_FRAME_SLOT for a slot outside the store.  No host sync."""
    a = L.FrameScatterArgs()
    a.store = store.to_c()
    a.num_frames = frame_slots.numel()
    a.frame_slots, a.status, a.slot_error = _p(frame_slots), _p(status), _p(slot_error)
    for k in ("sel_count", "row_off", "sel_idx", "sel_rows", "bank_cls", "bank_reg", "bank_edge", "bank_score"):
        setattr(a, k, _p(sel[k]))
    with L.timed("tscd_frame_scatter"):
        L.check(L.lib().tscd_frame_scatter(C.byref(a), _stream()), "tscd_frame_scatter")


def clip_assemble(store, clip_slots: torch.Tensor, B: int, F: int, Lf: int, row_cap: int, status: torch.Tensor,
                  out: Optional[dict] = None, want_idx: bool = True) -> dict:
    """tscd_clip_assemble: clip_slots [B, F] (int32 device tensor) -> the packed clip dict forward_from_bank consumes
    (sel_count, row_off, bank_cls/reg/edge/score with row_cap rows, sel_rows, sel_idx).  `out`: preallocated buffers of that
    shape to write instead (nothing is allocated then)."""
    dev = clip_slots.device
    nf, kmax, W = B * F, store.kmax, 7 + store.num_classes
    if out is None:
        out = dict(sel_count=torch.empty(nf, dtype=torch.int32, device=dev),
                   row_off=torch.empty(nf + 1, dtype=torch.int32, device=dev),
                   sel_idx=torch.empty(nf, kmax, dtype=torch.int32, device=dev) if want_idx else None,
                   sel_rows=torch.empty(nf, kmax, W, dtype=torch.float32, device=dev),
                   bank_score=torch.empty(row_cap, dtype=torch.float32, device=dev), max_keep=kmax)
        for k in ("bank_cls", "bank_reg", "bank_edge"):
            out[k] = torch.empty(row_cap, store.dim, dtype=store.dtype, device=dev)
    call("tscd_clip_assemble", L.ClipAssembleArgs, store=store.to_c(), B=B, F=F, L=Lf, row_cap=out["bank_cls"].shape[0],
         clip_slots=clip_slots, sel_count=out["sel_count"], row_off=out["row_off"], bank_cls=out["bank_cls"],
         bank_reg=out["bank_reg"], bank_edge=out["bank_edge"], bank_score=out["bank_score"], sel_idx=out.get("sel_idx"),
         sel_rows=out["sel_rows"], status=status)
    return out


# ----------------------------------------------------------------------------------------------- video pack
def video_pack(calls, frame_map: torch.Tensor, scale: Optional[torch.Tensor] = None, status: Optional[torch.Tensor] = None,
               out: Optional[dict] = None) -> dict:
    """tscd_video_pack: calls = [(rows [n, cap, 7], count [n], cand [n] or None), ...] (device tensors of the clip calls of a
    group), frame_map [frames, 3] int32 device tensor of (call, row, frame index in its video), scale [frames] fp32 or None.
    Returns {'packed' [frames * cap, 12], 'offsets' [frames + 1], 'det_cand' [frames], 'calls' (the device call array, kept
    alive with the launch)}; no host sync.  `out`: preallocated buffers of those shapes."""
    if not calls:
        raise RuntimeError("video_pack: no clip calls")
    cap = calls[0][0].shape[1]
    for rows, count, cand in calls:
        if rows.dim() != 3 or rows.shape[1] != cap or rows.shape[2] != 7 or rows.dtype != torch.float32 or not rows.is_contiguous():
            raise RuntimeError(f"video_pack: every call's rows must be contiguous fp32 [n, {cap}, 7], got {tuple(rows.shape)}")
        if count.dtype != torch.int32 or count.numel() < rows.shape[0]:
            raise RuntimeError("video_pack: counts must be int32 with one entry per row")
    dev = frame_map.device
    nf = frame_map.shape[0]
    arr = (L.VideoPackCall * len(calls))()
    for i, (rows, count, cand) in enumerate(calls):
        arr[i].rows, arr[i].count, arr[i].cand, arr[i].n_rows = _p(rows), _p(count), _p(cand), rows.shape[0]
    # the call array travels to the device with the launch (a pinned copy: stream-ordered, the host buffer is kept by torch
    # until the copy has run)
    host = torch.frombuffer(bytearray(C.string_at(arr, C.sizeof(arr))), dtype=torch.uint8).pin_memory()
    dcalls = host.to(dev, non_blocking=True)
    if out is None:
        out = dict(packed=torch.empty(max(nf * cap, 1), 12, dtype=torch.float32, device=dev),
                   offsets=torch.empty(nf + 1, dtype=torch.int32, device=dev),
                   det_cand=torch.empty(nf, dtype=torch.int32, device=dev))
    call("tscd_video_pack", L.VideoPackArgs, num_frames=nf, num_calls=len(calls), cap=cap, pad=0, calls=dcalls, map=frame_map,
         scale=scale, offsets=out["offsets"], packed=out["packed"], det_cand=out["det_cand"], status=status)
    out["calls"] = dcalls
    return out
