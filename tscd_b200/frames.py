"""Frame store: select and gather every video frame ONCE, assemble clips from it on the device.

A video is cut into overlapping clips (clips.demo_clips / clips.dataset_clips: `lframe` consecutive local frames + `gframe`
frames drawn from the rest of the video), so a frame takes part in many clips: about 4 times per video at OVIS TSCD-L (8 local
+ 24 global), about 32 times at VID TSCD-L (1 + 31).  Everything K1-K3 (selection, pre-NMS, bank gather, edge rows) produce
for a frame depends on that frame alone, and everything after them reads only the clip's packed bank.  So

    AggregationStage.ingest_frames(store, head, feats, feat_dtype, frame_slots)     K1-K3 once per frame -> store slots
    AggregationStage.forward_clips(store, clip_slots, L, time_embedding, ...)       tscd_clip_assemble + forward_from_bank

gives bit for bit what forward() gives on clip tensors built with index_select from the same frames.  The caller maps video
frames to slots, the same way CAFMState slots map to videos (INTEGRATION.md "Videos: select every frame once")."""
from typing import Optional

import numpy as np
import torch

from . import _lib as L

MAX_KEYS_PER_CLIP = 65536     # attention kernels: keys of one clip (csrc/attn.cu, 16-bit key index in row_meta)


def check_keys_per_clip(F: int, kmax: int):
    """The attention kernels' limit on keys per clip (F frames x kmax proposals, in 128-row tiles), shared by
    AggregationStage.forward and forward_clips."""
    if _r128(F * kmax) > MAX_KEYS_PER_CLIP:
        raise RuntimeError(f"{F} frames x {kmax} proposals per frame = {F * kmax} keys per clip exceed the attention kernels' "
                           f"capacity of {MAX_KEYS_PER_CLIP}; lower SelectionConfig.max_proposals")


def _r128(x: int) -> int:
    return (x + 127) // 128 * 128


class FrameStore:
    """Caller-owned pool of `frames` frame slots; each holds one frame's K1-K3 result at a fixed pitch of `kmax` rows
    (kmax = the stage's SelectionConfig.max_keep, so the wide tier's 2048 works as well as the default tier).

    Fields (views of ONE flat byte buffer `flat`, every field 16-byte aligned):
      count      [frames] int32         kept rows of the frame in the slot; -1 = never written
      status     [frames] int32         status of the ingest call that wrote the slot (0 ok, else a TSCD_ERR_* code)
      bank_cls, bank_reg, bank_edge     [frames, kmax, dim] 16-bit feature rows
      bank_score [frames, kmax] fp32    class confidence of each row (the MCA key score)
      sel_idx    [frames, kmax] int32   anchor ids
      sel_rows   [frames, kmax, 7+C] fp32  reference rows [x1,y1,x2,y2,obj,class_conf,class_pred,cls*C] (read for local frames)

    Bytes per slot: 8 + kmax * (6*dim + 8 + 4*(7+C)), i.e. at dim 256  8 + kmax * (1544 + 4*(7+C)):
    49 KB at OVIS mode A (kmax 30, C 25), 0.84 MB at OVIS-L mode B (kmax 500), 0.87 MB at VID-L (kmax 512, C 30), 3.5 MB on the
    wide tier (kmax 2048, C 30)."""

    def __init__(self, frames: int, kmax: int, num_classes: int, dim: int = 256, dtype: torch.dtype = torch.float16,
                 device="cuda"):
        if frames < 1 or kmax < 1 or num_classes < 1:
            raise RuntimeError(f"FrameStore: frames, kmax and num_classes must be positive (got {frames}, {kmax}, {num_classes})")
        if dtype not in (torch.float16, torch.bfloat16):
            raise RuntimeError(f"FrameStore: the bank is 16-bit (float16 / bfloat16), got {dtype}")
        self.frames, self.kmax, self.num_classes, self.dim, self.dtype = frames, kmax, num_classes, dim, dtype
        self.num_anchors = None            # anchors per frame of the frames ingested (set by the first ingest)
        W = 7 + num_classes
        rows = frames * kmax
        sizes = [("count", frames * 4), ("status", frames * 4), ("bank_cls", rows * dim * 2), ("bank_reg", rows * dim * 2),
                 ("bank_edge", rows * dim * 2), ("bank_score", rows * 4), ("sel_idx", rows * 4), ("sel_rows", rows * W * 4)]
        total = sum((n + 15) // 16 * 16 for _, n in sizes)
        self.flat = torch.zeros(total, dtype=torch.uint8, device=device)
        off, v = 0, {}
        for name, n in sizes:
            v[name] = self.flat[off:off + n]
            off += (n + 15) // 16 * 16
        self.count, self.status = v["count"].view(torch.int32), v["status"].view(torch.int32)
        self.bank_cls, self.bank_reg, self.bank_edge = (v[k].view(dtype).view(frames, kmax, dim) for k in ("bank_cls", "bank_reg", "bank_edge"))
        self.bank_score = v["bank_score"].view(torch.float32).view(frames, kmax)
        self.sel_idx = v["sel_idx"].view(torch.int32).view(frames, kmax)
        self.sel_rows = v["sel_rows"].view(torch.float32).view(frames, kmax, W)
        self.count.fill_(-1)

    @staticmethod
    def bytes_per_slot(kmax: int, num_classes: int, dim: int = 256) -> int:
        return 8 + kmax * (6 * dim + 8 + 4 * (7 + num_classes))

    @property
    def device(self):
        return self.flat.device

    def to_c(self) -> L.FrameStoreC:
        from .ops import _DT, _p
        s = L.FrameStoreC()
        s.frames, s.kmax, s.num_classes, s.dtype = self.frames, self.kmax, self.num_classes, _DT[self.dtype]
        for k in ("count", "status", "bank_cls", "bank_reg", "bank_edge", "bank_score", "sel_idx", "sel_rows"):
            setattr(s, k, _p(getattr(self, k)))
        return s


def _host_ints(x) -> np.ndarray:
    return np.asarray(x.cpu() if isinstance(x, torch.Tensor) else x, dtype=np.int64)


def check_clip_args(store: FrameStore, slots, kmax: int, num_classes: int, dim: int, dtype: torch.dtype, L: Optional[int] = None,
                    num_frames: Optional[int] = None):
    """Validates the slot arguments of one frame-store call (no device work; raises RuntimeError).

    L None: AggregationStage.ingest_frames -- `slots` is [num_frames] distinct slots.  L given: forward_clips -- `slots` is
    [B, F] (clip-major; a slot may repeat, within a clip too: the reference pads short videos and tail clips with their last
    frame) and L the local frames of each clip.  `slots` may be a list, a NumPy array, a CPU tensor or an int32 device tensor;
    the values of a device tensor are not read back (capture-safe), the others are checked against [0, store.frames).
    kmax / num_classes / dim / dtype are the stage's: a store of another shape is rejected, naming the expected value."""
    where = "forward_clips" if L is not None else "ingest_frames"
    for name, have, want in (("kmax", store.kmax, kmax), ("num_classes", store.num_classes, num_classes), ("dim", store.dim, dim),
                             ("dtype", store.dtype, dtype)):
        if have != want:
            extra = " (SelectionConfig.max_keep)" if name == "kmax" else ""
            raise RuntimeError(f"{where}: the FrameStore has {name} = {have}, this stage needs {name} = {want}{extra}; allocate "
                               f"FrameStore(frames, {kmax}, {num_classes}, dim={dim}, dtype={dtype})")
    dev = isinstance(slots, torch.Tensor) and slots.is_cuda
    if dev:
        if slots.dtype != torch.int32 or not slots.is_contiguous():
            raise RuntimeError(f"{where}: a device slot tensor must be a contiguous int32 tensor, got {slots.dtype}")
        shape = tuple(slots.shape)
    else:
        arr = _host_ints(slots)
        shape = arr.shape
    if L is None:
        if len(shape) != 1 or (num_frames is not None and shape[0] != num_frames):
            raise RuntimeError(f"{where}: frame_slots must be 1-D with one slot per frame ({num_frames} frames), got shape {shape}")
    else:
        if len(shape) != 2 or shape[0] < 1 or shape[1] < 1:
            raise RuntimeError(f"{where}: clip_slots must be [B, F] (one row of frame slots per clip), got shape {shape}")
        F = shape[1]
        if not 1 <= L <= F:
            raise RuntimeError(f"{where}: L = {L} local frames for clips of F = {F} frames; need 1 <= L <= F")
        check_keys_per_clip(F, kmax)
    if dev:
        return
    flat = arr.reshape(-1)
    bad = sorted({int(x) for x in flat if not 0 <= int(x) < store.frames})
    if bad:
        raise RuntimeError(f"{where}: frame slot(s) {bad} outside [0, {store.frames}) of the FrameStore")
    if L is None and len(set(int(x) for x in flat)) != len(flat):
        dup = sorted({int(x) for x in flat if (flat == x).sum() > 1})
        raise RuntimeError(f"{where}: duplicate frame slot(s) {dup} in one call; every frame of a call needs its own slot")
