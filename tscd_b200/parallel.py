"""Multi-GPU modes of the aggregation stage (SURVEY.md section 8e).

* clip-parallel (configs 3, 5): clips are independent units -> `shard_clips` gives every rank a contiguous block; there
  is NO data-path collective (bench.py --gpus N).
* one long clip sharded by frame (config 4): every rank selects / gathers ITS frames (K1-K3 are per frame), packs the bank
  rows of its GLOBAL frames into one buffer (tscd_bank_pack), the ranks exchange the buffers with ONE all-gather
  (ncclAllGather over NVLink/NVSwitch via torch.distributed; 1040 bytes per row: 0.75 MB per rank at 24 global frames x 30
  proposals), and tscd_bank_unpack builds the virtual clip [own local frames | every rank's global frames].  Queries stay
  sharded, so the attention needs no reduction.  The CAFM recurrence is a chain over consecutive local frames: rank r
  receives the CAFM memory from rank r-1 before its chain and sends it on afterwards -- ONE point-to-point message per hop
  (CAFMState.flat) instead of gathering all local rows.

`frame_plan`, `shard_clips`, `all_gather_bytes` and the state hand-over are device-agnostic and exercised with gloo on CPU
(tests/test_parallel_cpu.py); pack / unpack are CUDA kernels (tests/test_gpu_long_clip.py emulates the ranks on one GPU).
"""
from typing import Dict, Optional

import torch
import torch.distributed as dist

from . import _lib as L
from . import ops
from .selection import DEFAULT_TIER_MAX


def shard_clips(num_clips: int, rank: int, world: int):
    """Contiguous block of clips for `rank` (consecutive clips of one video stay together and in order)."""
    per = (num_clips + world - 1) // world
    lo = min(rank * per, num_clips)
    return lo, min(lo + per, num_clips)


def frame_plan(n_local: int, n_global: int, rank: int, world: int):
    """Frames of a long clip [n_local local | n_global global] owned by `rank`: consecutive blocks of the local frames in rank
    order (the CAFM chain walks them in order) and of the global frames.  Returns (local frame ids, global frame ids)."""
    if n_local % world or n_global % world:
        raise RuntimeError(f"long-clip mode: {n_local} local / {n_global} global frames must divide over {world} ranks")
    lr, gr = n_local // world, n_global // world
    return list(range(rank * lr, (rank + 1) * lr)), list(range(n_local + rank * gr, n_local + (rank + 1) * gr))


def all_gather_bytes(send: torch.Tensor, group=None) -> torch.Tensor:
    """ONE all-gather of a flat uint8 buffer per rank -> [world * nbytes]."""
    world = dist.get_world_size(group)
    recv = torch.empty(world * send.numel(), dtype=send.dtype, device=send.device)
    dist.all_gather_into_tensor(recv, send, group=group)
    return recv


def pack_global_bank(sel: Dict[str, torch.Tensor], n_local_frames: int, n_global_frames: int, kmax: int, dtype) -> torch.Tensor:
    nbytes = L.lib().tscd_bank_pack_bytes(n_global_frames, kmax)
    if nbytes < 0:
        raise RuntimeError(f"long-clip mode: {n_global_frames} global frames per rank exceed the exchange header (256)")
    send = torch.empty(nbytes, dtype=torch.uint8, device=sel["bank_cls"].device)
    ops.call("tscd_bank_pack", L.BankPackArgs, n_local_frames=n_local_frames, n_global_frames=n_global_frames, kmax=kmax, dtype=dtype,
             sel_count=sel["sel_count"], row_off=sel["row_off"], bank_cls=sel["bank_cls"], bank_reg=sel["bank_reg"],
             bank_score=sel["bank_score"], send=send)
    return send


def unpack_virtual_clip(sel: Dict[str, torch.Tensor], recv: torch.Tensor, world: int, n_local_frames: int, n_global_frames: int,
                        kmax: int, dtype):
    """Gathered buffers + own bank -> the `sel` dict of the virtual clip [own local frames | all ranks' global frames]."""
    dev = recv.device
    F_virt = n_local_frames + world * n_global_frames
    rows_cap = ((F_virt * kmax + 127) // 128) * 128 + 128
    D = sel["bank_cls"].shape[1]
    out = dict(sel_count=torch.empty(F_virt, dtype=torch.int32, device=dev), row_off=torch.empty(F_virt + 1, dtype=torch.int32, device=dev),
               bank_cls=torch.empty(rows_cap, D, dtype=dtype, device=dev), bank_reg=torch.empty(rows_cap, D, dtype=dtype, device=dev),
               bank_edge=torch.empty(rows_cap, D, dtype=dtype, device=dev), bank_score=torch.empty(rows_cap, dtype=torch.float32, device=dev))
    ops.call("tscd_bank_unpack", L.BankUnpackArgs, world=world, n_local_frames=n_local_frames, n_global_frames=n_global_frames, kmax=kmax,
             dtype=dtype, rank_bytes=recv.numel() // world, recv=recv, sel_count=sel["sel_count"], row_off=sel["row_off"],
             bank_cls=sel["bank_cls"], bank_reg=sel["bank_reg"], bank_edge=sel["bank_edge"], bank_score=sel["bank_score"],
             v_count=out["sel_count"], v_row_off=out["row_off"], v_bank_cls=out["bank_cls"], v_bank_reg=out["bank_reg"],
             v_bank_edge=out["bank_edge"], v_bank_score=out["bank_score"])
    out["sel_rows"], out["sel_idx"] = sel["sel_rows"], sel.get("sel_idx")
    return out, F_virt


def exchange_global_bank(sel, n_local_frames: int, n_global_frames: int, kmax: int, dtype=torch.float16, group=None):
    """pack -> ONE all-gather -> unpack.  Returns (virtual-clip sel dict, F_virt)."""
    world = dist.get_world_size(group)
    send = pack_global_bank(sel, n_local_frames, n_global_frames, kmax, dtype)
    recv = all_gather_bytes(send, group)
    return unpack_virtual_clip(sel, recv, world, n_local_frames, n_global_frames, kmax, dtype)


def send_state(state, dst: int, group=None):
    dist.send(state.flat, dst, group=group)              # one message: every field is a view of `flat`


def recv_state(state, src: int, group=None):
    dist.recv(state.flat, src, group=group)


def long_clip_forward(stage, sel, n_local_frames: int, n_global_frames: int, kmax: int, time_embedding_local,
                      state, resume_first: bool = False, group=None, trace: Optional[dict] = None):
    """Frame-sharded forward of ONE long clip.  `sel` = this rank's selection (frames ordered [local | global]);
    ranks hold consecutive blocks of the clip's local frames in rank order.  Returns the stage output for this rank's
    local frames (use AggregationStage.to_lists(out, 1, n_local_frames))."""
    if kmax > DEFAULT_TIER_MAX:
        raise RuntimeError(f"long_clip_forward: the long-clip mode supports the default tier only (<= {DEFAULT_TIER_MAX} "
                           f"proposals per frame), got {kmax}")
    rank, world = dist.get_rank(group), dist.get_world_size(group)
    virt, F_virt = exchange_global_bank(sel, n_local_frames, n_global_frames, kmax, stage.cfg.dtype, group)
    dev = virt["bank_cls"].device
    resume = torch.tensor([1 if (rank > 0 or resume_first) else 0], dtype=torch.int32, device=dev)

    def before(st):
        if rank > 0:
            recv_state(st, rank - 1, group)

    def after(st):
        if rank < world - 1:
            send_state(st, rank + 1, group)

    return stage.forward_from_bank(virt, 1, F_virt, n_local_frames, kmax, time_embedding_local, state=state,
                                   resume=resume, trace=trace, before_cafm=before, after_cafm=after)
