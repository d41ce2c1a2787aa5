#!/usr/bin/env python
"""bench.py -- clip-frames/s of the TSCD aggregation stage (BASELINE.json metric) on N B200s.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference|reference-gpu] [--config NAME] [--mode clips|long-clip]
                  [--dump-outputs DIR]
  N > 1:  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

Configurations (--config; BASELINE.json `configs`):
  ovis_a_k30    (default, the headline = configs[1]) TSCD-L OVIS, 25 classes, 32-frame clips (8 local + 24 global), 576x576
                (6804 anchors/frame), pre-NMS top-750 by objectness -> class-aware NMS 0.75 -> 30 proposals/frame, then the TSCD
                aggregation (agg + agg_iou MCA, CAFM, TaskAligned, prediction heads, final per-class NMS 0.5);
  ovis_l_modeB  what exps/TSCD_OVIS/ovis_tscd_large.py really runs: postprocess_widx, minimal_limit 50 / maximal_limit 500,
                no pre-NMS, ragged 50..500 proposals per frame;
  vid_l_c30     configs[2]: TSCD-L ImageNet-VID, 30 classes, gframe = 32 (L = 1, G = 31), minimal_limit 50, no maximal_limit;
  vid_l_16f     configs[0]: one 16-frame VID clip shape (L = 4, G = 12), 30 classes;
  gen1_msa      the gen-1 (YOLOV) pipeline of north_star items (1)-(4): top-750 -> NMS -> 30, MSA self-attention over N = 960;
  sweep         configs[4]: 64 clips x 32 frames, pre-NMS top-k P in {300..1500} x proposals/frame K in {30..100} (one line per point).
--mode long-clip  configs[3]: ONE 256-frame OVIS clip sharded by frame over the ranks (NCCL all-gather of the proposal bank).

Data: synthetic random-init.  Head logits / features at seam S1 (raw per-level conv outputs, fp16, channels_last: what the
drop-in head's conv towers emit), weights uniform(+-1/sqrt(fan_in)).

A STEP is one pass of the stage over `clips x replays` clips per GPU: `replays` CUDA-graph replays of a `clips`-clip batch,
rotating over `--sets` (>= 2) different input sets resident in HBM (each set >> the 126 MB L2: 348 MB per clip), so that a step
is >= 100 ms of GPU work, 20 steps are seconds, and the sustained peaks of MEASURED_PEAKS.json are the right roofline denominators.

value : whole-job clip-frames/s with the step's inputs resident in HBM.
e2e   : same metric through AggregationStage.forward_host_submit / forward_host_collect with HOST (pinned) inputs: H2D of what
        the kernels consume and D2H of the detections inside the timed region; `--e2e-depth` (4) calls are kept in flight the
        way a streaming caller double-buffers (e2e.sync_call_ms is the latency of a lone synchronous call).
roofline : the dominant kernel (largest time per step among single kernels, launches of identical shape averaged), measured live
        with CUDA events in this process; `kernels` lists EVERY kernel of the step the same way.
--impl reference : the UNMODIFIED reference (baseline/_ref, pip-installed `yolox`) running its stock TSCDHead.forward from the
        seam on the host cores (baseline/ref_runner.py), all host threads, one clip per step.  Falls back to the oracle port
        (`kind: "port"`) only if the package is absent.
--impl reference-gpu : the same stock forward on the B200 in eager fp32 / fp16 (the incumbent GPU path; not driver-run).
"""
import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "baseline"))

D = 256
HW = [(72, 72), (36, 36), (18, 18)]
A = sum(h * w for h, w in HW)
METRIC = "clip-frames/sec of TSCD aggregation stage"

CONFIGS = {
    "ovis_a_k30": dict(C=25, F=32, L=8, mode="A", pre_k=750, top_k=30, clips=148, replays=28, obj_means=[-3.0],
                       workload="TSCD-L OVIS 25cls, 32-frame clip (8 local + 24 global) @576x576 (6804 anchors), pre-NMS top-750 -> "
                                "NMS0.75 -> 30 proposals/frame, agg+agg_iou MCA + CAFM + TaskAligned + final NMS0.5"),
    "ovis_l_modeB": dict(C=25, F=32, L=8, mode="B", minimal_limit=50, maximal_limit=500, clips=64, replays=4,
                         obj_means=[-13.5, -8.0, -10.2, -10.6, -9.7, -11.0, -13.0, -9.9],
                         workload="TSCD-L OVIS 25cls (exps/TSCD_OVIS/ovis_tscd_large.py), 32-frame clip (8 local + 24 global) @576x576, "
                                  "postprocess_widx min 50 / max 500, no pre-NMS, ragged 50..500 proposals/frame, full TSCD tail"),
    "vid_l_c30": dict(C=30, F=32, L=1, mode="B", minimal_limit=50, maximal_limit=0, clips=32, replays=16,
                      obj_means=[-13.0, -10.6, -11.0, -11.5, -10.4, -12.5, -10.8, -11.2],
                      workload="TSCD-L ImageNet-VID 30cls (exps/TSCD_VID/vid_tscd_large.py), gframe=32 clip (1 local + 31 global) @576x576, "
                               "postprocess_widx min 50 / no max (capacity 512), no pre-NMS, full TSCD tail"),
    "vid_l_16f": dict(C=30, F=16, L=4, mode="B", minimal_limit=50, maximal_limit=0, clips=32, replays=16,
                      obj_means=[-13.0, -10.6, -11.0, -11.5, -10.4, -12.5, -10.8, -11.2],
                      workload="TSCD-L VID 30cls, 16-frame clip (4 local + 12 global) @576x576, postprocess_widx min 50 / no max, full TSCD tail"),
    "gen1_msa": dict(C=25, F=32, L=32, mode="A", pre_k=750, top_k=30, clips=64, replays=64, obj_means=[-3.0], gen1=True,
                     workload="gen-1 (YOLOV) 25cls, 32-frame clip @576x576, top-750 -> NMS0.75 -> 30 proposals/frame, MSA self-attention "
                              "over N=960 + linear_pred"),
}
SEAMS = {"rows": "S1 raw head logits in the drop-in head's fused layout (one 64 / 128-byte fp16 row [reg4|obj|cls C|pad] per anchor + "
                  "dense objectness plane, tscd_pack_head) and channels_last fp16 feature planes",
         "levels": "S1 raw per-level conv outputs, fp16, channels_last logits and features"}
SWEEP_P, SWEEP_K = (300, 500, 750, 1000, 1500), (30, 50, 75, 100)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        j = json.load(open(p))
        return dict(hbm=j["hbm_gbs"], tf_burst=j["bf16_tflops"], tf_sust=j.get("bf16_tflops_sustained", j["bf16_tflops"]),
                    src="measured (MEASURED_PEAKS.json)")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sust=1400.0, src="fallback (B200_PROFILING.md)")


# ------------------------------------------------------------------------------------------------- synthetic inputs
def synth_s1(cfg, B, device, seed, pin=False, dtype=torch.float16, channels_last=True, layout="levels"):
    """Seam S1 tensors for B clips: per level reg [BF,4,H,W], obj [BF,1,H,W], cls [BF,C,H,W] logits and three feature planes
    [BF,256,H,W].  obj logits ~ N(obj_mean(frame), 2^2) (cfg['obj_means'] cycles over the frames of a clip: controls how many
    anchors pass the 0.001 filter in mode B), cls logits ~ N(-3, 2^2), dx,dy ~ U(-0.5,1.5), dw,dh ~ N(1, 0.7^2)."""
    g = torch.Generator(device=device).manual_seed(seed)
    F, C = cfg["F"], cfg["C"]
    n = B * F
    om = cfg["obj_means"]
    mean = torch.tensor([om[(i % F) % len(om)] for i in range(n)], dtype=torch.float32, device=device).view(n, 1, 1, 1)
    fmt = torch.channels_last if channels_last else torch.contiguous_format
    out = dict(reg=[], obj=[], cls=[], f_cls=[], f_reg=[], f_edge=[])
    for (h, w) in HW:
        xy = torch.rand(n, 2, h, w, generator=g, device=device) * 2 - 0.5
        wh = torch.randn(n, 2, h, w, generator=g, device=device) * 0.7 + 1.0
        out["reg"].append(torch.cat([xy, wh], 1).to(dtype).contiguous(memory_format=fmt))
        out["obj"].append((torch.randn(n, 1, h, w, generator=g, device=device) * 2 + mean).to(dtype).contiguous(memory_format=fmt))
        out["cls"].append((torch.randn(n, C, h, w, generator=g, device=device) * 2 - 3).to(dtype).contiguous(memory_format=fmt))
        for k in ("f_cls", "f_reg", "f_edge"):
            t = torch.empty(n, D, h, w, dtype=dtype, device=device).contiguous(memory_format=fmt)
            for i in range(0, n, 64):       # chunked: bounds the fp32 temporary
                t[i:i + 64] = torch.randn(min(64, n - i), D, h, w, generator=g, device=device).to(dtype)
            out[k].append(t)
    if layout == "rows":       # the drop-in head's fused layout: one 64 / 128-byte row per anchor + dense objectness plane
        from tscd_b200 import ops
        packed = ops.pack_head(ops.HeadViews.from_levels(out["reg"], out["obj"], out["cls"], ops.AnchorSpec(HW)))
        rows, objp = packed._keep
        torch.cuda.synchronize()
        for k in ("reg", "obj", "cls"):
            del out[k]
        out["rows"], out["objp"] = [rows], [objp]
    if pin:
        out = {k: [t.pin_memory() for t in v] for k, v in out.items()}
    return out


def nbytes(d):
    return sum(t.numel() * t.element_size() for v in d.values() for t in v)


def views_of(inp, ops, C=None):
    an = ops.AnchorSpec(HW)
    if "rows" in inp:
        head = ops.HeadViews.from_rows(inp["rows"][0], inp["objp"][0], an, C)
    else:
        head = ops.HeadViews.from_levels(inp["reg"], inp["obj"], inp["cls"], an)
    feats = tuple(ops.view_levels(inp[k]) for k in ("f_cls", "f_reg", "f_edge"))
    return head, feats


def selection_of(cfg, selection):
    if cfg["mode"] == "A":
        return selection.SelectionConfig(mode="A", pre_k=cfg["pre_k"], top_k=cfg["top_k"], nms_thresh=0.75,
                                         max_proposals=max(512, cfg["top_k"]) if cfg.get("gen1") else 512)
    return selection.SelectionConfig(mode="B", minimal_limit=cfg["minimal_limit"], maximal_limit=cfg["maximal_limit"],
                                     use_pre_nms=False, nms_thresh=0.75)


def make_runner(cfg, dev):
    """Returns (stage, run(inp_views, B) -> out, counts_of(out))."""
    from tscd_b200 import gen1, selection, stage, weights
    C, F, L = cfg["C"], cfg["F"], cfg["L"]
    if cfg.get("gen1"):
        st = gen1.Gen1Stage(C, selection_of(cfg, selection), weights.random_state_dict(C, D, seed=2024, gen1=True), device=dev)

        def run(views, B, te):
            head, feats = views
            return st.forward(head, (feats[0], feats[1], feats[1]), torch.float16, B, F)
        return st, run
    st = stage.AggregationStage(stage.StageConfig(num_classes=C, selection=selection_of(cfg, selection)),
                                weights.random_state_dict(C, D, seed=2024), device=dev)

    def run(views, B, te):
        head, feats = views
        return st.forward(head, feats, torch.float16, te, B, F, L)
    return st, run


# ------------------------------------------------------------------------------------------------- --dump-outputs
DUMP_MAX_BYTES = 64_000_000
NPY_HEADER_BYTES = 128             # np.save header of a 1-D / 2-D float array


def caller_arrays(cfg, out, B):
    """What a caller receives from one forward of the stage: {name: (per-frame list of float32 arrays or None, columns,
    most rows a frame can hold)}.  TSCD stage: AggregationStage.to_lists (result / result_ori, per local frame [n,7] or None);
    gen-1 stage: the refined class logits of each frame's proposals."""
    from tscd_b200 import stage
    if cfg.get("gen1"):
        if int(out["status"].item()) != 0:
            raise RuntimeError("the gen-1 stage reported a capacity error")
        off = out["sel"]["row_off"][:B * cfg["F"] + 1].cpu().tolist()
        logits = out["logits"][:off[-1]].cpu().numpy()
        return {"logits": ([logits[a:b] for a, b in zip(off[:-1], off[1:])], logits.shape[1], out["sel"]["sel_rows"].shape[1])}
    host = {k: out[k].cpu() for k in ("status", "det_count", "ori_count", "det_cand", "det_rows", "ori_rows")}
    res, res_ori = stage.AggregationStage.to_lists(host, B, cfg["L"])
    return {name: ([None if t is None else t.numpy() for t in lst], host[name + "_rows"].shape[2], host[name + "_rows"].shape[1])
            for name, lst in (("det", res), ("ori", res_ori))}


def dump_outputs(path, arrays, max_bytes=DUMP_MAX_BYTES, seed=0):
    """Writes caller_arrays() to `path`: per name <name>_rows.npy (float32, the frames' rows concatenated in frame order) and
    <name>_counts.npy (float64, rows per frame, -1 where the caller gets None); frames.npy (float64) lists the frames written.
    When the frames could hold more than max_bytes at full capacity (headers included), a seeded sample of frames is written:
    the first k of a permutation drawn from the frame count and the seed, k set by the output buffers' row capacity.  Two builds
    with the same capacities dump the same frames; with different capacities one frame set contains the other."""
    import numpy as np
    n = len(next(iter(arrays.values()))[0])
    frame_bytes = sum(cols * cap * 4 + 8 for _, cols, cap in arrays.values()) + 8
    k = min(n, max(1, (max_bytes - NPY_HEADER_BYTES * (1 + 2 * len(arrays))) // frame_bytes))
    frames = np.arange(n) if k == n else np.sort(np.random.default_rng(seed).permutation(n)[:k])
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "frames.npy"), frames.astype(np.float64))
    for name, (lst, cols, _) in arrays.items():
        picked = [lst[f] for f in frames]
        rows = [a for a in picked if a is not None]
        np.save(os.path.join(path, name + "_rows.npy"),
                np.concatenate(rows).astype(np.float32) if rows else np.zeros((0, cols), np.float32))
        np.save(os.path.join(path, name + "_counts.npy"), np.array([-1 if a is None else len(a) for a in picked], np.float64))


# ------------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index, extra="", period_ms=100):
        self.index, self.rows, self.proc, self.period_ms = index, [], None, period_ms
        if extra:                       # e.g. the PCIe link state for the host-buffer path
            self.Q = self.Q + "," + extra
        self.extra = [x for x in extra.split(",") if x]

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", str(self.period_ms)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 6 for i in range(4) if r[2 + i].lower() == "active"})
        out = {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
               "reasons": reasons, "samples": len(sm)}
        for k, name in enumerate(self.extra):            # extra columns: the distinct values seen
            out[name] = sorted({r[6 + k] for r in self.rows if len(r) > 6 + k})
        return out


# ------------------------------------------------------------------------------------------------- reference arms
def reference_available():
    try:
        import ref_runner
        return ref_runner.available()
    except Exception:      # noqa: BLE001
        return False


class ReferenceStage:
    """The unmodified reference forward from the seam (baseline/ref_runner.py) on `device`, one clip per call."""

    def __init__(self, cfg, device="cpu", dtype=torch.float32):
        import ref_runner
        self.rr = ref_runner
        ref_runner.install(cpu_redirect=(device == "cpu"))
        args = dict(ref_runner.OVIS_L_ARGS if cfg["C"] == 25 else ref_runner.VID_L_ARGS)
        if cfg["mode"] == "B":
            args["minimal_limit"] = cfg["minimal_limit"]
            if cfg["maximal_limit"]:
                args["maximal_limit"] = cfg["maximal_limit"]
        self.cfg, self.device, self.dtype = cfg, device, dtype
        head = ref_runner.build_head(cfg["C"], args, seed=2024)
        self.head = ref_runner.attach_replay(head, selection=cfg["mode"]).to(device=device, dtype=dtype)
        from tscd_b200.weights import timing_signal_1d
        self.te = timing_signal_1d(torch.arange(cfg["L"]), 256).to(device=device, dtype=dtype)
        inp = synth_s1(cfg, 1, "cpu", seed=2024, dtype=torch.float32, channels_last=False)
        self.inp = {k: [t.to(device=device, dtype=dtype) for t in v] for k, v in inp.items()}

    def one_clip(self):
        i, c = self.inp, self.cfg
        return self.rr.run_tail(self.head, i["reg"], i["obj"], i["cls"], i["f_cls"], i["f_reg"], i["f_edge"], self.te, c["L"], c["F"] - c["L"])


def port_sample(cfg, n_clips, seed=2024):
    """Fallback CPU arm: the oracle port of the reference's fp32 PyTorch code.  Returns (clip_frames_per_s, seconds, threads)."""
    import oracle
    torch.set_num_threads(os.cpu_count() or 1)
    C, F, L = cfg["C"], cfg["F"], cfg["L"]
    head, feats = oracle.synth_head_outputs(F, HW, C, dim=D, seed=seed, obj_mean=[cfg["obj_means"][i % len(cfg["obj_means"])] for i in range(F)])
    if cfg.get("gen1"):
        sd = oracle.init_stage_weights(C, dim=D, seed=seed, gen1=True)

        def one():
            oracle.stage_gen1(sd, oracle.decode_outputs(head, HW, [8, 16, 32]), feats[0], feats[1], C, pre_k=cfg["pre_k"], top_k=cfg["top_k"])
    else:
        sd = oracle.init_stage_weights(C, dim=D, seed=seed)
        te = oracle.timing_signal_1d(torch.arange(L), 256)
        if cfg["mode"] == "A":
            kw = dict(selection="A", select_kwargs=dict(nms_thre=0.75, pre_k=cfg["pre_k"], top_k=cfg["top_k"]))
        else:
            kw = dict(selection="B", select_kwargs=dict(nms_thre=0.75, minimal_limit=cfg["minimal_limit"], maximal_limit=cfg["maximal_limit"], use_pre_nms=False))

        def one():
            oracle.stage_tscd(sd, oracle.decode_outputs(head, HW, [8, 16, 32]), feats[0], feats[1], feats[2], te, C, L, F - L, nms_thresh=0.5, **kw)
    one()
    t0 = time.perf_counter()
    for _ in range(n_clips):
        one()
    dt = time.perf_counter() - t0
    return n_clips * F / dt, dt, torch.get_num_threads()


def cpu_reference_sample(cfg, n_clips, warm=1):
    """(clip-frames/s, seconds, threads, kind, description) of the reference's CPU path on a bounded sample."""
    if reference_available() and not cfg.get("gen1"):
        torch.set_num_threads(os.cpu_count() or 1)
        rs = ReferenceStage(cfg, "cpu", torch.float32)
        for _ in range(warm):
            rs.one_clip()
        t0 = time.perf_counter()
        for _ in range(n_clips):
            rs.one_clip()
        dt = time.perf_counter() - t0
        return (n_clips * cfg["F"] / dt, dt, torch.get_num_threads(), "reference",
                f"{n_clips} clip(s) x {cfg['F']} frames of the same workload through the unmodified reference TSCDHead.forward from the seam "
                f"(baseline/_ref), fp32, {torch.get_num_threads()} threads, {dt:.1f} s")
    fps, dt, thr = port_sample(cfg, n_clips)
    return fps, dt, thr, "port", f"{n_clips} clip(s) x {cfg['F']} frames, fp32, {thr} threads, {dt:.1f} s (oracle port: reference package absent or gen-1 head broken upstream)"


def run_reference(args, cfg, rank):
    if rank != 0:
        return
    per_step = 1
    fps, dt, thr, kind, sample = cpu_reference_sample(cfg, per_step * args.steps, warm=max(1, min(args.warmup, 2)))
    line = {"impl": "reference", "metric": METRIC, "value": fps, "unit": "clip-frames/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": cfg["workload"], "name": args.config, "clips_per_step": per_step},
            "cpu_baseline": {"value": fps, "unit": "clip-frames/s", "cores": thr, "kind": kind, "sample": sample},
            "e2e": {"value": fps, "unit": "clip-frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


def reference_gpu_eager(cfg, dev, reps=3):
    """The incumbent GPU path: the stock reference forward from the seam, eager, on this GPU.  {dtype: clip-frames/s}."""
    out = {}
    for name, dt in (("fp32", torch.float32), ("fp16", torch.float16)):
        try:
            rs = ReferenceStage(cfg, str(dev), dt)
            for _ in range(2):
                rs.one_clip()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(reps):
                rs.one_clip()
            torch.cuda.synchronize()
            out[name] = reps * cfg["F"] / (time.perf_counter() - t0)
            del rs
        except Exception as e:      # noqa: BLE001
            out[name] = f"failed: {type(e).__name__}: {str(e)[:120]}"
    return out


# ------------------------------------------------------------------------------------------------- per-kernel roofline
KERNEL_OF = {"tscd_select": "select_rows_kernel (fused rows, mode A) / select_kernel (+ classmax_kernel for NCHW planes)",
             "tscd_nms": "nms_kernel / nms_matrix_kernel / nmsl_*", "tscd_cafm_wide": "cafm_wide_{begin,perm,qin,finish,end}_kernel",
             "tscd_frame_flash": "frame_flash_kernel",
             "tscd_gather": "rows_gather_kernel (+ offsets)", "tscd_local_offsets": "local_offsets_kernel", "tscd_attn_rowmeta": "attn_rowmeta_kernel",
             "tscd_qkv_project": "gemm_tn_kernel<256,.,EPI=1>", "tscd_linear": "gemm_tn_kernel", "tscd_attn_pv": "attn_pv_kernel",
             "tscd_attn_round2": "attn_round2_kernel", "tscd_attn_prep": "attn_prep_kernel", "tscd_transpose_clip": "transpose_clip_kernel",
             "tscd_cafm_prep": "cafm_prep_kernel", "tscd_cafm_cost": "cafm_cost16_kernel / cafm_cost_wide16_kernel / cafm_cost_kernel",
             "tscd_cafm_lap": "cafm_lap_small_kernel / cafm_lap_kernel",
             "tscd_cafm_chain": "cafm_chain_fast_kernel / cafm_chain_kernel", "tscd_frame_attention": "frame_attention16_kernel / frame_attention_kernel",
             "tscd_residual_ln2": "residual_ln2_kernel", "tscd_final_expand": "final_expand_kernel", "tscd_final_rows": "final_rows_kernel"}


def kernel_rows(cfg, events, linear_info, counts, cand_counts, B, pk, traffic):
    """One row per kernel of the step (launches of identical role averaged): time, bound, algorithmic work (DESIGN.md section 5: the
    SURVEY 8(d) figure and the reduced numerator the kernel really needs), achieved rate, fraction of the measured peak."""
    F, L, C = cfg["F"], cfg["L"], cfg["C"]
    s = 2
    nfr = B * F
    N = sum(counts)
    n_loc = sum(sum(counts[b * F:b * F + L]) for b in range(B))
    pairs = 0
    for b in range(B):
        if cfg.get("gen1"):
            nb = sum(counts[b * F:(b + 1) * F])
            pairs += nb * nb
        else:
            ng = sum(counts[b * F + L:(b + 1) * F])
            pairs += sum(n * (n + ng) for n in counts[b * F:b * F + L])
    P = sum(cand_counts)
    lin = {}
    for (M, Nn, K, md, tag, o16, o32) in linear_info:
        lin[tag] = (M if md is None else min(M, md), Nn, K, o16, o32)
    rows = []
    for key, evs in events.items():
        ms = statistics.mean(a.elapsed_time(b_) for a, b_ in evs)
        entry, _, tag = key.partition(":")
        flops = byts = survey = None
        if entry == "tscd_select":
            if cfg["mode"] == "A":     # objectness plane + the survivors' class / regression rows + candidate records
                byts = nfr * A * s + P * ((C + 4) * s + 28)
            else:                      # mode B: objectness + class rows of every anchor + candidate records
                byts = nfr * A * (1 + C) * s + P * (4 * s + 28)
            survey = nfr * A * (5 + C) * s + P * 32
        elif entry == "tscd_gather":
            byts = survey = 2 * N * 3 * D * s + N * (7 + C) * 4
        elif entry == "tscd_qkv_project":
            flops = 2.0 * N * 768 * 256
            byts = N * 256 * s * 5 + 768 * 256 * s          # x in, qn / kn / vn / V^T out
        elif entry == "tscd_linear" and tag in lin:
            M, Nn, K, o16, o32 = lin[tag]
            flops = 2.0 * M * Nn * K
            byts = M * K * s + Nn * K * s + M * Nn * (2 * o16 + 4 * o32)
        elif entry == "tscd_attn_pv":
            flops = pairs * (2048.0 if tag == "agg_iou" else 1536.0)
        elif entry == "tscd_attn_round2":
            flops = pairs * 1024.0
        elif entry == "tscd_cafm_cost":
            flops = sum(2.0 * 2 * n * n * 1024 for b in range(B) for n in counts[b * F:b * F + L])
        elif entry == "tscd_residual_ln2":
            byts = n_loc * 1024 * 4 * 2
        elif entry == "tscd_frame_attention":
            byts = n_loc * 1024 * (2 * 3 + 4)
        elif entry == "tscd_cafm_prep":
            byts = n_loc * (256 * 2 * 2 + 1024 * 4 * 2 + 256 * 2 * 2)
        t_fl = flops / (pk["tf_sust"] * 1e12) if flops else 0.0
        t_by = byts / (pk["hbm"] * 1e9) if byts else 0.0
        row = {"kernel": key, "cuda_kernel": KERNEL_OF.get(entry, entry), "launches_per_step": len(evs) // max(1, PROFILE_STEPS),
               "avg_launch_ms": round(ms, 5)}
        if flops or byts:
            if t_fl >= t_by:
                row.update(bound="tensor", work=flops, achieved=flops / (ms * 1e-3) / 1e12, peak=pk["tf_sust"], unit="TFLOP/s")
            else:
                row.update(bound="hbm", work=byts, achieved=byts / (ms * 1e-3) / 1e9, peak=pk["hbm"], unit="GB/s")
            row["frac"] = row["achieved"] / row["peak"]
            if survey is not None and survey != byts:
                row["work_survey_8d"] = survey
                row["achieved_survey_8d"] = survey / (ms * 1e-3) / 1e9
            if flops and byts:
                row["flops"], row["bytes"] = flops, byts
        else:
            row.update(bound="latency", work=None, achieved=None, peak=None, unit=None, frac=None)
        tr = traffic.get(key)
        if tr:
            row["traffic"] = tr
            if byts:
                row["traffic_ratio"] = tr / byts
        rows.append(row)
    rows.sort(key=lambda r: -r["avg_launch_ms"] * r["launches_per_step"])
    return rows


PROFILE_STEPS = 3


def load_traffic():
    """{kernel key: DRAM bytes per launch} from the committed ncu capture of the headline step (tools/make_profiles.py)."""
    p = os.path.join(ROOT, "profiles", "traffic_r2.json")
    if os.path.exists(p):
        j = json.load(open(p))
        return j.get("by_bench_key", {}), j.get("clips_per_replay")
    return {}, None


# ------------------------------------------------------------------------------------------------- main arm
def run_ours(args, cfg, rank, world, local):
    assert args.warmup >= 3, "timing rules: at least 3 warm-up steps"
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device: tscd_b200 has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    from tscd_b200 import _lib as L, ops, weights

    F, Lf, C = cfg["F"], cfg["L"], cfg["C"]
    B = args.clips or cfg["clips"]
    R = args.replays or cfg["replays"]
    nsets = max(2, args.sets)
    st, run = make_runner(cfg, dev)
    te = torch.cat([weights.timing_signal_1d(torch.arange(Lf), 256)] * B, 0).to(dev)
    sets = [synth_s1(cfg, B, dev, seed=2024 + 100 * i + rank, layout=args.head_layout) for i in range(nsets)]
    views = [views_of(s_, ops, C) for s_ in sets]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- eager warm-up (lazy module loading, attribute setting), capacity check ----
    for i in range(2):
        out = run(views[i % nsets], B, te)
    torch.cuda.synchronize()
    if int(out["status"].item()) != 0:
        raise RuntimeError("the stage reported a capacity error on the benchmark inputs")
    counts = out["sel"]["sel_count"].cpu().tolist()
    cand_counts = out["sel"]["cand"]["count"].cpu().tolist()
    L.launch_count = 0
    h0 = time.perf_counter()
    out = run(views[0], B, te)
    host_ms = 1e3 * (time.perf_counter() - h0)
    launches_per_replay = L.launch_count
    torch.cuda.synchronize()

    # ---- one CUDA graph per input set (the stage has no host sync) ----
    graphs, graph_outs = [], []
    if not args.no_graph:
        try:
            for i in range(nsets):
                g, g_out = st.capture_fn(lambda i=i: run(views[i], B, te)) if hasattr(st, "capture_fn") else _capture(lambda i=i: run(views[i], B, te), dev)
                graphs.append(g)
                graph_outs.append(g_out)
            torch.cuda.synchronize()
        except Exception as e:   # noqa: BLE001
            sys.stderr.write(f"CUDA graph capture failed ({e}); timing eager launches\n")
            graphs, graph_outs = [], []
            torch.cuda.synchronize()

    def step():
        for r in range(R):
            if graphs:
                graphs[r % nsets].replay()
                res = graph_outs[r % nsets]
            else:
                res = run(views[r % nsets], B, te)
        return res

    for _ in range(args.warmup):
        step()
    # ---- timed region ----
    clocks = ClockSampler(local)
    clocks.start()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    last = None
    e0.record()
    for _ in range(args.steps):
        last = step()
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    clk = clocks.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, caller_arrays(cfg, last, B))
    if world > 1:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    clips_per_step = B * R
    value = world * clips_per_step * F * args.steps / (ms / 1e3)

    # ---- per-kernel durations, measured live right after the timed region: the same launch sequence run eagerly on the
    #      launching stream with CUDA events around every kernel launch (inside a graph replay launches cannot be bracketed) ----
    L.profile = {"names": None, "events": {}}
    st.serialize = True          # no concurrent side stream in this pass: every kernel is timed alone
    for i in range(PROFILE_STEPS):
        run(views[i % nsets], B, te)
    torch.cuda.synchronize()
    st.serialize = False
    events = L.profile["events"]
    linear_info = [(M, N, K, None if md is None else int(md.item()), tag, o16, o32) for (M, N, K, md, tag, o16, o32) in L.profile.get("linear", [])]
    L.profile = None
    inp_mib = nbytes(sets[0]) / 2**20
    launch_mode = "cuda_graph" if graphs else "eager"

    # ---- e2e: host (pinned) inputs -> detections on the host ----
    e2e = None
    if not cfg.get("gen1") and not args.no_e2e:
        del graphs, graph_outs, last, sets, views, out
        torch.cuda.empty_cache()
        e2e = run_e2e(args, cfg, st, dev, rank, world, dist, barrier)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return None
    pk = peaks()
    traffic, traffic_clips = load_traffic()
    rows = kernel_rows(cfg, events, linear_info, counts, cand_counts, B, pk,
                       traffic if (args.config == "ovis_a_k30" and B == traffic_clips and args.head_layout == "rows") else {})
    serial_ms = sum(r["avg_launch_ms"] * r["launches_per_step"] for r in rows)
    for r in rows:
        r["share_of_serialised_step"] = round(r["avg_launch_ms"] * r["launches_per_step"] / serial_ms, 4)
    top = rows[0]
    roof = {"kernel": top["kernel"], "cuda_kernel": top["cuda_kernel"], "bound": top["bound"] if top["bound"] != "latency" else "hbm",
            "achieved": top["achieved"], "peak": top["peak"], "unit": top["unit"], "frac": top["frac"], "traffic": top.get("traffic"),
            "avg_launch_ms": top["avg_launch_ms"], "launches_per_step": top["launches_per_step"] * R,
            "share_of_step": top["share_of_serialised_step"],
            "peak_source": pk["src"] + ", sustained (steps are >= 100 ms of back-to-back GPU work)",
            "note": "dominant = largest time per replay among single kernels (launches of identical role averaged); durations measured with CUDA "
                    "events around each launch of an eager pass right after the timed region; `kernels` lists every kernel of the replay",
            "traffic_source": "profiles/traffic_r2.json (ncu dram__bytes_read.sum + dram__bytes_write.sum per launch)" if top.get("traffic") else None,
            "serialised_kernel_ms_per_replay": round(serial_ms, 4), "replay_ms": ms / args.steps / R}
    line = {"metric": METRIC, "value": value, "unit": "clip-frames/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f16", "data": "synthetic",
            "config": {"workload": cfg["workload"], "name": args.config, "clips_per_gpu_per_step": clips_per_step,
                       "clips_per_graph_replay": B, "graph_replays_per_step": R, "input_sets": nsets,
                       "proposals_per_frame": {"min": min(counts), "mean": round(sum(counts) / len(counts), 1), "max": max(counts)},
                       "seam": SEAMS[args.head_layout],
                       "l2": f"{nsets} rotating input sets of {inp_mib:.0f} MiB each (>> the 126 MB L2); no flush needed",
                       "parallelism": f"clip-parallel x{world}, no collective"},
            "clocks": clk, "gpu_launches": launches_per_replay * R * args.steps, "launch_mode": launch_mode,
            "host_ms_per_eager_replay": host_ms, "roofline": roof, "kernels": rows}
    if e2e is not None:
        line["e2e"] = e2e
    return line


def _capture(fn, dev):
    s = torch.cuda.Stream(device=dev, priority=-1)
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(2):
            fn()
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=s):
        out = fn()
    return g, out


def _host_info():
    """CPU budget of this container (the host-buffer path has a host part: one thread)."""
    info = {"cpu_count": os.cpu_count(), "torch_threads": torch.get_num_threads()}
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            info["cgroup_cpu"] = open(path).read().strip()
            break
        except OSError:
            pass
    return info


def run_e2e(args, cfg, st, dev, rank, world, dist, barrier):
    """Every step: H2D of what the kernels consume (copy stream, chunk-pipelined with compute), zero-copy gather of the kept
    proposals' feature rows out of the pinned feature planes, one D2H of the padded detections per chunk."""
    from tscd_b200 import weights
    F, Lf = cfg["F"], cfg["L"]
    Be = args.e2e_clips or min(32, cfg["clips"])
    dev_src = synth_s1(cfg, Be, dev, seed=99 + rank, layout=args.head_layout)
    host = {k: [(torch.empty(t.shape, dtype=t.dtype, pin_memory=True, memory_format=torch.channels_last) if t.dim() == 4 else
                 torch.empty(t.shape, dtype=t.dtype, pin_memory=True)).copy_(t) for t in v]
            for k, v in dev_src.items()}
    del dev_src
    torch.cuda.empty_cache()
    te_e = torch.cat([weights.timing_signal_1d(torch.arange(Lf), 256)] * Be, 0).pin_memory()

    depth = max(1, args.e2e_depth)

    def submit(i):
        return st.forward_host_submit(host, HW, te_e, Be, F, Lf, chunk_clips=args.e2e_chunk, slot=i % depth)

    for i in range(2 * depth):                                        # warm-up: builds / captures every slot's plan ...
        res, res_ori, h2d, d2h = st.forward_host_collect(submit(i))
    tw0, i = time.perf_counter(), 2 * depth
    while time.perf_counter() - tw0 < 0.5:                            # ... then keeps the GPU and the PCIe link busy for half a second
        res, res_ori, h2d, d2h = st.forward_host_collect(submit(i))   # (the pinned allocation above left them idle for seconds:
        i += 1                                                        # P-state / link speed ramp up)
    warm_calls = i
    # latency of one synchronous call (submit + collect, nothing else in flight)
    call_ms, call_split = [], []
    for i in range(3):
        tc0 = time.perf_counter()
        ticket = submit(i)
        tc1 = time.perf_counter()
        tm = {}
        st.forward_host_collect(ticket, timing=tm)
        call_ms.append(round(1e3 * (time.perf_counter() - tc0), 3))
        call_split.append({"submit": round(1e3 * (tc1 - tc0), 3), "wait": round(tm["wait"], 3), "unpack": round(tm["unpack"], 3)})
    import gc
    gc.collect()                       # the main arm left graphs / input sets behind: collect before, not inside, the timed region
    barrier()
    link = ClockSampler(torch.cuda.current_device(), extra="pstate,pcie.link.gen.current,pcie.link.width.current", period_ms=25)
    link.start()
    t0 = time.perf_counter()
    e2e_calls = args.steps * depth                                   # --steps steps of `depth` calls each
    # throughput: `depth` calls in flight (double buffering): the PCIe phases of step i+1 overlap the compute tail and the host-side
    # unpacking of step i.  Every step's copies, kernels, read-back and unpacking happen inside the timed region.
    inflight = []
    for i in range(e2e_calls):
        inflight.append(submit(i))
        if len(inflight) == depth:
            res, res_ori, h2d, d2h = st.forward_host_collect(inflight.pop(0))
    while inflight:
        res, res_ori, h2d, d2h = st.forward_host_collect(inflight.pop(0))
    barrier()
    e2e_s = time.perf_counter() - t0
    link_state = link.stop()
    if world > 1:
        t = torch.tensor([e2e_s], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())
    # where a call spends its time: GPU time of the captured launch sequence (events around one replay) vs the whole call
    gpu_ms = None
    plans = getattr(st, "_host_plans", {})
    if plans and list(plans.values())[-1]["graph"] is not None:
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        ev0.record()
        list(plans.values())[-1]["graph"].replay()
        ev1.record()
        torch.cuda.synchronize()
        gpu_ms = ev0.elapsed_time(ev1)
    return {"value": world * Be * F * e2e_calls / e2e_s, "unit": "clip-frames/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
            "ms_per_call": 1e3 * e2e_s / e2e_calls, "gpu_ms_per_call": gpu_ms, "sync_call_ms": call_ms, "sync_call_split_ms": call_split, "plans_built": getattr(st, "host_plan_builds", None), "host": _host_info(), "warmup_calls": warm_calls, "gpu_state": link_state,
            "clips_per_gpu_per_step": Be, "chunk_clips": args.e2e_chunk, "steps": args.steps, "calls": e2e_calls, "calls_in_flight": depth,
            "host_resident_input_bytes_per_step": nbytes(host),
            "note": "inputs are pinned HOST tensors; h2d counts the copied logits plus the rows read in place over PCIe"}


def run_sweep(args, rank, world, local):
    """configs[4]: P x K sweep, one JSON line per point (value only) and a summary line."""
    base = CONFIGS["ovis_a_k30"]
    points = []
    args.no_e2e = True
    for P in SWEEP_P:
        for K in SWEEP_K:
            cfg = dict(base, pre_k=P, top_k=K, workload=f"sweep point: pre-NMS top-{P} -> {K} proposals/frame, 64 clips x 32 frames per replay")
            a = argparse.Namespace(**vars(args))
            a.replays, a.warmup = args.replays or 4, 3
            line = run_ours(a, cfg, rank, world, local)
            if line is not None:
                pt = {"P": P, "K": K, "value": line["value"], "ms_per_replay": line["ms_per_step"] / a.replays,
                      "top_kernel": line["roofline"]["kernel"], "top_share": line["roofline"]["share_of_step"]}
                points.append(pt)
                print(json.dumps({"sweep_point": pt}), flush=True)
            torch.cuda.empty_cache()
    if rank == 0:
        print(json.dumps({"metric": METRIC, "unit": "clip-frames/s", "n_gpus": world, "config": {"name": "sweep", "workload": "64 clips x 32 frames, P x K"},
                          "sweep": points}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20, help="timed steps; the e2e leg times as many steps of --e2e-depth calls, "
                    "the sweep as many steps per point")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "reference-gpu"])
    ap.add_argument("--config", default="ovis_a_k30", choices=list(CONFIGS) + ["sweep"])
    ap.add_argument("--mode", default="clips", choices=["clips", "long-clip"])
    ap.add_argument("--clips", type=int, default=0, help="clips per GPU per graph replay (default: per config; 148 = one per SM for the headline)")
    ap.add_argument("--replays", type=int, default=0, help="graph replays per step (default: per config; 28 for the headline)")
    ap.add_argument("--sets", type=int, default=2, help="rotating input sets resident in HBM")
    ap.add_argument("--e2e-clips", type=int, default=0)
    ap.add_argument("--e2e-chunk", type=int, default=8, help="clips per pipelined chunk of the host-buffer path")
    ap.add_argument("--e2e-depth", type=int, default=4, help="forward_host calls kept in flight by the e2e loop (1 = synchronous calls)")
    ap.add_argument("--cpu-clips", type=int, default=6, help="clips timed for cpu_baseline (rank 0, N=1)")
    ap.add_argument("--head-layout", default="rows", choices=["rows", "levels"],
                    help="rows: fused 64-byte head rows + objectness plane (what the drop-in head emits); levels: per-level channels_last conv outputs")
    ap.add_argument("--no-graph", action="store_true", help="launch eagerly instead of replaying CUDA graphs")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline / reference-gpu legs")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last graph replay of the last step "
                    "returned to its caller as DIR/<name>.npy (float32 / float64, at most 64,000,000 bytes; rank 0 only); inputs are seeded, "
                    "so runs with the same arguments can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.mode != "clips" or args.config == "sweep" or args.impl != "ours"):
        ap.error("--dump-outputs applies to the timed stage: --impl ours, --mode clips, a single --config")
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    if args.mode == "long-clip":
        import bench_long_clip
        bench_long_clip.main(args, rank, world, local)
        return
    if args.config == "sweep":
        run_sweep(args, rank, world, local)
        return
    cfg = CONFIGS[args.config]
    if args.impl == "reference":
        run_reference(args, cfg, rank)
        return
    if args.impl == "reference-gpu":
        if rank == 0:
            torch.cuda.set_device(local)
            print(json.dumps({"impl": "reference-gpu", "metric": METRIC, "unit": "clip-frames/s", "config": {"name": args.config, "workload": cfg["workload"]},
                              "value": reference_gpu_eager(cfg, torch.device("cuda", local))}))
        return
    line = run_ours(args, cfg, rank, world, local)
    if line is None:
        return
    if world == 1 and not args.no_cpu:
        fps, dt, thr, kind, sample = cpu_reference_sample(cfg, args.cpu_clips)
        line["cpu_baseline"] = {"value": fps, "unit": "clip-frames/s", "cores": thr, "kind": kind, "sample": sample}
        if reference_available() and not cfg.get("gen1"):
            line["reference_gpu_eager"] = {"unit": "clip-frames/s", "value": reference_gpu_eager(cfg, torch.device("cuda", local)),
                                           "note": "the stock reference forward from the seam, eager PyTorch on this B200, 1 clip per call (the incumbent GPU path)"}
    print(json.dumps(line))
    if world > 1:
        import torch.distributed as dist
        if dist.is_initialized():
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
