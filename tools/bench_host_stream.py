#!/usr/bin/env python
"""Streaming videos through the host-buffer path: what the CAFM memory costs.

  python tools/bench_host_stream.py [--configs ovis_a_k30,ovis_l_modeB] [--clips 32] [--calls 24] [--depths 1,4] [--out FILE]

Synthetic videos (a fixed mix of clips per video) are scheduled by clips.ClipScheduler, one CAFMState slot per concurrent
video, and streamed through AggregationStage.forward_host_submit / forward_host_collect with bench.synth_s1 inputs in pinned
memory (the e2e leg of bench.py, fused head layout).  Every call is run twice on the same inputs and schedule: stateless (every
clip starts a new video) and stateful (state=pool, resume / state_slots of the schedule: the CAFM phases of the calls on the
pool are serialised in submission order).  Legs alternate, and the whole set is repeated, so the spread is visible.
Reports wall ms per call and clip-frames/s with `depth` calls in flight, and the GPU time of one call (CUDA events around one
graph replay).  The card's name and power limit are printed with the numbers."""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402

CLIPS_PER_VIDEO = [1, 2, 3, 5, 8, 4, 2, 6]      # cycled over the synthetic videos


def card():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit, max_sm_clock"] = q
    except (OSError, subprocess.SubprocessError) as e:
        info["power_limit, max_sm_clock"] = f"unavailable ({e.__class__.__name__})"
    return info


def schedule(B, n_calls, Lf):
    """The first n_calls full batches (B clips of B different videos) of a ClipScheduler over enough videos."""
    from tscd_b200 import clips
    per_video, v = [], 0
    while sum(len(x) for x in per_video) < 2 * B * n_calls:
        n = CLIPS_PER_VIDEO[v % len(CLIPS_PER_VIDEO)]
        per_video.append([([], list(range(c * Lf, (c + 1) * Lf))) for c in range(n)])
        v += 1
    out = []
    for batch in clips.ClipScheduler(per_video, world=1, slots=B).batches(0):
        if len(batch) < B or len(out) == n_calls:
            break
        out.append(batch)
    assert len(out) == n_calls
    return out


def run_leg(st, host, te, B, F, Lf, chunk, batches, depth, pool):
    def submit(i, batch):
        kw = {}
        if pool is not None:
            kw = dict(state=pool, resume=[c.resume for c in batch], state_slots=[c.slot for c in batch])
        return st.forward_host_submit(host, bench.HW, te, B, F, Lf, chunk_clips=chunk, slot=i % depth, **kw)

    for i in range(2 * depth):                          # builds / captures every slot's plan, warms the link
        st.forward_host_collect(submit(i, batches[i % len(batches)]))
    torch.cuda.synchronize()
    inflight = []
    t0 = time.perf_counter()
    for i, batch in enumerate(batches):
        inflight.append(submit(i, batch))
        if len(inflight) == depth:
            st.forward_host_collect(inflight.pop(0))
    while inflight:
        st.forward_host_collect(inflight.pop(0))
    ms = 1e3 * (time.perf_counter() - t0) / len(batches)
    # GPU time of one call: events around one replay of the slot-0 plan's graph, nothing else in flight
    ticket = submit(0, batches[0])
    st.forward_host_collect(ticket)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    gpu = []
    for _ in range(3):
        torch.cuda.synchronize()
        e0.record()
        ticket["graph"].replay()
        e1.record()
        torch.cuda.synchronize()
        gpu.append(e0.elapsed_time(e1))
    return ms, min(gpu)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="ovis_a_k30,ovis_l_modeB")
    ap.add_argument("--clips", type=int, default=32, help="clips per call (concurrent videos = CAFMState slots)")
    ap.add_argument("--calls", type=int, default=24, help="timed calls per leg")
    ap.add_argument("--depths", default="1,4")
    ap.add_argument("--chunk", type=int, default=8)
    ap.add_argument("--repeats", type=int, default=2)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_host_stream.py measures the GPU path; no CUDA device found")
    from tscd_b200 import ops, stage, weights
    dev = torch.device("cuda", 0)
    info = card()
    print(json.dumps({"card": info}), flush=True)
    results = []
    for name in args.configs.split(","):
        cfg = dict(bench.CONFIGS[name])
        F, Lf, B = cfg["F"], cfg["L"], args.clips
        st, _ = bench.make_runner(cfg, dev)
        src = bench.synth_s1(cfg, B, dev, seed=99, layout="rows")
        host = {k: [(torch.empty(t.shape, dtype=t.dtype, pin_memory=True, memory_format=torch.channels_last) if t.dim() == 4 else
                     torch.empty(t.shape, dtype=t.dtype, pin_memory=True)).copy_(t) for t in v] for k, v in src.items()}
        del src
        torch.cuda.empty_cache()
        te = torch.cat([weights.timing_signal_1d(torch.arange(Lf), 256)] * B, 0).pin_memory()
        kmax = st.cfg.selection.max_keep(ops.AnchorSpec(bench.HW).num_anchors)
        pool = stage.CAFMState(B, kmax, 256, dev)
        batches = schedule(B, args.calls, Lf)
        resumed = sum(c.resume for b in batches for c in b) / (B * len(batches))
        for rep in range(args.repeats):
            for depth in (int(x) for x in args.depths.split(",")):
                for stateful in (False, True):
                    ms, gpu = run_leg(st, host, te, B, F, Lf, args.chunk, batches, depth, pool if stateful else None)
                    r = dict(config=name, clips=B, depth=depth, stateful=stateful, repeat=rep, ms_per_call=round(ms, 3),
                             clip_frames_per_s=round(B * F / ms * 1e3), gpu_ms_per_call=round(gpu, 3),
                             resumed_fraction=round(resumed, 3))
                    results.append(r)
                    print(json.dumps(r), flush=True)
        st._host_plans.clear()
        del host, pool
        torch.cuda.empty_cache()
    print(json.dumps({"card": info}), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        json.dump({"card": info, "results": results}, open(args.out, "w"), indent=1)


if __name__ == "__main__":
    main()
