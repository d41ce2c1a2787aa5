"""Wide-tier measurements (SelectionConfig.max_proposals 2048) on one GPU.

  python tools/bench_wide.py [--clips B] [--steps K] [--out DIR]

* workload: VID TSCD-L shape (576 x 576 = 6804 anchors, 30 classes, F = 16 frames, L = 4 local), fused [F, A, 5+C] head layout, mode B with
  minimal_limit 50 and no maximal_limit; the local frames keep ~800 .. ~2000 proposals, the global ones 50 .. 300.  B clips per
  CUDA-graph replay; reports clip-frames/s (device events around K replays) and, in a separate pass, per-kernel CUDA times from
  torch.profiler;
* LSAP: tscd_cafm_lap on cosine-like tables of 512 / 1024 / 2048 rows (the CTA solver above 512 rows, the one-warp solver at
  512) beside scipy.optimize.linear_sum_assignment on the same tables on this host's CPU.
The card's name and power limit are written next to the numbers."""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import oracle  # noqa: E402

HW = [(72, 72), (36, 36), (18, 18)]


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                              text=True, timeout=30).stdout.strip()
    except Exception as e:  # pragma: no cover
        return f"unknown ({e})"


def wide_workload(B, steps, warmup, prof_dir):
    from tscd_b200 import ops, selection, stage
    C, F, Lf = 30, 16, 4
    sd = oracle.init_stage_weights(C, dim=256, seed=17)
    cfg = stage.StageConfig(num_classes=C, selection=selection.SelectionConfig(mode="B", minimal_limit=50, maximal_limit=0,
                                                                                use_pre_nms=False, max_proposals=2048))
    st = stage.AggregationStage(cfg, sd)
    means = [-7.75, -9.0, -8.4, -8.8] + [-10.5, -11.0, -9.9] * 4
    heads, planes = [], [[], [], []]
    for b in range(B):
        h, f = oracle.synth_head_outputs(F, HW, C, dim=256, seed=900 + b, clustered=True, obj_mean=means[:F], n_obj=3, n_mem=10)
        heads.append(oracle.decode_outputs(h, HW, [8, 16, 32]))
        for k in range(3):
            planes[k].append(f[k].half())
    an = ops.AnchorSpec(HW)
    head = ops.HeadViews.from_fused(torch.cat(heads, 0).cuda(), an, apply_sigmoid=False, apply_decode=False)
    views = tuple(ops.view_rowmajor(torch.cat(p, 0).cuda().contiguous(), an) for p in planes)
    te = torch.cat([oracle.timing_signal_1d(torch.arange(Lf), 256)] * B, 0)
    graph, out = st.capture(head, views, torch.float16, te, B, F, Lf, warmup=warmup)
    for _ in range(warmup):
        graph.replay()
    torch.cuda.synchronize()
    counts = out["sel"]["sel_count"].view(B, F)[:, :Lf].cpu()
    assert int(out["status"].item()) == 0, "capacity status set"
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        graph.replay()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    res = dict(clips=B, F=F, L=Lf, local_proposals=counts.tolist(), ms_per_replay=ms, clip_frames_per_s=B * F / (ms / 1e3))
    # per-kernel times: separate profiled pass (eager launches, profiler on)
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as p:
        st.forward(head, views, torch.float16, te, B, F, Lf)
        torch.cuda.synchronize()
    rows = sorted(((e.key, e.device_time_total / 1e3, e.count) for e in p.key_averages() if e.device_time_total > 0),
                  key=lambda r: -r[1])
    res["kernels_ms"] = [dict(name=k[:120], ms=round(t, 4), calls=c) for k, t, c in rows[:25]]
    if prof_dir:
        p.export_chrome_trace(os.path.join(prof_dir, "bench_wide_trace.json"))
    return res


def lap_bench():
    from scipy.optimize import linear_sum_assignment
    from tscd_b200 import _lib as L, ops
    out = []
    g = torch.Generator().manual_seed(4)
    for n in (512, 1024, 2048):
        a = torch.nn.functional.normalize(torch.randn(n, 64, generator=g), dim=1)
        b = torch.nn.functional.normalize(torch.randn(n, 64, generator=g), dim=1)
        c = (1.0 - a @ b.t()).contiguous()
        t0 = time.perf_counter()
        ri, ci = linear_sum_assignment(c.double().numpy())
        t_cpu = time.perf_counter() - t0
        cost = torch.zeros(1, n, n)
        cost[0] = c
        dcost = cost.cuda()
        lrow = torch.tensor([0, n], dtype=torch.int32).cuda()
        ref_n = torch.tensor([n], dtype=torch.int32).cuda()
        col = torch.empty(1, n, dtype=torch.int32).cuda()
        row = torch.empty(1, n, dtype=torch.int32).cuda()
        run = lambda: ops.call("tscd_cafm_lap", L.CafmLapArgs, num_frames=1, kmax=n, lrow_off=lrow, ref_n=ref_n, cost=dcost,  # noqa: E731
                               lap_col=col, lap_row=row)
        run()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(3):
            run()
        e1.record()
        torch.cuda.synchronize()
        same = col[0].cpu().tolist() == ci.tolist()             # square table: ri = 0 .. n-1
        out.append(dict(n=n, solver="cta" if n > 512 else "warp", gpu_ms=e0.elapsed_time(e1) / 3, scipy_cpu_ms=t_cpu * 1e3,
                        same_assignment=same))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--clips", type=int, default=4)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None, help="directory for the JSON result and the profiler trace")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_wide.py needs a GPU")
    if a.out:
        os.makedirs(a.out, exist_ok=True)
    res = dict(card=card(), lsap=lap_bench(), workload=wide_workload(a.clips, a.steps, a.warmup, a.out))
    s = json.dumps(res, indent=1)
    print(s)
    if a.out:
        with open(os.path.join(a.out, "bench_wide.json"), "w") as f:
            f.write(s)


if __name__ == "__main__":
    main()
