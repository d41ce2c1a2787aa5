"""Frame store measurements on one GPU: per-clip forward against ingest-once + forward_clips.

  python tools/bench_frame_store.py [--configs ovis_a_k30,ovis_l_modeB,vid_l_c30] [--videos V] [--frames N] [--clips B]
                                    [--replays R] [--out DIR]

Per configuration (bench.py CONFIGS: shapes, selection, synthetic seam-S1 inputs in the fused-row layout), one JSON line:
* workload: V seeded videos of N frames (576 x 576, 6804 anchors; 10.9 MB of head rows + feature planes per frame, GBs in all,
  far above the 126 MB L2), cut into clips by clips.demo_clips with a seeded rng (globals drawn from the whole video);
* per_clip: forward() on clip tensors materialised with index_select, CUDA-graph replays timed with device events exactly as
  bench.py times them (two input sets, each a different batch of B clips);
* store: ingest_frames of every frame of every video (`--ingest-chunk` frames per call; eager, and captured into one CUDA
  graph), then forward_clips CUDA-graph replays of the same two batches; `total_clip_frames_per_s` charges the whole graph
  ingest to the workload's clip-frames;
* assemble: tscd_clip_assemble alone (events around `--asm-iters` launches into preallocated outputs), its algorithmic bytes
  (rows and counts read from the store + written to the clip bank, computed from the counts) and GB/s against 7.7 TB/s;
* host: ingest_host_frames of the first video from pinned memory, H2D bytes per clip-frame against forward_host's bytes for
  the same clips (the same accounting forward_host reports: copied planes + rows read in place), and whether the store equals
  the device-ingested one;
* identical: to_lists detections, sel_count, row_off and bank rows of the timed replays, per_clip vs store.
The card's name and power limit are read in the same run."""
import argparse
import json
import os
import random
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402

HBM_PEAK_GBS = 7700.0      # HGX B200 data sheet, one GPU (at 1000 W)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
        name, pl, clk = [x.strip() for x in q.split(",")]
        return {"name": name, "power_limit": pl, "max_sm_clock": clk}
    except Exception as e:     # noqa: BLE001
        return {"name": torch.cuda.get_device_name(0), "power_limit": f"unavailable ({e})"}


def pick(inp, idx):
    """Clip tensors from per-frame tensors: rows / objp by index_select, feature planes keep their channels_last layout."""
    out = {k: [t.index_select(0, idx)] for k, t in (("rows", inp["rows"][0]), ("objp", inp["objp"][0]))}
    for k in ("f_cls", "f_reg", "f_edge"):
        out[k] = [t.permute(0, 2, 3, 1).index_select(0, idx).permute(0, 3, 1, 2) for t in inp[k]]
    return out


def timed_replays(graphs, R, steps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(2):
        for r in range(R):
            graphs[r % len(graphs)].replay()
    torch.cuda.synchronize()
    e0.record()
    for _ in range(steps):
        for r in range(R):
            graphs[r % len(graphs)].replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def same_out(st, a, b, B, L):
    sa, sb = a["sel"], b["sel"]
    if not (torch.equal(sa["sel_count"], sb["sel_count"]) and torch.equal(sa["row_off"], sb["row_off"])):
        return False
    n = int(sa["row_off"][-1])
    if not all(torch.equal(sa[k][:n], sb[k][:n]) for k in ("bank_cls", "bank_reg", "bank_edge", "bank_score")):
        return False
    ra, rb = st.to_lists(a, B, L), st.to_lists(b, B, L)
    eq = lambda x, y: all((p is None) == (q is None) and (p is None or torch.equal(p, q)) for p, q in zip(x, y))  # noqa: E731
    return eq(ra[0], rb[0]) and eq(ra[1], rb[1])


def run_config(name, args, dev):
    from tscd_b200 import clips, frames, ops
    cfg = bench.CONFIGS[name]
    C, F, L = cfg["C"], cfg["F"], cfg["L"]
    G = F - L
    st, _ = bench.make_runner(cfg, dev)
    an = ops.AnchorSpec(bench.HW)
    kmax = st.cfg.selection.max_keep(an.num_anchors)
    V, N = args.videos, args.frames
    inp = bench.synth_s1(dict(cfg, F=N), V, dev, seed=4242, layout="rows")       # V*N frames, video-major
    rng = random.Random(2026)
    per_video = [clips.demo_clips(N, L, G, rng=rng) for _ in range(V)]
    all_clips = [([v * N + f for f in c], p) for v, (cl, pa) in enumerate(per_video) for c, p in zip(cl, pa)]
    workload_cf = len(all_clips) * F
    B = min(args.clips or cfg["clips"], len(all_clips) // 2)
    batches = [all_clips[i * B:(i + 1) * B] for i in range(2)]
    tes = [torch.cat([clips.time_embedding(p) for _, p in b], 0).to(dev) for b in batches]

    # ---- per-clip forward over materialised clip tensors (graph replays, as bench.py) ----
    sets = [pick(inp, torch.tensor([f for c, _ in b for f in c], device=dev)) for b in batches]
    views = [bench.views_of(s, ops, C) for s in sets]
    g_ref, o_ref = zip(*[st.capture_fn(lambda i=i: st.forward(views[i][0], views[i][1], torch.float16, tes[i], B, F, L)) for i in range(2)])
    ms_ref = timed_replays(g_ref, args.replays, args.steps)
    ref_cf_s = B * F * args.replays * args.steps / (ms_ref / 1e3)

    # ---- ingest once + forward_clips ----
    store = frames.FrameStore(V * N, kmax, C)
    head_all, feats_all = bench.views_of(inp, ops, C)
    slots_all = torch.arange(V * N, dtype=torch.int32, device=dev)
    st.ingest_frames(store, head_all, feats_all, torch.float16, slots_all)       # warm-up (module loading)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    chunk = args.ingest_chunk
    e0.record()
    for f0 in range(0, V * N, chunk):
        sub = {k: [t[f0:f0 + chunk] for t in v] for k, v in inp.items()}
        h, fe = bench.views_of(sub, ops, C)
        st.ingest_frames(store, h, fe, torch.float16, slots_all[f0:f0 + chunk])
    e1.record()
    torch.cuda.synchronize()
    ingest_ms = e0.elapsed_time(e1)
    if int((store.status != 0).sum()) or int((store.count < 0).sum()):
        raise RuntimeError("ingest reported a capacity error / left a slot unwritten")
    # the same ingest captured into one CUDA graph (device slot tensor: nothing is read back), as a caller would replay it
    g_ing, _ = st.capture_fn(lambda: [st.ingest_frames(store, *bench.views_of({k: [t[f0:f0 + chunk] for t in v] for k, v in inp.items()},
                                                                              ops, C), torch.float16, slots_all[f0:f0 + chunk])
                                      for f0 in range(0, V * N, chunk)])
    ingest_graph_ms = timed_replays([g_ing], 1, args.steps) / args.steps
    slot_t = [torch.tensor([c for c, _ in b], dtype=torch.int32, device=dev) for b in batches]
    g_new, o_new = zip(*[st.capture_fn(lambda i=i: st.forward_clips(store, slot_t[i], L, tes[i])) for i in range(2)])
    ms_new = timed_replays(g_new, args.replays, args.steps)
    new_cf_s = B * F * args.replays * args.steps / (ms_new / 1e3)
    identical = all(same_out(st, o_ref[i], o_new[i], B, L) for i in range(2))
    total_s = ingest_graph_ms / 1e3 + workload_cf / new_cf_s

    # ---- tscd_clip_assemble alone ----
    status = torch.zeros(1, dtype=torch.int32, device=dev)
    row_cap = (B * F * kmax + 127) // 128 * 128 + 128
    asm_out = ops.clip_assemble(store, slot_t[0], B, F, L, row_cap, status)
    torch.cuda.synchronize()
    cnt = asm_out["sel_count"].tolist()
    W = 7 + C
    rows_all = sum(cnt)
    rows_loc = sum(c for i, c in enumerate(cnt) if i % F < L)
    nbytes = 2 * rows_all * (3 * 512 + 4 + 4) + 2 * rows_loc * W * 4 + B * F * (4 + 8 + 4 + 4) + 4
    for _ in range(3):
        ops.clip_assemble(store, slot_t[0], B, F, L, row_cap, status, out=asm_out)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(args.asm_iters):
        ops.clip_assemble(store, slot_t[0], B, F, L, row_cap, status, out=asm_out)
    e1.record()
    torch.cuda.synchronize()
    asm_us = 1e3 * e0.elapsed_time(e1) / args.asm_iters
    asm_gbs = nbytes / (asm_us * 1e-6) / 1e9

    # ---- host ingest of the first video (pinned) vs forward_host's bytes for its clips ----
    host = {}
    for k, v in inp.items():
        host[k] = [(torch.empty(t[:N].shape, dtype=t.dtype, pin_memory=True, memory_format=torch.channels_last) if t.dim() == 4 else
                    torch.empty(t[:N].shape, dtype=t.dtype, pin_memory=True)).copy_(t[:N]) for t in v]
    hstore = frames.FrameStore(N, kmax, C)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    hsel, copied = st.ingest_host_frames(hstore, host, bench.HW, list(range(N)))
    torch.cuda.synchronize()
    host_ms = 1e3 * (time.perf_counter() - t0)
    mode_a = cfg["mode"] == "A"
    row_b = host["rows"][0].shape[2] * 2
    sel_c = hsel["sel_count"].tolist()
    cand_c = hsel["cand"]["count"].tolist()
    per_frame = [host["objp"][0][0].numel() * 2 + (0 if mode_a else host["rows"][0][0].numel() * 2) + sel_c[f] * 3 * 512 +
                 ((cand_c[f] + sel_c[f]) * row_b if mode_a else 0) for f in range(N)]
    v0 = [c for c, _ in all_clips[:len(per_video[0][0])]]
    clip_bytes = sum(per_frame[f] for c in v0 for f in c) / (len(v0) * F)
    store_bytes = sum(per_frame) / (len(v0) * F)
    host_equal = torch.equal(hstore.count, store.count[:N]) and all(
            torch.equal(getattr(hstore, k)[f, :sel_c[f]], getattr(store, k)[f, :sel_c[f]])
            for f in range(N) for k in ("bank_cls", "bank_reg", "bank_edge", "bank_score", "sel_idx", "sel_rows"))
    assert copied == sum(host[k][0].numel() * 2 for k in (("objp",) if mode_a else ("objp", "rows")))
    del host, hstore

    return {"metric": "frame store: clip-frames/s, per-clip forward vs ingest once + forward_clips", "config": name,
            "workload": f"{V} videos x {N} frames, demo_clips L {L} / G {G} -> {len(all_clips)} clips ({workload_cf} clip-frames, "
                        f"{workload_cf / (V * N):.1f} per video frame); {B} clips per graph replay, 2 batches alternated",
            "kmax": kmax, "store_mb": round(store.flat.numel() / 2**20, 1),
            "proposals_per_frame": {"min": min(sel_c), "mean": round(sum(sel_c) / N, 1), "max": max(sel_c)},
            "per_clip": {"clip_frames_per_s": round(ref_cf_s), "replay_ms": round(ms_ref / args.steps / args.replays, 4)},
            "store": {"clip_frames_per_s_replay": round(new_cf_s), "replay_ms": round(ms_new / args.steps / args.replays, 4),
                      "ingest_ms_eager": round(ingest_ms, 3), "ingest_ms_graph": round(ingest_graph_ms, 3),
                      "ingest_frames_per_s_graph": round(V * N / (ingest_graph_ms / 1e3)),
                      "total_clip_frames_per_s": round(workload_cf / total_s),
                      "speedup_total": round(workload_cf / total_s / ref_cf_s, 3)},
            "assemble": {"us": round(asm_us, 2), "bytes": nbytes, "gbs": round(asm_gbs, 1), "frac_of_hbm_peak": round(asm_gbs / HBM_PEAK_GBS, 3),
                         "clip_frames": B * F, "rows": rows_all,
                         "note": "algorithmic bytes: rows + counts read from the store and written to the clip bank"},
            "host": {"h2d_bytes_per_clip_frame_forward_host": round(clip_bytes), "h2d_bytes_per_clip_frame_store": round(store_bytes),
                     "ingest_ms_first_video": round(host_ms, 2), "store_equals_device_ingest": bool(host_equal)},
            "identical": bool(identical)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="ovis_a_k30,ovis_l_modeB,vid_l_c30")
    ap.add_argument("--videos", type=int, default=2)
    ap.add_argument("--frames", type=int, default=200)
    ap.add_argument("--clips", type=int, default=0, help="clips per graph replay (default: bench.py's, at most half the workload)")
    ap.add_argument("--replays", type=int, default=8)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--asm-iters", type=int, default=50)
    ap.add_argument("--ingest-chunk", type=int, default=200, help="frames per ingest_frames call")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise RuntimeError("bench_frame_store.py needs a CUDA device: tscd_b200 has no CPU fallback")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    c = card()
    lines = []
    for name in args.configs.split(","):
        line = run_config(name, args, dev)
        line["card"] = c
        print(json.dumps(line), flush=True)
        lines.append(line)
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "bench_frame_store.jsonl"), "w") as f:
            f.write("".join(json.dumps(x) + "\n" for x in lines))


if __name__ == "__main__":
    main()
