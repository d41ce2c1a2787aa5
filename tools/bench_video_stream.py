"""VideoStream measurements on one GPU: whole videos from pinned host memory against forward_host per clip.

  python tools/bench_video_stream.py [--configs ovis_a_k30,ovis_l_modeB,vid_l_c30,vid_l_wide] [--videos V] [--frames N]
                                     [--clips-per-slot K] [--groups R] [--out DIR]

Per configuration (bench.py CONFIGS: shapes, selection, seeded synthetic inputs in the fused-row layout; vid_l_wide = vid_l_c30
with max_proposals 2048), one JSON line:
* workload: V videos of N frames (576 x 576, 6804 anchors) in one group, clips from clips.demo_clips with a seeded rng;
* stream: VideoStream(depth 2) submit / collect of R groups, two in flight (buffer sets alternate); wall clock over the R
  groups -> clip-frames/s end to end; how long each group's ingest ran while the previous group's clip calls were running
  (device events); the plan captures after the warm-up and at the end; H2D bytes per clip-frame (copied planes + rows and feature rows read in place, from the
  ingest counts); the device phase split of one group (ingest, clip calls, pack + header copy) and its host split;
* forward_host: the same clips, one clip of every video per call (stateful, resume / state slots of ClipScheduler), two calls in
  flight on two buffer sets (the pinned inputs of the first two batches, alternated; graph replays) -> clip-frames/s; the first
  two calls run on their own frames and their detections are compared with the stream's; not run on the wide tier
  (forward_host is default-tier only), where the device path below is the comparison;
* device: ingest_frames + chained forward_clips of the same group from device-resident frames (eager) -> clip-frames/s, its
  detections compared with the stream's;
* identical: every video's stream table equals pack_detections over the device path run one clip per call, byte for byte.
The card's name and power limit are read in the same run."""
import argparse
import dataclasses
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


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
        name, pl, clk = [x.strip() for x in q.split(",")]
        return {"name": name, "power_limit": pl, "max_sm_clock": clk}
    except Exception as e:     # noqa: BLE001
        return {"name": torch.cuda.get_device_name(0), "power_limit": f"unavailable ({e})"}


def write_staging(buf, inp, f0, n):
    for k in ("rows", "objp"):
        buf[k][0][:n].copy_(inp[k][0][f0:f0 + n])
    for k in ("f_cls", "f_reg", "f_edge"):
        for t, s in zip(buf[k], inp[k]):
            t[:n].copy_(s[f0:f0 + n])


def reference_table(st, store, base, item, L):
    """Device path one clip per call with resume, frame-ordered rows -> pack_detections (host copies)."""
    from tscd_b200 import clips, evalglue, stage
    from tscd_b200.video import local_frames
    pool = stage.CAFMState(1, store.kmax)
    outs = [st.forward_clips(store, [[base + f for f in c]], L, clips.time_embedding(p).cuda(), state=pool, resume=[int(i > 0)],
                             state_slots=[0]) for i, (c, p) in enumerate(zip(item["clips"], item["paths"]))]
    where = local_frames(item["clips"], item["paths"], item["num_frames"])
    rows = torch.stack([outs[c]["det_rows"][l] for c, l in where]).contiguous()
    cnt = torch.stack([outs[c]["det_count"][l] for c, l in where]).contiguous()
    packed, off = evalglue.pack_detections(rows, cnt, torch.tensor(item["ratios"]))
    off = off.cpu()
    return packed[:int(off[-1])].cpu(), off


def same_as_tables(tables, items, batch, result, L):
    """Per-local-frame results of one call (the reference's list layout) against the stream's tables: every frame a clip of
    the batch owns (its first local occurrence) must have the same rows, in packed form (ratio 1)."""
    from tscd_b200.video import local_frames
    for j, c in enumerate(batch):
        where = local_frames(items[c.video]["clips"], items[c.video]["paths"], items[c.video]["num_frames"])
        t = tables[c.video]
        for l in range(L):
            f = c.frames[l]
            if where[f] != (c.clip, l):
                continue
            rows = t["packed"][int(t["offsets"][f]):int(t["offsets"][f + 1])]
            r = result[j * L + l]
            if r is None:
                if rows.shape[0] or int(t["det_cand"][f]):
                    return False
                continue
            r = r.cpu()
            if rows.shape[0] != r.shape[0] or not all(torch.equal(rows[:, a], r[:, b]) for a, b in
                                                       ((1, 0), (2, 1), (8, 2), (9, 3), (7, 4), (10, 5), (6, 6))):
                return False
    return True


def run_config(name, args, dev):
    from tscd_b200 import clips, frames, ops, stage, weights
    from tscd_b200.video import VideoStream
    wide = name.endswith("_wide")
    cfg = bench.CONFIGS["vid_l_c30" if wide else name]
    C, F, L = cfg["C"], cfg["F"], cfg["L"]
    G = F - L
    st, _ = bench.make_runner(cfg, dev)
    if wide:
        sc = dataclasses.replace(st.cfg, selection=dataclasses.replace(st.cfg.selection, max_proposals=2048))
        st = stage.AggregationStage(sc, weights.random_state_dict(C, 256, seed=2024), device=dev)
    V, N = args.videos, args.frames
    inp = bench.synth_s1(dict(cfg, F=N), V, dev, seed=4242, layout="rows")
    rng = random.Random(2026)
    items = []
    for v in range(V):
        cl, pa = clips.demo_clips(N, L, G, rng=rng)
        items.append(dict(first_frame=v * N, num_frames=N, clips=cl, paths=pa, ratios=[1.0] * N))
    cf = sum(len(it["clips"]) for it in items) * F

    # ---- the stream ----
    vs = VideoStream(st, bench.HW, max_frames=V * N, slots=V, clips_per_slot=args.clips_per_slot, depth=2,
                     ingest_chunk=args.ingest_chunk)
    for i in range(2):
        write_staging(vs.staging(i), inp, 0, V * N)
    for i in range(2):                                               # warm-up: module loading, allocator
        vs.collect(vs.submit(i, items))
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    pending, tables, evs = [], None, []
    for g in range(args.groups):
        if len(pending) == 2:
            tables = vs.collect(pending.pop(0))
        pending.append(vs.submit(g % 2, items))
        evs.append(pending[-1]["events"])
    while pending:
        tables = vs.collect(pending.pop(0))
    wall = time.perf_counter() - t0
    builds_warm = vs.plan_builds
    # overlap of group g+1's ingest (i/o stream) with group g's clip calls (compute stream), device events, ms
    base = evs[0]["ingest0"]
    at = lambda e: base.elapsed_time(e)     # noqa: E731
    overlap = [max(0.0, min(at(x["calls"]), at(y["ingested"])) - max(at(x["ingested"]), at(y["ingest0"]))) for x, y in zip(evs, evs[1:])]
    stream_cf_s = cf * args.groups / wall
    timing = {}
    tables = vs.collect(vs.submit(0, items), timing=timing)
    t = vs.collect(vs.submit(1, items))
    del t
    mode_a = cfg["mode"] == "A"
    row_b = vs.buffers[0]["rows"][0].shape[2] * 2
    t_ing = vs.submit(0, items)
    sels = [p["sel"] for p in t_ing["plans"][:len(t_ing["ingest"])]]      # the ingest plans' K1-K3 outputs of this group
    vs.collect(t_ing)
    sel_rows = sum(int(s["sel_count"].sum()) for s in sels)
    cand_rows = sum(int(s["cand"]["count"].sum()) for s in sels) if mode_a else 0
    in_place = sel_rows * 3 * 512 + ((cand_rows + sel_rows) * row_b if mode_a else 0)
    h2d_cf = (t_ing["h2d"] + in_place) / cf
    del t_ing, sels

    # ---- device-resident frames: ingest_frames + chained forward_clips (eager) ----
    kmax = st.cfg.selection.max_keep(ops.AnchorSpec(bench.HW).num_anchors)
    store = frames.FrameStore(V * N, kmax, C)
    head_all, feats_all = bench.views_of(inp, ops, C)
    slots_all = torch.arange(V * N, dtype=torch.int32, device=dev)
    pool = stage.CAFMState(V, kmax)

    dev_lists = []

    def device_pass():
        dev_lists.clear()
        for f0 in range(0, V * N, args.ingest_chunk):
            sub = {k: [x[f0:f0 + args.ingest_chunk] for x in v] for k, v in inp.items()}
            h, fe = bench.views_of(sub, ops, C)
            st.ingest_frames(store, h, fe, torch.float16, slots_all[f0:f0 + args.ingest_chunk])
        per_video = [list(zip(it["clips"], it["paths"])) for it in items]
        for batch in clips.ClipScheduler(per_video, world=1, slots=V, clips_per_slot=args.clips_per_slot).batches(0):
            chain = [c.chain for c in batch]
            te = torch.cat([clips.time_embedding(c.frame_numbers) for c in batch], 0).to(dev)
            o = st.forward_clips(store, [[items[c.video]["first_frame"] + f for f in c.frames] for c in batch], L, te, state=pool,
                                 resume=[c.resume for c in batch], state_slots=[c.slot for c in batch], chain=chain if any(chain) else None)
            dev_lists.append((batch, o))
    device_pass()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(args.groups):
        device_pass()
    torch.cuda.synchronize()
    device_cf_s = cf * args.groups / (time.perf_counter() - t0)

    device_same = all(same_as_tables(tables, items, b, st.to_lists(o, len(b), L)[0], L) for b, o in dev_lists)
    dev_lists.clear()
    identical = True
    for v in range(V):
        want_p, want_o = reference_table(st, store, v * N, items[v], L)
        identical &= torch.equal(tables[v]["offsets"], want_o) and torch.equal(tables[v]["packed"].view(torch.int32), want_p.view(torch.int32))

    # ---- forward_host: one clip of every video per call, stateful, two calls in flight ----
    fh = None
    if not wide:
        per_video = [list(zip(it["clips"], it["paths"])) for it in items]
        batches = list(clips.ClipScheduler(per_video, world=1, slots=V).batches(0))
        hosts = []
        for b in batches[:2]:
            idx = torch.tensor([items[c.video]["first_frame"] + f for c in b for f in c.frames], device=dev)
            h = {k: [inp[k][0].index_select(0, idx).cpu().pin_memory()] for k in ("rows", "objp")}
            for k in ("f_cls", "f_reg", "f_edge"):
                h[k] = [torch.empty((len(idx),) + tuple(t.shape[1:]), dtype=t.dtype, pin_memory=True,
                                    memory_format=torch.channels_last).copy_(t.index_select(0, idx)) for t in inp[k]]
            hosts.append(h)
        hpool = stage.CAFMState(V, kmax)

        def fh_call(j, slot):
            b = batches[j]
            te = torch.cat([clips.time_embedding(c.frame_numbers) for c in b], 0)
            return st.forward_host_submit(hosts[j % 2], bench.HW, te, len(b), F, L, slot=slot, state=hpool,
                                          resume=[c.resume for c in b], state_slots=[c.slot for c in b])
        n_calls = len(batches)
        fh_same = True
        for j in range(2):                   # the first two calls run on their own frames: compared with the stream
            r = st.forward_host_collect(fh_call(j, j))[0]
            fh_same &= same_as_tables(tables, items, batches[j], r, L)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        pend, fcf = [], 0
        for g in range(args.groups):
            for j in range(n_calls):
                if len(pend) == 2:
                    st.forward_host_collect(pend.pop(0))
                pend.append(fh_call(j, j % 2))
                fcf += len(batches[j]) * F
        while pend:
            st.forward_host_collect(pend.pop(0))
        fh = {"clip_frames_per_s": round(fcf / (time.perf_counter() - t0)), "calls_per_group": n_calls, "first_two_calls_identical": bool(fh_same),
              "note": "one clip of every video per call, stateful, two calls in flight; timed on the pinned inputs of the first two "
                      "calls, alternated (all calls' inputs would not fit in pinned memory); the first two calls' detections are "
                      "compared with the stream's"}
        del hosts

    cnt = store.count[:V * N]
    return {"metric": "video stream: clip-frames/s end to end from pinned host memory", "config": name,
            "workload": f"{V} videos x {N} frames in one group, demo_clips L {L} / G {G} -> {cf // F} clips ({cf} clip-frames); "
                        f"{args.clips_per_slot} clips per slot chained; {args.groups} groups, 2 in flight",
            "kmax": kmax, "proposals_per_frame": {"min": int(cnt.min()), "mean": round(float(cnt.float().mean()), 1), "max": int(cnt.max())},
            "stream": {"clip_frames_per_s": round(stream_cf_s), "plan_builds": {"warm": builds_warm, "end": vs.plan_builds},
                       "ingest_overlap_ms": [round(x, 3) for x in overlap], "h2d_bytes_per_clip_frame": round(h2d_cf),
                       "phase_ms": {k: round(float(timing[k]), 3) for k in ("ingest", "calls", "pack", "wait", "readback", "unpack")},
                       "d2h_bytes_per_group": timing["d2h"]},
            "forward_host": fh, "device_resident": {"clip_frames_per_s": round(device_cf_s), "identical": bool(device_same),
                                "note": "ingest_frames + chained forward_clips, eager"},
            "identical": bool(identical)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="ovis_a_k30,ovis_l_modeB,vid_l_c30,vid_l_wide")
    ap.add_argument("--videos", type=int, default=4)
    ap.add_argument("--frames", type=int, default=64)
    ap.add_argument("--clips-per-slot", type=int, default=4)
    ap.add_argument("--ingest-chunk", type=int, default=64)
    ap.add_argument("--groups", type=int, default=4)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise RuntimeError("bench_video_stream.py needs a CUDA device: tscd_b200 has no CPU fallback")
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
        with open(os.path.join(args.out, "video_stream_b200.jsonl"), "w") as f:
            f.write("".join(json.dumps(x) + "\n" for x in lines))


if __name__ == "__main__":
    main()
