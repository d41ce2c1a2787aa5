#!/usr/bin/env python
"""REPP of one video straight from the stage's packed detections (REPPB200.from_detections: tscd_repp_prep -> link -> tubelets ->
emit, one read-back of the per-frame counts, one copy of the predictions) beside the dict path the packed table fed before
(evalglue.repp_predictions + REPPB200.__call__).  Synthetic stage rows [frames, cap, 7] of objects moving through a 480 x 854 video,
packed with the resize ratio as scale.  Times: wall clock of each path end to end (median of --reps), and device events around
from_detections (prep, the read-back of the per-frame counts, link, tubelets, emit: everything but the final copy and the dicts).
Outputs are compared.

  python tools/bench_repp_video.py [--frames 300] [--objects 45] [--reps 5] [--out FILE]"""
import argparse
import json
import os
import statistics
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def stage_rows(T, nobj, cap, ratio, seed=5, ih=480, iw=854):
    rng = np.random.default_rng(seed)
    pos = rng.uniform([-20, -20], [iw - 150, ih - 150], size=(nobj, 2))
    vel = rng.normal(0, 4, size=(nobj, 2))
    size = rng.uniform(25, 140, size=(nobj, 2))
    cls = rng.integers(0, 30, size=nobj)
    rows = np.zeros((T, cap, 7), dtype=np.float32)
    counts = []
    for t in range(T):
        dets = []
        for o in range(nobj):
            for rep in range(int(rng.integers(0, 3))):
                xy = pos[o] + vel[o] * t * 0.3 + rng.normal(0, 2.5, 2)
                wh = size[o] * (1 + rng.normal(0, 0.05, 2))
                c = cls[o] if rep == 0 else int(rng.integers(0, 30))
                dets.append([xy[0] * ratio, xy[1] * ratio, (xy[0] + wh[0]) * ratio, (xy[1] + wh[1]) * ratio,
                             rng.uniform(0.05, 0.95), rng.uniform(0.02, 0.9), c])
        n = min(cap, len(dets))
        rows[t, :n] = np.asarray(dets[:n], dtype=np.float32).reshape(-1, 7)
        counts.append(n)
    return rows, counts


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=300)
    ap.add_argument("--objects", type=int, default=45)
    ap.add_argument("--cap", type=int, default=128)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from tscd_b200 import evalglue
    from tscd_b200.repp import REPPB200
    g = json.load(open(os.path.join(ROOT, "tests", "golden", "repp.json")))
    cfg = g["cases"][0]["cfg"]
    ratio = 576 / 854
    rows, counts = stage_rows(args.frames, args.objects, args.cap, ratio)
    sizes, ids = [(480, 854)] * args.frames, [f"v/{t:06d}" for t in range(args.frames)]
    d_rows, d_cnt = torch.from_numpy(rows).cuda(), torch.tensor(counts, dtype=torch.int32).cuda()
    packed, offsets = evalglue.pack_detections(d_rows, d_cnt, torch.full((args.frames,), ratio))
    post = REPPB200(logreg=g["logreg"], **cfg)

    def dict_path():
        table, off = evalglue.to_host(packed, offsets)
        video = {str(f): p for f, p in enumerate(evalglue.repp_predictions(table, off, counts, sizes, ids))}
        return post(video)

    def packed_path():
        return post.from_detections(packed, offsets, counts, sizes, ids).predictions()

    want, got = dict_path(), packed_path()                     # warm-up (module load, allocator)
    walls = {"packed": [], "dicts": []}
    dev_ms = []
    for _ in range(args.reps):
        for name, fn in (("packed", packed_path), ("dicts", dict_path)):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            fn()
            walls[name].append(time.perf_counter() - t0)
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        s.record()
        r = post.from_detections(packed, offsets, counts, sizes, ids)
        e.record()
        torch.cuda.synchronize()
        dev_ms.append(s.elapsed_time(e))
        del r
    name = torch.cuda.get_device_name()
    line = {"frames": args.frames, "detections": int(sum(counts)), "predictions": len(got), "identical": got == want,
            "packed_wall_ms": round(1e3 * statistics.median(walls["packed"]), 3),
            "dicts_wall_ms": round(1e3 * statistics.median(walls["dicts"]), 3),
            "packed_events_ms": round(statistics.median(dev_ms), 3), "reps": args.reps, "gpu": name}
    print(json.dumps(line))
    if args.out:
        with open(args.out, "a") as f:
            f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
