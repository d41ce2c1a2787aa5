"""CPU test of bench.py --dump-outputs: the arrays written are the caller's view of the stage's output (TSCD: to_lists, per local
frame [n,7] rows or None; gen-1: each frame's logits rows), in float32 / float64, and the sample taken above the size cap is the
same whatever the outputs hold."""
import numpy as np
import torch

import bench


def _stage_out(nlf, det_cap, ori_cap, seed):
    g = torch.Generator().manual_seed(seed)
    det_n = torch.randint(0, det_cap + 1, (nlf,), generator=g, dtype=torch.int32)
    ori_n = torch.minimum(det_n, torch.tensor(ori_cap, dtype=torch.int32))
    cand = det_n.clone()
    cand[::3] = 0                                        # no candidate -> the caller gets None for both lists
    return dict(status=torch.zeros(1, dtype=torch.int32), det_count=det_n, ori_count=ori_n, det_cand=cand,
                det_rows=torch.randn(nlf, det_cap, 7, generator=g), ori_rows=torch.randn(nlf, ori_cap, 7, generator=g))


def _load(d, name):
    return np.load(d / (name + ".npy"))


def test_dump_writes_the_callers_lists(tmp_path):
    cfg = dict(bench.CONFIGS["ovis_a_k30"])
    B, Lf = 3, cfg["L"]
    out = _stage_out(B * Lf, 20, 4, seed=1)
    bench.dump_outputs(str(tmp_path), bench.caller_arrays(cfg, out, B))
    assert sorted(p.name for p in tmp_path.iterdir()) == ["det_counts.npy", "det_rows.npy", "frames.npy", "ori_counts.npy", "ori_rows.npy"]
    assert _load(tmp_path, "frames").dtype == np.float64 and _load(tmp_path, "frames").tolist() == list(range(B * Lf))
    for name in ("det", "ori"):
        rows, counts = _load(tmp_path, name + "_rows"), _load(tmp_path, name + "_counts")
        assert rows.dtype == np.float32 and counts.dtype == np.float64 and rows.shape[1] == 7
        want = []
        for f in range(B * Lf):
            if int(out["det_cand"][f]) == 0:
                assert counts[f] == -1
                continue
            n = int(out[name + "_count"][f])
            assert counts[f] == n
            want.append(out[name + "_rows"][f, :n].numpy())
        np.testing.assert_array_equal(rows, np.concatenate(want))


def test_dump_sample_is_capped_and_independent_of_the_outputs(tmp_path):
    cfg = dict(bench.CONFIGS["ovis_a_k30"])
    B, Lf = 16, cfg["L"]
    cap = 40 * (20 * 7 * 4 + 4 * 7 * 4 + 24) + 5 * bench.NPY_HEADER_BYTES   # room for 40 of the 128 frames at full capacity
    picked = []
    for seed in (1, 2):
        d = tmp_path / str(seed)
        bench.dump_outputs(str(d), bench.caller_arrays(cfg, _stage_out(B * Lf, 20, 4, seed), B), max_bytes=cap)
        frames = _load(d, "frames")
        assert len(frames) == 40 and np.all(np.diff(frames) > 0)
        assert sum(p.stat().st_size for p in d.iterdir()) <= cap
        assert len(_load(d, "det_counts")) == len(_load(d, "ori_counts")) == 40
        picked.append(frames.tolist())
    assert picked[0] == picked[1]


def test_dump_gen1_logits_split_by_frame(tmp_path):
    cfg = dict(bench.CONFIGS["gen1_msa"])
    B, F, kmax, C1 = 2, cfg["F"], 5, cfg["C"] + 1
    g = torch.Generator().manual_seed(4)
    counts = torch.randint(0, kmax + 1, (B * F,), generator=g)
    row_off = torch.cat([torch.zeros(1, dtype=torch.int64), counts.cumsum(0)]).to(torch.int32)
    n = int(row_off[-1])
    logits = torch.randn(n + 128, C1, generator=g)            # rows past row_off[-1] are padding the caller never reads
    out = dict(status=torch.zeros(1, dtype=torch.int32), logits=logits,
               sel=dict(row_off=row_off, sel_rows=torch.zeros(B * F, kmax, 7 + cfg["C"])))
    bench.dump_outputs(str(tmp_path), bench.caller_arrays(cfg, out, B))
    assert sorted(p.name for p in tmp_path.iterdir()) == ["frames.npy", "logits_counts.npy", "logits_rows.npy"]
    assert _load(tmp_path, "logits_counts").tolist() == counts.tolist()
    rows = _load(tmp_path, "logits_rows")
    assert rows.dtype == np.float32
    np.testing.assert_array_equal(rows, logits[:n].numpy())
