"""GPU tests of the wide tier (513 .. 2048 proposals per frame, SelectionConfig.max_proposals > 512): the CTA-cooperative LSAP
solver against scipy.optimize.linear_sum_assignment, the final NMS above 16384 candidate rows against the oracle's
torchvision restatement, the whole stage against oracle.stage_tscd at the VID TSCD-L shape with local frames of up to ~2000
proposals, the default tier against the wide tier on the same inputs, and the limits that stay loud."""
import pytest
import torch

import oracle
import parity
from test_gpu_nms_large import _expanded_frame
from test_gpu_stage import _decisive_weights, _report, _run_case

pytestmark = pytest.mark.gpu

HW = [(72, 72), (36, 36), (18, 18)]          # 576 x 576: 6804 anchors


def _lap_device(cost, shapes, kmax):
    from tscd_b200 import _lib as L, ops
    nf = len(shapes)
    lrow = torch.tensor([0] + list(torch.tensor([n for _, n in shapes]).cumsum(0)), dtype=torch.int32).cuda()
    ref_n = torch.tensor([np_ for np_, _ in shapes], dtype=torch.int32).cuda()
    lap_col = torch.full((nf, kmax), -7, dtype=torch.int32).cuda()
    lap_row = torch.full((nf, kmax), -7, dtype=torch.int32).cuda()
    ops.call("tscd_cafm_lap", L.CafmLapArgs, num_frames=nf, kmax=kmax, lrow_off=lrow, ref_n=ref_n, cost=cost.cuda().contiguous(),
             lap_col=lap_col, lap_row=lap_row)
    torch.cuda.synchronize()
    return lap_col.cpu(), lap_row.cpu()


def _assert_scipy(cost, shapes, lap_col, lap_row):
    from scipy.optimize import linear_sum_assignment
    for f, (np_, n) in enumerate(shapes):
        ri, ci = linear_sum_assignment(cost[f, :np_, :n].double().numpy())
        want_col, want_row = [-1] * np_, [-1] * n
        for r, c in zip(ri.tolist(), ci.tolist()):
            want_col[r] = c
            want_row[c] = r
        assert lap_col[f, :np_].tolist() == want_col, f"frame {f} shape {(np_, n)}: lap_col differs from scipy"
        assert lap_row[f, :n].tolist() == want_row, f"frame {f} shape {(np_, n)}: lap_row differs from scipy"


def _cosine_table(g, np_, n):
    a = torch.nn.functional.normalize(torch.randn(np_, 64, generator=g), dim=1)
    b = torch.nn.functional.normalize(torch.randn(n, 64, generator=g), dim=1)
    a2 = torch.nn.functional.normalize(torch.randn(np_, 32, generator=g), dim=1)
    b2 = torch.nn.functional.normalize(torch.randn(n, 32, generator=g), dim=1)
    return 1.0 - (a @ b.t() + a2 @ b2.t()) / 2


def test_lap_wide_vs_scipy():
    """Shapes up to 2048 x 2048, rectangular both ways down to 1 x 2048 / 2048 x 1, on cosine-like fp32 tables and on
    tie-heavy ones (small integers, rank-1: every assignment optimal), in ONE launch with problems of <= 512 (one-warp solvers)
    and > 512 (CTA solver): identical lap_col / lap_row."""
    g = torch.Generator().manual_seed(21)
    kmax = 2048
    spec = [((2048, 2048), "cos"), ((2048, 700), "cos"), ((700, 2048), "cos"), ((1, 2048), "cos"), ((2048, 1), "cos"),
            ((1024, 1024), "int"), ((1500, 1300), "rank1"), ((600, 600), "int"), ((513, 40), "cos"),
            ((300, 300), "cos"), ((512, 512), "int"), ((40, 40), "int"), ((20, 33), "rank1")]
    shapes = [s for s, _ in spec]
    cost = torch.zeros(len(spec), kmax, kmax)
    for f, ((np_, n), kind) in enumerate(spec):
        if kind == "cos":
            c = _cosine_table(g, np_, n)
        elif kind == "int":
            c = torch.randint(0, 3, (np_, n), generator=g).float()
        else:
            c = torch.randint(0, 4, (np_, 1), generator=g).float() + torch.randint(0, 4, (1, n), generator=g).float()
        cost[f, :np_, :n] = c
    lap_col, lap_row = _lap_device(cost, shapes, kmax)
    _assert_scipy(cost, shapes, lap_col, lap_row)


def test_lap_default_tier_unchanged_under_wide_kmax():
    """Problems of <= 512 rows and columns give the same assignment whether the launch's kmax is 512 (default tier) or 2048."""
    g = torch.Generator().manual_seed(22)
    shapes = [(500, 300), (300, 500), (512, 512), (100, 100), (33, 7), (1, 400)]
    small = torch.zeros(len(shapes), 512, 512)
    for f, (np_, n) in enumerate(shapes):
        small[f, :np_, :n] = _cosine_table(g, np_, n) if f % 2 == 0 else torch.randint(0, 4, (np_, n), generator=g).float()
    wide = torch.zeros(len(shapes), 2048, 2048)
    wide[:, :512, :512] = small
    c512, r512 = _lap_device(small, shapes, 512)
    c2k, r2k = _lap_device(wide, shapes, 2048)
    assert torch.equal(c512, c2k[:, :512]) and torch.equal(r512, r2k[:, :512])


def test_final_nms_2048x30_vs_oracle():
    """Final per-class NMS at the wide tier's VID pitch (2048 proposals x 30 classes = 61 440 rows): a dense frame, a frame whose
    class bands overlap with a real cross-class suppression (negative coordinates: the exact general path in global memory),
    a class with all 2048 proposals as members, and a small frame in the same launch.  Keep lists identical to
    oracle.batched_nms, in the same order, with and without a keep cap."""
    g = torch.Generator().manual_seed(31)
    C, P = 30, 2048
    cap = P * C
    Fn = 4
    box = torch.zeros(Fn, cap, 4)
    score = torch.zeros(Fn, cap)
    cls = torch.zeros(Fn, cap, dtype=torch.int32)
    count = torch.zeros(Fn, dtype=torch.int32)
    # frame 0: dense
    b, s, c = _expanded_frame(g, P, C, spread=520.0)
    box[0, :len(s)], score[0, :len(s)], cls[0, :len(s)], count[0] = b, s, c, len(s)
    # frame 1: negative coordinates + an engineered cross-class hit
    b, s, c = _expanded_frame(g, P - 2, C, spread=400.0, neg=60.0)
    M = 700.0
    b = torch.cat([b, torch.tensor([[M - 10, M - 10, M, M], [-11.0, -11.0, -1.0, -1.0]])])
    s = torch.cat([s, torch.tensor([1.5, 1.4])])
    c = torch.cat([c, torch.tensor([3, 4], dtype=torch.int32)])
    n1 = len(s)
    assert float(b.max()) == M
    box[1, :n1], score[1, :n1], cls[1, :n1], count[1] = b, s, c, n1
    want = oracle.batched_nms(b, s, c.float(), 0.5).tolist()
    assert (n1 - 2) in want and (n1 - 1) not in want             # really a cross-class suppression
    # frame 2: every proposal in class 5 (2048 members) plus the other classes sparsely
    b, s, c = _expanded_frame(g, P, C, spread=520.0, dup_scores=True)
    n2 = len(s)
    c = c.clone()
    c[torch.arange(0, n2, C)] = 5
    assert int((c == 5).sum()) >= 2048
    box[2, :n2], score[2, :n2], cls[2, :n2], count[2] = b, s, c, n2
    # frame 3: small
    b, s, c = _expanded_frame(g, 120, C, spread=300.0)
    box[3, :len(s)], score[3, :len(s)], cls[3, :len(s)], count[3] = b, s, c, len(s)
    assert int(count[:3].min()) > 16384
    _check(box, score, cls, count, 0.5, label="wide 0.5")
    _check(box, score, cls, count, 0.5, max_keep=3000, label="wide keep 3000")


def _check(box, score, cls, count, thr, max_keep=None, label=""):
    from tscd_b200 import ops
    keep, kc, status = ops.nms(box.cuda(), score.cuda(), cls.cuda(), count.cuda(), thr, max_keep=max_keep, wide=True)
    torch.cuda.synchronize()
    assert int(status.item()) == 0
    for f in range(box.shape[0]):
        n = int(count[f])
        want = oracle.batched_nms(box[f, :n], score[f, :n], cls[f, :n].float(), thr).tolist()
        if max_keep is not None:
            want = want[:max_keep]
        got = keep[f, :int(kc[f])].cpu().tolist()
        assert got == want, f"{label} frame {f} n {n}: {len(got)} vs {len(want)} kept"


def _wide_sel(limit):
    return dict(minimal_limit=50, maximal_limit=0, use_pre_nms=False, max_proposals=limit)


O_SEL = dict(nms_thre=0.75, minimal_limit=50, maximal_limit=0, use_pre_nms=False)


def test_stage_wide_vid_l_val_shape_with_resume():
    """(a) VID TSCD-L val shape: F = 32 (1 local + 31 global), C = 30, 576 x 576; the local frame keeps ~1800 proposals, the
    global frames 50 .. 300.  Two calls with resume: the second call's LSAP is ~1800 x ~1800 against the carried state."""
    def means(call, b):
        return [-7.9 if i == 0 else [-10.5, -9.9, -11.5, -10.2][i % 4] for i in range(32)]
    st = _run_case("B", B=1, F=32, Lf=1, hw=HW, C=30, sel_kw=_wide_sel(2048), o_sel_kw=O_SEL, seeds=[300, 400], calls=2,
                   obj_means=means, synth_kw=dict(n_obj=3, n_mem=10))
    _report(st, "wide VID-L val shape", max_flip_frac=0.5)


def test_stage_wide_chain_of_wide_lsaps():
    """(b) F = 16, L = 4: local frames of ~600 .. ~2000 proposals, so every step of the CAFM chain solves a wide LSAP."""
    def means(call, b):
        return [[-7.75, -9.3, -8.5, -9.0][i] if i < 4 else [-10.5, -11.0, -9.9][i % 3] for i in range(16)]
    st = _run_case("B", B=1, F=16, Lf=4, hw=HW, C=30, sel_kw=_wide_sel(2048), o_sel_kw=O_SEL, seeds=[500], calls=1,
                   obj_means=means, synth_kw=dict(n_obj=3, n_mem=10))
    _report(st, "wide chain L=4", max_flip_frac=0.5)


def _forward(cfg_limit, head, views, te, B, F, Lf, sd, C):
    from tscd_b200 import selection, stage
    cfg = stage.StageConfig(num_classes=C, selection=selection.SelectionConfig(mode="B", **_wide_sel(cfg_limit)))
    st = stage.AggregationStage(cfg, sd)
    trace = {}
    out = st.forward(head, views, torch.float16, te, B, F, Lf, trace=trace)
    torch.cuda.synchronize()
    res, ori = st.to_lists(out, B, Lf)
    return out, trace, res, ori


def test_default_and_wide_tier_agree_below_512():
    """The same inputs, every frame <= 512 proposals, at max_proposals 512 and 2048: identical selection, assignments and
    detections; float tensors within the parity bars."""
    from tscd_b200 import ops
    C, F, Lf, B = 30, 16, 4, 1
    sd = _decisive_weights(C, 256)
    means = [-9.8, -10.0, -11.0, -9.9] + [-10.5, -11.0, -9.9] * 4
    h, f = oracle.synth_head_outputs(F, HW, C, dim=256, seed=77, clustered=True, obj_mean=means[:F], n_obj=3, n_mem=10)
    an = ops.AnchorSpec(HW)
    head = ops.HeadViews.from_fused(oracle.decode_outputs(h, HW, [8, 16, 32]).cuda(), an, apply_sigmoid=False, apply_decode=False)
    views = tuple(ops.view_rowmajor(p.half().cuda().contiguous(), an) for p in f)
    te = oracle.timing_signal_1d(torch.arange(Lf), 256)
    o1, t1, r1, ori1 = _forward(512, head, views, te, B, F, Lf, sd, C)
    o2, t2, r2, ori2 = _forward(2048, head, views, te, B, F, Lf, sd, C)
    cnt = o1["sel"]["sel_count"].cpu()
    assert torch.equal(cnt, o2["sel"]["sel_count"].cpu()) and int(cnt.max()) <= 512 and int(cnt[:Lf].min()) > 100
    for fr in range(B * F):
        n = int(cnt[fr])
        assert torch.equal(o1["sel"]["sel_idx"][fr, :n].cpu(), o2["sel"]["sel_idx"][fr, :n].cpu())
    n_loc = int(o1["layout"].lrow_off[-1])
    assert torch.equal(t1["perm"][:n_loc].cpu(), t2["perm"][:n_loc].cpu())
    assert t2["cafm_lap_col"].shape[1] == 2048
    ref_n = t1["cafm_ref_n"].cpu().tolist()
    assert ref_n == t2["cafm_ref_n"].cpu().tolist()
    for lf in range(B * Lf):
        n = int(cnt[(lf // Lf) * F + lf % Lf])
        assert torch.equal(t1["cafm_lap_col"][lf, :ref_n[lf]].cpu(), t2["cafm_lap_col"][lf, :ref_n[lf]].cpu())
        assert torch.equal(t1["cafm_lap_row"][lf, :n].cpu(), t2["cafm_lap_row"][lf, :n].cpu())
    for name in ("agg_cls", "iou_cls", "iou_reg", "matched", "obj_ref", "cls_logits", "obj_logits", "reg_deltas"):
        en, er = parity.float_err(t2[name][:n_loc].float().cpu(), t1[name][:n_loc].float().cpu())
        assert en <= parity.TOL_NORM and er <= parity.TOL_REL, f"{name}: {en} / {er}"
    for a, b in zip(r1 + ori1, r2 + ori2):
        assert (a is None) == (b is None)
        if a is not None:
            assert a.shape == b.shape and torch.equal(a[:, 6], b[:, 6])
            torch.testing.assert_close(a, b, rtol=1e-3, atol=2e-2)


def test_wide_limits_stay_loud():
    """A frame above 2048 proposals raises (naming the limit); max_proposals = 2049 and 2048 x 40 classes are rejected at
    construction; F = 64 x 2048 keys per clip is rejected at forward; the host-buffer path refuses a wide-tier stage."""
    from tscd_b200 import ops, selection, stage
    C, F, Lf = 30, 4, 1
    sd = oracle.init_stage_weights(C, dim=256, seed=3)
    cfg = stage.StageConfig(num_classes=C, selection=selection.SelectionConfig(mode="B", **_wide_sel(2048)))
    st = stage.AggregationStage(cfg, sd)
    h, f = oracle.synth_head_outputs(F, HW, C, dim=256, seed=5, obj_mean=[-6.0, -11.0, -11.0, -11.0])   # frame 0: ~4000
    an = ops.AnchorSpec(HW)
    head = ops.HeadViews.from_fused(oracle.decode_outputs(h, HW, [8, 16, 32]).cuda(), an, apply_sigmoid=False, apply_decode=False)
    views = tuple(ops.view_rowmajor(p.half().cuda().contiguous(), an) for p in f)
    out = st.forward(head, views, torch.float16, oracle.timing_signal_1d(torch.arange(Lf), 256), 1, F, Lf)
    with pytest.raises(RuntimeError, match="2048"):
        st.to_lists(out, 1, Lf)
    with pytest.raises(RuntimeError, match="2048"):
        stage.AggregationStage(stage.StageConfig(num_classes=C, selection=selection.SelectionConfig(mode="B", **_wide_sel(2049))), sd)
    with pytest.raises(RuntimeError, match="NMS capacity of 65536"):
        stage.AggregationStage(stage.StageConfig(num_classes=40, selection=selection.SelectionConfig(mode="B", **_wide_sel(2048))),
                               oracle.init_stage_weights(40, dim=256, seed=3))
    hw64 = [(40, 40), (20, 20), (10, 10)]                       # 2100 anchors >= 2048: kmax = 2048, 64 x 2048 keys per clip
    an64 = ops.AnchorSpec(hw64)
    head64 = ops.HeadViews.from_fused(torch.zeros(64, an64.num_anchors, 5 + C).cuda(), an64, apply_sigmoid=False, apply_decode=False)
    with pytest.raises(RuntimeError, match="keys per clip"):
        st.forward(head64, None, torch.float16, oracle.timing_signal_1d(torch.arange(1), 256), 1, 64, 1)
    with pytest.raises(RuntimeError, match="default tier only"):
        st.forward_host({}, HW, oracle.timing_signal_1d(torch.arange(Lf), 256), 1, F, Lf)
