"""GPU parity: K4 cross-frame attention aggregation (tcgen05) vs the oracle's restatement of
MCA_tscd_g2l_reg / Attention_mca_g2l and MSA_yolov, at module level (after the output Linears).  Tolerance: max error
relative to the tensor's max <= 1e-2 (north_star; 16-bit operands, fp32 accumulation), no rows excluded.  For clustered
features the ragged-clip test does not compare with the oracle at all -- their similarities sit at the 0.75 / 0.99
thresholds, where the masks may flip -- and checks only that two runs are bit-identical and finite.  The kernels
themselves are checked element by element, masks included, in test_gpu_attn_kernels.py."""
import pytest
import torch

import oracle

pytestmark = pytest.mark.gpu


def _make_case(B, F, L, counts, seed, clustered):
    g = torch.Generator().manual_seed(seed)
    N = sum(counts)
    if clustered:
        base = torch.randn(40, 256, generator=g)
        idc = torch.randint(0, 40, (N,), generator=g)
        xc = base[idc] + 0.35 * torch.randn(N, 256, generator=g)
        xr = base[torch.randint(0, 40, (N,), generator=g)] + 0.05 * torch.randn(N, 256, generator=g)
    else:
        xc, xr = torch.randn(N, 256, generator=g), torch.randn(N, 256, generator=g)
    score = torch.rand(N, generator=g) * 0.9 + 0.05
    return xc, xr, score


def _rel(a, b):
    return float((a.float().cpu() - b).abs().max() / b.abs().max())


@pytest.mark.parametrize("clustered", [False, True])
@pytest.mark.parametrize("dtype", [torch.float16])
def test_mca_module_vs_oracle(clustered, dtype):
    from tscd_b200 import aggregate, ops
    B, F, L = 3, 6, 2
    g = torch.Generator().manual_seed(11)
    counts = torch.randint(20, 41, (B * F,), generator=g).tolist()
    counts[1] = 7
    xc, xr, score = _make_case(B, F, L, counts, 5, clustered)
    sd = oracle.init_stage_weights(25, dim=256, seed=3)
    # the product consumes 16-bit features: give the oracle the same rounded values
    xc, xr = xc.to(dtype).float(), xr.to(dtype).float()
    sd16 = {k: v.to(dtype).float() if v.dim() == 2 else v for k, v in sd.items()}
    N = sum(counts)
    row_cap = ((N + 127) // 128 + 1) * 128
    cnt = torch.tensor(counts, dtype=torch.int32).cuda()
    loc_total = sum(sum(counts[b * F:b * F + L]) for b in range(B))
    lay = aggregate.make_layout(cnt, B, F, L, row_cap, ((loc_total + 127) // 128) * 128, 256, dtype)
    bank_c = torch.zeros(row_cap, 256, dtype=dtype).cuda(); bank_c[:N] = xc.to(dtype).cuda()
    bank_r = torch.zeros(row_cap, 256, dtype=dtype).cuda(); bank_r[:N] = xr.to(dtype).cuda()
    bscore = torch.zeros(row_cap).cuda(); bscore[:N] = score.cuda()
    n_dev = torch.tensor([N], dtype=torch.int32).cuda()
    nl_dev = torch.tensor([loc_total], dtype=torch.int32).cuda()
    w = aggregate.MCAWeights(sd, "agg_iou.", dtype)
    dbg = {}
    (c16, c32), (o16, o32) = aggregate.mca_forward(lay, w, bank_c, bank_r, bscore, n_dev, nl_dev, need_reg=True, debug=dbg)
    torch.cuda.synchronize()

    # oracle per clip
    off = [0]
    for c in counts:
        off.append(off[-1] + c)
    lpos = 0
    for b in range(B):
        s, e = off[b * F], off[(b + 1) * F]
        ppf = counts[b * F:(b + 1) * F]
        nl = sum(ppf[:L])
        tc, to = oracle.mca_tscd_g2l_reg(sd16, "agg_iou.", xc[s:e].unsqueeze(0), xr[s:e].unsqueeze(0), score[s:e], ppf, L)
        # intermediate: attention part (x before `linear`) of local frame 0
        assert _rel(c32[lpos:lpos + nl], tc) < 1e-2, f"clip {b} cls"
        assert _rel(o32[lpos:lpos + nl], to) < 1e-2, f"clip {b} obj"
        assert _rel(c16[lpos:lpos + nl], tc) < 1e-2
        lpos += nl


def test_msa_yolov_self_attention_vs_oracle():
    """Gen-1 MSA (north_star item 4): self-attention over all proposals of each clip, both softmax branches,
    cosine masks, round 2 on linear1's output, linear2."""
    from tscd_b200 import aggregate, ops
    dtype = torch.float16
    B, F = 2, 4
    g = torch.Generator().manual_seed(21)
    counts = [30, 30, 17, 30, 30, 30, 30, 9]
    xc, xr, score = _make_case(B, F, F, counts, 9, True)
    xc, xr = xc.to(dtype).float(), xr.to(dtype).float()
    sd = oracle.init_stage_weights(25, dim=256, seed=5, gen1=True)
    sd16 = {k: v.to(dtype).float() if v.dim() == 2 else v for k, v in sd.items()}
    N = sum(counts)
    row_cap = ((N + 127) // 128 + 1) * 128
    cnt = torch.tensor(counts, dtype=torch.int32).cuda()
    lay = aggregate.make_layout(cnt, B, F, F, row_cap, row_cap, 128, dtype)
    lay.self_attn = True
    lay.lrow_off = lay.row_off
    bank_c = torch.zeros(row_cap, 256, dtype=dtype).cuda(); bank_c[:N] = xc.to(dtype).cuda()
    bank_r = torch.zeros(row_cap, 256, dtype=dtype).cuda(); bank_r[:N] = xr.to(dtype).cuda()
    bscore = torch.zeros(row_cap).cuda(); bscore[:N] = score.cuda()
    n_dev = torch.tensor([N], dtype=torch.int32).cuda()
    w = aggregate.MSAWeights(sd, "trans.", dtype)
    o16, o32 = aggregate.msa_forward(lay, w, bank_c, bank_r, bscore, n_dev)
    torch.cuda.synchronize()
    off = 0
    for b in range(B):
        n = sum(counts[b * F:(b + 1) * F])
        want, _ = oracle.msa_yolov(sd16, "trans.", xc[off:off + n].unsqueeze(0), xr[off:off + n].unsqueeze(0), score[off:off + n])
        assert _rel(o32[off:off + n], want) < 1e-2, f"clip {b}"
        off += n


@pytest.mark.parametrize("clustered", [False, True])
def test_mca_ragged_clip_sizes_and_determinism(clustered):
    """Clips of 6 / 64 / 65 / 129 / 257 proposals in one batch (key tiles of 64: one partial tile, exactly full, one
    key over, ...; 128 local rows = exactly one query tile, 1-row frames): every ring / barrier wrap-around of the
    pipelined attention kernels.  Two runs must be bit-identical (no race), and -- for unclustered features, whose
    cosine similarities are far from the 0.75 / 0.99 thresholds -- within 1e-2 of the oracle."""
    from tscd_b200 import aggregate
    dtype = torch.float16
    B, F, L = 5, 6, 2
    counts = [1, 1, 1, 1, 1, 1,   30, 30, 1, 1, 1, 1,   30, 31, 1, 1, 1, 1,   40, 25, 30, 30, 2, 2,   64, 64, 64, 63, 1, 1]
    assert [sum(counts[b * F:(b + 1) * F]) for b in range(B)] == [6, 64, 65, 129, 257]
    xc, xr, score = _make_case(B, F, L, counts, 17, clustered)
    sd = oracle.init_stage_weights(25, dim=256, seed=4)
    xc, xr = xc.to(dtype).float(), xr.to(dtype).float()
    sd16 = {k: v.to(dtype).float() if v.dim() == 2 else v for k, v in sd.items()}
    N = sum(counts)
    row_cap = ((N + 127) // 128 + 1) * 128
    cnt = torch.tensor(counts, dtype=torch.int32).cuda()
    loc_total = sum(sum(counts[b * F:b * F + L]) for b in range(B))
    lay = aggregate.make_layout(cnt, B, F, L, row_cap, ((loc_total + 127) // 128) * 128, 384, dtype)
    bank_c = torch.zeros(row_cap, 256, dtype=dtype).cuda(); bank_c[:N] = xc.to(dtype).cuda()
    bank_r = torch.zeros(row_cap, 256, dtype=dtype).cuda(); bank_r[:N] = xr.to(dtype).cuda()
    bscore = torch.zeros(row_cap).cuda(); bscore[:N] = score.cuda()
    n_dev = torch.tensor([N], dtype=torch.int32).cuda()
    nl_dev = torch.tensor([loc_total], dtype=torch.int32).cuda()
    w = aggregate.MCAWeights(sd, "agg_iou.", dtype)
    runs = []
    for _ in range(3):
        (c16, c32), (o16, o32) = aggregate.mca_forward(lay, w, bank_c, bank_r, bscore, n_dev, nl_dev, need_reg=True)
        torch.cuda.synchronize()
        runs.append((c32[:loc_total].clone(), o32[:loc_total].clone()))
    for c, o in runs[1:]:
        assert torch.equal(c, runs[0][0]) and torch.equal(o, runs[0][1])
    assert torch.isfinite(runs[0][0]).all() and torch.isfinite(runs[0][1]).all()
    if clustered:
        return
    off = [0]
    for c in counts:
        off.append(off[-1] + c)
    lpos = 0
    for b in range(B):
        s, e = off[b * F], off[(b + 1) * F]
        ppf = counts[b * F:(b + 1) * F]
        nl = sum(ppf[:L])
        tc, to = oracle.mca_tscd_g2l_reg(sd16, "agg_iou.", xc[s:e].unsqueeze(0), xr[s:e].unsqueeze(0), score[s:e], ppf, L)
        assert _rel(runs[0][0][lpos:lpos + nl], tc) < 1e-2, f"clip {b} cls"
        assert _rel(runs[0][1][lpos:lpos + nl], to) < 1e-2, f"clip {b} obj"
        lpos += nl


def test_mca_long_clip_vs_oracle():
    """One long clip (128 frames x 30 proposals = 3840 keys = 60 key tiles, 480 local rows = 4 query tiles): the
    barrier phases of the pipelined attention kernels wrap many times; result within 1e-2 of the oracle."""
    from tscd_b200 import aggregate
    dtype = torch.float16
    B, F, L = 1, 128, 16
    counts = [30] * (B * F)
    xc, xr, score = _make_case(B, F, L, counts, 23, False)
    sd = oracle.init_stage_weights(25, dim=256, seed=6)
    xc, xr = xc.to(dtype).float(), xr.to(dtype).float()
    sd16 = {k: v.to(dtype).float() if v.dim() == 2 else v for k, v in sd.items()}
    N = sum(counts)
    row_cap = ((N + 127) // 128 + 1) * 128
    cnt = torch.tensor(counts, dtype=torch.int32).cuda()
    loc_total = sum(counts[:L])
    lay = aggregate.make_layout(cnt, B, F, L, row_cap, ((loc_total + 127) // 128) * 128, ((N + 127) // 128) * 128, dtype)
    bank_c = torch.zeros(row_cap, 256, dtype=dtype).cuda(); bank_c[:N] = xc.to(dtype).cuda()
    bank_r = torch.zeros(row_cap, 256, dtype=dtype).cuda(); bank_r[:N] = xr.to(dtype).cuda()
    bscore = torch.zeros(row_cap).cuda(); bscore[:N] = score.cuda()
    n_dev = torch.tensor([N], dtype=torch.int32).cuda()
    nl_dev = torch.tensor([loc_total], dtype=torch.int32).cuda()
    w = aggregate.MCAWeights(sd, "agg_iou.", dtype)
    (c16, c32), (o16, o32) = aggregate.mca_forward(lay, w, bank_c, bank_r, bscore, n_dev, nl_dev, need_reg=True)
    torch.cuda.synchronize()
    tc, to = oracle.mca_tscd_g2l_reg(sd16, "agg_iou.", xc.unsqueeze(0), xr.unsqueeze(0), score, counts, L)
    assert _rel(c32[:loc_total], tc) < 1e-2
    assert _rel(o32[:loc_total], to) < 1e-2


def test_gen1_stage_vs_oracle_full_size():
    """BASELINE configs[1] as the gen-1 (YOLOV) pipeline the north_star items (1)-(4) describe: 32 frames at 576x576, top-750 ->
    NMS 0.75 -> 30 proposals/frame -> MSA self-attention over all N = 960 proposals -> linear_pred; selection exact, refined
    class logits within 1e-2 (max-normalised) of the oracle's stage_gen1."""
    from tscd_b200 import gen1, ops, selection
    dtype = torch.float16
    C, F, B = 25, 32, 2
    hw = [(72, 72), (36, 36), (18, 18)]
    sd = oracle.init_stage_weights(C, dim=256, seed=6, gen1=True)
    sd16 = {k: v.to(dtype).float() if v.dim() == 2 else v for k, v in sd.items()}
    st = gen1.Gen1Stage(C, selection.SelectionConfig(mode="A", pre_k=750, top_k=30, nms_thresh=0.75), sd)
    heads, planes = [], []
    for b in range(B):
        h, f = oracle.synth_head_outputs(F, hw, C, dim=256, seed=300 + b, clustered=True)
        heads.append(oracle.decode_outputs(h, hw, [8, 16, 32]))
        planes.append([p.to(dtype).float() for p in f])
    an = ops.AnchorSpec(hw)
    head = ops.HeadViews.from_fused(torch.cat(heads, 0).cuda(), an, apply_sigmoid=False, apply_decode=False)
    dev_feats = [torch.cat([planes[b][k] for b in range(B)], 0).to(dtype).cuda().contiguous() for k in range(2)]
    views = (ops.view_rowmajor(dev_feats[0], an), ops.view_rowmajor(dev_feats[1], an), ops.view_rowmajor(dev_feats[1], an))
    out = st.forward(head, views, dtype, B, F)
    torch.cuda.synchronize()
    assert int(out["status"].item()) == 0
    cnt = out["sel"]["sel_count"].cpu().tolist()
    off = out["sel"]["row_off"].cpu().tolist()
    for b in range(B):
        rows, idxs, logits = oracle.stage_gen1(sd16, heads[b], planes[b][0], planes[b][1], C, pre_k=750, top_k=30)
        for f in range(F):
            assert out["sel"]["sel_idx"][b * F + f, :cnt[b * F + f]].cpu().tolist() == idxs[f].tolist()
        got = out["logits"][off[b * F]:off[(b + 1) * F], :C + 1].cpu()
        assert got.shape == logits.shape
        err = _rel(got, logits)
        print(f"gen-1 stage clip {b}: N = {got.shape[0]}, refined logits max-normalised error {err:.2e}")
        assert err < 1e-2
