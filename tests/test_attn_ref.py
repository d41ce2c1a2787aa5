"""CPU: the float64 attention reference of tests/attn_ref.py (the masked whole-clip form the GPU attention tests compare
csrc/attn.cu with) equals the reference's per-local-frame restatement, oracle.attention_mca_g2l, and its self-attention,
oracle.attention_msa -- so a wrong reference can neither pass nor fail the GPU tests by itself.  Both sides run in float64
on the same projections; agreement to 1e-10 is rounding-order noise only."""
import pytest
import torch
import torch.nn.functional as F

import oracle
from attn_ref import attention, frame_of_rows, round2, round2_weights, similarity, visibility

D = 256


def _nrm(t):
    return (t.view(t.shape[0], 4, 64) / t.view(t.shape[0], 4, 64).norm(dim=-1, keepdim=True)).reshape(t.shape[0], D)


def _features(n, seed):
    """Clustered features (near-duplicates of six bases), so that the 0.75 / 0.99 masks keep some keys and drop others."""
    g = torch.Generator().manual_seed(seed)
    base = torch.randn(6, D, generator=g, dtype=torch.float64)
    xc = base[torch.randint(0, 6, (n,), generator=g)] + 0.3 * torch.randn(n, D, generator=g, dtype=torch.float64)
    xr = base[torch.randint(0, 6, (n,), generator=g)] + 0.05 * torch.randn(n, D, generator=g, dtype=torch.float64)
    score = torch.rand(n, generator=g, dtype=torch.float64) * 0.9 + 0.05
    return xc, xr, score


def _operands(wq_c, wkv_c, wq_r, wkv_r, xc, xr, score):
    """The kernels' operands in float64: per-head normalised q / k / v, 25 * score folded into k_cls, 25 into k_reg."""
    kvc, kvr = F.linear(xc, wkv_c), F.linear(xr, wkv_r)
    return dict(qc=_nrm(F.linear(xc, wq_c)), kc=_nrm(kvc[:, :D]) * 25 * score[:, None], vc=kvc[:, D:],
                qr=_nrm(F.linear(xr, wq_r)), kr=_nrm(kvr[:, :D]) * 25, vr=kvr[:, D:])


@pytest.mark.parametrize("counts,L", [([5, 9, 0, 7, 6], 2),       # empty global frame
                                      ([4, 0, 11, 3], 2),         # empty local frame
                                      ([6, 8, 5], 3)])            # no global frames (F == L)
def test_reference_matches_mca_oracle(counts, L):
    sd = {k: v.double() for k, v in oracle.init_stage_weights(5, dim=D, seed=3).items()}
    p = "agg_iou.mca."
    n = sum(counts)
    xc, xr, score = _features(n, 7)
    o = _operands(sd[p + "q_cls_local.weight"], sd[p + "kv_cls.weight"], sd[p + "q_reg_local.weight"], sd[p + "kv_reg.weight"],
                  xc, xr, score)
    frame = frame_of_rows(counts)
    nloc = sum(counts[:L])
    vis = visibility(frame[:nloc], frame, L, False)
    ref = attention(o["qc"][:nloc], o["kc"], o["qr"][:nloc], o["kr"], o["vc"], o["vr"], vis)
    sim = similarity(_nrm(o["vc"])[:nloc], _nrm(o["vc"]))
    osim = similarity(_nrm(o["vr"])[:nloc], _nrm(o["vr"]))
    w, wo = round2_weights(ref["amean"], vis, sim, osim, 0.75, 0.99)
    r2c, _ = round2(w, o["vc"])
    r2o, _ = round2(wo, o["vr"])
    assert 0 < int((w > 0).sum()) < int(vis.sum()) and int((wo > 0).sum()) < int((w > 0).sum()), "masks decide nothing"
    start = 0
    for f in range(L):
        m = counts[f]
        if m == 0:
            continue
        rows = torch.cat([torch.arange(start, start + m), torch.arange(nloc, n)])
        oc, orr = oracle.attention_mca_g2l(sd, p, xc[rows][None], xr[rows][None], score[rows], m)
        q = slice(start, start + m)
        xlin_c = F.linear(torch.cat([ref["x_cls"][q], o["vc"][q]], -1), sd[p + "linear.weight"], sd[p + "linear.bias"])
        xlin_r = F.linear(torch.cat([ref["x_reg"][q], o["vr"][q]], -1), sd[p + "linear_reg.weight"], sd[p + "linear_reg.bias"])
        for name, got, want in (("r2c", r2c[q], oc[:, :D]), ("r2o", r2o[q], orr[:, :D]), ("x_c linear", xlin_c, oc[:, D:]),
                                ("x_r linear", xlin_r, orr[:, D:])):
            err = float((got - want).abs().max())
            assert err < 1e-10, f"frame {f}: {name} differs from the oracle by {err:.3e}"
        start += m


def test_reference_matches_msa_oracle():
    sd = {k: v.double() for k, v in oracle.init_stage_weights(5, dim=D, seed=5, gen1=True).items()}
    p = "trans.msa."
    counts = [7, 0, 12, 9]
    n = sum(counts)
    xc, xr, score = _features(n, 9)
    wc, wr = sd[p + "qkv_cls.weight"], sd[p + "qkv_reg.weight"]
    o = _operands(wc[:D], wc[D:], wr[:D], wr[D:], xc, xr, score)
    frame = frame_of_rows(counts)
    vis = visibility(frame, frame, len(counts), True)
    ref = attention(o["qc"], o["kc"], o["qr"], o["kr"], o["vc"], o["vr"], vis)
    w, wo = round2_weights(ref["amean"], vis, similarity(_nrm(o["vc"]), _nrm(o["vc"])), similarity(_nrm(o["vr"]), _nrm(o["vr"])),
                           0.75, 0.99)
    x_c, x_r, r2c, r2o = oracle.attention_msa(sd, p, xc[None], xr[None], score)
    for name, got, want in (("attn @ v_cls", ref["x_cls"], x_c[0, :, :D]), ("attn @ v_reg", ref["x_reg"], x_r[0, :, :D]),
                            ("r2c", w / w.sum(-1, keepdim=True), r2c), ("r2o", wo / wo.sum(-1, keepdim=True), r2o)):
        err = float((got - want).abs().max())
        assert err < 1e-10, f"{name} differs from the oracle by {err:.3e}"
