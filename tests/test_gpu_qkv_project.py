"""GPU: the fused q|k|v projection (tscd_qkv_project) at the stage's batch shapes.  Every element that the attention
kernels and the MCA linear read must be written: qn of query rows, kn / vn of every row, V^T with its zeroed pad
columns up to the next multiple of 128, x_ori of query rows.  The outputs are checked against the unfused pair
(tscd_linear + tscd_attn_prep) within fp16 tolerance, starting from buffers filled with NaN, and repeated launches must
give identical bytes, also with need_reg=False (the `agg` module), which leaves out the reg branch's V^T and x_ori."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

SENTINEL = -1   # int16 0xffff: a NaN in fp16


def _counts(case, rng):
    if case == "headline":          # OVIS mode A: 148 clips x 32 frames x 30 proposals, 8 local frames
        return 148, 32, 8, [30] * (148 * 32)
    if case == "ovis_l_ragged":     # OVIS-L mode B: 50-500 proposals per frame
        return 6, 12, 4, rng.integers(50, 501, 6 * 12).tolist()
    if case == "vid_l":             # VID-L: one local frame and 31 global frames per clip
        return 32, 32, 1, [30] * (32 * 32)
    # small clips that straddle 128-row tiles, empty frames, and a partial last tile
    c = rng.integers(0, 46, 7 * 5)
    c[3] = 0
    c[10:13] = 0
    return 7, 5, 2, c.tolist()


@pytest.mark.parametrize("case", ["headline", "ovis_l_ragged", "vid_l", "straddle"])
def test_qkv_project_matches_unfused(case):
    from tscd_b200 import aggregate, ops
    dt = torch.float16
    rng = np.random.default_rng(7)
    B, F, L, counts = _counts(case, rng)
    N = sum(counts)
    clip_rows = [sum(counts[b * F:(b + 1) * F]) for b in range(B)]
    loc_rows = [sum(counts[b * F:b * F + L]) for b in range(B)]
    loc_total = sum(loc_rows)
    row_cap = ((N + 127) // 128 + 1) * 128           # the device row count is below the launch's row count
    loc_cap = ((loc_total + 127) // 128) * 128
    nk_pitch = max(128, ((max(clip_rows) + 127) // 128) * 128)
    g = torch.Generator(device="cuda").manual_seed(3)
    cnt = torch.tensor(counts, dtype=torch.int32, device="cuda")
    lay = aggregate.make_layout(cnt, B, F, L, row_cap, loc_cap, nk_pitch, dt)
    bank_c = torch.randn(row_cap, 256, device="cuda", generator=g).to(dt)
    bank_r = torch.randn(row_cap, 256, device="cuda", generator=g).to(dt)
    score = torch.rand(row_cap, device="cuda", generator=g) * 0.9 + 0.05
    w_c = (torch.randn(768, 256, device="cuda", generator=g) / 16).to(dt)
    w_r = (torch.randn(768, 256, device="cuda", generator=g) / 16).to(dt)
    n_dev = torch.tensor([N], dtype=torch.int32, device="cuda")

    def fused(need_reg=True):
        bufs = {n: torch.full((row_cap, 256), SENTINEL, dtype=torch.int16, device="cuda").view(dt)
                for n in ("qn_cls", "kn_cls", "vn_cls", "qn_reg", "kn_reg", "vn_reg")}
        for n in ("vt_cls", "vt_reg")[:2 if need_reg else 1]:
            bufs[n] = torch.full((B * 256, nk_pitch), SENTINEL, dtype=torch.int16, device="cuda").view(dt)
        bufs["row_frame"] = torch.empty(row_cap, dtype=torch.int32, device="cuda")
        bufs["row_meta"] = torch.empty(row_cap, dtype=torch.int32, device="cuda")
        xo_c = torch.full((loc_cap, 512), SENTINEL, dtype=torch.int16, device="cuda").view(dt)
        xo_r = torch.full((loc_cap, 512), SENTINEL, dtype=torch.int16, device="cuda").view(dt)
        ops.qkv_project_fused(lay, bank_c, bank_r, w_c, w_r, score, n_dev, xori_cls=xo_c[:, 256:],
                              xori_reg=xo_r[:, 256:] if need_reg else None, bufs=bufs, need_reg=need_reg)
        return bufs, xo_c[:, 256:], xo_r[:, 256:]

    bufs, xo_c, xo_r = fused()
    bufs2, xo_c2, xo_r2 = fused()
    bufs3, xo_c3, xo_r3 = fused(need_reg=False)   # the `agg` module: no reg V^T, no reg x_ori
    qkv_c, _ = ops.linear(bank_c, w_c, m_dev=n_dev)
    qkv_r, _ = ops.linear(bank_r, w_r, m_dev=n_dev)
    rx_c = torch.empty(loc_cap, 256, dtype=dt, device="cuda")
    rx_r = torch.empty(loc_cap, 256, dtype=dt, device="cuda")
    ref = ops.attn_prep(lay, qkv_c, qkv_r, score, xori_cls=rx_c, xori_reg=rx_r)
    torch.cuda.synchronize()

    starts = np.concatenate([[0], np.cumsum(clip_rows)])
    qrows = torch.from_numpy(np.concatenate([np.arange(starts[b], starts[b] + loc_rows[b]) for b in range(B)])).cuda()

    def check(name, got, want):
        got, want = got.float(), want.float()
        assert not torch.isnan(got).any(), f"{case}: {name} has elements the projection never wrote"
        err = float((got - want).abs().max() / want.abs().max().clamp_min(1e-6))
        assert err < 5e-3, f"{case}: {name} max relative error {err:.2e}"

    for br in ("cls", "reg"):
        check("qn_" + br, bufs["qn_" + br][qrows], ref["qn_" + br][qrows])
        for n in ("kn_", "vn_"):
            check(n + br, bufs[n + br][:N], ref[n + br][:N])
        vt, vt_ref = bufs["vt_" + br].view(B, 256, nk_pitch), ref["vt_" + br].view(B, 256, nk_pitch)
        for b in range(B):
            n, pad = clip_rows[b], min(((clip_rows[b] + 127) // 128) * 128, nk_pitch)
            if n:
                check(f"vt_{br}[clip {b}]", vt[b, :, :n], vt_ref[b, :, :n])
            assert bool((vt[b, :, n:pad].view(torch.int16) == 0).all()), f"{case}: V^T pad of clip {b} is not zero"
    check("x_ori cls", xo_c[:loc_total], rx_c[:loc_total])
    check("x_ori reg", xo_r[:loc_total], rx_r[:loc_total])

    # launches are deterministic: the same bytes in every element read downstream, also when the reg V^T / x_ori are off
    for other, xc_o, reg_vt in ((bufs2, xo_c2, True), (bufs3, xo_c3, False)):
        for br in ("cls", "reg"):
            assert torch.equal(bufs["qn_" + br][qrows].view(torch.int16), other["qn_" + br][qrows].view(torch.int16))
            for n in ("kn_", "vn_"):
                assert torch.equal(bufs[n + br][:N].view(torch.int16), other[n + br][:N].view(torch.int16))
        assert torch.equal(bufs["vt_cls"].view(torch.int16), other["vt_cls"].view(torch.int16))
        assert ("vt_reg" in other) == reg_vt
        assert torch.equal(xo_c[:loc_total].view(torch.int16), xc_o[:loc_total].view(torch.int16))
    assert torch.equal(bufs["vt_reg"].view(torch.int16), bufs2["vt_reg"].view(torch.int16))
    assert torch.equal(xo_r[:loc_total].view(torch.int16), xo_r2[:loc_total].view(torch.int16))
    assert bool((xo_r3.view(torch.int16) == SENTINEL).all()), "x_ori of the reg branch was written with need_reg=False"
