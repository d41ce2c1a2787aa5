"""GPU: the fused q|k|v projection (tscd_qkv_project) at the stage's batch shapes, fp16 and BF16.  Every element that the
attention kernels and the MCA linear read must be written: qn of query rows, kn / vn of every row, V^T with its zeroed pad
columns up to the next multiple of 128, x_ori of query rows.  Both the fused projection and the unfused pair (tscd_linear +
tscd_attn_prep) are checked element by element against a float64 reference of the same 16-bit bank and weights --
per-head L2 normalisation without epsilon, 25 * score folded into kn_cls and 25 into kn_reg, raw v in V^T and x_ori --
starting from buffers filled with NaN, and repeated launches must give identical bytes, also with need_reg=False (the `agg`
module), which leaves out the reg branch's V^T and x_ori.

Bound (u = 2^-11 fp16, 2^-8 BF16): the GEMM sums 256 products in fp32, so an output y_k of x @ w^T is within
e_k = 256 * 2^-23 * (|x| @ |w|^T)_k of exact (one ulp per addition).  Raw v: |v - ref| <= e + u|ref| (16-bit store).  A
per-head normalised output s * y / |y| moves by at most 2 s |e_h| / |y_h| (|e_h| the norm of e over the head) plus the
16-bit store u s |ref|; the unfused pair first stores y in 16 bits, which adds 2 u s, and a few fp32 ulp of s cover the
norm itself."""
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


U = {torch.float16: 2.0 ** -11, torch.bfloat16: 2.0 ** -8}


def _reference(x, w, key_score, scale):
    """float64 (qn, kn, v) of one branch plus their error bounds' ingredients, rows of x."""
    x, w = x.double(), w.double()
    y = x @ w.T
    e = 256 * 2.0 ** -23 * (x.abs() @ w.abs().T)
    out = {}
    for name, c0, s in (("qn", 0, torch.ones(x.shape[0], 1, dtype=torch.float64, device=x.device)),
                        ("kn", 256, scale * (key_score.double()[:, None] if key_score is not None else 1.0) * torch.ones(x.shape[0], 1, dtype=torch.float64, device=x.device)),
                        ("vn", 512, torch.ones(x.shape[0], 1, dtype=torch.float64, device=x.device))):
        yh, eh = y[:, c0:c0 + 256].view(-1, 4, 64), e[:, c0:c0 + 256].view(-1, 4, 64)
        nrm = yh.norm(dim=-1, keepdim=True)
        out[name] = ((yh / nrm) * s[:, :, None]).reshape(-1, 256)
        out[name + "_err"] = (2 * eh.norm(dim=-1, keepdim=True) / nrm * s[:, :, None]).expand(-1, 4, 64).reshape(-1, 256)
        out[name + "_scale"] = s
    out["v"], out["v_err"] = y[:, 512:], e[:, 512:]
    return out


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16], ids=["fp16", "bf16"])
@pytest.mark.parametrize("case", ["headline", "ovis_l_ragged", "vid_l", "straddle"])
def test_qkv_project_matches_unfused(case, dtype):
    from tscd_b200 import aggregate, ops
    dt = dtype
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

    u = U[dt]
    worst = {}

    def check(name, got, want, err_bound, scale, fused):
        got = got.double()
        assert not torch.isnan(got).any(), f"{case}: {name} has elements the projection never wrote"
        bound = err_bound + u * want.abs() + 8 * 2.0 ** -24 * scale + (0.0 if fused else 2 * u * scale)
        r = (got - want).abs() / bound
        k = int(torch.argmax(r))
        key = name.split(" (clip")[0]
        worst[key] = max(worst.get(key, 0.0), float(r.reshape(-1)[k]))
        assert float(r.reshape(-1)[k]) <= 1.0, (f"{case} / {dt}: {name} row {k // r.shape[1]} column {k % r.shape[1]}: "
                                             f"{float(got.reshape(-1)[k]):.6g} vs {float(want.reshape(-1)[k]):.6g}, error "
                                             f"{float(r.reshape(-1)[k]):.3g} x the bound")

    for br, bank, w, ks in (("cls", bank_c, w_c, score), ("reg", bank_r, w_r, None)):
        R = _reference(bank[:N], w, None if ks is None else ks[:N], 25.0)
        qsel = qrows
        for fused, got in ((True, bufs), (False, ref)):
            tag = ("fused " if fused else "unfused ") + br
            check(tag + " qn", got["qn_" + br][qsel], R["qn"][qsel], R["qn_err"][qsel], R["qn_scale"][qsel], fused)
            for n in ("kn", "vn"):
                check(f"{tag} {n}", got[f"{n}_{br}"][:N], R[n], R[n + "_err"], R[n + "_scale"], fused)
            vt = got["vt_" + br].view(B, 256, nk_pitch)
            for b in range(B):
                n, pad = clip_rows[b], min(((clip_rows[b] + 127) // 128) * 128, nk_pitch)
                if n:
                    s0 = int(starts[b])
                    check(f"{tag} V^T (clip {b})", vt[b, :, :n].T, R["v"][s0:s0 + n], R["v_err"][s0:s0 + n], 0.0, True)
                assert bool((vt[b, :, n:pad].view(torch.int16) == 0).all()), f"{case}: {tag} V^T pad of clip {b} is not zero"
        for fused, xo in ((True, xo_c if br == "cls" else xo_r), (False, rx_c if br == "cls" else rx_r)):
            check(("fused " if fused else "unfused ") + br + " x_ori", xo[:loc_total], R["v"][qrows], R["v_err"][qrows], 0.0, True)
    print(f"\n{case} / {dt}: worst error / bound " + ", ".join(f"{k} {v:.3f}" for k, v in worst.items()))

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
