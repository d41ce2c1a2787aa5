"""GPU: the per-frame attentions (tscd_frame_flash, the 16-bit tscd_frame_attention) and the LayerNorm pair
(tscd_residual_ln2 at dim 1024 with the fused objectness head) element by element against float64 references.

Attention reference: per item and head, q and k L2-normalised, no scale, softmax(q^ k^T) v.  The kernels round the
probabilities to 16 bits (u = 2^-11 fp16, 2^-8 BF16) and accumulate in fp32; the output is fp32, so there is no 16-bit store:
    |y - ref| <= 3u * sum_j p_ij |v_jk|  +  16 * 2^-24 * max_j |v_jk|
(one u for the probabilities, the rest covers the fp32 cosines -- at most 128 products -- and accumulation).

LayerNorm reference: y = LN_b(LN_a(x + r)), eps 1e-5, head = <y, head_w> + head_b.  With U32 = 2^-24 and per row
kappa = max|x + r| * rstd_a (large when the mean dwarfs the spread): the first LayerNorm's centred, normalised values are within
E1 = 64 U32 kappa (x + r rounded, the mean from 38 fp32 additions, rstd) of exact, so |dy1_k| <= |w_a_k| E1 (1 + |z1_k|)
+ U32 |y1_k|; the second adds |dy2_k| <= |w_b_k| (2 rstd_b max|dy1| + 64 U32)(1 + |z2_k|); out32 adds U32 |y2|, out16 u |y2|,
head_out sum_k |head_w_k| |dy2_k| + 1024 U32 sum_k |head_w_k y2_k|."""
import pytest
import torch

pytestmark = pytest.mark.gpu

U = {torch.float16: 2.0 ** -11, torch.bfloat16: 2.0 ** -8}
U32 = 2.0 ** -24
DTYPES = [torch.float16, torch.bfloat16]


def _cos_attention(q, k, v, heads):
    """float64 softmax(q^ k^T) v per head, and sum_j p |v| (the bound's scale)."""
    m, n, hd = q.shape[0], k.shape[0], q.shape[1] // heads
    qh = q.view(m, heads, hd) / q.view(m, heads, hd).norm(dim=-1, keepdim=True)
    kh = k.view(n, heads, hd) / k.view(n, heads, hd).norm(dim=-1, keepdim=True)
    p = torch.softmax(torch.einsum("ihd,jhd->hij", qh, kh), -1)
    vh = v.view(n, heads, hd)
    return (torch.einsum("hij,jhd->ihd", p, vh).reshape(m, heads * hd), torch.einsum("hij,jhd->ihd", p, vh.abs()).reshape(m, heads * hd),
            vh.abs().amax(0).reshape(1, heads * hd))


def _check_items(name, out, items, q, k, v, heads, dt):
    u = U[dt]
    worst = 0.0
    for i, (qb, nq, kb, nk) in enumerate(items):
        got = out[qb:qb + nq].double()
        if nk == 0:       # current behaviour: an item without keys leaves its output rows untouched
            assert bool(torch.isnan(got).all()), f"{name}: item {i} has no keys but its rows were written"
            continue
        ref, ref_abs, vmax = _cos_attention(q[qb:qb + nq].double(), k[kb:kb + nk].double(), v[kb:kb + nk].double(), heads)
        r = (got - ref).abs() / (3 * u * ref_abs + 16 * U32 * vmax)
        r = torch.where(torch.isfinite(got), r, torch.full_like(r, float("inf")))
        j = int(torch.argmax(r))
        worst = max(worst, float(r.view(-1)[j]))
        assert float(r.view(-1)[j]) <= 1.0, (f"{name} / {dt}: item {i} (nq {nq}, nk {nk}) query row {j // r.shape[1]} column "
                                             f"{j % r.shape[1]}: {float(got.view(-1)[j]):.6g} vs {float(ref.view(-1)[j]):.6g}")
    print(f"\n{name} / {dt}: worst error / bound {worst:.3f}")


def _ranges(sizes_q, sizes_k, gap):
    """Item row ranges with `gap` unused rows before every item (rows outside every range exist)."""
    items, rq, rk = [], gap, gap
    for nq, nk in zip(sizes_q, sizes_k):
        items.append((rq, nq, rk, nk))
        rq += nq + gap
        rk += nk + gap
    return items, rq, rk


def _untouched_rows(out, items, rows):
    mask = torch.ones(rows, dtype=torch.bool, device=out.device)
    for qb, nq, _, _ in items:
        mask[qb:qb + nq] = False
    return bool(torch.isnan(out[mask]).all())


SIZES = [1, 15, 16, 17, 63, 64, 65, 500, 2048]


def _flash(items, q, k, v, out, heads, hd, dt, max_q):
    from tscd_b200 import ops
    dev = q.device
    t = lambda xs: torch.tensor(xs, dtype=torch.int32, device=dev)           # noqa: E731
    ops.call("tscd_frame_flash", ops.L.FrameFlashArgs, num_items=len(items), heads=heads, head_dim=hd, dtype=dt, max_q=max_q,
             q_beg=t([a for a, _, _, _ in items]), q_end=t([a + b for a, b, _, _ in items]),
             kv_beg=t([c for _, _, c, _ in items]), kv_end=t([c + d for _, _, c, d in items]),
             q=q, ldq=q.stride(0), k=k, ldk=k.stride(0), v=v, ldv=v.stride(0), out=out, ldo=out.stride(0))


@pytest.mark.parametrize("dt", DTYPES)
def test_frame_flash_task_aligned(dt):
    """head_dim 128 x 8 heads, queries = keys = values' rows (TaskAligned); v is the column slice at 1024 of a 2048-pitch tkv."""
    g = torch.Generator(device="cuda").manual_seed(1)
    items, rows, _ = _ranges(SIZES, SIZES, 3)
    q = torch.randn(rows, 1024, generator=g, device="cuda").to(dt)
    tkv = torch.randn(rows, 2048, generator=g, device="cuda").to(dt)
    out = torch.full((rows, 1024), float("nan"), device="cuda")
    _flash(items, q, tkv, tkv[:, 1024:], out, 8, 128, dt, max(SIZES) + 64)
    torch.cuda.synchronize()
    assert _untouched_rows(out, items, rows), "rows outside every item were written"
    _check_items("frame_flash hd128", out, items, q, tkv[:, :1024], tkv[:, 1024:], 8, dt)


@pytest.mark.parametrize("dt", DTYPES)
def test_frame_flash_cafm_step(dt):
    """head_dim 32 x 8 heads, the wide CAFM step: query rows and key / value rows are different ranges, nq != nk, and one
    item has no keys."""
    g = torch.Generator(device="cuda").manual_seed(2)
    sq = SIZES + [40]
    sk = SIZES[3:] + SIZES[:3] + [0]
    items, rq, rk = _ranges(sq, sk, 5)
    q = torch.randn(rq, 256, generator=g, device="cuda").to(dt)
    k = torch.randn(rk, 256, generator=g, device="cuda").to(dt)
    v = torch.randn(rk, 256, generator=g, device="cuda").to(dt)
    out = torch.full((rq, 256), float("nan"), device="cuda")
    _flash(items, q, k, v, out, 8, 32, dt, max(sq) + 100)
    torch.cuda.synchronize()
    assert _untouched_rows(out, [it for it in items if it[3] > 0], rq), "rows outside every item were written"
    _check_items("frame_flash hd32", out, items, q, k, v, 8, dt)


@pytest.mark.parametrize("dt", DTYPES)
def test_frame_attention_16bit(dt):
    """tscd_frame_attention on 16-bit q / k / v (frames of up to 32 rows, head_dim 128 x 8 heads, k | v from one 2048-pitch tkv)."""
    from tscd_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(3)
    sizes = [1, 2, 7, 8, 15, 16, 17, 31, 32, 0, 5, 32, 24]
    lrow = [0]
    for s in sizes:
        lrow.append(lrow[-1] + s)
    rows = lrow[-1] + 16
    q = torch.randn(rows, 1024, generator=g, device="cuda").to(dt)
    tkv = torch.randn(rows, 2048, generator=g, device="cuda").to(dt)
    out = torch.full((rows, 1024), float("nan"), device="cuda")
    ops.call("tscd_frame_attention", ops.L.FrameAttentionArgs, num_frames=len(sizes), heads=8, head_dim=128, in_dtype=dt,
             lrow_off=torch.tensor(lrow, dtype=torch.int32, device="cuda"), q=q, ldq=q.stride(0), k=tkv, ldk=tkv.stride(0),
             v=tkv[:, 1024:], ldv=tkv.stride(0), out=out, ldo=out.stride(0))
    torch.cuda.synchronize()
    assert bool(torch.isnan(out[lrow[-1]:]).all()), "rows past the last frame were written"
    items = [(lrow[i], s, lrow[i], s) for i, s in enumerate(sizes) if s > 0]
    _check_items("frame_attention16", out, items, q, tkv[:, :1024], tkv[:, 1024:], 8, dt)


@pytest.mark.parametrize("dt", DTYPES)
def test_residual_ln2_with_objectness_head(dt):
    """dim 1024, rows_cap above 148 * 8 * 8 = 9472 (the capped grid loops), n_rows < rows_cap (rows past it untouched), and
    rows with a large common offset (mean >> spread)."""
    from tscd_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(4)
    D, rows_cap, n = 1024, 10240, 10000
    x = torch.randn(rows_cap, D, generator=g, device="cuda")
    r = torch.randn(rows_cap, D, generator=g, device="cuda")
    x[:64] += 1000.0                         # mean 1000, spread ~1.4
    r[64:128] = r[64:128] * 0.01 - 300.0
    w_a = 1 + 0.2 * torch.randn(D, generator=g, device="cuda")
    b_a = 0.1 * torch.randn(D, generator=g, device="cuda")
    w_b = 1 + 0.2 * torch.randn(D, generator=g, device="cuda")
    b_b = 0.1 * torch.randn(D, generator=g, device="cuda")
    head_w = torch.randn(D, generator=g, device="cuda") / 32
    head_b = torch.randn(1, generator=g, device="cuda")
    out32 = torch.full((rows_cap, D), float("nan"), device="cuda")
    out16 = torch.full((rows_cap, D), -1, dtype=torch.int16, device="cuda").view(dt)
    head = torch.full((rows_cap,), float("nan"), device="cuda")
    ops.call("tscd_residual_ln2", ops.L.ResidualLn2Args, rows_cap=rows_cap, dim=D,
             n_rows=torch.tensor([n], dtype=torch.int32, device="cuda"), x=x, r=r, w_a=w_a, b_a=b_a, w_b=w_b, b_b=b_b, out_dtype=dt,
             out16=out16, out32=out32, head_w=head_w, head_b=head_b, head_out=head)
    torch.cuda.synchronize()
    assert bool(torch.isnan(out32[n:]).all()) and bool(torch.isnan(head[n:]).all()), "rows past n_rows were written"
    assert bool((out16[n:].view(torch.int16) == -1).all()), "rows past n_rows were written (out16)"

    def ln(t, w, b):
        mu = t.mean(-1, keepdim=True)
        rstd = 1 / ((t - mu).pow(2).mean(-1, keepdim=True) + 1e-5).sqrt()
        z = (t - mu) * rstd
        return z * w + b, z, rstd

    v = x[:n].double() + r[:n].double()
    y1, z1, rstd_a = ln(v, w_a.double(), b_a.double())
    y2, z2, rstd_b = ln(y1, w_b.double(), b_b.double())
    hd = y2 @ head_w.double() + float(head_b)
    kappa = v.abs().amax(-1, keepdim=True) * rstd_a
    dy1 = w_a.double().abs() * (64 * U32 * kappa) * (1 + z1.abs()) + U32 * y1.abs()
    dy2 = w_b.double().abs() * (2 * rstd_b * dy1.amax(-1, keepdim=True) + 64 * U32) * (1 + z2.abs())
    for name, got, bound in (("out32", out32[:n].double(), dy2 + U32 * y2.abs()),
                             ("out16", out16[:n].double(), dy2 + U[dt] * y2.abs())):
        rt = (got - y2).abs() / bound
        j = int(torch.argmax(rt))
        print(f"\nresidual_ln2 {name} / {dt}: worst error / bound {float(rt.view(-1)[j]):.3f}")
        assert float(rt.view(-1)[j]) <= 1.0, f"residual_ln2 {name}: row {j // D} column {j % D}: error {float(rt.view(-1)[j]):.3g} x the bound"
    hb = (head_w.double().abs() * dy2).sum(-1) + 1024 * U32 * (head_w.double() * y2).abs().sum(-1)
    rt = (head[:n].double() - hd).abs() / hb
    j = int(torch.argmax(rt))
    print(f"residual_ln2 head_out / {dt}: worst error / bound {float(rt[j]):.3f}")
    assert float(rt[j]) <= 1.0, f"residual_ln2 head_out: row {j}: error {float(rt[j]):.3g} x the bound"
