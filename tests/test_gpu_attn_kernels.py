"""GPU: the MCA / MSA attention kernels (tscd_attn_pv, tscd_attn_round2) element by element against the float64 reference
of tests/attn_ref.py, computed from the kernels' own 16-bit operands (qn / kn / vn, V^T) as the q|k|v projection left them.

Every case is a layout the stage or the frame store builds (see _layout), run in three operand modes: fp16 (two-pass
statistics), BF16 with max_logit = 25 (single pass, the production default) and BF16 with max_logit = 0 (two-pass).
Every operand and output buffer starts as a NaN sentinel, so rows the projection never writes (qn of non-query rows, all
rows from N up to row_cap, bank rows past N) are poisoned: a kernel that multiplies an invalid key instead of masking it by
select, or lets a tile that runs past a clip leak into another row, produces a NaN or a wrong value.

Bounds (u = 2^-11 for fp16, 2^-8 for BF16; U32 = 2^-24).  For an output y_ik = sum_j c_ij v_jk / sum_j c_ij the kernels round
the probabilities / weights to 16 bits, accumulate in fp32 and store 16 bits:
    |y - ref| <= 3u * sum_j c_ij |v_jk| / sum_j c_ij  +  u * |ref|  +  floor,
    floor = n_keys(i) * 2^-25 * max_j |v_jk|  (fp16 two-pass: probabilities below 2^-14 are fp16 subnormals of spacing 2^-24
            and the row sum is >= 1)  +  16 * U32 * max_j |v_jk|  (a few fp32 ulp; every path).
stats: a logit is an fp32 sum of 64 products, so it is within  e = 64 * 2^-23 * |q_ih| * max_j |k_jh|  of the exact dot product
(one ulp per addition, allowing truncating accumulation).  Maxima: |m - ref| <= e.  Sums: relative error
<= 2e (every term and the maximum) + 2^-16 (rounding of the exp2 argument, up to 72, and ex2.approx) + n_keys * U32 (fp32
accumulation).  Single-pass mode: stats[0..7] == max_logit exactly.
w_out: exactly 0 where the key is invisible or masked off; elsewhere |w - ref| <= (u + 4 max e + 2^-15) * ref (16-bit rounding;
the head-mean attention is within 4e + 2^-15 of exact); the mask decision equals the reference's for every key outside the
ambiguity band.
Ambiguity band: the kernel forms the similarities as fp32 sums of 256 products (drift ~1e-5), so a key with
|sim - thresh| <= 1e-4 (or the same for osim) may flip; only the rows holding such a key are left out of that output's element
check, their number is printed and must stay below 1 % of the case's query rows.

Clustered features are built so that the masks decide: per head, a cluster member is  c * base + sqrt(1 - c^2) * e_t  with the
e_t orthonormal, and the value projection is block-orthogonal per head, so two members' head-mean cosine is c_a * c_b with c
from LEVELS -- similarities at 1 (exact duplicates), 0.998 / 0.98 (around 0.99) and 0.758 / 0.7243 (around 0.75), all at least
8e-3 from 0.5, 0.75, 0.9 and 0.99, far outside the 16-bit rounding of the operands.  The reg bank has the cls bank's clusters,
and half of them its levels too, so the obj mask splits keys the cls mask keeps in every case.  Because no similarity comes
near a threshold by construction, the ambiguity band excludes no row in these cases (the printed count is 0); it is there
for features whose similarities do fall within 1e-4 of a threshold."""
import numpy as np
import pytest
import torch

from attn_ref import U32, attention, chunks, frame_of_rows, round2, round2_weights, similarity, visibility

pytestmark = pytest.mark.gpu

SENTINEL = -1                    # int16 0xffff: a NaN in fp16 and in BF16
U = {torch.float16: 2.0 ** -11, torch.bfloat16: 2.0 ** -8}
MODES = {"fp16": (torch.float16, 0.0), "bf16_single": (torch.bfloat16, 25.0), "bf16_two": (torch.bfloat16, 0.0)}
LEVELS = (1.0, 0.999, 0.98, 0.7735, 0.725)
BAND = 1e-4
X0, X1 = 256, 512                # column slice of the attn_pv outputs inside 768-wide buffers
O0, O1 = 256, 512                # column slice of the round-2 outputs inside 1024-wide buffers


def _r128(x):
    return (x + 127) // 128 * 128


def _layout(case, rng):
    """(B, F, L, counts, self_attn, nk_pitch or None for the stage's _r128(F * kmax))."""
    if case == "headline":               # OVIS mode A: 148 clips x 32 frames x 30 proposals, 8 local frames
        return 148, 32, 8, [30] * (148 * 32), False, None
    if case == "ovis_l":                 # OVIS-L mode B: 50-500 proposals per frame
        return 2, 32, 8, rng.integers(50, 501, 64).tolist(), False, None
    if case == "vid_l":                  # VID-L: one local frame, 31 global frames
        return 32, 32, 1, [30] * (32 * 32), False, None
    if case == "wide_vid_l":             # wide tier: a 2048-row local frame, globals up to 2048 rows (up to 32 768 keys)
        return 2, 16, 1, [2048] * 16 + [2048] + rng.integers(0, 2049, 15).tolist(), False, None
    if case == "straddle":
        # clips (local f0 f1 | global f2 f3): empty local frame, empty global frame, no local rows, no global rows; local rows
        # 1 / 50 / 0 / 127 / 128 / 129 / 255 / 257, keys 63 / 64 / 65 / 127 / 128 / 129 / 257 / 320; nk_pitch 128 above 384
        c = [1, 0, 40, 22, 30, 20, 0, 14, 0, 0, 33, 32, 100, 27, 0, 0, 128, 0, 0, 0, 64, 65, 0, 0, 200, 55, 1, 1, 1, 256, 60, 3]
        return 8, 4, 2, c, False, 512
    if case == "no_globals":             # F == L: every frame is local, queries see their own frame only
        c = rng.integers(1, 150, 12)
        c[5] = 0
        return 3, 4, 4, c.tolist(), False, None
    if case == "msa":                    # gen-1 MSA: self-attention over every proposal of the clip
        return 2, 32, 32, [30] * 64, True, None
    if case == "msa_ragged":
        return 2, 32, 32, rng.integers(0, 61, 64).tolist(), True, None
    raise KeyError(case)


def _sentinel(*shape, dtype):
    return torch.full(shape, SENTINEL, dtype=torch.int16, device="cuda").view(dtype)


def _clustered(clip_rows, g, like=None):
    """[n, 256] rows in clusters of about 8 rows of the same clip: per head, member t of cluster k is
    c * b_k + sqrt(1 - c^2) e_kt with b_k, e_kt orthonormal.  Returns (rows, (cluster, rank, level)).  like: the structure
    of another bank (the cls bank, when building the reg bank): the same clusters, fresh directions, and in half of the
    clusters the same levels, so that there the obj similarity equals the cls similarity and the obj mask (> 0.99) splits
    the keys the cls mask (> 0.75) keeps."""
    K = 16
    n = sum(clip_rows)
    ncl = torch.tensor([max(1, r // 8) for r in clip_rows], device="cuda")
    nc = int(ncl.sum())
    if like is None:
        clip = torch.repeat_interleave(torch.arange(len(clip_rows), device="cuda"), torch.tensor(clip_rows, device="cuda"))
        pick = torch.rand(n, generator=g, device="cuda")
        cid = (torch.cumsum(ncl, 0) - ncl)[clip] + (pick * ncl[clip]).long().clamp_max(ncl[clip] - 1)
        srt = torch.sort(cid, stable=True)
        rank = torch.empty(n, dtype=torch.long, device="cuda")
        rank[srt.indices] = torch.arange(n, device="cuda") - torch.searchsorted(srt.values, srt.values)
    else:
        cid, rank = like[0], like[1]
    basis = []
    for _ in range(K + 1):
        v = torch.randn(nc, 4, 64, generator=g, device="cuda")
        for b in basis:
            v -= (v * b).sum(-1, keepdim=True) * b
        basis.append(v / v.norm(dim=-1, keepdim=True))
    basis = torch.stack(basis, 2)                                            # [nc, 4, K+1, 64]
    level = torch.tensor(LEVELS, device="cuda")[torch.randint(0, len(LEVELS), (n,), generator=g, device="cuda")]
    if like is not None:
        shared = (torch.rand(nc, generator=g, device="cuda") < 0.5)[cid]
        level = torch.where(shared, like[2], level)
    c = level[:, None, None]
    t = rank.clamp_max(K - 1) + 1
    x = c * basis[cid, :, 0] + (1 - c * c).sqrt() * basis[cid, :, t]
    lone = rank >= K                                                         # clusters larger than K: the rest are loners
    x[lone] = torch.randn(int(lone.sum()), 4, 64, generator=g, device="cuda")
    return 4 * (x / x.norm(dim=-1, keepdim=True)).reshape(n, 256), (cid, rank, level)


def _weights(g, dt):
    """[768, 256] q | k | v projection; v block-orthogonal per head (keeps per-head cosines)."""
    wq = torch.randn(256, 256, generator=g, device="cuda") / 16
    wk = torch.randn(256, 256, generator=g, device="cuda") / 16
    wv = torch.zeros(256, 256, device="cuda")
    for h in range(4):
        wv[h * 64:(h + 1) * 64, h * 64:(h + 1) * 64] = torch.linalg.qr(torch.randn(64, 64, generator=g, device="cuda"))[0]
    return torch.cat([wq, wk, wv]).to(dt).contiguous()


def _build(case, mode, data, seed=5):
    """Seeded bank -> layout -> q|k|v projection (fused, or linear + attn_prep for MSA) into NaN-filled operand buffers."""
    from tscd_b200 import aggregate, ops
    dt, max_logit = MODES[mode]
    B, F, L, counts, self_attn, nk_pitch = _layout(case, np.random.default_rng(seed))
    kmax = max(counts)
    N = sum(counts)
    row_cap = _r128(B * F * kmax) + 128
    nk_pitch = nk_pitch or _r128(F * kmax)
    clip_rows = [sum(counts[b * F:(b + 1) * F]) for b in range(B)]
    loc_rows = clip_rows if self_attn else [sum(counts[b * F:b * F + L]) for b in range(B)]
    loc_cap = row_cap if self_attn else _r128(B * L * kmax)
    g = torch.Generator(device="cuda").manual_seed(seed)
    bank, like = [], None
    for _ in range(2):
        if data.startswith("clustered"):
            x, like = _clustered(clip_rows, g, like)
        else:
            x = torch.randn(N, 256, generator=g, device="cuda")
        t = _sentinel(row_cap, 256, dtype=dt)
        t[:N] = x.to(dt)
        bank.append(t)
    score = torch.full((row_cap,), float("nan"), device="cuda")
    lo, hi = (1e-3, 1e-2) if data.endswith("lowscore") else (0.05, 0.95)
    score[:N] = lo + (hi - lo) * torch.rand(N, generator=g, device="cuda")
    w_c, w_r = _weights(g, dt), _weights(g, dt)
    cnt = torch.tensor(counts, dtype=torch.int32, device="cuda")
    lay = aggregate.make_layout(cnt, B, F, L, row_cap, loc_cap, nk_pitch, dt)
    if self_attn:
        lay.self_attn, lay.lrow_off = True, lay.row_off
    n_dev = torch.tensor([N], dtype=torch.int32, device="cuda")
    bufs = {n: _sentinel(row_cap, 256, dtype=dt) for n in ("qn_cls", "kn_cls", "vn_cls", "qn_reg", "kn_reg", "vn_reg")}
    for n in ("vt_cls", "vt_reg"):
        bufs[n] = _sentinel(B * 256, nk_pitch, dtype=dt)
    bufs["row_frame"] = torch.zeros(row_cap, dtype=torch.int32, device="cuda")
    bufs["row_meta"] = torch.zeros(row_cap, dtype=torch.int32, device="cuda")
    if self_attn:
        qkv_c, _ = ops.linear(bank[0], w_c, m_dev=n_dev)
        qkv_r, _ = ops.linear(bank[1], w_r, m_dev=n_dev)
        ops.attn_prep(lay, qkv_c, qkv_r, score, bufs=bufs)
    else:
        ops.qkv_project_fused(lay, bank[0], bank[1], w_c, w_r, score, n_dev, bufs=bufs)
    off = np.concatenate([[0], np.cumsum(counts)]).tolist()
    lbase = np.concatenate([[0], np.cumsum(loc_rows)]).tolist()
    return dict(case=case, mode=mode, dt=dt, max_logit=max_logit, B=B, F=F, L=L, counts=counts, self_attn=self_attn, N=N,
                row_cap=row_cap, loc_cap=loc_cap, nk_pitch=nk_pitch, clip_rows=clip_rows, loc_rows=loc_rows, lay=lay,
                bufs=bufs, off=off, lbase=lbase, loc_total=sum(loc_rows), g=g)


def _run_pv(S, need_reg=True, drop_vt_reg=False):
    from tscd_b200 import ops
    bufs = {k: v for k, v in S["bufs"].items() if not (drop_vt_reg and k == "vt_reg")}
    xc, xr = _sentinel(S["loc_cap"], 768, dtype=S["dt"]), _sentinel(S["loc_cap"], 768, dtype=S["dt"])
    stats = torch.full((S["loc_cap"], 16), float("nan"), device="cuda")
    ops.attn_pv(S["lay"], bufs, xc[:, X0:X1], xr[:, X0:X1], stats, need_reg=need_reg, max_logit=S["max_logit"])
    return xc, xr, stats


def _run_r2(S, vt, stats, use_obj, thr, w_out=None, w_in=None):
    from tscd_b200 import ops
    out = _sentinel(S["loc_cap"], 1024, dtype=S["dt"])
    ops.attn_round2(S["lay"], S["bufs"], vt, stats, out[:, O0:O1], use_obj_mask=use_obj, sim_thresh=thr[0], conf_sim_thresh=thr[1],
                    w_out=w_out, w_in=w_in)
    return out


class Worst:
    """Worst error / bound per output over every (clip, query block); one host read at the end."""

    def __init__(self, S):
        self.S, self.items = S, {}

    def add(self, name, ratio, b, i0):
        flat = ratio.reshape(-1)
        k = torch.argmax(flat)
        self.items.setdefault(name, []).append((torch.stack([flat[k], k.double()]), b, i0, ratio.shape[1]))

    def check(self):
        S, failures = self.S, []
        for name, lst in self.items.items():
            v = torch.stack([t for t, *_ in lst]).cpu()
            i = int(torch.argmax(v[:, 0]))
            worst, k = float(v[i, 0]), int(v[i, 1])
            _, b, i0, ncol = lst[i]
            row, col = i0 + k // ncol, k % ncol
            print(f"  {name:28s} worst error / bound {worst:.3f}  (clip {b}, query row {row}, column {col})")
            if not worst <= 1.0:
                failures.append(f"{name}: {S['case']} / {S['mode']}: clip {b}, query row {row} (output row "
                                f"{S['lbase'][b] + row}), column {col}: error {worst:.3g} x the bound")
        assert not failures, "\n".join(failures)


def _ratio(got, ref, bound, rows_ok=None):
    r = (got - ref).abs() / bound.clamp_min(1e-300)
    r = torch.where(torch.isfinite(got), r, torch.full_like(r, float("inf")))
    return r if rows_ok is None else r * rows_ok[:, None]


def _views(vt, b, n):
    return vt[b * 256:(b + 1) * 256, :n].T.double()


def _check_case(S, thr, outs, V_r2):
    """Compare every output with the float64 reference.  outs: xc, xr, stats, w_out, r2 outputs by name; V_r2: the value
    matrix each round-2 output aggregated, by name (its V^T buffer)."""
    dt, u = S["dt"], U[S["dt"]]
    two_pass_fp16 = dt == torch.float16
    W = Worst(S)
    F, L = S["F"], S["L"]
    n_band_c = n_band_o = 0
    bufs = S["bufs"]
    qchunk = 256 if max(S["clip_rows"]) > 8192 else 512
    for b in range(S["B"]):
        n, nq = S["clip_rows"][b], S["loc_rows"][b]
        if nq == 0:
            continue
        s0, lb = S["off"][b * F], S["lbase"][b]
        frame = frame_of_rows(S["counts"][b * F:(b + 1) * F]).cuda()
        op = {k: bufs[k][s0:s0 + n].double() for k in ("qn_cls", "kn_cls", "qn_reg", "kn_reg", "vn_cls", "vn_reg")}
        vc, vr = _views(bufs["vt_cls"], b, n), _views(bufs["vt_reg"], b, n)
        Vs = {name: _views(vt, b, n) for name, vt in V_r2.items()}
        # max_j |v_jk| over the visible keys of each row: own frame's maximum combined with the globals' maximum
        def vmax_of(V):
            fm = torch.zeros(F, 256, dtype=torch.float64, device="cuda").index_reduce_(0, frame, V.abs(), "amax")
            if S["self_attn"]:
                return fm.amax(0, keepdim=True).expand(F, 256)
            return torch.maximum(fm, V[S["loc_rows"][b]:].abs().amax(0, keepdim=True) if n > nq else torch.zeros_like(fm[:1]))
        vmax = {k: vmax_of(V) for k, V in list(Vs.items()) + [("x_cls", vc), ("x_reg", vr)]}
        for i0, i1 in chunks(nq, qchunk):
            vis = visibility(frame[i0:i1], frame, L, S["self_attn"])
            nvis = vis.sum(1, keepdim=True).double()
            r = attention(op["qn_cls"][i0:i1], op["kn_cls"], op["qn_reg"][i0:i1], op["kn_reg"], vc, vr, vis, S["max_logit"])
            rows = slice(lb + i0, lb + i1)
            # ---- attn_pv: x_cls / x_reg ----
            for name, got in (("x_cls", outs["xc"]), ("x_reg", outs["xr"])):
                ref = r[name]
                vm = vmax[name][frame[i0:i1]]
                floor = (nvis * 2.0 ** -25 if two_pass_fp16 else 0.0) * vm + 16 * U32 * vm
                bound = 3 * u * r[name + "_abs"] + u * ref.abs() + floor
                W.add("attn_pv " + name, _ratio(got[rows, X0:X1].double(), ref, bound), b, i0)
            # ---- attn_pv: stats ----
            st = outs["stats"][rows].double()
            e = r["logit_err"]
            if S["max_logit"] > 0:
                W.add("attn_pv stats max (== max_logit)", torch.where(st[:, :8] == S["max_logit"], 0.0, float("inf")), b, i0)
            else:
                W.add("attn_pv stats max", _ratio(st[:, :8], r["stats"][:, :8], e), b, i0)
            rel = 2 * e + 2.0 ** -16 + nvis * U32
            W.add("attn_pv stats sum", _ratio(st[:, 8:], r["stats"][:, 8:], rel * r["stats"][:, 8:]), b, i0)
            # ---- attn_round2: masks, weights ----
            sim = similarity(op["vn_cls"][i0:i1], op["vn_cls"])
            osim = similarity(op["vn_reg"][i0:i1], op["vn_reg"])
            band_c = (vis & ((sim - thr[0]).abs() <= BAND)).any(1)
            band_o = band_c | (vis & ((osim - thr[1]).abs() <= BAND)).any(1)
            n_band_c += int(band_c.sum())
            n_band_o += int(band_o.sum())
            w, wo = round2_weights(r["amean"], vis, sim, osim, thr[0], thr[1])
            gw = outs["w_out"][rows, :n].double()
            wb = (u + 4 * e.amax(1, keepdim=True) + 2.0 ** -15) * w
            wr = _ratio(gw, w, wb, ~band_c)
            wr = torch.where(~vis & (gw != 0), float("inf"), wr)                          # invisible keys: exactly 0
            wr = torch.where(vis & ~band_c[:, None] & ((gw != 0) != (w > 0)), float("inf"), wr)   # mask decisions
            W.add("attn_round2 w_out", wr, b, i0)
            # ---- attn_round2 outputs ----
            for name, got in outs["r2"].items():
                use_obj = name.startswith("obj")
                ref, ref_abs = round2(wo if use_obj else w, Vs[name])
                vm = vmax[name][frame[i0:i1]]
                bound = 3 * u * ref_abs + u * ref.abs() + 16 * U32 * vm
                W.add("attn_round2 " + name, _ratio(got[rows, O0:O1].double(), ref, bound, ~(band_o if use_obj else band_c)), b, i0)
    nq_total = S["loc_total"]
    print(f"  band-excluded rows: {n_band_c} (cls masks), {n_band_o} (cls or obj masks) of {nq_total} query rows")
    W.check()
    assert n_band_o <= 0.01 * nq_total, f"{S['case']}: {n_band_o} of {nq_total} query rows hold a key in the ambiguity band"


def _assert_untouched(S, name, buf, c0, c1):
    """Rows at or past the local total, and columns outside [c0, c1), still hold the sentinel."""
    bits = buf.view(torch.int16) if buf.dtype != torch.float32 else None
    lt = S["loc_total"]
    if bits is not None:
        assert bool((bits[lt:] == SENTINEL).all()), f"{S['case']}: {name} written at rows >= {lt}"
        assert bool((bits[:, :c0] == SENTINEL).all()) and bool((bits[:, c1:] == SENTINEL).all()), \
            f"{S['case']}: {name} written outside its column slice"
    else:
        assert bool(torch.isnan(buf[lt:]).all()), f"{S['case']}: {name} written at rows >= {lt}"


def _same(a, b):
    return torch.equal(a.view(torch.int16) if a.dtype != torch.float32 else a.view(torch.int32),
                       b.view(torch.int16) if b.dtype != torch.float32 else b.view(torch.int32))


PARAMS = [(c, m, d) for c in ("headline", "ovis_l", "vid_l", "wide_vid_l", "no_globals", "msa", "msa_ragged")
          for m, d in (("fp16", "clustered"), ("bf16_single", "clustered_lowscore"), ("bf16_two", "plain"))]
PARAMS += [("straddle", m, d) for m in MODES for d in ("plain", "clustered", "clustered_lowscore")]


@pytest.mark.parametrize("case,mode,data", PARAMS)
def test_attn_kernels_vs_float64(case, mode, data):
    _attn_case(case, mode, data, (0.75, 0.99))


def test_attn_round2_thresholds_are_used():
    """Non-default thresholds (0.5 / 0.9): masks at other similarities than the defaults'."""
    _attn_case("straddle", "fp16", "clustered", (0.5, 0.9))


def _attn_case(case, mode, data, thr):
    from tscd_b200 import ops
    S = _build(case, mode, data)
    dt, lt, B, nk = S["dt"], S["loc_total"], S["B"], S["nk_pitch"]
    print(f"\n{case} / {mode} / {data} / thresholds {thr}: B {B}, F {S['F']}, L {S['L']}, N {S['N']}, query rows {lt}, nk_pitch {nk}")
    xc, xr, stats = _run_pv(S)
    w_out = _sentinel(S["loc_cap"], nk, dtype=dt)
    if S["self_attn"]:
        # gen-1 MSA: round 2 aggregates linear1's output (here a seeded 16-bit [N, 512] matrix) through tscd_transpose_clip,
        # one 256-column half per launch
        tc = _sentinel(S["row_cap"], 512, dtype=dt)
        tc[:S["N"]] = torch.randn(S["N"], 512, generator=S["g"], device="cuda").to(dt)
        tct = _sentinel(B * 512, nk, dtype=dt)
        ops.call("tscd_transpose_clip", ops.L.TransposeArgs, lay=S["lay"].to_c(), width=512, x=tc, ld_x=tc.stride(0), xt=tct)
        halves = [tct.view(B, 512, nk)[:, h * 256:(h + 1) * 256].contiguous().view(B * 256, nk) for h in range(2)]
        r2 = {"half0": _run_r2(S, halves[0], stats, False, thr, w_out=w_out), "half1": _run_r2(S, halves[1], stats, False, thr)}
        V_r2 = {"half0": halves[0], "half1": halves[1]}
    else:
        cls = _run_r2(S, S["bufs"]["vt_cls"], stats, False, thr, w_out=w_out)
        obj_win = _run_r2(S, S["bufs"]["vt_reg"], stats, True, thr, w_in=w_out)
        obj_re = _run_r2(S, S["bufs"]["vt_reg"], stats, True, thr)
        r2 = {"cls": cls, "obj (w_in)": obj_win, "obj (recompute)": obj_re}
        V_r2 = {"cls": S["bufs"]["vt_cls"], "obj (w_in)": S["bufs"]["vt_reg"], "obj (recompute)": S["bufs"]["vt_reg"]}
    torch.cuda.synchronize()

    # nothing is written outside the outputs
    for name, buf, c0, c1 in (("x_cls", xc, X0, X1), ("x_reg", xr, X0, X1), ("w_out", w_out, 0, nk)) + \
            tuple(("round 2 " + k, v, O0, O1) for k, v in r2.items()):
        _assert_untouched(S, name, buf, c0, c1)
    _assert_untouched(S, "stats", stats, 0, 16)

    _check_case(S, thr, dict(xc=xc, xr=xr, stats=stats, w_out=w_out, r2=r2), V_r2)

    if not S["self_attn"]:
        # the w_in launch reads no w_out column at or past its clip's key count
        w_poison = w_out.clone()
        for b in range(B):
            l0, l1 = S["lbase"][b], S["lbase"][b + 1]
            w_poison[l0:l1, S["clip_rows"][b]:] = float("nan")
        again = _run_r2(S, S["bufs"]["vt_reg"], stats, True, thr, w_in=w_poison)
        torch.cuda.synchronize()
        assert _same(again, r2["obj (w_in)"]), f"{case}: the w_in launch depends on w_out columns past the clip"

    # need_reg = 0 without a reg V^T: the same x_cls bytes, x_reg untouched
    xc0, xr0, st0 = _run_pv(S, need_reg=False, drop_vt_reg=True)
    torch.cuda.synchronize()
    assert _same(xc0, xc), f"{case}: x_cls differs between need_reg = 1 and need_reg = 0"
    assert bool((xr0.view(torch.int16) == SENTINEL).all()), f"{case}: x_reg written with need_reg = 0"
    assert _same(st0, stats), f"{case}: stats differ between need_reg = 1 and need_reg = 0"

    # rejected argument combinations launch nothing
    xc1, xr1, st1 = _sentinel(S["loc_cap"], 768, dtype=dt), _sentinel(S["loc_cap"], 768, dtype=dt), torch.full_like(stats, float("nan"))
    with pytest.raises(RuntimeError):
        ops.attn_pv(S["lay"], {k: v for k, v in S["bufs"].items() if k != "vt_reg"}, xc1[:, X0:X1], xr1[:, X0:X1], st1, need_reg=True,
                    max_logit=S["max_logit"])
    out1 = _sentinel(S["loc_cap"], 1024, dtype=dt)
    with pytest.raises(RuntimeError):
        ops.attn_round2(S["lay"], S["bufs"], S["bufs"]["vt_cls"], stats, out1[:, O0:O1], use_obj_mask=False, w_in=w_out)
    torch.cuda.synchronize()
    for t in (xc1, xr1, out1):
        assert bool((t.view(torch.int16) == SENTINEL).all()), f"{case}: a rejected call wrote its output"
    assert bool(torch.isnan(st1).all())

    # two further launches: identical bytes in every output
    for _ in range(2):
        xc2, xr2, st2 = _run_pv(S)
        w2 = _sentinel(S["loc_cap"], nk, dtype=dt)
        if S["self_attn"]:
            same = _same(_run_r2(S, V_r2["half0"], st2, False, thr, w_out=w2), r2["half0"])
        else:
            same = _same(_run_r2(S, S["bufs"]["vt_cls"], st2, False, thr, w_out=w2), r2["cls"]) and \
                _same(_run_r2(S, S["bufs"]["vt_reg"], st2, True, thr, w_in=w2), r2["obj (w_in)"])
        torch.cuda.synchronize()
        assert _same(xc2, xc) and _same(xr2, xr) and _same(st2, stats) and _same(w2, w_out) and same, f"{case}: launches differ"
