"""Float64 reference of the MCA / MSA attention kernels (csrc/attn.cu: tscd_attn_pv, tscd_attn_round2), computed from the
16-bit operand buffers the kernels consume, so that a test measures the kernel and not the rounding of its inputs.

Notation: clip b with n keys (bank rows [row_off[b*F], row_off[(b+1)*F])), query row i, 4 heads of 64 columns.
  K(i)      visible keys: the rows of i's own frame plus every row of a global frame (frame index >= L); with self_attn
            every row of the clip.
  s^c_hij = <qn_cls[i,h], kn_cls[j,h]>   (kn_cls already carries 25 * class score),   s^r_hij = <qn_reg[i,h], kn_reg[j,h]>
  a_hij   = (softmax_{j in K(i)}(s^c_hi.) + softmax_{j in K(i)}(s^r_hi.)) / 2
  x_cls[i,h] = sum_j a_hij v_cls[j,h],  x_reg likewise (v = the columns of V^T)
  stats[i] = max_j s^c (h 0..3), max_j s^r (h 0..3), then sum_j exp(s - m) in the same order; in single-pass mode
            (BF16, max_logit > 0) m is max_logit.
  sim_ij  = 1/4 sum_h <vn_cls[i,h], vn_cls[j,h]>,   osim_ij the same over vn_reg
  w_ij    = [j in K(i)] [sim_ij > sim_thresh] exp(1/4 sum_h a_hij)       (what attn_round2's w_out holds)
  wo_ij   = w_ij [osim_ij > conf_sim_thresh]
  round 2 = sum_j w_ij V[j] / sum_j w_ij  (wo for the obj output), V the value matrix the launch aggregates.

This masked whole-clip form equals the reference's per-local-frame loop (oracle.attention_mca_g2l) and its MSA
(oracle.attention_msa); tests/test_attn_ref.py checks that on the CPU.  Everything here is plain torch on float64 tensors of
whatever device they live on; callers chunk by query block (`chunks`) so memory stays bounded."""
import torch

H, HD = 4, 64
U32 = 2.0 ** -24          # fp32 unit roundoff


def frame_of_rows(counts_clip):
    """Frame index (within the clip) of every key of a clip, from its per-frame counts."""
    return torch.repeat_interleave(torch.arange(len(counts_clip)), torch.tensor(counts_clip, dtype=torch.long))


def visibility(frame_q, frame_k, L, self_attn):
    """[m, n] bool: key j is visible to query i."""
    if self_attn:
        return torch.ones(frame_q.numel(), frame_k.numel(), dtype=torch.bool, device=frame_k.device)
    return (frame_q[:, None] == frame_k[None, :]) | (frame_k[None, :] >= L)


def _heads(t):
    return t.reshape(t.shape[0], H, HD)


def attention(qc, kc, qr, kr, vc, vr, vis, max_logit=0.0):
    """attn_pv of one query block.  q* [m,256], k* / v* [n,256] float64, vis [m,n].  Returns dict:
      x_cls, x_reg [m,256]; x_cls_abs, x_reg_abs [m,256] = sum_j a_hij |v_jk| (the scale of the P@V rounding error);
      stats [m,16] as the kernel defines it (maxima of the reference, or max_logit in single-pass mode);
      logit_err [m,8] = 64 * 2^-23 * |q_ih| * max_j |k_jh|: a bound of the fp32 error of one logit (64 products, one
        ulp per addition, which also covers an accumulator that truncates);
      amean [m,n] = 1/4 sum_h a_hij (0 where invisible)."""
    out, a_sum, stats_m, stats_l, lerr = {}, None, [], [], []
    for br, q, k in (("c", qc, kc), ("r", qr, kr)):
        s = torch.einsum("ihd,jhd->hij", _heads(q), _heads(k)).masked_fill(~vis[None], float("-inf"))
        m = s.amax(-1)                                                   # [4, m]
        mu = torch.full_like(m, float(max_logit)) if max_logit > 0 else m
        e = torch.exp(s - mu[..., None])
        l = e.sum(-1)
        p = e / l[..., None]
        a_sum = p if a_sum is None else a_sum + p
        stats_m.append(mu.T)
        stats_l.append(l.T)
        lerr.append(64 * 2 * U32 * _heads(q).norm(dim=-1) * _heads(k).norm(dim=-1).amax(0)[None, :])
    a = 0.5 * a_sum                                                      # [4, m, n]
    for name, v in (("x_cls", vc), ("x_reg", vr)):
        vh = _heads(v)
        out[name] = torch.einsum("hij,jhd->ihd", a, vh).reshape(a.shape[1], H * HD)
        out[name + "_abs"] = torch.einsum("hij,jhd->ihd", a, vh.abs()).reshape(a.shape[1], H * HD)
    out["stats"] = torch.cat(stats_m + stats_l, 1)
    out["logit_err"] = torch.cat(lerr, 1)
    out["amean"] = a.mean(0)
    return out


def similarity(vn_q, vn_k):
    """Head-mean cosine of the normalised raw values: 1/4 sum_h <vn_q[i,h], vn_k[j,h]> = (vn_q @ vn_k^T) / 4."""
    return vn_q @ vn_k.T / H


def round2_weights(amean, vis, sim, osim, sim_thresh, conf_sim_thresh):
    """(w, wo): the cls-launch weights and the obj-launch weights."""
    w = torch.where(vis & (sim > sim_thresh), torch.exp(amean), torch.zeros_like(amean))
    return w, torch.where(osim > conf_sim_thresh, w, torch.zeros_like(w))


def round2(w, V):
    """(sum_j w_ij V_j / sum_j w_ij, sum_j w_ij |V_j| / sum_j w_ij)."""
    den = w.sum(-1, keepdim=True)
    return (w @ V) / den, (w @ V.abs()) / den


def chunks(n, size):
    for i0 in range(0, n, size):
        yield i0, min(n, i0 + size)
