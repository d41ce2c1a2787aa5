// Tail of the stage: TaskAligned cosine attention per frame, the two LayerNorms, and the final per-class
// expansion feeding the last class-aware NMS.
//
// Reference: TaskAligned.forward / CrossAttentionLayer.forward_post / MHAttention.forward
// (yolox/models/tscd_matching.py:1107-1139, 421-433, 159-181), decode_reg_preds5 (yolox/models/tscd_head.py:
// 914-949) and postprocess (yolox/models/post_process.py:9-85).
#include "common.cuh"
#include "mma.cuh"

namespace tscd {

// ---------------------------------------------------------------------------------------------- frame attention
// One CTA per (local frame, head).  Keys/values stream through shared memory in chunks of 64 (one chunk for the
// usual <= 64 proposals per frame) with an online softmax; each warp owns query rows, lanes own keys (scores) then
// output dims (weighted sum).  All shared-memory traffic is 128-bit: the kernel is shared-memory-bandwidth bound.
constexpr int kFaChunk = 64;

__global__ void __launch_bounds__(256, 2) frame_attention_kernel(const tscd_frame_attention_args a) {
    extern __shared__ __align__(16) float fa_smem[];
    const int hd = a.head_dim;           // multiple of 32, <= 128
    const int pitch = hd + 4;            // rows stay 16-byte aligned; 4-float skew keeps float4 row reads conflict-free
    float* sK = fa_smem;                  // [64][hd+4] normalised keys
    float* sV = sK + kFaChunk * pitch;    // [64][hd]
    float* sQ = sV + kFaChunk * hd;       // [8 warps][hd] normalised query rows
    const int lf = blockIdx.x, h = blockIdx.y;
    const int l0 = a.lrow_off[lf], n = a.lrow_off[lf + 1] - l0;
    if (n <= 0) return;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int nd = hd / 32;               // output dims per lane (<= 4)
    float* myq = sQ + warp * hd;
    const bool single = n <= kFaChunk;    // keys / values staged once for all query rows

    auto stage = [&](int k0, int kc) {
        for (int j = warp; j < kc; j += 8) {   // stage + normalise keys, copy values
            const float* kr = reinterpret_cast<const float*>(a.k) + (int64_t)(l0 + k0 + j) * a.ldk + h * hd;
            const float* vr = reinterpret_cast<const float*>(a.v) + (int64_t)(l0 + k0 + j) * a.ldv + h * hd;
            float kv[4], ks = 0.f;
#pragma unroll
            for (int t = 0; t < 4; ++t)
                if (t < nd) { kv[t] = kr[lane + 32 * t]; ks = fmaf(kv[t], kv[t], ks); sV[j * hd + lane + 32 * t] = vr[lane + 32 * t]; }
            ks = warp_sumf(ks);
            const float inv = 1.f / sqrtf(ks);
#pragma unroll
            for (int t = 0; t < 4; ++t)
                if (t < nd) sK[j * pitch + lane + 32 * t] = kv[t] * inv;
        }
    };
    if (single) { stage(0, n); __syncthreads(); }

    for (int rb = 0; rb < n; rb += 8) {   // 8 query rows per pass (one per warp)
        const int r = rb + warp;
        const bool r_ok = r < n;
        float qs = 0.f;
        if (r_ok) {
            for (int d = lane; d < hd; d += 32) { const float x = reinterpret_cast<const float*>(a.q)[(int64_t)(l0 + r) * a.ldq + h * hd + d]; myq[d] = x; qs = fmaf(x, x, qs); }
        }
        qs = warp_sumf(qs);
        if (r_ok) { const float inv = 1.f / sqrtf(qs); for (int d = lane; d < hd; d += 32) myq[d] *= inv; }
        __syncwarp();
        float m = -INFINITY, l = 0.f, acc[4] = {0.f, 0.f, 0.f, 0.f};
        for (int k0 = 0; k0 < n; k0 += kFaChunk) {
            const int kc = min(kFaChunk, n - k0);
            if (!single) {
                __syncthreads();
                stage(k0, kc);
                __syncthreads();
            }
            if (r_ok) {
                float s0 = 0.f, s1 = 0.f;
                const float4* q4 = reinterpret_cast<const float4*>(myq);
                const float4* ka = reinterpret_cast<const float4*>(sK + min(lane, kc - 1) * pitch);
                const float4* kb = reinterpret_cast<const float4*>(sK + min(lane + 32, kc - 1) * pitch);
                const bool two = kc > 32;
                for (int d = 0; d < hd / 4; ++d) {
                    const float4 qq = q4[d], x = ka[d];
                    s0 = fmaf(qq.x, x.x, fmaf(qq.y, x.y, fmaf(qq.z, x.z, fmaf(qq.w, x.w, s0))));
                    if (two) {
                        const float4 y = kb[d];
                        s1 = fmaf(qq.x, y.x, fmaf(qq.y, y.y, fmaf(qq.z, y.z, fmaf(qq.w, y.w, s1))));
                    }
                }
                if (lane >= kc) s0 = -INFINITY;
                if (lane + 32 >= kc) s1 = -INFINITY;
                const float mn = fmaxf(m, warp_maxf(fmaxf(s0, s1)));
                const float corr = expf(m - mn);
                const float p0 = (lane < kc) ? expf(s0 - mn) : 0.f;
                const float p1 = (lane + 32 < kc) ? expf(s1 - mn) : 0.f;
                l = l * corr + warp_sumf(p0 + p1);
#pragma unroll
                for (int t = 0; t < 4; ++t) acc[t] *= corr;
                for (int j = 0; j < kc; ++j) {
                    const float pj = __shfl_sync(0xffffffffu, j < 32 ? p0 : p1, j & 31);
#pragma unroll
                    for (int t = 0; t < 4; ++t)
                        if (t < nd) acc[t] = fmaf(pj, sV[j * hd + lane + 32 * t], acc[t]);
                }
                m = mn;
            }
        }
        if (r_ok) {
            const float inv = 1.f / l;
#pragma unroll
            for (int t = 0; t < 4; ++t)
                if (t < nd) a.out[(int64_t)(l0 + r) * a.ldo + h * hd + lane + 32 * t] = acc[t] * inv;
        }
        __syncwarp();
    }
}

// ---------------------------------------------------------------------------------------------- frame attention, tensor cores
// Frames of at most 32 proposals, head_dim 128, 16-bit q/k/v (the GEMM's 16-bit outputs).  One CTA per (frame, half of the
// heads): the frame's q, k, v head slices are staged with cp.async, warp = (head, 16-row tile).  S = q k^T on mma.sync
// (8 k-steps), cosine by scaling the fp32 scores with 1/|q_r| and 1/|k_j|, softmax in registers, P fed to P @ v straight
// from the accumulator layout.  Output fp32 (it feeds the residual LayerNorm).
constexpr int kFa16Pitch = 136;     // 16-bit elements per staged row: 128 + 8 (272 B -> ldmatrix conflict-free)
constexpr int kFa16Heads = 4;       // heads per CTA

template <typename T>
__global__ void __launch_bounds__(256, 2) frame_attention16_kernel(const tscd_frame_attention_args a) {
    extern __shared__ __align__(16) unsigned char fa16_smem[];
    T* sQ = reinterpret_cast<T*>(fa16_smem);                        // [4 heads][32][136]
    T* sK = sQ + kFa16Heads * 32 * kFa16Pitch;
    T* sV = sK + kFa16Heads * 32 * kFa16Pitch;
    float* sQn = reinterpret_cast<float*>(sV + kFa16Heads * 32 * kFa16Pitch);   // [4][32] 1/|q|
    float* sKn = sQn + kFa16Heads * 32;
    const int lf = blockIdx.x, h0 = blockIdx.y * kFa16Heads;
    const int l0 = a.lrow_off[lf], n = a.lrow_off[lf + 1] - l0;
    if (n <= 0) return;
    if (n > 32) __trap();                     // host contract: this variant is only launched for kmax <= 32
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int g = lane >> 2, t4 = lane & 3;
    const T* q = reinterpret_cast<const T*>(a.q);
    const T* k = reinterpret_cast<const T*>(a.k);
    const T* v = reinterpret_cast<const T*>(a.v);
    // stage: 3 matrices x 4 heads x n rows x 16 chunks of 16 bytes
    for (int i = tid; i < 3 * kFa16Heads * 32 * 16; i += 256) {
        const int ch = i & 15, r = (i >> 4) & 31, hh = (i >> 9) & 3, m = i >> 11;
        T* dst = (m == 0 ? sQ : (m == 1 ? sK : sV)) + (hh * 32 + r) * kFa16Pitch + ch * 8;
        if (r < n) {
            const T* src = (m == 0 ? q + (int64_t)(l0 + r) * a.ldq : (m == 1 ? k + (int64_t)(l0 + r) * a.ldk : v + (int64_t)(l0 + r) * a.ldv)) +
                           (h0 + hh) * 128 + ch * 8;
            cp_async16(dst, src);
        } else {
            *reinterpret_cast<uint4*>(dst) = make_uint4(0, 0, 0, 0);     // padding rows: finite (keys masked, values x 0)
        }
    }
    cp_async_commit();
    cp_async_wait_all();
    __syncthreads();
    // 1 / |q_r|, 1 / |k_j| per head: one thread per (matrix, head, row)
    {
        const int r = tid & 31, hh = (tid >> 5) & 3, m = tid >> 7;
        const T* row = (m == 0 ? sQ : sK) + (hh * 32 + r) * kFa16Pitch;
        float ss = 0.f;
#pragma unroll
        for (int c = 0; c < 16; ++c) {
            float x[8];
            load8(row + c * 8, x);
#pragma unroll
            for (int i = 0; i < 8; ++i) ss = fmaf(x[i], x[i], ss);
        }
        (m == 0 ? sQn : sKn)[hh * 32 + r] = 1.f / sqrtf(ss);
    }
    __syncthreads();
    const int hh = warp >> 1, mt = warp & 1;
    if (mt * 16 >= n) return;
    const T* Qh = sQ + hh * 32 * kFa16Pitch;
    const T* Kh = sK + hh * 32 * kFa16Pitch;
    const T* Vh = sV + hh * 32 * kFa16Pitch;
    float sc[4][4];
#pragma unroll
    for (int nt = 0; nt < 4; ++nt) sc[nt][0] = sc[nt][1] = sc[nt][2] = sc[nt][3] = 0.f;
#pragma unroll
    for (int ks = 0; ks < 8; ++ks) {
        uint32_t qa[4];
        ldsm_x4(qa, Qh + (mt * 16 + (lane & 15)) * kFa16Pitch + ks * 16 + (lane >> 4) * 8);
#pragma unroll
        for (int ntp = 0; ntp < 2; ++ntp) {       // two key n-tiles per ldmatrix.x4: (keys 16ntp..+7, k lo/hi), (keys +8.., k lo/hi)
            uint32_t kb[4];
            ldsm_x4(kb, Kh + (ntp * 16 + (lane & 7) + ((lane >> 4) & 1) * 8) * kFa16Pitch + ks * 16 + ((lane >> 3) & 1) * 8);
            mma16816<T>(sc[2 * ntp], qa, kb[0], kb[1]);
            mma16816<T>(sc[2 * ntp + 1], qa, kb[2], kb[3]);
        }
    }
    const int R0 = mt * 16 + g, R1 = R0 + 8;
    const float iq0 = sQn[hh * 32 + R0], iq1 = sQn[hh * 32 + R1];
    float mx0 = -INFINITY, mx1 = -INFINITY;
#pragma unroll
    for (int nt = 0; nt < 4; ++nt) {
        const int j0 = nt * 8 + 2 * t4;
        const float ik0 = sKn[hh * 32 + j0], ik1 = sKn[hh * 32 + j0 + 1];
        sc[nt][0] = j0 < n ? sc[nt][0] * iq0 * ik0 : -INFINITY;
        sc[nt][1] = j0 + 1 < n ? sc[nt][1] * iq0 * ik1 : -INFINITY;
        sc[nt][2] = j0 < n ? sc[nt][2] * iq1 * ik0 : -INFINITY;
        sc[nt][3] = j0 + 1 < n ? sc[nt][3] * iq1 * ik1 : -INFINITY;
        mx0 = fmaxf(mx0, fmaxf(sc[nt][0], sc[nt][1]));
        mx1 = fmaxf(mx1, fmaxf(sc[nt][2], sc[nt][3]));
    }
    mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 1)); mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 2));
    mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 1)); mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 2));
    float sum0 = 0.f, sum1 = 0.f;
#pragma unroll
    for (int nt = 0; nt < 4; ++nt) {
        sc[nt][0] = expf(sc[nt][0] - mx0); sc[nt][1] = expf(sc[nt][1] - mx0);
        sc[nt][2] = expf(sc[nt][2] - mx1); sc[nt][3] = expf(sc[nt][3] - mx1);
        sum0 += sc[nt][0] + sc[nt][1];
        sum1 += sc[nt][2] + sc[nt][3];
    }
    sum0 += __shfl_xor_sync(0xffffffffu, sum0, 1); sum0 += __shfl_xor_sync(0xffffffffu, sum0, 2);
    sum1 += __shfl_xor_sync(0xffffffffu, sum1, 1); sum1 += __shfl_xor_sync(0xffffffffu, sum1, 2);
    const float is0 = 1.f / sum0, is1 = 1.f / sum1;
    uint32_t pa[2][4];
#pragma unroll
    for (int ks = 0; ks < 2; ++ks) {
        pa[ks][0] = pack2<T>(sc[2 * ks][0] * is0, sc[2 * ks][1] * is0);
        pa[ks][1] = pack2<T>(sc[2 * ks][2] * is1, sc[2 * ks][3] * is1);
        pa[ks][2] = pack2<T>(sc[2 * ks + 1][0] * is0, sc[2 * ks + 1][1] * is0);
        pa[ks][3] = pack2<T>(sc[2 * ks + 1][2] * is1, sc[2 * ks + 1][3] * is1);
    }
    float* out0 = a.out + (int64_t)(l0 + R0) * a.ldo + (h0 + hh) * 128;
    float* out1 = a.out + (int64_t)(l0 + R1) * a.ldo + (h0 + hh) * 128;
#pragma unroll
    for (int ntp = 0; ntp < 8; ++ntp) {           // 16 output dims per iteration
        float o0[4] = {0.f, 0.f, 0.f, 0.f}, o1[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int ks = 0; ks < 2; ++ks) {
            uint32_t vb[4];
            ldsm_x4_trans(vb, Vh + (ks * 16 + (lane & 7) + ((lane >> 3) & 1) * 8) * kFa16Pitch + ntp * 16 + (lane >> 4) * 8);
            mma16816<T>(o0, pa[ks], vb[0], vb[1]);
            mma16816<T>(o1, pa[ks], vb[2], vb[3]);
        }
        const int col = ntp * 16 + 2 * t4;
        if (R0 < n) {
            *reinterpret_cast<float2*>(out0 + col) = make_float2(o0[0], o0[1]);
            *reinterpret_cast<float2*>(out0 + col + 8) = make_float2(o1[0], o1[1]);
        }
        if (R1 < n) {
            *reinterpret_cast<float2*>(out1 + col) = make_float2(o0[2], o0[3]);
            *reinterpret_cast<float2*>(out1 + col + 8) = make_float2(o1[2], o1[3]);
        }
    }
}

// ---------------------------------------------------------------------------------------------- LN(LN(x + r))
template <typename T>
__global__ void __launch_bounds__(256) residual_ln2_kernel(const tscd_residual_ln2_args a) {
    extern __shared__ __align__(16) float ln_smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n = min(a.rows_cap, a.n_rows ? __ldg(a.n_rows) : a.rows_cap);
    const int D = a.dim;
    if (D == 1024) {
        // TSCD-L width: the row lives in registers (8 float4 per lane, 16-byte loads), no shared memory
        for (int r = blockIdx.x * 8 + warp; r < n; r += gridDim.x * 8) {
            const float4* xp = reinterpret_cast<const float4*>(a.x + (int64_t)r * D);
            const float4* rp = reinterpret_cast<const float4*>(a.r + (int64_t)r * D);
            float4 v[8];
            float s = 0.f;
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const float4 p = __ldg(xp + i * 32 + lane), q = __ldg(rp + i * 32 + lane);
                v[i] = make_float4(p.x + q.x, p.y + q.y, p.z + q.z, p.w + q.w);
                s += (v[i].x + v[i].y) + (v[i].z + v[i].w);
            }
            float mean = warp_sumf(s) / D, var = 0.f;
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const float dx = v[i].x - mean, dy = v[i].y - mean, dz = v[i].z - mean, dw = v[i].w - mean;
                var = fmaf(dx, dx, fmaf(dy, dy, fmaf(dz, dz, fmaf(dw, dw, var))));
            }
            float rstd = rsqrtf(warp_sumf(var) / D + 1e-5f);
            s = 0.f;
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const float4 w = __ldg(reinterpret_cast<const float4*>(a.w_a) + i * 32 + lane), b = __ldg(reinterpret_cast<const float4*>(a.b_a) + i * 32 + lane);
                v[i] = make_float4((v[i].x - mean) * rstd * w.x + b.x, (v[i].y - mean) * rstd * w.y + b.y,
                                   (v[i].z - mean) * rstd * w.z + b.z, (v[i].w - mean) * rstd * w.w + b.w);
                s += (v[i].x + v[i].y) + (v[i].z + v[i].w);
            }
            mean = warp_sumf(s) / D; var = 0.f;
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const float dx = v[i].x - mean, dy = v[i].y - mean, dz = v[i].z - mean, dw = v[i].w - mean;
                var = fmaf(dx, dx, fmaf(dy, dy, fmaf(dz, dz, fmaf(dw, dw, var))));
            }
            rstd = rsqrtf(warp_sumf(var) / D + 1e-5f);
            float hd = 0.f;
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const float4 w = __ldg(reinterpret_cast<const float4*>(a.w_b) + i * 32 + lane), b = __ldg(reinterpret_cast<const float4*>(a.b_b) + i * 32 + lane);
                const float4 y = make_float4((v[i].x - mean) * rstd * w.x + b.x, (v[i].y - mean) * rstd * w.y + b.y,
                                             (v[i].z - mean) * rstd * w.z + b.z, (v[i].w - mean) * rstd * w.w + b.w);
                if (a.head_w) {
                    const float4 hw = __ldg(reinterpret_cast<const float4*>(a.head_w) + i * 32 + lane);
                    hd = fmaf(y.x, hw.x, fmaf(y.y, hw.y, fmaf(y.z, hw.z, fmaf(y.w, hw.w, hd))));
                }
                const int64_t o = (int64_t)r * D + (i * 32 + lane) * 4;
                if (a.out16) {
                    *reinterpret_cast<uint2*>(reinterpret_cast<T*>(a.out16) + o) = make_uint2(pack2<T>(y.x, y.y), pack2<T>(y.z, y.w));
                }
                if (a.out32) *reinterpret_cast<float4*>(a.out32 + o) = y;
            }
            if (a.head_w) {
                hd = warp_sumf(hd);
                if (lane == 0) a.head_out[r] = hd + __ldg(a.head_b);
            }
        }
        return;
    }
    float* buf = ln_smem + warp * D;
    for (int r = blockIdx.x * 8 + warp; r < n; r += gridDim.x * 8) {
        float s = 0.f;
        for (int c = lane; c < D; c += 32) { const float x = a.x[(int64_t)r * D + c] + a.r[(int64_t)r * D + c]; buf[c] = x; s += x; }
        float mean = warp_sumf(s) / D, v = 0.f;
        for (int c = lane; c < D; c += 32) { const float d = buf[c] - mean; v = fmaf(d, d, v); }
        float rstd = rsqrtf(warp_sumf(v) / D + 1e-5f);
        s = 0.f;
        for (int c = lane; c < D; c += 32) { const float y = (buf[c] - mean) * rstd * a.w_a[c] + a.b_a[c]; buf[c] = y; s += y; }
        mean = warp_sumf(s) / D; v = 0.f;
        for (int c = lane; c < D; c += 32) { const float d = buf[c] - mean; v = fmaf(d, d, v); }
        rstd = rsqrtf(warp_sumf(v) / D + 1e-5f);
        for (int c = lane; c < D; c += 32) {
            const float y = (buf[c] - mean) * rstd * a.w_b[c] + a.b_b[c];
            if (a.out16) reinterpret_cast<T*>(a.out16)[(int64_t)r * D + c] = cvt_from_float<T>(y);
            if (a.out32) a.out32[(int64_t)r * D + c] = y;
        }
    }
}

// ---------------------------------------------------------------------------------------------- final expansion
__global__ void __launch_bounds__(256) final_expand_kernel(const tscd_final_expand_args a) {
    __shared__ int scan[40];
    const int lf = blockIdx.x;
    const int b = lf / a.L, f = lf - b * a.L;
    const int fi = b * a.F + f;
    const int n = min(a.sel_count[fi], a.max_keep);
    const int l0 = a.lrow_off[lf];
    const int C = a.num_classes, W = 7 + C;
    const float* rows = a.sel_rows + (int64_t)fi * a.max_keep * W;
    const int64_t rbase = (int64_t)lf * a.max_keep * C, obase = (int64_t)lf * a.max_keep;
    const float thr = a.conf_thre;

    // ---- refined candidates: flattened (proposal, class) space, stable compaction ----
    const int total = n * C;
    const int chunk = (total + blockDim.x - 1) / blockDim.x;
    const int lo = min((int)threadIdx.x * chunk, total), hi = min(lo + chunk, total);
    int cnt = 0;
    for (int t = lo; t < hi; ++t) {
        const int p = t / C, c = t - p * C;
        const float cs = sigmoidf_ref(a.cls_logits[(int64_t)(l0 + p) * a.ld_cls + c]);
        const float ob = sigmoidf_ref(a.obj_logits[(int64_t)(l0 + p) * a.ld_obj]);
        cnt += (cs >= thr && __fmul_rn(ob, cs) >= thr) ? 1 : 0;
    }
    int tot;
    int o = block_excl_scan(cnt, scan, &tot);
    for (int t = lo; t < hi; ++t) {
        const int p = t / C, c = t - p * C;
        const float cs = sigmoidf_ref(a.cls_logits[(int64_t)(l0 + p) * a.ld_cls + c]);
        const float ob = sigmoidf_ref(a.obj_logits[(int64_t)(l0 + p) * a.ld_obj]);
        if (cs >= thr && __fmul_rn(ob, cs) >= thr) {
            // decode_reg_preds5 (tscd_head.py:914-949), deltas w.r.t. the still-detector box
            const float* r = rows + (int64_t)p * W;
            const float* d = a.reg_deltas + (int64_t)(l0 + p) * a.ld_reg;
            const float w = __fsub_rn(r[2], r[0]), h = __fsub_rn(r[3], r[1]);
            const float cx = __fadd_rn(r[0], __fmul_rn(0.5f, w)), cy = __fadd_rn(r[1], __fmul_rn(0.5f, h));
            const float dw = fminf(d[2], a.xform_clip), dh = fminf(d[3], a.xform_clip);
            const float pcx = __fadd_rn(__fmul_rn(d[0], w), cx), pcy = __fadd_rn(__fmul_rn(d[1], h), cy);
            const float pw = __fmul_rn(expf(dw), w), ph = __fmul_rn(expf(dh), h);
            float4 box = make_float4(__fsub_rn(pcx, __fmul_rn(0.5f, pw)), __fsub_rn(pcy, __fmul_rn(0.5f, ph)),
                                     __fadd_rn(pcx, __fmul_rn(0.5f, pw)), __fadd_rn(pcy, __fmul_rn(0.5f, ph)));
            reinterpret_cast<float4*>(a.r_box)[rbase + o] = box;
            a.r_score[rbase + o] = __fmul_rn(ob, cs);
            a.r_cls[rbase + o] = c;
            a.r_obj[rbase + o] = ob;
            a.r_cscore[rbase + o] = cs;
            ++o;
        }
    }
    if (threadIdx.x == 0) a.r_count[lf] = tot;

    // ---- still-detector candidates ----
    const int chunk2 = (n + blockDim.x - 1) / blockDim.x;
    const int lo2 = min((int)threadIdx.x * chunk2, n), hi2 = min(lo2 + chunk2, n);
    cnt = 0;
    for (int p = lo2; p < hi2; ++p) {
        const float* r = rows + (int64_t)p * W;
        cnt += (__fmul_rn(r[4], r[5]) >= thr) ? 1 : 0;
    }
    o = block_excl_scan(cnt, scan, &tot);
    for (int p = lo2; p < hi2; ++p) {
        const float* r = rows + (int64_t)p * W;
        if (__fmul_rn(r[4], r[5]) >= thr) {
            reinterpret_cast<float4*>(a.o_box)[obase + o] = make_float4(r[0], r[1], r[2], r[3]);
            a.o_score[obase + o] = __fmul_rn(r[4], r[5]);
            a.o_cls[obase + o] = (int)r[6];
            a.o_obj[obase + o] = r[4];
            a.o_cscore[obase + o] = r[5];
            ++o;
        }
    }
    if (threadIdx.x == 0) a.o_count[lf] = tot;
}

__global__ void final_rows_kernel(const tscd_final_rows_args a) {
    const int fr = blockIdx.x;
    const int n = min(a.keep_count[fr], a.keep_cap);
    for (int j = threadIdx.x; j < n; j += blockDim.x) {
        const int pos = a.keep[(int64_t)fr * a.keep_cap + j];
        const int64_t s = (int64_t)fr * a.cand_cap + pos;
        float* o = a.rows + ((int64_t)fr * a.keep_cap + j) * 7;
        const float4 bx = reinterpret_cast<const float4*>(a.box)[s];
        o[0] = bx.x; o[1] = bx.y; o[2] = bx.z; o[3] = bx.w;
        o[4] = a.obj[s]; o[5] = a.cscore[s]; o[6] = (float)a.cls[s];
    }
}

// Evaluator / Predictor glue (SURVEY.md section 8f-1): every detection of every frame as ONE packed table, in the units the
// reference's consumers compute per box in Python loops after a per-frame .cpu():
//   OVISEvaluator.convert_to_coco_format (yolox/evaluators/ovis_evaluator_v2.py:233-289):  bboxes /= scale; xyxy2xywh;
//   score = obj * cls_conf;   Predictor.to_repp_heavy (tools/val_to_imdb.py:193-218): output[:, :4] /= ratio, clipping to the image.
// Row (12 floats) = [frame, x1/s, y1/s, (x2/s - x1/s), (y2/s - y1/s), obj * cls, class, obj, x2/s, y2/s, cls_score, 0]
// (same operation order as the reference: divide, then subtract).
__global__ void __launch_bounds__(1024) pack_offsets_kernel(int num_frames, int cap, const int32_t* count, int32_t* offsets) {
    __shared__ int scan[40];
    int carry = 0;
    for (int f0 = 0; f0 < num_frames; f0 += blockDim.x) {
        const int f = f0 + threadIdx.x;
        const int c = f < num_frames ? min(count[f], cap) : 0;
        int tot;
        const int ex = block_excl_scan(c, scan, &tot);
        if (f < num_frames) offsets[f] = carry + ex;
        carry += tot;
    }
    if (threadIdx.x == 0) offsets[num_frames] = carry;
}

__global__ void pack_detections_kernel(const tscd_pack_detections_args a) {
    const int f = blockIdx.x;
    const int n = min(a.count[f], a.cap);
    const int o = a.offsets[f];
    const float s = a.scale ? a.scale[f] : 1.f;
    for (int j = threadIdx.x; j < n; j += blockDim.x)
        pack_detection_row(a.rows + ((int64_t)f * a.cap + j) * 7, (float)f, s, a.packed + (int64_t)(o + j) * 12);
}

// raw variant: the [n,7] rows themselves, frame after frame (forward_host's single read-back)
__global__ void pack_rows_kernel(const tscd_pack_rows_args a) {
    const int f = blockIdx.x;
    const int n = min(a.count[f], a.cap);
    const float* src = a.rows + (int64_t)f * a.cap * 7;
    float* dst = a.packed + (int64_t)a.offsets[f] * 7;
    for (int j = threadIdx.x; j < n * 7; j += blockDim.x) dst[j] = src[j];
}

}  // namespace tscd

extern "C" int tscd_pack_rows(const tscd_pack_rows_args* a, void* stream) {
    using namespace tscd;
    if (!a || a->num_frames <= 0 || a->cap <= 0 || !a->rows || !a->count || !a->offsets || !a->packed) return TSCD_ERR_INVALID_ARG;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    pack_offsets_kernel<<<1, 1024, 0, st>>>(a->num_frames, a->cap, a->count, a->offsets);
    TSCD_CUDA_CHECK_LAUNCH();
    pack_rows_kernel<<<a->num_frames, 256, 0, st>>>(*a);
    TSCD_CUDA_CHECK_LAUNCH();
    return TSCD_OK;
}

extern "C" int tscd_pack_detections(const tscd_pack_detections_args* a, void* stream) {
    using namespace tscd;
    if (!a || a->num_frames <= 0 || a->cap <= 0 || !a->rows || !a->count || !a->offsets || !a->packed) return TSCD_ERR_INVALID_ARG;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    pack_offsets_kernel<<<1, 1024, 0, st>>>(a->num_frames, a->cap, a->count, a->offsets);
    TSCD_CUDA_CHECK_LAUNCH();
    pack_detections_kernel<<<a->num_frames, 128, 0, st>>>(*a);
    TSCD_CUDA_CHECK_LAUNCH();
    return TSCD_OK;
}

extern "C" int tscd_frame_attention(const tscd_frame_attention_args* a, void* stream) {
    using namespace tscd;
    if (!a || a->num_frames <= 0 || a->heads <= 0 || a->head_dim <= 0 || a->head_dim % 32 || a->head_dim > 128) return TSCD_ERR_INVALID_ARG;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    if (a->in_dtype == TSCD_F16 || a->in_dtype == TSCD_BF16) {
        // tensor-core variant: 16-bit q/k/v, frames of <= 32 rows (caller guarantees kmax <= 32), head_dim 128
        if (a->head_dim != 128 || (a->heads % kFa16Heads) != 0 || (a->ldq % 8) || (a->ldk % 8) || (a->ldv % 8)) return TSCD_ERR_UNSUPPORTED;
        const size_t sm = (size_t)3 * kFa16Heads * 32 * kFa16Pitch * 2 + 2 * kFa16Heads * 32 * sizeof(float);
        const dim3 grid(a->num_frames, a->heads / kFa16Heads);
        if (a->in_dtype == TSCD_F16) {
            if (cudaFuncSetAttribute(frame_attention16_kernel<__half>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm) != cudaSuccess) return TSCD_ERR_CUDA;
            frame_attention16_kernel<__half><<<grid, 256, sm, st>>>(*a);
        } else {
            if (cudaFuncSetAttribute(frame_attention16_kernel<__nv_bfloat16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm) != cudaSuccess) return TSCD_ERR_CUDA;
            frame_attention16_kernel<__nv_bfloat16><<<grid, 256, sm, st>>>(*a);
        }
        TSCD_CUDA_CHECK_LAUNCH();
        return TSCD_OK;
    }
    if (a->in_dtype != TSCD_F32) return TSCD_ERR_UNSUPPORTED;
    const size_t smem = (size_t)(kFaChunk * (a->head_dim + 4) + kFaChunk * a->head_dim + 8 * a->head_dim) * sizeof(float);
    if (cudaFuncSetAttribute(frame_attention_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) return TSCD_ERR_CUDA;
    frame_attention_kernel<<<dim3(a->num_frames, a->heads), 256, smem, st>>>(*a);
    TSCD_CUDA_CHECK_LAUNCH();
    return TSCD_OK;
}

extern "C" int tscd_residual_ln2(const tscd_residual_ln2_args* a, void* stream) {
    using namespace tscd;
    if (!a || a->rows_cap <= 0 || a->dim <= 0 || a->dim > 4096 || (!a->out16 && !a->out32 && !a->head_w)) return TSCD_ERR_INVALID_ARG;
    if (a->head_w && (a->dim != 1024 || !a->head_b || !a->head_out)) return TSCD_ERR_UNSUPPORTED;
    const size_t smem = (size_t)8 * a->dim * sizeof(float);
    int grid = (a->rows_cap + 7) / 8;
    if (grid > 148 * 8) grid = 148 * 8;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    if (a->out_dtype == TSCD_BF16) {
        if (cudaFuncSetAttribute(residual_ln2_kernel<__nv_bfloat16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) return TSCD_ERR_CUDA;
        residual_ln2_kernel<__nv_bfloat16><<<grid, 256, smem, st>>>(*a);
    } else {
        if (cudaFuncSetAttribute(residual_ln2_kernel<__half>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) return TSCD_ERR_CUDA;
        residual_ln2_kernel<__half><<<grid, 256, smem, st>>>(*a);
    }
    TSCD_CUDA_CHECK_LAUNCH();
    return TSCD_OK;
}

extern "C" int tscd_final_expand(const tscd_final_expand_args* a, void* stream) {
    using namespace tscd;
    if (!a || a->B <= 0 || a->L <= 0 || a->num_classes <= 0 || a->max_keep <= 0) return TSCD_ERR_INVALID_ARG;
    final_expand_kernel<<<a->B * a->L, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(*a);
    TSCD_CUDA_CHECK_LAUNCH();
    return TSCD_OK;
}

extern "C" int tscd_final_rows(const tscd_final_rows_args* a, void* stream) {
    using namespace tscd;
    if (!a || a->num_frames <= 0) return TSCD_ERR_INVALID_ARG;
    final_rows_kernel<<<a->num_frames, 128, 0, reinterpret_cast<cudaStream_t>(stream)>>>(*a);
    TSCD_CUDA_CHECK_LAUNCH();
    return TSCD_OK;
}
