// K5: CAFM -- spatiotemporal context-aware feature matching (AwarePositionRegMatcher).
//
// Reference: yolox/models/tscd_matching.py:639-937 (forward :722-888, double_match_embds :912-937,
// ReferringCrossAttentionLayer.forward_post :566-589, SEModule :278-283, PositionMHAttention :31-60) and
// scipy.optimize.linear_sum_assignment (called at :935).
//
// The recurrence over local frames is inherently sequential (frame i's queries are frame i-1's outputs), so
// one CTA owns one clip and walks its frames; clips run in parallel on different SMs.  Everything that does
// not depend on the recurrence (value / key projections, SE gate of the key side, time embedding, norms) is
// computed up front by batched kernels (tscd_cafm_prep + tscd_linear).  Inside the chain:
//   cost      32x32 tiles of (prev, cur) pairs, 128-dim slabs of the 2x1024-dim embeddings staged in shared
//             memory, fp32:  1 - (cos_reg + cos_cls)/2  with the reference's (|x| + 1e-6) norms, NaN -> 0;
//   LSAP      shortest augmenting path in fp64 by one warp, SciPy's scan order and tie rules (among equal
//             minima prefer a column that is a new sink; `remaining` filled in reverse, swap-with-last);
//   attention 8 heads x 32, cosine (L2-normalised q,k, no scale), keys/values = the CURRENT frame only;
//   output    LayerNorm(identity + attn), scattered back to the original row order, then decoder_norm.
#include "common.cuh"
#include "mma.cuh"

namespace tscd {

constexpr int kChainThreads = 512;
constexpr int kChainMax = 512;                   // default tier: the one-warp LSAP, the generic one-CTA chain
constexpr int kWideMax = TSCD_MAX_PROPOSALS;     // wide tier: CTA LSAP, wide chain, wide cost kernel
constexpr int kCostSmem = 64 * 64;

__device__ __forceinline__ float se_gate(float a, float b, const float* w1, const float* w2) {
    float o0 = 0.f, o1 = 0.f;
#pragma unroll
    for (int j = 0; j < 32; ++j) {
        float h = fmaxf(0.f, fmaf(w1[2 * j + 1], b, w1[2 * j] * a));
        o0 = fmaf(w2[j], h, o0);
        o1 = fmaf(w2[32 + j], h, o1);
    }
    const float s0 = 1.f / (1.f + expf(-o0)), s1 = 1.f / (1.f + expf(-o1));
    return a * s0 + b * s1;
}

// Packed fp32 arithmetic (Blackwell FFMA2 / FMUL2: two IEEE round-to-nearest fp32 operations per instruction).  The SE
// gate is bound by the FMA pipe; pairing two elements per instruction halves its instruction count with bit-identical
// results (each half is an ordinary fp32 fma / mul).
__device__ __forceinline__ unsigned long long pk2(float lo, float hi) {
    unsigned long long r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void upk2(unsigned long long v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ unsigned long long fma2(unsigned long long a, unsigned long long b, unsigned long long c) {
    unsigned long long r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
    return r;
}
__device__ __forceinline__ unsigned long long mul2(unsigned long long a, unsigned long long b) {
    unsigned long long r;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}

// SE gate of 8 (a, b) pairs at once: the 32 hidden units' weights are read once per 8 elements (one LDS.128 each);
// per hidden unit and element:  h = relu(w1b * b + w1a * a);  o0 += w2[0] * h;  o1 += w2[1] * h  (same order as se_gate)
__device__ __forceinline__ void se_gate8(const float (&a)[8], const float (&b)[8], const float4* se, float (&out)[8]) {
    unsigned long long A2[4], B2[4], o0[4], o1[4];
#pragma unroll
    for (int p = 0; p < 4; ++p) { A2[p] = pk2(a[2 * p], a[2 * p + 1]); B2[p] = pk2(b[2 * p], b[2 * p + 1]); o0[p] = 0ull; o1[p] = 0ull; }
#pragma unroll 4
    for (int j = 0; j < 32; ++j) {
        const float4 w = se[j];
        const unsigned long long wx = pk2(w.x, w.x), wy = pk2(w.y, w.y), wz = pk2(w.z, w.z), ww = pk2(w.w, w.w);
#pragma unroll
        for (int p = 0; p < 4; ++p) {
            float h0, h1;
            upk2(fma2(wy, B2[p], mul2(wx, A2[p])), h0, h1);
            const unsigned long long h = pk2(fmaxf(0.f, h0), fmaxf(0.f, h1));
            o0[p] = fma2(wz, h, o0[p]);
            o1[p] = fma2(ww, h, o1[p]);
        }
    }
#pragma unroll
    for (int p = 0; p < 4; ++p) {
        float x0, x1, y0, y1;
        upk2(o0[p], x0, x1);
        upk2(o1[p], y0, y1);
        const float s00 = 1.f / (1.f + expf(-x0)), s01 = 1.f / (1.f + expf(-x1));
        const float s10 = 1.f / (1.f + expf(-y0)), s11 = 1.f / (1.f + expf(-y1));
        out[2 * p] = a[2 * p] * s00 + b[2 * p] * s10;
        out[2 * p + 1] = a[2 * p + 1] * s01 + b[2 * p + 1] * s11;
    }
}

__device__ __forceinline__ void store8(float* p, const float (&v)[8]) {
    *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
    *reinterpret_cast<float4*>(p + 4) = make_float4(v[4], v[5], v[6], v[7]);
}

// One warp per local row: lane owns 8 consecutive channels (16-byte loads / stores), the SE gate is register-blocked
// over them; then the warp reduces the two 1024-dim matching-embedding norms of the row.  grid = (local frames, ysplit).
template <typename T>
__global__ void __launch_bounds__(256) cafm_prep_kernel(const tscd_cafm_prep_args a) {
    __shared__ float4 se[32];
    if (threadIdx.x < 32) se[threadIdx.x] = make_float4(a.se_w1[2 * threadIdx.x], a.se_w1[2 * threadIdx.x + 1], a.se_w2[threadIdx.x], a.se_w2[32 + threadIdx.x]);
    __syncthreads();
    const int lf = blockIdx.x;  // local frame index b*L + f
    const int b = lf / a.L, f = lf - b * a.L;
    const int r0 = a.row_off[b * a.F + f];
    const int n = a.row_off[b * a.F + f + 1] - r0;
    const int l0 = a.lrow_off[lf];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int D = a.D, E = 4 * a.D;         // D == 256 (checked on the host)
    for (int j = warp + 8 * blockIdx.y; j < n; j += 8 * gridDim.y) {
        const T* fr = reinterpret_cast<const T*>(a.bank_reg) + (int64_t)(r0 + j) * D;
        const T* er = reinterpret_cast<const T*>(a.bank_edge) + (int64_t)(r0 + j) * D;
        const int64_t o = (int64_t)(l0 + j) * D + lane * 8;
        float x[8], e[8], k[8], tm[8];
        const uint4 xraw = __ldg(reinterpret_cast<const uint4*>(fr + lane * 8));
        load8(reinterpret_cast<const T*>(&xraw), x);
        load8(er + lane * 8, e);
        load8(a.time_emb + (int64_t)lf * D + lane * 8, tm);
        se_gate8(x, e, se, k);
#pragma unroll
        for (int i = 0; i < 8; ++i) k[i] += tm[i];
        if (a.feat) store8(a.feat + o, x);
        if (a.edge) store8(a.edge + o, e);
        if (a.kin) store8(a.kin + o, k);
        *reinterpret_cast<uint4*>(reinterpret_cast<T*>(a.feat16) + o) = xraw;
        uint4 kp;
        kp.x = pack2<T>(k[0], k[1]); kp.y = pack2<T>(k[2], k[3]); kp.z = pack2<T>(k[4], k[5]); kp.w = pack2<T>(k[6], k[7]);
        *reinterpret_cast<uint4*>(reinterpret_cast<T*>(a.kin16) + o) = kp;
        if (a.emb_dtype != TSCD_F32) continue;      // 16-bit matching embeddings: tscd_cafm_cost computes the norms itself
        float sr = 0.f, sc = 0.f;
        const float4* pr = reinterpret_cast<const float4*>(a.emb_reg + (int64_t)(l0 + j) * E);
        const float4* pc = reinterpret_cast<const float4*>(a.emb_cls + (int64_t)(l0 + j) * E);
#pragma unroll 4
        for (int c = lane; c < E / 4; c += 32) {
            const float4 u = pr[c], w = pc[c];
            sr = fmaf(u.x, u.x, fmaf(u.y, u.y, fmaf(u.z, u.z, fmaf(u.w, u.w, sr))));
            sc = fmaf(w.x, w.x, fmaf(w.y, w.y, fmaf(w.z, w.z, fmaf(w.w, w.w, sc))));
        }
        sr = warp_sumf(sr); sc = warp_sumf(sc);
        if (lane == 0) { a.norm_reg[l0 + j] = sqrtf(sr) + 1e-6f; a.norm_cls[l0 + j] = sqrtf(sc) + 1e-6f; }
    }
}

// ---------------------------------------------------------------------------------------------- matching costs, wide frames
// Frames of more than 32 proposals with 16-bit copies of the matching embeddings: one CTA (8 warps) per (local frame,
// 128 reference rows, 64 current rows).  Both 1024-dim embeddings stream through shared memory in 64-dim chunks (cp.async,
// double buffered, 144-byte rows: ldmatrix conflict-free); warp w owns reference rows [16w, 16w+16) x all 64 columns:
// 8 n-tiles of mma.sync m16n8k16 per k-step, fp32 accumulation, the two cosines kept in separate accumulators.  Norms are the
// fp32 ones of tscd_cafm_prep (or of the carried state, whose fp32 embeddings are converted while they are staged).
constexpr int kCwRows = 128, kCwCols = 64, kCwPitch = 72, kCwThreads = 256;

template <typename T>
__global__ void __launch_bounds__(kCwThreads) cafm_cost_wide16_kernel(const tscd_cafm_cost_args a) {
    extern __shared__ __align__(16) unsigned char cw_smem[];
    T* sA = reinterpret_cast<T*>(cw_smem);                        // [2][128][72]
    T* sB = sA + 2 * kCwRows * kCwPitch;                          // [2][64][72]
    const int lf = blockIdx.x, b = lf / a.L, f = lf - b * a.L;
    const int l0 = a.lrow_off[lf], n = a.lrow_off[lf + 1] - l0;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t4 = lane & 3;
    if (n <= 0) {
        if (a.ref_n && blockIdx.y == 0 && blockIdx.z == 0 && tid == 0) a.ref_n[lf] = 0;
        return;
    }
    constexpr int E = 1024;
    const int KM = a.kmax;
    // reference side: previous non-empty local frame, else the carried state (resume), else the frame itself
    const T *Rp = nullptr, *Cp = nullptr;
    const float *sR = nullptr, *sC = nullptr, *nRp = nullptr, *nCp = nullptr;
    int np = 0;
    for (int p = f - 1; p >= 0 && np == 0; --p) {
        const int pl0 = a.lrow_off[b * a.L + p], pn = a.lrow_off[b * a.L + p + 1] - pl0;
        if (pn > 0) {
            np = pn;
            Rp = reinterpret_cast<const T*>(a.emb_reg16) + (int64_t)pl0 * E; Cp = reinterpret_cast<const T*>(a.emb_cls16) + (int64_t)pl0 * E;
            nRp = a.norm_reg + pl0; nCp = a.norm_cls + pl0;
        }
    }
    if (np == 0) {
        const int sb = a.slot ? a.slot[b] : b;       // state slot of clip b
        const int sn = (a.resume && a.resume[b]) ? a.st_n[sb] : 0;
        if (sn > 0) {
            np = sn;
            sR = a.st_reg + (int64_t)sb * KM * E; sC = a.st_cls + (int64_t)sb * KM * E;
            nRp = a.st_nreg + (int64_t)sb * KM; nCp = a.st_ncls + (int64_t)sb * KM;
        } else {
            np = n;
            Rp = reinterpret_cast<const T*>(a.emb_reg16) + (int64_t)l0 * E; Cp = reinterpret_cast<const T*>(a.emb_cls16) + (int64_t)l0 * E;
            nRp = a.norm_reg + l0; nCp = a.norm_cls + l0;
        }
    }
    if (a.ref_n && blockIdx.y == 0 && blockIdx.z == 0 && tid == 0) a.ref_n[lf] = (np > KM || n > KM) ? 0 : np;
    const int rb = blockIdx.y * kCwRows, cb = blockIdx.z * kCwCols;
    if (rb >= np || cb >= n || np > KM || n > KM) return;
    const T* Rc = reinterpret_cast<const T*>(a.emb_reg16) + (int64_t)l0 * E;
    const T* Cc = reinterpret_cast<const T*>(a.emb_cls16) + (int64_t)l0 * E;

    auto stage = [&](int s, int buf) {                  // chunk s: embedding s >> 4, dims [(s & 15) * 64, +64)
        const int which = s >> 4, d0 = (s & 15) * 64;
        T* dA = sA + buf * kCwRows * kCwPitch;
        T* dB = sB + buf * kCwCols * kCwPitch;
        const T* P16 = which == 0 ? Rp : Cp;
        const float* P32 = which == 0 ? sR : sC;
        for (int i = tid; i < kCwRows * 8; i += kCwThreads) {
            const int r = i >> 3, c = (i & 7) * 8;
            T* dst = dA + r * kCwPitch + c;
            if (rb + r >= np) { *reinterpret_cast<uint4*>(dst) = make_uint4(0, 0, 0, 0); continue; }
            if (P16) {
                cp_async16(dst, P16 + (int64_t)(rb + r) * E + d0 + c);
            } else {                                    // carried fp32 state: convert while staging
                const float4 u = *reinterpret_cast<const float4*>(P32 + (int64_t)(rb + r) * E + d0 + c);
                const float4 v = *reinterpret_cast<const float4*>(P32 + (int64_t)(rb + r) * E + d0 + c + 4);
                uint4 o;
                o.x = pack2<T>(u.x, u.y); o.y = pack2<T>(u.z, u.w); o.z = pack2<T>(v.x, v.y); o.w = pack2<T>(v.z, v.w);
                *reinterpret_cast<uint4*>(dst) = o;
            }
        }
        const T* Q16 = which == 0 ? Rc : Cc;
        for (int i = tid; i < kCwCols * 8; i += kCwThreads) {
            const int r = i >> 3, c = (i & 7) * 8;
            T* dst = dB + r * kCwPitch + c;
            if (cb + r < n) cp_async16(dst, Q16 + (int64_t)(cb + r) * E + d0 + c);
            else *reinterpret_cast<uint4*>(dst) = make_uint4(0, 0, 0, 0);
        }
        cp_async_commit();
    };

    float acc[2][8][4];
#pragma unroll
    for (int w = 0; w < 2; ++w)
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) acc[w][nt][0] = acc[w][nt][1] = acc[w][nt][2] = acc[w][nt][3] = 0.f;
    stage(0, 0);
#pragma unroll 1
    for (int s = 0; s < 32; ++s) {
        const int buf = s & 1;
        cp_async_wait_all();
        __syncthreads();                                 // chunk s landed; every warp is done with the other buffer
        if (s + 1 < 32) stage(s + 1, buf ^ 1);
        const T* tA = sA + buf * kCwRows * kCwPitch;
        const T* tB = sB + buf * kCwCols * kCwPitch;
#pragma unroll
        for (int ks = 0; ks < 4; ++ks) {
            uint32_t fa[4];
            ldsm_x4(fa, tA + (warp * 16 + (lane & 15)) * kCwPitch + ks * 16 + (lane >> 4) * 8);
#pragma unroll
            for (int ntp = 0; ntp < 4; ++ntp) {
                uint32_t fb[4];
                ldsm_x4(fb, tB + (ntp * 16 + (lane & 7) + ((lane >> 4) & 1) * 8) * kCwPitch + ks * 16 + ((lane >> 3) & 1) * 8);
                if (s < 16) { mma16816<T>(acc[0][2 * ntp], fa, fb[0], fb[1]); mma16816<T>(acc[0][2 * ntp + 1], fa, fb[2], fb[3]); }
                else { mma16816<T>(acc[1][2 * ntp], fa, fb[0], fb[1]); mma16816<T>(acc[1][2 * ntp + 1], fa, fb[2], fb[3]); }
            }
        }
    }
    float* out = a.cost + (int64_t)lf * KM * KM;
#pragma unroll
    for (int hr = 0; hr < 2; ++hr) {
        const int r = rb + warp * 16 + g + hr * 8;
        if (r >= np) continue;
        const float nr = nRp[r], nc = nCp[r];
#pragma unroll
        for (int nt = 0; nt < 8; ++nt)
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const int c = cb + nt * 8 + 2 * t4 + e;
                if (c >= n) continue;
                const float cr = acc[0][nt][hr * 2 + e] / (nr * a.norm_reg[l0 + c]);
                const float cq = acc[1][nt][hr * 2 + e] / (nc * a.norm_cls[l0 + c]);
                float v = 1.f - (cr + cq) / 2.f;
                if (v != v) v = 0.f;                     // tscd_matching.py:930 NaN -> 0
                out[(int64_t)r * KM + c] = v;
            }
    }
}

constexpr int kSmall = 32;   // frames with <= kSmall proposals keep their whole working set in shared memory

struct LapSmem {
    double u[kChainMax], v[kChainMax], spc[kChainMax];
    int path[kChainMax], col4row[kChainMax], row4col[kChainMax], remaining[kChainMax];
    unsigned char SR[kChainMax], SC[kChainMax];
    float cost_s[kCostSmem];          // cost table kept on chip when n_ref * n_cur fits (the common case)
};

struct ChainSmem {
    int perm[kChainMax], prow[kChainMax], ord_prev[kChainMax];
    float w1[64], w2[64];
    float pbuf[kChainThreads / 32][kChainMax];
    float x0[kSmall * 256];           // query input, then pre-norm output
    float x1[kSmall * 256];           // q, then scratch for the decoder norm
    float xk[kSmall * 256];           // normalised keys
    float xv[kSmall * 256];           // values
};

// ---------------------------------------------------------------------------------------------- matching costs
// One CTA per (local frame, 32x32 tile): 128-dim slabs of the two 1024-dim embeddings staged in shared memory.
__global__ void __launch_bounds__(256) cafm_cost_kernel(const tscd_cafm_cost_args a) {
    __shared__ __align__(16) float tiles[2][32][132];                 // 4-float skew: float4 row reads are conflict-free
    float (*tileA)[132] = tiles[0];
    float (*tileB)[132] = tiles[1];
    const int lf = blockIdx.x, b = lf / a.L, f = lf - b * a.L;
    const int l0 = a.lrow_off[lf], n = a.lrow_off[lf + 1] - l0;
    if (n <= 0) {
        if (a.ref_n && blockIdx.y == 0 && blockIdx.z == 0 && threadIdx.x == 0) a.ref_n[lf] = 0;
        return;
    }
    const int E = 4 * a.D, KM = a.kmax;
    // reference side: previous non-empty local frame, else the carried state (resume), else the frame itself
    const float *Rp = nullptr, *Cp = nullptr, *nRp = nullptr, *nCp = nullptr;
    int np = 0;
    for (int p = f - 1; p >= 0 && np == 0; --p) {
        const int pl0 = a.lrow_off[b * a.L + p], pn = a.lrow_off[b * a.L + p + 1] - pl0;
        if (pn > 0) { np = pn; Rp = a.emb_reg + (int64_t)pl0 * E; Cp = a.emb_cls + (int64_t)pl0 * E; nRp = a.norm_reg + pl0; nCp = a.norm_cls + pl0; }
    }
    if (np == 0) {
        const int sb = a.slot ? a.slot[b] : b;       // state slot of clip b
        const int sn = (a.resume && a.resume[b]) ? a.st_n[sb] : 0;
        if (sn > 0) {
            np = sn;
            Rp = a.st_reg + (int64_t)sb * KM * E; Cp = a.st_cls + (int64_t)sb * KM * E;
            nRp = a.st_nreg + (int64_t)sb * KM; nCp = a.st_ncls + (int64_t)sb * KM;
        } else {
            np = n;
            Rp = a.emb_reg + (int64_t)l0 * E; Cp = a.emb_cls + (int64_t)l0 * E; nRp = a.norm_reg + l0; nCp = a.norm_cls + l0;
        }
    }
    if (a.ref_n && blockIdx.y == 0 && blockIdx.z == 0 && threadIdx.x == 0) a.ref_n[lf] = (np > KM || n > KM) ? 0 : np;
    const int rb = blockIdx.y * 32, cb = blockIdx.z * 32;
    if (rb >= np || cb >= n || np > KM || n > KM) return;
    const float* Rc = a.emb_reg + (int64_t)l0 * E;
    const float* Cc = a.emb_cls + (int64_t)l0 * E;
    // Register tiling: the CTA's 4 groups of 64 threads each take 32 of a slab's 128 dims and ALL 32x32 pairs; a thread
    // owns the 4x4 pairs (rows ty + 8i, columns tx + 8j), so one slab step costs 8 conflict-free 16-byte shared loads for
    // 64 FMAs (the 1-output-column mapping it replaces was shared-memory-bandwidth bound at 5 loads per 16 FMAs).
    const int grp = threadIdx.x >> 6, tg = threadIdx.x & 63, ty = tg & 7, tx = tg >> 3;
    float accR[16], accC[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) { accR[i] = 0.f; accC[i] = 0.f; }
    // slabs of 128 dims; each thread moves four float4 per matrix and slab (row = t / 32 + 8 k, 16-byte column t % 32);
    // the next slab is fetched into registers while the current one is multiplied (one barrier pair per slab)
    const int lr = threadIdx.x >> 5, lc4 = threadIdx.x & 31;
    float4 pa[4], pb[4];
    auto fetch = [&](int s) {
        const int which = s >> 3, d0 = (s & 7) * 128;
        const float* P = which == 0 ? Rp : Cp;
        const float* Q = which == 0 ? Rc : Cc;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int rr = lr + 8 * k;
            pa[k] = (rb + rr < np) ? __ldg(reinterpret_cast<const float4*>(P + (int64_t)(rb + rr) * E + d0) + lc4) : make_float4(0.f, 0.f, 0.f, 0.f);
            pb[k] = (cb + rr < n) ? __ldg(reinterpret_cast<const float4*>(Q + (int64_t)(cb + rr) * E + d0) + lc4) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
    };
    fetch(0);
    for (int s = 0; s < 16; ++s) {
        __syncthreads();
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            *reinterpret_cast<float4*>(&tileA[lr + 8 * k][lc4 * 4]) = pa[k];
            *reinterpret_cast<float4*>(&tileB[lr + 8 * k][lc4 * 4]) = pb[k];
        }
        __syncthreads();
        if (s + 1 < 16) fetch(s + 1);
        // packed fp32 FMAs (FFMA2): each accumulator pair holds the partial sums of the even / odd dims of its dot product
        unsigned long long x2[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) x2[i] = 0ull;
#pragma unroll 2
        for (int d4 = grp * 8; d4 < grp * 8 + 8; ++d4) {
            ulonglong2 p4[4], q4[4];          // a float4 viewed as two packed float pairs (x,y) (z,w)
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                p4[i] = reinterpret_cast<const ulonglong2*>(tileA[ty + 8 * i])[d4];
                q4[i] = reinterpret_cast<const ulonglong2*>(tileB[tx + 8 * i])[d4];
            }
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    x2[i * 4 + j] = fma2(p4[i].x, q4[j].x, fma2(p4[i].y, q4[j].y, x2[i * 4 + j]));
        }
#pragma unroll
        for (int i = 0; i < 16; ++i) {
            float lo, hi;
            upk2(x2[i], lo, hi);
            if (s < 8) accR[i] += lo + hi; else accC[i] += lo + hi;
        }
    }
    // reduce the four dim-groups through shared memory (the tiles are free now): red[grp][which][row][col]
    __syncthreads();
    float* red = &tiles[0][0][0];
    static_assert(sizeof(float) * 2 * 32 * 132 >= sizeof(float) * 4 * 2 * 32 * 32, "reduction scratch must fit in the two tiles");
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int r = ty + 8 * i, c = tx + 8 * j;
            red[((grp * 2 + 0) * 32 + r) * 32 + c] = accR[i * 4 + j];
            red[((grp * 2 + 1) * 32 + r) * 32 + c] = accC[i * 4 + j];
        }
    __syncthreads();
    float* out = a.cost + (int64_t)lf * KM * KM;
    for (int t = threadIdx.x; t < 32 * 32; t += 256) {
        const int rr = t >> 5, cc = t & 31;
        const int r = rb + rr, c = cb + cc;
        if (r < np && c < n) {
            float dr = 0.f, dc = 0.f;
#pragma unroll
            for (int gq = 0; gq < 4; ++gq) { dr += red[((gq * 2 + 0) * 32 + rr) * 32 + cc]; dc += red[((gq * 2 + 1) * 32 + rr) * 32 + cc]; }
            const float cr = dr / (nRp[r] * a.norm_reg[l0 + c]);
            const float cq = dc / (nCp[r] * a.norm_cls[l0 + c]);
            float v = 1.f - (cr + cq) / 2.f;
            if (v != v) v = 0.f;                    // tscd_matching.py:930 NaN -> 0
            out[(int64_t)r * KM + c] = v;
        }
    }
}

// ---------------------------------------------------------------------------------------------- matching costs, 16-bit
// Frames of at most 32 proposals with 16-bit matching embeddings (the agg_iou GEMM outputs as the tensor cores produced
// them): one CTA (4 warps) per local frame.  The two 1024-dim embeddings of the reference rows and of the current rows
// stream through shared memory in 64-dim chunks (cp.async, double buffered, rows padded to 144 bytes so ldmatrix is
// conflict-free); warp w owns embedding (w >> 1) and the 16 reference rows (w & 1): 4 n-tiles of mma.sync m16n8k16 per
// k-step, fp32 accumulation.  Every thread also accumulates the squared norm of one (matrix, row) from the same chunks, so
// the (|x| + 1e-6) norms of tscd_matching.py:914-927 come from exactly the values the dot products use and the 126 MB norm
// pass over fp32 embeddings in tscd_cafm_prep disappears.  The current frame's norms are written out for the state carry.
constexpr int kC16Pitch = 72;                 // halves per smem row: 64 + 8 pad
constexpr int kC16Chunk = 64;

template <typename T>
__global__ void __launch_bounds__(128) cafm_cost16_kernel(const tscd_cafm_cost_args a) {
    __shared__ __align__(16) T tile[2][4][32][kC16Pitch];     // [stage][ref_reg, cur_reg, ref_cls, cur_cls][row][k]
    __shared__ float nrm[4][32];
    __shared__ float cosv[2][32][33];
    const int lf = blockIdx.x, b = lf / a.L, f = lf - b * a.L;
    const int l0 = a.lrow_off[lf], n = a.lrow_off[lf + 1] - l0;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (n <= 0) {
        if (tid == 0) a.ref_n[lf] = 0;
        return;
    }
    constexpr int E = 1024;
    const int KM = a.kmax;
    // reference side: previous non-empty local frame, else the carried state (resume), else the frame itself
    const T *Rp = nullptr, *Cp = nullptr;
    const float *sR = nullptr, *sC = nullptr;
    int np = 0;
    for (int p = f - 1; p >= 0 && np == 0; --p) {
        const int pl0 = a.lrow_off[b * a.L + p], pn = a.lrow_off[b * a.L + p + 1] - pl0;
        if (pn > 0) { np = pn; Rp = reinterpret_cast<const T*>(a.emb_reg) + (int64_t)pl0 * E; Cp = reinterpret_cast<const T*>(a.emb_cls) + (int64_t)pl0 * E; }
    }
    if (np == 0) {
        const int sb = a.slot ? a.slot[b] : b;       // state slot of clip b
        const int sn = (a.resume && a.resume[b]) ? a.st_n[sb] : 0;
        if (sn > 0) { np = sn; sR = a.st_reg + (int64_t)sb * KM * E; sC = a.st_cls + (int64_t)sb * KM * E; }
        else { np = n; Rp = reinterpret_cast<const T*>(a.emb_reg) + (int64_t)l0 * E; Cp = reinterpret_cast<const T*>(a.emb_cls) + (int64_t)l0 * E; }
    }
    if (np > KM || n > KM || np > 32 || n > 32) {          // the chain kernel reports the capacity error
        if (tid == 0) a.ref_n[lf] = 0;
        return;
    }
    if (tid == 0) a.ref_n[lf] = np;
    const T* Rc = reinterpret_cast<const T*>(a.emb_reg) + (int64_t)l0 * E;
    const T* Cc = reinterpret_cast<const T*>(a.emb_cls) + (int64_t)l0 * E;
    // zero the rows no load will touch (both stages)
    for (int i = tid; i < 2 * 4 * 32 * (kC16Pitch / 8); i += 128) {
        const int st = i / (4 * 32 * (kC16Pitch / 8)), rem = i % (4 * 32 * (kC16Pitch / 8));
        const int m = rem / (32 * (kC16Pitch / 8)), r = (rem / (kC16Pitch / 8)) % 32;
        if (r >= ((m & 1) ? n : np)) reinterpret_cast<uint4*>(&tile[st][m][r][0])[rem % (kC16Pitch / 8)] = make_uint4(0u, 0u, 0u, 0u);
    }
    auto load_chunk = [&](int st, int kc) {
        // 4 matrices x 32 rows x 8 16-byte pieces = 1024 pieces, 8 per thread
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const int i = u * 128 + tid;
            const int m = i >> 8, r = (i >> 3) & 31, pc = i & 7;
            const int rows = (m & 1) ? n : np;
            if (r >= rows) continue;
            T* dst = &tile[st][m][r][pc * 8];
            if (m & 1) {
                cp_async16(dst, (m == 1 ? Rc : Cc) + (int64_t)r * E + kc * kC16Chunk + pc * 8);
            } else if (Rp) {
                cp_async16(dst, (m == 0 ? Rp : Cp) + (int64_t)r * E + kc * kC16Chunk + pc * 8);
            } else {                                        // carried state: fp32 copies of 16-bit values
                const float* src = (m == 0 ? sR : sC) + (int64_t)r * E + kc * kC16Chunk + pc * 8;
                const float4 x = __ldg(reinterpret_cast<const float4*>(src)), y = __ldg(reinterpret_cast<const float4*>(src) + 1);
                uint4 pk;
                pk.x = pack2<T>(x.x, x.y); pk.y = pack2<T>(x.z, x.w); pk.z = pack2<T>(y.x, y.y); pk.w = pack2<T>(y.z, y.w);
                *reinterpret_cast<uint4*>(dst) = pk;
            }
        }
        cp_async_commit();
    };
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
    float sq = 0.f;                                         // squared norm of (matrix tid >> 5, row tid & 31)
    const int e = warp >> 1, mt = warp & 1;
    __syncthreads();
    load_chunk(0, 0);
    constexpr int NCH = E / kC16Chunk;
    for (int kc = 0; kc < NCH; ++kc) {
        const int st = kc & 1;
        if (kc + 1 < NCH) load_chunk(st ^ 1, kc + 1);
        if (kc + 1 < NCH) asm volatile("cp.async.wait_group 1;\n" ::: "memory"); else cp_async_wait_all();
        __syncthreads();
        {   // norms
            const uint4* row = reinterpret_cast<const uint4*>(&tile[st][warp][lane][0]);
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                const uint4 raw = row[q];
                const T* h = reinterpret_cast<const T*>(&raw);
#pragma unroll
                for (int t = 0; t < 8; ++t) { const float x = ldf_reg(h[t]); sq = fmaf(x, x, sq); }
            }
        }
#pragma unroll
        for (int ks = 0; ks < kC16Chunk / 16; ++ks) {
            uint32_t af[4], bf0[4], bf1[4];
            // A: reference rows mt*16 .. +16, k ks*16 .. +16  (row-major): matrices (r0-7,k0-7) (r8-15,k0-7) (r0-7,k8-15) (r8-15,k8-15)
            ldsm_x4(af, &tile[st][2 * e][mt * 16 + (lane & 15)][ks * 16 + (lane >> 4) * 8]);
            // B: current rows as [n][k]: x4 = (n0-7,k0-7) (n0-7,k8-15) (n8-15,k0-7) (n8-15,k8-15)
            ldsm_x4(bf0, &tile[st][2 * e + 1][(lane & 7) + ((lane >> 4) << 3)][ks * 16 + ((lane >> 3) & 1) * 8]);
            ldsm_x4(bf1, &tile[st][2 * e + 1][16 + (lane & 7) + ((lane >> 4) << 3)][ks * 16 + ((lane >> 3) & 1) * 8]);
            mma16816<T>(acc[0], af, bf0[0], bf0[1]);
            mma16816<T>(acc[1], af, bf0[2], bf0[3]);
            mma16816<T>(acc[2], af, bf1[0], bf1[1]);
            mma16816<T>(acc[3], af, bf1[2], bf1[3]);
        }
        __syncthreads();
    }
    nrm[warp][lane] = sqrtf(sq) + 1e-6f;
    __syncthreads();
    // cos = dot / (|ref| |cur|); fragment layout of m16n8: rows lane/4 (+8), cols 2*(lane%4) (+1)
#pragma unroll
    for (int nt = 0; nt < 4; ++nt)
#pragma unroll
        for (int h = 0; h < 4; ++h) {
            const int r = mt * 16 + (lane >> 2) + ((h >> 1) << 3), c = nt * 8 + 2 * (lane & 3) + (h & 1);
            cosv[e][r][c] = acc[nt][h] / (nrm[2 * e][r] * nrm[2 * e + 1][c]);
        }
    __syncthreads();
    float* out = a.cost + (int64_t)lf * KM * KM;
    for (int t = tid; t < 32 * 32; t += 128) {
        const int r = t >> 5, c = t & 31;
        if (r < np && c < n) {
            float v = 1.f - (cosv[0][r][c] + cosv[1][r][c]) / 2.f;
            if (v != v) v = 0.f;                            // tscd_matching.py:930 NaN -> 0
            out[(int64_t)r * KM + c] = v;
        }
    }
    if (tid < n) { const_cast<float*>(a.norm_reg)[l0 + tid] = nrm[1][tid]; const_cast<float*>(a.norm_cls)[l0 + tid] = nrm[3][tid]; }
}

// Rectangular LSAP by warp 0.  C is the [n_prev x n_cur] cost (row-major, fp32).  Solves the problem with
// rows = the smaller side exactly like scipy (transposing when n_cur < n_prev).  Results in s.col4row / s.row4col.
__device__ void lap_warp(const float* C, int ldc, int n_prev, int n_cur, LapSmem& s, int lane) {
    const bool tr = n_cur < n_prev;
    const int nr = tr ? n_cur : n_prev, nc = tr ? n_prev : n_cur;
    for (int j = lane; j < nc; j += 32) { s.v[j] = 0.0; s.row4col[j] = -1; s.path[j] = -1; }
    for (int i = lane; i < nr; i += 32) { s.u[i] = 0.0; s.col4row[i] = -1; }
    __syncwarp();
    for (int cur = 0; cur < nr; ++cur) {
        for (int it = lane; it < nc; it += 32) { s.remaining[it] = nc - it - 1; s.spc[it] = INFINITY; s.SC[it] = 0; }
        for (int i = lane; i < nr; i += 32) s.SR[i] = 0;
        __syncwarp();
        double min_val = 0.0;
        int i = cur, num_rem = nc, sink = -1;
        while (sink == -1) {
            if (lane == 0) s.SR[i] = 1;
            const double ui = s.u[i];
            // candidate key: (value, tb) ascending; tb encodes SciPy's tie rule -- among equal minima a column that is a
            // new sink wins and the LAST such sink in scan order is taken, otherwise the FIRST minimum
            double best = INFINITY;
            unsigned best_tb = 0xffffffffu;
            for (int it = lane; it < num_rem; it += 32) {
                const int j = s.remaining[it];
                const double c = (double)(tr ? C[(int64_t)j * ldc + i] : C[(int64_t)i * ldc + j]);
                const double r = min_val + c - ui - s.v[j];
                if (r < s.spc[j]) { s.path[j] = i; s.spc[j] = r; }
                const double sj = s.spc[j];
                const unsigned tb = (s.row4col[j] == -1) ? (unsigned)(kChainMax - 1 - it) : (0x10000u | (unsigned)it);
                if (sj < best || (sj == best && tb < best_tb)) { best = sj; best_tb = tb; }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const double ob = __shfl_xor_sync(0xffffffffu, best, o);
                const unsigned otb = __shfl_xor_sync(0xffffffffu, best_tb, o);
                if (ob < best || (ob == best && otb < best_tb)) { best = ob; best_tb = otb; }
            }
            const int best_it = (best_tb == 0xffffffffu) ? -1 : ((best_tb & 0x10000u) ? (int)(best_tb & 0xffffu) : kChainMax - 1 - (int)best_tb);
            min_val = best;
            if (best_it < 0 || best == INFINITY) { sink = -2; break; }   // infeasible (cannot happen: finite costs)
            const int j = s.remaining[best_it];
            if (s.row4col[j] == -1) sink = j; else i = s.row4col[j];
            __syncwarp();
            if (lane == 0) { s.SC[j] = 1; s.remaining[best_it] = s.remaining[num_rem - 1]; }
            --num_rem;
            __syncwarp();
        }
        if (sink < 0) break;
        if (lane == 0) s.u[cur] += min_val;
        for (int r = lane; r < nr; r += 32)
            if (s.SR[r] && r != cur) s.u[r] += min_val - s.spc[s.col4row[r]];
        for (int j = lane; j < nc; j += 32)
            if (s.SC[j]) s.v[j] -= min_val - s.spc[j];
        __syncwarp();
        if (lane == 0) {
            int j = sink;
            for (;;) {
                const int r = s.path[j];
                s.row4col[j] = r;
                const int t = s.col4row[r];
                s.col4row[r] = j;
                j = t;
                if (r == cur) break;
            }
        }
        __syncwarp();
    }
}

// Same algorithm for problems with at most 32 rows and columns, with the whole solver state in REGISTERS: lane j owns
// column j (v, shortest-path cost, predecessor, matched row, its position in SciPy's `remaining` list) and lane i owns
// row i (u, matched column).  A Dijkstra step is one shared-memory load (the cost), a double-precision warp minimum and
// one hardware integer reduction for the tie rule -- no shared-memory round trips, no __syncwarp.  Scan order and tie
// rules are those of lap_warp / SciPy: among equal minima an unassigned column wins, the LAST such column in scan order,
// otherwise the FIRST minimum; a removed column is replaced by the last one of the list.
__device__ void lap_warp_fast(const float* C, int ldc, int n_prev, int n_cur, int lane, int* col4row_out, int* row4col_out) {
    const bool tr = n_cur < n_prev;
    const int nr = tr ? n_cur : n_prev, nc = tr ? n_prev : n_cur;
    double v = 0.0, u = 0.0;
    int row4col = -1, col4row = -1, path = -1;
    for (int cur = 0; cur < nr; ++cur) {
        double spc = INFINITY;
        int pos = lane < nc ? nc - 1 - lane : -1;      // remaining[it] = nc - it - 1
        bool SC = false, SR = false;
        double min_val = 0.0;
        int i = cur, num_rem = nc, sink = -1;
        while (sink == -1) {
            if (lane == i) SR = true;
            const double ui = __shfl_sync(0xffffffffu, u, i);
            if (pos >= 0) {
                const double c = (double)(tr ? C[(int64_t)lane * ldc + i] : C[(int64_t)i * ldc + lane]);
                const double r = min_val + c - ui - v;
                if (r < spc) { path = i; spc = r; }
            }
            const double sj = pos >= 0 ? spc : INFINITY;
            double m = sj;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) m = fmin(m, __shfl_xor_sync(0xffffffffu, m, o));
            if (m == INFINITY) { sink = -2; break; }           // infeasible (cannot happen: finite costs)
            const unsigned tb = (pos >= 0 && sj == m) ? (row4col == -1 ? (unsigned)(kChainMax - 1 - pos) : (0x10000u | (unsigned)pos)) : 0xffffffffu;
            const unsigned best_tb = __reduce_min_sync(0xffffffffu, tb);
            const int jwin = __ffs(__ballot_sync(0xffffffffu, tb == best_tb)) - 1;
            min_val = m;
            const int rw = __shfl_sync(0xffffffffu, row4col, jwin);
            if (rw == -1) sink = jwin; else i = rw;
            // remove jwin from the list: the last element takes its place
            const int pwin = __shfl_sync(0xffffffffu, pos, jwin);
            if (pos == num_rem - 1) pos = pwin;
            if (lane == jwin) { SC = true; pos = -1; }
            --num_rem;
        }
        if (sink < 0) break;
        // dual updates
        {
            const double spc_of_match = __shfl_sync(0xffffffffu, spc, col4row < 0 ? 0 : col4row);
            if (lane == cur) u += min_val;
            else if (SR) u += min_val - spc_of_match;
            if (SC) v -= min_val - spc;
        }
        // augment along the alternating path back to `cur`
        int j = sink;
        for (;;) {
            const int r = __shfl_sync(0xffffffffu, path, j);
            if (lane == j) row4col = r;
            const int t = __shfl_sync(0xffffffffu, col4row, r);
            if (lane == r) col4row = j;
            j = t;
            if (r == cur) break;
        }
    }
    *col4row_out = col4row;
    *row4col_out = row4col;
}

__global__ void __launch_bounds__(32) cafm_lap_kernel(const tscd_cafm_lap_args a) {
    extern __shared__ __align__(16) unsigned char lap_smem[];
    LapSmem& s = *reinterpret_cast<LapSmem*>(lap_smem);
    const int lf = blockIdx.x, lane = threadIdx.x;
    const int n = a.lrow_off[lf + 1] - a.lrow_off[lf];
    const int np = a.ref_n[lf];
    if (n <= 0 || np <= 0 || max(n, np) > kChainMax) return;      // wide problems: cafm_lap_cta_kernel
    const int KM = a.kmax;
    const float* C = a.cost + (int64_t)lf * KM * KM;
    int ldc = KM;
    if (np * n <= kCostSmem) {                       // stage the table on chip: every Dijkstra step reads one row / column
        for (int t = lane; t < np * n; t += 32) { const int r = t / n, c = t - r * n; s.cost_s[t] = C[(int64_t)r * KM + c]; }
        __syncwarp();
        C = s.cost_s;
        ldc = n;
    }
    const bool tr = n < np;       // the solvers work with rows = the smaller side
    int32_t* col = a.lap_col + (int64_t)lf * KM;
    int32_t* row = a.lap_row + (int64_t)lf * KM;
    if (np <= 32 && n <= 32) {
        int c4r, r4c;
        lap_warp_fast(C, ldc, np, n, lane, &c4r, &r4c);
        // lane r holds col4row[r] of solver row r, lane c holds row4col[c] of solver column c
        if (!tr) {
            if (lane < np) col[lane] = c4r;
            if (lane < n) row[lane] = r4c;
        } else {                  // transposed problem: its rows are the current columns
            if (lane < np) col[lane] = r4c;
            if (lane < n) row[lane] = c4r;
        }
        return;
    }
    lap_warp(C, ldc, np, n, s, lane);
    __syncwarp();
    if (!tr) {
        for (int r = lane; r < np; r += 32) col[r] = s.col4row[r];
        for (int c = lane; c < n; c += 32) row[c] = s.row4col[c];
    } else {                      // transposed problem: its rows are the current columns
        for (int r = lane; r < np; r += 32) col[r] = s.row4col[r];
        for (int c = lane; c < n; c += 32) row[c] = s.col4row[c];
    }
}

// Wide problems (max(n_prev, n) > kChainMax, up to kWideMax): the same shortest-augmenting-path algorithm with the whole
// CTA on every Dijkstra step.  The column scan is spread over the block; the arg-min is a warp reduction of (value, tie key)
// followed by warp 0 over the per-warp winners, which also removes the winner from `remaining` (swap with the last entry)
// before the second barrier of the step.  Tie keys are those of lap_warp (an unassigned column wins, the LAST one in scan
// order; otherwise the FIRST minimum), so the result is SciPy's assignment, not only its cost.  State in shared memory,
// sized by kmax: fp64 potentials u / v and path costs, path / col4row / row4col / remaining, SR / SC flags (86 KB at 2048).
constexpr int kLapCtaThreads = 512;

__global__ void __launch_bounds__(kLapCtaThreads, 1) cafm_lap_cta_kernel(const tscd_cafm_lap_args a) {
    extern __shared__ __align__(16) unsigned char lap_smem[];
    constexpr int NW = kLapCtaThreads / 32;
    __shared__ double red_v[NW];
    __shared__ unsigned red_tb[NW];
    __shared__ double bc_min;
    __shared__ int bc_j, bc_r4c;
    const int lf = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int n = a.lrow_off[lf + 1] - a.lrow_off[lf];
    const int np = a.ref_n[lf];
    if (n <= 0 || np <= 0 || max(n, np) <= kChainMax) return;     // default-tier problems: cafm_lap_kernel
    const int KM = a.kmax;
    double* u = reinterpret_cast<double*>(lap_smem);
    double* v = u + KM;
    double* spc = v + KM;
    int* path = reinterpret_cast<int*>(spc + KM);
    int* col4row = path + KM;
    int* row4col = col4row + KM;
    int* remaining = row4col + KM;
    unsigned char* SR = reinterpret_cast<unsigned char*>(remaining + KM);
    unsigned char* SC = SR + KM;
    const float* C = a.cost + (int64_t)lf * KM * KM;
    const bool tr = n < np;
    const int nr = tr ? n : np, nc = tr ? np : n;
    for (int j = tid; j < nc; j += kLapCtaThreads) { v[j] = 0.0; row4col[j] = -1; path[j] = -1; }
    for (int i = tid; i < nr; i += kLapCtaThreads) { u[i] = 0.0; col4row[i] = -1; }
    __syncthreads();
    for (int cur = 0; cur < nr; ++cur) {
        for (int it = tid; it < nc; it += kLapCtaThreads) { remaining[it] = nc - it - 1; spc[it] = INFINITY; SC[it] = 0; }
        for (int i = tid; i < nr; i += kLapCtaThreads) SR[i] = (i == cur) ? 1 : 0;
        __syncthreads();
        double min_val = 0.0;
        int i = cur, num_rem = nc, sink = -1;
        while (sink == -1) {
            const double ui = u[i];
            double best = INFINITY;
            unsigned best_tb = 0xffffffffu;
            for (int it = tid; it < num_rem; it += kLapCtaThreads) {
                const int j = remaining[it];
                const double c = (double)(tr ? C[(int64_t)j * KM + i] : C[(int64_t)i * KM + j]);
                const double r = min_val + c - ui - v[j];
                if (r < spc[j]) { path[j] = i; spc[j] = r; }
                const double sj = spc[j];
                const unsigned tb = (row4col[j] == -1) ? (unsigned)(0xffff - it) : (0x10000u | (unsigned)it);
                if (sj < best || (sj == best && tb < best_tb)) { best = sj; best_tb = tb; }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const double ob = __shfl_xor_sync(0xffffffffu, best, o);
                const unsigned otb = __shfl_xor_sync(0xffffffffu, best_tb, o);
                if (ob < best || (ob == best && otb < best_tb)) { best = ob; best_tb = otb; }
            }
            if (lane == 0) { red_v[warp] = best; red_tb[warp] = best_tb; }
            __syncthreads();
            if (warp == 0) {
                best = lane < NW ? red_v[lane] : INFINITY;
                best_tb = lane < NW ? red_tb[lane] : 0xffffffffu;
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    const double ob = __shfl_xor_sync(0xffffffffu, best, o);
                    const unsigned otb = __shfl_xor_sync(0xffffffffu, best_tb, o);
                    if (ob < best || (ob == best && otb < best_tb)) { best = ob; best_tb = otb; }
                }
                if (lane == 0) {
                    const int best_it = (best_tb == 0xffffffffu) ? -1 : ((best_tb & 0x10000u) ? (int)(best_tb & 0xffffu) : 0xffff - (int)best_tb);
                    bc_min = best;
                    if (best_it < 0 || best == INFINITY) {
                        bc_j = -1;
                    } else {
                        const int j = remaining[best_it];
                        bc_j = j;
                        bc_r4c = row4col[j];
                        SC[j] = 1;
                        remaining[best_it] = remaining[num_rem - 1];
                        if (row4col[j] != -1) SR[row4col[j]] = 1;
                    }
                }
            }
            __syncthreads();
            min_val = bc_min;
            const int j = bc_j;
            if (j < 0 || min_val == INFINITY) { sink = -2; break; }     // infeasible (cannot happen: finite costs)
            if (bc_r4c == -1) sink = j; else i = bc_r4c;
            --num_rem;
        }
        if (sink < 0) break;
        for (int r = tid; r < nr; r += kLapCtaThreads)
            if (r == cur) u[r] += min_val;
            else if (SR[r]) u[r] += min_val - spc[col4row[r]];
        for (int j = tid; j < nc; j += kLapCtaThreads)
            if (SC[j]) v[j] -= min_val - spc[j];
        __syncthreads();
        if (tid == 0) {
            int j = sink;
            for (;;) {
                const int r = path[j];
                row4col[j] = r;
                const int t = col4row[r];
                col4row[r] = j;
                j = t;
                if (r == cur) break;
            }
        }
        __syncthreads();
    }
    int32_t* col = a.lap_col + (int64_t)lf * KM;
    int32_t* row = a.lap_row + (int64_t)lf * KM;
    if (!tr) {
        for (int r = tid; r < np; r += kLapCtaThreads) col[r] = col4row[r];
        for (int c = tid; c < n; c += kLapCtaThreads) row[c] = row4col[c];
    } else {                      // transposed problem: its rows are the current columns
        for (int r = tid; r < np; r += kLapCtaThreads) col[r] = row4col[r];
        for (int c = tid; c < n; c += kLapCtaThreads) row[c] = col4row[c];
    }
}

// Frames of <= 32 proposals (kmax <= 32): 32 problems per CTA, one warp each, 4 KB of staged costs per warp.  A matching is a
// latency-bound serial algorithm; as 1-warp CTAs with the general 37 KB scratch the B*L problems took two waves spread thinly
// over every SM -- packed 32 to a CTA they run in ONE wave on a quarter of the SMs, and the rest of the GPU stays free for the
// classification branch's tensor-core kernels on the side stream.
constexpr int kLapPack = 32;
__global__ void __launch_bounds__(kLapPack * 32) cafm_lap_small_kernel(const tscd_cafm_lap_args a) {
    extern __shared__ __align__(16) unsigned char lap_smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int lf = blockIdx.x * kLapPack + warp;
    if (lf >= a.num_frames) return;
    const int n = a.lrow_off[lf + 1] - a.lrow_off[lf];
    const int np = a.ref_n[lf];
    if (n <= 0 || np <= 0) return;
    const int KM = a.kmax;                           // <= 32
    const float* C = a.cost + (int64_t)lf * KM * KM;
    float* cost_s = reinterpret_cast<float*>(lap_smem) + warp * 1024;
    for (int t = lane; t < np * n; t += 32) { const int r = t / n, c = t - r * n; cost_s[t] = C[(int64_t)r * KM + c]; }
    __syncwarp();
    const bool tr = n < np;
    int32_t* col = a.lap_col + (int64_t)lf * KM;
    int32_t* row = a.lap_row + (int64_t)lf * KM;
    int c4r, r4c;
    lap_warp_fast(cost_s, n, np, n, lane, &c4r, &r4c);
    if (!tr) {
        if (lane < np) col[lane] = c4r;
        if (lane < n) row[lane] = r4c;
    } else {
        if (lane < np) col[lane] = r4c;
        if (lane < n) row[lane] = c4r;
    }
}

__device__ __forceinline__ void layer_norm_row(const float* x, const float* w, const float* b, float* y, int D, int lane) {
    float s = 0.f;
    for (int c = lane; c < D; c += 32) s += x[c];
    const float mean = warp_sumf(s) / D;
    float v = 0.f;
    for (int c = lane; c < D; c += 32) { const float d = x[c] - mean; v = fmaf(d, d, v); }
    const float rstd = rsqrtf(warp_sumf(v) / D + 1e-5f);
    for (int c = lane; c < D; c += 32) y[c] = (x[c] - mean) * rstd * w[c] + b[c];
}

// per-phase cycle counters of block 0 (debug aid, read with tscd_debug_chain_clocks)
__device__ long long g_chain_clk[8];
#define CHAIN_TICK(i)                                                                     \
    do {                                                                                  \
        if (blockIdx.x == 0 && threadIdx.x == 0) { const long long now__ = clock64(); g_chain_clk[i] += now__ - tick__; tick__ = now__; } \
    } while (0)

template <typename T>
__global__ void __launch_bounds__(kChainThreads, 1) cafm_chain_kernel(const tscd_cafm_chain_args a) {
    extern __shared__ __align__(16) unsigned char chain_smem[];
    ChainSmem& s = *reinterpret_cast<ChainSmem*>(chain_smem);
    const int b = blockIdx.x;
    const int sb = a.slot ? a.slot[b] : b;   // state slot of clip b (scratch, bank and resume stay indexed by b)
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int D = a.D, E = 4 * a.D, KM = a.kmax;
    constexpr int NW = kChainThreads / 32;
    if (tid < 64) { s.w1[tid] = a.se_w1[tid]; s.w2[tid] = a.se_w2[tid]; }

    float* st_out = a.st_out + (int64_t)sb * KM * D;
    float* st_edge = a.st_edge + (int64_t)sb * KM * D;
    float* st_time = a.st_time + (int64_t)sb * D;
    float* g_qin = a.sc_qin + (int64_t)b * KM * D;
    float* g_q = a.sc_q + (int64_t)b * KM * D;
    float* g_k = a.sc_k + (int64_t)b * KM * D;

    const bool resume = a.resume ? (a.resume[b] != 0) : false;
    int n_prev = resume ? a.st_n[sb] : 0;   // 0 = no memory
    for (int r = tid; r < kChainMax; r += kChainThreads) s.ord_prev[r] = r;   // carried state is already in matched order
    int last_l0 = -1;
    __syncthreads();
    long long tick__ = clock64();

    for (int f = 0; f < a.L; ++f) {
        const int lf = b * a.L + f;
        const int l0 = a.lrow_off[lf];
        const int n = a.lrow_off[lf + 1] - l0;
        if (n == 0) {
            if (f == 0 && !resume) n_prev = 0;      // tscd_matching.py:762-771
            continue;
        }
        if (n > KM || n > kChainMax || n_prev > KM) {
            if (tid == 0) atomicMin(a.status, TSCD_ERR_CAPACITY);
            continue;
        }
        const bool first = (f == 0 && !resume) || n_prev == 0;
        const int np = first ? n : n_prev;           // rows on the reference side of the matching (== ref_n[lf])
        const bool small = n <= kSmall;
        float* qin = small ? s.x0 : g_qin;
        float* qv = small ? s.x1 : g_q;
        float* kh = small ? s.xk : g_k;
        const float* featc = a.feat + (int64_t)l0 * D;
        const float* edgec = a.edge + (int64_t)l0 * D;
        const float* kinc = a.kin + (int64_t)l0 * D;
        const float* kp = a.kproj + (int64_t)l0 * D;
        const float* vg = a.vproj + (int64_t)l0 * D;
        const float* vp = small ? s.xv : vg;

        // ---- assignment: re-index the frame's (order-independent) LSAP solution by how the reference frame
        //      remembers its rows (tscd_matching.py:813-844) ---------------------------------------------
        if (small) for (int t = tid; t < n * D; t += kChainThreads) s.xv[t] = vg[t];
        if (tid == 0) {
            const int32_t* colo = a.lap_col + (int64_t)lf * KM;
            const int32_t* rowo = a.lap_row + (int64_t)lf * KM;
            if (np <= n) {
                for (int r = 0; r < np; ++r) { s.perm[r] = colo[first ? r : s.ord_prev[r]]; s.prow[r] = r; }
                int t = np;
                for (int c = 0; c < n && t < n; ++c)
                    if (rowo[c] == -1) { s.perm[t] = c; s.prow[t] = -1 - c; ++t; }
            } else {
                int t = 0;
                for (int r = 0; r < np && t < n; ++r) {
                    const int c = colo[s.ord_prev[r]];
                    if (c >= 0) { s.perm[t] = c; s.prow[t] = r; ++t; }
                }
            }
        }
        __syncthreads();
        CHAIN_TICK(0);
        // ---- query input ----------------------------------------------------------------------------
        for (int t = tid; t < n * D; t += kChainThreads) {
            const int r = t / D, c = t - r * D;
            float v;
            if (first) {
                v = kinc[(int64_t)r * D + c];                  // SE(feat, edge) + time of this frame
            } else {
                const int p = s.prow[r];
                const float tg = p >= 0 ? st_out[(int64_t)p * D + c] : featc[(int64_t)(-1 - p) * D + c];
                const float ed = p >= 0 ? st_edge[(int64_t)p * D + c] : edgec[(int64_t)(-1 - p) * D + c];
                v = se_gate(tg, ed, s.w1, s.w2) + st_time[c];
            }
            qin[t] = v;
        }
        __syncthreads();
        CHAIN_TICK(1);
        // ---- q = W_q qin  (thread = output channel; each half of the CTA owns every other block of 16 rows,
        //      so W_q^T is streamed from L2 once per 16 rows with coalesced loads) ------------------------
        {
            const int c = tid % D, g = tid / D, ng = kChainThreads / D;
            for (int r0 = g * 16; r0 < n; r0 += ng * 16) {
                float acc[16];
#pragma unroll
                for (int i = 0; i < 16; ++i) acc[i] = 0.f;
#pragma unroll 4
                for (int k = 0; k < D; ++k) {
                    const float w = __ldg(a.wq_t + (int64_t)k * D + c);
#pragma unroll
                    for (int i = 0; i < 16; ++i) acc[i] = fmaf(qin[(int64_t)min(r0 + i, n - 1) * D + k], w, acc[i]);
                }
#pragma unroll
                for (int i = 0; i < 16; ++i)
                    if (r0 + i < n) qv[(int64_t)(r0 + i) * D + c] = acc[i];
            }
        }
        __syncthreads();
        CHAIN_TICK(2);
        // ---- per-head L2 normalisation of q and k (8 heads x 32) --------------------------------------
        for (int t = warp; t < n * 8 * 2; t += NW) {
            const int which = t & 1, rh = t >> 1, r = rh >> 3, h = rh & 7;
            const float x = which == 0 ? qv[(int64_t)r * D + h * 32 + lane] : kp[(int64_t)r * D + h * 32 + lane];
            const float nn = sqrtf(warp_sumf(x * x));
            if (which == 0) qv[(int64_t)r * D + h * 32 + lane] = x / nn; else kh[(int64_t)r * D + h * 32 + lane] = x / nn;
        }
        __syncthreads();
        CHAIN_TICK(3);
        // ---- attention over the current frame; qin is reused as the pre-norm output buffer [n, D] ----
        for (int t = warp; t < n * 8; t += NW) {
            const int r = t >> 3, h = t & 7;
            const float* qs = qv + (int64_t)r * D + h * 32;
            float* p = s.pbuf[warp];
            float mx = -INFINITY;
            for (int j = lane; j < n; j += 32) {
                const float* kr = kh + (int64_t)j * D + h * 32;
                float sc = 0.f;
#pragma unroll
                for (int d = 0; d < 32; ++d) {       // rotated index: lanes hit distinct banks when q / k live in shared memory
                    const int dd = (d + lane) & 31;
                    sc = fmaf(qs[dd], kr[dd], sc);
                }
                p[j] = sc;
                mx = fmaxf(mx, sc);
            }
            mx = warp_maxf(mx);
            __syncwarp();
            float sum = 0.f;
            for (int j = lane; j < n; j += 32) { const float e = expf(p[j] - mx); p[j] = e; sum += e; }
            sum = warp_sumf(sum);
            __syncwarp();
            float acc = 0.f;
            for (int j = 0; j < n; ++j) acc = fmaf(p[j], vp[(int64_t)j * D + h * 32 + lane], acc);
            const int idr = first ? r : s.perm[r];
            qin[(int64_t)r * D + h * 32 + lane] = featc[(int64_t)idr * D + h * 32 + lane] + acc / sum;
            __syncwarp();
        }
        __syncthreads();
        CHAIN_TICK(4);
        // ---- norms, state update, scatter to the original order --------------------------------------
        for (int r = warp; r < n; r += NW) {
            layer_norm_row(qin + (int64_t)r * D, a.ln_w, a.ln_b, st_out + (int64_t)r * D, D, lane);   // new last_outputs
            __syncwarp();
            const int dst = l0 + s.perm[r];
            float* tmp = qv + (int64_t)r * D;    // q no longer needed
            layer_norm_row(st_out + (int64_t)r * D, a.dec_w, a.dec_b, tmp, D, lane);
            __syncwarp();
            for (int c = lane; c < D; c += 32) {
                reinterpret_cast<T*>(a.out16)[(int64_t)dst * D + c] = cvt_from_float<T>(tmp[c]);
                if (a.out32) a.out32[(int64_t)dst * D + c] = tmp[c];
            }
            if (a.perm && lane == 0) a.perm[l0 + r] = s.perm[r];
            const int src = first ? r : s.perm[r];   // order in which this frame is remembered
            for (int c = lane; c < D; c += 32) st_edge[(int64_t)r * D + c] = edgec[(int64_t)src * D + c];
        }
        for (int c = tid; c < D; c += kChainThreads) st_time[c] = a.time_emb[(int64_t)lf * D + c];
        __syncthreads();
        for (int r = tid; r < n; r += kChainThreads) s.ord_prev[r] = first ? r : s.perm[r];
        n_prev = n;
        last_l0 = l0;
        __syncthreads();
        CHAIN_TICK(5);
    }
    // ---- carry the last frame's matching embeddings (in matched order) to the next call ----------------
    if (last_l0 >= 0) {
        float* st_reg = a.st_reg + (int64_t)sb * KM * E;
        float* st_cls = a.st_cls + (int64_t)sb * KM * E;
        const float* Rc = a.emb_reg + (int64_t)last_l0 * E;
        const float* Cc = a.emb_cls + (int64_t)last_l0 * E;
        for (int t = tid; t < n_prev * (E / 4); t += kChainThreads) {
            const int r = t / (E / 4), c4 = t - r * (E / 4);
            const int src = s.ord_prev[r];
            reinterpret_cast<float4*>(st_reg)[(int64_t)r * (E / 4) + c4] = reinterpret_cast<const float4*>(Rc)[(int64_t)src * (E / 4) + c4];
            reinterpret_cast<float4*>(st_cls)[(int64_t)r * (E / 4) + c4] = reinterpret_cast<const float4*>(Cc)[(int64_t)src * (E / 4) + c4];
        }
        for (int r = tid; r < n_prev; r += kChainThreads) {
            a.st_nreg[(int64_t)sb * KM + r] = a.norm_reg[last_l0 + s.ord_prev[r]];
            a.st_ncls[(int64_t)sb * KM + r] = a.norm_cls[last_l0 + s.ord_prev[r]];
        }
    }
    if (tid == 0) a.st_n[sb] = n_prev;
    __syncthreads();
    CHAIN_TICK(6);
}


// ================================================================================================================
// Fast chain for frames of at most 32 proposals (kmax <= 32: the mode-A / BASELINE configuration, K = 30).
//
// One CTA (16 warps) per clip.  The whole per-frame working set lives in shared memory and the two small matrix
// products of every step run on the tensor cores with warp-level mma.sync (m16n8k16, 16-bit operands, fp32
// accumulation) -- a 30-row problem is latency-bound, far below the 128-row tcgen05 tile:
//   * W_q (256x256) is held in REGISTERS for the whole chain: warp w owns output channels [16w, 16w+16), i.e. the
//     B fragments of 2 n-tiles x 16 k-steps = 64 registers per thread, loaded once per clip;
//   * k_reg / v_reg projections, raw features, edge features, time embedding and the frame's LSAP solution of frame
//     i+1 are prefetched with cp.async into the second half of a double buffer while frame i is computed;
//   * q is kept un-normalised (16-bit) with its per-(row, head) squared norms; the cosine of the attention is
//     S * (1/|q_r|) * (1/|k_j|), applied to the fp32 accumulators;  softmax in registers;  P feeds the P.V product
//     straight from the accumulator layout (no shared-memory round trip);
//   * LayerNorm(identity + attn) is written in place as the next frame's `last_outputs`.
// ================================================================================================================
constexpr int kFR = 32;        // rows per frame (capacity of the fast path)
constexpr int kFS = 264;       // padded row pitch (16-bit elements) of the ldmatrix operands: 528 B -> conflict-free
constexpr int kFastThreads = 512;

template <typename T>
struct FastBuf {
    T k[kFR * kFS];
    T v[kFR * kFS];
    T feat[kFR * 256];
    T edge[kFR * 256];
    float time[256];
    int col[kFR], row[kFR];
};

template <typename T>
struct FastSmem {
    FastBuf<T> buf[2];
    T qin[kFR * kFS];
    T q[kFR * kFS];
    float x[kFR * 256];          // pre-norm output of the current frame, then (in place) last_outputs
    float qss[kFR][16];          // squared norm partials of q: [row][warp]; head h = warps 2h, 2h+1
    float ln[4][256];            // ln_w, ln_b, dec_w, dec_b
    float4 se[32];               // (w1[j][0], w1[j][1], w2[0][j], w2[1][j])
    int perm[kFR], prow[kFR], ord_prev[kFR], frames[64];
};

template <typename T>
__device__ __forceinline__ void fast_prefetch(const tscd_cafm_chain_args& a, FastBuf<T>& dst, int b, int f, int tid) {
    const int lf = b * a.L + f;
    const int l0 = a.lrow_off[lf], n = a.lrow_off[lf + 1] - l0;
    const int r0 = a.row_off[b * a.F + f];
    const T* kp = reinterpret_cast<const T*>(a.kproj16) + (int64_t)l0 * 256;
    const T* vp = reinterpret_cast<const T*>(a.vproj16) + (int64_t)l0 * 256;
    const T* fp = reinterpret_cast<const T*>(a.bank_reg) + (int64_t)r0 * 256;
    const T* ep = reinterpret_cast<const T*>(a.bank_edge) + (int64_t)r0 * 256;
    for (int i = tid; i < n * 32; i += kFastThreads) {
        const int r = i >> 5, c = (i & 31) * 8;
        cp_async16(&dst.k[r * kFS + c], kp + r * 256 + c);
        cp_async16(&dst.v[r * kFS + c], vp + r * 256 + c);
        cp_async16(&dst.feat[r * 256 + c], fp + r * 256 + c);
        cp_async16(&dst.edge[r * 256 + c], ep + r * 256 + c);
    }
    for (int i = n * 32 + tid; i < kFR * 32; i += kFastThreads) {          // padding rows: keys are masked, values must be finite
        const int r = i >> 5, c = (i & 31) * 8;
        *reinterpret_cast<uint4*>(&dst.k[r * kFS + c]) = make_uint4(0, 0, 0, 0);
        *reinterpret_cast<uint4*>(&dst.v[r * kFS + c]) = make_uint4(0, 0, 0, 0);
    }
    if (tid < 64) cp_async16(&dst.time[tid * 4], a.time_emb + (int64_t)lf * 256 + tid * 4);
    if (tid >= 64 && tid < 64 + kFR) {
        const int i = tid - 64;
        if (i < a.kmax) {
            cp_async4(&dst.col[i], a.lap_col + (int64_t)lf * a.kmax + i);
            cp_async4(&dst.row[i], a.lap_row + (int64_t)lf * a.kmax + i);
        }
    }
    cp_async_commit();
}

template <typename T>
__global__ void __launch_bounds__(kFastThreads, 1) cafm_chain_fast_kernel(const tscd_cafm_chain_args a) {
    extern __shared__ __align__(16) unsigned char chain_smem[];
    FastSmem<T>& s = *reinterpret_cast<FastSmem<T>*>(chain_smem);
    const int b = blockIdx.x;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int g = lane >> 2, t4 = lane & 3;
    const int KM = a.kmax, E = 4 * 256;

    // ---- one-time setup: weights, list of non-empty frames, carried state --------------------------------
    if (tid < 32) s.se[tid] = make_float4(a.se_w1[2 * tid], a.se_w1[2 * tid + 1], a.se_w2[tid], a.se_w2[32 + tid]);
    for (int c = tid; c < 256; c += kFastThreads) {
        s.ln[0][c] = a.ln_w[c]; s.ln[1][c] = a.ln_b[c]; s.ln[2][c] = a.dec_w[c]; s.ln[3][c] = a.dec_b[c];
    }
    const bool resume = a.resume ? (a.resume[b] != 0) : false;
    int n_prev = resume ? a.st_n[a.slot ? a.slot[b] : b] : 0;
    bool bad = n_prev > kFR;
    int m = 0;                                   // number of non-empty frames (uniform: every thread scans the offsets)
    for (int f = 0; f < a.L; ++f) {
        const int n = a.lrow_off[b * a.L + f + 1] - a.lrow_off[b * a.L + f];
        if (n > kFR || n > KM) bad = true;
        if (n > 0) { if (tid == 0 && m < 64) s.frames[m] = f; ++m; }
    }
    if (bad || a.L > 64) {
        if (tid == 0) atomicMin(a.status, TSCD_ERR_CAPACITY);
        return;
    }
    // W_q fragments: warp w owns output channels [16w, 16w+16); B[k][n] = W[n][k] -> thread (g, t4) holds
    // W[n0 + g][k0 + 2*t4 .. +1] and W[n0 + g][k0 + 8 + 2*t4 .. +1]
    uint32_t wq[2][16][2];
    {
        const T* W = reinterpret_cast<const T*>(a.wq16);
#pragma unroll
        for (int nt = 0; nt < 2; ++nt)
#pragma unroll
            for (int ks = 0; ks < 16; ++ks) {
                const T* p = W + (int64_t)(warp * 16 + nt * 8 + g) * 256 + ks * 16 + 2 * t4;
                wq[nt][ks][0] = __ldg(reinterpret_cast<const uint32_t*>(p));
                wq[nt][ks][1] = __ldg(reinterpret_cast<const uint32_t*>(p + 8));
            }
    }
    if (tid < kFR) s.ord_prev[tid] = tid;        // carried state is already in matched order
    __syncthreads();                             // s.frames visible
    if (m > 0) fast_prefetch<T>(a, s.buf[0], b, s.frames[0], tid);
    if (n_prev > 0) {                            // resume: last_outputs -> x, last edge / time -> the "previous" buffer
        const int sb = a.slot ? a.slot[b] : b;   // state slot of clip b (re-read where needed: no register held across the loop)
        const float* so = a.st_out + (int64_t)sb * KM * 256;
        const float* se = a.st_edge + (int64_t)sb * KM * 256;
        for (int i = tid; i < n_prev * 256; i += kFastThreads) {
            s.x[i] = so[i];
            s.buf[1].edge[i] = cvt_from_float<T>(se[i]);          // exact: edge features are 16-bit bank values
        }
        for (int c = tid; c < 256; c += kFastThreads) s.buf[1].time[c] = a.st_time[(int64_t)sb * 256 + c];
    }
    int slot = 0, last_l0 = -1;

    for (int fi = 0; fi < m; ++fi) {
        const int f = s.frames[fi];
        const int lf = b * a.L + f;
        const int l0 = a.lrow_off[lf], n = a.lrow_off[lf + 1] - l0;
        FastBuf<T>& cur = s.buf[slot];
        FastBuf<T>& prv = s.buf[slot ^ 1];
        const bool first = (f == 0 && !resume) || n_prev == 0;
        const int np = first ? n : n_prev;
        cp_async_wait_all();
        __syncthreads();                                          // cur is loaded; previous frame's writes are visible

        // ---- assignment: re-index the frame's LSAP solution by how the reference frame remembers its rows ----
        if (warp == 0) {
            if (np <= n) {
                if (lane < np) {
                    s.perm[lane] = cur.col[first ? lane : s.ord_prev[lane]];
                    s.prow[lane] = first ? (-1 - lane) : lane;
                }
                const bool un = lane < n && cur.row[lane] == -1;
                const unsigned bal = __ballot_sync(0xffffffffu, un);
                const int pos = np + __popc(bal & ((1u << lane) - 1u));
                if (un && pos < n) { s.perm[pos] = lane; s.prow[pos] = -1 - lane; }
            } else {
                const int c = lane < np ? cur.col[s.ord_prev[lane]] : -1;
                const bool mt = c >= 0;
                const unsigned bal = __ballot_sync(0xffffffffu, mt);
                const int pos = __popc(bal & ((1u << lane) - 1u));
                if (mt && pos < n) { s.perm[pos] = c; s.prow[pos] = lane; }
            }
        }
        __syncthreads();

        // ---- query input  SE(tgt, query_edge) + query_pos  (tscd_matching.py:566-575), 16-bit A operand ------------
        {
            const float* tm = first ? cur.time : prv.time;
#pragma unroll 1
            for (int pass = 0; pass < 2; ++pass) {
                const int r = (tid >> 5) + pass * 16, c0 = (tid & 31) * 8;
                uint4 packed = make_uint4(0, 0, 0, 0);
                if (r < n) {
                    const int p = s.prow[r];
                    float ta[8], ed[8], o[8];
                    if (p >= 0) { load8(&s.x[p * 256 + c0], ta); load8(&prv.edge[s.ord_prev[p] * 256 + c0], ed); }
                    else        { load8(&cur.feat[(-1 - p) * 256 + c0], ta); load8(&cur.edge[(-1 - p) * 256 + c0], ed); }
                    se_gate8(ta, ed, s.se, o);
                    float tv[8];
                    load8(&tm[c0], tv);
                    packed.x = pack2<T>(o[0] + tv[0], o[1] + tv[1]); packed.y = pack2<T>(o[2] + tv[2], o[3] + tv[3]);
                    packed.z = pack2<T>(o[4] + tv[4], o[5] + tv[5]); packed.w = pack2<T>(o[6] + tv[6], o[7] + tv[7]);
                }
                *reinterpret_cast<uint4*>(&s.qin[r * kFS + c0]) = packed;
            }
        }
        __syncthreads();
        // the previous frame's buffer is free now: prefetch the next non-empty frame into it
        if (fi + 1 < m) fast_prefetch<T>(a, prv, b, s.frames[fi + 1], tid);

        // ---- q = W_q qin on the tensor cores; un-normalised q (16-bit) + per-(row, warp) squared norms ------------
        {
            const int mts = n > 16 ? 2 : 1;
#pragma unroll 1
            for (int mt = 0; mt < mts; ++mt) {
                float acc[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}};
                const T* arow = &s.qin[(mt * 16 + (lane & 15)) * kFS + (lane >> 4) * 8];
#pragma unroll
                for (int ks = 0; ks < 16; ++ks) {
                    uint32_t af[4];
                    ldsm_x4(af, arow + ks * 16);
                    mma16816<T>(acc[0], af, wq[0][ks][0], wq[0][ks][1]);
                    mma16816<T>(acc[1], af, wq[1][ks][0], wq[1][ks][1]);
                }
                float ss0 = 0.f, ss1 = 0.f;
#pragma unroll
                for (int nt = 0; nt < 2; ++nt) {
                    const int col = warp * 16 + nt * 8 + 2 * t4;
                    *reinterpret_cast<uint32_t*>(&s.q[(mt * 16 + g) * kFS + col]) = pack2<T>(acc[nt][0], acc[nt][1]);
                    *reinterpret_cast<uint32_t*>(&s.q[(mt * 16 + g + 8) * kFS + col]) = pack2<T>(acc[nt][2], acc[nt][3]);
                    ss0 = fmaf(acc[nt][0], acc[nt][0], fmaf(acc[nt][1], acc[nt][1], ss0));
                    ss1 = fmaf(acc[nt][2], acc[nt][2], fmaf(acc[nt][3], acc[nt][3], ss1));
                }
                ss0 += __shfl_xor_sync(0xffffffffu, ss0, 1); ss0 += __shfl_xor_sync(0xffffffffu, ss0, 2);
                ss1 += __shfl_xor_sync(0xffffffffu, ss1, 1); ss1 += __shfl_xor_sync(0xffffffffu, ss1, 2);
                if (t4 == 0) { s.qss[mt * 16 + g][warp] = ss0; s.qss[mt * 16 + g + 8][warp] = ss1; }
            }
        }
        __syncthreads();

        // ---- 8-head cosine attention over the CURRENT frame only: warp = (head, 16-row tile) -------------------
        {
            const int h = warp >> 1, mt = warp & 1;
            if (mt * 16 < n) {
                // 1 / |k_j| of this head, lane = key
                float invk;
                {
                    float ssk = 0.f;
#pragma unroll
                    for (int c = 0; c < 4; ++c) {
                        float kv[8];
                        load8(&cur.k[lane * kFS + h * 32 + c * 8], kv);
#pragma unroll
                        for (int i = 0; i < 8; ++i) ssk = fmaf(kv[i], kv[i], ssk);
                    }
                    invk = 1.f / sqrtf(ssk);
                }
                uint32_t qa[2][4];
                const T* qrow = &s.q[(mt * 16 + (lane & 15)) * kFS + h * 32 + (lane >> 4) * 8];
                ldsm_x4(qa[0], qrow);
                ldsm_x4(qa[1], qrow + 16);
                float sc[4][4];
#pragma unroll
                for (int nt = 0; nt < 4; ++nt) {
                    uint32_t kb[4];
                    ldsm_x4(kb, &cur.k[(nt * 8 + (lane & 7)) * kFS + h * 32 + (lane >> 3) * 8]);
                    sc[nt][0] = sc[nt][1] = sc[nt][2] = sc[nt][3] = 0.f;
                    mma16816<T>(sc[nt], qa[0], kb[0], kb[1]);
                    mma16816<T>(sc[nt], qa[1], kb[2], kb[3]);
                }
                const int R0 = mt * 16 + g, R1 = R0 + 8;
                const float iq0 = 1.f / sqrtf(s.qss[R0][2 * h] + s.qss[R0][2 * h + 1]);
                const float iq1 = 1.f / sqrtf(s.qss[R1][2 * h] + s.qss[R1][2 * h + 1]);
                float mx0 = -INFINITY, mx1 = -INFINITY;
#pragma unroll
                for (int nt = 0; nt < 4; ++nt) {
                    const int j0 = nt * 8 + 2 * t4;
                    const float ik0 = __shfl_sync(0xffffffffu, invk, j0), ik1 = __shfl_sync(0xffffffffu, invk, j0 + 1);
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
                float o[4][4];
#pragma unroll
                for (int nt = 0; nt < 4; ++nt) o[nt][0] = o[nt][1] = o[nt][2] = o[nt][3] = 0.f;
#pragma unroll
                for (int ks = 0; ks < 2; ++ks) {
                    uint32_t pa[4];
                    pa[0] = pack2<T>(sc[2 * ks][0] * is0, sc[2 * ks][1] * is0);
                    pa[1] = pack2<T>(sc[2 * ks][2] * is1, sc[2 * ks][3] * is1);
                    pa[2] = pack2<T>(sc[2 * ks + 1][0] * is0, sc[2 * ks + 1][1] * is0);
                    pa[3] = pack2<T>(sc[2 * ks + 1][2] * is1, sc[2 * ks + 1][3] * is1);
#pragma unroll
                    for (int ntp = 0; ntp < 2; ++ntp) {
                        uint32_t vb[4];
                        ldsm_x4_trans(vb, &cur.v[(ks * 16 + (lane & 7) + ((lane >> 3) & 1) * 8) * kFS + h * 32 + ntp * 16 + (lane >> 4) * 8]);
                        mma16816<T>(o[2 * ntp], pa, vb[0], vb[1]);
                        mma16816<T>(o[2 * ntp + 1], pa, vb[2], vb[3]);
                    }
                }
                // identity + attention -> pre-norm output (tscd_matching.py:585-586)
#pragma unroll
                for (int half = 0; half < 2; ++half) {
                    const int R = half ? R1 : R0;
                    if (R < n) {
                        const int idr = first ? R : s.perm[R];
#pragma unroll
                        for (int nt = 0; nt < 4; ++nt) {
                            const int col = h * 32 + nt * 8 + 2 * t4;
                            const float i0 = ldf_reg(cur.feat[idr * 256 + col]), i1 = ldf_reg(cur.feat[idr * 256 + col + 1]);
                            *reinterpret_cast<float2*>(&s.x[R * 256 + col]) = make_float2(i0 + o[nt][2 * half], i1 + o[nt][2 * half + 1]);
                        }
                    }
                }
            }
        }
        __syncthreads();

        // ---- LayerNorm (new last_outputs, in place) + decoder_norm -> output in the original row order ------------
        for (int r = warp; r < n; r += 16) {
            float v[8], y[8], z[8];
            load8(&s.x[r * 256 + lane * 8], v);
            float sm = 0.f;
#pragma unroll
            for (int i = 0; i < 8; ++i) sm += v[i];
            float mean = warp_sumf(sm) / 256.f, var = 0.f;
#pragma unroll
            for (int i = 0; i < 8; ++i) { const float d = v[i] - mean; var = fmaf(d, d, var); }
            float rstd = rsqrtf(warp_sumf(var) / 256.f + 1e-5f);
#pragma unroll
            for (int i = 0; i < 8; ++i) y[i] = (v[i] - mean) * rstd * s.ln[0][lane * 8 + i] + s.ln[1][lane * 8 + i];
            *reinterpret_cast<float4*>(&s.x[r * 256 + lane * 8]) = make_float4(y[0], y[1], y[2], y[3]);
            *reinterpret_cast<float4*>(&s.x[r * 256 + lane * 8 + 4]) = make_float4(y[4], y[5], y[6], y[7]);
            sm = 0.f;
#pragma unroll
            for (int i = 0; i < 8; ++i) sm += y[i];
            mean = warp_sumf(sm) / 256.f; var = 0.f;
#pragma unroll
            for (int i = 0; i < 8; ++i) { const float d = y[i] - mean; var = fmaf(d, d, var); }
            rstd = rsqrtf(warp_sumf(var) / 256.f + 1e-5f);
#pragma unroll
            for (int i = 0; i < 8; ++i) z[i] = (y[i] - mean) * rstd * s.ln[2][lane * 8 + i] + s.ln[3][lane * 8 + i];
            const int64_t dst = (int64_t)(l0 + s.perm[r]) * 256 + lane * 8;
            uint4 pk;
            pk.x = pack2<T>(z[0], z[1]); pk.y = pack2<T>(z[2], z[3]); pk.z = pack2<T>(z[4], z[5]); pk.w = pack2<T>(z[6], z[7]);
            *reinterpret_cast<uint4*>(reinterpret_cast<T*>(a.out16) + dst) = pk;
            if (a.out32) {
                *reinterpret_cast<float4*>(a.out32 + dst) = make_float4(z[0], z[1], z[2], z[3]);
                *reinterpret_cast<float4*>(a.out32 + dst + 4) = make_float4(z[4], z[5], z[6], z[7]);
            }
            if (a.perm && lane == 0) a.perm[l0 + r] = s.perm[r];
        }
        __syncthreads();
        if (tid < n) s.ord_prev[tid] = first ? tid : s.perm[tid];   // order in which this frame is remembered
        n_prev = n;
        last_l0 = l0;
        slot ^= 1;
    }
    __syncthreads();

    // ---- write the memory back (tscd_matching.py:876-878) for the next call ------------------------------------
    const int sb = a.slot ? a.slot[b] : b;
    if (last_l0 >= 0) {
        const FastBuf<T>& lastb = s.buf[slot ^ 1];
        float* so = a.st_out + (int64_t)sb * KM * 256;
        float* se = a.st_edge + (int64_t)sb * KM * 256;
        for (int i = tid; i < n_prev * 256; i += kFastThreads) {
            const int r = i >> 8, c = i & 255;
            so[i] = s.x[i];
            se[i] = ldf_reg(lastb.edge[s.ord_prev[r] * 256 + c]);
        }
        for (int c = tid; c < 256; c += kFastThreads) a.st_time[(int64_t)sb * 256 + c] = lastb.time[c];
        float* st_reg = a.st_reg + (int64_t)sb * KM * E;
        float* st_cls = a.st_cls + (int64_t)sb * KM * E;
        if (a.emb_dtype != TSCD_F32) {
            // 16-bit matching embeddings: widened to fp32 in the state (exact), 8 values per 16-byte load
            const T* Rc16 = reinterpret_cast<const T*>(a.emb_reg) + (int64_t)last_l0 * E;
            const T* Cc16 = reinterpret_cast<const T*>(a.emb_cls) + (int64_t)last_l0 * E;
            for (int i = tid; i < n_prev * (E / 8); i += kFastThreads) {
                const int r = i / (E / 8), c8 = i - r * (E / 8);
                const int src = s.ord_prev[r];
                float vr[8], vc[8];
                load8(Rc16 + (int64_t)src * E + c8 * 8, vr);
                load8(Cc16 + (int64_t)src * E + c8 * 8, vc);
                store8(st_reg + (int64_t)r * E + c8 * 8, vr);
                store8(st_cls + (int64_t)r * E + c8 * 8, vc);
            }
        } else {
        const float* Rc = a.emb_reg + (int64_t)last_l0 * E;
            const float* Cc = a.emb_cls + (int64_t)last_l0 * E;
            // 2 x n_prev x 4 KB: batches of four independent 16-byte loads per matrix before the stores (latency-bound otherwise)
            for (int i0 = 0; i0 < n_prev * (E / 4); i0 += 4 * kFastThreads) {
                float4 vr[4], vc[4];
    #pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const int i = i0 + u * kFastThreads + tid;
                    if (i < n_prev * (E / 4)) {
                        const int r = i / (E / 4), c4 = i - r * (E / 4);
                        const int src = s.ord_prev[r];
                        vr[u] = __ldg(reinterpret_cast<const float4*>(Rc) + (int64_t)src * (E / 4) + c4);
                        vc[u] = __ldg(reinterpret_cast<const float4*>(Cc) + (int64_t)src * (E / 4) + c4);
                    }
                }
    #pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const int i = i0 + u * kFastThreads + tid;
                    if (i < n_prev * (E / 4)) {
                        reinterpret_cast<float4*>(st_reg)[i] = vr[u];
                        reinterpret_cast<float4*>(st_cls)[i] = vc[u];
                    }
                }
            }
        }
        for (int r = tid; r < n_prev; r += kFastThreads) {
            a.st_nreg[(int64_t)sb * KM + r] = a.norm_reg[last_l0 + s.ord_prev[r]];
            a.st_ncls[(int64_t)sb * KM + r] = a.norm_cls[last_l0 + s.ord_prev[r]];
        }
    }
    if (tid == 0) a.st_n[sb] = n_prev;
}


// ================================================================================================================
// Wide chain (frames of MORE than 32 proposals: mode B, 50..500 per frame).  The recurrence is sequential over the local
// frames of a clip, but one frame's step is a large parallel problem (SE gate on n x 256 elements, a 256 x 256
// projection, an n x n attention over 8 heads, two LayerNorms): run by ONE CTA per clip it kept a handful of SMs busy
// for ~1 ms per frame.  Here every step is a short sequence of batch-wide launches over ALL clips:
//     tscd_cafm_wide(phase 0)            once: n_prev / ord_prev from the carried state
//     for f in 0 .. L-1:
//         tscd_cafm_wide(phase 1, f)     permutation of the frame (block scans) + query input rows (SE gate) -> 16-bit
//         tscd_linear                    q = W_q qin                 (tcgen05 GEMM over B * kmax rows)
//         tscd_frame_flash               softmax(q^ k^T) v           (mma.sync flash kernel, 8 heads x 32)
//         tscd_cafm_wide(phase 2, f)     identity + LayerNorm -> new memory, decoder norm -> output rows, state update
//     tscd_cafm_wide(phase 3)            once: matching embeddings of the last frame into the carried state
// Same arithmetic as cafm_chain_kernel (tscd_matching.py:722-888) except that q / k / v enter the two products as 16-bit
// operands, like the fast chain for small frames.
// ================================================================================================================
struct WideCtl { int n, np, first, l0, skip, pad0, pad1, pad2; };

__global__ void cafm_wide_begin_kernel(const tscd_cafm_wide_args w) {
    const tscd_cafm_chain_args& a = w.base;
    const int b = blockIdx.x, KM = a.kmax;
    const bool resume = a.resume ? (a.resume[b] != 0) : false;
    for (int r = threadIdx.x; r < KM; r += blockDim.x) w.ord_prev[(int64_t)b * KM + r] = r;
    if (threadIdx.x == 0) { w.n_prev[b] = resume ? a.st_n[a.slot ? a.slot[b] : b] : 0; w.last_l0[b] = -1; }
}

// one CTA (512 threads, rows in chunks of 512) per clip: control block + perm / prow of frame f (tscd_matching.py:813-844)
__global__ void __launch_bounds__(512) cafm_wide_perm_kernel(const tscd_cafm_wide_args w, int f) {
    __shared__ int scan[40];
    const tscd_cafm_chain_args& a = w.base;
    const int b = blockIdx.x, KM = a.kmax, tid = threadIdx.x;
    const int lf = b * a.L + f;
    const int l0 = a.lrow_off[lf], n = a.lrow_off[lf + 1] - l0;
    const bool resume = a.resume ? (a.resume[b] != 0) : false;
    int n_prev = w.n_prev[b];
    WideCtl* ctl = reinterpret_cast<WideCtl*>(w.ctl) + b;
    int* perm = w.perm_s + (int64_t)b * KM;
    int* prow = w.prow_s + (int64_t)b * KM;
    const int* ord = w.ord_prev + (int64_t)b * KM;
    __syncthreads();                                 // every thread has read n_prev before thread 0 may reset it
    if (n == 0 || n > KM || n > kWideMax || n_prev > KM) {
        if (tid == 0) {
            if (n == 0) { if (f == 0 && !resume) w.n_prev[b] = 0; }
            else atomicMin(a.status, TSCD_ERR_CAPACITY);
            ctl->n = 0; ctl->skip = 1; ctl->l0 = l0; ctl->first = 0; ctl->np = 0;
            w.q_beg[b] = b * KM; w.q_end[b] = b * KM; w.kv_beg[b] = l0; w.kv_end[b] = l0;
        }
        return;
    }
    const bool first = (f == 0 && !resume) || n_prev == 0;
    const int np = first ? n : n_prev;
    const int32_t* colo = a.lap_col + (int64_t)lf * KM;
    const int32_t* rowo = a.lap_row + (int64_t)lf * KM;
    int carry = 0;
    if (np <= n) {
        for (int r = tid; r < np; r += 512) { perm[r] = colo[first ? r : ord[r]]; prow[r] = r; }
        // unmatched current columns follow in ascending order
        for (int c0 = 0; c0 < n; c0 += 512) {
            const int c = c0 + tid;
            const int flag = (c < n && rowo[c] == -1) ? 1 : 0;
            int tot;
            const int ex = carry + block_excl_scan(flag, scan, &tot);
            if (flag && np + ex < n) { perm[np + ex] = c; prow[np + ex] = -1 - c; }
            carry += tot;
        }
    } else {
        for (int r0 = 0; r0 < np; r0 += 512) {
            const int r = r0 + tid;
            int c = -1;
            if (r < np) c = colo[ord[r]];
            const int flag = c >= 0 ? 1 : 0;
            int tot;
            const int ex = carry + block_excl_scan(flag, scan, &tot);
            if (flag && ex < n) { perm[ex] = c; prow[ex] = r; }
            carry += tot;
        }
    }
    if (tid == 0) {
        ctl->n = n; ctl->np = np; ctl->first = first ? 1 : 0; ctl->l0 = l0; ctl->skip = 0;
        w.q_beg[b] = b * KM; w.q_end[b] = b * KM + n; w.kv_beg[b] = l0; w.kv_end[b] = l0 + n;
    }
}

// query input rows (ReferringCrossAttentionLayer: SE(tgt, query_edge) + query_pos), 8 rows per CTA, thread = channel
template <typename T>
__global__ void __launch_bounds__(256) cafm_wide_qin_kernel(const tscd_cafm_wide_args w) {
    __shared__ float w1[64], w2[64];
    const tscd_cafm_chain_args& a = w.base;
    const int b = blockIdx.x, KM = a.kmax, D = a.D, c = threadIdx.x;
    const WideCtl ctl = reinterpret_cast<const WideCtl*>(w.ctl)[b];
    if (threadIdx.x < 64) { w1[threadIdx.x] = a.se_w1[threadIdx.x]; w2[threadIdx.x] = a.se_w2[threadIdx.x]; }
    __syncthreads();
    T* qin = reinterpret_cast<T*>(w.qin16) + (int64_t)b * KM * D;
    const int sb = a.slot ? a.slot[b] : b;           // state slot of clip b
    const float* st_out = a.st_out + (int64_t)sb * KM * D;
    const float* st_edge = a.st_edge + (int64_t)sb * KM * D;
    const float tm = a.st_time[(int64_t)sb * D + c];
    const int* prow = w.prow_s + (int64_t)b * KM;
    for (int r = blockIdx.y * 8; r < min(KM, blockIdx.y * 8 + 8); ++r) {
        float v = 0.f;
        if (!ctl.skip && r < ctl.n) {
            if (ctl.first) {
                v = a.kin[(int64_t)(ctl.l0 + r) * D + c];                  // SE(feat, edge) + time of this frame
            } else {
                const int p = prow[r];
                const float tg = p >= 0 ? st_out[(int64_t)p * D + c] : a.feat[(int64_t)(ctl.l0 - 1 - p) * D + c];
                const float ed = p >= 0 ? st_edge[(int64_t)p * D + c] : a.edge[(int64_t)(ctl.l0 - 1 - p) * D + c];
                v = se_gate(tg, ed, w1, w2) + tm;
            }
        }
        qin[(int64_t)r * D + c] = cvt_from_float<T>(v);
    }
}

// identity + attention -> LayerNorm (new last_outputs) -> decoder norm (output rows); state update.  Warp per row.
template <typename T>
__global__ void __launch_bounds__(256) cafm_wide_finish_kernel(const tscd_cafm_wide_args w, int f) {
    __shared__ float xs[8][256], ys[8][256];
    const tscd_cafm_chain_args& a = w.base;
    const int b = blockIdx.x, KM = a.kmax, D = a.D, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const WideCtl ctl = reinterpret_cast<const WideCtl*>(w.ctl)[b];
    if (ctl.skip) return;
    const int lf = b * a.L + f, n = ctl.n, l0 = ctl.l0;
    const bool first = ctl.first != 0;
    const int* perm = w.perm_s + (int64_t)b * KM;
    const int sb = a.slot ? a.slot[b] : b;           // state slot of clip b
    float* st_out = a.st_out + (int64_t)sb * KM * D;
    float* st_edge = a.st_edge + (int64_t)sb * KM * D;
    const int r = blockIdx.y * 8 + warp;
    if (r < n) {
        const int pr = perm[r];
        const int idr = first ? r : pr;
        for (int c = lane; c < D; c += 32)
            xs[warp][c] = a.feat[(int64_t)(l0 + idr) * D + c] + w.attn[((int64_t)b * KM + r) * D + c];
        __syncwarp();
        layer_norm_row(xs[warp], a.ln_w, a.ln_b, ys[warp], D, lane);
        __syncwarp();
        for (int c = lane; c < D; c += 32) st_out[(int64_t)r * D + c] = ys[warp][c];          // new last_outputs
        layer_norm_row(ys[warp], a.dec_w, a.dec_b, xs[warp], D, lane);
        __syncwarp();
        const int dst = l0 + pr;
        for (int c = lane; c < D; c += 32) {
            reinterpret_cast<T*>(a.out16)[(int64_t)dst * D + c] = cvt_from_float<T>(xs[warp][c]);
            if (a.out32) a.out32[(int64_t)dst * D + c] = xs[warp][c];
            st_edge[(int64_t)r * D + c] = a.edge[(int64_t)(l0 + idr) * D + c];
        }
        if (lane == 0) {
            if (a.perm) a.perm[l0 + r] = pr;
            w.ord_prev[(int64_t)b * KM + r] = idr;
        }
    }
    if (blockIdx.y == 0) {
        for (int c = threadIdx.x; c < D; c += blockDim.x) a.st_time[(int64_t)sb * D + c] = a.time_emb[(int64_t)lf * D + c];
        if (threadIdx.x == 0) { w.n_prev[b] = n; w.last_l0[b] = l0; }
    }
}

// carry the last frame's matching embeddings (in matched order) to the next call
__global__ void __launch_bounds__(256) cafm_wide_end_kernel(const tscd_cafm_wide_args w) {
    const tscd_cafm_chain_args& a = w.base;
    const int b = blockIdx.x, KM = a.kmax, E = 4 * a.D, tid = blockIdx.y * blockDim.x + threadIdx.x;
    const int nthreads = gridDim.y * blockDim.x;
    const int n_prev = w.n_prev[b], last_l0 = w.last_l0[b];
    const int* ord = w.ord_prev + (int64_t)b * KM;
    const int sb = a.slot ? a.slot[b] : b;           // state slot of clip b
    if (last_l0 >= 0) {
        float* st_reg = a.st_reg + (int64_t)sb * KM * E;
        float* st_cls = a.st_cls + (int64_t)sb * KM * E;
        const float* Rc = a.emb_reg + (int64_t)last_l0 * E;
        const float* Cc = a.emb_cls + (int64_t)last_l0 * E;
        for (int t = tid; t < n_prev * (E / 4); t += nthreads) {
            const int r = t / (E / 4), c4 = t - r * (E / 4);
            const int src = ord[r];
            reinterpret_cast<float4*>(st_reg)[(int64_t)r * (E / 4) + c4] = reinterpret_cast<const float4*>(Rc)[(int64_t)src * (E / 4) + c4];
            reinterpret_cast<float4*>(st_cls)[(int64_t)r * (E / 4) + c4] = reinterpret_cast<const float4*>(Cc)[(int64_t)src * (E / 4) + c4];
        }
        for (int r = tid; r < n_prev; r += nthreads) {
            a.st_nreg[(int64_t)sb * KM + r] = a.norm_reg[last_l0 + ord[r]];
            a.st_ncls[(int64_t)sb * KM + r] = a.norm_cls[last_l0 + ord[r]];
        }
    }
    if (tid == 0) a.st_n[sb] = n_prev;
}

}  // namespace tscd

extern "C" int tscd_cafm_wide(const tscd_cafm_wide_args* w, int phase, int frame, void* stream) {
    using namespace tscd;
    if (!w) return TSCD_ERR_INVALID_ARG;
    const tscd_cafm_chain_args& a = w->base;
    if (a.B <= 0 || a.L <= 0 || a.D != 256 || a.kmax <= 0 || a.kmax > kWideMax || frame < 0 || frame >= a.L) return TSCD_ERR_INVALID_ARG;
    if (a.emb_dtype != TSCD_F32 || !w->ctl || !w->perm_s || !w->prow_s || !w->ord_prev || !w->n_prev || !w->last_l0 || !w->q_beg ||
        !w->q_end || !w->kv_beg || !w->kv_end || !w->qin16 || !w->attn)
        return TSCD_ERR_INVALID_ARG;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    const dim3 rows(a.B, (a.kmax + 7) / 8);
    switch (phase) {
        case 0: cafm_wide_begin_kernel<<<a.B, 256, 0, st>>>(*w); break;
        case 1:
            cafm_wide_perm_kernel<<<a.B, 512, 0, st>>>(*w, frame);
            if (a.out_dtype == TSCD_F16) cafm_wide_qin_kernel<__half><<<rows, 256, 0, st>>>(*w);
            else if (a.out_dtype == TSCD_BF16) cafm_wide_qin_kernel<__nv_bfloat16><<<rows, 256, 0, st>>>(*w);
            else return TSCD_ERR_UNSUPPORTED;
            break;
        case 2:
            if (a.out_dtype == TSCD_F16) cafm_wide_finish_kernel<__half><<<rows, 256, 0, st>>>(*w, frame);
            else if (a.out_dtype == TSCD_BF16) cafm_wide_finish_kernel<__nv_bfloat16><<<rows, 256, 0, st>>>(*w, frame);
            else return TSCD_ERR_UNSUPPORTED;
            break;
        case 3: cafm_wide_end_kernel<<<dim3(a.B, 32), 256, 0, st>>>(*w); break;
        default: return TSCD_ERR_INVALID_ARG;
    }
    TSCD_CUDA_CHECK_LAUNCH();
    return TSCD_OK;
}

namespace tscd {
}  // namespace tscd

extern "C" int tscd_cafm_prep(const tscd_cafm_prep_args* a, void* stream) {
    using namespace tscd;
    if (!a || a->B <= 0 || a->L <= 0 || a->D <= 0 || (a->D % 32) != 0) return TSCD_ERR_INVALID_ARG;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    if (a->D != 256) return TSCD_ERR_UNSUPPORTED;
    const dim3 grid(a->B * a->L, 4);
    if (a->bank_dtype == TSCD_F16) cafm_prep_kernel<__half><<<grid, 256, 0, st>>>(*a);
    else if (a->bank_dtype == TSCD_BF16) cafm_prep_kernel<__nv_bfloat16><<<grid, 256, 0, st>>>(*a);
    else return TSCD_ERR_UNSUPPORTED;
    TSCD_CUDA_CHECK_LAUNCH();
    return TSCD_OK;
}

extern "C" int tscd_cafm_cost(const tscd_cafm_cost_args* a, void* stream) {
    using namespace tscd;
    if (!a || a->B <= 0 || a->L <= 0 || a->D != 256 || a->kmax <= 0 || a->kmax > kWideMax) return TSCD_ERR_INVALID_ARG;
    // above kChainMax only the tensor-core kernel of the wide frames (16-bit copies of the embeddings)
    if (a->kmax > kChainMax && (a->emb_dtype != TSCD_F32 || !a->emb_reg16 || !a->emb_cls16)) return TSCD_ERR_UNSUPPORTED;
    const int tiles = (a->kmax + 31) / 32;
    if (a->emb_dtype != TSCD_F32) {                        // 16-bit matching embeddings: tensor-core kernel, frames <= 32 proposals
        if (a->kmax > 32 || !a->norm_reg || !a->norm_cls || !a->ref_n) return TSCD_ERR_INVALID_ARG;
        if (a->emb_dtype == TSCD_F16) cafm_cost16_kernel<__half><<<a->B * a->L, 128, 0, reinterpret_cast<cudaStream_t>(stream)>>>(*a);
        else if (a->emb_dtype == TSCD_BF16) cafm_cost16_kernel<__nv_bfloat16><<<a->B * a->L, 128, 0, reinterpret_cast<cudaStream_t>(stream)>>>(*a);
        else return TSCD_ERR_UNSUPPORTED;
        TSCD_CUDA_CHECK_LAUNCH();
        return TSCD_OK;
    }
    if (a->emb_reg16 && a->emb_cls16 && a->kmax > 32) {      // wide frames, 16-bit copies available: tensor-core kernel
        const size_t sm = (size_t)2 * (kCwRows + kCwCols) * kCwPitch * 2;
        const dim3 grid(a->B * a->L, (a->kmax + kCwRows - 1) / kCwRows, (a->kmax + kCwCols - 1) / kCwCols);
        cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
        if (a->emb16_dtype == TSCD_F16) {
            if (cudaFuncSetAttribute(cafm_cost_wide16_kernel<__half>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm) != cudaSuccess) return TSCD_ERR_CUDA;
            cafm_cost_wide16_kernel<__half><<<grid, kCwThreads, sm, st>>>(*a);
        } else if (a->emb16_dtype == TSCD_BF16) {
            if (cudaFuncSetAttribute(cafm_cost_wide16_kernel<__nv_bfloat16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm) != cudaSuccess) return TSCD_ERR_CUDA;
            cafm_cost_wide16_kernel<__nv_bfloat16><<<grid, kCwThreads, sm, st>>>(*a);
        } else {
            return TSCD_ERR_UNSUPPORTED;
        }
        TSCD_CUDA_CHECK_LAUNCH();
        return TSCD_OK;
    }
    cafm_cost_kernel<<<dim3(a->B * a->L, tiles, tiles), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(*a);
    TSCD_CUDA_CHECK_LAUNCH();
    return TSCD_OK;
}

extern "C" int tscd_cafm_lap(const tscd_cafm_lap_args* a, void* stream) {
    using namespace tscd;
    if (!a || a->num_frames <= 0 || a->kmax <= 0 || a->kmax > kWideMax) return TSCD_ERR_INVALID_ARG;
    if (a->kmax <= 32) {
        const size_t sm = (size_t)kLapPack * 1024 * sizeof(float);
        if (cudaFuncSetAttribute(cafm_lap_small_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm) != cudaSuccess) return TSCD_ERR_CUDA;
        cafm_lap_small_kernel<<<(a->num_frames + kLapPack - 1) / kLapPack, kLapPack * 32, sm, reinterpret_cast<cudaStream_t>(stream)>>>(*a);
        TSCD_CUDA_CHECK_LAUNCH();
        return TSCD_OK;
    }
    const size_t smem = sizeof(LapSmem);
    if (cudaFuncSetAttribute(cafm_lap_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) return TSCD_ERR_CUDA;
    cafm_lap_kernel<<<a->num_frames, 32, smem, reinterpret_cast<cudaStream_t>(stream)>>>(*a);
    TSCD_CUDA_CHECK_LAUNCH();
    if (a->kmax > kChainMax) {       // the solver is picked per problem on the device: each kernel skips the other's problems
        const size_t smem_w = (size_t)a->kmax * (3 * sizeof(double) + 4 * sizeof(int) + 2);
        if (cudaFuncSetAttribute(cafm_lap_cta_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_w) != cudaSuccess) return TSCD_ERR_CUDA;
        cafm_lap_cta_kernel<<<a->num_frames, kLapCtaThreads, smem_w, reinterpret_cast<cudaStream_t>(stream)>>>(*a);
        TSCD_CUDA_CHECK_LAUNCH();
    }
    return TSCD_OK;
}

extern "C" int tscd_debug_chain_clocks(long long* out, int reset) {
    using namespace tscd;
    if (cudaMemcpyFromSymbol(out, g_chain_clk, sizeof(long long) * 8) != cudaSuccess) return TSCD_ERR_CUDA;
    if (reset) {
        long long z[8] = {0, 0, 0, 0, 0, 0, 0, 0};
        if (cudaMemcpyToSymbol(g_chain_clk, z, sizeof(z)) != cudaSuccess) return TSCD_ERR_CUDA;
    }
    return TSCD_OK;
}

extern "C" int tscd_cafm_chain(const tscd_cafm_chain_args* a, void* stream) {
    using namespace tscd;
    if (!a || a->B <= 0 || a->L <= 0 || a->D != 256 || a->kmax <= 0 || a->kmax > kChainMax) return TSCD_ERR_INVALID_ARG;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    if (a->kproj16 && a->vproj16 && a->wq16) {            // fast path: every frame holds <= 32 proposals (kmax <= 32)
        if (a->kmax > kFR || a->L > 64 || !a->bank_reg || !a->bank_edge) return TSCD_ERR_INVALID_ARG;
        if (a->out_dtype == TSCD_F16) {
            const size_t sm = sizeof(FastSmem<__half>);
            if (cudaFuncSetAttribute(cafm_chain_fast_kernel<__half>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm) != cudaSuccess) return TSCD_ERR_CUDA;
            cafm_chain_fast_kernel<__half><<<a->B, kFastThreads, sm, st>>>(*a);
        } else if (a->out_dtype == TSCD_BF16) {
            const size_t sm = sizeof(FastSmem<__nv_bfloat16>);
            if (cudaFuncSetAttribute(cafm_chain_fast_kernel<__nv_bfloat16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm) != cudaSuccess) return TSCD_ERR_CUDA;
            cafm_chain_fast_kernel<__nv_bfloat16><<<a->B, kFastThreads, sm, st>>>(*a);
        } else {
            return TSCD_ERR_UNSUPPORTED;
        }
        TSCD_CUDA_CHECK_LAUNCH();
        return TSCD_OK;
    }
    const size_t smem = sizeof(ChainSmem);
    if (a->out_dtype == TSCD_F16) {
        if (cudaFuncSetAttribute(cafm_chain_kernel<__half>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) return TSCD_ERR_CUDA;
        cafm_chain_kernel<__half><<<a->B, kChainThreads, smem, st>>>(*a);
    } else if (a->out_dtype == TSCD_BF16) {
        if (cudaFuncSetAttribute(cafm_chain_kernel<__nv_bfloat16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) return TSCD_ERR_CUDA;
        cafm_chain_kernel<__nv_bfloat16><<<a->B, kChainThreads, smem, st>>>(*a);
    } else {
        return TSCD_ERR_UNSUPPORTED;
    }
    TSCD_CUDA_CHECK_LAUNCH();
    return TSCD_OK;
}
