// K4: cross-frame attention aggregation on tcgen05 tensor cores (see include/tscd_b200.h for semantics).
//
// Reference: Attention_mca_g2l.forward (yolox/models/post_trans.py:601-714) / Attention_msa.forward (:734-826).
//
// Layout of the work: one CTA per (clip, 128-query tile).  Queries of a clip are its local rows; keys are
// all rows of the clip with a per-(query,key) visibility mask (own frame or global frame), which is how the
// reference's per-local-frame loop (post_trans.py:1143-1151) collapses into one masked attention problem
// and the global K/V projections are computed once instead of once per local frame.
//
// Every matrix product runs on the 5th-gen tensor cores (tcgen05.mma, fp32 accumulators in TMEM):
//   S_cls/S_reg = Qn Kn^T per head (K-major operands straight from TMA, 128-byte swizzle),
//   attn @ V     with the probabilities written to shared memory by the softmax warps as a swizzled K-major
//                A operand and V^T tiles as the B operand,
//   the head-mean raw-v cosine similarity as ONE K=256 product of the per-head-normalised rows,
//   the round-2 weights @ V.
// Softmax statistics are exact two-pass (row max, then exp/sum) so fp16 probabilities never underflow.
// The CTA runs its phases in lock step (TMA -> MMA -> softmax warps); concurrency comes from the other
// clips' CTAs.  Warps 0-3 own the 128 TMEM lanes (thread == query row); warp 4 issues TMA and MMA.
#include <cuda.h>

#include "common.cuh"
#include "tc.cuh"

namespace tscd {

int make_tmap_kmajor(CUtensorMap* m, const void* ptr, int is_bf16, int64_t rows, int64_t K, int64_t ld, int box_rows);

constexpr int kAttnThreads = 160;
constexpr float kLog2e = 1.4426950408889634f;

// -------------------------------------------------------------------------------------------------------
// prep: normalise / scale / transpose
// -------------------------------------------------------------------------------------------------------
template <typename T>
__device__ __forceinline__ float2 ld2(const T* p);
template <> __device__ __forceinline__ float2 ld2<__half>(const __half* p) { return __half22float2(*reinterpret_cast<const __half2*>(p)); }
template <> __device__ __forceinline__ float2 ld2<__nv_bfloat16>(const __nv_bfloat16* p) {
    return __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(p));
}
template <typename T>
__device__ __forceinline__ void st2(T* p, float a, float b);
template <> __device__ __forceinline__ void st2<__half>(__half* p, float a, float b) { *reinterpret_cast<__half2*>(p) = __floats2half2_rn(a, b); }
template <> __device__ __forceinline__ void st2<__nv_bfloat16>(__nv_bfloat16* p, float a, float b) {
    *reinterpret_cast<__nv_bfloat162*>(p) = __floats2bfloat162_rn(a, b);
}

constexpr int kPrepRowPitch = 264;  // 16-bit elements per staged v row: 256 + 8 padding (rows stay 16-byte aligned)

template <typename T>
__device__ __forceinline__ void unpack8(const uint4& raw, float (&v)[8]) {
    const T* e = reinterpret_cast<const T*>(&raw);
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = ldf_reg(e[i]);
}
template <typename T>
__device__ __forceinline__ uint4 pack8(const float (&v)[8], float scale) {
    uint4 o;
    T* e = reinterpret_cast<T*>(&o);
#pragma unroll
    for (int i = 0; i < 8; ++i) e[i] = cvt_from_float<T>(v[i] * scale);
    return o;
}
// sum of squares over the 8 lanes that share a head (lane owns 8 of the head's 64 channels)
__device__ __forceinline__ float head_sumsq(const float (&v)[8]) {
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) s = fmaf(v[i], v[i], s);
    s += __shfl_xor_sync(0xffffffffu, s, 1);
    s += __shfl_xor_sync(0xffffffffu, s, 2);
    s += __shfl_xor_sync(0xffffffffu, s, 4);
    return s;
}

// One CTA per (64 keys, clip); one warp per bank row, lane = 8 consecutive channels (16-byte loads / stores), all four
// heads of a row normalised at once (8 lanes per head).  The un-normalised v rows are staged in shared memory and
// written out transposed (V^T: 64 consecutive keys = 128 bytes per channel row).
constexpr int kPrepThreads = 384;     // 12 warps x 3 CTAs/SM (67.6 KB of staging each): 36 resident warps instead of 24

template <typename T>
__global__ void __launch_bounds__(kPrepThreads) attn_prep_kernel(const tscd_attn_prep_args a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    T* tile_c = reinterpret_cast<T*>(smem_raw);        // [64 keys][kPrepRowPitch]
    T* tile_r = tile_c + 64 * kPrepRowPitch;
    const tscd_attn_layout& lay = a.lay;
    const int b = blockIdx.y, k0 = blockIdx.x * 64;
    const int s0 = lay.row_off[b * lay.F];
    const int n_clip = lay.row_off[(b + 1) * lay.F] - s0;
    const int n_loc = lay.self_attn ? n_clip : (lay.row_off[b * lay.F + lay.L] - s0);
    const int n_pad = min((n_clip + 127) & ~127, lay.nk_pitch);
    if (k0 >= n_pad) return;
    const int lbase = lay.lrow_off[b * lay.L];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int c = lane * 8;

    constexpr int NW = kPrepThreads / 32;
#pragma unroll 2
    for (int rr = warp; rr < 64; rr += NW) {
        const int r = k0 + rr;                 // key index within the clip
        const int row = s0 + r;                // bank row
        const bool valid = r < n_clip;
        if (valid) {                           // frame of the row: lanes test one frame each
            for (int f0 = 0; f0 < lay.F; f0 += 32) {
                const int f = f0 + lane;
                const bool in = f < lay.F && lay.row_off[b * lay.F + f] <= row && row < lay.row_off[b * lay.F + f + 1];
                const unsigned bal = __ballot_sync(0xffffffffu, in);
                if (bal) { if (lane == 0) a.row_frame[row] = f0 + __ffs(bal) - 1; break; }
            }
        }
        const float kscale_c = valid ? a.scale * __ldg(a.key_score + row) : 0.f;
#pragma unroll
        for (int br = 0; br < 2; ++br) {
            const T* src = reinterpret_cast<const T*>(br == 0 ? a.qkv_cls : a.qkv_reg) + (int64_t)row * a.ld_qkv + c;
            T* tile = (br == 0 ? tile_c : tile_r) + (r - k0) * kPrepRowPitch + c;
            if (!valid) {                       // padding keys: V^T columns must be finite (they are multiplied by zero weights)
                *reinterpret_cast<uint4*>(tile) = make_uint4(0, 0, 0, 0);
                continue;
            }
            const bool is_query = r < n_loc;                   // q of the global rows is never read
            const uint4 kraw = __ldg(reinterpret_cast<const uint4*>(src + 256));
            const uint4 vraw = __ldg(reinterpret_cast<const uint4*>(src + 512));
            float k[8], v[8];
            unpack8<T>(kraw, k); unpack8<T>(vraw, v);
            const float ik = (br == 0 ? kscale_c : a.scale) / sqrtf(head_sumsq(k)), iv = 1.f / sqrtf(head_sumsq(v));
            T* kn = reinterpret_cast<T*>(br == 0 ? a.kn_cls : a.kn_reg) + (int64_t)row * 256 + c;
            T* vn = reinterpret_cast<T*>(br == 0 ? a.vn_cls : a.vn_reg) + (int64_t)row * 256 + c;
            *reinterpret_cast<uint4*>(kn) = pack8<T>(k, ik);
            *reinterpret_cast<uint4*>(vn) = pack8<T>(v, iv);
            if (is_query) {                                    // uniform over the warp
                const uint4 qraw = __ldg(reinterpret_cast<const uint4*>(src));
                float q[8];
                unpack8<T>(qraw, q);
                const float iq = 1.f / sqrtf(head_sumsq(q));
                T* qn = reinterpret_cast<T*>(br == 0 ? a.qn_cls : a.qn_reg) + (int64_t)row * 256 + c;
                *reinterpret_cast<uint4*>(qn) = pack8<T>(q, iq);
            }
            T* xori = reinterpret_cast<T*>(br == 0 ? a.xori_cls : a.xori_reg);
            if (xori && r < n_loc) *reinterpret_cast<uint4*>(xori + (int64_t)(lbase + r) * a.ld_xori + c) = vraw;
            *reinterpret_cast<uint4*>(tile) = vraw;
        }
    }
    __syncthreads();
    // transposed store: channel ch -> 64 consecutive keys (128 bytes); lane = two consecutive keys
    for (int ch = warp; ch < 256; ch += NW) {
#pragma unroll
        for (int br = 0; br < 2; ++br) {
            const uint16_t* tile = reinterpret_cast<const uint16_t*>(br == 0 ? tile_c : tile_r);
            const uint32_t lo = tile[(2 * lane) * kPrepRowPitch + ch], hi = tile[(2 * lane + 1) * kPrepRowPitch + ch];
            T* vt = reinterpret_cast<T*>(br == 0 ? a.vt_cls : a.vt_reg) + ((int64_t)b * 256 + ch) * lay.nk_pitch + k0;
            *reinterpret_cast<uint32_t*>(vt + 2 * lane) = lo | (hi << 16);
        }
    }
}

// Row metadata for the fused q|k|v projection (tscd_qkv_project) and the attention kernels: frame of every bank row,
// (clip, key index) of every bank row, and zero fill of the V^T padding columns [n_clip, round_up(n_clip, 128)) that
// the P @ V / W @ V products read with zero weights.  grid (nk_pitch / 64, B), one thread per key.
template <typename T>
__global__ void __launch_bounds__(64) attn_rowmeta_kernel(const tscd_attn_rowmeta_args a) {
    const tscd_attn_layout& lay = a.lay;
    const int b = blockIdx.y, r = blockIdx.x * 64 + threadIdx.x;
    const int s0 = lay.row_off[b * lay.F];
    const int n_clip = lay.row_off[(b + 1) * lay.F] - s0;
    const int n_pad = min((n_clip + 127) & ~127, lay.nk_pitch);
    if (r >= n_pad) return;
    if (r < n_clip) {
        const int row = s0 + r;
        int lo = 0, hi = lay.F;               // frame f with row_off[b*F+f] <= row < row_off[b*F+f+1] (last such f: empty frames)
        while (hi - lo > 1) {
            const int mid = (lo + hi) >> 1;
            if (lay.row_off[b * lay.F + mid] <= row) lo = mid; else hi = mid;
        }
        a.row_frame[row] = lo;
        a.row_meta[row] = (b << 16) | r;
    } else {
        T* vc = reinterpret_cast<T*>(a.vt_cls) + (int64_t)b * 256 * lay.nk_pitch + r;
        T* vr = a.vt_reg ? reinterpret_cast<T*>(a.vt_reg) + (int64_t)b * 256 * lay.nk_pitch + r : nullptr;
        for (int c = 0; c < 256; ++c) {
            vc[(int64_t)c * lay.nk_pitch] = cvt_from_float<T>(0.f);
            if (vr) vr[(int64_t)c * lay.nk_pitch] = cvt_from_float<T>(0.f);
        }
    }
}

// per-clip transpose (64 keys x 64 channels tiles through shared memory)
template <typename T>
__global__ void __launch_bounds__(256) transpose_clip_kernel(const tscd_transpose_args a) {
    __shared__ T tile[64][66];
    const tscd_attn_layout& lay = a.lay;
    const int b = blockIdx.z, k0 = blockIdx.x * 64, c0 = blockIdx.y * 64;
    const int s0 = lay.row_off[b * lay.F];
    const int n_clip = lay.row_off[(b + 1) * lay.F] - s0;
    const int n_pad = min((n_clip + 127) & ~127, lay.nk_pitch);
    if (k0 >= n_pad) return;
    const int tx = threadIdx.x & 63, ty = threadIdx.x >> 6;
    for (int r = ty; r < 64; r += 4) {
        const int key = k0 + r;
        T v = cvt_from_float<T>(0.f);
        if (key < n_clip) v = reinterpret_cast<const T*>(a.x)[(int64_t)(s0 + key) * a.ld_x + c0 + tx];
        tile[r][tx] = v;
    }
    __syncthreads();
    for (int c = ty; c < 64; c += 4)
        reinterpret_cast<T*>(a.xt)[((int64_t)b * a.width + c0 + c) * lay.nk_pitch + k0 + tx] = tile[tx][c];
}

// -------------------------------------------------------------------------------------------------------
// shared pieces of the two tensor-core kernels
// -------------------------------------------------------------------------------------------------------
struct ClipInfo {
    int s0, n_clip, n_loc, lbase, q0;
};
__device__ __forceinline__ ClipInfo clip_info(const tscd_attn_layout& lay, int b, int qtile) {
    ClipInfo c;
    c.s0 = lay.row_off[b * lay.F];
    c.n_clip = min(lay.row_off[(b + 1) * lay.F] - c.s0, lay.nk_pitch);
    c.n_loc = lay.self_attn ? c.n_clip : (lay.row_off[b * lay.F + lay.L] - c.s0);
    c.lbase = lay.lrow_off[b * lay.L];
    c.q0 = qtile * 128;
    return c;
}

// 16-byte chunk `chunk` (8 x 16-bit) of row `row` inside a [rows x 64] K-major tile with 128-byte swizzle
__device__ __forceinline__ uint32_t sw128_off(int row, int chunk) { return (uint32_t)(row * 128 + ((chunk ^ (row & 7)) << 4)); }

template <bool BF16>
__device__ __forceinline__ uint32_t pack2(float a, float b) {
    if (BF16) {
        __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
        return *reinterpret_cast<uint32_t*>(&h);
    } else {
        __half2 h = __floats2half2_rn(a, b);
        return *reinterpret_cast<uint32_t*>(&h);
    }
}

// Debug build (-DTSCD_R2_PROF): clocks one lane per role of CTA (0,0) spends in each barrier wait, by wait-site tag
// (attn_pv tags 300.., attn_round2 tags 400..); read back with tscd_debug_r2_waits (tools/r2_waits.py).
#ifdef TSCD_R2_PROF
__device__ unsigned long long g_r2_wait[64];
__device__ unsigned long long g_pv_wait[64];
__device__ __forceinline__ void wait_prof(unsigned long long* acc, uint64_t* bar, uint32_t parity, int tag, int base) {
    const long long t0 = clock64();
    tc::mbar_wait(bar, parity, tag);
    const long long dt = clock64() - t0;
    if (blockIdx.x == 0 && blockIdx.y == 0 && (threadIdx.x == 0 || (threadIdx.x >= 512 && (threadIdx.x & 31) == 0)))
        atomicAdd(&acc[tag - base], (unsigned long long)dt);
}
#define R2_WAIT(bar, parity, tag) wait_prof(g_r2_wait, bar, parity, tag, 400)
#define PV_WAIT(bar, parity, tag) wait_prof(g_pv_wait, bar, parity, tag, 300)
#else
#define R2_WAIT mbar_wait
#define PV_WAIT mbar_wait
#endif

struct PvTmaps {
    CUtensorMap qc, kc, qr, kr, k64c, k64r, vtc, vtr;
};

// -------------------------------------------------------------------------------------------------------
// attn_pv: row max (pass A), exp/sum + P@V (pass B) -- warp-specialised, mbarrier-pipelined
//
//   warp 16 (one thread) TMA producer: Q tiles (double-buffered per head) and a 3-stage ring of key tiles
//                        (pass A: Kc|Kr of 128 keys, 32 KB; pass B: Kc|Kr of 64 keys, the first 16 KB of a stage);
//   warp 19 (one thread) TMA producer of the value tiles of pass B (Vc^T|Vr^T, the second 16 KB of a stage) -- its own
//                        ring: a key tile is free again as soon as its scores exist, a value tile only after P@V, so
//                        the key loads run up to three tiles ahead of the softmax instead of waiting for P@V;
//   warp 17 (one thread) tcgen05.mma issuer of the scores S = Q K^T (two TMEM score buffers: tile g+1 is computed
//                        while the softmax warps work on tile g);
//   warp 18 (one thread) tcgen05.mma issuer of P(g) @ V(g) (pass B).  (One issuing thread pays ~15 dependent
//                        instructions per UMMA; two issuers halve that serial chain.)
//   warps 0-15           softmax: thread == query row == TMEM lane, warp w owns lanes 32 * (w % 4) and column quarter
//                        w / 4 of every tile (four warps per scheduler hide the TMEM-load -> ex2 -> store chain);
//                        visibility mask from the row's own frame range (no shared-memory side table), exp2, fp16/bf16
//                        probabilities written as the swizzled K-major A operand of the P@V products (two P buffers).
//   TMEM: pass A  2 x (S_cls 128 | S_reg 128);   pass B  2 x (S_cls 64 | S_reg 64) | O_cc O_cr O_rc O_rr (64 each).
// -------------------------------------------------------------------------------------------------------
constexpr int kPvThreads = 640;     // 16 softmax warps (4 per scheduler), 2 TMA warps, 2 MMA warps
constexpr int kPvStages = 3;

struct PvBars {
    uint64_t k_full[kPvStages], k_empty[kPvStages];
    uint64_t v_full[kPvStages], v_empty[kPvStages];
    uint64_t q_full[2], q_empty[2];
    uint64_t s_full[2], s_empty[2];
    uint64_t p_full[2], p_empty[2];
    uint64_t o_full, o_empty;
    uint32_t tmem_base;
    float xch[4][128];         // partial row sums exchanged between the four column quarters of a row (cls, then reg:
                               // the 227 KB window has no room for both at once)
};

static_assert(65536 + kPvStages * 32768 + 65536 + sizeof(PvBars) <= 232448, "attn_pv: over the 227 KB shared-memory window");

__device__ __forceinline__ float ex2_approx(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;\n" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ void softmax_bar_sync() { asm volatile("bar.sync 1, 512;\n" ::: "memory"); }

template <bool BF16>
__global__ void __launch_bounds__(kPvThreads, 1) attn_pv_kernel(const __grid_constant__ PvTmaps tm, const tscd_attn_pv_args a) {
    using namespace tc;
    const tscd_attn_layout& lay = a.lay;
    const int b = blockIdx.y;
    const ClipInfo ci = clip_info(lay, b, blockIdx.x);
    if (ci.q0 >= ci.n_loc) return;
#ifdef TSCD_R2_PROF
    const long long tk0 = clock64();
#endif

    extern __shared__ __align__(1024) unsigned char smem_raw[];
    unsigned char* smem = smem_raw;                      // no static shared memory: the window starts 1024-byte aligned
    if ((smem_u32(smem) & 1023u) != 0) __trap();
    unsigned char* sQ = smem;                            // 2 x (Qc 16K | Qr 16K)
    unsigned char* sKV = smem + 65536;                   // 3 x 32K
    unsigned char* sP = smem + 65536 + kPvStages * 32768;  // 2 x (Pc 16K | Pr 16K)
    PvBars& bars = *reinterpret_cast<PvBars*>(sP + 65536);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 512) {
        tma_prefetch_desc(&tm.qc); tma_prefetch_desc(&tm.kc); tma_prefetch_desc(&tm.qr); tma_prefetch_desc(&tm.kr);
        tma_prefetch_desc(&tm.k64c); tma_prefetch_desc(&tm.k64r); tma_prefetch_desc(&tm.vtc); tma_prefetch_desc(&tm.vtr);
        for (int i = 0; i < kPvStages; ++i) {
            mbar_init(&bars.k_full[i], 1); mbar_init(&bars.k_empty[i], 1);
            mbar_init(&bars.v_full[i], 1); mbar_init(&bars.v_empty[i], 1);
        }
        for (int i = 0; i < 2; ++i) {
            mbar_init(&bars.q_full[i], 1); mbar_init(&bars.q_empty[i], 1);
            mbar_init(&bars.s_full[i], 1); mbar_init(&bars.s_empty[i], 16);
            mbar_init(&bars.p_full[i], 16); mbar_init(&bars.p_empty[i], 1);
        }
        mbar_init(&bars.o_full, 1); mbar_init(&bars.o_empty, 16);
        fence_barrier_init();
    }
    if (warp == 17) tmem_alloc<512>(&bars.tmem_base);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = bars.tmem_base;

    // Single-pass mode (a.max_logit > 0, BF16 operands only): the logits are bounded (|q^ . k^| <= 1 times the key scale), so
    // exp(s - max_logit) needs no row maximum -- IF the probabilities keep their exponent range, which BF16's 8-bit exponent
    // does and fp16's does not (a row whose true maximum lies 20 below the bound would underflow).  Pass A (every score read
    // out of TMEM a second time at 64 B/clk -- the kernel's bound) disappears; the row sums and the statistics handed to
    // attn_round2 (m = max_logit, l) stay exact in fp32.  fp16 operands keep the exact two-pass statistics: a BF16 P
    // against an fp16 V in one tcgen05.mma (mixed a/b formats) is an illegal instruction on sm_100a (tried).
    const bool single = BF16 && a.max_logit > 0.f;
    const int GA = single ? 0 : (ci.n_clip + 127) / 128;       // key tiles of pass A
    const int GB = (ci.n_clip + 63) / 64;         // key tiles of pass B
    const bool need_reg = a.need_reg != 0;

    // softmax-thread state
    const int row = threadIdx.x & 127;
    const int quarter = (threadIdx.x >> 7) & 3;  // softmax warps 4q .. 4q+3 own column quarter q of every tile
    const bool is_sm = warp < 16;
    const int q = ci.q0 + row;
    const bool q_ok = is_sm && q < ci.n_loc;
    const bool self_attn = lay.self_attn != 0;
    int lo = 0, hi = 0;                            // own frame's key range (clip-local); empty for padding rows
    if (q_ok && !self_attn) {
        const int qf = a.row_frame[ci.s0 + q];
        lo = lay.row_off[b * lay.F + qf] - ci.s0;
        hi = lay.row_off[b * lay.F + qf + 1] - ci.s0;
    }
    const int n_glob0 = self_attn ? 0 : ci.n_loc;  // keys >= n_glob0 are visible to every query
    const uint32_t lane_base = tmem + ((uint32_t)((warp & 3) * 32) << 16);
    float mxc[4], mxr[4];

    // ======================================= pass A: row maxima =======================================
    const int HA = single ? 0 : 4;                 // heads visited by pass A
    if (warp == 16) {
        if (lane == 0) {
            uint32_t it = 0;
            for (int h = 0; h < HA; ++h) {
                const int qb = h & 1, uq = h >> 1;
                PV_WAIT(&bars.q_empty[qb], (uq & 1) ^ 1, 300);
                mbar_expect_tx(&bars.q_full[qb], 32768);
                tma_load_2d(sQ + qb * 32768, &tm.qc, &bars.q_full[qb], h * 64, ci.s0 + ci.q0);
                tma_load_2d(sQ + qb * 32768 + 16384, &tm.qr, &bars.q_full[qb], h * 64, ci.s0 + ci.q0);
                for (int g = 0; g < GA; ++g, ++it) {
                    const int st = it % kPvStages;
                    PV_WAIT(&bars.k_empty[st], ((it / kPvStages) & 1) ^ 1, 301);
                    mbar_expect_tx(&bars.k_full[st], 32768);
                    tma_load_2d(sKV + st * 32768, &tm.kc, &bars.k_full[st], h * 64, ci.s0 + g * 128);
                    tma_load_2d(sKV + st * 32768 + 16384, &tm.kr, &bars.k_full[st], h * 64, ci.s0 + g * 128);
                }
            }
        }
    } else if (warp == 17) {
        {   // the whole warp walks the loop (warp-uniform operands stay in uniform registers); one elected lane issues
            const uint32_t idesc128 = make_idesc_f16(BF16, 128, 128);
            uint32_t it = 0;
            for (int h = 0; h < HA; ++h) {
                const int qb = h & 1, uq = h >> 1;
                PV_WAIT(&bars.q_full[qb], uq & 1, 310);
                const uint64_t dqc = make_smem_desc_sw128(smem_u32(sQ + qb * 32768));
                const uint64_t dqr = make_smem_desc_sw128(smem_u32(sQ + qb * 32768 + 16384));
                for (int g = 0; g < GA; ++g, ++it) {
                    const int st = it % kPvStages, sb = it & 1;
                    PV_WAIT(&bars.k_full[st], (it / kPvStages) & 1, 311);
                    PV_WAIT(&bars.s_empty[sb], ((it >> 1) & 1) ^ 1, 312);
                    tc_fence_after();
                    const uint64_t dkc = make_smem_desc_sw128(smem_u32(sKV + st * 32768));
                    const uint64_t dkr = make_smem_desc_sw128(smem_u32(sKV + st * 32768 + 16384));
                    if (elect_one()) {
#pragma unroll
                        for (int k = 0; k < 4; ++k) umma_f16(tmem + sb * 256, dqc + 2 * k, dkc + 2 * k, idesc128, k ? 1u : 0u);
#pragma unroll
                        for (int k = 0; k < 4; ++k) umma_f16(tmem + sb * 256 + 128, dqr + 2 * k, dkr + 2 * k, idesc128, k ? 1u : 0u);
                        umma_commit(&bars.k_empty[st]);
                        umma_commit(&bars.s_full[sb]);
                    }
                    __syncwarp();
                }
                if (elect_one()) umma_commit(&bars.q_empty[qb]);
                __syncwarp();
            }
        }
    } else if (is_sm) {
        uint32_t it = 0;
        for (int h = 0; h < HA; ++h) {
            float mc = -INFINITY, mr = -INFINITY;
            for (int g = 0; g < GA; ++g, ++it) {
                const int sb = it & 1, kbase = g * 128;
                PV_WAIT(&bars.s_full[sb], (it >> 1) & 1, 320);
                tc_fence_after();
                const bool all_vis = kbase >= n_glob0 && kbase + 128 <= ci.n_clip;
                {
                    const int c0 = quarter * 32;
                    uint32_t rc[32], rr[32];
                    tmem_ld_32x32(lane_base + sb * 256 + c0, rc);
                    tmem_ld_32x32(lane_base + sb * 256 + 128 + c0, rr);
                    tmem_ld_wait();
                    float m0 = -INFINITY, m1 = -INFINITY, m2 = -INFINITY, m3 = -INFINITY;
                    if (all_vis) {
#pragma unroll
                        for (int j = 0; j < 32; j += 2) {
                            m0 = fmaxf(m0, __uint_as_float(rc[j])); m1 = fmaxf(m1, __uint_as_float(rc[j + 1]));
                            m2 = fmaxf(m2, __uint_as_float(rr[j])); m3 = fmaxf(m3, __uint_as_float(rr[j + 1]));
                        }
                    } else {
#pragma unroll
                        for (int j = 0; j < 32; ++j) {
                            const int k = kbase + c0 + j;
                            const bool ok = k < ci.n_clip && (k >= n_glob0 || (k >= lo && k < hi));
                            if (ok) { m0 = fmaxf(m0, __uint_as_float(rc[j])); m2 = fmaxf(m2, __uint_as_float(rr[j])); }
                        }
                    }
                    mc = fmaxf(mc, fmaxf(m0, m1)); mr = fmaxf(mr, fmaxf(m2, m3));
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&bars.s_empty[sb]);
            }
            reinterpret_cast<float*>(sP)[(quarter * 128 + row) * 8 + h] = mc;      // sP is idle during pass A
            reinterpret_cast<float*>(sP)[(quarter * 128 + row) * 8 + 4 + h] = mr;
        }
    }
    __syncthreads();      // every pass-A score tile has been consumed: TMEM is re-partitioned for pass B
#ifdef TSCD_R2_PROF
    if (blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0) atomicAdd(&g_pv_wait[62], (unsigned long long)(clock64() - tk0));
#endif
    if (is_sm) {
#pragma unroll
        for (int h = 0; h < 4; ++h) {
            const float* x0 = reinterpret_cast<const float*>(sP) + row * 8;
            mxc[h] = fmaxf(fmaxf(x0[h], x0[1024 + h]), fmaxf(x0[2048 + h], x0[3072 + h]));
            mxr[h] = fmaxf(fmaxf(x0[4 + h], x0[1024 + 4 + h]), fmaxf(x0[2048 + 4 + h], x0[3072 + 4 + h]));
            if (single) { mxc[h] = a.max_logit; mxr[h] = a.max_logit; }
        }
        softmax_bar_sync();  // every quarter has read the maxima before sP is written again
    }

    // ============================== pass B: exp / row sums / P @ V ================================
    const uint32_t itA = 4u * (uint32_t)GA;       // barrier use counters continue across the passes
    if (warp == 16) {
        if (lane == 0) {
            uint32_t it = itA;
            for (int h = 0; h < 4; ++h) {
                const int qb = h & 1, uq = (single ? 0 : 2) + (h >> 1);
                PV_WAIT(&bars.q_empty[qb], (uq & 1) ^ 1, 330);
                mbar_expect_tx(&bars.q_full[qb], 32768);
                tma_load_2d(sQ + qb * 32768, &tm.qc, &bars.q_full[qb], h * 64, ci.s0 + ci.q0);
                tma_load_2d(sQ + qb * 32768 + 16384, &tm.qr, &bars.q_full[qb], h * 64, ci.s0 + ci.q0);
                for (int g = 0; g < GB; ++g, ++it) {
                    const int st = it % kPvStages;
                    unsigned char* base = sKV + st * 32768;
                    PV_WAIT(&bars.k_empty[st], ((it / kPvStages) & 1) ^ 1, 331);
                    mbar_expect_tx(&bars.k_full[st], 16384);
                    tma_load_2d(base, &tm.k64c, &bars.k_full[st], h * 64, ci.s0 + g * 64);
                    tma_load_2d(base + 8192, &tm.k64r, &bars.k_full[st], h * 64, ci.s0 + g * 64);
                }
            }
        }
    } else if (warp == 19) {
        if (lane == 0) {        // value tiles: their own ring (second half of every stage), counted from 0 in pass B
            uint32_t iv = 0;
            for (int h = 0; h < 4; ++h)
                for (int g = 0; g < GB; ++g, ++iv) {
                    const int st = iv % kPvStages;
                    unsigned char* base = sKV + st * 32768 + 16384;
                    PV_WAIT(&bars.v_empty[st], ((iv / kPvStages) & 1) ^ 1, 332);
                    mbar_expect_tx(&bars.v_full[st], need_reg ? 16384 : 8192);
                    tma_load_2d(base, &tm.vtc, &bars.v_full[st], g * 64, b * 256 + h * 64);
                    if (need_reg) tma_load_2d(base + 8192, &tm.vtr, &bars.v_full[st], g * 64, b * 256 + h * 64);
                }
        }
    } else if (warp == 17) {
        {                       // scores of every tile (whole warp walks the loop, one elected lane issues: uniform operands)
            const uint32_t idesc64 = make_idesc_f16(BF16, 128, 64);
            uint32_t it = itA;          // key-tile counter (ring stage / score buffer of tile `it`)
            for (int h = 0; h < 4; ++h) {
                const int qb = h & 1, uq = (single ? 0 : 2) + (h >> 1);
                PV_WAIT(&bars.q_full[qb], uq & 1, 340);
                const uint64_t dqc = make_smem_desc_sw128(smem_u32(sQ + qb * 32768));
                const uint64_t dqr = make_smem_desc_sw128(smem_u32(sQ + qb * 32768 + 16384));
                for (int g = 0; g < GB; ++g, ++it) {
                    const int st = it % kPvStages, sb = it & 1;
                    PV_WAIT(&bars.k_full[st], (it / kPvStages) & 1, 341);
                    PV_WAIT(&bars.s_empty[sb], ((it >> 1) & 1) ^ 1, 342);
                    tc_fence_after();
                    const uint64_t dkc = make_smem_desc_sw128(smem_u32(sKV + st * 32768));
                    const uint64_t dkr = make_smem_desc_sw128(smem_u32(sKV + st * 32768 + 8192));
                    if (elect_one()) {
#pragma unroll
                        for (int k = 0; k < 4; ++k) umma_f16(tmem + sb * 128, dqc + 2 * k, dkc + 2 * k, idesc64, k ? 1u : 0u);
#pragma unroll
                        for (int k = 0; k < 4; ++k) umma_f16(tmem + sb * 128 + 64, dqr + 2 * k, dkr + 2 * k, idesc64, k ? 1u : 0u);
                        umma_commit(&bars.k_empty[st]);
                        umma_commit(&bars.s_full[sb]);
                    }
                    __syncwarp();
                }
                if (elect_one()) umma_commit(&bars.q_empty[qb]);
                __syncwarp();
            }
        }
    } else if (warp == 18) {
        {                       // P @ V of every tile
            const uint32_t idesc64 = make_idesc_f16(BF16, 128, 64);
            const uint32_t idesc128b = make_idesc_f16(BF16, 128, 128);
            uint32_t ip = 0;            // P@V counter (tile whose probabilities are consumed next)
            for (int h = 0; h < 4; ++h) {
                for (int g = 0; g < GB; ++g, ++ip) {
                    const int st = ip % kPvStages, pb = ip & 1;
                    PV_WAIT(&bars.v_full[st], (ip / kPvStages) & 1, 345);
                    PV_WAIT(&bars.p_full[pb], (ip >> 1) & 1, 343);
                    if (g == 0 && h > 0) PV_WAIT(&bars.o_empty, (h - 1) & 1, 344);   // previous head's O has been read
                    tc_fence_after();
                    const uint64_t dpc = make_smem_desc_sw128(smem_u32(sP + pb * 32768));
                    const uint64_t dpr = make_smem_desc_sw128(smem_u32(sP + pb * 32768 + 16384));
                    const uint64_t dvc = make_smem_desc_sw128(smem_u32(sKV + st * 32768 + 16384));
                    if (elect_one()) {
#pragma unroll
                        for (int k = 0; k < 4; ++k) {
                            const uint32_t acc = (g > 0 || k) ? 1u : 0u;
                            if (need_reg) {
                                // Vc^T and Vr^T tiles are adjacent in the stage: one N = 128 product per probability
                                // matrix (the A operand is read from shared memory once instead of twice)
                                umma_f16(tmem + 256, dpc + 2 * k, dvc + 2 * k, idesc128b, acc);   // O_cc | O_cr
                                umma_f16(tmem + 384, dpr + 2 * k, dvc + 2 * k, idesc128b, acc);   // O_rc | O_rr
                            } else {
                                umma_f16(tmem + 256, dpc + 2 * k, dvc + 2 * k, idesc64, acc);     // O_cc
                                umma_f16(tmem + 320, dpr + 2 * k, dvc + 2 * k, idesc64, acc);     // O_rc
                            }
                        }
                        umma_commit(&bars.v_empty[st]);
                        umma_commit(&bars.p_empty[pb]);
                    }
                    __syncwarp();
                }
                if (elect_one()) umma_commit(&bars.o_full);
                __syncwarp();
            }
        }
    } else if (is_sm) {
        uint32_t it = itA, ip = 0;
        float lsum_c[4], lsum_r[4];
        for (int h = 0; h < 4; ++h) {
            const float mc = mxc[h] * kLog2e, mr = mxr[h] * kLog2e;
            float lc = 0.f, lr = 0.f;
            for (int g = 0; g < GB; ++g, ++it, ++ip) {
                const int sb = it & 1, pb = ip & 1, kbase = g * 64;
                PV_WAIT(&bars.s_full[sb], (it >> 1) & 1, 350);
                PV_WAIT(&bars.p_empty[pb], ((ip >> 1) & 1) ^ 1, 351);
                tc_fence_after();
                unsigned char* sPc = sP + pb * 32768;
                unsigned char* sPr = sPc + 16384;
                const bool all_vis = kbase >= n_glob0 && kbase + 64 <= ci.n_clip;
                {
                    const int c0 = quarter * 16;
                    uint32_t rc[16], rr[16];
                    tmem_ld_32x16(lane_base + sb * 128 + c0, rc);
                    tmem_ld_32x16(lane_base + sb * 128 + 64 + c0, rr);
                    tmem_ld_wait();
                    float ec[16], er[16];
                    float l0 = 0.f, l1 = 0.f, l2 = 0.f, l3 = 0.f;
                    if (all_vis) {
#pragma unroll
                        for (int j = 0; j < 16; j += 2) {
                            ec[j] = ex2_approx(fmaf(__uint_as_float(rc[j]), kLog2e, -mc));
                            ec[j + 1] = ex2_approx(fmaf(__uint_as_float(rc[j + 1]), kLog2e, -mc));
                            er[j] = ex2_approx(fmaf(__uint_as_float(rr[j]), kLog2e, -mr));
                            er[j + 1] = ex2_approx(fmaf(__uint_as_float(rr[j + 1]), kLog2e, -mr));
                            l0 += ec[j]; l1 += ec[j + 1]; l2 += er[j]; l3 += er[j + 1];
                        }
                    } else {
#pragma unroll
                        for (int j = 0; j < 16; ++j) {
                            const int k = kbase + c0 + j;
                            const bool ok = k < ci.n_clip && (k >= n_glob0 || (k >= lo && k < hi));
                            ec[j] = ok ? ex2_approx(fmaf(__uint_as_float(rc[j]), kLog2e, -mc)) : 0.f;
                            er[j] = ok ? ex2_approx(fmaf(__uint_as_float(rr[j]), kLog2e, -mr)) : 0.f;
                            l0 += ec[j]; l2 += er[j];
                        }
                    }
                    lc += l0 + l1; lr += l2 + l3;
#pragma unroll
                    for (int cc = 0; cc < 2; ++cc) {
                        const uint32_t off = sw128_off(row, (c0 >> 3) + cc);
                        *reinterpret_cast<uint4*>(sPc + off) =
                            make_uint4(pack2<BF16>(ec[cc * 8], ec[cc * 8 + 1]), pack2<BF16>(ec[cc * 8 + 2], ec[cc * 8 + 3]),
                                       pack2<BF16>(ec[cc * 8 + 4], ec[cc * 8 + 5]), pack2<BF16>(ec[cc * 8 + 6], ec[cc * 8 + 7]));
                        *reinterpret_cast<uint4*>(sPr + off) =
                            make_uint4(pack2<BF16>(er[cc * 8], er[cc * 8 + 1]), pack2<BF16>(er[cc * 8 + 2], er[cc * 8 + 3]),
                                       pack2<BF16>(er[cc * 8 + 4], er[cc * 8 + 5]), pack2<BF16>(er[cc * 8 + 6], er[cc * 8 + 7]));
                    }
                }
                fence_proxy_async();
                tc_fence_before();
                __syncwarp();
                if (lane == 0) { mbar_arrive(&bars.s_empty[sb]); mbar_arrive(&bars.p_full[pb]); }
            }
            // the row's four column quarters exchange their partial sums
            bars.xch[quarter][row] = lc;
            softmax_bar_sync();
            lc = (bars.xch[0][row] + bars.xch[1][row]) + (bars.xch[2][row] + bars.xch[3][row]);
            softmax_bar_sync();
            bars.xch[quarter][row] = lr;
            softmax_bar_sync();
            lr = (bars.xch[0][row] + bars.xch[1][row]) + (bars.xch[2][row] + bars.xch[3][row]);
            softmax_bar_sync();
            lsum_c[h] = lc; lsum_r[h] = lr;
            // head epilogue: x = (O_c / l_c + O_r / l_r) / 2; each quarter drains 16 of the head's 64 output columns
            PV_WAIT(&bars.o_full, h & 1, 352);
            tc_fence_after();
            const float ic = 0.5f / lc, ir = 0.5f / lr;
            for (int br = 0; br < (need_reg ? 2 : 1); ++br) {
                uint16_t* dst = reinterpret_cast<uint16_t*>(br == 0 ? a.x_cls : a.x_reg);
                const int c0 = quarter * 16;
                uint32_t oc[16], orr[16];
                // TMEM: need_reg  O_cc 256 | O_cr 320 | O_rc 384 | O_rr 448;   else  O_cc 256 | O_rc 320
                tmem_ld_32x16(lane_base + (need_reg ? 256 + br * 64 : 256) + c0, oc);
                tmem_ld_32x16(lane_base + (need_reg ? 384 + br * 64 : 320) + c0, orr);
                tmem_ld_wait();
                if (q_ok) {
                    uint32_t pk[8];
#pragma unroll
                    for (int j = 0; j < 8; ++j)
                        pk[j] = pack2<BF16>(__uint_as_float(oc[2 * j]) * ic + __uint_as_float(orr[2 * j]) * ir,
                                            __uint_as_float(oc[2 * j + 1]) * ic + __uint_as_float(orr[2 * j + 1]) * ir);
                    uint4* o = reinterpret_cast<uint4*>(dst + (int64_t)(ci.lbase + q) * a.ld_x + h * 64 + c0);
#pragma unroll
                    for (int j = 0; j < 2; ++j) o[j] = make_uint4(pk[4 * j], pk[4 * j + 1], pk[4 * j + 2], pk[4 * j + 3]);
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&bars.o_empty);
        }
        if (q_ok && quarter == 0) {
            float4* st = reinterpret_cast<float4*>(a.stats + (int64_t)(ci.lbase + q) * 16);
            st[0] = make_float4(mxc[0], mxc[1], mxc[2], mxc[3]);
            st[1] = make_float4(mxr[0], mxr[1], mxr[2], mxr[3]);
            st[2] = make_float4(lsum_c[0], lsum_c[1], lsum_c[2], lsum_c[3]);
            st[3] = make_float4(lsum_r[0], lsum_r[1], lsum_r[2], lsum_r[3]);
        }
    }
#ifdef TSCD_R2_PROF
    if (blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0) atomicAdd(&g_pv_wait[63], (unsigned long long)(clock64() - tk0));
#endif
    tc_fence_before();
    __syncthreads();
    if (warp == 17) {
        tc_fence_after();
        tmem_dealloc<512>(tmem);
    }
}

// -------------------------------------------------------------------------------------------------------
// attn_round2: masks from head-mean raw-v cosine, exp(head-mean attention), renormalise, @ V
// -------------------------------------------------------------------------------------------------------
struct R2Tmaps {
    CUtensorMap q128c, q128r, k64c, k64r, vn128c, vn128r, vn64c, vn64r, vt;
};

// Warp-specialised like attn_pv.  The kernel is bound by the latency of L2 -> shared-memory operand traffic and of the
// single-thread UMMA issue, so
//  * the A operands that every key tile re-uses stay RESIDENT in shared memory for the whole CTA (loaded once):
//      cls launch (no w_in):  the 8 query head slices  Q[h][branch]  [128 x 64]   (8 x 16K = 128K)
//      obj launch (w_in):     the 4 raw-v query atoms of the reg branch [128 x 64] (4 x 16K)
//  * the rest streams through TWO independent pipelines, each one TMA warp -> ring of 8 KB slots -> one MMA warp
//    (single producer, single consumer per ring: every waiter sees every phase of its barriers):
//      S pipeline (cls launch only, 4 slots):  the 8 score units of every tile; item = K head slice [64 x 64], 1 slot
//      X pipeline (6 / 16 slots):  raw(0), then per tile kt:  W(kt-1) @ V^T halves | raw-v atoms of tile kt+1
//          raw atom  = Vn(query) [128 x 64] 16K + Vn(keys) [64 x 64] 8K           3 slots  (cls launch)
//                      Vn(keys) only, the query atom is resident                   1 slot   (obj launch)
//          V^T half  = [128 dims x 64 keys]                                       2 slots
//    An item takes contiguous slots; one that would straddle the end of its ring restarts at the ring's first slot.
// TMEM: U 256 | R_cls 64 | R_reg 64 | two score units of 64 columns (obj launch: the two R regions double-buffer the
// reg-branch similarity).  The 16 softmax warps read the raw-v similarities of a tile first (mask bits -> registers),
// then the 8 score units (head-sum of the normalised attention, exact statistics from attn_pv), then write the
// round-2 weights as the A operand of W @ V^T.
constexpr int kR2Threads = 640;      // 16 softmax warps + (TMA, MMA) of the S pipeline + (TMA, MMA) of the X pipeline
constexpr int kR2MaxSlots = 16;
constexpr int kR2SlotBytes = 8192;
constexpr int kR2SmemBytes = 229376;      // resident operands + rings + weight buffers (mode-dependent split)

struct R2Bars {
    uint64_t full[kR2MaxSlots], empty[kR2MaxSlots];
    uint64_t res_full;
    uint64_t r_full[2], r_empty[2];
    uint64_t s_full[2], s_empty[2];
    uint64_t w_full[2], w_empty[2];
    uint64_t u_full;
    uint32_t tmem_base;
    float xch[4][128];
};

static_assert(kR2SmemBytes + sizeof(R2Bars) <= 232448, "attn_round2: over the 227 KB shared-memory window");

// One side of a ring: slot cursor + per-slot barrier parities (the producer tracks `empty`, the consumer `full`).
struct R2Ring {
    int first, count;        // slots [first, first + count)
    int pos;
    uint32_t ph;
    __device__ __forceinline__ R2Ring(int f, int c) : first(f), count(c), pos(f), ph(0) {}
    // next(n): first slot of the next item of n slots.  parity(s): this side's phase bit of slot s, then flipped -- the
    // producer calls it for every slot of an item (all `empty` barriers cycle), the consumer for the first only (`full`).
    __device__ __forceinline__ int next(int n) {
        if (pos + n > first + count) pos = first;
        const int s = pos;
        pos += n;
        return s;
    }
    __device__ __forceinline__ uint32_t parity(int s) {
        const uint32_t p = (ph >> s) & 1u;
        ph ^= 1u << s;
        return p;
    }
};

// X pipeline order.  f(kind, kt, i): kind 1 = raw atom i of tile kt, 2 = V^T half i of tile kt
template <class F>
__device__ __forceinline__ void r2_x_schedule(int KT, int atom0, int atom1, F&& f) {
    for (int x = atom0; x < atom1; ++x) f(1, 0, x);
    for (int kt = 0; kt < KT; ++kt) {
        if (kt >= 1) { f(2, kt - 1, 0); f(2, kt - 1, 1); }
        if (kt + 1 < KT)
            for (int x = atom0; x < atom1; ++x) f(1, kt + 1, x);
    }
    f(2, KT - 1, 0); f(2, KT - 1, 1);
}

template <bool BF16>
__global__ void __launch_bounds__(kR2Threads, 1) attn_round2_kernel(const __grid_constant__ R2Tmaps tm,
                                                                     const tscd_attn_round2_args a) {
    using namespace tc;
    const tscd_attn_layout& lay = a.lay;
    const int b = blockIdx.y;
    const ClipInfo ci = clip_info(lay, b, blockIdx.x);
    if (ci.q0 >= ci.n_loc) return;
#ifdef TSCD_R2_PROF
    const long long tk0 = clock64();
#endif

    extern __shared__ __align__(1024) unsigned char smem_raw[];
    unsigned char* smem = smem_raw;                       // no static shared memory: the window starts 1024-byte aligned
    if ((smem_u32(smem) & 1023u) != 0) __trap();
    const bool use_obj = a.use_obj_mask != 0;
    // w_in: the cls-output launch of the same module already stored  sim_mask * exp(mean attention)  (its weights): this
    // launch only needs the reg-branch raw-v similarity (obj mask) -- no score units, no exponentials
    const bool reuse = a.w_in != nullptr;
    const int n_atoms = use_obj ? 8 : 4;
    const int n_s = reuse ? 0 : 4, n_x = reuse ? 16 : 6;          // ring slots of the S / X pipelines
    const int atom0 = reuse ? 4 : 0, atom1 = reuse ? 8 : n_atoms;
    unsigned char* sRes = smem;                                   // resident A operands: 4 or 8 x 16K
    unsigned char* sRing = smem + (reuse ? 65536 : 131072);       // 16 or 10 x 8K
    unsigned char* sW = sRing + (n_s + n_x) * kR2SlotBytes;       // 2 or 1 x 16K weights [128 x 64 keys]
    R2Bars& bars = *reinterpret_cast<R2Bars*>(smem + kR2SmemBytes);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 512) {
        tma_prefetch_desc(&tm.q128c); tma_prefetch_desc(&tm.q128r); tma_prefetch_desc(&tm.k64c); tma_prefetch_desc(&tm.k64r);
        tma_prefetch_desc(&tm.vn128c); tma_prefetch_desc(&tm.vn128r); tma_prefetch_desc(&tm.vn64c); tma_prefetch_desc(&tm.vn64r);
        tma_prefetch_desc(&tm.vt);
        for (int i = 0; i < kR2MaxSlots; ++i) { mbar_init(&bars.full[i], 1); mbar_init(&bars.empty[i], 1); }
        mbar_init(&bars.res_full, 1);
        for (int i = 0; i < 2; ++i) {
            mbar_init(&bars.r_full[i], 1); mbar_init(&bars.r_empty[i], 16);
            mbar_init(&bars.s_full[i], 1); mbar_init(&bars.s_empty[i], 16);
            mbar_init(&bars.w_full[i], 16); mbar_init(&bars.w_empty[i], 1);
        }
        mbar_init(&bars.u_full, 1);
        fence_barrier_init();
    }
    if (warp == 17) tmem_alloc<512>(&bars.tmem_base);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = bars.tmem_base;
    const int KT = (ci.n_clip + 63) / 64;
    if (warp == 16) {
        // ------------------------------------------------ S pipeline: TMA producer ------------------------------------------------
        if (lane == 0) {
            // resident A operands
            if (reuse) {
                mbar_expect_tx(&bars.res_full, 4 * 16384);
                for (int at = 0; at < 4; ++at) tma_load_2d(sRes + at * 16384, &tm.vn128r, &bars.res_full, at * 64, ci.s0 + ci.q0);
            } else {
                mbar_expect_tx(&bars.res_full, 8 * 16384);
                for (int u = 0; u < 8; ++u)
                    tma_load_2d(sRes + u * 16384, (u & 1) == 0 ? &tm.q128c : &tm.q128r, &bars.res_full, (u >> 1) * 64, ci.s0 + ci.q0);
                R2Ring ring(0, n_s);
                for (int kt = 0; kt < KT; ++kt)
                    for (int u = 0; u < 8; ++u) {
                        const int sl = ring.next(1);
                        R2_WAIT(&bars.empty[sl], ring.parity(sl) ^ 1u, 400);
                        mbar_expect_tx(&bars.full[sl], 8192);
                        tma_load_2d(sRing + sl * kR2SlotBytes, (u & 1) == 0 ? &tm.k64c : &tm.k64r, &bars.full[sl], (u >> 1) * 64, ci.s0 + kt * 64);
                    }
            }
        }
    } else if (warp == 18) {
        // ------------------------------------------------ X pipeline: TMA producer ------------------------------------------------
        if (lane == 0) {
            R2Ring ring(n_s, n_x);
            r2_x_schedule(KT, atom0, atom1, [&](int kind, int kt, int i) {
                const int n = kind == 2 ? 2 : (reuse ? 1 : 3);
                const int sl = ring.next(n);
                for (int j = 0; j < n; ++j) R2_WAIT(&bars.empty[sl + j], ring.parity(sl + j) ^ 1u, 401);
                uint64_t* fb = &bars.full[sl];
                unsigned char* d = sRing + sl * kR2SlotBytes;
                mbar_expect_tx(fb, n * 8192);
                if (kind == 1) {
                    const int br = i >> 2, at = i & 3;
                    if (reuse) {
                        tma_load_2d(d, &tm.vn64r, fb, at * 64, ci.s0 + kt * 64);
                    } else {
                        tma_load_2d(d, br == 0 ? &tm.vn128c : &tm.vn128r, fb, at * 64, ci.s0 + ci.q0);
                        tma_load_2d(d + 16384, br == 0 ? &tm.vn64c : &tm.vn64r, fb, at * 64, ci.s0 + kt * 64);
                    }
                } else {
                    tma_load_2d(d, &tm.vt, fb, kt * 64, b * 256 + i * 128);
                    tma_load_2d(d + 8192, &tm.vt, fb, kt * 64, b * 256 + i * 128 + 64);
                }
            });
        }
    } else if (warp == 17) {
        // ------------------------------------------------ S pipeline: MMA issuer (score units) ------------------------------------------------
        if (!reuse) {             // whole warp walks the loop (uniform operands), one elected lane issues
            const uint32_t idesc64 = make_idesc_f16(BF16, 128, 64);
            R2Ring ring(0, n_s);
            R2_WAIT(&bars.res_full, 0, 414);
            tc_fence_after();
            uint32_t iu = 0;
            for (int kt = 0; kt < KT; ++kt)
                for (int u = 0; u < 8; ++u, ++iu) {          // score unit u = 2 * head + branch
                    const int su = iu & 1;
                    R2_WAIT(&bars.s_empty[su], ((iu >> 1) & 1) ^ 1, 412);
                    const int sl = ring.next(1);
                    R2_WAIT(&bars.full[sl], ring.parity(sl), 410);
                    tc_fence_after();
                    const uint64_t dq = make_smem_desc_sw128(smem_u32(sRes + u * 16384));
                    const uint64_t dk = make_smem_desc_sw128(smem_u32(sRing + sl * kR2SlotBytes));
                    if (elect_one()) {
#pragma unroll
                        for (int k = 0; k < 4; ++k) umma_f16(tmem + 384 + su * 64, dq + 2 * k, dk + 2 * k, idesc64, k ? 1u : 0u);
                        umma_commit(&bars.empty[sl]);
                        umma_commit(&bars.s_full[su]);
                    }
                    __syncwarp();
                }
        }
    } else if (warp == 19) {
        // ------------------------------------------------ X pipeline: MMA issuer (raw-v similarity, W @ V^T) ------------------------------------------------
        {
            const uint32_t idesc64 = make_idesc_f16(BF16, 128, 64);
            const uint32_t idesc128 = make_idesc_f16(BF16, 128, 128);
            R2Ring ring(n_s, n_x);
            if (reuse) {
                R2_WAIT(&bars.res_full, 0, 414);
                tc_fence_after();
            }
            r2_x_schedule(KT, atom0, atom1, [&](int kind, int kt, int i) {
                const int n = kind == 2 ? 2 : (reuse ? 1 : 3);
                if (kind == 1) {                 // raw-v similarity atom (K = 256 as four 64-dim atoms per branch)
                    const int br = i >> 2, at = i & 3;
                    const int rb = reuse ? (kt & 1) : 0, use = reuse ? (kt >> 1) : kt;
                    if (i == atom0) {
                        R2_WAIT(&bars.r_empty[rb], (use & 1) ^ 1, 411);
                        tc_fence_after();
                    }
                    const int sl = ring.next(n);
                    R2_WAIT(&bars.full[sl], ring.parity(sl), 415);
                    tc_fence_after();
                    unsigned char* d = sRing + sl * kR2SlotBytes;
                    const uint64_t da = make_smem_desc_sw128(smem_u32(reuse ? sRes + at * 16384 : d));
                    const uint64_t db = make_smem_desc_sw128(smem_u32(reuse ? d : d + 16384));
                    const uint32_t col = tmem + 256 + (reuse ? rb : br) * 64;
                    if (elect_one()) {
#pragma unroll
                        for (int k = 0; k < 4; ++k) umma_f16(col, da + 2 * k, db + 2 * k, idesc64, (at | k) ? 1u : 0u);
                        for (int j = 0; j < n; ++j) umma_commit(&bars.empty[sl + j]);
                        if (i == atom1 - 1) umma_commit(&bars.r_full[rb]);
                    }
                    __syncwarp();
                } else {                         // U += W(kt) @ V^T(kt), 128-dim half i
                    const int wb = reuse ? (kt & 1) : 0, use = reuse ? (kt >> 1) : kt;
                    if (i == 0) {
                        R2_WAIT(&bars.w_full[wb], use & 1, 413);
                        tc_fence_after();
                    }
                    const int sl = ring.next(2);
                    R2_WAIT(&bars.full[sl], ring.parity(sl), 415);
                    tc_fence_after();
                    const uint64_t dw = make_smem_desc_sw128(smem_u32(sW + wb * 16384));
                    const uint64_t dv = make_smem_desc_sw128(smem_u32(sRing + sl * kR2SlotBytes));
                    if (elect_one()) {
#pragma unroll
                        for (int k = 0; k < 4; ++k) umma_f16(tmem + i * 128, dw + 2 * k, dv + 2 * k, idesc128, (kt | k) ? 1u : 0u);
                        umma_commit(&bars.empty[sl]);
                        umma_commit(&bars.empty[sl + 1]);
                        if (i == 1) umma_commit(&bars.w_empty[wb]);
                    }
                    __syncwarp();
                }
            });
            if (elect_one()) umma_commit(&bars.u_full);
            __syncwarp();
        }
    } else {
        // ------------------------------------------------ softmax / weight warps ------------------------------------------------
        // 16 warps: warp w owns TMEM lanes 32 * (w % 4) .. +31 (query rows) and column quarter w / 4 of every 64-key unit.
        // (Four warps per scheduler: the per-unit chain  TMEM load -> ex2 -> accumulate  is latency-bound with two.)
        constexpr int NC = 16;
        const int row = threadIdx.x & 127;
        const int quarter = (threadIdx.x >> 7) & 3;
        const int q = ci.q0 + row;
        const bool q_ok = q < ci.n_loc;
        const bool self_attn = lay.self_attn != 0;
        int lo = 0, hi = 0;
        if (q_ok && !self_attn) {
            const int qf = a.row_frame[ci.s0 + q];
            lo = lay.row_off[b * lay.F + qf] - ci.s0;
            hi = lay.row_off[b * lay.F + qf + 1] - ci.s0;
        }
        const int n_glob0 = self_attn ? 0 : ci.n_loc;
        const uint32_t lane_base = tmem + ((uint32_t)((warp & 3) * 32) << 16);
        float mcl[8], il[8];       // per unit u = 2*h + br: row max * log2e, 0.5 / row sum
#pragma unroll
        for (int u = 0; u < 8; ++u) { mcl[u] = 0.f; il[u] = 0.f; }
        if (q_ok && !reuse) {
            const float* st = a.stats + (int64_t)(ci.lbase + q) * 16;
#pragma unroll
            for (int h = 0; h < 4; ++h) {
                mcl[2 * h] = st[h] * kLog2e; mcl[2 * h + 1] = st[4 + h] * kLog2e;
                il[2 * h] = 0.5f / st[8 + h]; il[2 * h + 1] = 0.5f / st[12 + h];
            }
        }
        const int c0 = quarter * NC;
        // bits j of the NC columns starting at key `base` that fall into [k0, k1)
        auto range_bits = [](int k0, int k1, int base) -> uint32_t {
            const int x0 = min(max(k0 - base, 0), NC), x1 = min(max(k1 - base, 0), NC);
            return x1 > x0 ? (((1u << x1) - 1u) & ~((1u << x0) - 1u)) : 0u;
        };
        float den = 0.f;
        uint32_t iu = 0;
        for (int kt = 0; kt < KT; ++kt) {
            const int kbase = kt * 64;
            // ---- mask bits of this tile: visibility, head-mean raw-v cosine thresholds ----
            uint32_t bits = range_bits(n_glob0, ci.n_clip, kbase + c0) | range_bits(lo, min(hi, ci.n_clip), kbase + c0);
            const int rb = reuse ? (kt & 1) : 0, ruse = reuse ? (kt >> 1) : kt;
            R2_WAIT(&bars.r_full[rb], ruse & 1, 420);
            tc_fence_after();
            {
                uint32_t rc[NC], rr[NC];
                if (!reuse) tmem_ld_32x16(lane_base + 256 + c0, rc);
                if (use_obj) tmem_ld_32x16(lane_base + (reuse ? 256 + rb * 64 : 320) + c0, rr);
                tmem_ld_wait();
                uint32_t pass = 0;
#pragma unroll
                for (int j = 0; j < NC; ++j) {
                    bool ok = true;
                    if (!reuse) ok = __uint_as_float(rc[j]) * 0.25f > a.sim_thresh;                    // (already folded into w_in)
                    if (use_obj) ok = ok && (__uint_as_float(rr[j]) * 0.25f > a.conf_sim_thresh);
                    pass |= ok ? (1u << j) : 0u;
                }
                bits &= pass;
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&bars.r_empty[rb]);
            float w[NC];
            if (!reuse) {
                // ---- head-sum of the normalised attention over the 8 (head, branch) score units ----
                float as[NC];
#pragma unroll
                for (int j = 0; j < NC; ++j) as[j] = 0.f;
#pragma unroll
                for (int u = 0; u < 8; ++u, ++iu) {
                    const int su = iu & 1;
                    R2_WAIT(&bars.s_full[su], (iu >> 1) & 1, 421);
                    tc_fence_after();
                    uint32_t r[NC];
                    tmem_ld_32x16(lane_base + 384 + su * 64 + c0, r);
                    tmem_ld_wait();
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&bars.s_empty[su]);      // the unit is in registers: release it before the math
                    const float m = mcl[u], sc = il[u];
#pragma unroll
                    for (int j = 0; j < NC; ++j) as[j] = fmaf(ex2_approx(fmaf(__uint_as_float(r[j]), kLog2e, -m)), sc, as[j]);
                }
                // ---- weights: mask * exp(mean attention) ----
#pragma unroll
                for (int j = 0; j < NC; ++j) w[j] = ((bits >> j) & 1u) ? ex2_approx(as[j] * (0.25f * kLog2e)) : 0.f;
            } else {
                // ---- weights of the cls launch (16-bit, sim mask applied) gated by the obj mask ----
                const uint4* src = reinterpret_cast<const uint4*>(reinterpret_cast<const uint16_t*>(a.w_in) +
                                                                  (int64_t)(ci.lbase + min(q, ci.n_loc - 1)) * lay.nk_pitch + kbase + c0);
#pragma unroll
                for (int cc = 0; cc < NC / 8; ++cc) {
                    const uint4 raw = __ldg(src + cc);
                    const uint32_t wd[4] = {raw.x, raw.y, raw.z, raw.w};
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        float lo16, hi16;
                        if (BF16) {
                            lo16 = __uint_as_float(wd[e] << 16); hi16 = __uint_as_float(wd[e] & 0xffff0000u);
                        } else {
                            const __half2 h2 = *reinterpret_cast<const __half2*>(&wd[e]);
                            lo16 = __low2float(h2); hi16 = __high2float(h2);
                        }
                        const int j = cc * 8 + e * 2;
                        w[j] = ((bits >> j) & 1u) ? lo16 : 0.f;
                        w[j + 1] = ((bits >> (j + 1)) & 1u) ? hi16 : 0.f;
                    }
                }
            }
            float d0 = 0.f, d1 = 0.f;
#pragma unroll
            for (int j = 0; j < NC; j += 2) { d0 += w[j]; d1 += w[j + 1]; }
            den += d0 + d1;
            const int wb = reuse ? (kt & 1) : 0;
            R2_WAIT(&bars.w_empty[wb], (ruse & 1) ^ 1, 422);
            unsigned char* sWb = sW + wb * 16384;
#pragma unroll
            for (int cc = 0; cc < NC / 8; ++cc) {
                const uint4 pk = make_uint4(pack2<BF16>(w[cc * 8], w[cc * 8 + 1]), pack2<BF16>(w[cc * 8 + 2], w[cc * 8 + 3]),
                                            pack2<BF16>(w[cc * 8 + 4], w[cc * 8 + 5]), pack2<BF16>(w[cc * 8 + 6], w[cc * 8 + 7]));
                *reinterpret_cast<uint4*>(sWb + sw128_off(row, (c0 >> 3) + cc)) = pk;
                if (a.w_out && q_ok)     // keep the weights for the obj launch of the same module
                    *reinterpret_cast<uint4*>(reinterpret_cast<uint16_t*>(a.w_out) + (int64_t)(ci.lbase + q) * lay.nk_pitch + kbase + c0 + cc * 8) = pk;
            }
            fence_proxy_async();
            __syncwarp();
            if (lane == 0) mbar_arrive(&bars.w_full[wb]);
        }
        // ---- U / den: each column quarter of a row drains 64 of the 256 output columns ----
        bars.xch[quarter][row] = den;
        asm volatile("bar.sync 1, 512;\n" ::: "memory");
        den = (bars.xch[0][row] + bars.xch[1][row]) + (bars.xch[2][row] + bars.xch[3][row]);
        R2_WAIT(&bars.u_full, 0, 423);
        tc_fence_after();
        const float inv = 1.f / den;
        uint16_t* dst = reinterpret_cast<uint16_t*>(a.out);
#pragma unroll 1
        for (int cb = quarter * 64; cb < quarter * 64 + 64; cb += 32) {
            uint32_t u[32];
            tmem_ld_32x32(lane_base + cb, u);
            tmem_ld_wait();
            if (q_ok) {
                uint32_t pk[16];
#pragma unroll
                for (int j = 0; j < 16; ++j) pk[j] = pack2<BF16>(__uint_as_float(u[2 * j]) * inv, __uint_as_float(u[2 * j + 1]) * inv);
                uint4* o = reinterpret_cast<uint4*>(dst + (int64_t)(ci.lbase + q) * a.ld_out + cb);
#pragma unroll
                for (int j = 0; j < 4; ++j) o[j] = make_uint4(pk[4 * j], pk[4 * j + 1], pk[4 * j + 2], pk[4 * j + 3]);
            }
        }
    }
#ifdef TSCD_R2_PROF
    if (blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0) atomicAdd(&g_r2_wait[63], (unsigned long long)(clock64() - tk0));
#endif
    tc_fence_before();
    __syncthreads();
    if (warp == 17) {
        tc_fence_after();
        tmem_dealloc<512>(tmem);
    }
}

static bool layout_ok(const tscd_attn_layout& l) {
    return l.B > 0 && l.F > 0 && l.L > 0 && l.L <= l.F && l.row_cap > 0 && l.nk_pitch > 0 && (l.nk_pitch % 128) == 0 &&
           l.row_off && l.lrow_off && (l.dtype == TSCD_F16 || l.dtype == TSCD_BF16);
}

}  // namespace tscd

extern "C" int tscd_attn_prep(const tscd_attn_prep_args* a, void* stream) {
    using namespace tscd;
    if (!a || !layout_ok(a->lay)) return TSCD_ERR_INVALID_ARG;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    dim3 grid(a->lay.nk_pitch / 64, a->lay.B);
    const size_t smem = 2 * 64 * kPrepRowPitch * 2;
    if (a->lay.dtype == TSCD_F16) {
        if (cudaFuncSetAttribute(attn_prep_kernel<__half>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) return TSCD_ERR_CUDA;
        attn_prep_kernel<__half><<<grid, kPrepThreads, smem, st>>>(*a);
    } else {
        if (cudaFuncSetAttribute(attn_prep_kernel<__nv_bfloat16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) return TSCD_ERR_CUDA;
        attn_prep_kernel<__nv_bfloat16><<<grid, kPrepThreads, smem, st>>>(*a);
    }
    TSCD_CUDA_CHECK_LAUNCH();
    return TSCD_OK;
}

extern "C" int tscd_transpose_clip(const tscd_transpose_args* a, void* stream) {
    using namespace tscd;
    if (!a || !layout_ok(a->lay) || a->width <= 0 || (a->width % 64) != 0) return TSCD_ERR_INVALID_ARG;
    dim3 grid(a->lay.nk_pitch / 64, a->width / 64, a->lay.B);
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    if (a->lay.dtype == TSCD_F16) transpose_clip_kernel<__half><<<grid, 256, 0, st>>>(*a);
    else transpose_clip_kernel<__nv_bfloat16><<<grid, 256, 0, st>>>(*a);
    TSCD_CUDA_CHECK_LAUNCH();
    return TSCD_OK;
}

extern "C" int tscd_attn_pv(const tscd_attn_pv_args* a, void* stream) {
    using namespace tscd;
    if (!a || !layout_ok(a->lay)) return TSCD_ERR_INVALID_ARG;
    const tscd_attn_layout& l = a->lay;
    const int bf = l.dtype == TSCD_BF16;
    PvTmaps tm;
    int rc = 0;
    rc |= make_tmap_kmajor(&tm.qc, a->qn_cls, bf, l.row_cap, 256, 256, 128);
    rc |= make_tmap_kmajor(&tm.kc, a->kn_cls, bf, l.row_cap, 256, 256, 128);
    rc |= make_tmap_kmajor(&tm.qr, a->qn_reg, bf, l.row_cap, 256, 256, 128);
    rc |= make_tmap_kmajor(&tm.kr, a->kn_reg, bf, l.row_cap, 256, 256, 128);
    rc |= make_tmap_kmajor(&tm.k64c, a->kn_cls, bf, l.row_cap, 256, 256, 64);
    rc |= make_tmap_kmajor(&tm.k64r, a->kn_reg, bf, l.row_cap, 256, 256, 64);
    rc |= make_tmap_kmajor(&tm.vtc, a->vt_cls, bf, (int64_t)l.B * 256, l.nk_pitch, l.nk_pitch, 64);
    if (a->need_reg && !a->vt_reg) return TSCD_ERR_INVALID_ARG;
    // without need_reg the reg V^T is never loaded (and may be NULL): its map points at vt_cls
    rc |= make_tmap_kmajor(&tm.vtr, a->need_reg ? a->vt_reg : a->vt_cls, bf, (int64_t)l.B * 256, l.nk_pitch, l.nk_pitch, 64);
    if (rc) return TSCD_ERR_CUDA;
    const size_t smem = 65536 + kPvStages * 32768 + 65536 + sizeof(PvBars);
    dim3 grid((l.nk_pitch + 127) / 128, l.B);      // query tiles are bounded by the clip size; empty tiles exit at once
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    if (bf) {
        if (cudaFuncSetAttribute(attn_pv_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) return TSCD_ERR_CUDA;
        attn_pv_kernel<true><<<grid, kPvThreads, smem, st>>>(tm, *a);
    } else {
        if (cudaFuncSetAttribute(attn_pv_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) return TSCD_ERR_CUDA;
        attn_pv_kernel<false><<<grid, kPvThreads, smem, st>>>(tm, *a);
    }
    TSCD_CUDA_CHECK_LAUNCH();
    return TSCD_OK;
}

extern "C" int tscd_attn_round2(const tscd_attn_round2_args* a, void* stream) {
    using namespace tscd;
    if (!a || !layout_ok(a->lay)) return TSCD_ERR_INVALID_ARG;
    if (a->w_in && !a->use_obj_mask) return TSCD_ERR_INVALID_ARG;      // w_in is the cls launch's weights: only the obj launch re-uses them
    const tscd_attn_layout& l = a->lay;
    const int bf = l.dtype == TSCD_BF16;
    R2Tmaps tm;
    int rc = 0;
    rc |= make_tmap_kmajor(&tm.q128c, a->qn_cls, bf, l.row_cap, 256, 256, 128);
    rc |= make_tmap_kmajor(&tm.q128r, a->qn_reg, bf, l.row_cap, 256, 256, 128);
    rc |= make_tmap_kmajor(&tm.k64c, a->kn_cls, bf, l.row_cap, 256, 256, 64);
    rc |= make_tmap_kmajor(&tm.k64r, a->kn_reg, bf, l.row_cap, 256, 256, 64);
    rc |= make_tmap_kmajor(&tm.vn128c, a->vn_cls, bf, l.row_cap, 256, 256, 128);
    rc |= make_tmap_kmajor(&tm.vn128r, a->vn_reg, bf, l.row_cap, 256, 256, 128);
    rc |= make_tmap_kmajor(&tm.vn64c, a->vn_cls, bf, l.row_cap, 256, 256, 64);
    rc |= make_tmap_kmajor(&tm.vn64r, a->vn_reg, bf, l.row_cap, 256, 256, 64);
    rc |= make_tmap_kmajor(&tm.vt, a->vt, bf, (int64_t)l.B * 256, l.nk_pitch, l.nk_pitch, 64);
    if (rc) return TSCD_ERR_CUDA;
    const size_t smem = kR2SmemBytes + sizeof(R2Bars);
    dim3 grid((l.nk_pitch + 127) / 128, l.B);
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    if (bf) {
        if (cudaFuncSetAttribute(attn_round2_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) return TSCD_ERR_CUDA;
        attn_round2_kernel<true><<<grid, kR2Threads, smem, st>>>(tm, *a);
    } else {
        if (cudaFuncSetAttribute(attn_round2_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) return TSCD_ERR_CUDA;
        attn_round2_kernel<false><<<grid, kR2Threads, smem, st>>>(tm, *a);
    }
    TSCD_CUDA_CHECK_LAUNCH();
    return TSCD_OK;
}

#ifdef TSCD_R2_PROF
extern "C" int tscd_debug_r2_waits(unsigned long long* out, int reset) {      // out[0..63] attn_round2, out[64..127] attn_pv
    if (reset) {
        unsigned long long z[64] = {};
        return cudaMemcpyToSymbol(tscd::g_r2_wait, z, sizeof(z)) == cudaSuccess && cudaMemcpyToSymbol(tscd::g_pv_wait, z, sizeof(z)) == cudaSuccess ? 0 : -1;
    }
    return cudaMemcpyFromSymbol(out, tscd::g_r2_wait, sizeof(unsigned long long) * 64) == cudaSuccess &&
                   cudaMemcpyFromSymbol(out + 64, tscd::g_pv_wait, sizeof(unsigned long long) * 64) == cudaSuccess ? 0 : -1;
}
#endif

extern "C" int tscd_attn_rowmeta(const tscd_attn_rowmeta_args* a, void* stream) {
    using namespace tscd;
    if (!a || !layout_ok(a->lay) || !a->row_frame || !a->row_meta || !a->vt_cls || a->lay.B > 32767 || a->lay.nk_pitch > 65536) return TSCD_ERR_INVALID_ARG;
    dim3 grid(a->lay.nk_pitch / 64, a->lay.B);
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    if (a->lay.dtype == TSCD_F16) attn_rowmeta_kernel<__half><<<grid, 64, 0, st>>>(*a);
    else attn_rowmeta_kernel<__nv_bfloat16><<<grid, 64, 0, st>>>(*a);
    TSCD_CUDA_CHECK_LAUNCH();
    return TSCD_OK;
}
