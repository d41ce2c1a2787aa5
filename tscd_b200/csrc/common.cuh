// Shared device helpers for the TSCD aggregation-stage kernels (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <cuda_bf16.h>
#include <stdint.h>

#include "../../include/tscd_b200.h"

extern "C" void tscd_set_last_cuda_error(int code, const char* where);
#define TSCD_CUDA_CHECK_LAUNCH()                                   \
    do {                                                           \
        cudaError_t e__ = cudaGetLastError();                      \
        if (e__ != cudaSuccess) {                                  \
            tscd_set_last_cuda_error((int)e__, __FILE__);          \
            return TSCD_ERR_CUDA;                                  \
        }                                                          \
    } while (0)

namespace tscd {

constexpr int kWarp = 32;

// ---- order-preserving float <-> uint32 (larger float -> larger uint) --------------------------------
__device__ __forceinline__ uint32_t f2ord(float f) {
    uint32_t u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float ord2f(uint32_t u) {
    return __uint_as_float((u & 0x80000000u) ? (u & 0x7fffffffu) : ~u);
}

// ---- element loads (boundary tensors may be fp32 / fp16 / bf16) --------------------------------------
template <typename T> __device__ __forceinline__ float ldf(const T* p);
template <> __device__ __forceinline__ float ldf<float>(const float* p) { return __ldg(p); }
template <> __device__ __forceinline__ float ldf<__half>(const __half* p) { return __half2float(__ldg(p)); }
template <> __device__ __forceinline__ float ldf<__nv_bfloat16>(const __nv_bfloat16* p) {
    return __bfloat162float(__ldg(p));
}
__device__ __forceinline__ float ldf_reg(float v) { return v; }
__device__ __forceinline__ float ldf_reg(__half v) { return __half2float(v); }
__device__ __forceinline__ float ldf_reg(__nv_bfloat16 v) { return __bfloat162float(v); }
template <typename T> __device__ __forceinline__ T cvt_from_float(float v);
template <> __device__ __forceinline__ float cvt_from_float<float>(float v) { return v; }
template <> __device__ __forceinline__ __half cvt_from_float<__half>(float v) { return __float2half_rn(v); }
template <> __device__ __forceinline__ __nv_bfloat16 cvt_from_float<__nv_bfloat16>(float v) {
    return __float2bfloat16_rn(v);
}

// sigmoid matching ATen's  1 / (1 + exp(-x))  expression (used at seam S1 only)
__device__ __forceinline__ float sigmoidf_ref(float x) { return __fdiv_rn(1.f, __fadd_rn(1.f, expf(-x))); }

// ---- warp / block reductions ------------------------------------------------------------------------
__device__ __forceinline__ int warp_sum(int v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float warp_sumf(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float warp_maxf(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ int warp_incl_scan(int v, int lane) {
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        int t = __shfl_up_sync(0xffffffffu, v, o);
        if (lane >= o) v += t;
    }
    return v;
}

// Block-wide exclusive scan of one int per thread; returns exclusive prefix, writes total to *total.
// scratch: >= 33 ints of shared memory.  All threads must call.  blockDim.x multiple of 32, <= 1024.
__device__ __forceinline__ int block_excl_scan(int v, int* scratch, int* total) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
    int inc = warp_incl_scan(v, lane);
    if (lane == 31) scratch[wid] = inc;
    __syncthreads();
    if (wid == 0) {
        int w = lane < nw ? scratch[lane] : 0;
        int winc = warp_incl_scan(w, lane);
        scratch[lane] = winc - w;
        if (lane == 31) scratch[32] = winc;
    }
    __syncthreads();
    int res = inc - v + scratch[wid];
    *total = scratch[32];
    __syncthreads();
    return res;
}

// One packed detection row (tscd_pack_detections, tscd_video_pack): stage row r = [x1,y1,x2,y2,obj,cls_score,cls] of frame
// `frame`, resize scale s -> d = [frame, x1/s, y1/s, (x2/s - x1/s), (y2/s - y1/s), obj * cls, class, obj, x2/s, y2/s, cls_score, 0]
// (the reference's operation order: divide, then subtract; explicit rounding, no contraction).
__device__ __forceinline__ void pack_detection_row(const float* r, float frame, float s, float* d) {
    const float x1 = __fdiv_rn(r[0], s), y1 = __fdiv_rn(r[1], s), x2 = __fdiv_rn(r[2], s), y2 = __fdiv_rn(r[3], s);
    d[0] = frame; d[1] = x1; d[2] = y1; d[3] = __fsub_rn(x2, x1); d[4] = __fsub_rn(y2, y1);
    d[5] = __fmul_rn(r[4], r[5]); d[6] = r[6]; d[7] = r[4];
    d[8] = x2; d[9] = y2; d[10] = r[5]; d[11] = 0.f;
}

// ---- block-wide bitonic sort, descending, 64-bit keys ---------------------------------------------------
// E keys per thread in registers (element index = tid * E + r, E * blockDim.x keys in total, both powers of two).
// Compare-exchange distances below E stay inside the thread, distances below 32 * E go through warp shuffles, only
// the remaining ones use shared memory and a CTA barrier (10 of the 55 steps for 1024 keys on 512 threads).
// `smem` must hold E * blockDim.x keys.  All threads must call.
template <int E, typename KT>
__device__ __forceinline__ void bitonic_sort_regs_desc(KT (&v)[E], KT* smem) {
    const int tid = threadIdx.x;
    const int N = E * (int)blockDim.x;
    for (int k = 2; k <= N; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            if (j < E) {
#pragma unroll
                for (int r = 0; r < E; ++r) {
                    if ((r & j) == 0 && r + j < E) {
                        const bool desc = (((tid * E + r) & k) == 0);
                        const KT x = v[r], y = v[r + j < E ? r + j : r];
                        const bool sw = desc ? (x < y) : (x > y);
                        v[r] = sw ? y : x;
                        v[r + j < E ? r + j : r] = sw ? x : y;
                    }
                }
            } else if (j < 32 * E) {
#pragma unroll
                for (int r = 0; r < E; ++r) {
                    const int idx = tid * E + r;
                    const KT o = __shfl_xor_sync(0xffffffffu, v[r], j / E);
                    const bool keep_max = (((idx & j) == 0) == ((idx & k) == 0));
                    v[r] = keep_max ? (v[r] > o ? v[r] : o) : (v[r] < o ? v[r] : o);
                }
            } else {
#pragma unroll
                for (int r = 0; r < E; ++r) smem[tid * E + r] = v[r];
                __syncthreads();
#pragma unroll
                for (int r = 0; r < E; ++r) {
                    const int idx = tid * E + r;
                    const KT o = smem[idx ^ j];
                    const bool keep_max = (((idx & j) == 0) == ((idx & k) == 0));
                    v[r] = keep_max ? (v[r] > o ? v[r] : o) : (v[r] < o ? v[r] : o);
                }
                __syncthreads();
            }
        }
    }
}

// Sort the first `n` (<= cap) keys of smem_keys[0..cap) descending in place; cap = E * blockDim.x exactly.
// Entries at or beyond n are treated as 0 (they sort last).  Ends with the sorted keys visible to the whole CTA.
template <int E, typename KT>
__device__ __forceinline__ void block_sort_desc64(KT* smem_keys, int n) {
    KT v[E];
    const int tid = threadIdx.x;
#pragma unroll
    for (int r = 0; r < E; ++r) { const int i = tid * E + r; v[r] = i < n ? smem_keys[i] : (KT)0; }
    __syncthreads();
    bitonic_sort_regs_desc<E, KT>(v, smem_keys);
#pragma unroll
    for (int r = 0; r < E; ++r) smem_keys[tid * E + r] = v[r];
    __syncthreads();
}
// run-time dispatch on cap / blockDim.x (a power of two between 1 and 16); keys are 64- or 32-bit unsigned
template <typename KT>
__device__ __forceinline__ void block_sort_desc64_dyn(KT* smem_keys, int n, int cap) {
    const int e = cap / (int)blockDim.x;
    if (e <= 1) block_sort_desc64<1, KT>(smem_keys, n);
    else if (e == 2) block_sort_desc64<2, KT>(smem_keys, n);
    else if (e == 4) block_sort_desc64<4, KT>(smem_keys, n);
    else if (e == 8) block_sort_desc64<8, KT>(smem_keys, n);
    else block_sort_desc64<16, KT>(smem_keys, n);
}

// ---- block radix select (k-th largest key), shared by K1 and K2 ---------------------------------------
struct SelSmem {
    int hist[256];
    int scan[40];
    int misc[8];
};

// k-th largest key among keys[0..n) (k >= 1, k <= n).  Returns the threshold key T and the number of
// elements equal to T that belong to the top-k (r_eq); elements > T number k - r_eq.
template <typename KT>
__device__ void radix_select_kth(const KT* keys, int n, int k, SelSmem* s, uint32_t* T_out, int* req_out) {
    uint32_t prefix = 0, mask = 0;
    int remaining = k;
    constexpr int kPasses = (int)sizeof(KT);       // 8-bit digits, most significant first
    for (int pass = 0; pass < kPasses; ++pass) {
        const int shift = 8 * (kPasses - 1 - pass);
        for (int i = threadIdx.x; i < 256; i += blockDim.x) s->hist[i] = 0;
        __syncthreads();
        // histogram of the digit among the keys that still match the prefix.  Sigmoid scores share a few exponent
        // digits, so a plain shared-memory atomic per key would serialise on one bin in the first pass: the lanes
        // that agree with the first active lane's digit are counted with one ballot (leader adds the population),
        // the others (few, spread over many bins in the later passes) add themselves.
        for (int i0 = 0; i0 < n; i0 += blockDim.x) {
            const int i = i0 + threadIdx.x;
            const uint32_t u = i < n ? (uint32_t)keys[i] : 0u;
            const bool in = i < n && (u & mask) == prefix;
            const unsigned act = __ballot_sync(0xffffffffu, in);
            if (act == 0u) continue;
            const uint32_t d = (u >> shift) & 255;
            const int first = __ffs(act) - 1;
            const uint32_t d0 = __shfl_sync(0xffffffffu, d, first);
            const unsigned same = __ballot_sync(0xffffffffu, in && d == d0);
            if ((int)(threadIdx.x & 31) == first) atomicAdd(&s->hist[d0], __popc(same));
            else if (in && d != d0) atomicAdd(&s->hist[d], 1);
        }
        __syncthreads();
        if (threadIdx.x < 32) {
            // warp 0: lane l owns digits [8l, 8l+8); suffix sums from the top digit down
            const int lane = threadIdx.x;
            int loc[8], tot = 0;
#pragma unroll
            for (int j = 0; j < 8; ++j) { loc[j] = s->hist[255 - (lane * 8 + j)]; tot += loc[j]; }
            int inc = warp_incl_scan(tot, lane);
            int before = inc - tot;  // count of keys in strictly higher digit groups
            if (before < remaining && remaining <= inc) {
                int cum = before;
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    if (cum < remaining && remaining <= cum + loc[j]) {
                        s->misc[0] = 255 - (lane * 8 + j);
                        s->misc[1] = remaining - cum;
                    }
                    cum += loc[j];
                }
            }
        }
        __syncthreads();
        prefix |= (uint32_t)s->misc[0] << shift;
        mask |= 255u << shift;
        remaining = s->misc[1];
        __syncthreads();
    }
    *T_out = prefix;
    *req_out = remaining;
}

// Class max / arg-max of every anchor as its own streaming kernel (mode A, planar head layouts): thread = 8 anchors x all
// class planes, 8 independent 16-byte loads in flight per batch, thousands of small CTAs -> the class planes (83 % of the
// stage's mandatory HBM bytes) are read at streaming bandwidth instead of inside the per-frame selection CTA, whose
// on-chip phases (radix select, scans, sort) would otherwise stall the loads.  Results go to a [F, ws_pitch] workspace
// that select_kernel<T, true> reads back for the ~pre_k survivors only (L2 hits).

// ---- anchor geometry ----------------------------------------------------------------------------------
struct AnchorPos {
    int level;
    int local;  // index within the level
    float gx, gy, stride;
};
__device__ __forceinline__ AnchorPos anchor_pos(const tscd_anchors& an, int a) {
    AnchorPos p;
    int l = 0;
#pragma unroll
    for (int i = 1; i < TSCD_MAX_LEVELS; ++i)
        if (i < an.num_levels && a >= an.level_start[i]) l = i;
    p.level = l;
    p.local = a - an.level_start[l];
    int w = an.level_w[l];
    int y = p.local / w;
    p.gx = (float)(p.local - y * w);
    p.gy = (float)y;
    p.stride = (float)an.level_stride[l];
    return p;
}

template <typename T>
__device__ __forceinline__ const T* view_ptr(const tscd_view& v, int level, int frame, int local) {
    return reinterpret_cast<const T*>(v.ptr[level]) + (int64_t)frame * v.frame_stride[level] +
           (int64_t)local * v.anchor_stride[level];
}

// Box of one anchor as the reference computes it: decode_outputs (tscd_head.py:768-769) then
// cxcywh->xyxy (tscd_head.py:1561-1566).  Explicit round-to-nearest ops: no FMA contraction.
// cxcywh regression outputs of one anchor -> xyxy box, with explicit round-to-nearest ops (no FMA contraction)
__device__ __forceinline__ float4 box_from_reg(float cx, float cy, float w, float h, const AnchorPos& p, bool decode) {
    if (decode) {
        cx = __fmul_rn(__fadd_rn(cx, p.gx), p.stride);
        cy = __fmul_rn(__fadd_rn(cy, p.gy), p.stride);
        w = __fmul_rn(expf(w), p.stride);
        h = __fmul_rn(expf(h), p.stride);
    }
    float hw = __fmul_rn(w, 0.5f), hh = __fmul_rn(h, 0.5f);  // w/2 is exact either way
    return make_float4(__fsub_rn(cx, hw), __fsub_rn(cy, hh), __fadd_rn(cx, hw), __fadd_rn(cy, hh));
}

template <typename T>
__device__ __forceinline__ float4 anchor_box(const tscd_view& reg, const AnchorPos& p, int frame, bool decode) {
    const T* r = view_ptr<T>(reg, p.level, frame, p.local);
    const int64_t cs = reg.chan_stride[p.level];
    return box_from_reg(ldf(r), ldf(r + cs), ldf(r + 2 * cs), ldf(r + 3 * cs), p, decode);
}

// csrc/select_rows.cu: the fused [reg4|obj|cls C|pad] row layout (row pitch in elements, or 0) and its mode-A kernel
int fused_rows_pitch(const tscd_anchors& an, const tscd_view& reg, const tscd_view& obj, const tscd_view& cls, int num_classes,
                     int head_dtype, bool need_flat_obj);
int select_rows_try(const tscd_select_args* a, cudaStream_t st);

}  // namespace tscd
