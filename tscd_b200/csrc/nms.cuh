// Shared pieces of the NMS kernels (csrc/nms.cu: frames of up to 4096 candidates in shared memory; csrc/nms_large.cu:
// up to 65536 candidates through a global-memory workspace).
#pragma once
#include "common.cuh"

namespace tscd {

constexpr int kNmsCap = 4096;          // one-CTA-per-frame kernels (shared-memory sort)
constexpr int kNmsLargeCap = 16384;    // workspace path, per-frame merge in one CTA's shared memory
constexpr int kNmsWideCap = 65536;     // workspace path, merge through global memory (wide tier: 2048 proposals x <= 32 classes)

// torchvision's nms predicate on two (offset) boxes: inter / (Sa + Sb - inter) > thr, every operation rounded to nearest
// single precision exactly once (no FMA contraction), the comparison in double like the CPU kernel.
__device__ __forceinline__ bool iou_gt(const float4& a, float sa, const float4& b, float sb, double thr) {
    float xx1 = fmaxf(a.x, b.x), yy1 = fmaxf(a.y, b.y);
    float xx2 = fminf(a.z, b.z), yy2 = fminf(a.w, b.w);
    // disjoint boxes (every pair of different classes after the coordinate-trick offset): inter = 0, and
    // 0/u > thr is false for thr >= 0 (0/0 = NaN compares false too) -- skip the division
    if (!(xx2 > xx1) || !(yy2 > yy1)) return false;
    float w = fmaxf(0.f, __fsub_rn(xx2, xx1)), h = fmaxf(0.f, __fsub_rn(yy2, yy1));
    float inter = __fmul_rn(w, h);
    float uni = __fsub_rn(__fadd_rn(sa, sb), inter);
    float ovr = __fdiv_rn(inter, uni);
    return (double)ovr > thr;
}

// boxes + class_id * (boxes.max() + 1)   (torchvision _batched_nms_coordinate_trick)
__device__ __forceinline__ float4 offset_box(float4 b, int cls, float off_unit) {
    const float off = __fmul_rn((float)cls, off_unit);
    b.x = __fadd_rn(b.x, off); b.y = __fadd_rn(b.y, off);
    b.z = __fadd_rn(b.z, off); b.w = __fadd_rn(b.w, off);
    return b;
}
__device__ __forceinline__ float box_area(const float4& b) { return __fmul_rn(__fsub_rn(b.z, b.x), __fsub_rn(b.w, b.y)); }

// launched by tscd_nms for cand_cap > kNmsCap
int nms_large_launch(const tscd_nms_args& a, cudaStream_t st);

}  // namespace tscd
