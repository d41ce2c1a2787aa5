// Frame store: K1-K3 once per video frame, clips assembled on the device (tscd_b200/frames.py).
//
// Videos are cut into OVERLAPPING clips (tools/tscd_demo.py:223-241, vid.py:601-683: L consecutive local frames + G frames
// drawn from the rest of the video), so one frame is selected and gathered by several clips.  Everything K1-K3 produce for a
// frame depends on that frame alone, so the store keeps one frame's result per slot at a fixed pitch of kmax rows and a clip
// is rebuilt from its slots by a copy:
//   frame_scatter   packed K3 output of N frames (tscd_gather layout: rows at row_off[i]) -> rows at slot * kmax;
//   clip_assemble   clip_slots [B*F] -> counts + exclusive prefix (one CTA), then the rows of every frame back into the packed
//                   clip bank tscd_gather would have written for those frames (one CTA per frame and 64-row chunk).
// Both copy whole 512-byte feature rows with 16-byte vector loads, one row per warp, two rows in flight per warp.
#include "common.cuh"

namespace tscd {

constexpr int kStoreChunkRows = 64;             // rows of one frame copied by one CTA (grid.y = ceil(kmax / 64))

// Rows [j0, j1) of one frame: three 16-bit 256-wide planes (512 bytes each), the score, the anchor id and, when `rows_w` > 0,
// the reference row of rows_w fp32 values.
// src / dst: first plane row of the frame on each side; src_p / dst_p: its row in the [*, kmax] pitched sel_idx / sel_rows.
__device__ __forceinline__ void copy_frame_rows(const void* s_cls, const void* s_reg, const void* s_edge, const float* s_score,
                                                void* d_cls, void* d_reg, void* d_edge, float* d_score, int64_t src, int64_t dst,
                                                int j0, int j1, const int32_t* s_idx, int32_t* d_idx, int64_t src_p, int64_t dst_p,
                                                const float* s_rows, float* d_rows, int rows_w) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    const uint4* sc = reinterpret_cast<const uint4*>(s_cls);
    const uint4* sr = reinterpret_cast<const uint4*>(s_reg);
    const uint4* se = reinterpret_cast<const uint4*>(s_edge);
    uint4* dc = reinterpret_cast<uint4*>(d_cls);
    uint4* dr = reinterpret_cast<uint4*>(d_reg);
    uint4* de = reinterpret_cast<uint4*>(d_edge);
    for (int j = j0 + 2 * warp; j < j1; j += 2 * nw) {          // two rows per warp in flight: six 16-byte loads per lane
        const bool two = j + 1 < j1;
        const int64_t a = (src + j) * 32 + lane, b = (dst + j) * 32 + lane;
        const uint4 c0 = __ldg(sc + a), r0 = __ldg(sr + a), e0 = __ldg(se + a);
        uint4 c1, r1, e1;
        if (two) { c1 = __ldg(sc + a + 32); r1 = __ldg(sr + a + 32); e1 = __ldg(se + a + 32); }
        dc[b] = c0; dr[b] = r0; de[b] = e0;
        if (two) { dc[b + 32] = c1; dr[b + 32] = r1; de[b + 32] = e1; }
        if (lane < (two ? 2 : 1)) {
            d_score[dst + j + lane] = s_score[src + j + lane];
            if (d_idx) d_idx[dst_p + j + lane] = s_idx[src_p + j + lane];
        }
    }
    if (rows_w > 0 && j1 > j0) {                                // the frame's reference rows are contiguous on both sides
        const float* s = s_rows + (src_p + j0) * rows_w;
        float* d = d_rows + (dst_p + j0) * rows_w;
        const int n = (j1 - j0) * rows_w;
        if (((reinterpret_cast<uintptr_t>(s) | reinterpret_cast<uintptr_t>(d)) & 15) == 0) {
            const int n4 = n >> 2;
            for (int i = threadIdx.x; i < n4; i += blockDim.x)
                reinterpret_cast<float4*>(d)[i] = __ldg(reinterpret_cast<const float4*>(s) + i);
            for (int i = 4 * n4 + threadIdx.x; i < n; i += blockDim.x) d[i] = s[i];
        } else {
            for (int i = threadIdx.x; i < n; i += blockDim.x) d[i] = s[i];
        }
    }
}

__global__ void __launch_bounds__(256) frame_scatter_kernel(const tscd_frame_scatter_args a) {
    const tscd_frame_store& st = a.store;
    const int i = blockIdx.x;
    const int slot = a.frame_slots[i];
    if (slot < 0 || slot >= st.frames) {
        if (blockIdx.y == 0 && threadIdx.x == 0 && a.slot_error) atomicMin(a.slot_error, TSCD_ERR_FRAME_SLOT);
        return;
    }
    const int n = min(a.sel_count[i], st.kmax);
    const int j0 = blockIdx.y * kStoreChunkRows, j1 = min(n, j0 + kStoreChunkRows);
    if (blockIdx.y == 0 && threadIdx.x == 0) {
        st.count[slot] = n;
        // the capacity flags of K1 / K2 / the edge rows are per call: every frame of the call carries them.  `status` is only
        // read here (a bad slot goes to the separate `slot_error` word), so every block sees the same value.
        st.status[slot] = *a.status;
    }
    const int64_t own = (int64_t)slot * st.kmax;
    copy_frame_rows(a.bank_cls, a.bank_reg, a.bank_edge, a.bank_score, st.bank_cls, st.bank_reg, st.bank_edge, st.bank_score,
                    a.row_off[i], own, j0, j1, a.sel_idx, st.sel_idx, (int64_t)i * st.kmax, own, a.sel_rows, st.sel_rows,
                    7 + st.num_classes);
}

// One CTA: per clip frame the slot's count (0 and TSCD_ERR_FRAME_SLOT for a bad slot), exclusive prefix, status hand-over.
__global__ void __launch_bounds__(1024) clip_offsets_kernel(const tscd_clip_assemble_args a) {
    __shared__ int scan[40];
    const tscd_frame_store& st = a.store;
    const int nf = a.B * a.F;
    int carry = 0;
    for (int f0 = 0; f0 < nf; f0 += blockDim.x) {
        const int f = f0 + threadIdx.x;
        int c = 0;
        if (f < nf) {
            const int s = a.clip_slots[f];
            const int cnt = (s >= 0 && s < st.frames) ? st.count[s] : -1;
            if (cnt < 0) {
                atomicMin(a.status, TSCD_ERR_FRAME_SLOT);
            } else {
                c = min(cnt, st.kmax);
                const int e = st.status[s];
                if (e != 0) atomicMin(a.status, e);
            }
        }
        int tot;
        const int ex = block_excl_scan(c, scan, &tot);
        if (f < nf) { a.sel_count[f] = c; a.row_off[f] = carry + ex; }
        carry += tot;
    }
    if (threadIdx.x == 0) a.row_off[nf] = carry;
}

__global__ void __launch_bounds__(256) clip_rows_kernel(const tscd_clip_assemble_args a) {
    const tscd_frame_store& st = a.store;
    const int f = blockIdx.x;
    const int n = a.sel_count[f];
    const int j0 = blockIdx.y * kStoreChunkRows, j1 = min(n, j0 + kStoreChunkRows);
    if (j0 >= j1) return;                      // also every frame of a bad slot (count 0)
    const int64_t slot = a.clip_slots[f];
    const int W = 7 + st.num_classes;
    const bool local = (f % a.F) < a.L;        // reference rows are read for the local frames only (final expansion)
    const int64_t r0 = a.row_off[f];
    copy_frame_rows(st.bank_cls, st.bank_reg, st.bank_edge, st.bank_score, a.bank_cls, a.bank_reg, a.bank_edge, a.bank_score,
                    slot * st.kmax, r0, j0, j1, st.sel_idx, a.sel_idx, slot * st.kmax, (int64_t)f * st.kmax, st.sel_rows, a.sel_rows,
                    local ? W : 0);
}

static bool store_ok(const tscd_frame_store& s) {
    return s.frames > 0 && s.kmax > 0 && s.kmax <= TSCD_MAX_PROPOSALS && s.num_classes > 0 && s.count && s.status && s.bank_cls &&
           s.bank_reg && s.bank_edge && s.bank_score && s.sel_idx && s.sel_rows && (s.dtype == TSCD_F16 || s.dtype == TSCD_BF16);
}

}  // namespace tscd

extern "C" int tscd_frame_scatter(const tscd_frame_scatter_args* a, void* stream) {
    using namespace tscd;
    if (!a || !store_ok(a->store) || a->num_frames < 0 || !a->status) return TSCD_ERR_INVALID_ARG;
    if (a->num_frames == 0) return TSCD_OK;
    if (!a->frame_slots || !a->sel_count || !a->row_off || !a->sel_idx || !a->sel_rows || !a->bank_cls || !a->bank_reg ||
        !a->bank_edge || !a->bank_score)
        return TSCD_ERR_INVALID_ARG;
    const dim3 grid(a->num_frames, (a->store.kmax + kStoreChunkRows - 1) / kStoreChunkRows);
    frame_scatter_kernel<<<grid, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(*a);
    TSCD_CUDA_CHECK_LAUNCH();
    return TSCD_OK;
}

extern "C" int tscd_clip_assemble(const tscd_clip_assemble_args* a, void* stream) {
    using namespace tscd;
    if (!a || !store_ok(a->store) || a->B <= 0 || a->F <= 0 || a->L < 1 || a->L > a->F || !a->clip_slots || !a->status)
        return TSCD_ERR_INVALID_ARG;
    if (!a->sel_count || !a->row_off || !a->bank_cls || !a->bank_reg || !a->bank_edge || !a->bank_score || !a->sel_rows)
        return TSCD_ERR_INVALID_ARG;
    if (a->row_cap < (int64_t)a->B * a->F * a->store.kmax) return TSCD_ERR_CAPACITY;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    clip_offsets_kernel<<<1, 1024, 0, st>>>(*a);
    TSCD_CUDA_CHECK_LAUNCH();
    const dim3 grid(a->B * a->F, (a->store.kmax + kStoreChunkRows - 1) / kStoreChunkRows);
    clip_rows_kernel<<<grid, 256, 0, st>>>(*a);
    TSCD_CUDA_CHECK_LAUNCH();
    return TSCD_OK;
}
