// Video pack: the detections of a group of whole videos, gathered from the clip calls that produced them, in frame order
// (tscd_b200/video.py VideoStream).  Replaces the host-side stitching of to_lists per call + splitting by video + trimming the
// padded tail frames + pack_detections per video with one pass on the device.
//   video_offsets_kernel   one CTA: per group frame the count of its (call, row), exclusive prefix, candidate counts;
//   video_pack_kernel      one CTA per frame: the rows through pack_detection_row (common.cuh), bit-identical to
//                          tscd_pack_detections.
#include "common.cuh"

namespace tscd {

// rows of frame i's source (call, row), or -1 when the map entry lies outside the calls
__device__ __forceinline__ int video_src(const tscd_video_pack_args& a, int i, const float** rows, int* cand) {
    const int c = a.map[3 * i], r = a.map[3 * i + 1];
    if (c < 0 || c >= a.num_calls) return -1;
    const tscd_video_pack_call k = a.calls[c];
    if (r < 0 || r >= k.n_rows) return -1;
    if (rows) *rows = k.rows + (int64_t)r * a.cap * 7;
    if (cand) *cand = k.cand ? k.cand[r] : 1;
    return min(k.count[r], a.cap);
}

__global__ void __launch_bounds__(1024) video_offsets_kernel(const tscd_video_pack_args a) {
    __shared__ int scan[40];
    int carry = 0;
    for (int f0 = 0; f0 < a.num_frames; f0 += blockDim.x) {
        const int f = f0 + threadIdx.x;
        int n = 0;
        if (f < a.num_frames) {
            int cand = 0;
            n = video_src(a, f, nullptr, &cand);
            if (n < 0) {
                n = 0;
                cand = 0;
                if (a.status) atomicMin(a.status, TSCD_ERR_INVALID_ARG);
            }
            if (a.det_cand) a.det_cand[f] = cand;
        }
        int tot;
        const int ex = block_excl_scan(n, scan, &tot);
        if (f < a.num_frames) a.offsets[f] = carry + ex;
        carry += tot;
    }
    if (threadIdx.x == 0) a.offsets[a.num_frames] = carry;
}

__global__ void __launch_bounds__(128) video_pack_kernel(const tscd_video_pack_args a) {
    const int f = blockIdx.x;
    const float* rows = nullptr;
    const int n = video_src(a, f, &rows, nullptr);
    const int o = a.offsets[f];
    const float s = a.scale ? a.scale[f] : 1.f;
    const float frame = (float)a.map[3 * f + 2];
    for (int j = threadIdx.x; j < n; j += blockDim.x)
        pack_detection_row(rows + (int64_t)j * 7, frame, s, a.packed + (int64_t)(o + j) * 12);
}

}  // namespace tscd

extern "C" int tscd_video_pack(const tscd_video_pack_args* a, void* stream) {
    using namespace tscd;
    if (!a || a->num_frames < 0 || a->num_calls <= 0 || a->cap <= 0 || !a->calls || !a->offsets) return TSCD_ERR_INVALID_ARG;
    if (a->num_frames > 0 && (!a->map || !a->packed)) return TSCD_ERR_INVALID_ARG;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    video_offsets_kernel<<<1, 1024, 0, st>>>(*a);
    TSCD_CUDA_CHECK_LAUNCH();
    if (a->num_frames == 0) return TSCD_OK;
    video_pack_kernel<<<a->num_frames, 128, 0, st>>>(*a);
    TSCD_CUDA_CHECK_LAUNCH();
    return TSCD_OK;
}
