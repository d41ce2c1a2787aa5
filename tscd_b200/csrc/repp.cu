// REPP detection linking on the device (SURVEY.md 8f-3): the O(n1 * n2) part of the reference's tubelet post-processing.
//
// Reference: tools/REPP.py:82-133 (get_video_pairs + solve_distances_def) with the linking scores of :52-79
// (distance_def / distance_logreg) and the pair features of tools/repp_utils.py:34-109.  The reference fills an n1 x n2
// distance matrix with a Python double loop (one sklearn predict_proba call per pair) and then repeatedly takes the global
// minimum (first in row-major order among equals), erasing its row and column, until only INF is left.
//
// Here one CTA handles one pair of consecutive frames: every thread evaluates linking distances (same operation order and
// precision as the numpy expressions: box / ratio / IoU arithmetic in fp32, the centre distance's square root, the
// logistic model and the score algebra in fp64), the finite ones are appended to a candidate list in the workspace, and the
// greedy matching is a loop of block-wide arg-min reductions over the surviving candidates with (distance, row-major index)
// as the key -- exactly the order the reference extracts pairs in, which the tubelet builder depends on.
#include <cfloat>

#include "common.cuh"

namespace tscd {

constexpr int kReppThreads = 256;
constexpr int kReppMaxDet = 4096;          // detections per frame (row / column "used" bitmaps live in shared memory)
constexpr double kReppInf = 9e15;          // REPP.py:16

// repp_utils.py:53-109 on (x, y, w, h) fp32 boxes; every operation rounded to fp32 like the numpy float32 scalars
__device__ __forceinline__ float repp_iou(float4 p, float4 q) {
    const float px2 = __fadd_rn(p.z, p.x), py2 = __fadd_rn(p.w, p.y), qx2 = __fadd_rn(q.z, q.x), qy2 = __fadd_rn(q.w, q.y);
    const float xl = fmaxf(p.x, q.x), yt = fmaxf(p.y, q.y), xr = fminf(px2, qx2), yb = fminf(py2, qy2);
    if (xr < xl || yb < yt) return 0.f;
    const float inter = __fmul_rn(__fsub_rn(xr, xl), __fsub_rn(yb, yt));
    const float a1 = __fmul_rn(__fsub_rn(px2, p.x), __fsub_rn(py2, p.y)), a2 = __fmul_rn(__fsub_rn(qx2, q.x), __fsub_rn(qy2, q.y));
    return __fdiv_rn(inter, __fsub_rn(__fadd_rn(a1, a2), inter));
}

__device__ __forceinline__ double repp_distance(const tscd_repp_link_args& a, int i, int j) {
    const float4 p = reinterpret_cast<const float4*>(a.bbox)[i], q = reinterpret_cast<const float4*>(a.bbox)[j];
    const double si = a.score[i], sj = a.score[j];
    const double dot = a.cls[i] == a.cls[j] ? __dmul_rn(si, sj) : 0.0;       // one-hot score vectors (REPP.py:251-253)
    const float iou = repp_iou(p, q);
    if (a.distance_func == 0) {                                               // distance_def :52-57
        const double div = __dmul_rn((double)iou, dot);
        return div == 0.0 ? kReppInf : __ddiv_rn(1.0, div);
    }
    const float wrel = __fdiv_rn(fminf(p.z, q.z), fmaxf(p.z, q.z)), hrel = __fdiv_rn(fminf(p.w, q.w), fmaxf(p.w, q.w));
    const float2 c1 = reinterpret_cast<const float2*>(a.center)[i], c2 = reinterpret_cast<const float2*>(a.center)[j];
    const float dx = __fsub_rn(c2.x, c1.x), dy = __fsub_rn(c2.y, c1.y);
    const double cd = sqrt((double)__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)));   // math.sqrt of the fp32 sum
    // features in the model's order: center_distances_corrected, height_rel, iou, width_rel (matching_model_logreg.pckl)
    double d = __dmul_rn(cd, a.coef[0]);
    d = __dadd_rn(d, __dmul_rn((double)hrel, a.coef[1]));
    d = __dadd_rn(d, __dmul_rn((double)iou, a.coef[2]));
    d = __dadd_rn(d, __dmul_rn((double)wrel, a.coef[3]));
    d = __dadd_rn(d, a.intercept);
    double sc = __ddiv_rn(1.0, __dadd_rn(1.0, exp(-d)));                      // predict_proba[:, 1] = expit(decision)
    if (sc < a.clf_thr) return kReppInf;
    if (a.clf_mode == 0) sc = __dmul_rn(dot, sc);                             // 'dot'
    else if (a.clf_mode == 1) sc = __dmul_rn(__dmul_rn(si, sj), sc);          // 'max' (one-hot vectors: max = the score)
    else if (a.clf_mode == 2) sc = __dadd_rn(dot, sc);                        // 'dot_plus'
    return __dsub_rn(1.0, sc);                                                // 'raw' = 3: unchanged
}

__global__ void __launch_bounds__(kReppThreads) repp_link_kernel(const tscd_repp_link_args a) {
    __shared__ uint32_t used_r[kReppMaxDet / 32], used_c[kReppMaxDet / 32];
    __shared__ double red_d[kReppThreads / 32];
    __shared__ long long red_i[kReppThreads / 32];
    __shared__ int s_count, s_pairs;
    __shared__ long long s_best;
    const int f = blockIdx.x;                                   // links frame f -> f + 1
    const int o1 = a.frame_off[f], o2 = a.frame_off[f + 1], o3 = a.frame_off[f + 2];
    const int n1 = o2 - o1, n2 = o3 - o2;
    int32_t* pairs = a.pairs + (int64_t)f * a.max_det * 2;
    if (n1 <= 0 || n2 <= 0 || n1 > a.max_det || n2 > a.max_det || n1 > kReppMaxDet || n2 > kReppMaxDet) {
        if (threadIdx.x == 0) {
            a.pair_count[f] = 0;
            if (n1 > 0 && n2 > 0 && a.status) atomicMin(a.status, TSCD_ERR_CAPACITY);
        }
        return;
    }
    double* cd = a.ws_dist + (int64_t)f * a.ws_pitch;            // candidate distances
    int32_t* ci = a.ws_idx + (int64_t)f * a.ws_pitch;            // candidate row-major indices  i * n2 + j
    for (int w = threadIdx.x; w < kReppMaxDet / 32; w += blockDim.x) { used_r[w] = 0u; used_c[w] = 0u; }
    if (threadIdx.x == 0) { s_count = 0; s_pairs = 0; }
    __syncthreads();
    const int64_t total = (int64_t)n1 * n2;
    for (int64_t e = threadIdx.x; e < total; e += blockDim.x) {
        const int i = (int)(e / n2), j = (int)(e - (int64_t)i * n2);
        const double d = repp_distance(a, o1 + i, o2 + j);
        if (d != kReppInf) {
            const int slot = atomicAdd(&s_count, 1);
            if (slot < a.ws_pitch) { cd[slot] = d; ci[slot] = (int)e; }
        }
    }
    __syncthreads();
    const int m = s_count;
    if (m > a.ws_pitch) {
        if (threadIdx.x == 0) { a.pair_count[f] = 0; if (a.status) atomicMin(a.status, TSCD_ERR_CAPACITY); }
        return;
    }
    // greedy: global minimum (ties: lowest row-major index) among candidates whose row and column are still free
    while (true) {
        double bd = kReppInf;
        long long bi = -1;
        for (int k = threadIdx.x; k < m; k += blockDim.x) {
            const int e = ci[k];
            if (e < 0) continue;
            const int i = e / n2, j = e - i * n2;
            if (((used_r[i >> 5] >> (i & 31)) & 1u) || ((used_c[j >> 5] >> (j & 31)) & 1u)) { ci[k] = -1; continue; }
            const double d = cd[k];
            if (d < bd || (d == bd && (long long)e < bi) || bi < 0) { bd = d; bi = e; }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const double od = __shfl_xor_sync(0xffffffffu, bd, o);
            const long long oi = __shfl_xor_sync(0xffffffffu, bi, o);
            if (oi >= 0 && (bi < 0 || od < bd || (od == bd && oi < bi))) { bd = od; bi = oi; }
        }
        if ((threadIdx.x & 31) == 0) { red_d[threadIdx.x >> 5] = bd; red_i[threadIdx.x >> 5] = bi; }
        __syncthreads();
        if (threadIdx.x == 0) {
            for (int w = 1; w < kReppThreads / 32; ++w) {
                const double od = red_d[w];
                const long long oi = red_i[w];
                if (oi >= 0 && (bi < 0 || od < bd || (od == bd && oi < bi))) { bd = od; bi = oi; }
            }
            s_best = bi;
            if (bi >= 0) {
                const int i = (int)(bi / n2), j = (int)(bi - (long long)i * n2);
                used_r[i >> 5] |= 1u << (i & 31);
                used_c[j >> 5] |= 1u << (j & 31);
                pairs[2 * s_pairs] = i;
                pairs[2 * s_pairs + 1] = j;
                ++s_pairs;
            }
        }
        __syncthreads();
        if (s_best < 0) break;
    }
    if (threadIdx.x == 0) a.pair_count[f] = s_pairs;
}


// ---- the bookkeeping after the linking (tscd_repp_prep / _tubelets / _emit) ------------------------------------------------
// Integer scans and scalar fp64 in the reference's order.  Scans over frames / pairs / tubelets / output units run in one CTA
// of kReppScanThreads (chunks of 1024 with a carry); the per-tubelet work is CTA-per-tubelet in a grid-stride loop.
constexpr int kReppScanThreads = 1024;
constexpr int kReppGrid = 148 * 8;

// largest f in [0, n) with off[f] <= v (off non-decreasing, off[0] <= v)
__device__ __forceinline__ int repp_find(const int32_t* off, int n, int v) {
    int lo = 0, hi = n - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (off[mid] <= v) lo = mid; else hi = mid - 1;
    }
    return lo;
}

// One packed row through Predictor.to_repp_heavy (val_to_imdb.py:201-216, as evalglue.repp_predictions types it) and the
// filter / one-hot of REPP.__call__ (REPP.py:247-256).  max(0, x) keeps the int 0 unless x > 0, min(iw, x) keeps the int iw
// unless x < iw; a coordinate that stays an int is exact in fp32, so the fp32 arithmetic below is NumPy's float32 scalar
// arithmetic with the ints converted -- except the centre of an axis clipped on both sides, where only Python ints and
// floats meet (fp64).
struct ReppDet {
    float4 box;
    float2 ctr;
    float sc;
    int cls, kind;
};

__device__ __forceinline__ bool repp_prep_row(const tscd_repp_prep_args& a, int f, int r, ReppDet& d) {
    const float* p = a.packed + (int64_t)r * 12;
    const int ih = a.img_size[2 * f], iw = a.img_size[2 * f + 1];
    const int wdiff = ih > iw ? (ih - iw) / 2 : 0, hdiff = iw > ih ? (iw - ih) / 2 : 0, mx = max(iw, ih);
    const float x1 = p[1], y1 = p[2], x2 = p[8], y2 = p[9];
    const bool lx = !(x1 > 0.f), ly = !(y1 > 0.f), rx = !(x2 < (float)iw), ry = !(y2 < (float)ih);
    const float xmin = lx ? 0.f : x1, ymin = ly ? 0.f : y1, xmax = rx ? (float)iw : x2, ymax = ry ? (float)ih : y2;
    const float w = __fsub_rn(xmax, xmin), h = __fsub_rn(ymax, ymin);
    if (w <= 0.f || h <= 0.f) return false;
    d.sc = __fmul_rn(p[7], p[10]);
    if (a.thr_f32 ? !(d.sc >= (float)a.min_tubelet_score) : !((double)d.sc >= a.min_tubelet_score)) return false;
    d.cls = (int)p[6];
    d.box = make_float4(xmin, ymin, w, h);
    d.kind = (lx ? 2 : 1) | (ly ? 2 : 1) | (lx && rx ? 2 : 1) | (ly && ry ? 2 : 1);
    d.ctr.x = lx && rx ? __double2float_rn(__ddiv_rn(__dadd_rn((double)wdiff, 0.5 * iw), (double)mx))
                       : __fdiv_rn(__fadd_rn(__fadd_rn(xmin, (float)wdiff), __fdiv_rn(w, 2.f)), (float)mx);
    d.ctr.y = ly && ry ? __double2float_rn(__ddiv_rn(__dadd_rn((double)hdiff, 0.5 * ih), (double)mx))
                       : __fdiv_rn(__fadd_rn(__fadd_rn(ymin, (float)hdiff), __fdiv_rn(h, 2.f)), (float)mx);
    return true;
}

__global__ void __launch_bounds__(256) repp_prep_count_kernel(const tscd_repp_prep_args a) {
    const int f = blockIdx.x, o = a.offsets[f], n = a.det_cand[f] ? a.offsets[f + 1] - o : 0;
    int kept = 0;
    for (int j0 = 0; j0 < n; j0 += blockDim.x) {
        ReppDet d;
        kept += __syncthreads_count(j0 + threadIdx.x < n && repp_prep_row(a, f, o + j0 + threadIdx.x, d));
    }
    if (threadIdx.x == 0) a.count[f] = kept;
}

// exclusive scan of n ints (out[n] = total), one CTA
__global__ void __launch_bounds__(kReppScanThreads) repp_scan_kernel(const int32_t* in, int n, int32_t* out) {
    __shared__ int scan[40];
    int carry = 0;
    for (int i0 = 0; i0 < n; i0 += blockDim.x) {
        const int i = i0 + threadIdx.x;
        int tot;
        const int ex = block_excl_scan(i < n ? in[i] : 0, scan, &tot);
        if (i < n) out[i] = carry + ex;
        carry += tot;
    }
    if (threadIdx.x == 0) out[n] = carry;
}

__global__ void __launch_bounds__(256) repp_prep_write_kernel(const tscd_repp_prep_args a) {
    __shared__ int scan[40];
    const int f = blockIdx.x, o = a.offsets[f], n = a.det_cand[f] ? a.offsets[f + 1] - o : 0;
    int base = a.frame_off[f];
    for (int j0 = 0; j0 < n; j0 += blockDim.x) {
        const int r = o + j0 + threadIdx.x;
        ReppDet d;
        const bool keep = j0 + threadIdx.x < n && repp_prep_row(a, f, r, d);
        int tot;
        const int i = base + block_excl_scan(keep ? 1 : 0, scan, &tot);
        base += tot;
        if (!keep) continue;
        if (d.cls < 0 || d.cls >= a.num_classes) atomicMin(a.status, TSCD_ERR_INVALID_ARG);   // q["scores"][idx] = sc
        reinterpret_cast<float4*>(a.bbox)[i] = d.box;
        reinterpret_cast<float2*>(a.center)[i] = d.ctr;
        a.score[i] = (double)d.sc;
        a.cls[i] = d.cls;
        a.box64[4 * i] = d.box.x; a.box64[4 * i + 1] = d.box.y; a.box64[4 * i + 2] = d.box.z; a.box64[4 * i + 3] = d.box.w;
        a.kind[i] = d.kind;
        a.src[i] = r;
    }
}

// next / has_prev per detection from the pairs of frame pair f (CTA f owns next[] of frame f and has_prev[] of frame f + 1)
__global__ void __launch_bounds__(256) repp_links_kernel(const tscd_repp_tubelets_args a) {
    const int f = blockIdx.x, P = a.num_frames - 1;
    const int o1 = a.frame_off[f], o2 = a.frame_off[f + 1], o3 = a.frame_off[f + 2];
    for (int g = o1 + threadIdx.x; g < o2; g += blockDim.x) a.next[g] = -1;
    for (int g = o2 + threadIdx.x; g < o3; g += blockDim.x) a.has_prev[g] = 0;
    if (f == 0)
        for (int g = o1 + threadIdx.x; g < o2; g += blockDim.x) a.has_prev[g] = 0;
    if (f == P - 1)
        for (int g = o2 + threadIdx.x; g < o3; g += blockDim.x) a.next[g] = -1;
    __syncthreads();
    const int32_t* pr = a.pairs + (int64_t)f * a.max_det * 2;
    for (int k = threadIdx.x; k < a.pair_count[f]; k += blockDim.x) {
        a.next[o1 + pr[2 * k]] = o2 + pr[2 * k + 1];
        a.has_prev[o2 + pr[2 * k + 1]] = 1;
    }
}

// data row of detection `local` of linking frame `pos`, read through the insertion-order frame at the same position
__device__ __forceinline__ int repp_data_row(const tscd_repp_tubelets_args& a, int pos, int local) {
    if (!a.data_off) return a.frame_off[pos] + local;
    if (local >= a.data_cnt[pos]) { atomicMin(a.status, TSCD_ERR_INVALID_ARG); return 0; }
    return a.data_off[pos] + local;
}

// get_tubelets: starts = pairs whose source has no incoming link, numbered in [frame pair, extraction index] order (the
// reference always restarts at the earliest frame with pairs left, and a chain consumes every linked successor); each start
// walks its chain once for the length and, after a scan, once for the members.  Then the singletons.
__global__ void __launch_bounds__(kReppScanThreads) repp_chains_kernel(const tscd_repp_tubelets_args a) {
    __shared__ int scan[40];
    const int P = a.num_frames - 1, tid = threadIdx.x, bd = blockDim.x;
    int32_t* pair_off = a.ws;
    int32_t* head_g = a.ws + P + 1;
    int32_t* head_f = head_g + a.cap;
    int carry = 0, tot;
    for (int f0 = 0; f0 < P; f0 += bd) {
        const int f = f0 + tid;
        const int ex = block_excl_scan(f < P ? a.pair_count[f] : 0, scan, &tot);
        if (f < P) pair_off[f] = carry + ex;
        carry += tot;
    }
    if (tid == 0) pair_off[P] = carry;
    __syncthreads();
    const int npairs = carry;
    int ntub = 0;
    for (int e0 = 0; e0 < npairs; e0 += bd) {
        const int e = e0 + tid;
        int st = 0, g = 0, f = 0;
        if (e < npairs) {
            f = repp_find(pair_off, P, e);
            g = a.frame_off[f] + a.pairs[((int64_t)f * a.max_det + (e - pair_off[f])) * 2];
            st = !a.has_prev[g];
        }
        const int t = ntub + block_excl_scan(st, scan, &tot);
        if (st && t < a.cap) { head_g[t] = g; head_f[t] = f; }
        ntub += tot;
    }
    if (ntub > a.cap) {
        if (tid == 0) atomicMin(a.status, TSCD_ERR_CAPACITY);
        ntub = a.cap;
    }
    for (int t = tid; t < ntub; t += bd) {
        int g = head_g[t], len = 1;
        while (a.next[g] >= 0) { g = a.next[g]; ++len; }
        a.tub_off[t] = len;
    }
    __syncthreads();
    carry = 0;
    for (int t0 = 0; t0 < ntub; t0 += bd) {
        const int t = t0 + tid;
        const int ex = block_excl_scan(t < ntub ? a.tub_off[t] : 0, scan, &tot);
        if (t < ntub) a.tub_off[t] = carry + ex;
        carry += tot;
    }
    if (tid == 0) a.tub_off[ntub] = carry;
    __syncthreads();
    for (int t = tid; t < ntub; t += bd) {
        int g = head_g[t], pos = head_f[t], j = a.tub_off[t];
        while (true) {
            a.members[j] = repp_data_row(a, pos, g - a.frame_off[pos]);
            const int nx = a.next[g];
            if (nx < 0) break;
            g = nx; ++pos; ++j;
        }
        a.tail_of[g] = t;
    }
    __syncthreads();
    int ns = 0;
    if (a.add_unmatched) {                                       // REPP.py:109, :235-243
        const int nodes = a.frame_off[P];                        // frames 0 .. n-2
        for (int g0 = 0; g0 < nodes; g0 += bd) {
            const int g = g0 + tid;
            const int s = g < nodes && a.next[g] < 0;
            const int i = ns + block_excl_scan(s, scan, &tot);
            if (s) {
                const int pos = repp_find(a.frame_off, P, g);
                a.single[i] = repp_data_row(a, pos, g - a.frame_off[pos]);
                a.single_tub[i] = a.has_prev[g] ? a.tail_of[g] : -1;
            }
            ns += tot;
        }
    }
    if (tid == 0) { a.counts[0] = ntub; a.counts[1] = ns; }
}

// rescore_tubelets (REPP.py:193-202) and recoordinate_tubelets_full (:205-218), one CTA per tubelet.
//   rescoring: np.mean over one-hot fp64 rows = per class a sequential sum in member order, then one division by M;
//   re-coordination: ndimage.convolve(column, w / sum(w), mode="reflect") = per output a sequential fp64 sum over the window
//   in index order, reflect indices (d c b a | a b c d | d c b a), taps with |w| <= DBL_EPSILON dropped (scipy's footprint);
//   the window of a length-M tubelet is the centred slice of the one long window, normalised by its left-to-right sum.
__global__ void __launch_bounds__(256) repp_smooth_kernel(const tscd_repp_emit_args a) {
    extern __shared__ double wn[];
    __shared__ double s_sum;
    __shared__ int s_kind;
    const int ntub = a.counts[0], C = a.num_classes, tid = threadIdx.x;
    for (int t = blockIdx.x; t < ntub; t += gridDim.x) {
        const int o = a.tub_off[t], M = a.tub_off[t + 1] - o;
        if (tid < 32) {
            int k = 0;
            for (int c0 = 0; c0 < C; c0 += 32) {
                const int c = c0 + tid;
                bool pass = false;
                if (c < C) {
                    double s = 0.0;
                    for (int m = 0; m < M; ++m) {
                        const int d = a.members[o + m];
                        if (a.cls[d] == c) s = __dadd_rn(s, a.score[d]);
                    }
                    s = __ddiv_rn(s, (double)M);
                    a.tub_score[(int64_t)t * C + c] = s;
                    pass = !(s < a.min_pred_score);
                }
                k += __popc(__ballot_sync(0xffffffffu, pass));
            }
            if (tid == 0) a.tub_k[t] = k;
        }
        if (!a.recoordinate) continue;
        const int W = 2 * M - 1;
        const double* w = a.window + (a.num_frames - M);
        if (tid == 0) {
            double s = 0.0;
            for (int j = 0; j < W; ++j) s = __dadd_rn(s, w[j]);
            s_sum = s;
            s_kind = 0;
        }
        __syncthreads();
        for (int j = tid; j < W; j += blockDim.x) wn[j] = __ddiv_rn(w[j], s_sum);
        for (int m = tid; m < M; m += blockDim.x) atomicOr(&s_kind, a.kind[a.members[o + m]]);
        __syncthreads();
        const int kind = s_kind;
        for (int q = tid; q < 4 * M; q += blockDim.x) {
            const int i = q >> 2, k = q & 3;
            double acc = 0.0;
            for (int j = 0; j < W; ++j) {
                const double wj = wn[j];
                if (!(fabs(wj) > DBL_EPSILON)) continue;
                int p = i + j - (M - 1);
                p = p < 0 ? -p - 1 : (p >= M ? 2 * M - 1 - p : p);
                acc = __dadd_rn(acc, __dmul_rn(a.box64[4 * a.members[o + p] + k], wj));
            }
            // the convolution writes into the column's own dtype: float32 rounds, int64 truncates
            a.mem_box[4 * (o + i) + k] = kind == 1 ? (double)__double2float_rn(acc) : kind == 2 ? (double)(long long)acc : acc;
        }
        __syncthreads();
    }
}

// classes a one-hot singleton emits (tubelets_to_predictions: skip s < min_pred_score)
__device__ __forceinline__ int repp_onehot_k(const tscd_repp_emit_args& a, int d) {
    return (0.0 < a.min_pred_score ? 0 : a.num_classes - 1) + (a.score[d] < a.min_pred_score ? 0 : 1);
}

__global__ void __launch_bounds__(kReppScanThreads) repp_rows_kernel(const tscd_repp_emit_args a) {
    __shared__ int scan[40];
    const int ntub = a.counts[0], U = ntub + a.counts[1];
    int carry = 0, tot;
    for (int u0 = 0; u0 < U; u0 += blockDim.x) {
        const int u = u0 + threadIdx.x;
        int rows = 0;
        if (u < ntub) {
            rows = (a.tub_off[u + 1] - a.tub_off[u]) * a.tub_k[u];
        } else if (u < U) {
            const int st = a.single_tub[u - ntub];
            rows = st >= 0 ? a.tub_k[st] : repp_onehot_k(a, a.single[u - ntub]);
        }
        const int ex = block_excl_scan(rows, scan, &tot);
        if (u < U) a.row_off[u] = carry + ex;
        carry += tot;
    }
    if (threadIdx.x == 0) {
        a.row_off[U] = carry;
        if ((int64_t)carry > a.row_cap) atomicMin(a.status, TSCD_ERR_CAPACITY);
        *a.n_out = (int64_t)carry > a.row_cap ? (int)a.row_cap : carry;
    }
}

// tubelets_to_predictions (REPP.py:221-233): tubelets then singletons (track id = unit index), members in chain order, classes
// ascending.  A singleton that is a tubelet's tail shares that tubelet's scores and box (one dict in the reference).
__global__ void __launch_bounds__(256) repp_write_kernel(const tscd_repp_emit_args a) {
    const int ntub = a.counts[0], U = ntub + a.counts[1], C = a.num_classes;
    for (int u = blockIdx.x; u < U; u += gridDim.x) {
        const int base = a.row_off[u], nrow = a.row_off[u + 1] - base;
        if ((int64_t)base + nrow > a.row_cap) continue;
        const int st = u < ntub ? u : a.single_tub[u - ntub];
        const int d0 = u < ntub ? -1 : a.single[u - ntub];
        const int k = st >= 0 ? a.tub_k[st] : 1;
        for (int r = threadIdx.x; r < nrow; r += blockDim.x) {
            int d, slot = -1, c = 0, j = st >= 0 ? r % k : r;
            double s = 0.0;
            if (st >= 0) {
                slot = u < ntub ? a.tub_off[u] + r / k : a.tub_off[st + 1] - 1;
                d = a.members[slot];
                const double* ts = a.tub_score + (int64_t)st * C;
                for (c = 0; c < C; ++c)
                    if (!(ts[c] < a.min_pred_score) && j-- == 0) break;
                s = ts[c];
            } else {
                d = d0;
                for (c = 0; c < C; ++c) {
                    s = c == a.cls[d] ? a.score[d] : 0.0;
                    if (!(s < a.min_pred_score) && j-- == 0) break;
                }
            }
            const double4 bx = reinterpret_cast<const double4*>(a.recoordinate && slot >= 0 ? a.mem_box : a.box64)[a.recoordinate && slot >= 0 ? slot : d];
            double4* out = reinterpret_cast<double4*>(a.out + (int64_t)(base + r) * 8);
            out[0] = make_double4(d, bx.x, bx.y, bx.z);
            out[1] = make_double4(bx.w, s, c, u);
        }
    }
}

}  // namespace tscd

extern "C" int tscd_repp_link(const tscd_repp_link_args* a, void* stream) {
    using namespace tscd;
    if (!a || a->num_frames < 0 || a->max_det <= 0 || a->ws_pitch <= 0 || !a->frame_off || !a->bbox || !a->center || !a->score ||
        !a->cls || !a->pairs || !a->pair_count || !a->ws_dist || !a->ws_idx)
        return TSCD_ERR_INVALID_ARG;
    if (a->distance_func != 0 && a->distance_func != 1) return TSCD_ERR_INVALID_ARG;
    if (a->clf_mode < 0 || a->clf_mode > 3) return TSCD_ERR_INVALID_ARG;
    if (a->max_det > kReppMaxDet) return TSCD_ERR_CAPACITY;
    if (a->num_frames < 2) return TSCD_OK;
    repp_link_kernel<<<a->num_frames - 1, kReppThreads, 0, reinterpret_cast<cudaStream_t>(stream)>>>(*a);
    TSCD_CUDA_CHECK_LAUNCH();
    return TSCD_OK;
}

extern "C" int tscd_repp_prep(const tscd_repp_prep_args* a, void* stream) {
    using namespace tscd;
    if (!a || a->num_frames <= 0 || a->num_classes <= 0 || !a->packed || !a->offsets || !a->det_cand || !a->img_size || !a->count ||
        !a->frame_off || !a->bbox || !a->center || !a->score || !a->cls || !a->box64 || !a->kind || !a->src || !a->status)
        return TSCD_ERR_INVALID_ARG;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    repp_prep_count_kernel<<<a->num_frames, 256, 0, st>>>(*a);
    TSCD_CUDA_CHECK_LAUNCH();
    repp_scan_kernel<<<1, kReppScanThreads, 0, st>>>(a->count, a->num_frames, a->frame_off);
    TSCD_CUDA_CHECK_LAUNCH();
    repp_prep_write_kernel<<<a->num_frames, 256, 0, st>>>(*a);
    TSCD_CUDA_CHECK_LAUNCH();
    return TSCD_OK;
}

extern "C" int tscd_repp_tubelets(const tscd_repp_tubelets_args* a, void* stream) {
    using namespace tscd;
    if (!a || a->num_frames <= 0 || a->max_det <= 0 || a->cap <= 0 || !a->frame_off || (!a->data_off != !a->data_cnt) ||
        (a->num_frames > 1 && (!a->pairs || !a->pair_count)) || !a->next || !a->has_prev || !a->tail_of || !a->ws || !a->counts ||
        !a->tub_off || !a->members || !a->single || !a->single_tub || !a->status)
        return TSCD_ERR_INVALID_ARG;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    if (a->num_frames > 1) {
        repp_links_kernel<<<a->num_frames - 1, 256, 0, st>>>(*a);
        TSCD_CUDA_CHECK_LAUNCH();
    }
    repp_chains_kernel<<<1, kReppScanThreads, 0, st>>>(*a);
    TSCD_CUDA_CHECK_LAUNCH();
    return TSCD_OK;
}

extern "C" int tscd_repp_emit(const tscd_repp_emit_args* a, void* stream) {
    using namespace tscd;
    if (!a || a->num_frames <= 0 || a->num_classes <= 0 || a->cap <= 0 || a->row_cap < 0 || (a->recoordinate && !a->window) ||
        !a->box64 || !a->kind || !a->score || !a->cls || !a->counts || !a->tub_off || !a->members || !a->single || !a->single_tub ||
        !a->tub_score || !a->tub_k || !a->mem_box || !a->row_off || !a->out || !a->n_out || !a->status)
        return TSCD_ERR_INVALID_ARG;
    if (2 * (int64_t)a->cap * a->num_classes > INT32_MAX) return TSCD_ERR_CAPACITY;      // row offsets are int32
    const size_t smem = a->recoordinate ? (size_t)(2 * a->num_frames - 1) * sizeof(double) : 0;
    if (smem > 200 * 1024) return TSCD_ERR_CAPACITY;                                        // window of a 12800-frame video
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    const int grid = a->cap < kReppGrid ? a->cap : kReppGrid;
    if (cudaFuncSetAttribute(repp_smooth_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) return TSCD_ERR_CUDA;
    repp_smooth_kernel<<<grid, 256, smem, st>>>(*a);
    TSCD_CUDA_CHECK_LAUNCH();
    repp_rows_kernel<<<1, kReppScanThreads, 0, st>>>(*a);
    TSCD_CUDA_CHECK_LAUNCH();
    repp_write_kernel<<<grid, 256, 0, st>>>(*a);
    TSCD_CUDA_CHECK_LAUNCH();
    return TSCD_OK;
}
