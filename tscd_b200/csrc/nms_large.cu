// K2 for frames of more than 4096 candidates (up to 16384): the final per-class NMS of post_process.py:36-65 expands every
// proposal into one row per class above the 0.001 filter -- 500 proposals x 25 classes = 12 500 rows per frame for the
// shipped OVIS-L limits (exps/TSCD_OVIS/ovis_tscd_large.py:45,49) -- far beyond what one CTA sorts and resolves in shared
// memory.  Same semantics as csrc/nms.cu (torchvision batched_nms, coordinate trick, bit-exact keep lists), three kernels
// over a caller-provided workspace:
//
//   nmsl_partition  one CTA per frame: boxes.max()+1, class histogram -> class offsets, unordered scatter of the
//                   candidate positions into per-class lists, x-band of every class's offset boxes;
//   nmsl_class      one CTA per (frame, class): sort the class's members by (score desc, position asc), offset boxes in
//                   shared memory, lazy greedy suppression in chunks of 32 -> one `kept` flag per candidate.  After the
//                   coordinate-trick offset, boxes of different classes interact only where the classes' x-bands overlap
//                   (negative coordinates); greedy NMS decomposes EXACTLY into per-class problems as long as no cross-class
//                   pair exceeds the IoU threshold, so exactly those pairs are tested here and a hit marks the frame;
//   nmsl_merge      one CTA per frame: sort the kept candidates by (score desc, position asc) -> keep list.  Marked frames
//                   (cross-class hit, class ids outside [0,256), a class of more than kClassCap members) are redone with
//                   the general algorithm: full sort + lazy greedy over all candidates (slow, exact).
//
// Frames of more than 16384 candidates (up to 65536: the wide tier's 2048 proposals x 30 classes = 61 440 rows) keep the
// first two kernels; their candidates no longer fit one CTA's sort, so the merge goes through global memory:
//   nmsw_run        one CTA per (frame, run of 16384 positions): the run's kept candidates (every candidate of a marked frame)
//                   sorted by (score desc, position asc) in shared memory, written to the workspace;
//   nmsw_rank       one thread per sorted entry: its rank in the frame = its rank in its run + the number of larger keys in
//                   each other run (binary search; keys are unique, they carry the position) -> the merged order, and the keep
//                   list of an unmarked frame;
//   nmsw_final      one CTA per frame: keep count / overflow status, and for marked frames the general algorithm's lazy
//                   greedy over the merged order in global memory.
#include "nms.cuh"

namespace tscd {

constexpr int kClassCap = 2048;        // members of one class handled by nmsl_class
constexpr int kPartThreads = 512, kClassThreads = 256, kMergeThreads = 1024;
constexpr int kClassSlots = 32;        // grid.y of nmsl_class: classes are dealt round-robin over the slots

constexpr int kRun = 16384, kRunsMax = kNmsWideCap / kRun;   // wide path: sorted runs per frame

struct LargeWs {
    float* off_unit;        // [F]
    int* fallback;          // [F]
    int* ncl;               // [F]
    int* class_off;         // [F][257]
    float* lo;              // [F][256]
    float* hi;              // [F][256]
    unsigned char* ids;     // [F][256]
    int* list;              // [F][cap]
    unsigned char* flag;    // [F][cap]
    // wide path only (cap > kNmsLargeCap)
    int* run_n;                     // [F][kRunsMax] entries of every run
    unsigned long long* run_key;    // [F][cap] run r at [r * kRun, r * kRun + run_n)
    unsigned long long* merged;     // [F][cap] every run's entries in frame order
    int* kept;                      // [F][cap] marked frames: merged ranks of the boxes kept so far
};

__host__ __device__ inline size_t r16(size_t x) { return (x + 15) & ~(size_t)15; }

__host__ inline size_t large_ws_bytes(int F, int cap) {
    size_t b = r16((size_t)F * 4) * 3 + r16((size_t)F * 257 * 4) + r16((size_t)F * 256 * 4) * 2 + r16((size_t)F * 256) +
               r16((size_t)F * cap * 4) + r16((size_t)F * cap);
    if (cap > kNmsLargeCap) b += r16((size_t)F * kRunsMax * 4) + 2 * r16((size_t)F * cap * 8) + r16((size_t)F * cap * 4);
    return b;
}
__host__ inline LargeWs carve_large_ws(void* p, int F, int cap) {
    unsigned char* c = reinterpret_cast<unsigned char*>(p);
    LargeWs w;
    w.off_unit = reinterpret_cast<float*>(c); c += r16((size_t)F * 4);
    w.fallback = reinterpret_cast<int*>(c); c += r16((size_t)F * 4);
    w.ncl = reinterpret_cast<int*>(c); c += r16((size_t)F * 4);
    w.class_off = reinterpret_cast<int*>(c); c += r16((size_t)F * 257 * 4);
    w.lo = reinterpret_cast<float*>(c); c += r16((size_t)F * 256 * 4);
    w.hi = reinterpret_cast<float*>(c); c += r16((size_t)F * 256 * 4);
    w.ids = c; c += r16((size_t)F * 256);
    w.list = reinterpret_cast<int*>(c); c += r16((size_t)F * cap * 4);
    w.flag = c; c += r16((size_t)F * cap);
    w.run_n = nullptr; w.run_key = nullptr; w.merged = nullptr; w.kept = nullptr;
    if (cap > kNmsLargeCap) {
        w.run_n = reinterpret_cast<int*>(c); c += r16((size_t)F * kRunsMax * 4);
        w.run_key = reinterpret_cast<unsigned long long*>(c); c += r16((size_t)F * cap * 8);
        w.merged = reinterpret_cast<unsigned long long*>(c); c += r16((size_t)F * cap * 8);
        w.kept = reinterpret_cast<int*>(c);
    }
    return w;
}

__device__ __forceinline__ unsigned long long nms_key(float score, int pos) {
    return ((unsigned long long)f2ord(score) << 32) | (unsigned long long)(0xffffffffu - (uint32_t)pos);
}
__device__ __forceinline__ int key_pos(unsigned long long k) { return (int)(0xffffffffu - (uint32_t)(k & 0xffffffffull)); }

// ------------------------------------------------------------------------------------------------ partition
__global__ void __launch_bounds__(kPartThreads) nmsl_partition_kernel(const tscd_nms_args args, const LargeWs ws) {
    __shared__ int hist[257];
    __shared__ int cursor[256];
    __shared__ uint32_t lo_u[256], hi_u[256];
    __shared__ float red[kPartThreads / 32];
    __shared__ int s_bad, s_ncl;
    const int frame = blockIdx.x, tid = threadIdx.x, lane = tid & 31;
    const int n = min(args.count[frame], args.cand_cap);
    if (n <= 0) {
        if (tid == 0) { ws.ncl[frame] = 0; ws.fallback[frame] = 0; }
        return;
    }
    const int64_t base = (int64_t)frame * args.cand_cap;
    const float4* gbox = reinterpret_cast<const float4*>(args.box) + base;
    const int32_t* gcls = args.cls + base;
    for (int c = tid; c < 257; c += blockDim.x) hist[c] = 0;
    for (int c = tid; c < 256; c += blockDim.x) { cursor[c] = 0; lo_u[c] = 0xffffffffu; hi_u[c] = 0u; }
    if (tid == 0) s_bad = 0;
    __syncthreads();
    float mx = -INFINITY;
    int bad = 0;
    for (int i = tid; i < n; i += blockDim.x) {
        const float4 b = gbox[i];
        mx = fmaxf(mx, fmaxf(fmaxf(b.x, b.y), fmaxf(b.z, b.w)));
        const int c = gcls[i];
        if (c < 0 || c > 255) bad = 1; else atomicAdd(&hist[c + 1], 1);
    }
    mx = warp_maxf(mx);
    if (lane == 0) red[tid >> 5] = mx;
    if (bad) s_bad = 1;
    __syncthreads();
    mx = red[0];
#pragma unroll
    for (int w = 1; w < kPartThreads / 32; ++w) mx = fmaxf(mx, red[w]);
    const float off_unit = __fadd_rn(mx, 1.f);          // boxes.max() + 1
    if (tid == 0) { ws.off_unit[frame] = off_unit; ws.fallback[frame] = s_bad; }
    if (s_bad) {                                         // general path only
        if (tid == 0) ws.ncl[frame] = 0;
        return;
    }
    if (tid < 32) {                                      // prefix over the 256 class counts (8 per lane) + non-empty class ids
        int loc[8], tot = 0;
#pragma unroll
        for (int j = 0; j < 8; ++j) { loc[j] = hist[1 + lane * 8 + j]; tot += loc[j]; }
        const int inc = warp_incl_scan(tot, lane);
        int run = inc - tot;
#pragma unroll
        for (int j = 0; j < 8; ++j) { run += loc[j]; hist[1 + lane * 8 + j] = run; }
        __syncwarp();
        int ncl = 0;
        unsigned char* ids = ws.ids + (int64_t)frame * 256;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int c = j * 32 + lane;
            const bool ne = hist[c + 1] - hist[c] > 0;
            const unsigned bal = __ballot_sync(0xffffffffu, ne);
            if (ne) ids[ncl + __popc(bal & ((1u << lane) - 1u))] = (unsigned char)c;
            ncl += __popc(bal);
        }
        if (lane == 0) s_ncl = ncl;
    }
    __syncthreads();
    int* list = ws.list + (int64_t)frame * args.cand_cap;
    for (int i = tid; i < n; i += blockDim.x) {
        const int c = gcls[i];
        const int slot = atomicAdd(&cursor[c], 1);
        list[hist[c] + slot] = i;                        // order inside a class is irrelevant: the sort key carries the position
        const float4 b = offset_box(gbox[i], c, off_unit);
        atomicMin(&lo_u[c], f2ord(b.x));
        atomicMax(&hi_u[c], f2ord(b.z));
    }
    __syncthreads();
    for (int c = tid; c < 257; c += blockDim.x) ws.class_off[(int64_t)frame * 257 + c] = hist[c];
    for (int c = tid; c < 256; c += blockDim.x) {
        ws.lo[(int64_t)frame * 256 + c] = ord2f(lo_u[c]);
        ws.hi[(int64_t)frame * 256 + c] = ord2f(hi_u[c]);
    }
    if (tid == 0) ws.ncl[frame] = s_ncl;
}

// ------------------------------------------------------------------------------------------------ per class
__global__ void __launch_bounds__(kClassThreads) nmsl_class_kernel(const tscd_nms_args args, const LargeWs ws, int class_cap) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    unsigned long long* skey = reinterpret_cast<unsigned long long*>(smem_raw);      // [class_cap]
    float4* sbox = reinterpret_cast<float4*>(skey + class_cap);                       // [class_cap] sorted, offset boxes
    float* sarea = reinterpret_cast<float*>(sbox + class_cap);                        // [class_cap]
    unsigned short* kept = reinterpret_cast<unsigned short*>(sarea + class_cap);      // [class_cap] sorted ranks of the kept boxes
    __shared__ unsigned int cmask[32];
    __shared__ unsigned int s_deadbits;
    __shared__ int s_nkept;
    const int frame = blockIdx.x, tid = threadIdx.x;
    const int n = min(args.count[frame], args.cand_cap);
    if (n <= 0 || ws.fallback[frame]) return;            // (a marked frame is redone from scratch by nmsl_merge)
    const int ncl = ws.ncl[frame];
    const int64_t base = (int64_t)frame * args.cand_cap;
    const float* gscore = args.score + base;
    const float4* gbox = reinterpret_cast<const float4*>(args.box) + base;
    const int* list = ws.list + base;
    unsigned char* flag = ws.flag + base;
    const int* coff = ws.class_off + (int64_t)frame * 257;
    const unsigned char* ids = ws.ids + (int64_t)frame * 256;
    const float* blo = ws.lo + (int64_t)frame * 256;
    const float* bhi = ws.hi + (int64_t)frame * 256;
    const float off_unit = ws.off_unit[frame];
    const double thr = (double)args.iou_thresh;

    for (int ci = blockIdx.y; ci < ncl; ci += gridDim.y) {
        const int c = ids[ci];
        const int o0 = coff[c], m = coff[c + 1] - o0;
        if (m > class_cap) {                             // uniform branch
            if (tid == 0) ws.fallback[frame] = 1;
            continue;
        }
        int cap = kClassThreads;
        while (cap < m) cap <<= 1;
        __syncthreads();                                 // previous class's shared data is dead
        for (int i = tid; i < m; i += blockDim.x) { const int pos = list[o0 + i]; skey[i] = nms_key(gscore[pos], pos); }
        __syncthreads();
        block_sort_desc64_dyn<unsigned long long>(skey, m, cap);
        for (int r = tid; r < m; r += blockDim.x) {
            const float4 b = offset_box(gbox[key_pos(skey[r])], c, off_unit);
            sbox[r] = b;
            sarea[r] = box_area(b);
        }
        if (tid == 0) s_nkept = 0;
        __syncthreads();
        // lazy greedy, 32 sorted boxes per step: chunk vs the boxes kept so far, 32 x 32 intra-chunk bitmask, warp 0 resolves
        for (int c0 = 0; c0 < m; c0 += 32) {
            const int cn = min(32, m - c0);
            if (tid < 32) cmask[tid] = 0u;
            if (tid == 0) s_deadbits = 0u;
            __syncthreads();
            const int nk0 = s_nkept;
            {
                const int l = tid & 31;
                if (l < cn) {
                    const float4 bl = sbox[c0 + l];
                    const float sl = sarea[c0 + l];
                    bool dead = false;
                    for (int k = tid >> 5; k < nk0 && !dead; k += kClassThreads / 32) {
                        const int i = kept[k];
                        dead = iou_gt(sbox[i], sarea[i], bl, sl, thr);
                    }
                    if (dead) atomicOr(&s_deadbits, 1u << l);
                }
            }
            for (int pr = tid; pr < 32 * 32; pr += blockDim.x) {
                const int l = pr >> 5, j = pr & 31;
                if (j < l && l < cn && iou_gt(sbox[c0 + j], sarea[c0 + j], sbox[c0 + l], sarea[c0 + l], thr)) atomicOr(&cmask[l], 1u << j);
            }
            __syncthreads();
            if (tid < 32) {
                const int lane = tid;
                const bool alive = (lane < cn) && !((s_deadbits >> lane) & 1u);
                const unsigned alive_bits = __ballot_sync(0xffffffffu, alive);
                const unsigned my = cmask[lane];
                unsigned kb = 0u;
#pragma unroll
                for (int l = 0; l < 32; ++l) {
                    const unsigned mm = __shfl_sync(0xffffffffu, my, l);
                    if (((alive_bits >> l) & 1u) && !(mm & kb)) kb |= 1u << l;
                }
                const bool mine = (kb >> lane) & 1u;
                if (mine) kept[nk0 + __popc(kb & ((1u << lane) - 1u))] = (unsigned short)(c0 + lane);
                if (lane < cn) flag[key_pos(skey[c0 + lane])] = mine ? 1 : 0;
                if (lane == 0) s_nkept = nk0 + __popc(kb);
            }
            __syncthreads();
        }
        // cross-class pairs against every later class whose x-band overlaps this one
        const float l_c = blo[c], h_c = bhi[c];
        for (int di = ci + 1; di < ncl; ++di) {
            const int d = ids[di];
            const float l_d = blo[d], h_d = bhi[d];
            if (!(fminf(h_c, h_d) > fmaxf(l_c, l_d))) continue;
            const int od = coff[d], nd = coff[d + 1] - od;
            bool hit = false;
            for (int jj = tid; jj < nd; jj += blockDim.x) {
                const float4 bj = offset_box(gbox[list[od + jj]], d, off_unit);
                if (!(bj.z > l_c) || !(bj.x < h_c)) continue;           // does not reach into this class's band
                const float sj = box_area(bj);
                for (int i = 0; i < m && !hit; ++i) {
                    const float4 bi = sbox[i];
                    if (fminf(bi.z, bj.z) > fmaxf(bi.x, bj.x)) hit = iou_gt(bi, sarea[i], bj, sj, thr);
                }
            }
            if (hit) ws.fallback[frame] = 1;
        }
    }
}

// ------------------------------------------------------------------------------------------------ merge / general path
__global__ void __launch_bounds__(kMergeThreads) nmsl_merge_kernel(const tscd_nms_args args, const LargeWs ws, int sort_cap) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    unsigned long long* skey = reinterpret_cast<unsigned long long*>(smem_raw);      // [sort_cap]
    int* s_kept = reinterpret_cast<int*>(skey + sort_cap);                            // [sort_cap] (general path)
    __shared__ int s_cnt;
    __shared__ float4 cbox[32];
    __shared__ float carea[32];
    __shared__ unsigned int cmask[32];
    __shared__ unsigned int s_deadbits;
    const int frame = blockIdx.x, tid = threadIdx.x;
    const int n = min(args.count[frame], args.cand_cap);
    const int max_keep = args.max_keep;
    int32_t* keep = args.keep + (int64_t)frame * max_keep;
    if (n <= 0) {
        if (tid == 0) args.keep_count[frame] = 0;
        return;
    }
    const int64_t base = (int64_t)frame * args.cand_cap;
    const float* gscore = args.score + base;
    const float4* gbox = reinterpret_cast<const float4*>(args.box) + base;
    const int32_t* gcls = args.cls + base;
    if (!ws.fallback[frame]) {
        const unsigned char* flag = ws.flag + base;
        if (tid == 0) s_cnt = 0;
        __syncthreads();
        for (int i = tid; i < n; i += blockDim.x)
            if (flag[i]) skey[atomicAdd(&s_cnt, 1)] = nms_key(gscore[i], i);
        __syncthreads();
        const int k = s_cnt;
        int cap = kMergeThreads;
        while (cap < k) cap <<= 1;
        block_sort_desc64_dyn<unsigned long long>(skey, k, cap);
        const int out = min(k, max_keep);
        for (int j = tid; j < out; j += blockDim.x) keep[j] = key_pos(skey[j]);
        if (tid == 0) {
            args.keep_count[frame] = out;
            if (args.strict_keep && k > max_keep) atomicMin(args.status, TSCD_ERR_CAPACITY);
        }
        return;
    }
    // ---- general path: every candidate, any class id, cross-class suppression included ----------------------------
    const float off_unit = ws.off_unit[frame];
    const double thr = (double)args.iou_thresh;
    for (int i = tid; i < n; i += blockDim.x) skey[i] = nms_key(gscore[i], i);
    __syncthreads();
    int cap = kMergeThreads;
    while (cap < n) cap <<= 1;
    block_sort_desc64_dyn<unsigned long long>(skey, n, cap);
    if (tid == 0) s_cnt = 0;
    __syncthreads();
    const int limit = args.strict_keep ? n : max_keep;   // strict: count every survivor to detect the overflow
    for (int c0 = 0; c0 < n; c0 += 32) {
        const int cn = min(32, n - c0);
        if (tid < 32) {
            cmask[tid] = 0u;
            if (tid < cn) {
                const int pos = key_pos(skey[c0 + tid]);
                const float4 b = offset_box(gbox[pos], gcls[pos], off_unit);
                cbox[tid] = b;
                carea[tid] = box_area(b);
            }
        }
        if (tid == 0) s_deadbits = 0u;
        __syncthreads();
        const int nk0 = s_cnt;
        {
            const int l = tid & 31;
            if (l < cn) {
                const float4 bl = cbox[l];
                const float sl = carea[l];
                bool dead = false;
                for (int k = tid >> 5; k < nk0 && !dead; k += kMergeThreads / 32) {
                    const int pos = key_pos(skey[s_kept[k]]);
                    const float4 bk = offset_box(gbox[pos], gcls[pos], off_unit);
                    if (fminf(bk.z, bl.z) > fmaxf(bk.x, bl.x)) dead = iou_gt(bk, box_area(bk), bl, sl, thr);
                }
                if (dead) atomicOr(&s_deadbits, 1u << l);
            }
        }
        {
            const int l = tid >> 5, j = tid & 31;        // 1024 threads = the 32 x 32 pairs of the chunk
            if (j < l && l < cn && iou_gt(cbox[j], carea[j], cbox[l], carea[l], thr)) atomicOr(&cmask[l], 1u << j);
        }
        __syncthreads();
        if (tid < 32) {
            const int lane = tid;
            const bool alive = (lane < cn) && !((s_deadbits >> lane) & 1u);
            const unsigned alive_bits = __ballot_sync(0xffffffffu, alive);
            const unsigned my = cmask[lane];
            unsigned kb = 0u;
#pragma unroll
            for (int l = 0; l < 32; ++l) {
                const unsigned mm = __shfl_sync(0xffffffffu, my, l);
                if (((alive_bits >> l) & 1u) && !(mm & kb)) kb |= 1u << l;
            }
            const int rank = nk0 + __popc(kb & ((1u << lane) - 1u));
            if ((kb >> lane) & 1u) {
                s_kept[rank] = c0 + lane;
                if (rank < max_keep) keep[rank] = key_pos(skey[c0 + lane]);
            }
            if (lane == 0) s_cnt = nk0 + __popc(kb);
        }
        __syncthreads();
        if (s_cnt >= limit) break;
    }
    if (tid == 0) {
        args.keep_count[frame] = min(s_cnt, max_keep);
        if (args.strict_keep && s_cnt > max_keep) atomicMin(args.status, TSCD_ERR_CAPACITY);
    }
}

// ------------------------------------------------------------------------------------------------ wide merge (> 16384)
__global__ void __launch_bounds__(kMergeThreads) nmsw_run_kernel(const tscd_nms_args args, const LargeWs ws) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    unsigned long long* skey = reinterpret_cast<unsigned long long*>(smem_raw);      // [kRun]
    __shared__ int s_cnt;
    const int frame = blockIdx.x, run = blockIdx.y, tid = threadIdx.x;
    const int n = min(args.count[frame], args.cand_cap);
    const int lo = run * kRun, hi = min(lo + kRun, n);
    const int64_t base = (int64_t)frame * args.cand_cap;
    if (hi <= lo) {
        if (tid == 0) ws.run_n[frame * kRunsMax + run] = 0;
        return;
    }
    const bool all = ws.fallback[frame] != 0;          // marked frame: the general path orders every candidate
    const float* gscore = args.score + base;
    const unsigned char* flag = ws.flag + base;
    if (tid == 0) s_cnt = 0;
    __syncthreads();
    for (int i = lo + tid; i < hi; i += blockDim.x)
        if (all || flag[i]) skey[atomicAdd(&s_cnt, 1)] = nms_key(gscore[i], i);
    __syncthreads();
    const int k = s_cnt;
    int cap = kMergeThreads;
    while (cap < k) cap <<= 1;
    block_sort_desc64_dyn<unsigned long long>(skey, k, cap);
    unsigned long long* out = ws.run_key + base + lo;
    for (int j = tid; j < k; j += blockDim.x) out[j] = skey[j];
    if (tid == 0) ws.run_n[frame * kRunsMax + run] = k;
}

__global__ void __launch_bounds__(256) nmsw_rank_kernel(const tscd_nms_args args, const LargeWs ws) {
    const int frame = blockIdx.y;
    const int e = blockIdx.x * blockDim.x + threadIdx.x;          // entry e of run e / kRun
    const int run = e / kRun, t = e - run * kRun;
    if (run >= kRunsMax || (int64_t)run * kRun >= args.cand_cap) return;
    const int* rn = ws.run_n + frame * kRunsMax;
    if (t >= rn[run]) return;
    const int64_t base = (int64_t)frame * args.cand_cap;
    const unsigned long long key = ws.run_key[base + e];
    int rank = t;
    for (int r = 0; r < kRunsMax && (int64_t)r * kRun < args.cand_cap; ++r) {
        if (r == run) continue;
        const unsigned long long* rk = ws.run_key + base + (int64_t)r * kRun;
        int lo = 0, hi = rn[r];                                    // descending run: count the entries > key
        while (lo < hi) {
            const int mid = (lo + hi) >> 1;
            if (rk[mid] > key) lo = mid + 1; else hi = mid;
        }
        rank += lo;
    }
    ws.merged[base + rank] = key;
    if (!ws.fallback[frame] && rank < args.max_keep) args.keep[(int64_t)frame * args.max_keep + rank] = key_pos(key);
}

// keep count of every frame; marked frames: nmsl_merge's general path with the sorted keys and the kept list in global memory
__global__ void __launch_bounds__(kMergeThreads) nmsw_final_kernel(const tscd_nms_args args, const LargeWs ws) {
    __shared__ int s_cnt;
    __shared__ float4 cbox[32];
    __shared__ float carea[32];
    __shared__ unsigned int cmask[32];
    __shared__ unsigned int s_deadbits;
    const int frame = blockIdx.x, tid = threadIdx.x;
    const int n = min(args.count[frame], args.cand_cap);
    const int max_keep = args.max_keep;
    int32_t* keep = args.keep + (int64_t)frame * max_keep;
    if (n <= 0) {
        if (tid == 0) args.keep_count[frame] = 0;
        return;
    }
    const int64_t base = (int64_t)frame * args.cand_cap;
    if (!ws.fallback[frame]) {
        if (tid == 0) {
            int k = 0;
            for (int r = 0; r < kRunsMax && (int64_t)r * kRun < args.cand_cap; ++r) k += ws.run_n[frame * kRunsMax + r];
            args.keep_count[frame] = min(k, max_keep);
            if (args.strict_keep && k > max_keep) atomicMin(args.status, TSCD_ERR_CAPACITY);
        }
        return;
    }
    const unsigned long long* skey = ws.merged + base;
    int* g_kept = ws.kept + base;
    const float4* gbox = reinterpret_cast<const float4*>(args.box) + base;
    const int32_t* gcls = args.cls + base;
    const float off_unit = ws.off_unit[frame];
    const double thr = (double)args.iou_thresh;
    if (tid == 0) s_cnt = 0;
    __syncthreads();
    const int limit = args.strict_keep ? n : max_keep;   // strict: count every survivor to detect the overflow
    for (int c0 = 0; c0 < n; c0 += 32) {
        const int cn = min(32, n - c0);
        if (tid < 32) {
            cmask[tid] = 0u;
            if (tid < cn) {
                const int pos = key_pos(skey[c0 + tid]);
                const float4 b = offset_box(gbox[pos], gcls[pos], off_unit);
                cbox[tid] = b;
                carea[tid] = box_area(b);
            }
        }
        if (tid == 0) s_deadbits = 0u;
        __syncthreads();
        const int nk0 = s_cnt;
        {
            const int l = tid & 31;
            if (l < cn) {
                const float4 bl = cbox[l];
                const float sl = carea[l];
                bool dead = false;
                for (int k = tid >> 5; k < nk0 && !dead; k += kMergeThreads / 32) {
                    const int pos = key_pos(skey[g_kept[k]]);
                    const float4 bk = offset_box(gbox[pos], gcls[pos], off_unit);
                    if (fminf(bk.z, bl.z) > fmaxf(bk.x, bl.x)) dead = iou_gt(bk, box_area(bk), bl, sl, thr);
                }
                if (dead) atomicOr(&s_deadbits, 1u << l);
            }
        }
        {
            const int l = tid >> 5, j = tid & 31;        // 1024 threads = the 32 x 32 pairs of the chunk
            if (j < l && l < cn && iou_gt(cbox[j], carea[j], cbox[l], carea[l], thr)) atomicOr(&cmask[l], 1u << j);
        }
        __syncthreads();
        if (tid < 32) {
            const int lane = tid;
            const bool alive = (lane < cn) && !((s_deadbits >> lane) & 1u);
            const unsigned alive_bits = __ballot_sync(0xffffffffu, alive);
            const unsigned my = cmask[lane];
            unsigned kb = 0u;
#pragma unroll
            for (int l = 0; l < 32; ++l) {
                const unsigned mm = __shfl_sync(0xffffffffu, my, l);
                if (((alive_bits >> l) & 1u) && !(mm & kb)) kb |= 1u << l;
            }
            const int rank = nk0 + __popc(kb & ((1u << lane) - 1u));
            if ((kb >> lane) & 1u) {
                g_kept[rank] = c0 + lane;
                if (rank < max_keep) keep[rank] = key_pos(skey[c0 + lane]);
            }
            if (lane == 0) s_cnt = nk0 + __popc(kb);
        }
        __syncthreads();                                 // also orders the g_kept writes before the next chunk's reads
        if (s_cnt >= limit) break;
    }
    if (tid == 0) {
        args.keep_count[frame] = min(s_cnt, max_keep);
        if (args.strict_keep && s_cnt > max_keep) atomicMin(args.status, TSCD_ERR_CAPACITY);
    }
}

int nms_large_launch(const tscd_nms_args& a, cudaStream_t st) {
    if (a.cand_cap > kNmsWideCap) return TSCD_ERR_CAPACITY;
    if (!a.ws || a.ws_bytes < (int64_t)large_ws_bytes(a.num_frames, a.cand_cap)) return TSCD_ERR_INVALID_ARG;
    const LargeWs ws = carve_large_ws(a.ws, a.num_frames, a.cand_cap);
    nmsl_partition_kernel<<<a.num_frames, kPartThreads, 0, st>>>(a, ws);
    TSCD_CUDA_CHECK_LAUNCH();
    int class_cap = kClassThreads;
    while (class_cap < a.cand_cap && class_cap < kClassCap) class_cap <<= 1;
    const size_t smem_c = (size_t)class_cap * (8 + 16 + 4 + 2);
    if (cudaFuncSetAttribute(nmsl_class_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_c) != cudaSuccess) return TSCD_ERR_CUDA;
    nmsl_class_kernel<<<dim3(a.num_frames, kClassSlots), kClassThreads, smem_c, st>>>(a, ws, class_cap);
    TSCD_CUDA_CHECK_LAUNCH();
    if (a.cand_cap > kNmsLargeCap) {
        const int runs = (a.cand_cap + kRun - 1) / kRun;
        const size_t smem_r = (size_t)kRun * 8;
        if (cudaFuncSetAttribute(nmsw_run_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_r) != cudaSuccess) return TSCD_ERR_CUDA;
        nmsw_run_kernel<<<dim3(a.num_frames, runs), kMergeThreads, smem_r, st>>>(a, ws);
        TSCD_CUDA_CHECK_LAUNCH();
        nmsw_rank_kernel<<<dim3(runs * kRun / 256, a.num_frames), 256, 0, st>>>(a, ws);
        TSCD_CUDA_CHECK_LAUNCH();
        nmsw_final_kernel<<<a.num_frames, kMergeThreads, 0, st>>>(a, ws);
        TSCD_CUDA_CHECK_LAUNCH();
        return TSCD_OK;
    }
    int sort_cap = kMergeThreads;
    while (sort_cap < a.cand_cap) sort_cap <<= 1;
    const size_t smem_m = (size_t)sort_cap * (8 + 4);
    if (cudaFuncSetAttribute(nmsl_merge_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_m) != cudaSuccess) return TSCD_ERR_CUDA;
    nmsl_merge_kernel<<<a.num_frames, kMergeThreads, smem_m, st>>>(a, ws, sort_cap);
    TSCD_CUDA_CHECK_LAUNCH();
    return TSCD_OK;
}

}  // namespace tscd

extern "C" int64_t tscd_nms_workspace_bytes(int32_t num_frames, int32_t cand_cap) {
    if (num_frames <= 0 || cand_cap <= tscd::kNmsCap) return 0;
    return (int64_t)tscd::large_ws_bytes(num_frames, cand_cap);
}
