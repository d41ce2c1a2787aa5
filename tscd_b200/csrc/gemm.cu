// Linear layers of the aggregation stage as a hand-written tcgen05 GEMM:
//     C[M,N] = A[M,K] * W[N,K]^T (+ bias[N]),  A/W fp16 or bf16 (K contiguous), fp32 accumulation in TMEM.
//
// Replaces the F.linear / cuBLAS calls at yolox/models/post_trans.py:613-618,687-689,1159-1161,
// yolox/models/tscd_matching.py:37-39,165-167,756 and yolox/models/tscd_head.py:507,515-520.
//
// Structure (one 128 x BN output tile per CTA, 192 threads):
//   warp 0     TMA producer: cp.async.bulk.tensor 2D loads of the A (128x64) and W (BNx64) k-blocks into a
//              3-stage shared-memory ring (128-byte swizzle), completion on "full" mbarriers;
//   warp 1     allocates TMEM and issues tcgen05.mma (one elected thread, 4 x K=16 per k-block), releasing
//              ring slots with tcgen05.commit on "empty" mbarriers and signalling the epilogue at the end;
//   warps 2-5  epilogue: tcgen05.ld (32 lanes x 32 columns per instruction; thread == output row), bias,
//              conversion and direct 64/128-byte row-segment stores to global memory.
// The row count may live in device memory (`m_dev`): CTAs whose rows are all beyond it exit immediately,
// which is how the ragged, data-dependent proposal counts are handled without a host sync.
#include <cuda.h>

#include "common.cuh"
#include "tc.cuh"

namespace tscd {

constexpr int kGemmBM = 128;
constexpr int kGemmBK = 64;
constexpr int kGemmStages = 3;
constexpr int kGemmThreads = 320;   // TMA warp, MMA warp, 8 epilogue warps
constexpr int kGemmThreadsFused = 576;   // fused q|k|v epilogue: 16 epilogue warps, one head each (the epilogue is latency-bound)
__host__ __device__ constexpr int gemm_epi_warps(int epi) { return epi ? 16 : 8; }

struct GemmParams {
    int M, N, K;
    const int* m_dev;     // optional device row count (min(M, *m_dev) rows are valid)
    const float* bias;    // optional [N]
    void* out16;          // optional 16-bit output (same type as the operands), pitch ld16 elements
    float* out32;         // optional fp32 output, pitch ld32 elements
    int ld16, ld32;
    int is_bf16;
    // fused q|k|v epilogue (EPI = 1): per-head L2 normalisation, key scaling, V^T / x_ori scatter (see tscd_qkv_project)
    const int32_t* row_meta;   // [rows] (clip << 16) | key index within the clip
    const int32_t* row_off;    // [B*F+1]
    const int32_t* lrow_off;   // [B*L+1]
    int B, F, L, self_attn, nk_pitch;
    const float* key_score;    // [rows] or NULL
    float scale;
    void *qn, *kn, *vn, *vt, *xori;
    int ld_xori;
};

// Debug build (-DTSCD_R2_PROF): clocks lane 0 of warps 0 (TMA), 1 (MMA) and 2 (epilogue) of CTA 0 of the FUSED projection
// kernel spend in each barrier wait; read back with tscd_debug_gemm_waits (tools/r2_waits.py).
#ifdef TSCD_R2_PROF
__device__ unsigned long long g_gemm_wait[8];
template <int EPI>
__device__ __forceinline__ void gemm_wait_prof(uint64_t* bar, uint32_t parity, int tag, int slot) {
    const long long t0 = clock64();
    tc::mbar_wait(bar, parity, tag);
    if (EPI == 1 && blockIdx.x == 0 && (threadIdx.x & 31) == 0 && threadIdx.x < 96) atomicAdd(&g_gemm_wait[slot], (unsigned long long)(clock64() - t0));
}
#define GEMM_WAIT(bar, parity, tag, slot) gemm_wait_prof<EPI>(bar, parity, tag, slot)
#else
#define GEMM_WAIT(bar, parity, tag, slot) mbar_wait(bar, parity, tag)
#endif

// Persistent, warp-specialised: every CTA walks tiles  t = blockIdx.x, blockIdx.x + gridDim.x, ...  (n fastest, so
// CTAs running at the same time share their A rows in L2).  Two TMEM accumulator stages let the epilogue of tile i
// overlap the TMA/MMA main loop of tile i+1; the smem ring keeps filling across tile boundaries.
// Resident weights: when the K loop has exactly as many blocks as the ring has stages (K = 256 with 128x256 tiles),
// k-block kb of every tile lands in stage kb, so the weight half of a stage already holds the right block whenever two
// consecutive tiles of a CTA share their column block -- tiles are then ordered m-fastest and the producer skips the
// weight load (192 KB -> 64 KB of L2 -> shared-memory traffic per tile).
constexpr int kAccStages = 2;

// Fused q|k|v projection (EPI = 1) schedule: the grid is G groups of 3 CTAs.  Group g walks m-tiles g, g + G, g + 2G, ...
// in rounds; in every round its three CTAs compute the q, k and v tiles of the same 128 bank rows at the same time, so
// those rows come from DRAM once and the other two CTAs read them from L2 (the m-fastest order of the plain kernel reads
// every row three times: all q tiles, then all k tiles, then all v tiles).  CTA j of a group computes column block
// (j + phase) % 3, where the phase (0, 1, 2) is the third of the rounds the round falls in: every CTA keeps one weight
// tile resident for a third of its tiles and gets an equal share of the three epilogues (v writes V^T and x_ori too).
// q is only stored for query rows (the first L frames of a clip), so a q tile without one is skipped altogether: no
// loads, MMA or epilogue.  The CTA then moves on to its next round.  Which of its q rounds hold a query row is worked out
// once at kernel start into a byte per round (rounds beyond kQFlagCap, i.e. more than 2048 x 49 m-tiles, are not skipped).
constexpr int kQkvGroup = 3;
constexpr int kQFlagCap = 2048;

template <int BN, bool BF16, int EPI = 0>
__global__ void __launch_bounds__(EPI ? kGemmThreadsFused : kGemmThreads) gemm_tn_kernel(const __grid_constant__ CUtensorMap tmap_a,
                                                                const __grid_constant__ CUtensorMap tmap_w,
                                                                const GemmParams p) {
    using namespace tc;
    constexpr int STAGES = BN == 256 ? 4 : 3;      // 128x256 tiles: 48 KB per stage, one CTA per SM, all 512 TMEM columns
    int M = p.M;
    if (p.m_dev) M = min(M, __ldg(p.m_dev));
    const int tiles_n = (p.N + BN - 1) / BN;
    const int tiles_m = (M + kGemmBM - 1) / kGemmBM;      // only tiles with valid rows exist
    const int num_tiles = tiles_m * tiles_n;
    // EPI = 1: group, member and round count of the grouped schedule (the host launches a multiple of 3 CTAs)
    const int groups = EPI ? (int)gridDim.x / kQkvGroup : 0;
    const int grp = EPI ? (int)blockIdx.x / kQkvGroup : 0, member = EPI ? (int)blockIdx.x % kQkvGroup : 0;
    const int rounds = EPI ? (tiles_m + groups - 1) / groups : 0;
    // uniform over the CTA, before any barrier / TMEM state exists
    if (EPI ? grp >= tiles_m : (int)blockIdx.x >= num_tiles) return;
#ifdef TSCD_R2_PROF
    const long long tk0 = clock64();
#endif

    // No static shared memory in this kernel: the dynamic window then starts at the CTA's shared base, which honours
    // the 1024-byte alignment the 128-byte swizzle needs (no over-allocation -> two CTAs fit in 227 KB).
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    unsigned char* smem = smem_raw;
    constexpr int kABytes = kGemmBM * kGemmBK * 2;
    constexpr int kWBytes = BN * kGemmBK * 2;
    unsigned char* sA = smem;
    unsigned char* sW = smem + STAGES * kABytes;
    unsigned char* sStage = sW + STAGES * kWBytes;      // 8 epilogue warps x (32 rows x 64 B)
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(sStage + gemm_epi_warps(EPI) * 2048);
    uint64_t* empty_bar = full_bar + STAGES;
    uint64_t* tmem_full_bar = empty_bar + STAGES;
    uint64_t* tmem_empty_bar = tmem_full_bar + kAccStages;
    uint32_t& tmem_base_smem = *reinterpret_cast<uint32_t*>(tmem_empty_bar + kAccStages);
    if ((smem_u32(smem) & 1023u) != 0) __trap();             // alignment contract violated

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int num_kb = (p.K + kGemmBK - 1) / kGemmBK;
    const bool w_resident = num_kb == STAGES;
    unsigned char* qflag = reinterpret_cast<unsigned char*>(full_bar) + 128;   // EPI = 1: [kQFlagCap] per round
    // The CTA's next tile: `cur` is the tile index (plain kernel) or the round (EPI = 1); false when the CTA is done.
    // Every role of the CTA walks the same sequence with its own cursor.
    auto next_tile = [&](int& cur, int& m0, int& n0) -> bool {
        if constexpr (EPI == 1) {
            for (;; ++cur) {
                const int mt = grp + groups * cur;
                if (mt >= tiles_m) return false;
                const int kind = (member + kQkvGroup * cur / rounds) % kQkvGroup;
                if (kind == 0 && cur < kQFlagCap && !qflag[cur]) continue;
                m0 = mt * kGemmBM;
                n0 = kind * BN;
                ++cur;
                return true;
            }
        } else {
            if (cur >= num_tiles) return false;
            if (w_resident) { m0 = (cur % tiles_m) * kGemmBM; n0 = (cur / tiles_m) * BN; }
            else { m0 = (cur / tiles_n) * kGemmBM; n0 = (cur % tiles_n) * BN; }
            cur += gridDim.x;
            return true;
        }
    };
    const int cur0 = EPI ? 0 : (int)blockIdx.x;

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&tmap_a);
        tma_prefetch_desc(&tmap_w);
        for (int s = 0; s < STAGES; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
        for (int s = 0; s < kAccStages; ++s) { mbar_init(&tmem_full_bar[s], 1); mbar_init(&tmem_empty_bar[s], gemm_epi_warps(EPI)); }
        fence_barrier_init();
    }
    if (warp == 1) tmem_alloc<kAccStages * BN>(&tmem_base_smem);
    if constexpr (EPI == 1) {
        // epilogue threads: does the q tile of round r hold a query row?  Rows [row_off[c*F], row_off[c*F+L]) of clip c
        // are its queries (the whole clip for self-attention); walk the clips that start inside the tile.
        if (warp >= 2) {
            for (int r = threadIdx.x - 64; r < min(rounds, kQFlagCap); r += blockDim.x - 64) {
                const int mt = grp + groups * r;
                bool hq = true;
                if (mt < tiles_m && (member + kQkvGroup * r / rounds) % kQkvGroup == 0) {
                    const int m_end = min(M, (mt + 1) * kGemmBM);
                    int row = mt * kGemmBM;
                    const int meta = __ldg(p.row_meta + row);
                    if (meta >= 0) {
                        hq = false;
                        for (int cb = meta >> 16; row < m_end && cb < p.B; ++cb) {
                            const int qend = __ldg(p.row_off + (p.self_attn ? (cb + 1) * p.F : cb * p.F + p.L));
                            if (row < qend) { hq = true; break; }
                            row = __ldg(p.row_off + (cb + 1) * p.F);
                        }
                    }
                }
                qflag[r] = hq;
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_base_smem;

    if (warp == 0) {
        if (lane == 0) {
            uint32_t it = 0;   // running k-block counter across tiles -> ring stage / phase
            int n_prev = -1;   // column block whose weights the stages hold (w_resident)
            int cur = cur0, m0, n0;
            while (next_tile(cur, m0, n0)) {
                const bool load_w = !(w_resident && n0 == n_prev);
                for (int kb = 0; kb < num_kb; ++kb, ++it) {
                    const int s = it % STAGES;
                    const uint32_t ph = (it / STAGES) & 1;
                    GEMM_WAIT(&empty_bar[s], ph ^ 1, 100 + s, 0);
                    mbar_expect_tx(&full_bar[s], load_w ? kABytes + kWBytes : kABytes);
                    tma_load_2d(sA + s * kABytes, &tmap_a, &full_bar[s], kb * kGemmBK, m0);
                    if (load_w) tma_load_2d(sW + s * kWBytes, &tmap_w, &full_bar[s], kb * kGemmBK, n0);
                }
                n_prev = n0;
            }
        }
    } else if (warp == 1) {
        {   // the whole warp walks the tile loop (warp-uniform operands stay in uniform registers: no per-instruction broadcast
            // loop in front of every tcgen05.mma), one elected lane issues
            const uint32_t idesc = make_idesc_f16(BF16, kGemmBM, BN);
            uint32_t it = 0, ti = 0;
            int cur = cur0, m0, n0;
            for (; next_tile(cur, m0, n0); ++ti) {
                const int acc = ti % kAccStages;
                const uint32_t aph = (ti / kAccStages) & 1;
                GEMM_WAIT(&tmem_empty_bar[acc], aph ^ 1, 130 + acc, 1);     // epilogue has drained this accumulator
                tc_fence_after();
                const uint32_t d = tmem_base + (uint32_t)(acc * BN);
                for (int kb = 0; kb < num_kb; ++kb, ++it) {
                    const int s = it % STAGES;
                    const uint32_t ph = (it / STAGES) & 1;
                    GEMM_WAIT(&full_bar[s], ph, 110 + s, 2);
                    tc_fence_after();
                    const uint64_t adesc = make_smem_desc_sw128(smem_u32(sA + s * kABytes));
                    const uint64_t bdesc = make_smem_desc_sw128(smem_u32(sW + s * kWBytes));
                    if (elect_one()) {
#pragma unroll
                        for (int k = 0; k < kGemmBK / 16; ++k) {
                            // advance 16 elements (32 bytes) along K inside the 128-byte swizzle row: +2 in 16-byte units
                            umma_f16(d, adesc + (uint64_t)(k * 2), bdesc + (uint64_t)(k * 2), idesc, (kb | k) ? 1u : 0u);
                        }
                        umma_commit(&empty_bar[s]);
                    }
                    __syncwarp();
                }
                if (elect_one()) umma_commit(&tmem_full_bar[acc]);
                __syncwarp();
            }
        }
    } else {
        // 8 epilogue warps: warp % 4 selects the TMEM lane quadrant (hardware rule), (warp - 2) / 4 the column half.
        // TMEM loads are software-pipelined: chunk c+1 is in flight while chunk c is converted and stored.
        const int q = warp & 3;
        const int half = (warp - 2) >> 2;
        constexpr int kChunks = BN / 64;                    // 32-column chunks per warp (half of the tile's columns)
        unsigned char* stg = sStage + (warp - 2) * 2048;
        const bool al16 = p.out16 && (p.ld16 % 8) == 0 && (reinterpret_cast<uintptr_t>(p.out16) & 15) == 0;
        const bool al32 = p.out32 && (p.ld32 % 4) == 0 && (reinterpret_cast<uintptr_t>(p.out32) & 15) == 0;
        uint32_t ti = 0;
        int cur = cur0, m0, n0;
        for (; next_tile(cur, m0, n0); ++ti) {
            const int acc = ti % kAccStages;
            const uint32_t aph = (ti / kAccStages) & 1;
            const int row_base = m0 + q * 32;
            const int row = row_base + lane;
            const bool row_ok = row < M;
            // fused epilogue: the row metadata (three dependent L2 reads) is fetched BEFORE waiting for the accumulator
            int meta = -1, lb = 0;
            bool is_query = false;
            if constexpr (EPI == 1) {
                meta = row_ok ? __ldg(p.row_meta + row) : -1;
                if (meta >= 0) {
                    const int cb0 = meta >> 16;
                    const int s0 = __ldg(p.row_off + cb0 * p.F);
                    const int n_loc = (p.self_attn ? __ldg(p.row_off + (cb0 + 1) * p.F) : __ldg(p.row_off + cb0 * p.F + p.L)) - s0;
                    is_query = (meta & 0xffff) < n_loc;
                    lb = __ldg(p.lrow_off + cb0 * p.L);
                }
            }
            GEMM_WAIT(&tmem_full_bar[acc], aph, 120 + acc, 3);
            tc_fence_after();
            const uint32_t tsrc = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(acc * BN + half * (BN / 2));
            if constexpr (EPI == 1) {
                // ---- fused q|k|v epilogue: this 256-column tile is the q (0), k (1) or v (2) projection of 128 bank rows;
                //      the warp's 128 columns are two heads; thread == row holds a head's 64 values in registers ----
                static_assert(BN == 256 || EPI == 0, "the fused epilogue works on 256-column tiles");
                const int kind = n0 >> 8;
                const bool valid = meta >= 0;
                const int cb = valid ? (meta >> 16) : 0, kr = meta & 0xffff;
                auto pk2h = [](float a, float b) -> uint32_t {
                    if (BF16) { __nv_bfloat162 h = __floats2bfloat162_rn(a, b); return *reinterpret_cast<uint32_t*>(&h); }
                    __half2 h = __floats2half2_rn(a, b);
                    return *reinterpret_cast<uint32_t*>(&h);
                };
                {
                    const int head = (warp - 2) >> 2;              // 16 epilogue warps: lane quadrant x head
                    const uint32_t tsrc_h = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(acc * BN + head * 64);
                    uint32_t r0[32], r1[32];
                    tmem_ld_32x32(tsrc_h, r0);
                    tmem_ld_32x32(tsrc_h + 32u, r1);
                    tmem_ld_wait();
                    float ss = 0.f;
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        ss = fmaf(__uint_as_float(r0[j]), __uint_as_float(r0[j]), ss);
                        ss = fmaf(__uint_as_float(r1[j]), __uint_as_float(r1[j]), ss);
                    }
                    // 16-bit row-segment stores go through the warp's 32 x 64-byte staging tile (as in the plain epilogue):
                    // one store instruction then writes 8 rows x 64 contiguous bytes instead of 32 scattered 16-byte pieces.
                    // `dest` = destination row of this lane's bank row (-1: nothing to store), fetched per staged row by shuffle.
                    auto staged_store = [&](const uint32_t (&w16)[16], uint16_t* base, int64_t dest, int ld, int col) {
                        __syncwarp();
#pragma unroll
                        for (int j = 0; j < 4; ++j)
                            *reinterpret_cast<uint4*>(stg + lane * 64 + ((j ^ ((lane >> 1) & 3)) << 4)) =
                                make_uint4(w16[4 * j], w16[4 * j + 1], w16[4 * j + 2], w16[4 * j + 3]);
                        __syncwarp();
#pragma unroll
                        for (int k = 0; k < 4; ++k) {
                            const int rr = 8 * k + (lane >> 2), ch = lane & 3;
                            const uint4 val = *reinterpret_cast<const uint4*>(stg + rr * 64 + ((ch ^ ((rr >> 1) & 3)) << 4));
                            const long long d = __shfl_sync(0xffffffffu, (long long)dest, rr);
                            if (d >= 0) *reinterpret_cast<uint4*>(base + d * ld + col + ch * 8) = val;
                        }
                    };
                    float sc = valid ? 1.f / sqrtf(ss) : 0.f;
                    if (kind == 1 && valid) sc *= p.key_score ? p.scale * __ldg(p.key_score + row) : p.scale;
                    uint16_t* nbase = reinterpret_cast<uint16_t*>(kind == 0 ? p.qn : (kind == 1 ? p.kn : p.vn));
                    const int64_t ndest = (valid && (kind != 0 || is_query)) ? (int64_t)row : -1;     // q of the global rows is never read
                    uint32_t w16[16];
#pragma unroll
                    for (int j = 0; j < 16; ++j) w16[j] = pk2h(__uint_as_float(r0[2 * j]) * sc, __uint_as_float(r0[2 * j + 1]) * sc);
                    staged_store(w16, nbase, ndest, 256, head * 64);
#pragma unroll
                    for (int j = 0; j < 16; ++j) w16[j] = pk2h(__uint_as_float(r1[2 * j]) * sc, __uint_as_float(r1[2 * j + 1]) * sc);
                    staged_store(w16, nbase, ndest, 256, head * 64 + 32);
                    if (kind == 2) {
                        // raw v: x_ori rows of the queries, and V^T (lanes are consecutive keys -> 64 contiguous bytes per channel)
                        if (p.xori) {
                            const int64_t xdest = (valid && is_query) ? (int64_t)(lb + kr) : -1;
#pragma unroll
                            for (int j = 0; j < 16; ++j) w16[j] = pk2h(__uint_as_float(r0[2 * j]), __uint_as_float(r0[2 * j + 1]));
                            staged_store(w16, reinterpret_cast<uint16_t*>(p.xori), xdest, p.ld_xori, head * 64);
#pragma unroll
                            for (int j = 0; j < 16; ++j) w16[j] = pk2h(__uint_as_float(r1[2 * j]), __uint_as_float(r1[2 * j + 1]));
                            staged_store(w16, reinterpret_cast<uint16_t*>(p.xori), xdest, p.ld_xori, head * 64 + 32);
                        }
                        if (valid && p.vt) {
                            uint16_t* vt = reinterpret_cast<uint16_t*>(p.vt) + ((int64_t)cb * 256 + head * 64) * p.nk_pitch + kr;
#pragma unroll
                            for (int j = 0; j < 32; ++j) {
                                vt[(int64_t)j * p.nk_pitch] = (uint16_t)(pk2h(__uint_as_float(r0[j]), 0.f) & 0xffffu);
                                vt[(int64_t)(32 + j) * p.nk_pitch] = (uint16_t)(pk2h(__uint_as_float(r1[j]), 0.f) & 0xffffu);
                            }
                        }
                    }
                    __syncwarp();
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&tmem_empty_bar[acc]);
                continue;
            }
            uint32_t rbuf[2][32];
            tmem_ld_32x32(tsrc, rbuf[0]);
            tmem_ld_wait();
#pragma unroll
            for (int c = 0; c < kChunks; ++c) {
                if (c + 1 < kChunks) tmem_ld_32x32(tsrc + (uint32_t)((c + 1) * 32), rbuf[(c + 1) & 1]);
                const uint32_t* r = rbuf[c & 1];
                const int col0 = n0 + half * (BN / 2) + c * 32;
                if (col0 < p.N) {
                    float v[32];
                    if (p.bias) {
#pragma unroll
                        for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]) + ((col0 + j < p.N) ? __ldg(p.bias + col0 + j) : 0.f);
                    } else {
#pragma unroll
                        for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]);
                    }
                    const bool full = (col0 + 32 <= p.N);
                    // Every chunk goes through a per-warp 32 x 64-byte staging tile (16-byte pieces XOR-swizzled by
                    // row) so that a store instruction writes 8 rows x 64 contiguous bytes (whole sectors) instead of
                    // 32 scattered 16-byte pieces.  Register arrays are only ever indexed statically (no local memory);
                    // the ragged / unaligned edge reads single elements back from the staging tile.
                    if (p.out16) {
                        uint32_t pk[16];
#pragma unroll
                        for (int j = 0; j < 16; ++j) {
                            if (BF16) {
                                __nv_bfloat162 h = __floats2bfloat162_rn(v[2 * j], v[2 * j + 1]);
                                pk[j] = *reinterpret_cast<uint32_t*>(&h);
                            } else {
                                __half2 h = __floats2half2_rn(v[2 * j], v[2 * j + 1]);
                                pk[j] = *reinterpret_cast<uint32_t*>(&h);
                            }
                        }
                        uint16_t* obase = reinterpret_cast<uint16_t*>(p.out16);
                        __syncwarp();
#pragma unroll
                        for (int j = 0; j < 4; ++j)
                            *reinterpret_cast<uint4*>(stg + lane * 64 + ((j ^ ((lane >> 1) & 3)) << 4)) =
                                make_uint4(pk[4 * j], pk[4 * j + 1], pk[4 * j + 2], pk[4 * j + 3]);
                        __syncwarp();
                        if (full && al16) {
#pragma unroll
                            for (int k = 0; k < 4; ++k) {
                                const int rr = 8 * k + (lane >> 2), ch = lane & 3;
                                const uint4 val = *reinterpret_cast<const uint4*>(stg + rr * 64 + ((ch ^ ((rr >> 1) & 3)) << 4));
                                if (row_base + rr < M)
                                    *reinterpret_cast<uint4*>(obase + (int64_t)(row_base + rr) * p.ld16 + col0 + ch * 8) = val;
                            }
                        } else if (row_ok) {
                            uint16_t* o = obase + (int64_t)row * p.ld16 + col0;
                            const int nc = min(32, p.N - col0);
                            for (int j = 0; j < nc; ++j)
                                o[j] = *reinterpret_cast<const uint16_t*>(stg + lane * 64 + (((j >> 3) ^ ((lane >> 1) & 3)) << 4) + (j & 7) * 2);
                        }
                    }
                    if (p.out32) {
#pragma unroll
                        for (int hh = 0; hh < 2; ++hh) {
                            __syncwarp();
#pragma unroll
                            for (int j = 0; j < 4; ++j)
                                *reinterpret_cast<float4*>(stg + lane * 64 + ((j ^ ((lane >> 1) & 3)) << 4)) =
                                    make_float4(v[hh * 16 + 4 * j], v[hh * 16 + 4 * j + 1], v[hh * 16 + 4 * j + 2], v[hh * 16 + 4 * j + 3]);
                            __syncwarp();
                            if (full && al32) {
#pragma unroll
                                for (int k = 0; k < 4; ++k) {
                                    const int rr = 8 * k + (lane >> 2), ch = lane & 3;
                                    const float4 val = *reinterpret_cast<const float4*>(stg + rr * 64 + ((ch ^ ((rr >> 1) & 3)) << 4));
                                    if (row_base + rr < M)
                                        *reinterpret_cast<float4*>(p.out32 + (int64_t)(row_base + rr) * p.ld32 + col0 + hh * 16 + ch * 4) = val;
                                }
                            } else if (row_ok) {
                                float* o = p.out32 + (int64_t)row * p.ld32 + col0 + hh * 16;
                                const int nc = min(16, p.N - col0 - hh * 16);
                                for (int j = 0; j < nc; ++j)
                                    o[j] = *reinterpret_cast<const float*>(stg + lane * 64 + (((j >> 2) ^ ((lane >> 1) & 3)) << 4) + (j & 3) * 4);
                            }
                        }
                    }
                }
                if (c + 1 < kChunks) tmem_ld_wait();
            }
            // this warp has read its part of the accumulator: release it to the MMA warp
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&tmem_empty_bar[acc]);
        }
    }
#ifdef TSCD_R2_PROF
    if (EPI == 1 && blockIdx.x == 0 && (threadIdx.x & 31) == 0 && threadIdx.x < 96) atomicAdd(&g_gemm_wait[4 + warp], (unsigned long long)(clock64() - tk0));
#endif
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc<kAccStages * BN>(tmem_base);
    }
}

// ---- host side ----------------------------------------------------------------------------------------
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static PFN_encodeTiled get_encode() {
    static PFN_encodeTiled fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess) return nullptr;
        if (q != cudaDriverEntryPointSuccess) return nullptr;
        fn = reinterpret_cast<PFN_encodeTiled>(p);
    }
    return fn;
}

// 2-D K-major operand [rows, K] with row pitch ld (elements); box = 64 (K) x box_rows, 128-byte swizzle.
int make_tmap_kmajor(CUtensorMap* m, const void* ptr, int is_bf16, int64_t rows, int64_t K, int64_t ld, int box_rows) {
    PFN_encodeTiled enc = get_encode();
    if (!enc) return TSCD_ERR_CUDA;
    if ((ld * 2) % 16 != 0 || (reinterpret_cast<uintptr_t>(ptr) & 15) != 0) return TSCD_ERR_INVALID_ARG;
    cuuint64_t dims[2] = {(cuuint64_t)K, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)(ld * 2)};
    cuuint32_t box[2] = {(cuuint32_t)kGemmBK, (cuuint32_t)box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(m, is_bf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2,
                     const_cast<void*>(ptr), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? TSCD_OK : TSCD_ERR_CUDA;
}

template <int BN, bool BF16, int EPI = 0>
static int launch_gemm(const CUtensorMap& ta, const CUtensorMap& tw, const GemmParams& p, cudaStream_t st) {
    constexpr int STAGES = BN == 256 ? 4 : 3;
    constexpr size_t smem = (size_t)STAGES * (kGemmBM * kGemmBK * 2 + BN * kGemmBK * 2) + gemm_epi_warps(EPI) * 2048 + 128 +
                            (EPI ? kQFlagCap : 0);   // 229504 + 2048 bytes for the fused projection, under the 227 KB limit
    // per-DEVICE caches (the attribute is per device; a process may drive several GPUs)
    static bool attr_set[64] = {};
    static int num_sms_dev[64] = {};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return TSCD_ERR_CUDA;
    if (!attr_set[dev]) {
        if (cudaFuncSetAttribute(gemm_tn_kernel<BN, BF16, EPI>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
            return TSCD_ERR_CUDA;
        if (cudaDeviceGetAttribute(&num_sms_dev[dev], cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return TSCD_ERR_CUDA;
        attr_set[dev] = true;
    }
    const int num_sms = num_sms_dev[dev];
    const int tiles = ((p.N + BN - 1) / BN) * ((p.M + kGemmBM - 1) / kGemmBM);
    const int ctas_per_sm = BN == 256 ? 1 : 2;                       // 113 KB smem and 2*BN TMEM columns per CTA (BN <= 128)
    int grid = tiles < ctas_per_sm * num_sms ? tiles : ctas_per_sm * num_sms;
    if (EPI) {   // whole groups of kQkvGroup CTAs, at most one group per m-tile
        const int tiles_m = (p.M + kGemmBM - 1) / kGemmBM;
        grid = kQkvGroup * min(tiles_m, num_sms / kQkvGroup);
    }
    gemm_tn_kernel<BN, BF16, EPI><<<grid, EPI ? kGemmThreadsFused : kGemmThreads, smem, st>>>(ta, tw, p);
    return cudaGetLastError() == cudaSuccess ? TSCD_OK : TSCD_ERR_CUDA;
}

}  // namespace tscd

extern "C" int tscd_linear(const tscd_linear_args* a, void* stream) {
    using namespace tscd;
    if (!a || a->M <= 0 || a->N <= 0 || a->K <= 0 || !a->x || !a->w) return TSCD_ERR_INVALID_ARG;
    if (a->dtype != TSCD_F16 && a->dtype != TSCD_BF16) return TSCD_ERR_UNSUPPORTED;
    if (!a->out16 && !a->out32) return TSCD_ERR_INVALID_ARG;
    const int is_bf16 = a->dtype == TSCD_BF16;
    // 128x128 tiles need 128 B/clk of operand reads from shared memory (its full bandwidth), 128x256 tiles 96 B/clk:
    // the wide tile is used where the main loop dominates (K >= 512); short-K GEMMs are epilogue-bound and keep two
    // smaller CTAs (16 epilogue warps) per SM
    const int BN = a->N <= 64 ? 64 : ((a->N % 256) == 0 && a->K >= 256 ? 256 : 128);
    CUtensorMap ta, tw;
    int rc = make_tmap_kmajor(&ta, a->x, is_bf16, a->M, a->K, a->ldx, kGemmBM);
    if (rc != TSCD_OK) return rc;
    rc = make_tmap_kmajor(&tw, a->w, is_bf16, a->N, a->K, a->ldw, BN);
    if (rc != TSCD_OK) return rc;
    GemmParams p = {};
    p.M = a->M; p.N = a->N; p.K = a->K;
    p.m_dev = a->m_dev; p.bias = a->bias;
    p.out16 = a->out16; p.out32 = a->out32;
    p.ld16 = a->ld16; p.ld32 = a->ld32;
    p.is_bf16 = is_bf16;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    if (is_bf16) return BN == 64 ? launch_gemm<64, true>(ta, tw, p, st) : (BN == 128 ? launch_gemm<128, true>(ta, tw, p, st) : launch_gemm<256, true>(ta, tw, p, st));
    return BN == 64 ? launch_gemm<64, false>(ta, tw, p, st) : (BN == 128 ? launch_gemm<128, false>(ta, tw, p, st) : launch_gemm<256, false>(ta, tw, p, st));
}

extern "C" int tscd_qkv_project(const tscd_qkv_project_args* a, void* stream) {
    using namespace tscd;
    if (!a || a->rows <= 0 || !a->x || !a->w || !a->row_meta || !a->qn || !a->kn || !a->vn) return TSCD_ERR_INVALID_ARG;
    const tscd_attn_layout& l = a->lay;
    if (l.dtype != TSCD_F16 && l.dtype != TSCD_BF16) return TSCD_ERR_UNSUPPORTED;
    if (l.B <= 0 || l.F <= 0 || l.L <= 0 || l.L > l.F || !l.row_off || !l.lrow_off || (l.nk_pitch % 128) != 0 || l.nk_pitch > 65536) return TSCD_ERR_INVALID_ARG;
    const int is_bf16 = l.dtype == TSCD_BF16;
    CUtensorMap ta, tw;
    int rc = make_tmap_kmajor(&ta, a->x, is_bf16, a->rows, 256, a->ldx, kGemmBM);
    if (rc != TSCD_OK) return rc;
    rc = make_tmap_kmajor(&tw, a->w, is_bf16, 768, 256, 256, 256);
    if (rc != TSCD_OK) return rc;
    GemmParams p = {};
    p.M = a->rows; p.N = 768; p.K = 256;
    p.m_dev = a->m_dev;
    p.is_bf16 = is_bf16;
    p.row_meta = a->row_meta; p.row_off = l.row_off; p.lrow_off = l.lrow_off;
    p.B = l.B; p.F = l.F; p.L = l.L; p.self_attn = l.self_attn; p.nk_pitch = l.nk_pitch;
    p.key_score = a->key_score; p.scale = a->scale;
    p.qn = a->qn; p.kn = a->kn; p.vn = a->vn; p.vt = a->vt; p.xori = a->xori; p.ld_xori = a->ld_xori;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    return is_bf16 ? launch_gemm<256, true, 1>(ta, tw, p, st) : launch_gemm<256, false, 1>(ta, tw, p, st);
}

#ifdef TSCD_R2_PROF
extern "C" int tscd_debug_gemm_waits(unsigned long long* out, int reset) {
    if (reset) {
        unsigned long long z[8] = {};
        return cudaMemcpyToSymbol(tscd::g_gemm_wait, z, sizeof(z)) == cudaSuccess ? 0 : -1;
    }
    return cudaMemcpyFromSymbol(out, tscd::g_gemm_wait, sizeof(unsigned long long) * 8) == cudaSuccess ? 0 : -1;
}
#endif
