// Volume-weighted snapshot SVD by the method of snapshots (device side of compute_svd, utils.py:302-346):
//   B = sqrt(vol) * (A - mean_t(A)),  G = B^T B  [T,T],  G = V diag(s^2) V^T,  U = B V / s / sqrt(vol) = (A - mean) V / s.
// The row means, the Gram contraction and the projection are hand-written kernels; the small dense T x T
// eigen-decomposition is left to the host (torch.linalg.eigh, fp64).
//
// Gram contraction, 2*M*T^2 flop (the only GEMM-shaped work of the S^3 path, SURVEY 8a row a14):
//   method 1/2 (default 1): tcgen05 tensor cores. gram_prepare_kernel centres and scales the rows and writes them as
//     TF32 "hi" (+ "lo" residual for the 3xTF32 split, method 1) planes in a [T/32][rows][32] layout; gram_tc_kernel
//     is warp-specialised: one TMA producer thread (3-D boxes, 128B swizzle with 32B atoms, 4-stage mbarrier ring), one
//     thread issuing tcgen05.mma.kind::tf32 with both operands MN-major straight from the swizzled stages
//     (D[128x256] += A_l*B_h + A_h*B_l + A_h*B_h), fp32 accumulators double-buffered in TMEM (2 x 256 columns),
//     and eight epilogue warps that pull every finished K-segment (a few stages) out of TMEM with tcgen05.ld,
//     sum segments in fp32 registers and flush to fp64 partials, while the next segment is already running.
//     (The tensor core's own fp32 accumulation truncates; short TMEM segments bound that drift. Measured on a
//     262144 x 2000 matrix, segment length x flush interval -> time, max error vs fp64: 4 x 32 -> 6.7 ms, 5.5e-7;
//     8 x 128 (default) -> 5.9 ms, 1.2e-6; 16 x 1000 -> 5.6 ms, 2.9e-6; the drains compete with the MMAs for TMEM.)
//     Optionally (default) the two CTAs of a cluster work on tiles that share B and fetch it once with TMA multicast;
//     that halves the L2 -> SM operand traffic but measured the same speed (6.72 vs 6.74 ms): the kernel is bound
//     by the tensor pipe + TMEM drains, not by operand traffic.
//   method 0: fp32 CUDA-core tiles (kept as the on-device cross-check of the tensor-core path).
// Projection U = (A - mean) V / s, 2*M*T*r flop: the same planes contracted over t on tcgen05 (project_tc_kernel, K-major
//   TF32 operands, 3xTF32, a few TMEM segments against accumulation drift; tf32_split_kernel splits (V / s)^T),
//   262144 x 2000 rows onto r = 50 / 150 / 256 modes in 1.8 / 2.3 / 2.6 ms (of which 1.1 ms is the prepare pass) instead
//   of 4.2 / 12.2 / 16.0 ms on the fp32 CUDA-core kernel, max error vs fp64 2e-6 .. 8e-6 of the largest entry.
// Residual of a low-rank model (s3_lowrank_error): lowrank_error_kernel, the operand forms of the projection with both
//   factors split by tf32_split_kernel, and lowrank_reduce_kernel. The inline PTX of these kernels is in tma.cuh.
#include "tma.cuh"
#include "../../include/s3b200.h"

namespace s3 {

// ---------------------------------------------------------------- row means
__global__ void __launch_bounds__(256)
row_mean_kernel(const float* __restrict__ a, int64_t m, int64_t t, float* __restrict__ mean) {
    const int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (row >= m) return;
    const float* p = a + row * t;
    double acc = 0.0;
    for (int64_t i = lane; i < t; i += 32) acc += (double)p[i];
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane == 0) mean[row] = (float)(acc / (double)t);
}

// ---------------------------------------------------------------- Gram: G[i][j] = sum_m vol_m (a_mi - mu_m)(a_mj - mu_m)
constexpr int kGT = 128;     // output tile (kGT x kGT) per CTA
constexpr int kGK = 16;      // rows of A per shared-memory step
constexpr int kGThreads = 256;
// rows of A per K-split at most: a split sums its rows in fp32 before the fp64 reduce, and that error grows with its
// length (600 000 x 2000 in 5 splits of 120 000 rows: 5.8e-5 of sqrt(G_ii G_jj) on a B200, against 2e-5 as the bound)
constexpr int64_t kGSplitRows = 8192;

__global__ void __launch_bounds__(kGThreads)
gram_kernel(const float* __restrict__ a, const float* __restrict__ mean, const float* __restrict__ vol, int vol_div,
            int64_t row0, int64_t m, int64_t t, int tiles, int64_t rows_per_split, float* __restrict__ partial) {
    __shared__ float sa[kGK][kGT];
    __shared__ float sb[kGK][kGT];
    // upper-triangular tile pair (ti <= tj) from the linear tile id
    int tid_lin = blockIdx.x, ti = 0;
    while (tid_lin >= tiles - ti) { tid_lin -= tiles - ti; ++ti; }
    const int tj = ti + tid_lin;
    const int64_t r0 = row0 + (int64_t)blockIdx.y * rows_per_split;
    const int64_t r1 = (r0 + rows_per_split) < m ? (r0 + rows_per_split) : m;
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;     // 16 x 16 threads, 8 x 8 outputs each
    float acc[8][8];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
    for (int64_t rr = r0; rr < r1; rr += kGK) {
        // load kGK rows x 128 columns of both column tiles, centred and scaled by sqrt(vol)
        for (int e = threadIdx.x; e < kGK * kGT; e += kGThreads) {
            const int kk = e / kGT, c = e % kGT;
            const int64_t row = rr + kk;
            float va = 0.f, vb = 0.f;
            if (row < r1) {
                const float mu = mean[row];
                const float s = sqrtf(vol[row / vol_div]);
                const int64_t ca = (int64_t)ti * kGT + c, cb = (int64_t)tj * kGT + c;
                if (ca < t) va = (a[row * t + ca] - mu) * s;
                if (cb < t) vb = (a[row * t + cb] - mu) * s;
            }
            sa[kk][c] = va;
            sb[kk][c] = vb;
        }
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < kGK; ++kk) {
            float ra[8], rb[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) ra[i] = sa[kk][ty * 8 + i];
#pragma unroll
            for (int j = 0; j < 8; ++j) rb[j] = sb[kk][tx * 8 + j];
#pragma unroll
            for (int i = 0; i < 8; ++i)
#pragma unroll
                for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(ra[i], rb[j], acc[i][j]);
        }
        __syncthreads();
    }
    float* out = partial + (int64_t)blockIdx.y * t * t;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const int64_t gi = (int64_t)ti * kGT + ty * 8 + i;
        if (gi >= t) continue;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int64_t gj = (int64_t)tj * kGT + tx * 8 + j;
            if (gj < t) out[gi * t + gj] = acc[i][j];
        }
    }
}

// sum the K-splits in fp64 (and add to g: accumulate) and mirror the upper triangle
__global__ void __launch_bounds__(256)
gram_reduce_kernel(const float* __restrict__ partial, int splits, int64_t t, int accumulate, double* __restrict__ g) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= t * t) return;
    const int64_t i = e / t, j = e % t;
    const int64_t ti = i / kGT, tj = j / kGT;
    // tiles with ti <= tj were computed; take (i,j) from there, or its transpose
    const int64_t src = (ti <= tj) ? (i * t + j) : (j * t + i);
    double acc = accumulate ? g[e] : 0.0;
    for (int s = 0; s < splits; ++s) acc += (double)partial[(int64_t)s * t * t + src];
    g[e] = acc;
}

// ---------------------------------------------------------------- projection: U[m][j] = sum_t (a[m][t] - mu_m) * vs[t][j]
constexpr int kPM = 128, kPN = 64, kPK = 16;

__global__ void __launch_bounds__(256)
project_kernel(const float* __restrict__ a, const float* __restrict__ mean, const float* __restrict__ vs, int64_t m,
               int64_t t, int r, float* __restrict__ u) {
    __shared__ float sa[kPK][kPM + 1];
    __shared__ float sv[kPK][kPN];
    const int64_t row0 = (int64_t)blockIdx.x * kPM;
    const int col0 = blockIdx.y * kPN;
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;      // 16 x 16 threads: 8 rows x 4 cols each
    float acc[8][4];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
    for (int64_t k0 = 0; k0 < t; k0 += kPK) {
        for (int e = threadIdx.x; e < kPM * kPK; e += 256) {
            const int rr = e / kPK, kk = e % kPK;                 // consecutive threads read consecutive t of one row
            const int64_t row = row0 + rr, tt = k0 + kk;
            float v = 0.f;
            if (row < m && tt < t) v = a[row * t + tt] - mean[row];
            sa[kk][rr] = v;
        }
        for (int e = threadIdx.x; e < kPK * kPN; e += 256) {
            const int kk = e / kPN, c = e % kPN;
            const int64_t tt = k0 + kk;
            sv[kk][c] = (tt < t && col0 + c < r) ? vs[tt * r + col0 + c] : 0.f;
        }
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < kPK; ++kk) {
            float ra[8], rb[4];
#pragma unroll
            for (int i = 0; i < 8; ++i) ra[i] = sa[kk][ty * 8 + i];
#pragma unroll
            for (int j = 0; j < 4; ++j) rb[j] = sv[kk][tx * 4 + j];
#pragma unroll
            for (int i = 0; i < 8; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(ra[i], rb[j], acc[i][j]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const int64_t row = row0 + ty * 8 + i;
        if (row >= m) continue;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int c = col0 + tx * 4 + j;
            if (c < r) u[row * r + c] = acc[i][j];
        }
    }
}


// ================================================================== tensor-core Gram (tcgen05 / TMEM / TMA)
constexpr int kTcBM = 128;                                   // rows of a G tile = UMMA M (TMEM lanes)
constexpr int kTcBN = 256;                                   // columns of a G tile = UMMA N (TMEM columns)
constexpr int kTcKB = 16;                                    // rows of the planes per pipeline stage (2 UMMA K-steps)
constexpr int kTcStages = 4;
constexpr int kTcGroupBytes = kTcKB * 128;                   // one 32-column group of a stage: KB rows x 128 B
constexpr int kTcABytes = (kTcBM / 32) * kTcGroupBytes;      // 8 KB
constexpr int kTcBBytes = (kTcBN / 32) * kTcGroupBytes;      // 16 KB
constexpr int kTcStageBytes = 2 * (kTcABytes + kTcBBytes);   // [A_hi][A_lo][B_hi][B_lo] = 48 KB
constexpr int kTcEpiWarps = 8;                               // two warps per TMEM lane quarter, 128 columns each
constexpr int kTcThreads = (2 + kTcEpiWarps) * 32;           // warp 0 TMA, warp 1 MMA + TMEM alloc, warps 2..9 epilogue
constexpr int kTcTmemCols = 2 * kTcBN;                       // two accumulator buffers
constexpr size_t kTcSmemBytes = (size_t)kTcStages * kTcStageBytes + 1024;
int g_tc_seg_kblocks = 8;      // K-blocks accumulated in TMEM before the epilogue takes over (s3_set_tuning key 10)
int g_tc_pair = 1;             // clusters of two CTAs sharing B via TMA multicast (s3_set_tuning key 14)
int g_tc_flush_segments = 128;  // TMEM segments summed in fp32 registers per fp64 flush (s3_set_tuning key 11)
int g_plane_rows_cap = 0;       // rows per plane chunk of gram_tc / project_tc at most (key 17; tests reach the chunked
                                // accumulation at small sizes), 0 = planes of up to 2 GB

// Centre, scale and split the rows [row0, row0 + n_rows) of A into TF32 planes, layout [n_groups][plane_rows][32]:
//   b = (a - mean) * sqrt(vol);  (hi, lo) = tf32_split(b).
// Rows past `m` and columns past `t` are written as zeros. One warp per row.
__global__ void __launch_bounds__(256)
gram_prepare_kernel(const float* __restrict__ a, const float* __restrict__ mean, const float* __restrict__ vol,
                    int vol_div, int64_t row0, int64_t n_rows_pad, int64_t m, int64_t t, int n_groups,
                    int64_t plane_rows, float* __restrict__ hi, float* __restrict__ lo) {
    const int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (r >= n_rows_pad) return;
    const int64_t row = row0 + r;
    const bool live = row < m;
    float mu = 0.f, s = 0.f;
    if (live) {
        mu = mean[row];
        s = sqrtf(vol[row / vol_div]);
    }
    const float* p = a + row * t;
    for (int g = 0; g < n_groups; ++g) {
        const int64_t c = (int64_t)g * 32 + lane;
        float b = 0.f;
        if (live && c < t) b = (p[c] - mu) * s;
        float h, l;
        tf32_split(b, h, l);
        const int64_t o = ((int64_t)g * plane_rows + r) * 32 + lane;
        hi[o] = h;
        if (lo) lo[o] = l;
    }
}

// TF32 planes [n_i_pad][n_c_pad] of a strided fp32 matrix: (hi, lo)[i][c] = tf32_split(src[i * s_i + c * s_c]) for
// i < n_i, c < n_c, zeros in the padding; no lo plane when `lo` is NULL. The K-major operands W^T = (V / s)^T of the
// projection and left / right_t of the low-rank residual.
__global__ void __launch_bounds__(256)
tf32_split_kernel(const float* __restrict__ src, int64_t s_i, int64_t s_c, int64_t n_i, int64_t n_c, int64_t n_i_pad,
                  int64_t n_c_pad, float* __restrict__ hi, float* __restrict__ lo) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n_i_pad * n_c_pad) return;
    const int64_t i = e / n_c_pad, c = e % n_c_pad;
    float h, l;
    tf32_split((i < n_i && c < n_c) ? src[i * s_i + c * s_c] : 0.f, h, l);
    hi[e] = h;
    if (lo) lo[e] = l;
}

// first j-tile (256 columns) that reaches the upper triangle of i-tile ti (128 rows)
__host__ __device__ __forceinline__ int tc_first_tj(int ti) { return (ti * kTcBM) / kTcBN; }

// paired mode: tiles are enumerated j-tile major, i-tiles 0 .. 2 tj + 1 of a j-tile (an even count when T is padded to
// 256 columns), so that the two CTAs of a cluster work on (2p, tj) and (2p + 1, tj) and share the B operand
__host__ __device__ __forceinline__ int tc_pair_count(int tj, int n_i) { return (2 * tj + 2) < n_i ? (2 * tj + 2) : n_i; }

// One CTA per (G tile, K split). partial: fp64 [n_items][kTcBN][kTcBM] (column of the tile major, rows contiguous).
// PAIR: clusters of two CTAs whose tiles share the 256 columns of B: each CTA fetches half of every B stage and TMA
// multicasts it into both shared memories (L2 -> SM operand traffic 32 KB instead of 48 KB per CTA and stage -- the
// single-CTA kernel is bound by exactly that traffic); a stage is released to both producers by multicast commits.
template <bool PAIR>
__global__ void __launch_bounds__(kTcThreads, 1)
gram_tc_kernel(const __grid_constant__ CUtensorMap map_hi, const __grid_constant__ CUtensorMap map_lo, int n_i, int n_j,
               int splits, int n_kblocks, int seg_kblocks, int flush_segments, int passes, double* __restrict__ partial) {
    extern __shared__ __align__(1024) unsigned char tc_smem_raw[];
    __shared__ __align__(8) uint64_t full_bar[kTcStages];
    __shared__ __align__(8) uint64_t empty_bar[kTcStages];
    __shared__ __align__(8) uint64_t acc_full_bar[2];
    __shared__ __align__(8) uint64_t acc_empty_bar[2];
    __shared__ uint32_t tmem_base_slot;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    // 1024-byte aligned stage ring (the 128B swizzle pattern is a function of the address bits [7,10))
    const uint32_t raw = smem_u32(tc_smem_raw);
    const uint32_t ring = (raw + 1023u) & ~1023u;
    unsigned char* ring_ptr = tc_smem_raw + (ring - raw);

    // work item -> (ti, tj, split)
    const uint32_t rank = PAIR ? cluster_rank() : 0u;
    int item, tile, split, ti = 0, tj = 0;
    if (PAIR) {
        const int cl = blockIdx.x >> 1;
        split = cl % splits;
        tile = 2 * (cl / splits) + (int)rank;
        int acc_tiles = 0;
        while (tj < n_j) {
            const int cnt = tc_pair_count(tj, n_i);
            if (tile < acc_tiles + cnt) break;
            acc_tiles += cnt;
            ++tj;
        }
        ti = tile - acc_tiles;
        item = tile * splits + split;
    } else {
        item = blockIdx.x;
        tile = item / splits;
        split = item % splits;
        int acc_tiles = 0;
        while (ti < n_i) {
            const int cnt = n_j - tc_first_tj(ti);
            if (tile < acc_tiles + cnt) break;
            acc_tiles += cnt;
            ++ti;
        }
        tj = tc_first_tj(ti) + (tile - acc_tiles);
    }
    const int per_split = (n_kblocks + splits - 1) / splits;
    const int kb0 = split * per_split;
    const int kb1 = (kb0 + per_split) < n_kblocks ? (kb0 + per_split) : n_kblocks;
    const int n_kb = kb1 > kb0 ? (kb1 - kb0) : 0;
    const int n_seg = (n_kb + seg_kblocks - 1) / seg_kblocks;

    if (threadIdx.x == 0) {
        for (int s = 0; s < kTcStages; ++s) {
            mbar_init(&full_bar[s], 1);
            mbar_init(&empty_bar[s], PAIR ? 2 : 1);            // paired: both CTAs' MMAs must be done with the stage
        }
        for (int b = 0; b < 2; ++b) {
            mbar_init(&acc_full_bar[b], 1);
            mbar_init(&acc_empty_bar[b], kTcEpiWarps * 32);
        }
        tma_prefetch(&map_hi);
        tma_prefetch(&map_lo);
    }
    if (warp == 1) tmem_alloc(&tmem_base_slot, (uint32_t)kTcTmemCols);
    tc_fence_before();
    __syncthreads();
    if (PAIR) cluster_sync_all();                          // the peer's barriers exist before anything arrives on them
    tc_fence_after();
    const uint32_t tmem_base = tmem_base_slot;

    if (warp == 0) {
        // ------------------------------------------------------------------ TMA producer (one thread)
        if (lane == 0) {
            const uint32_t stage_tx = (uint32_t)(passes == 3 ? kTcStageBytes : kTcStageBytes / 2);
            for (int it = 0; it < n_kb; ++it) {
                const int s = it % kTcStages;
                const uint32_t round = (uint32_t)(it / kTcStages);
                if (round > 0) mbar_wait_wd(&empty_bar[s], (round - 1) & 1u);
                unsigned char* st = ring_ptr + (size_t)s * kTcStageBytes;
                const int row = (kb0 + it) * kTcKB;
                mbar_expect_tx(&full_bar[s], stage_tx);
                tma_load_3d(st, &map_hi, 0, row, ti * (kTcBM / 32), &full_bar[s]);
                if (passes == 3) tma_load_3d(st + kTcABytes, &map_lo, 0, row, ti * (kTcBM / 32), &full_bar[s]);
                if (PAIR) {
                    // my half of B (4 of its 8 column groups) goes to both CTAs; the other half arrives from the peer
                    const int g = tj * (kTcBN / 32) + 4 * (int)rank;
                    const size_t off = (size_t)rank * (kTcBBytes / 2);
                    tma_load_3d_multicast(st + 2 * kTcABytes + off, &map_hi, 0, row, g, &full_bar[s], 0x3);
                    if (passes == 3)
                        tma_load_3d_multicast(st + 2 * kTcABytes + kTcBBytes + off, &map_lo, 0, row, g, &full_bar[s], 0x3);
                } else {
                    tma_load_3d(st + 2 * kTcABytes, &map_hi, 0, row, tj * (kTcBN / 32), &full_bar[s]);
                    tma_load_3d(st + 2 * kTcABytes + kTcBBytes / 2, &map_hi, 0, row, tj * (kTcBN / 32) + 4, &full_bar[s]);
                    if (passes == 3) {
                        tma_load_3d(st + 2 * kTcABytes + kTcBBytes, &map_lo, 0, row, tj * (kTcBN / 32), &full_bar[s]);
                        tma_load_3d(st + 2 * kTcABytes + kTcBBytes + kTcBBytes / 2, &map_lo, 0, row, tj * (kTcBN / 32) + 4,
                                    &full_bar[s]);
                    }
                }
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        // ------------------------------------------------------------------ MMA issuer (one thread)
        if (lane == 0) {
            constexpr uint32_t idesc = umma_idesc_tf32_mn(kTcBM, kTcBN);
            int it = 0;
            for (int seg = 0; seg < n_seg; ++seg) {
                const int b = seg & 1;
                if (seg >= 2) {
                    mbar_wait_wd(&acc_empty_bar[b], (uint32_t)((seg >> 1) - 1) & 1u);
                    tc_fence_after();
                }
                const uint32_t d_tmem = tmem_base + (uint32_t)(b * kTcBN);
                const int seg_end = (seg + 1) * seg_kblocks < n_kb ? (seg + 1) * seg_kblocks : n_kb;
                uint32_t accumulate = 0;
                for (; it < seg_end; ++it) {
                    const int s = it % kTcStages;
                    mbar_wait_wd(&full_bar[s], (uint32_t)(it / kTcStages) & 1u);
                    tc_fence_after();
                    const uint32_t st = ring + (uint32_t)s * kTcStageBytes;
#pragma unroll
                    for (int ks = 0; ks < kTcKB / 8; ++ks) {
                        const uint32_t koff = (uint32_t)ks * 1024u;
                        const uint64_t a_hi = umma_desc_mn_sw128_32b(st + koff, kTcGroupBytes, 512);
                        const uint64_t b_hi = umma_desc_mn_sw128_32b(st + 2 * kTcABytes + koff, kTcGroupBytes, 512);
                        if (passes == 3) {
                            const uint64_t a_lo = umma_desc_mn_sw128_32b(st + kTcABytes + koff, kTcGroupBytes, 512);
                            const uint64_t b_lo =
                                umma_desc_mn_sw128_32b(st + 2 * kTcABytes + kTcBBytes + koff, kTcGroupBytes, 512);
                            umma_tf32(d_tmem, a_lo, b_hi, idesc, accumulate);
                            umma_tf32(d_tmem, a_hi, b_lo, idesc, 1u);
                            umma_tf32(d_tmem, a_hi, b_hi, idesc, 1u);
                        } else {
                            umma_tf32(d_tmem, a_hi, b_hi, idesc, accumulate);
                        }
                        accumulate = 1u;
                    }
                    // the stage is free once these MMAs have read it (paired: tell both producers)
                    if (PAIR) umma_commit_multicast(&empty_bar[s], 0x3);
                    else umma_commit(&empty_bar[s]);
                }
                umma_commit(&acc_full_bar[b]);         // the segment's accumulator is complete
            }
        }
        __syncwarp();
    } else {
        // ------------------------------------------------------------------ epilogue warps
        // The tensor core adds into its fp32 accumulator with truncation, so a long accumulation chain drifts
        // (measured: 2e-5 relative after 768 MMAs). The MMA thread therefore accumulates only `seg_kblocks` stages
        // in TMEM; the epilogue warps pull every finished segment into fp32 registers (round-to-nearest adds) and
        // move the running sums to the fp64 partials every `flush_segments` segments.
        const int q = warp & 3;                        // TMEM lane quarter this warp may access
        const int half = (warp - 2) >> 2;              // which 128 of the tile's 256 columns
        const int row = q * 32 + lane;                 // row of the G tile
        double* out = partial + ((size_t)item * kTcBN + (size_t)half * (kTcBN / 2)) * kTcBM + row;
        float acc[kTcBN / 2];
#pragma unroll
        for (int c = 0; c < kTcBN / 2; ++c) acc[c] = 0.f;
        bool first_flush = true;
        int pending = 0;
        for (int seg = 0; seg < n_seg; ++seg) {
            const int b = seg & 1;
            mbar_wait_wd(&acc_full_bar[b], (uint32_t)(seg >> 1) & 1u);
            tc_fence_after();
            const uint32_t taddr =
                tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(b * kTcBN + half * (kTcBN / 2));
#pragma unroll
            for (int c0 = 0; c0 < kTcBN / 2; c0 += 32) {
                uint32_t v[32];
                tmem_ld32(taddr + (uint32_t)c0, v);
#pragma unroll
                for (int c = 0; c < 32; ++c) acc[c0 + c] = __fadd_rn(acc[c0 + c], __uint_as_float(v[c]));
            }
            // everything of this buffer is in registers: hand it back to the MMA thread
            tc_fence_before();
            mbar_arrive_cta(&acc_empty_bar[b]);
            if (++pending == flush_segments || seg + 1 == n_seg) {
                if (first_flush) {
#pragma unroll
                    for (int c = 0; c < kTcBN / 2; ++c) out[(size_t)c * kTcBM] = (double)acc[c];
                } else {
#pragma unroll
                    for (int c = 0; c < kTcBN / 2; ++c) out[(size_t)c * kTcBM] += (double)acc[c];
                }
#pragma unroll
                for (int c = 0; c < kTcBN / 2; ++c) acc[c] = 0.f;
                first_flush = false;
                pending = 0;
            }
        }
        if (n_seg == 0) {
#pragma unroll 1
            for (int c = 0; c < kTcBN / 2; ++c) out[(size_t)c * kTcBM] = 0.0;
        }
    }
    tc_fence_before();
    __syncthreads();
    if (PAIR) cluster_sync_all();                          // the peer may still multicast into / arrive on this CTA
    if (warp == 1) tmem_dealloc(tmem_base, (uint32_t)kTcTmemCols);
}

// G[i][j] (+)= sum over splits of the tile partials; both triangles are written from the same upper-triangle entry.
__global__ void __launch_bounds__(256)
gram_tc_reduce_kernel(const double* __restrict__ partial, int splits, int n_i, int n_j, int64_t t, int accumulate,
                      int paired, double* __restrict__ g) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= t * t) return;
    int64_t i = e / t, j = e % t;
    if (j < i) { const int64_t x = i; i = j; j = x; }
    const int ti = (int)(i / kTcBM), tj = (int)(j / kTcBN);
    int tile = 0;
    if (paired) {
        for (int u = 0; u < tj; ++u) tile += tc_pair_count(u, n_i);
        tile += ti;
    } else {
        for (int u = 0; u < ti; ++u) tile += n_j - tc_first_tj(u);
        tile += tj - tc_first_tj(ti);
    }
    const double* p = partial + ((size_t)tile * splits * kTcBN + (size_t)(j % kTcBN)) * kTcBM + (size_t)(i % kTcBM);
    double acc = accumulate ? g[e] : 0.0;
    for (int s = 0; s < splits; ++s) acc += p[(size_t)s * kTcBN * kTcBM];
    g[e] = acc;
}

// ================================================================== tensor-core projection
//   U[m][j] = (1 / sqrt(vol_m)) * sum_t B[m][t] * W[t][j],   B = sqrt(vol) (A - mean) (the planes of the Gram kernel),
//   W = V / s  [T, r]
// Here the contraction runs over t, which is the contiguous direction of the planes ([T/32][rows][32]): a TMA box of
// {32 t, 128 rows} written with the plain 128B swizzle is the canonical K-major UMMA tile (8-row x 128-byte atoms,
// SBO = 1024), and W is passed transposed ([r_pad][T_pad], t contiguous) so that it is K-major as well. One CTA per
// 128 rows: warp 0 = TMA producer, warp 1 = MMA issuer (3xTF32: B_l W_h + B_h W_l + B_h W_h), warps 2..5 = epilogue
// (tcgen05.ld, scale by 1/sqrt(vol), store the r columns of the row). Accumulator: 128 lanes x r_pad TMEM columns.
constexpr int kPjBM = 128;
constexpr int kPjStages = 2;
constexpr int kPjThreads = 6 * 32;
constexpr int kPjABytes = kPjBM * 128;                       // one plane tile: 128 rows x 32 floats
// 32-column groups per TMEM segment at most (3xTF32: 384 MMAs, the chain length of T = 2000 at r = 256); longer t ranges
// run as several launches that add into U. One launch with two segments of 128 / 256 groups (r = 256, T = 8192 / 16 384)
// measured 3.2e-5 / 5.1e-5 of the largest entry on a B200, split launches 7e-6 (tests/test_svd_scale_gpu.py).
constexpr int kPjSegGroups = 32;

__global__ void __launch_bounds__(kPjThreads, 1)
project_tc_kernel(const __grid_constant__ CUtensorMap map_hi, const __grid_constant__ CUtensorMap map_lo,
                  const __grid_constant__ CUtensorMap map_whi, const __grid_constant__ CUtensorMap map_wlo, int g0,
                  int n_groups, int r_pad, int tmem_cols, int n_seg, int passes, const float* __restrict__ vol, int vol_div,
                  int64_t row0, int64_t m, int r, int col0, int add, float* __restrict__ u) {
    extern __shared__ __align__(1024) unsigned char pj_smem_raw[];
    __shared__ __align__(8) uint64_t full_bar[kPjStages];
    __shared__ __align__(8) uint64_t empty_bar[kPjStages];
    __shared__ __align__(8) uint64_t acc_bar;
    __shared__ uint32_t tmem_base_slot;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t raw = smem_u32(pj_smem_raw);
    const uint32_t ring = (raw + 1023u) & ~1023u;
    unsigned char* ring_ptr = pj_smem_raw + (ring - raw);
    const uint32_t w_bytes = (uint32_t)r_pad * 128u;                  // one W^T tile: r_pad rows x 32 floats
    const uint32_t stage_bytes = 2u * kPjABytes + 2u * w_bytes;       // [B_hi][B_lo][W_hi][W_lo]
    const int tile_row = blockIdx.x * kPjBM;                          // first plane row of this CTA

    if (threadIdx.x == 0) {
        for (int s = 0; s < kPjStages; ++s) {
            mbar_init(&full_bar[s], 1);
            mbar_init(&empty_bar[s], 1);
        }
        mbar_init(&acc_bar, 1);
        tma_prefetch(&map_hi);
        tma_prefetch(&map_whi);
    }
    if (warp == 1) tmem_alloc(&tmem_base_slot, (uint32_t)tmem_cols);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_base_slot;

    if (warp == 0) {
        if (lane == 0) {
            const uint32_t tx = passes == 3 ? stage_bytes : (kPjABytes + w_bytes);
            for (int g = 0; g < n_groups; ++g) {
                const int s = g % kPjStages;
                const uint32_t round = (uint32_t)(g / kPjStages);
                if (round > 0) mbar_wait_wd(&empty_bar[s], (round - 1) & 1u);
                unsigned char* st = ring_ptr + (size_t)s * stage_bytes;
                mbar_expect_tx(&full_bar[s], tx);
                tma_load_3d(st, &map_hi, 0, tile_row, g0 + g, &full_bar[s]);
                tma_load_2d(st + 2 * kPjABytes, &map_whi, (g0 + g) * 32, 0, &full_bar[s]);
                if (passes == 3) {
                    tma_load_3d(st + kPjABytes, &map_lo, 0, tile_row, g0 + g, &full_bar[s]);
                    tma_load_2d(st + 2 * kPjABytes + w_bytes, &map_wlo, (g0 + g) * 32, 0, &full_bar[s]);
                }
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        if (lane == 0) {
            const uint32_t idesc = umma_idesc_tf32_k(kPjBM, r_pad);
            // The tensor core's fp32 accumulation truncates, so the error grows with the length of the chain: the t
            // range is cut into n_seg segments with their own TMEM columns, summed (round to nearest) in the epilogue.
            const int per_seg = (n_groups + n_seg - 1) / n_seg;
            uint32_t accumulate = 0;
            for (int g = 0; g < n_groups; ++g) {
                const int s = g % kPjStages;
                mbar_wait_wd(&full_bar[s], (uint32_t)(g / kPjStages) & 1u);
                tc_fence_after();
                const uint32_t st = ring + (uint32_t)s * stage_bytes;
                const uint32_t d_tmem = tmem_base + (uint32_t)((g / per_seg) * r_pad);
                if (g % per_seg == 0) accumulate = 0;
                umma_stage_k(d_tmem, st, st + kPjABytes, st + 2 * kPjABytes, st + 2 * kPjABytes + w_bytes, idesc, passes,
                             accumulate);
                accumulate = 1u;
                umma_commit(&empty_bar[s]);
            }
            umma_commit(&acc_bar);
        }
        __syncwarp();
    } else {
        const int q = warp & 3;                                       // TMEM lane quarter of this warp
        const int64_t row = row0 + tile_row + q * 32 + lane;
        mbar_wait_wd(&acc_bar, 0);
        tc_fence_after();
        const float scale = row < m ? rsqrtf(vol[row / vol_div]) : 0.f;
        const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16);
        const int per_seg = (n_groups + n_seg - 1) / n_seg;
        const int used_seg = (n_groups + per_seg - 1) / per_seg;      // segments that received at least one stage
        for (int c0 = 0; c0 < r_pad; c0 += 32) {
            float acc[32];
#pragma unroll
            for (int c = 0; c < 32; ++c) acc[c] = 0.f;
            for (int sg = 0; sg < used_seg; ++sg) {
                uint32_t v[32];
                tmem_ld32(taddr + (uint32_t)(sg * r_pad + c0), v);    // warp-collective: all lanes, also dead rows
#pragma unroll
                for (int c = 0; c < 32; ++c) acc[c] = __fadd_rn(acc[c], __uint_as_float(v[c]));
            }
            if (row < m) {
                float* o = u + row * r + col0 + c0;
#pragma unroll
                for (int c = 0; c < 32; ++c)
                    if (col0 + c0 + c < r) o[c] = add ? __fadd_rn(o[c], acc[c] * scale) : acc[c] * scale;
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem_base, (uint32_t)tmem_cols);
}

// ================================================================== residual of a low-rank model (s3_lowrank_error)
//   e[m][t] = (a[m][t] - mean[m]) - sum_j left[m][j] * right_t[t][j],   j < q <= 512
// The product runs on tcgen05 with the operand forms of project_tc_kernel: left (K = q contiguous) takes the role of the
// planes, right_t the role of W^T; both are split into TF32 hi / lo planes ([rows_pad][q_pad], zero padded) by
// tf32_split_kernel and contracted 3xTF32 into one 128 x 256 fp32 tile in TMEM (q_pad / 8 * 3 <= 192 MMAs, one
// segment). The epilogue warps pull the tile with tcgen05.ld, read the matching 128 x 256 tile of `a` from HBM once and
// form e in fp64. Work unit: a row tile (128 rows) over ALL column tiles, so that the row sums stay in registers of one
// CTA; row tiles are dealt out in fixed groups of consecutive tiles (the grouping depends on m only), a group's column
// partials are added up by one thread per column in tile order, and a second kernel sums the groups in group order:
// the results do not depend on the number of CTAs. Accumulator double-buffered in TMEM (2 x 256 columns), so the MMAs of
// the next column tile run under the epilogue of this one. Warp 0 = TMA, warp 1 = MMA, warps 2..5 = epilogue (one per
// TMEM lane quarter; with eight, the register budget of 10 warps per SM spilled the fp64 reductions).
constexpr int kLrBM = 128, kLrBN = 256, kLrMaxQ = 512;
constexpr int kLrStages = 2;
constexpr int kLrABytes = kLrBM * 128;                       // 128 rows x 32 floats
constexpr int kLrBBytes = kLrBN * 128;                       // 256 rows x 32 floats
constexpr int kLrStageBytes = 2 * (kLrABytes + kLrBBytes);   // [A_hi][A_lo][B_hi][B_lo] = 96 KB
constexpr int kLrEpiWarps = 4;                               // one per TMEM lane quarter (6 warps: up to 255 registers)
constexpr int kLrThreads = (2 + kLrEpiWarps) * 32;
constexpr int kLrTmemCols = 2 * kLrBN;
constexpr size_t kLrSmemBytes = (size_t)kLrStages * kLrStageBytes + 1024;
constexpr int kLrMaxGroups = 1024;                           // row-tile groups at most (scratch: groups x 3 x vol_div x t)
int g_lowrank_cap = 0;                                       // CTAs at most (s3x_tune key 19; tests), 0 = one per SM

// Sum over the 32 lanes of a warp of each of 32 columns, value(j) = this lane's entry of column j (reduce-scatter
// butterfly, 31 shuffles): returns the sum (max: the maximum) of column `lane`. The order of the adds is fixed by the lane
// numbers. The first step consumes the values as they are formed, so only 16 partials are ever live.
template <typename F>
__device__ __forceinline__ double warp_column_reduce(F value, bool max, int lane) {
    double v[16];
    {
        const bool upper = (lane & 16) != 0;
#pragma unroll
        for (int i = 0; i < 16; ++i) {
            const double lo = value(i), hi = value(i + 16);
            const double recv = shfl_xor_d(upper ? lo : hi, 16);
            v[i] = max ? fmax(upper ? hi : lo, recv) : (upper ? hi : lo) + recv;
        }
    }
#pragma unroll
    for (int k = 8; k >= 1; k >>= 1) {
        const bool upper = (lane & k) != 0;
#pragma unroll
        for (int i = 0; i < k; ++i) {
            const double send = upper ? v[i] : v[i + k];
            const double keep = upper ? v[i + k] : v[i];
            const double recv = shfl_xor_d(send, k);
            v[i] = max ? fmax(keep, recv) : keep + recv;
        }
    }
    return v[0];
}

// part: fp64 [n_groups][3][vol_div][t] (sq_err, sq_ref, max_abs of the group's rows)
__global__ void __launch_bounds__(kLrThreads, 1)
lowrank_error_kernel(const __grid_constant__ CUtensorMap map_lhi, const __grid_constant__ CUtensorMap map_llo,
                     const __grid_constant__ CUtensorMap map_rhi, const __grid_constant__ CUtensorMap map_rlo,
                     const float* __restrict__ a, const float* __restrict__ mean, const float* __restrict__ vol,
                     int vol_div, int64_t m, int64_t t, int n_kgroups, int n_ct, int64_t n_rt, int64_t tiles_per_group,
                     int64_t n_groups, double* __restrict__ part, double* __restrict__ row_sq_err) {
    extern __shared__ __align__(1024) unsigned char lr_smem_raw[];
    __shared__ __align__(8) uint64_t full_bar[kLrStages];
    __shared__ __align__(8) uint64_t empty_bar[kLrStages];
    __shared__ __align__(8) uint64_t acc_full_bar[2];
    __shared__ __align__(8) uint64_t acc_empty_bar[2];
    __shared__ uint32_t tmem_base_slot;
    __shared__ double red[4][3][32];                         // [lane quarter][quantity][column]

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t raw = smem_u32(lr_smem_raw);
    const uint32_t ring = (raw + 1023u) & ~1023u;
    unsigned char* ring_ptr = lr_smem_raw + (ring - raw);

    if (threadIdx.x == 0) {
        for (int s = 0; s < kLrStages; ++s) {
            mbar_init(&full_bar[s], 1);
            mbar_init(&empty_bar[s], 1);
        }
        for (int b = 0; b < 2; ++b) {
            mbar_init(&acc_full_bar[b], 1);
            mbar_init(&acc_empty_bar[b], kLrEpiWarps * 32);
        }
        tma_prefetch(&map_lhi);
        tma_prefetch(&map_rhi);
    }
    if (warp == 1) tmem_alloc(&tmem_base_slot, (uint32_t)kLrTmemCols);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_base_slot;

    if (warp == 0) {
        if (lane == 0) {
            int it = 0;
            for (int64_t grp = blockIdx.x; grp < n_groups; grp += gridDim.x) {
                const int64_t rt1 = (grp + 1) * tiles_per_group < n_rt ? (grp + 1) * tiles_per_group : n_rt;
                for (int64_t rt = grp * tiles_per_group; rt < rt1; ++rt)
                    for (int ct = 0; ct < n_ct; ++ct)
                        for (int g = 0; g < n_kgroups; ++g, ++it) {
                            const int s = it % kLrStages;
                            const uint32_t round = (uint32_t)(it / kLrStages);
                            if (round > 0) mbar_wait_wd(&empty_bar[s], (round - 1) & 1u);
                            unsigned char* st = ring_ptr + (size_t)s * kLrStageBytes;
                            mbar_expect_tx(&full_bar[s], (uint32_t)kLrStageBytes);
                            tma_load_2d(st, &map_lhi, g * 32, (int)(rt * kLrBM), &full_bar[s]);
                            tma_load_2d(st + kLrABytes, &map_llo, g * 32, (int)(rt * kLrBM), &full_bar[s]);
                            tma_load_2d(st + 2 * kLrABytes, &map_rhi, g * 32, ct * kLrBN, &full_bar[s]);
                            tma_load_2d(st + 2 * kLrABytes + kLrBBytes, &map_rlo, g * 32, ct * kLrBN, &full_bar[s]);
                        }
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        if (lane == 0) {
            constexpr uint32_t idesc = umma_idesc_tf32_k(kLrBM, kLrBN);
            int it = 0, item = 0;
            for (int64_t grp = blockIdx.x; grp < n_groups; grp += gridDim.x) {
                const int64_t rt1 = (grp + 1) * tiles_per_group < n_rt ? (grp + 1) * tiles_per_group : n_rt;
                for (int64_t rt = grp * tiles_per_group; rt < rt1; ++rt)
                    for (int ct = 0; ct < n_ct; ++ct, ++item) {
                        const int b = item & 1;
                        if (item >= 2) {
                            mbar_wait_wd(&acc_empty_bar[b], (uint32_t)((item >> 1) - 1) & 1u);
                            tc_fence_after();
                        }
                        const uint32_t d_tmem = tmem_base + (uint32_t)(b * kLrBN);
                        uint32_t accumulate = 0;
                        for (int g = 0; g < n_kgroups; ++g, ++it) {
                            const int s = it % kLrStages;
                            mbar_wait_wd(&full_bar[s], (uint32_t)(it / kLrStages) & 1u);
                            tc_fence_after();
                            const uint32_t st = ring + (uint32_t)s * kLrStageBytes;
                            umma_stage_k(d_tmem, st, st + kLrABytes, st + 2 * kLrABytes, st + 2 * kLrABytes + kLrBBytes,
                                         idesc, 3, accumulate);
                            accumulate = 1u;
                            umma_commit(&empty_bar[s]);
                        }
                        umma_commit(&acc_full_bar[b]);
                    }
            }
        }
        __syncwarp();
    } else {
        const int qd = warp & 3;                             // TMEM lane quarter
        // 16-byte row loads when every row starts 16-byte aligned (a lane reads its own row: a quarter of the load
        // instructions of the scalar path, each touching the same 32 rows)
        const bool vec4 = t % 4 == 0 && (reinterpret_cast<uintptr_t>(a) & 15) == 0;
        int item = 0;
        for (int64_t grp = blockIdx.x; grp < n_groups; grp += gridDim.x) {
            const int64_t rt0 = grp * tiles_per_group;
            const int64_t rt1 = rt0 + tiles_per_group < n_rt ? rt0 + tiles_per_group : n_rt;
            for (int64_t rt = rt0; rt < rt1; ++rt) {
                const int64_t row = rt * kLrBM + qd * 32 + lane;
                const bool live = row < m;
                const double mu = (live && mean) ? (double)mean[row] : 0.0;
                const double w = live ? (vol ? (double)vol[row / vol_div] : 1.0) : 0.0;
                const int comp = (int)(row % vol_div);
                const float* arow = a + (live ? row : 0) * t;
                double row_acc = 0.0;
                for (int ct = 0; ct < n_ct; ++ct, ++item) {
                    const int b = item & 1;
                    const uint32_t taddr = tmem_base + ((uint32_t)(qd * 32) << 16) + (uint32_t)(b * kLrBN);
#pragma unroll 1
                    for (int c0 = 0; c0 < kLrBN; c0 += 32) {
                        const int64_t col0 = (int64_t)ct * kLrBN + c0;
                        float av[32];
                        if (vec4) {                                       // t % 4 == 0: a float4 is all in or all out
#pragma unroll
                            for (int j = 0; j < 32; j += 4) {
                                const float4 v = (live && col0 + j < t) ? __ldg(reinterpret_cast<const float4*>(arow + col0 + j))
                                                                        : make_float4(0.f, 0.f, 0.f, 0.f);
                                av[j] = v.x; av[j + 1] = v.y; av[j + 2] = v.z; av[j + 3] = v.w;
                            }
                        } else {
#pragma unroll
                            for (int j = 0; j < 32; ++j) av[j] = (live && col0 + j < t) ? __ldg(arow + col0 + j) : 0.f;
                        }
                        if (c0 == 0) {                                    // (the first loads are in flight meanwhile)
                            mbar_wait_wd(&acc_full_bar[b], (uint32_t)(item >> 1) & 1u);
                            tc_fence_after();
                        }
                        uint32_t pv[32];
                        tmem_ld32(taddr + (uint32_t)c0, pv);             // warp-collective: all lanes, also dead rows
                        if (c0 + 32 == kLrBN) {                       // the whole buffer is in registers
                            tc_fence_before();
                            mbar_arrive_cta(&acc_empty_bar[b]);
                        }
                        // the residual is formed in fp64 (no cancellation between a - mean and the product) and kept
                        // rounded to fp32 (6e-8 of itself) for the reductions, which square and sum it in fp64; an fp64
                        // copy of the chunk does not fit beside the butterfly in 255 registers. 0 past column t.
                        float e[32];
#pragma unroll
                        for (int j = 0; j < 32; ++j) {
                            e[j] = col0 + j < t ? (float)(((double)av[j] - mu) - (double)__uint_as_float(pv[j])) : 0.f;
                            row_acc = fma((double)e[j], (double)e[j], row_acc);
                        }
                        const bool first = rt == rt0;
#pragma unroll 1
                        for (int c = 0; c < vol_div; ++c) {
                            const double wc = comp == c ? w : 0.0;
                            const bool in_c = live && comp == c;
                            // one quantity at a time (k = 0: sum vol e^2, 1: sum vol (a - mean)^2, 2: max |e|): three
                            // independent butterflies in flight at once would not fit the register budget
#pragma unroll 1
                            for (int k = 0; k < 3; ++k)
                                red[qd][k][lane] = warp_column_reduce([&](int j) {
                                    const double x = k == 1 ? (double)av[j] - mu : (double)e[j];
                                    return k == 2 ? (in_c ? fabs(x) : 0.0) : wc * (x * x);
                                }, k == 2, lane);
                            named_bar(1, kLrEpiWarps * 32);
                            // quarters 0..2 each combine one quantity over the four quarters, in order
                            const int64_t col = col0 + lane;
                            if (qd < 3 && col < t) {
                                const double* r4 = &red[0][qd][lane];
                                double sum;
                                if (qd == 2) sum = fmax(fmax(r4[0], r4[3 * 32]), fmax(r4[6 * 32], r4[9 * 32]));
                                else sum = ((r4[0] + r4[3 * 32]) + r4[6 * 32]) + r4[9 * 32];
                                double* o = part + ((grp * 3 + qd) * vol_div + c) * t + col;
                                if (!first) sum = qd == 2 ? fmax(*o, sum) : *o + sum;
                                *o = sum;
                            }
                            named_bar(1, kLrEpiWarps * 32);
                        }
                    }
                }
                if (row_sq_err && live) row_sq_err[row] += row_acc;
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem_base, (uint32_t)kLrTmemCols);
}

// out[k][c][col] = sum (k = 0, 1) / max (k = 2) over the groups, in group order; part [n_groups][3][vol_div][t]
__global__ void __launch_bounds__(256)
lowrank_reduce_kernel(const double* __restrict__ part, int64_t n_groups, int vol_div, int64_t t,
                      double* __restrict__ sq_err, double* __restrict__ sq_ref, double* __restrict__ max_abs) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t n = 3 * (int64_t)vol_div * t;
    if (e >= n) return;
    const int k = (int)(e / ((int64_t)vol_div * t));
    double acc = 0.0;
    for (int64_t g = 0; g < n_groups; ++g) {
        const double v = part[g * n + e];
        acc = k == 2 ? fmax(acc, v) : acc + v;
    }
    const int64_t o = e % ((int64_t)vol_div * t);
    (k == 0 ? sq_err : k == 1 ? sq_ref : max_abs)[o] = acc;
}

}  // namespace s3

using namespace s3;

extern "C" int s3_svd_row_means(const float* d_a, int64_t m, int64_t t, float* d_mean, void* stream) {
    S3_REQUIRE(d_a && d_mean, "s3_svd_row_means: NULL argument");
    S3_REQUIRE(m >= 0 && t >= 1, "s3_svd_row_means: bad sizes");
    if (m == 0) return S3_OK;
    row_mean_kernel<<<(unsigned)ceil_div(m * 32, 256), 256, 0, (cudaStream_t)stream>>>(d_a, m, t, d_mean);
    S3_LAUNCH_CHECK();
    note_launch(1);
    return S3_OK;
}

static int gram_simt(const float* d_a, const float* d_mean, const float* d_vol, int vol_div, int64_t m, int64_t t,
                     double* d_gram, cudaStream_t st) {
    const int tiles = (int)ceil_div(t, kGT);
    const int n_pairs = tiles * (tiles + 1) / 2;
    // enough K-splits to fill the GPU, of at most kGSplitRows rows each
    int64_t splits = ceil_div(4 * kNumSMs, n_pairs);
    if (splits < 1) splits = 1;
    const int64_t max_splits_mem = (int64_t)(2ll << 30) / (t * t * 4);
    if (splits > max_splits_mem) splits = max_splits_mem > 0 ? max_splits_mem : 1;
    if (splits > ceil_div(m, kGK)) splits = ceil_div(m, kGK);
    int64_t rows_per_split = ceil_div(ceil_div(m, splits), kGK) * kGK;
    if (rows_per_split > kGSplitRows) rows_per_split = kGSplitRows;
    splits = ceil_div(m, rows_per_split);
    // splits per launch, bounded by the scratch they need; later passes add into the fp64 result
    int64_t per_pass = splits < max_splits_mem ? splits : (max_splits_mem > 0 ? max_splits_mem : 1);
    if (per_pass > 65535) per_pass = 65535;
    Scratch scratch(st);
    float* partial = nullptr;
    S3_TRY(scratch.alloc(&partial, (size_t)per_pass * t * t));
    S3_CUDA(cudaMemsetAsync(partial, 0, sizeof(float) * (size_t)per_pass * t * t, st));
    for (int64_t s0 = 0; s0 < splits; s0 += per_pass) {
        const int64_t n = (splits - s0) < per_pass ? (splits - s0) : per_pass;
        dim3 grid((unsigned)n_pairs, (unsigned)n);
        gram_kernel<<<grid, kGThreads, 0, st>>>(d_a, d_mean, d_vol, vol_div, s0 * rows_per_split, m, t, tiles,
                                                rows_per_split, partial);
        gram_reduce_kernel<<<(unsigned)ceil_div(t * t, 256), 256, 0, st>>>(partial, (int)n, t, s0 > 0, d_gram);
        S3_LAUNCH_CHECK();
        note_launch(2);
    }
    return S3_OK;
}

// Rows of A per plane chunk of gram_tc / project_tc: each plane at most 2 GB (and at most g_plane_rows_cap rows), a
// multiple of the `tile` rows that a kernel step consumes, no more than the rows of A padded to that tile.
static int64_t plane_rows_for(int64_t m, int64_t t_pad, int64_t tile) {
    int64_t plane_rows = ((int64_t)(1ll << 31) / (t_pad * 4)) & ~(tile - 1);
    if (g_plane_rows_cap > 0 && plane_rows > g_plane_rows_cap) plane_rows = g_plane_rows_cap & ~(tile - 1);
    if (plane_rows < tile) plane_rows = tile;
    const int64_t m_pad = ceil_div(m, tile) * tile;
    return plane_rows < m_pad ? plane_rows : m_pad;
}

static int gram_tc(const float* d_a, const float* d_mean, const float* d_vol, int vol_div, int64_t m, int64_t t,
                   int passes, double* d_gram, cudaStream_t st) {
    // paired kernel (clusters of two CTAs sharing B by TMA multicast): needs an even number of i-tiles per j-tile
    const bool paired = g_tc_pair != 0;
    const int64_t t_pad = paired ? ceil_div(t, kTcBN) * kTcBN : ceil_div(t, kTcBM) * kTcBM;
    const int n_groups = (int)(t_pad / 32);
    const int n_i = (int)(t_pad / kTcBM);
    const int n_j = (int)ceil_div(t_pad, kTcBN);
    int tiles = 0;
    if (paired) for (int tj = 0; tj < n_j; ++tj) tiles += tc_pair_count(tj, n_i);
    else for (int ti = 0; ti < n_i; ++ti) tiles += n_j - tc_first_tj(ti);
    const int64_t plane_rows = plane_rows_for(m, t_pad, kTcKB);
    int splits_max = (kNumSMs + tiles / 2) / tiles;
    if (splits_max < 1) splits_max = 1;

    Scratch scratch(st);
    float *hi = nullptr, *lo = nullptr;
    double* partial = nullptr;
    S3_TRY(scratch.alloc(&hi, (size_t)plane_rows * t_pad));
    if (passes == 3) S3_TRY(scratch.alloc(&lo, (size_t)plane_rows * t_pad));
    S3_TRY(scratch.alloc(&partial, (size_t)tiles * splits_max * kTcBN * kTcBM));

    CUtensorMap map_hi, map_lo;
    S3_TRY(tma_map_f32(&map_hi, "hi", hi, {32, plane_rows, n_groups}, {32, kTcKB, 4}, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B));
    S3_TRY(tma_map_f32(&map_lo, "lo", passes == 3 ? lo : hi, {32, plane_rows, n_groups}, {32, kTcKB, 4},
                       CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B));
    S3_CUDA(cudaFuncSetAttribute(gram_tc_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kTcSmemBytes));
    S3_CUDA(cudaFuncSetAttribute(gram_tc_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kTcSmemBytes));

    int chunk = 0;
    for (int64_t row0 = 0; row0 < m; row0 += plane_rows, ++chunk) {
        const int64_t rows = (m - row0) < plane_rows ? (m - row0) : plane_rows;
        const int64_t rows_pad = ceil_div(rows, kTcKB) * kTcKB;
        gram_prepare_kernel<<<(unsigned)ceil_div(rows_pad * 32, 256), 256, 0, st>>>(
            d_a, d_mean, d_vol, vol_div, row0, rows_pad, m, t, n_groups, plane_rows, hi, lo);
        const int n_kblocks = (int)(rows_pad / kTcKB);
        int splits = splits_max < n_kblocks ? splits_max : n_kblocks;
        const int per_split = (int)ceil_div(n_kblocks, splits);
        splits = (int)ceil_div(n_kblocks, per_split);          // no empty split
        if (paired) {
            cudaLaunchConfig_t cfg;
            memset(&cfg, 0, sizeof(cfg));
            cfg.gridDim = dim3((unsigned)(tiles * splits));       // tiles is even: cluster = (tile 2p, tile 2p + 1) of a split
            cfg.blockDim = dim3(kTcThreads);
            cfg.dynamicSmemBytes = kTcSmemBytes;
            cfg.stream = st;
            cudaLaunchAttribute attr[1];
            attr[0].id = cudaLaunchAttributeClusterDimension;
            attr[0].val.clusterDim.x = 2;
            attr[0].val.clusterDim.y = 1;
            attr[0].val.clusterDim.z = 1;
            cfg.attrs = attr;
            cfg.numAttrs = 1;
            S3_CUDA(cudaLaunchKernelEx(&cfg, gram_tc_kernel<true>, map_hi, map_lo, n_i, n_j, splits, n_kblocks,
                                       g_tc_seg_kblocks, g_tc_flush_segments, passes, partial));
        } else {
            gram_tc_kernel<false><<<(unsigned)(tiles * splits), kTcThreads, kTcSmemBytes, st>>>(
                map_hi, map_lo, n_i, n_j, splits, n_kblocks, g_tc_seg_kblocks, g_tc_flush_segments, passes, partial);
        }
        gram_tc_reduce_kernel<<<(unsigned)ceil_div(t * t, 256), 256, 0, st>>>(partial, splits, n_i, n_j, t, chunk > 0,
                                                                              paired ? 1 : 0, d_gram);
        S3_LAUNCH_CHECK();
        note_launch(3);
    }
    return S3_OK;
}

extern "C" int s3_svd_gram(const float* d_a, const float* d_mean, const float* d_vol, int vol_div, int64_t m, int64_t t,
                           int method, double* d_gram, void* stream) {
    S3_REQUIRE(d_a && d_mean && d_vol && d_gram, "s3_svd_gram: NULL argument");
    S3_REQUIRE(m >= 1 && t >= 1 && vol_div >= 1, "s3_svd_gram: bad sizes");
    S3_REQUIRE(t <= 16384, "s3_svd_gram: too many snapshots (%lld)", (long long)t);
    S3_REQUIRE(method >= 0 && method <= 2, "s3_svd_gram: method must be 0 (fp32 CUDA cores), 1 (3xTF32) or 2 (TF32)");
    cudaStream_t st = (cudaStream_t)stream;
    if (method == 0) return gram_simt(d_a, d_mean, d_vol, vol_div, m, t, d_gram, st);
    return gram_tc(d_a, d_mean, d_vol, vol_div, m, t, method == 1 ? 3 : 1, d_gram, st);
}

extern "C" int s3_svd_project(const float* d_a, const float* d_mean, const float* d_vs, int64_t m, int64_t t, int r,
                              float* d_u, void* stream) {
    S3_REQUIRE(d_a && d_mean && d_vs && d_u, "s3_svd_project: NULL argument");
    S3_REQUIRE(m >= 0 && t >= 1 && r >= 1, "s3_svd_project: bad sizes");
    if (m == 0) return S3_OK;
    dim3 grid((unsigned)ceil_div(m, kPM), (unsigned)ceil_div(r, kPN));
    S3_REQUIRE(grid.y <= 65535, "s3_svd_project: rank too large");
    project_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(d_a, d_mean, d_vs, m, t, r, d_u);
    S3_LAUNCH_CHECK();
    note_launch(1);
    return S3_OK;
}

// U = (A - mean) vs on the tensor cores (see project_tc_kernel); vs [t, r] fp32, u [m, r] fp32.
static int project_tc(const float* d_a, const float* d_mean, const float* d_vol, int vol_div, const float* d_vs,
                      int64_t m, int64_t t, int r, int passes, float* d_u, cudaStream_t st) {
    const int64_t t_pad = ceil_div(t, (int64_t)32) * 32;
    const int n_groups = (int)(t_pad / 32);
    const int64_t plane_rows = plane_rows_for(m, t_pad, kPjBM);
    const int r_blk_max = r < 256 ? (int)(ceil_div((int64_t)r, (int64_t)32) * 32) : 256;   // columns per pass, multiple of 32

    Scratch scratch(st);
    float *hi = nullptr, *lo = nullptr, *whi = nullptr, *wlo = nullptr;
    S3_TRY(scratch.alloc(&hi, (size_t)plane_rows * t_pad));
    if (passes == 3) S3_TRY(scratch.alloc(&lo, (size_t)plane_rows * t_pad));
    S3_TRY(scratch.alloc(&whi, (size_t)r_blk_max * t_pad));
    if (passes == 3) S3_TRY(scratch.alloc(&wlo, (size_t)r_blk_max * t_pad));

    CUtensorMap map_hi, map_lo;
    S3_TRY(tma_map_f32(&map_hi, "projection hi", hi, {32, plane_rows, n_groups}, {32, kPjBM, 1},
                       CU_TENSOR_MAP_SWIZZLE_128B));
    S3_TRY(tma_map_f32(&map_lo, "projection lo", passes == 3 ? lo : hi, {32, plane_rows, n_groups}, {32, kPjBM, 1},
                       CU_TENSOR_MAP_SWIZZLE_128B));
    for (int col0 = 0; col0 < r; col0 += 256) {
        const int r_blk = (r - col0) < 256 ? (r - col0) : 256;
        const int r_pad = (int)(ceil_div((int64_t)r_blk, (int64_t)32) * 32);
        // TMEM: up to 256 columns (two CTAs may share an SM), 512 when the stages leave room for one CTA only
        const int tmem_cols = r_pad > 128 ? 512 : 256;
        int n_seg = tmem_cols / r_pad;
        if (n_seg > 8) n_seg = 8;
        const int launch_groups = n_seg * kPjSegGroups;            // t range of one launch: segments of <= kPjSegGroups
        if (n_seg > n_groups) n_seg = n_groups;
        // W^T [r_pad][t_pad]: W^T[j][tt] = vs[tt][col0 + j]
        tf32_split_kernel<<<(unsigned)ceil_div((int64_t)r_pad * t_pad, (int64_t)256), 256, 0, st>>>(
            d_vs + col0, 1, r, r_blk, t, r_pad, t_pad, whi, wlo);
        CUtensorMap map_whi, map_wlo;
        S3_TRY(tma_map_f32(&map_whi, "projection W hi", whi, {t_pad, r_pad}, {32, r_pad}, CU_TENSOR_MAP_SWIZZLE_128B));
        S3_TRY(tma_map_f32(&map_wlo, "projection W lo", passes == 3 ? wlo : whi, {t_pad, r_pad}, {32, r_pad},
                           CU_TENSOR_MAP_SWIZZLE_128B));
        const size_t smem = (size_t)kPjStages * (2 * kPjABytes + 2 * (size_t)r_pad * 128) + 1024;
        S3_CUDA(cudaFuncSetAttribute(project_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        for (int64_t row0 = 0; row0 < m; row0 += plane_rows) {
            const int64_t rows = (m - row0) < plane_rows ? (m - row0) : plane_rows;
            const int64_t rows_pad = ceil_div(rows, (int64_t)kPjBM) * kPjBM;
            gram_prepare_kernel<<<(unsigned)ceil_div(rows_pad * 32, (int64_t)256), 256, 0, st>>>(
                d_a, d_mean, d_vol, vol_div, row0, rows_pad, m, t, n_groups, plane_rows, hi, lo);
            for (int g0 = 0; g0 < n_groups; g0 += launch_groups) {
                const int lg = (n_groups - g0) < launch_groups ? (n_groups - g0) : launch_groups;
                project_tc_kernel<<<(unsigned)(rows_pad / kPjBM), kPjThreads, smem, st>>>(
                    map_hi, map_lo, map_whi, map_wlo, g0, lg, r_pad, tmem_cols, n_seg < lg ? n_seg : lg, passes, d_vol,
                    vol_div, row0, m, r, col0, g0 > 0, d_u);
                note_launch(1);
            }
            S3_LAUNCH_CHECK();
            note_launch(1);
        }
        note_launch(1);
    }
    return S3_OK;
}

extern "C" int s3_svd_project_tc(const float* d_a, const float* d_mean, const float* d_vol, int vol_div,
                                 const float* d_vs, int64_t m, int64_t t, int r, int method, float* d_u, void* stream) {
    S3_REQUIRE(d_a && d_mean && d_vol && d_vs && d_u, "s3_svd_project_tc: NULL argument");
    S3_REQUIRE(m >= 0 && t >= 1 && r >= 1 && vol_div >= 1, "s3_svd_project_tc: bad sizes");
    S3_REQUIRE(method == 1 || method == 2, "s3_svd_project_tc: method must be 1 (3xTF32) or 2 (TF32)");
    if (m == 0) return S3_OK;
    return project_tc(d_a, d_mean, d_vol, vol_div, d_vs, m, t, r, method == 1 ? 3 : 1, d_u, (cudaStream_t)stream);
}

// e = (a - mean) - left right_t^T on the tensor cores with fused fp64 reductions (see lowrank_error_kernel)
extern "C" int s3_lowrank_error(const float* d_a, int64_t m, int64_t t, const float* d_mean, const float* d_vol,
                                int vol_div, const float* d_left, const float* d_right_t, int q, double* d_sq_err,
                                double* d_sq_ref, double* d_max_abs, double* d_row_sq_err, void* stream) {
    S3_REQUIRE(d_a && d_left && d_right_t, "s3_lowrank_error: NULL argument");
    S3_REQUIRE(d_sq_err && d_sq_ref && d_max_abs, "s3_lowrank_error: NULL result");
    S3_REQUIRE(m >= 1 && t >= 1 && vol_div >= 1, "s3_lowrank_error: bad sizes (m %lld, t %lld, vol_div %d)",
               (long long)m, (long long)t, vol_div);
    S3_REQUIRE(m % vol_div == 0, "s3_lowrank_error: m = %lld rows is not a multiple of vol_div = %d", (long long)m,
               vol_div);
    S3_REQUIRE(m <= ((int64_t)1 << 31) - kLrBM && t <= ((int64_t)1 << 31) - kLrBN,
               "s3_lowrank_error: too many rows or columns (%lld x %lld)", (long long)m, (long long)t);
    if (q < 1 || q > kLrMaxQ) {
        s3::set_error("s3_lowrank_error: q = %d columns of left / right_t, supported 1..%d (one 3xTF32 TMEM segment)", q,
                      kLrMaxQ);
        return S3_ERR_UNSUPPORTED;
    }
    cudaStream_t st = (cudaStream_t)stream;
    const int q_pad = (int)(ceil_div((int64_t)q, (int64_t)32) * 32);
    const int64_t m_pad = ceil_div(m, (int64_t)kLrBM) * kLrBM, t_pad = ceil_div(t, (int64_t)kLrBN) * kLrBN;
    const int64_t n_rt = m_pad / kLrBM;
    const int n_ct = (int)(t_pad / kLrBN);
    // row tiles per group: a function of m only, so that the sums do not depend on the CTA count
    const int64_t tiles_per_group = ceil_div(n_rt, (int64_t)kLrMaxGroups);
    const int64_t n_groups = ceil_div(n_rt, tiles_per_group);
    int64_t ctas = n_groups < kNumSMs ? n_groups : kNumSMs;
    if (g_lowrank_cap > 0 && ctas > g_lowrank_cap) ctas = g_lowrank_cap;

    Scratch scratch(st);
    float *lhi = nullptr, *llo = nullptr, *rhi = nullptr, *rlo = nullptr;
    double* part = nullptr;
    S3_TRY(scratch.alloc(&lhi, (size_t)m_pad * q_pad));
    S3_TRY(scratch.alloc(&llo, (size_t)m_pad * q_pad));
    S3_TRY(scratch.alloc(&rhi, (size_t)t_pad * q_pad));
    S3_TRY(scratch.alloc(&rlo, (size_t)t_pad * q_pad));
    S3_TRY(scratch.alloc(&part, (size_t)n_groups * 3 * vol_div * t));
    tf32_split_kernel<<<(unsigned)ceil_div(m_pad * q_pad, (int64_t)256), 256, 0, st>>>(d_left, q, 1, m, q, m_pad, q_pad,
                                                                                     lhi, llo);
    tf32_split_kernel<<<(unsigned)ceil_div(t_pad * q_pad, (int64_t)256), 256, 0, st>>>(d_right_t, q, 1, t, q, t_pad,
                                                                                     q_pad, rhi, rlo);
    CUtensorMap maps[4];
    S3_TRY(tma_map_f32(&maps[0], "low-rank left hi", lhi, {q_pad, m_pad}, {32, kLrBM}, CU_TENSOR_MAP_SWIZZLE_128B));
    S3_TRY(tma_map_f32(&maps[1], "low-rank left lo", llo, {q_pad, m_pad}, {32, kLrBM}, CU_TENSOR_MAP_SWIZZLE_128B));
    S3_TRY(tma_map_f32(&maps[2], "low-rank right hi", rhi, {q_pad, t_pad}, {32, kLrBN}, CU_TENSOR_MAP_SWIZZLE_128B));
    S3_TRY(tma_map_f32(&maps[3], "low-rank right lo", rlo, {q_pad, t_pad}, {32, kLrBN}, CU_TENSOR_MAP_SWIZZLE_128B));
    S3_CUDA(cudaFuncSetAttribute(lowrank_error_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kLrSmemBytes));
    lowrank_error_kernel<<<(unsigned)ctas, kLrThreads, kLrSmemBytes, st>>>(
        maps[0], maps[1], maps[2], maps[3], d_a, d_mean, d_vol, vol_div, m, t, q_pad / 32, n_ct, n_rt, tiles_per_group,
        n_groups, part, d_row_sq_err);
    lowrank_reduce_kernel<<<(unsigned)ceil_div(3 * (int64_t)vol_div * t, (int64_t)256), 256, 0, st>>>(
        part, n_groups, vol_div, t, d_sq_err, d_sq_ref, d_max_abs);
    S3_LAUNCH_CHECK();
    note_launch(4);
    return S3_OK;
}
