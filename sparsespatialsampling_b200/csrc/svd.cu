// Volume-weighted snapshot SVD by the method of snapshots (device side of compute_svd, utils.py:302-346):
//   B = sqrt(vol) * (A - mean_t(A)),  G = B^T B  [T,T],  G = V diag(s^2) V^T,  U = B V / s / sqrt(vol) = (A - mean) V / s.
// The row means, the Gram contraction and the projection are hand-written kernels; the small dense T x T
// eigen-decomposition is left to the host (torch.linalg.eigh, fp64).
//
// Gram contraction, 2*M*T^2 flop (the only GEMM-shaped work of the S^3 path, SURVEY 8a row a14):
//   method 1/2 (default 1): tcgen05 tensor cores. A prepare kernel centres and scales the rows and writes them as
//     TF32 "hi" (+ "lo" residual for the 3xTF32 split, method 1) planes in a [T/32][rows][32] layout; the Gram
//     kernel is warp-specialised: one TMA producer thread (3-D boxes, 128B swizzle with 32B atoms, 4-stage mbarrier ring), one
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
//   TF32 operands, 3xTF32, a few TMEM segments against accumulation drift), 262144 x 2000 rows onto r = 50 / 150 / 256
//   modes in 1.8 / 2.3 / 2.6 ms (of which 1.1 ms is the prepare pass) instead of 4.2 / 12.2 / 16.0 ms on the fp32
//   CUDA-core kernel, max error vs fp64 2e-6 .. 8e-6 of the largest entry.
#include <cuda.h>
#include "common.cuh"
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
//   b = (a - mean) * sqrt(vol);  hi = tf32_rna(b);  lo = b - hi  (exact in fp32; the tensor core drops lo's low bits).
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
        uint32_t hbits;
        asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(hbits) : "f"(b));
        const float h = __uint_as_float(hbits);
        const int64_t o = ((int64_t)g * plane_rows + r) * 32 + lane;
        hi[o] = h;
        if (lo) lo[o] = b - h;
    }
}

__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* map, int c0, int c1, int c2, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::
            "r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
        : "memory");
}
// mbarrier wait with a watchdog: a protocol error must surface as a launch failure, not as a hung GPU
__device__ __forceinline__ void mbar_wait_wd(uint64_t* bar, uint32_t phase) {
    uint32_t done = 0;
    const long long t0 = clock64();
    while (true) {
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
            "selp.u32 %0, 1, 0, p;\n"
            "}\n"
            : "=r"(done)
            : "r"(smem_u32(bar)), "r"(phase)
            : "memory");
        if (done) break;
        if (clock64() - t0 > 8000000000ll) __trap();
    }
}
// the same box written to the same shared-memory offset of every CTA in `cta_mask`; each destination CTA's mbarrier at
// the same offset receives the complete_tx for the bytes that landed in that CTA
__device__ __forceinline__ void tma_load_3d_multicast(void* dst, const CUtensorMap* map, int c0, int c1, int c2,
                                                      uint64_t* bar, uint16_t cta_mask) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster"
        " [%0], [%1, {%3, %4, %5}], [%2], %6;" ::"r"(smem_u32(dst)),
        "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "h"(cta_mask)
        : "memory");
}
__device__ __forceinline__ uint32_t cluster_rank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\nbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_cta(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// Shared-memory matrix descriptor of an MN-major TF32 operand. 32-bit MN-major operands have exactly one legal
// swizzled layout, "128B swizzle with 32B atoms" (UMMA layout type 1; CUTLASS: Layout_MN_SW128_32B_Atom):
//   (byte address) Swizzle<2,5,2> o ((32 floats, n), (4, k)) : ((4 B, LBO), (128 B, SBO))
// i.e. 128-byte rows of 32 MN-contiguous floats, 4 K-rows per 512-byte atom, the 32-byte chunk index of a row is
// XOR-ed with (row & 3); LBO = byte distance between 32-float MN groups, SBO = byte distance between 4-row K atoms.
// This is what a TMA box {32 floats, rows, groups} written with CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B looks like.
__device__ __forceinline__ uint64_t umma_desc_mn_sw128_32b(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr & 0x3FFFFu) >> 4);
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16;
    d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32;
    d |= (uint64_t)1 << 46;     // descriptor version 1 (Blackwell)
    d |= (uint64_t)1 << 61;     // layout type SWIZZLE_128B_BASE32B
    return d;
}
// instruction descriptor: D fp32, A/B TF32, both MN-major ("transposed"), M x N
__host__ __device__ constexpr uint32_t umma_idesc_tf32_mn(int M, int N) {
    return (1u << 4) | (2u << 7) | (2u << 10) | (1u << 15) | (1u << 16) | ((uint32_t)(N >> 3) << 17) |
           ((uint32_t)(M >> 4) << 24);
}
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                          uint32_t accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
                 : "memory");
}
// the same, arriving on the mbarrier at this offset in every CTA of `cta_mask`
__device__ __forceinline__ void umma_commit_multicast(uint64_t* bar, uint16_t cta_mask) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::
                     "r"(smem_u32(bar)), "h"(cta_mask)
                 : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
          "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
          "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
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
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_hi) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_lo) : "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_slot)),
                     "r"((uint32_t)kTcTmemCols)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
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
    if (warp == 1) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)kTcTmemCols)
                     : "memory");
    }
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

__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, int c0, int c1, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::
            "r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
        : "memory");
}
// K-major TF32 operand, 128B swizzle: rows of 32 K-contiguous floats, 8-row atoms of 1024 bytes (SBO), LBO unused
__device__ __forceinline__ uint64_t umma_desc_k_sw128(uint32_t saddr) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr & 0x3FFFFu) >> 4);
    d |= (uint64_t)1 << 16;                      // LBO (ignored for swizzled K-major layouts)
    d |= (uint64_t)(1024 >> 4) << 32;            // SBO
    d |= (uint64_t)1 << 46;                      // descriptor version 1 (Blackwell)
    d |= (uint64_t)2 << 61;                      // layout type SWIZZLE_128B
    return d;
}
// instruction descriptor: D fp32, A/B TF32, both K-major, M x N
__host__ __device__ constexpr uint32_t umma_idesc_tf32_k(int M, int N) {
    return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// W^T planes: wt[j][tt] = tf32 split of vs[tt][col0 + j] (zero beyond r / t), [r_pad][t_pad]
__global__ void __launch_bounds__(256)
project_prepare_w_kernel(const float* __restrict__ vs, int64_t t, int r, int col0, int r_pad, int64_t t_pad,
                         float* __restrict__ hi, float* __restrict__ lo) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= (int64_t)r_pad * t_pad) return;
    const int j = (int)(e / t_pad);
    const int64_t tt = e % t_pad;
    float w = 0.f;
    if (col0 + j < r && tt < t) w = vs[tt * r + col0 + j];
    uint32_t hbits;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(hbits) : "f"(w));
    const float h = __uint_as_float(hbits);
    hi[e] = h;
    if (lo) lo[e] = w - h;
}

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
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_hi) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_whi) : "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_slot)),
                     "r"((uint32_t)tmem_cols)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
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
#pragma unroll
                for (int ks = 0; ks < 4; ++ks) {                      // 32 floats per stage = 4 UMMA K-steps of 8
                    const uint32_t koff = (uint32_t)ks * 32u;
                    const uint64_t a_hi = umma_desc_k_sw128(st + koff);
                    const uint64_t b_hi = umma_desc_k_sw128(st + 2 * kPjABytes + koff);
                    if (passes == 3) {
                        const uint64_t a_lo = umma_desc_k_sw128(st + kPjABytes + koff);
                        const uint64_t b_lo = umma_desc_k_sw128(st + 2 * kPjABytes + w_bytes + koff);
                        umma_tf32(d_tmem, a_lo, b_hi, idesc, accumulate);
                        umma_tf32(d_tmem, a_hi, b_lo, idesc, 1u);
                        umma_tf32(d_tmem, a_hi, b_hi, idesc, 1u);
                    } else {
                        umma_tf32(d_tmem, a_hi, b_hi, idesc, accumulate);
                    }
                    accumulate = 1u;
                }
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
    if (warp == 1) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)tmem_cols)
                     : "memory");
    }
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

typedef CUresult (*PFN_encodeTiledSvd)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                       const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                       CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

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

static int gram_tc(const float* d_a, const float* d_mean, const float* d_vol, int vol_div, int64_t m, int64_t t,
                   int passes, double* d_gram, cudaStream_t st) {
    static PFN_encodeTiledSvd encode = nullptr;
    if (!encode) {
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult qres;
        S3_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
        S3_REQUIRE(fn != nullptr && qres == cudaDriverEntryPointSuccess, "cuTensorMapEncodeTiled not available");
        encode = (PFN_encodeTiledSvd)fn;
    }
    // paired kernel (clusters of two CTAs sharing B by TMA multicast): needs an even number of i-tiles per j-tile
    const bool paired = g_tc_pair != 0;
    const int64_t t_pad = paired ? ceil_div(t, kTcBN) * kTcBN : ceil_div(t, kTcBM) * kTcBM;
    const int n_groups = (int)(t_pad / 32);
    const int n_i = (int)(t_pad / kTcBM);
    const int n_j = (int)ceil_div(t_pad, kTcBN);
    int tiles = 0;
    if (paired) for (int tj = 0; tj < n_j; ++tj) tiles += tc_pair_count(tj, n_i);
    else for (int ti = 0; ti < n_i; ++ti) tiles += n_j - tc_first_tj(ti);
    // rows of A per chunk: each plane at most 2 GB
    int64_t plane_rows = ((int64_t)(1ll << 31) / (t_pad * 4)) & ~(int64_t)(kTcKB - 1);
    if (g_plane_rows_cap > 0 && plane_rows > g_plane_rows_cap) plane_rows = g_plane_rows_cap & ~(int64_t)(kTcKB - 1);
    if (plane_rows < kTcKB) plane_rows = kTcKB;
    const int64_t m_pad = ceil_div(m, kTcKB) * kTcKB;
    if (plane_rows > m_pad) plane_rows = m_pad;
    int splits_max = (kNumSMs + tiles / 2) / tiles;
    if (splits_max < 1) splits_max = 1;

    Scratch scratch(st);
    float *hi = nullptr, *lo = nullptr;
    double* partial = nullptr;
    S3_TRY(scratch.alloc(&hi, (size_t)plane_rows * t_pad));
    if (passes == 3) S3_TRY(scratch.alloc(&lo, (size_t)plane_rows * t_pad));
    S3_TRY(scratch.alloc(&partial, (size_t)tiles * splits_max * kTcBN * kTcBM));

    CUtensorMap map_hi, map_lo;
    memset(&map_hi, 0, sizeof(map_hi));
    memset(&map_lo, 0, sizeof(map_lo));
    {
        const cuuint64_t gdim[3] = {32, (cuuint64_t)plane_rows, (cuuint64_t)n_groups};
        const cuuint64_t gstride[2] = {128, (cuuint64_t)plane_rows * 128};
        const cuuint32_t box[3] = {32, (cuuint32_t)kTcKB, 4};
        const cuuint32_t estride[3] = {1, 1, 1};
        CUresult cr = encode(&map_hi, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, hi, gdim, gstride, box, estride,
                             CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B,
                             CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        S3_REQUIRE(cr == CUDA_SUCCESS, "cuTensorMapEncodeTiled(hi) failed with code %d", (int)cr);
        cr = encode(&map_lo, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, passes == 3 ? lo : hi, gdim, gstride, box, estride,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        S3_REQUIRE(cr == CUDA_SUCCESS, "cuTensorMapEncodeTiled(lo) failed with code %d", (int)cr);
    }
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
    static PFN_encodeTiledSvd encode = nullptr;
    if (!encode) {
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult qres;
        S3_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
        S3_REQUIRE(fn != nullptr && qres == cudaDriverEntryPointSuccess, "cuTensorMapEncodeTiled not available");
        encode = (PFN_encodeTiledSvd)fn;
    }
    const int64_t t_pad = ceil_div(t, (int64_t)32) * 32;
    const int n_groups = (int)(t_pad / 32);
    // rows of A per chunk: each plane at most 2 GB, a multiple of the 128-row tile
    int64_t plane_rows = ((int64_t)(1ll << 31) / (t_pad * 4)) & ~(int64_t)(kPjBM - 1);
    if (g_plane_rows_cap > 0 && plane_rows > g_plane_rows_cap) plane_rows = g_plane_rows_cap & ~(int64_t)(kPjBM - 1);
    if (plane_rows < kPjBM) plane_rows = kPjBM;
    const int64_t m_pad = ceil_div(m, (int64_t)kPjBM) * kPjBM;
    if (plane_rows > m_pad) plane_rows = m_pad;
    const int r_blk_max = r < 256 ? (int)(ceil_div((int64_t)r, (int64_t)32) * 32) : 256;   // columns per pass, multiple of 32

    Scratch scratch(st);
    float *hi = nullptr, *lo = nullptr, *whi = nullptr, *wlo = nullptr;
    S3_TRY(scratch.alloc(&hi, (size_t)plane_rows * t_pad));
    if (passes == 3) S3_TRY(scratch.alloc(&lo, (size_t)plane_rows * t_pad));
    S3_TRY(scratch.alloc(&whi, (size_t)r_blk_max * t_pad));
    if (passes == 3) S3_TRY(scratch.alloc(&wlo, (size_t)r_blk_max * t_pad));

    CUtensorMap map_hi, map_lo;
    memset(&map_hi, 0, sizeof(map_hi));
    memset(&map_lo, 0, sizeof(map_lo));
    {
        const cuuint64_t gdim[3] = {32, (cuuint64_t)plane_rows, (cuuint64_t)n_groups};
        const cuuint64_t gstride[2] = {128, (cuuint64_t)plane_rows * 128};
        const cuuint32_t box[3] = {32, (cuuint32_t)kPjBM, 1};
        const cuuint32_t estride[3] = {1, 1, 1};
        CUresult cr = encode(&map_hi, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, hi, gdim, gstride, box, estride,
                             CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                             CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        S3_REQUIRE(cr == CUDA_SUCCESS, "cuTensorMapEncodeTiled(projection hi) failed with code %d", (int)cr);
        cr = encode(&map_lo, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, passes == 3 ? lo : hi, gdim, gstride, box, estride,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        S3_REQUIRE(cr == CUDA_SUCCESS, "cuTensorMapEncodeTiled(projection lo) failed with code %d", (int)cr);
    }
    for (int col0 = 0; col0 < r; col0 += 256) {
        const int r_blk = (r - col0) < 256 ? (r - col0) : 256;
        const int r_pad = (int)(ceil_div((int64_t)r_blk, (int64_t)32) * 32);
        // TMEM: up to 256 columns (two CTAs may share an SM), 512 when the stages leave room for one CTA only
        const int tmem_cols = r_pad > 128 ? 512 : 256;
        int n_seg = tmem_cols / r_pad;
        if (n_seg > 8) n_seg = 8;
        const int launch_groups = n_seg * kPjSegGroups;            // t range of one launch: segments of <= kPjSegGroups
        if (n_seg > n_groups) n_seg = n_groups;
        project_prepare_w_kernel<<<(unsigned)ceil_div((int64_t)r_pad * t_pad, (int64_t)256), 256, 0, st>>>(
            d_vs, t, r, col0, r_pad, t_pad, whi, wlo);
        CUtensorMap map_whi, map_wlo;
        memset(&map_whi, 0, sizeof(map_whi));
        memset(&map_wlo, 0, sizeof(map_wlo));
        {
            const cuuint64_t gdim[2] = {(cuuint64_t)t_pad, (cuuint64_t)r_pad};
            const cuuint64_t gstride[1] = {(cuuint64_t)t_pad * 4};
            const cuuint32_t box[2] = {32, (cuuint32_t)r_pad};
            const cuuint32_t estride[2] = {1, 1};
            CUresult cr = encode(&map_whi, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, whi, gdim, gstride, box, estride,
                                 CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                                 CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
            S3_REQUIRE(cr == CUDA_SUCCESS, "cuTensorMapEncodeTiled(projection W hi) failed with code %d", (int)cr);
            cr = encode(&map_wlo, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, passes == 3 ? wlo : whi, gdim, gstride, box, estride,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
            S3_REQUIRE(cr == CUDA_SUCCESS, "cuTensorMapEncodeTiled(projection W lo) failed with code %d", (int)cr);
        }
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
