// Export-stage interpolation of snapshot rows onto the sampled grid:
//   out[c, d, t] = sum_j w[c, j] * data[idx[c, j], d, t]
// Replaces interpolate_data (sparseSpatialSampling/export.py:446-468), which materialises
// data[idx] ([chunk, k, D, T]) and reduces it on the CPU.
//
// Layout: the reference's [N, D, T] with T contiguous, described by strides (row_stride between source points,
// comp_stride between the D components of a point, both in elements). A row pitch that is a multiple of 128 bytes is
// the layout this kernel is built for: every 512-byte warp request then covers exactly four 128-byte lines. With the
// reference's dense pitch (T = 1000 -> 4000 B) three rows in four start 32/64/96 bytes into a line and every
// 128-bit warp load costs 6 L1 wavefronts instead of 4 (the two half-warp requests each straddle a third line) --
// measured 0.68 of the HBM roofline instead of the aligned figure (DESIGN.md 3).
//
// Work distribution: one warp per cell, the warps of a CTA work on CONSECUTIVE cells of the processing order (callers
// pass cells in Morton order): neighbouring cells share most of their source rows, so the same 512-byte row segments
// are requested by several warps of the CTA within a few hundred cycles and are served by L1; the CTAs in flight
// cover a compact window of the grid, so the second use of a row by a neighbouring CTA is an L2 hit and every source
// row crosses HBM once (ncu: DRAM bytes = 0.995 x algorithmic bytes). The lanes sweep the row, V contiguous columns
// per lane and step (one 128-bit vector), UNROLL steps at a time; a cell's (index, weight) pairs live in registers
// (lane j holds neighbour j) and are broadcast with shuffles, or parked in shared memory and read back with one
// uniform LDS.64 per neighbour (PAIRS).
#include <stdlib.h>
#include <type_traits>
#include "common.cuh"
#include "../../include/s3b200.h"

namespace s3 {

// ---- knobs of the A/B harness (s3x_tune, not part of the public C-ABI) -----------------------------------------
static int g_warps_per_cta = 8;    // key 1: cells (= warps) per CTA
static int g_unroll = 0;           // key 2: column vectors per lane and step, 0 = by k
static int g_pairs = -1;           // key 3: (idx, w) broadcast: 0 = SHFL, 1 = shared-memory pairs, -1 = by k
static int g_chunk_cols = 0;       // key 4: columns per blockIdx.y window, 0 = whole row
static int g_carveout = -1;        // key 5: shared-memory carve-out in percent, -1 = driver default
static int g_wide = -1;            // key 6: 256-bit loads (fp32 in/out, pointers and pitches multiples of 32 B): -1 = whenever possible
static int g_wide64 = 1;           // key 16: 256-bit path of the fp64-result mode
static int g_dense = 1;            // key 9: 1 = dense fp32 batches with k <= 16 take interp_dense_kernel
static int g_kunroll = 0;          // key 7: neighbour-loop unroll (row loads in flight per lane): 1, 4 or 8; 0 = by row length
static int g_persistent = -1;      // key 8: part-warp persistent kernel: -1 = short rows (see launch_interp), 0 = never, 1 = whenever possible
static int g_lanes_per_cell = 0;   // key 13: lanes per cell of that kernel (16 or 32), 0 = by row length
static int g_persist_ctas = 0;     // key 12: resident CTAs per SM it is compiled for (3: 80 registers, 4: 64), 0 = by row length
static int g_persist_cap = 0;      // key 15: at most this many CTAs of that kernel (tests: several sweeps at small sizes), 0 = no cap
extern int g_tc_seg_kblocks;
extern int g_tc_flush_segments;
extern int g_tc_pair;
extern int g_plane_rows_cap;       // key 17 (csrc/svd.cu): rows per TF32 plane chunk of the Gram / projection kernels, 0 = no cap
extern int g_lowrank_cap;          // key 19 (csrc/svd.cu): CTAs of s3_lowrank_error at most, 0 = one per SM
extern int g_curve;          // csrc/knn.cu: 0 = Morton, 1 = Hilbert order of the KNN index and of the processing order (key 30)

template <typename T, int V>
struct alignas(sizeof(T) * V) Vec {
    T v[V];
};

template <typename T, int V>
__device__ __forceinline__ Vec<T, V> ld_vec(const T* p) {
    // plain (allocating) loads: the row segments are re-used by the neighbouring cells of the CTA
    return *reinterpret_cast<const Vec<T, V>*>(p);
}
template <>
__device__ __forceinline__ Vec<float, 8> ld_vec<float, 8>(const float* p) {
    Vec<float, 8> r;
    asm volatile("ld.global.v8.f32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=f"(r.v[0]), "=f"(r.v[1]), "=f"(r.v[2]), "=f"(r.v[3]), "=f"(r.v[4]), "=f"(r.v[5]), "=f"(r.v[6]),
                   "=f"(r.v[7])
                 : "l"(p));
    return r;
}
template <>
__device__ __forceinline__ Vec<double, 4> ld_vec<double, 4>(const double* p) {
    Vec<double, 4> r;
    asm volatile("ld.global.v4.f64 {%0, %1, %2, %3}, [%4];" : "=d"(r.v[0]), "=d"(r.v[1]), "=d"(r.v[2]), "=d"(r.v[3]) : "l"(p));
    return r;
}
template <typename T, int V>
__device__ __forceinline__ void st_vec(T* p, const Vec<T, V>& x) {
    *reinterpret_cast<Vec<T, V>*>(p) = x;
}
template <>
__device__ __forceinline__ void st_vec<double, 4>(double* p, const Vec<double, 4>& x) {
    asm volatile("st.global.v4.f64 [%0], {%1, %2, %3, %4};" ::"l"(p), "d"(x.v[0]), "d"(x.v[1]), "d"(x.v[2]), "d"(x.v[3]) : "memory");
}
template <>
__device__ __forceinline__ void st_vec<double, 8>(double* p, const Vec<double, 8>& x) {      // two 256-bit stores
    asm volatile("st.global.v4.f64 [%0], {%1, %2, %3, %4};" ::"l"(p), "d"(x.v[0]), "d"(x.v[1]), "d"(x.v[2]), "d"(x.v[3]) : "memory");
    asm volatile("st.global.v4.f64 [%0], {%1, %2, %3, %4};" ::"l"(p + 4), "d"(x.v[4]), "d"(x.v[5]), "d"(x.v[6]), "d"(x.v[7]) : "memory");
}
template <>
__device__ __forceinline__ void st_vec<float, 8>(float* p, const Vec<float, 8>& x) {
    asm volatile("st.global.v8.f32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(p), "f"(x.v[0]), "f"(x.v[1]),
                 "f"(x.v[2]), "f"(x.v[3]), "f"(x.v[4]), "f"(x.v[5]), "f"(x.v[6]), "f"(x.v[7])
                 : "memory");
}

struct InterpGeom {
    int64_t row_stride, comp_stride;          // source: elements between points / between components
    int64_t out_row_stride, out_comp_stride;  // result
    int64_t n_cols;                           // T: columns per component
    int64_t chunk_cols;                       // columns per blockIdx.y window (multiple of the warp step)
    int n_chunks;                             // windows per component
    int lead;                                 // columns the first warp step is shortened by so that all following
                                              // steps start on a 128-byte line (common misalignment of all rows)
};

// MODE 0: fp32 FMA accumulation (fast path). MODE 1: fp64 products, then sequential adds without contraction -- the
// reference's (w * data[idx]).sum(dim=1) evaluation order (export.py:463-466).
// KU: unroll factor of the neighbour loop = row loads a lane keeps in flight (ptxas batches the loads of an unrolled
// group in front of their FMAs); the 32-register variants (64 resident warps per SM) and the batched ones trade
// occupancy against memory-level parallelism per warp -- both are instantiated, the launcher picks by measurement.
template <typename Tin, typename Tw, typename Tout, int V, int MODE, int UNROLL, bool PAIRS, int KU>
__global__ void __launch_bounds__(512, (MODE == 0 && sizeof(Tin) * V * UNROLL <= 16 && KU == 1) ? 4 : 0)
interp_warpcell_kernel(const Tin* __restrict__ data, const int32_t* __restrict__ idx, const Tw* __restrict__ w,
                       int64_t n_cells, int k, const int32_t* __restrict__ out_row, Tout* __restrict__ out,
                       const InterpGeom g) {
    const int warps = blockDim.x >> 5;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t cell = (int64_t)blockIdx.x * warps + warp;
    if (cell >= n_cells) return;
    const int comp = (int)(blockIdx.y / g.n_chunks), chunk = (int)(blockIdx.y % g.n_chunks);

    int32_t idx_lo = 0, idx_hi = 0;
    Tw w_lo = (Tw)0, w_hi = (Tw)0;
    if (lane < k) { idx_lo = idx[cell * k + lane]; w_lo = w[cell * k + lane]; }
    if (lane + 32 < k) { idx_hi = idx[cell * k + lane + 32]; w_hi = w[cell * k + lane + 32]; }
    const int64_t orow = out_row ? (int64_t)out_row[cell] : cell;

    extern __shared__ __align__(16) unsigned char s_raw[];
    struct alignas(2 * sizeof(Tw)) Pair { int32_t i; Tw w; };       // one LDS.64 (fp32 weights) / LDS.128 (fp64)
    Pair* my_pairs = reinterpret_cast<Pair*>(s_raw) + (size_t)warp * k;
    if (PAIRS) {
        if (lane < k) my_pairs[lane] = Pair{idx_lo, w_lo};
        if (lane + 32 < k) my_pairs[lane + 32] = Pair{idx_hi, w_hi};
        __syncwarp();
    }

    const Tin* src0 = data + (int64_t)comp * g.comp_stride;
    Tout* dst = out + orow * g.out_row_stride + (int64_t)comp * g.out_comp_stride;
    constexpr int STEP = 32 * V;
    // window [c_begin, c_end) of this CTA row; steps are laid out from -lead so that step boundaries are line aligned
    const int64_t w_begin = (int64_t)chunk * g.chunk_cols - g.lead;
    const int64_t c_begin = w_begin < 0 ? 0 : w_begin;
    const int64_t w_end = w_begin + g.chunk_cols;
    const int64_t c_end = (chunk == g.n_chunks - 1 || w_end > g.n_cols) ? g.n_cols : w_end;
    const int64_t c_vec_end = c_end - (c_end % V);      // last column covered by whole vectors (n_cols % V tail below)

    for (int64_t col0 = w_begin; col0 < c_vec_end; col0 += (int64_t)STEP * UNROLL) {
        Tw acc[UNROLL][V];
        bool in[UNROLL];
#pragma unroll
        for (int u = 0; u < UNROLL; ++u) {
            const int64_t c = col0 + u * STEP + lane * V;
            in[u] = c >= c_begin && c < c_vec_end;
#pragma unroll
            for (int e = 0; e < V; ++e) acc[u][e] = (Tw)0;
        }
        const Tin* colbase = src0 + col0 + lane * V;
#pragma unroll KU
        for (int j = 0; j < k; ++j) {
            int32_t r;
            Tw wj;
            if (PAIRS) {
                const Pair pr = my_pairs[j];
                r = pr.i;
                wj = pr.w;
            } else {
                r = __shfl_sync(0xffffffffu, (j & 32) ? idx_hi : idx_lo, j & 31);
                wj = __shfl_sync(0xffffffffu, (j & 32) ? w_hi : w_lo, j & 31);
            }
            const Tin* src = colbase + (int64_t)r * g.row_stride;
#pragma unroll
            for (int u = 0; u < UNROLL; ++u) {
                if (in[u]) {
                    const Vec<Tin, V> x = ld_vec<Tin, V>(src + u * STEP);
#pragma unroll
                    for (int e = 0; e < V; ++e) {
                        if (MODE == 0) acc[u][e] = fmaf((float)wj, (float)x.v[e], (float)acc[u][e]);
                        else acc[u][e] = __dadd_rn((double)acc[u][e], __dmul_rn((double)wj, (double)x.v[e]));
                    }
                }
            }
        }
#pragma unroll
        for (int u = 0; u < UNROLL; ++u) {
            if (in[u]) {
                Vec<Tout, V> ov;
#pragma unroll
                for (int e = 0; e < V; ++e) ov.v[e] = (Tout)acc[u][e];
                st_vec<Tout, V>(dst + col0 + u * STEP + lane * V, ov);
            }
        }
    }
    // the n_cols % V columns behind the last whole vector (V > 1 only): one column per lane, scalar accesses
    if (V > 1 && c_end == g.n_cols && c_vec_end < c_end) {
        const int64_t c = c_vec_end + lane;
        const bool mine = c < c_end;
        Tw acc = (Tw)0;
        for (int j = 0; j < k; ++j) {
            const int32_t r = __shfl_sync(0xffffffffu, (j & 32) ? idx_hi : idx_lo, j & 31);
            const Tw wj = __shfl_sync(0xffffffffu, (j & 32) ? w_hi : w_lo, j & 31);
            if (mine) {
                const Tin x = src0[(int64_t)r * g.row_stride + c];
                if (MODE == 0) acc = fmaf((float)wj, (float)x, (float)acc);
                else acc = __dadd_rn((double)acc, __dmul_rn((double)wj, (double)x));
            }
        }
        if (mine) dst[c] = (Tout)acc;
    }
}

// Dense fp32 batches (row pitch = row length on both sides) whose rows are 16- but not 32-byte aligned, so that the
// 256-bit path does not apply: the round-1 formulation of the same loop, kept because ptxas schedules it best among the
// 128-bit variants for k = 8 (four predicated row loads in flight at 32 registers = 64 resident warps per SM; C2: 0.391
// ms per step against 0.405-0.48 for the strided 128-bit instantiations, 0.375 for the 256-bit kernel on this layout).
__global__ void __launch_bounds__(512)
interp_dense_kernel(const float* __restrict__ data, int64_t row_len, const int32_t* __restrict__ idx,
                    const float* __restrict__ w, int64_t n_cells, int k, const int32_t* __restrict__ out_row,
                    float* __restrict__ out) {
    const int warps = blockDim.x >> 5;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t cell = (int64_t)blockIdx.x * warps + warp;
    if (cell >= n_cells) return;
    int32_t idx_lo = 0, idx_hi = 0;
    float w_lo = 0.f, w_hi = 0.f;
    if (lane < k) { idx_lo = idx[cell * k + lane]; w_lo = w[cell * k + lane]; }
    if (lane + 32 < k) { idx_hi = idx[cell * k + lane + 32]; w_hi = w[cell * k + lane + 32]; }
    const int64_t orow = out_row ? (int64_t)out_row[cell] : cell;
    float* o = out + orow * row_len;
    constexpr int V = 4, STEP = 32 * V;
    for (int64_t col0 = 0; col0 < row_len; col0 += (int64_t)STEP) {
        float acc[V];
#pragma unroll
        for (int e = 0; e < V; ++e) acc[e] = 0.f;
        for (int j = 0; j < k; ++j) {
            const int32_t r = __shfl_sync(0xffffffffu, (j & 32) ? idx_hi : idx_lo, j & 31);
            const float wj = __shfl_sync(0xffffffffu, (j & 32) ? w_hi : w_lo, j & 31);
            const float* src = data + (int64_t)r * row_len + col0 + lane * V;
            if (col0 + lane * V < row_len) {
                const Vec<float, V> x = ld_vec<float, V>(src);
#pragma unroll
                for (int e = 0; e < V; ++e) acc[e] = fmaf(wj, x.v[e], acc[e]);
            }
        }
        const int64_t c = col0 + lane * V;
        if (c < row_len) {
            Vec<float, V> ov;
#pragma unroll
            for (int e = 0; e < V; ++e) ov.v[e] = acc[e];
            *reinterpret_cast<Vec<float, V>*>(o + c) = ov;
        }
    }
}

// Short rows (the time windows of a sharded export: 125-500 snapshots per rank; k = 8: up to ~750 columns).
// interp_warpcell_kernel spends a whole warp and a CTA slot on one cell: for a 500-byte row that is one 128-bit load
// per neighbour behind a dependent table load, ~500 issued instructions per cell, and the SM is issue bound (ncu: 84 %
// issue-active at 0.34 of the HBM roofline). Here the warps are persistent and split into PART-WARPS of LPC lanes:
//   * a part-warp walks the cells  first + i * stride  on its own (no CTA barrier anywhere); one 256-bit vector per
//     lane, so a warp request still covers 1 KB of row segments -- of two cells at a time for rows <= 128 columns;
//   * lane j fetches neighbour j's (index, weight) of the NEXT cell while the rows of the current one are in flight,
//     parks them in the part-warp's shared-memory slot, and all lanes read them back with uniform LDS.64;
//   * the components of a point are looped inside (tables read once per cell, not once per component);
//   * KU row segments are in flight per lane before their FMAs are issued in neighbour order.
// The part-warps resident on the GPU at any time cover one compact window of consecutive cells (the warps of a CTA:
// 8-16 consecutive cells, for L1; all CTAs: a few thousand, for L2). A source vector that straddles the end of a row
// is loaded whole (pitches are multiples of 32 bytes, so the load stays inside the 32-byte sector of the row's last
// valid column) and stored column by column. Same products in the same order as interp_warpcell_kernel: same bits.
// KR = table registers per lane (k <= KR * LPC); CTAS = resident CTAs per SM the register budget is cut for.
template <int LPC, int KU, int KR, int CTAS>
__global__ void __launch_bounds__(256, CTAS)
interp_partwarp_kernel(const float* __restrict__ data, const int32_t* __restrict__ idx, const float* __restrict__ w,
                       int64_t n_cells, int k, const int32_t* __restrict__ out_row, float* __restrict__ out,
                       const InterpGeom g, int n_comp, int store_w) {
    extern __shared__ __align__(16) unsigned char s_raw[];
    struct alignas(8) Pair { int32_t i; float w; };
    constexpr int SUB = 32 / LPC;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, warps = blockDim.x >> 5;
    const int sub = lane / LPC, sl = lane % LPC;
    Pair* my_pairs = reinterpret_cast<Pair*>(s_raw) + (size_t)(warp * SUB + sub) * (KR * LPC);
    const int64_t stride = (int64_t)gridDim.x * warps * SUB;
    const int64_t warp_first = ((int64_t)blockIdx.x * warps + warp) * SUB;      // uniform loop bound of the warp
    int64_t cell = warp_first + sub;

    Pair nxt[KR];
    int32_t orow_n = 0;
    auto fetch = [&](int64_t c) {
#pragma unroll
        for (int q = 0; q < KR; ++q) {
            const int j = sl + q * LPC;
            nxt[q] = Pair{0, 0.f};
            if (c < n_cells && j < k) nxt[q] = Pair{idx[c * k + j], w[c * k + j]};
        }
        orow_n = c < n_cells ? (out_row ? out_row[c] : (int32_t)c) : 0;
    };
    fetch(cell);
    for (int64_t first = warp_first; first < n_cells; first += stride, cell += stride) {
#pragma unroll
        for (int q = 0; q < KR; ++q) my_pairs[sl + q * LPC] = nxt[q];
        const int64_t orow = orow_n;
        __syncwarp();
        fetch(cell + stride);
        if (cell < n_cells) {
            for (int comp = 0; comp < n_comp; ++comp) {
                float* dst = out + orow * g.out_row_stride + (int64_t)comp * g.out_comp_stride;
                for (int col = sl * 8; col < (int)g.n_cols; col += LPC * 8) {
                    float acc[8];
#pragma unroll
                    for (int e = 0; e < 8; ++e) acc[e] = 0.f;
                    const float* colbase = data + (int64_t)comp * g.comp_stride + col;
                    int j = 0;
                    for (; j + KU <= k; j += KU) {
                        Vec<float, 8> x[KU];
                        float wj[KU];
#pragma unroll
                        for (int u = 0; u < KU; ++u) {
                            const Pair p = my_pairs[j + u];
                            wj[u] = p.w;
                            x[u] = ld_vec<float, 8>(colbase + (int64_t)p.i * g.row_stride);
                        }
#pragma unroll
                        for (int u = 0; u < KU; ++u)
#pragma unroll
                            for (int e = 0; e < 8; ++e) acc[e] = fmaf(wj[u], x[u].v[e], acc[e]);
                    }
                    for (; j < k; ++j) {
                        const Pair p = my_pairs[j];
                        const Vec<float, 8> x = ld_vec<float, 8>(colbase + (int64_t)p.i * g.row_stride);
#pragma unroll
                        for (int e = 0; e < 8; ++e) acc[e] = fmaf(p.w, x.v[e], acc[e]);
                    }
                    // result rows need not share the alignment of the source rows (a dense [Nc, D, 250] result has
                    // 8-byte aligned rows): store_w = widest vector (in floats) every result segment is aligned for
                    if (col + 8 <= (int)g.n_cols && store_w == 8) {
                        Vec<float, 8> ov;
#pragma unroll
                        for (int e = 0; e < 8; ++e) ov.v[e] = acc[e];
                        st_vec<float, 8>(dst + col, ov);
                    } else if (col + 8 <= (int)g.n_cols && store_w == 4) {
#pragma unroll
                        for (int h = 0; h < 2; ++h) {
                            Vec<float, 4> ov;
#pragma unroll
                            for (int e = 0; e < 4; ++e) ov.v[e] = acc[4 * h + e];
                            st_vec<float, 4>(dst + col + 4 * h, ov);
                        }
                    } else if (col + 8 <= (int)g.n_cols && store_w == 2) {
#pragma unroll
                        for (int h = 0; h < 4; ++h) {
                            Vec<float, 2> ov;
                            ov.v[0] = acc[2 * h];
                            ov.v[1] = acc[2 * h + 1];
                            st_vec<float, 2>(dst + col + 2 * h, ov);
                        }
                    } else {
#pragma unroll
                        for (int e = 0; e < 8; ++e)
                            if (col + e < (int)g.n_cols) dst[col + e] = acc[e];
                    }
                }
            }
        }
        __syncwarp();
    }
}

template <typename Tin, typename Tw, typename Tout, int MODE>
static int launch_interp(const void* data, const int32_t* idx, const void* w, int64_t n_cells, int k,
                         const int32_t* out_row, void* out, int n_comp, InterpGeom g, cudaStream_t stream) {
    constexpr int VFULL = 16 / sizeof(Tin);
    const int warps = g_warps_per_cta;
    const int64_t blocks = ceil_div(n_cells, warps);
    S3_REQUIRE(blocks < ((int64_t)1 << 31), "s3_interp_gather: too many cells");
    // vector path: every (row, component) segment starts on a 16-byte boundary, for the source and for the result
    const bool vec_ok = ((uintptr_t)data % 16 == 0) && ((uintptr_t)out % (sizeof(Tout) * VFULL) == 0) &&
                        g.row_stride % VFULL == 0 && g.comp_stride % VFULL == 0 && g.out_row_stride % VFULL == 0 &&
                        g.out_comp_stride % VFULL == 0;
    // Launch shape by measurement (C2 tables k = 8, T = 1000 and 3-D tables k = 26, T = 2000; scripts/interp_lab.py,
    // profiles/r2_interp_lab.md): 256-bit row loads with the (index, weight) pairs in shared memory whenever pointers
    // and pitches are 32-byte aligned (k = 8: 0.378 ms per C2 step on 128-byte pitched rows against 0.387 with two
    // 128-bit vectors per lane and 0.46 with one; k = 26: 8.1-8.5 ms against 9.5-9.7), one column vector per lane for
    // k <= 16 and two beyond, two 128-bit vectors otherwise.
    const bool wide_ok = vec_ok && MODE == 0 && std::is_same<Tin, float>::value && std::is_same<Tout, float>::value &&
                         (uintptr_t)data % 32 == 0 && (uintptr_t)out % 32 == 0 && g.row_stride % 8 == 0 &&
                         g.comp_stride % 8 == 0 && g.out_row_stride % 8 == 0 && g.out_comp_stride % 8 == 0;
    // short rows (time windows of a sharded export): a 256-column warp step would leave most lanes idle
    const bool wide = wide_ok && (g_wide == 1 || (g_wide < 0 && g.n_cols >= 384));
    // the reference's result dtype (fp64 sums): 256-bit loads (8 floats / 4 doubles per lane), 256-bit stores
    constexpr int VW64 = 32 / sizeof(Tin);
    const bool wide64 = MODE == 1 && std::is_same<Tout, double>::value && g_wide64 && vec_ok &&
                        (uintptr_t)data % 32 == 0 && (uintptr_t)out % 32 == 0 && g.row_stride % VW64 == 0 &&
                        g.comp_stride % VW64 == 0 && g.out_row_stride % 4 == 0 && g.out_comp_stride % 4 == 0 &&
                        (g_wide == 1 || (g_wide < 0 && g.n_cols >= 384));
    const int unroll = g_unroll != 0 ? g_unroll : ((wide || wide64) ? (k > 16 ? 2 : 1) : (g.n_cols > 128 ? 2 : 1));
    const bool pairs = g_pairs >= 0 ? g_pairs != 0 : (wide || wide64 || k > 16);
    // Rows of one or two warp steps (the time windows of a sharded export): the warp is bound by the chain
    // index -> row load -> FMA, one load latency per neighbour; eight neighbours' loads are issued as a batch there.
    // Long rows keep one load in flight per warp (more only thrashes the L1, profiles/r2_interp_lab.md).
    const int kunroll = g_kunroll != 0 ? g_kunroll : (g.n_cols <= 256 ? 8 : 1);
    if constexpr (std::is_same<Tin, float>::value && std::is_same<Tout, float>::value && MODE == 0) {
        // measured cross-over against the warp-per-cell kernel (profiles/r2_interp_lab.md, run 8): k = 8 wins up to 750
        // columns (T = 1000: 0.352 against 0.346 ms); k = 26 on the 10 M-point C4 cloud wins at 250 (0.98 against 1.22 ms)
        // and loses at 500 (2.31 against 1.96 ms)
        const bool short_rows = g.n_cols <= (k <= 16 ? 768 : 256);
        // 256-bit loads need 32-byte aligned SOURCE segments only; the stores adapt to the result's alignment
        const bool src_wide_ok = (uintptr_t)data % 32 == 0 && g.row_stride % 8 == 0 && g.comp_stride % 8 == 0;
        const uintptr_t out_bits = (uintptr_t)out | (uintptr_t)(g.out_row_stride * 4) | (uintptr_t)(g.out_comp_stride * 4);
        const int store_w = out_bits % 32 == 0 ? 8 : out_bits % 16 == 0 ? 4 : out_bits % 8 == 0 ? 2 : 1;
        if (src_wide_ok && k <= 64 && g.n_cols < (1 << 30) && g_chunk_cols == 0 &&
            (g_persistent == 1 || (g_persistent < 0 && short_rows))) {
            int lpc = g_lanes_per_cell ? g_lanes_per_cell : (g.n_cols <= 128 ? 16 : 32);
            if (k > 2 * lpc) lpc = 32;
            const int kr = k <= lpc ? 1 : 2;
            const int ku = g_kunroll == 8 ? 8 : 4;
            // whole-warp rows with few neighbours run best at 4 CTAs (32 warps) per SM, the two-cells-per-warp shape and
            // k = 26 at 3 (T = 500: 0.181 against 0.191 ms, T = 125: 0.066 against 0.065)
            const int per_sm_built = g_persist_ctas ? g_persist_ctas : (lpc == 32 && k <= 16 ? 4 : 3);
            const int sub = 32 / lpc;
            const int pw = warps > 8 ? 8 : warps;                  // __launch_bounds__(256, ...)
            const int threads = pw * 32;
            const size_t sm = (size_t)pw * sub * kr * lpc * 8;
            const float* d_f = reinterpret_cast<const float*>(data);
            const float* w_f = reinterpret_cast<const float*>(w);
            float* o_f = reinterpret_cast<float*>(out);
            int dev = 0;
            cudaGetDevice(&dev);
            // resident CTAs of the whole device per (device, instantiation, CTA size): queried once, the launch itself
            // stays free of driver queries (benign race: every thread computes the same number)
            static int s_resident[16][2][2][3][9];
            int* slot = (dev >= 0 && dev < 16) ? &s_resident[dev][lpc == 32][kr - 1][ku == 8 ? 0 : per_sm_built - 2][pw] : nullptr;
#define S3_PARTWARP(L, K_, R, C)                                                                                   \
    do {                                                                                                           \
        auto kern = interp_partwarp_kernel<L, K_, R, C>;                                                           \
        int resident = slot ? *slot : 0;                                                                           \
        if (resident <= 0) {                                                                                       \
            int per_sm = 1, n_sm = 148;                                                                            \
            cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev);                                    \
            cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, threads, sm);                             \
            resident = n_sm * (per_sm < 1 ? 1 : per_sm);                                                           \
            if (slot) *slot = resident;                                                                            \
        }                                                                                                          \
        const int64_t want = ceil_div(n_cells, (int64_t)pw * sub);                                                 \
        int64_t ctas = want < (int64_t)resident ? want : (int64_t)resident;                                        \
        if (g_persist_cap > 0 && ctas > g_persist_cap) ctas = g_persist_cap;                                       \
        kern<<<(unsigned)ctas, threads, sm, stream>>>(d_f, idx, w_f, n_cells, k, out_row, o_f, g, n_comp, store_w); \
    } while (0)
#define S3_PARTWARP_C(L, K_, R) do { if (ku == 8) S3_PARTWARP(L, 8, R, 2); else if (per_sm_built == 4) S3_PARTWARP(L, 4, R, 4); else S3_PARTWARP(L, 4, R, 3); } while (0)
#define S3_PARTWARP_R(L) do { if (kr == 1) S3_PARTWARP_C(L, 0, 1); else S3_PARTWARP_C(L, 0, 2); } while (0)
            if (lpc == 16) S3_PARTWARP_R(16); else S3_PARTWARP_R(32);
#undef S3_PARTWARP_R
#undef S3_PARTWARP_C
#undef S3_PARTWARP
            S3_LAUNCH_CHECK();
            note_launch(1);
            return S3_OK;
        }
    }
    if constexpr (std::is_same<Tin, float>::value && std::is_same<Tout, float>::value && MODE == 0) {
        if (g_dense && !wide && vec_ok && k <= 16 && n_comp == 1 && g.n_cols % 4 == 0 && g.row_stride == g.n_cols &&
            g.out_row_stride == g.n_cols && g_chunk_cols == 0) {
            interp_dense_kernel<<<(unsigned)blocks, warps * 32, 0, stream>>>(
                reinterpret_cast<const float*>(data), g.n_cols, idx, reinterpret_cast<const float*>(w), n_cells, k,
                out_row, reinterpret_cast<float*>(out));
            S3_LAUNCH_CHECK();
            note_launch(1);
            return S3_OK;
        }
    }
    const int v = wide ? 8 : wide64 ? VW64 : (vec_ok ? VFULL : 1);
    const int64_t step = (int64_t)32 * v * unroll;
    // all rows share their offset inside a 128-byte line when the pitches are multiples of 128 bytes: shorten the
    // first step by that offset so that every later warp request is line aligned
    g.lead = 0;
    if (v > 1 && (g.row_stride * sizeof(Tin)) % 128 == 0 && (g.comp_stride * sizeof(Tin)) % 128 == 0) {
        const int off = (int)(((uintptr_t)data % 128) / sizeof(Tin));           // multiple of v (16/32-byte aligned)
        g.lead = off;
    }
    int64_t chunk = g_chunk_cols > 0 ? ceil_div(g_chunk_cols, step) * step : g.n_cols + g.lead;
    int64_t n_chunks = ceil_div(g.n_cols + g.lead, chunk);
    if (n_chunks * n_comp > 65535) {
        chunk = ceil_div(ceil_div(g.n_cols + g.lead, 65535 / n_comp), step) * step;
        n_chunks = ceil_div(g.n_cols + g.lead, chunk);
    }
    S3_REQUIRE(n_chunks * n_comp <= 65535, "s3_interp_gather: too many components (%d)", n_comp);
    g.chunk_cols = chunk;
    g.n_chunks = (int)n_chunks;
    const dim3 grid((unsigned)blocks, (unsigned)(n_chunks * n_comp));
    const size_t smem = pairs ? (size_t)warps * k * 2 * sizeof(Tw) : 0;
    const Tin* d_p = reinterpret_cast<const Tin*>(data);
    const Tw* w_p = reinterpret_cast<const Tw*>(w);
    Tout* o_p = reinterpret_cast<Tout*>(out);
#define S3_WARPCELL(VV, UU, PP)                                                                                   \
    do {                                                                                                          \
        auto kern = kunroll == 8 ? interp_warpcell_kernel<Tin, Tw, Tout, VV, MODE, UU, PP, 8>                      \
                  : kunroll == 4 ? interp_warpcell_kernel<Tin, Tw, Tout, VV, MODE, UU, PP, 4>                      \
                                 : interp_warpcell_kernel<Tin, Tw, Tout, VV, MODE, UU, PP, 1>;                     \
        if (g_carveout >= 0) cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, g_carveout); \
        kern<<<grid, warps * 32, smem, stream>>>(d_p, idx, w_p, n_cells, k, out_row, o_p, g);                      \
    } while (0)
#define S3_WARPCELL_UP(VV)                                                                                        \
    do {                                                                                                          \
        if (unroll == 2) { if (pairs) S3_WARPCELL(VV, 2, true); else S3_WARPCELL(VV, 2, false); }                  \
        else { if (pairs) S3_WARPCELL(VV, 1, true); else S3_WARPCELL(VV, 1, false); }                              \
    } while (0)
    if constexpr (std::is_same<Tin, float>::value && std::is_same<Tout, float>::value && MODE == 0) {
        if (wide) {
            S3_WARPCELL_UP(8);
            S3_LAUNCH_CHECK();
            note_launch(1);
            return S3_OK;
        }
    }
    if constexpr (MODE == 1 && std::is_same<Tout, double>::value) {
        if (wide64) {
            S3_WARPCELL_UP(VW64);
            S3_LAUNCH_CHECK();
            note_launch(1);
            return S3_OK;
        }
    }
    if (vec_ok) S3_WARPCELL_UP(VFULL); else S3_WARPCELL_UP(1);
#undef S3_WARPCELL_UP
#undef S3_WARPCELL
    S3_LAUNCH_CHECK();
    note_launch(1);
    return S3_OK;
}

// ---- reconstruction error of a sampled grid (s3_recon_error) ----------------------------------------------------
// The sampled field is gathered back onto the original points with the tables of the other direction (N original points
// queried among the Nc cell centres) and compared there without materialising the [N, D, T] reconstruction:
//   r = sum_j w[p, j] * sampled[idx[p, j], d, t]   (fp32 FMA chain in neighbour order: the gather's MODE 0 products)
//   e = (double) r - (double) original[out_row[p], d, t]
// Grid: one CTA per (point block, component, column tile), the tiles and components of one block adjacent in launch
// order, so that they run together and the block's table rows and original rows are served from L2 to all of them. The
// warps of a CTA walk the points of the block (warp w: points w, w + 8, ...; neighbouring points of the Morton order
// share sampled rows, which L1 serves), each lane owns 8 columns of the 256-column tile. The fp64 column partials of the
// warps are combined in shared memory in warp order, one partial per (block, column) goes to scratch and a second kernel
// reduces them in block order. The reduction tree therefore depends on N only: the results are the same bits for any
// CTA count (key 18) and for any set of other columns in the launch (a time window gives the full launch's columns).
constexpr int kReconWarps = 8;          // warps per CTA
constexpr int kReconBlock = 512;        // points per block: fixed, the order of every sum depends on it
constexpr int kReconTile = 256;         // columns per tile: 32 lanes x 8
constexpr int kReconGroup = 256;        // block partials per group of the first column-reduction pass
static int g_recon_cap = 0;             // key 18: at most this many CTAs per (component, tile), 0 = no cap (tests)

struct ReconGeom {
    int64_t s_row, s_comp;              // sampled: elements between cells / between components
    int64_t o_row, o_comp;              // original: elements between points / between components
    int64_t n_cols;
    int n_comp, n_tiles;
};

// WIDE: one 256-bit load per lane and row (base pointers and strides multiples of 32 bytes; a vector that straddles the
// end of a row stays inside the 32-byte sector of the row's last column and its columns past the end are not used).
// Otherwise the lane owns columns lane + 32 e with scalar loads, and nothing past a row is read.
template <bool WIDE>
__global__ void __launch_bounds__(kReconWarps * 32, 2)
recon_error_kernel(const float* __restrict__ sampled, const float* __restrict__ original, const int32_t* __restrict__ idx,
                   const float* __restrict__ w, const int32_t* __restrict__ out_row, int64_t n_points, int k,
                   const ReconGeom g, int64_t n_blocks, int64_t n_slots, double* __restrict__ col_part,
                   double* __restrict__ pt_part) {
    __shared__ double s_red[3][kReconWarps][kReconTile];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n_xt = g.n_comp * g.n_tiles;
    const int xt = (int)(blockIdx.x % n_xt);
    const int64_t slot = blockIdx.x / n_xt;
    const int comp = xt / g.n_tiles, tile = xt % g.n_tiles;
    const int64_t n_cols = g.n_cols, dt = (int64_t)g.n_comp * n_cols;
    const int64_t tile0 = (int64_t)tile * kReconTile;
    const float* s_base = sampled + (int64_t)comp * g.s_comp;
    const float* o_base = original + (int64_t)comp * g.o_comp;
    auto col_in_tile = [&](int e) { return WIDE ? lane * 8 + e : lane + 32 * e; };

    for (int64_t pb = slot; pb < n_blocks; pb += n_slots) {
        double se[8], sr[8], mx[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) se[e] = sr[e] = mx[e] = 0.0;
        const int64_t p_end = min(n_points, (pb + 1) * kReconBlock);
        for (int64_t p = pb * kReconBlock + warp; p < p_end; p += kReconWarps) {
            int32_t idx_lo = 0, idx_hi = 0;
            float w_lo = 0.f, w_hi = 0.f;
            if (lane < k) { idx_lo = idx[p * k + lane]; w_lo = w[p * k + lane]; }
            if (lane + 32 < k) { idx_hi = idx[p * k + lane + 32]; w_hi = w[p * k + lane + 32]; }
            const int64_t orow = out_row ? (int64_t)out_row[p] : p;
            const float* orig = o_base + orow * g.o_row;
            float o[8], acc[8];
#pragma unroll
            for (int e = 0; e < 8; ++e) { o[e] = 0.f; acc[e] = 0.f; }
            const int64_t c0 = tile0 + lane * 8;
            if (WIDE) {
                if (c0 < n_cols) {
                    const Vec<float, 8> x = ld_vec<float, 8>(orig + c0);
#pragma unroll
                    for (int e = 0; e < 8; ++e) o[e] = x.v[e];
                }
            } else {
#pragma unroll
                for (int e = 0; e < 8; ++e) {
                    const int64_t c = tile0 + col_in_tile(e);
                    if (c < n_cols) o[e] = orig[c];
                }
            }
#pragma unroll 4
            for (int j = 0; j < k; ++j) {
                const int32_t r = __shfl_sync(0xffffffffu, (j & 32) ? idx_hi : idx_lo, j & 31);
                const float wj = __shfl_sync(0xffffffffu, (j & 32) ? w_hi : w_lo, j & 31);
                const float* src = s_base + (int64_t)r * g.s_row;
                if (WIDE) {
                    if (c0 < n_cols) {
                        const Vec<float, 8> x = ld_vec<float, 8>(src + c0);
#pragma unroll
                        for (int e = 0; e < 8; ++e) acc[e] = fmaf(wj, x.v[e], acc[e]);
                    }
                } else {
#pragma unroll
                    for (int e = 0; e < 8; ++e) {
                        const int64_t c = tile0 + col_in_tile(e);
                        if (c < n_cols) acc[e] = fmaf(wj, src[c], acc[e]);
                    }
                }
            }
            double ps = 0.0;                                  // sum over this lane's columns of e^2
#pragma unroll
            for (int e = 0; e < 8; ++e) {
                if (tile0 + col_in_tile(e) < n_cols) {       // the n_cols % 8 tail of the last vector is not a column
                    const double d = (double)acc[e] - (double)o[e];
                    const double d2 = d * d;
                    se[e] += d2;
                    sr[e] += (double)o[e] * (double)o[e];
                    mx[e] = fmax(mx[e], fabs(d));
                    ps += d2;
                }
            }
            if (pt_part) {
#pragma unroll
                for (int off = 16; off > 0; off >>= 1) ps += __shfl_xor_sync(0xffffffffu, ps, off);
                if (lane == 0) pt_part[((int64_t)tile * n_points + p) * g.n_comp + comp] = ps;
            }
        }
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            s_red[0][warp][col_in_tile(e)] = se[e];
            s_red[1][warp][col_in_tile(e)] = sr[e];
            s_red[2][warp][col_in_tile(e)] = mx[e];
        }
        __syncthreads();
        const int t = threadIdx.x;
        if (tile0 + t < n_cols) {
            double a = 0.0, b = 0.0, m = 0.0;
#pragma unroll
            for (int q = 0; q < kReconWarps; ++q) {
                a += s_red[0][q][t];
                b += s_red[1][q][t];
                m = fmax(m, s_red[2][q][t]);
            }
            double* part = col_part + pb * 3 * dt + (int64_t)comp * n_cols + tile0 + t;
            part[0] = a;
            part[dt] = b;
            part[2 * dt] = m;
        }
        __syncthreads();
    }
}

// in: rows of [3][dt] partials (sum, sum, max); group y reduces rows [y * rows_per_group, ...) in row order into
// out{0,1,2}[y * ld_out + c]
__global__ void recon_reduce_cols_kernel(const double* __restrict__ in, int64_t n_rows, int64_t rows_per_group,
                                         int64_t dt, double* out0, double* out1, double* out2, int64_t ld_out) {
    const int64_t c3 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c3 >= 3 * dt) return;
    const int plane = (int)(c3 / dt);
    const int64_t c = c3 % dt;
    const int64_t r0 = (int64_t)blockIdx.y * rows_per_group;
    const int64_t r1 = min(n_rows, r0 + rows_per_group);
    double acc = 0.0;
    for (int64_t r = r0; r < r1; ++r) {
        const double v = in[r * 3 * dt + c3];
        acc = plane == 2 ? fmax(acc, v) : acc + v;
    }
    double* out = plane == 0 ? out0 : plane == 1 ? out1 : out2;
    out[blockIdx.y * ld_out + c] = acc;
}

// point_sq_err[out_row[p], d] += sum over the tiles, in tile order, of the (point, tile) partials
__global__ void recon_reduce_points_kernel(const double* __restrict__ pt_part, int64_t n_points, int n_comp, int n_tiles,
                                           const int32_t* __restrict__ out_row, double* __restrict__ point_sq_err) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t n = n_points * n_comp;
    if (i >= n) return;
    double s = 0.0;
    for (int t = 0; t < n_tiles; ++t) s += pt_part[(int64_t)t * n + i];
    const int64_t p = i / n_comp;
    const int64_t orow = out_row ? (int64_t)out_row[p] : p;
    point_sq_err[orow * n_comp + i % n_comp] += s;
}

static int launch_recon_error(const float* sampled, const float* original, const int32_t* idx, const float* w,
                              const int32_t* out_row, int64_t n_points, int k, ReconGeom g, double* sq_err,
                              double* sq_ref, double* max_abs, double* point_sq_err, cudaStream_t stream) {
    const int64_t dt = (int64_t)g.n_comp * g.n_cols;
    const int64_t n_blocks = ceil_div(n_points, kReconBlock);
    const int64_t n_xt = (int64_t)g.n_comp * g.n_tiles;
    int64_t n_slots = n_blocks;
    if (g_recon_cap > 0 && n_slots > g_recon_cap) n_slots = g_recon_cap;
    S3_REQUIRE(n_xt * n_slots < ((int64_t)1 << 31), "s3_recon_error: too many CTAs (%lld tiles x %lld blocks)",
               (long long)n_xt, (long long)n_slots);
    const int64_t n_groups = ceil_div(n_blocks, kReconGroup);
    S3_REQUIRE(n_groups <= 65535, "s3_recon_error: too many points (%lld)", (long long)n_points);
    Scratch scratch(stream);
    double *col_part = nullptr, *grp_part = nullptr, *pt_part = nullptr;
    S3_TRY(scratch.alloc(&col_part, (size_t)(n_blocks * 3 * dt)));
    if (point_sq_err) S3_TRY(scratch.alloc(&pt_part, (size_t)(g.n_tiles * n_points * g.n_comp)));
    const bool wide = (uintptr_t)sampled % 32 == 0 && (uintptr_t)original % 32 == 0 && g.s_row % 8 == 0 &&
                      g.s_comp % 8 == 0 && g.o_row % 8 == 0 && g.o_comp % 8 == 0;
    const unsigned ctas = (unsigned)(n_xt * n_slots);
    if (wide)
        recon_error_kernel<true><<<ctas, kReconWarps * 32, 0, stream>>>(sampled, original, idx, w, out_row, n_points, k,
                                                                         g, n_blocks, n_slots, col_part, pt_part);
    else
        recon_error_kernel<false><<<ctas, kReconWarps * 32, 0, stream>>>(sampled, original, idx, w, out_row, n_points, k,
                                                                          g, n_blocks, n_slots, col_part, pt_part);
    S3_LAUNCH_CHECK();
    const unsigned col_ctas = (unsigned)ceil_div(3 * dt, 256);
    if (n_groups == 1) {
        recon_reduce_cols_kernel<<<dim3(col_ctas, 1), 256, 0, stream>>>(col_part, n_blocks, n_blocks, dt, sq_err,
                                                                         sq_ref, max_abs, 0);
        S3_LAUNCH_CHECK();
    } else {
        S3_TRY(scratch.alloc(&grp_part, (size_t)(n_groups * 3 * dt)));
        recon_reduce_cols_kernel<<<dim3(col_ctas, (unsigned)n_groups), 256, 0, stream>>>(
            col_part, n_blocks, kReconGroup, dt, grp_part, grp_part + dt, grp_part + 2 * dt, 3 * dt);
        S3_LAUNCH_CHECK();
        recon_reduce_cols_kernel<<<dim3(col_ctas, 1), 256, 0, stream>>>(grp_part, n_groups, n_groups, dt, sq_err,
                                                                         sq_ref, max_abs, 0);
        S3_LAUNCH_CHECK();
    }
    if (point_sq_err) {
        recon_reduce_points_kernel<<<(unsigned)ceil_div(n_points * g.n_comp, 256), 256, 0, stream>>>(
            pt_part, n_points, g.n_comp, g.n_tiles, out_row, point_sq_err);
        S3_LAUNCH_CHECK();
    }
    note_launch(point_sq_err ? (n_groups == 1 ? 3 : 4) : (n_groups == 1 ? 2 : 3));
    return S3_OK;
}

}  // namespace s3

using namespace s3;

// A/B harness hook (scripts/, tests of the variants): NOT declared in include/s3b200.h. Keys: see the knobs above;
// 10 / 11 / 14 / 17 belong to the tensor-core Gram and projection kernels (csrc/svd.cu).
extern "C" int s3x_tune(int key, int value) {
    switch (key) {
        case 1: S3_REQUIRE(value >= 1 && value <= 16, "s3x_tune: warps per CTA must be 1..16"); g_warps_per_cta = value; return S3_OK;
        case 2: S3_REQUIRE(value >= 0 && value <= 2, "s3x_tune: unroll must be 0 (by k), 1 or 2"); g_unroll = value; return S3_OK;
        case 3: S3_REQUIRE(value >= -1 && value <= 1, "s3x_tune: pairs must be -1 (by k), 0 or 1"); g_pairs = value; return S3_OK;
        case 4: S3_REQUIRE(value >= 0, "s3x_tune: window columns must be >= 0"); g_chunk_cols = value; return S3_OK;
        case 5: S3_REQUIRE(value >= -1 && value <= 100, "s3x_tune: carve-out must be -1 or 0..100"); g_carveout = value; return S3_OK;
        case 6: S3_REQUIRE(value >= -1 && value <= 1, "s3x_tune: wide must be -1 (auto), 0 or 1"); g_wide = value; return S3_OK;
        case 16: S3_REQUIRE(value == 0 || value == 1, "s3x_tune: fp64 wide path must be 0 or 1"); g_wide64 = value; return S3_OK;
        case 9: S3_REQUIRE(value == 0 || value == 1, "s3x_tune: dense kernel must be 0 or 1"); g_dense = value; return S3_OK;
        case 7: S3_REQUIRE(value == 0 || value == 1 || value == 4 || value == 8, "s3x_tune: neighbour-loop unroll must be 0 (auto), 1, 4 or 8"); g_kunroll = value; return S3_OK;
        case 8: S3_REQUIRE(value >= -1 && value <= 1, "s3x_tune: part-warp kernel must be -1 (short rows), 0 (never) or 1 (whenever possible)"); g_persistent = value; return S3_OK;
        case 12: S3_REQUIRE(value == 0 || value == 3 || value == 4, "s3x_tune: resident CTAs per SM must be 0 (by row length), 3 or 4"); g_persist_ctas = value; return S3_OK;
        case 15: S3_REQUIRE(value >= 0 && value <= (1 << 20), "s3x_tune: part-warp CTA cap must be 0 (none) or >= 1"); g_persist_cap = value; return S3_OK;
        case 13: S3_REQUIRE(value == 0 || value == 16 || value == 32, "s3x_tune: lanes per cell must be 0 (by row length), 16 or 32"); g_lanes_per_cell = value; return S3_OK;
        case 30: S3_REQUIRE(value == 0 || value == 1, "s3x_tune: curve must be 0 (Morton) or 1 (Hilbert)"); g_curve = value; return S3_OK;
        case 10: S3_REQUIRE(value >= 1 && value <= (1 << 20), "s3x_tune: K-blocks per TMEM segment must be >= 1"); g_tc_seg_kblocks = value; return S3_OK;
        case 11: S3_REQUIRE(value >= 1 && value <= (1 << 20), "s3x_tune: segments per fp64 flush must be >= 1"); g_tc_flush_segments = value; return S3_OK;
        case 14: S3_REQUIRE(value == 0 || value == 1, "s3x_tune: paired Gram kernel must be 0 or 1"); g_tc_pair = value; return S3_OK;
        case 17: S3_REQUIRE(value >= 0, "s3x_tune: plane-row cap must be 0 (none) or >= 1"); g_plane_rows_cap = value; return S3_OK;
        case 18: S3_REQUIRE(value >= 0, "s3x_tune: reconstruction-error CTA cap must be 0 (none) or >= 1"); g_recon_cap = value; return S3_OK;
        case 19: S3_REQUIRE(value >= 0, "s3x_tune: low-rank error CTA cap must be 0 (none) or >= 1"); g_lowrank_cap = value; return S3_OK;
    }
    s3::set_error("s3x_tune: unknown key %d", key);
    return S3_ERR_INVALID;
}

extern "C" int s3_interp_gather_strided(const void* d_data, int data_dtype, int64_t n_src, int n_comp, int64_t n_cols,
                                        int64_t row_stride, int64_t comp_stride, const int32_t* d_idx, const void* d_w,
                                        int64_t n_cells, int k, const int32_t* d_out_row, void* d_out, int out_dtype,
                                        int64_t out_row_stride, int64_t out_comp_stride, void* stream) {
    S3_REQUIRE(n_cells >= 0 && n_cols >= 0 && n_comp >= 0, "s3_interp_gather: bad sizes");
    if (n_cells == 0 || n_cols == 0 || n_comp == 0) return S3_OK;     // empty grids / rows: nothing to do (buffers may be NULL)
    S3_REQUIRE(d_data && d_idx && d_w && d_out, "s3_interp_gather: NULL argument");
    S3_REQUIRE(k >= 1 && k <= 64, "s3_interp_gather: k=%d out of range [1, 64]", k);
    S3_REQUIRE(n_src >= 1, "s3_interp_gather: bad sizes");
    S3_REQUIRE(comp_stride >= n_cols || n_comp == 1, "s3_interp_gather: component stride %lld < %lld columns",
               (long long)comp_stride, (long long)n_cols);
    S3_REQUIRE(out_comp_stride >= n_cols || n_comp == 1, "s3_interp_gather: result component stride too small");
    S3_REQUIRE(row_stride >= (n_comp - 1) * comp_stride + n_cols && out_row_stride >= (n_comp - 1) * out_comp_stride + n_cols,
               "s3_interp_gather: row stride smaller than a row");
    cudaStream_t st = (cudaStream_t)stream;
    InterpGeom g{};
    g.row_stride = row_stride; g.comp_stride = comp_stride;
    g.out_row_stride = out_row_stride; g.out_comp_stride = out_comp_stride;
    g.n_cols = n_cols;
    // dense components on both sides: one long row per point (fewer partial warp steps)
    if (n_comp > 1 && comp_stride == n_cols && out_comp_stride == n_cols) {
        g.n_cols = n_cols * n_comp;
        n_comp = 1;
    }
    if (n_comp == 1) {                      // a single component: its stride means nothing (and must not spoil the alignment tests)
        g.comp_stride = 0;
        g.out_comp_stride = 0;
    }
    if (data_dtype == S3_F32 && out_dtype == S3_F32)
        return launch_interp<float, float, float, 0>(d_data, d_idx, d_w, n_cells, k, d_out_row, d_out, n_comp, g, st);
    if (data_dtype == S3_F32 && out_dtype == S3_F64)
        return launch_interp<float, double, double, 1>(d_data, d_idx, d_w, n_cells, k, d_out_row, d_out, n_comp, g, st);
    if (data_dtype == S3_F64 && out_dtype == S3_F64)
        return launch_interp<double, double, double, 1>(d_data, d_idx, d_w, n_cells, k, d_out_row, d_out, n_comp, g, st);
    s3::set_error("s3_interp_gather: unsupported dtype combination data=%d out=%d", data_dtype, out_dtype);
    return S3_ERR_UNSUPPORTED;
}

extern "C" int s3_recon_error(const void* d_sampled, int sampled_dtype, int64_t n_sampled, int n_comp, int64_t n_cols,
                              int64_t s_row_stride, int64_t s_comp_stride, const void* d_original, int original_dtype,
                              int64_t n_points, int64_t o_row_stride, int64_t o_comp_stride, const int32_t* d_idx,
                              const float* d_w, const int32_t* d_out_row, int k, double* d_sq_err, double* d_sq_ref,
                              double* d_max_abs, double* d_point_sq_err, void* stream) {
    S3_REQUIRE(n_points >= 0 && n_cols >= 0 && n_comp >= 0 && n_sampled >= 0, "s3_recon_error: bad sizes");
    if (sampled_dtype != S3_F32 || original_dtype != S3_F32) {
        s3::set_error("s3_recon_error: fields must be fp32 (sampled dtype %d, original dtype %d); the error of fp64 "
                      "fields is not implemented", sampled_dtype, original_dtype);
        return S3_ERR_UNSUPPORTED;
    }
    S3_REQUIRE(k >= 1 && k <= 64, "s3_recon_error: k=%d out of range [1, 64]", k);
    if (n_cols == 0 || n_comp == 0) return S3_OK;
    S3_REQUIRE(d_sq_err && d_sq_ref && d_max_abs, "s3_recon_error: NULL result");
    cudaStream_t st = (cudaStream_t)stream;
    if (n_points == 0) {                    // no points: zero sums, nothing added to the point map
        const size_t bytes = (size_t)n_comp * n_cols * sizeof(double);
        S3_CUDA(cudaMemsetAsync(d_sq_err, 0, bytes, st));
        S3_CUDA(cudaMemsetAsync(d_sq_ref, 0, bytes, st));
        S3_CUDA(cudaMemsetAsync(d_max_abs, 0, bytes, st));
        return S3_OK;
    }
    S3_REQUIRE(d_sampled && d_original && d_idx && d_w, "s3_recon_error: NULL argument");
    S3_REQUIRE(n_sampled >= 1, "s3_recon_error: no sampled cells");
    S3_REQUIRE((s_comp_stride >= n_cols && o_comp_stride >= n_cols) || n_comp == 1,
               "s3_recon_error: component stride smaller than a row");
    S3_REQUIRE(s_row_stride >= (n_comp - 1) * s_comp_stride + n_cols && o_row_stride >= (n_comp - 1) * o_comp_stride + n_cols,
               "s3_recon_error: row stride smaller than a row");
    ReconGeom g{};
    g.s_row = s_row_stride; g.s_comp = n_comp == 1 ? 0 : s_comp_stride;
    g.o_row = o_row_stride; g.o_comp = n_comp == 1 ? 0 : o_comp_stride;
    g.n_cols = n_cols;
    g.n_comp = n_comp;
    g.n_tiles = (int)ceil_div(n_cols, kReconTile);
    S3_REQUIRE(ceil_div(n_cols, kReconTile) * n_comp < (1 << 20), "s3_recon_error: too many columns");
    return launch_recon_error(reinterpret_cast<const float*>(d_sampled), reinterpret_cast<const float*>(d_original),
                              d_idx, d_w, d_out_row, n_points, k, g, d_sq_err, d_sq_ref, d_max_abs, d_point_sq_err, st);
}

extern "C" int s3_interp_gather(const void* d_data, int data_dtype, int64_t n_src, int64_t row_len,
                                const int32_t* d_idx, const void* d_w, int64_t n_cells, int k,
                                const int32_t* d_out_row, void* d_out, int out_dtype, void* stream) {
    return s3_interp_gather_strided(d_data, data_dtype, n_src, 1, row_len, row_len, row_len, d_idx, d_w, n_cells, k,
                                    d_out_row, d_out, out_dtype, row_len, row_len, stream);
}
