// Level-synchronous octree/quadtree refinement kernels (device side of SamplingTree, s_cube.py).
//
// Cell state is a structure of arrays indexed by the reference's cell index (creation order):
//   center fp64 [cap, dim], level int32 [cap], gain fp64 [cap], metric fp64 [cap], flags uint8 [cap].
#include "common.cuh"
#include "geometry.cuh"
#include "stl.cuh"
#include "knn.cuh"
#include "radix_sort.cuh"
#include "../../include/s3b200.h"

namespace s3 {

const KnnIndex* knn_index_of(const s3_knn_t* h);

constexpr uint8_t kFlagLeaf = 1;
constexpr uint8_t kFlagInvalid = 2;

// child / node offsets, order CH = swu, nwu, neu, seu, swl, nwl, nel, sel (s_cube.py:29, :188-194)
__device__ __forceinline__ void direction(int dim, int c, int* d) {
    const int dx[4] = {-1, -1, 1, 1};
    const int dy[4] = {-1, 1, 1, -1};
    d[0] = dx[c & 3];
    d[1] = dy[c & 3];
    if (dim == 3) d[2] = (c < 4) ? 1 : -1;
}

// ---------------------------------------------------------------- children (s_cube.py:399-445, :865-902)
__global__ void __launch_bounds__(256)
cells_refine_kernel(double* __restrict__ center, int32_t* __restrict__ level, uint8_t* __restrict__ flags,
                    const int64_t* __restrict__ parents, int64_t n_parents, int64_t first_child, int dim, double width) {
    const int nch = 1 << dim;
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_parents * nch) return;
    const int64_t pi = t / nch;
    const int c = (int)(t % nch);
    const int64_t p = parents[pi];
    const int64_t child = first_child + t;
    const int lp = level[p];
    // offset = (+-1 * 0.25 * width) / 2^level : exact power-of-two scaling of width (s_cube.py:441)
    const double off = ldexp(width, -(lp + 2));
    int d[3];
    direction(dim, c, d);
    for (int a = 0; a < dim; ++a) {
        const double pc = center[p * dim + a];
        center[child * dim + a] = __dadd_rn(pc, d[a] > 0 ? off : -off);
    }
    level[child] = lp + 1;
    flags[child] = kFlagLeaf;
    if (c == 0) flags[p] = (uint8_t)(flags[p] & ~kFlagLeaf);
}

// ---------------------------------------------------------------- gain (s_cube.py:207-241, :1840-1859)
// One CTA per cell: warp 0 predicts the metric at the cell centre, warps 1..2^d at the centres of the
// would-be children; thread 0 then evaluates sum|m0 - mj| and the gain in the reference's rounding order.
template <int DIM>
__global__ void __launch_bounds__(32 * ((1 << DIM) + 1))
cells_gain_kernel(KnnView ix, const double* __restrict__ center, const int32_t* __restrict__ level,
                  const int64_t* __restrict__ cells, int64_t first, int64_t n, int k, double width, double gain0,
                  int sdm_order, double* __restrict__ metric, double* __restrict__ gain) {
    constexpr int NW = (1 << DIM) + 1;
    __shared__ double s_lb[NW][kKnnStack];
    __shared__ int32_t s_node[NW][kKnnStack];
    __shared__ double s_pred[NW];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t cell = cells ? cells[blockIdx.x] : first + blockIdx.x;
    const int lv = level[cell];
    double q[3];
    if (warp == 0) {
#pragma unroll
        for (int a = 0; a < DIM; ++a) q[a] = center[cell * DIM + a];
    } else {
        const double off = ldexp(width, -(lv + 2));
        int d[3];
        direction(DIM, warp - 1, d);
#pragma unroll
        for (int a = 0; a < DIM; ++a) q[a] = __dadd_rn(center[cell * DIM + a], d[a] > 0 ? off : -off);
    }
    WarpTopK best = warp_knn_search<DIM>(ix, q, k, s_lb[warp], s_node[warp]);
    const double pred = warp_idw_predict(best, k, ix.values);
    if (lane == 0) s_pred[warp] = pred;
    __syncthreads();
    if (threadIdx.x == 0) {
        const double m0 = s_pred[0];
        double a[1 << DIM];
#pragma unroll
        for (int j = 0; j < (1 << DIM); ++j) a[j] = fabs(__dsub_rn(m0, s_pred[j + 1]));
        double sdm;
        if (DIM == 3 && sdm_order == 1) {
            // torch fp64 sum(dim=1) over 8 columns on AVX2/AVX512 hosts (probed):
            sdm = __dadd_rn(__dadd_rn(__dadd_rn(__dadd_rn(a[0], a[4]), __dadd_rn(a[1], a[5])), __dadd_rn(a[2], a[6])),
                            __dadd_rn(a[3], a[7]));
        } else {
            sdm = a[0];
#pragma unroll
            for (int j = 1; j < (1 << DIM); ++j) sdm = __dadd_rn(sdm, a[j]);
        }
        // numba fastmath form of s_cube.py:1859 (probed): (((1/2^d) * c^d) * sdm) / gain0, c = width / 2^level
        const double c = ldexp(width, -lv);
        double qd = __dmul_rn(c, c);
        if (DIM == 3) qd = __dmul_rn(qd, c);
        const double g = __ddiv_rn(__dmul_rn(__dmul_rn(1.0 / (1 << DIM), qd), sdm), gain0);
        gain[cell] = g;
        metric[cell] = m0;
    }
}

// ---------------------------------------------------------------- geometry mask (s_cube.py:669-732, :1816-1837)
// STL geometries evaluated beforehand by stl_inside_kernel (one flag per node): slot i holds geometry geom[i]
constexpr int kMaxStlPre = 4;
struct StlPre {
    const uint8_t* inside[kMaxStlPre];
    int geom[kMaxStlPre];
    int n;
};
__device__ __forceinline__ const uint8_t* stl_pre_of(const StlPre& pre, int g) {
    for (int i = 0; i < pre.n; ++i)
        if (pre.geom[i] == g) return pre.inside[i];
    return nullptr;
}

__global__ void __launch_bounds__(128)
cells_mask_kernel(const double* __restrict__ center, const int32_t* __restrict__ level,
                  const int64_t* __restrict__ cells, int64_t first, int64_t n, int dim, double width,
                  const int32_t* __restrict__ geom_hdr, const double* __restrict__ geom_par, int n_geoms,
                  int only_geom, int refine_mode, int apply, uint8_t* __restrict__ out_invalid,
                  uint8_t* __restrict__ flags, double* __restrict__ gain, const StlPre pre) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    const int64_t cell = cells ? cells[t] : first + t;
    const int nn = 1 << dim;
    const double h = ldexp(width, -(level[cell] + 1));  // 0.5 * width / 2^level (s_cube.py:698)
    double node[8][3];
    for (int j = 0; j < nn; ++j) {
        int d[3];
        direction(dim, j, d);
        for (int a = 0; a < dim; ++a) node[j][a] = __dadd_rn(center[cell * dim + a], d[a] > 0 ? h : -h);
    }
    bool invalid = false;
    for (int g = 0; g < n_geoms && !invalid; ++g) {
        if (only_geom >= 0 && g != only_geom) continue;
        GeomHdr hd;
        hd.type = geom_hdr[4 * g];
        hd.keep_inside = geom_hdr[4 * g + 1];
        hd.offset = geom_hdr[4 * g + 2];
        hd.n_extra = geom_hdr[4 * g + 3];
        if (hd.type == GEOM_CUSTOM) continue;
        int n_in = 0;
        const uint8_t* staged = hd.type == GEOM_STL ? stl_pre_of(pre, g) : nullptr;
        if (staged) {
            for (int j = 0; j < nn; ++j) n_in += staged[t * nn + j];
        } else {
            for (int j = 0; j < nn; ++j) n_in += point_in_geometry(hd, geom_par + hd.offset, node[j], dim) ? 1 : 0;
        }
        invalid = apply_mask(n_in, nn, hd.keep_inside != 0, refine_mode != 0);
    }
    out_invalid[t] = invalid ? 1 : 0;
    if (apply && invalid) {
        // s_cube.py:721-731: children = [], gain = 0, removed from the leaf set
        flags[cell] = kFlagInvalid;
        gain[cell] = 0.0;
    }
}

// check_cell on explicit node sets: nodes fp64 [n, nn, dim]
__global__ void __launch_bounds__(128)
nodes_mask_kernel(const double* __restrict__ nodes, int64_t n, int nn, int dim, const int32_t* __restrict__ geom_hdr,
                  const double* __restrict__ geom_par, int n_geoms, int only_geom, int refine_mode,
                  uint8_t* __restrict__ out_invalid, const StlPre pre) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    bool invalid = false;
    for (int g = 0; g < n_geoms && !invalid; ++g) {
        if (only_geom >= 0 && g != only_geom) continue;
        GeomHdr hd;
        hd.type = geom_hdr[4 * g];
        hd.keep_inside = geom_hdr[4 * g + 1];
        hd.offset = geom_hdr[4 * g + 2];
        hd.n_extra = geom_hdr[4 * g + 3];
        if (hd.type == GEOM_CUSTOM) continue;
        int n_in = 0;
        const uint8_t* staged = hd.type == GEOM_STL ? stl_pre_of(pre, g) : nullptr;
        for (int j = 0; j < nn; ++j) {
            if (staged) { n_in += staged[t * nn + j]; continue; }
            double p[3] = {0, 0, 0};
            for (int a = 0; a < dim; ++a) p[a] = nodes[(t * nn + j) * dim + a];
            n_in += point_in_geometry(hd, geom_par + hd.offset, p, dim) ? 1 : 0;
        }
        invalid = apply_mask(n_in, nn, hd.keep_inside != 0, refine_mode != 0);
    }
    out_invalid[t] = invalid ? 1 : 0;
}

__global__ void __launch_bounds__(128)
points_inside_kernel(const double* __restrict__ pts, int64_t n, int dim, const int32_t* __restrict__ geom_hdr,
                     const double* __restrict__ geom_par, int g, uint8_t* __restrict__ out_inside) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    GeomHdr hd;
    hd.type = geom_hdr[4 * g];
    hd.keep_inside = geom_hdr[4 * g + 1];
    hd.offset = geom_hdr[4 * g + 2];
    hd.n_extra = geom_hdr[4 * g + 3];
    double p[3] = {0, 0, 0};
    for (int a = 0; a < dim; ++a) p[a] = pts[t * dim + a];
    out_inside[t] = point_in_geometry(hd, geom_par + hd.offset, p, dim) ? 1 : 0;
}

// ---------------------------------------------------------------- selection (s_cube.py:599-602)
// top-k leaves by (gain descending, index ascending)
struct SelectState {
    uint64_t prefix;      // key bits decided so far (high bits)
    uint64_t remaining;   // how many still to take among keys matching the prefix
    uint32_t hist[256];
    uint32_t ticket;
    uint32_t pad;
};

constexpr int kSelTile = 2048;

__device__ __forceinline__ uint64_t leaf_key(const double* gain, const uint8_t* flags, int64_t i) {
    return (flags[i] & kFlagLeaf) ? f64_to_ordered(gain[i]) : 0ull;
}

__global__ void select_init_kernel(SelectState* st, uint64_t k) {
    if (threadIdx.x == 0) { st->prefix = 0; st->remaining = k; st->ticket = 0; }
    st->hist[threadIdx.x] = 0;
}

// One radix-select pass over byte `pass` (7 = most significant): histogram of that byte among the
// keys whose higher bytes equal the prefix; the last CTA to finish picks the digit that contains the
// remaining-th largest key.
__global__ void __launch_bounds__(256)
select_pass_kernel(const double* __restrict__ gain, const uint8_t* __restrict__ flags, int64_t n, int pass,
                   SelectState* st) {
    __shared__ uint32_t sh[256];
    __shared__ bool is_last;
    sh[threadIdx.x] = 0;
    __syncthreads();
    const int shift = pass * 8;
    const uint64_t prefix = st->prefix;
    const uint64_t himask = pass == 7 ? 0ull : (~0ull << (shift + 8));
    const int64_t base = (int64_t)blockIdx.x * kSelTile;
    for (int j = threadIdx.x; j < kSelTile; j += 256) {
        const int64_t i = base + j;
        if (i < n && (flags[i] & kFlagLeaf)) {
            const uint64_t key = f64_to_ordered(gain[i]);
            if ((key & himask) == (prefix & himask)) atomicAdd(&sh[(key >> shift) & 255u], 1u);
        }
    }
    __syncthreads();
    if (sh[threadIdx.x]) atomicAdd(&st->hist[threadIdx.x], sh[threadIdx.x]);
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) is_last = (atomicAdd(&st->ticket, 1u) == gridDim.x - 1);
    __syncthreads();
    if (!is_last) return;
    __threadfence();
    if (threadIdx.x == 0) {
        uint64_t rem = st->remaining;
        int digit = 0;
        for (int d = 255; d >= 0; --d) {
            const uint32_t c = ((volatile uint32_t*)st->hist)[d];
            if (rem <= c) { digit = d; break; }
            rem -= c;
        }
        st->prefix = (prefix & himask) | ((uint64_t)digit << shift);
        st->remaining = rem;
        st->ticket = 0;
    }
    __syncthreads();
    ((volatile uint32_t*)st->hist)[threadIdx.x] = 0;
}

// counts per tile: keys > T and keys == T (T = st->prefix after the 8 passes)
__global__ void __launch_bounds__(256)
select_count_kernel(const double* __restrict__ gain, const uint8_t* __restrict__ flags, int64_t n,
                    const SelectState* st, uint32_t* __restrict__ cnt_gt, uint32_t* __restrict__ cnt_eq) {
    __shared__ uint32_t s_gt, s_eq;
    if (threadIdx.x == 0) { s_gt = 0; s_eq = 0; }
    __syncthreads();
    const uint64_t T = st->prefix;
    const int64_t base = (int64_t)blockIdx.x * kSelTile;
    uint32_t gt = 0, eq = 0;
    for (int j = threadIdx.x; j < kSelTile; j += 256) {
        const int64_t i = base + j;
        if (i < n && (flags[i] & kFlagLeaf)) {
            const uint64_t key = f64_to_ordered(gain[i]);
            gt += key > T;
            eq += key == T;
        }
    }
    for (int o = 16; o > 0; o >>= 1) {
        gt += __shfl_xor_sync(0xffffffffu, gt, o);
        eq += __shfl_xor_sync(0xffffffffu, eq, o);
    }
    if ((threadIdx.x & 31) == 0) { atomicAdd(&s_gt, gt); atomicAdd(&s_eq, eq); }
    __syncthreads();
    if (threadIdx.x == 0) { cnt_gt[blockIdx.x] = s_gt; cnt_eq[blockIdx.x] = s_eq; }
}

// exclusive scans of both tile-count arrays (single CTA; nblocks is small)
__global__ void __launch_bounds__(1024)
select_scan_kernel(uint32_t* __restrict__ cnt_gt, uint32_t* __restrict__ cnt_eq, int nblocks, uint32_t* totals) {
    __shared__ uint32_t pg[1024], pe[1024];
    const int t = threadIdx.x;
    const int chunk = (nblocks + 1023) / 1024;
    const int lo = t * chunk, hi = min(lo + chunk, nblocks);
    uint32_t sg = 0, se = 0;
    for (int i = lo; i < hi; ++i) { sg += cnt_gt[i]; se += cnt_eq[i]; }
    pg[t] = sg; pe[t] = se;
    __syncthreads();
    for (int off = 1; off < 1024; off <<= 1) {
        uint32_t a = t >= off ? pg[t - off] : 0, b = t >= off ? pe[t - off] : 0;
        __syncthreads();
        pg[t] += a; pe[t] += b;
        __syncthreads();
    }
    uint32_t rg = t ? pg[t - 1] : 0, re = t ? pe[t - 1] : 0;
    for (int i = lo; i < hi; ++i) {
        uint32_t a = cnt_gt[i], b = cnt_eq[i];
        cnt_gt[i] = rg; cnt_eq[i] = re;
        rg += a; re += b;
    }
    if (t == 1023) { totals[0] = pg[1023]; totals[1] = pe[1023]; }
}

// ordered compaction: all keys > T (index order), then the first `remaining` keys == T (index order)
__global__ void __launch_bounds__(256)
select_scatter_kernel(const double* __restrict__ gain, const uint8_t* __restrict__ flags, int64_t n,
                      const SelectState* st, const uint32_t* __restrict__ off_gt, const uint32_t* __restrict__ off_eq,
                      const uint32_t* __restrict__ totals, uint64_t* __restrict__ out_key, uint32_t* __restrict__ out_idx) {
    __shared__ uint32_t w_gt[8], w_eq[8];
    __shared__ uint32_t run_gt, run_eq;
    const uint64_t T = st->prefix;
    const uint32_t take_eq = (uint32_t)st->remaining;
    const uint32_t total_gt = totals[0];
    if (threadIdx.x == 0) { run_gt = off_gt[blockIdx.x]; run_eq = off_eq[blockIdx.x]; }
    __syncthreads();
    const int64_t base = (int64_t)blockIdx.x * kSelTile;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int j0 = 0; j0 < kSelTile; j0 += 256) {
        const int64_t i = base + j0 + threadIdx.x;
        uint64_t key = 0;
        bool gt = false, eq = false;
        if (i < n && (flags[i] & kFlagLeaf)) {
            key = f64_to_ordered(gain[i]);
            gt = key > T;
            eq = key == T;
        }
        const uint32_t bg = __ballot_sync(0xffffffffu, gt), be = __ballot_sync(0xffffffffu, eq);
        if (lane == 0) { w_gt[warp] = __popc(bg); w_eq[warp] = __popc(be); }
        __syncthreads();
        uint32_t pre_g = run_gt, pre_e = run_eq;
        for (int w = 0; w < warp; ++w) { pre_g += w_gt[w]; pre_e += w_eq[w]; }
        const uint32_t lt = (1u << lane) - 1u;
        if (gt) {
            const uint32_t pos = pre_g + __popc(bg & lt);
            out_key[pos] = ~key;  // ascending sort of ~key == descending gain
            out_idx[pos] = (uint32_t)i;
        } else if (eq) {
            const uint32_t r = pre_e + __popc(be & lt);
            if (r < take_eq) {
                out_key[total_gt + r] = ~key;
                out_idx[total_gt + r] = (uint32_t)i;
            }
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            uint32_t sg = 0, se = 0;
            for (int w = 0; w < 8; ++w) { sg += w_gt[w]; se += w_eq[w]; }
            run_gt += sg; run_eq += se;
        }
        __syncthreads();
    }
}

__global__ void widen_idx_kernel(const uint32_t* __restrict__ in, int64_t n, int64_t* __restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = (int64_t)in[i];
}

// ---------------------------------------------------------------- fused selection (one cooperative launch)
// The adaptive loop is a chain of small dependent steps, so the 38 launches of the multi-kernel selection above cost
// more than the work. This kernel does the whole top-k in one launch of at most one CTA per SM (cooperative launch:
// all CTAs are co-resident, so a global barrier is legal): a radix select over the 96-bit composite key
// (ordered gain, ~index) -- unique per cell, hence no tie handling -- in nine 11/10-bit digits with a grid barrier
// after each histogram, an unordered append of the k winners, and a bitonic sort of the winners by CTA 0.
constexpr int kFusedThreads = 256;
constexpr int kFusedBins = 2048;
constexpr int kFusedPasses = 9;
constexpr int kFusedMaxSortK = 8192;                 // winners sorted in shared memory (12 bytes each)
__constant__ int kFusedShift[kFusedPasses] = {85, 74, 63, 52, 42, 32, 21, 10, 0};
__constant__ int kFusedBits[kFusedPasses] = {11, 11, 11, 11, 10, 10, 11, 11, 10};

struct FusedSelectState {
    uint32_t hist[kFusedPasses][kFusedBins];
    uint32_t barrier;
    uint32_t n_out;
};

struct Key96 {
    uint64_t hi;   // ordered gain
    uint32_t lo;   // ~index: smaller index = larger key
};

__device__ __forceinline__ uint32_t key96_digit(const Key96& k, int shift, int bits) {
    // bits [shift, shift + bits) of the 96-bit number (hi << 32) | lo
    const uint32_t mask = (1u << bits) - 1u;
    if (shift >= 32) return (uint32_t)(k.hi >> (shift - 32)) & mask;
    // digits never straddle the hi/lo boundary with the chosen widths (shift + bits <= 32 here)
    return (k.lo >> shift) & mask;
}
// do the bits above `shift` of a and b agree?
__device__ __forceinline__ bool key96_prefix_equal(const Key96& a, const Key96& b, int shift) {
    if (shift >= 96) return true;
    if (shift >= 32) {
        const int s = shift - 32;
        return s >= 64 ? true : ((a.hi >> s) == (b.hi >> s));
    }
    return a.hi == b.hi && (shift >= 32 ? true : ((a.lo >> shift) == (b.lo >> shift)));
}
// is the part of a above bit `shift` >= the same part of b?
__device__ __forceinline__ bool key96_top_ge(const Key96& a, const Key96& b, int shift) {
    if (shift >= 32) {
        const int s = shift - 32;
        return (a.hi >> s) >= (b.hi >> s);
    }
    return a.hi > b.hi || (a.hi == b.hi && (a.lo >> shift) >= (b.lo >> shift));
}
__device__ __forceinline__ bool key96_ge(const Key96& a, const Key96& b) {
    return a.hi > b.hi || (a.hi == b.hi && a.lo >= b.lo);
}
__device__ __forceinline__ bool key96_gt(const Key96& a, const Key96& b) {
    return a.hi > b.hi || (a.hi == b.hi && a.lo > b.lo);
}

__device__ __forceinline__ void fused_grid_barrier(uint32_t* counter, uint32_t& generation) {
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        const uint32_t target = (generation + 1u) * gridDim.x;
        atomicAdd(counter, 1u);
        while (*((volatile uint32_t*)counter) < target) { }
        __threadfence();
    }
    ++generation;
    __syncthreads();
}

__global__ void __launch_bounds__(kFusedThreads, 1)
select_fused_kernel(const double* __restrict__ gain, const uint8_t* __restrict__ flags, int64_t n, uint32_t k,
                    FusedSelectState* st, uint64_t* __restrict__ win_key, uint32_t* __restrict__ win_idx,
                    int64_t* __restrict__ out, int sort_in_kernel, uint32_t max_candidates) {
    extern __shared__ __align__(16) unsigned char fused_smem[];
    uint32_t* s_hist = reinterpret_cast<uint32_t*>(fused_smem);            // [kFusedBins], re-used by the sort
    __shared__ uint32_t s_digit, s_rem, s_cnt;
    int final_shift = 0;
    uint32_t n_cand = k;
    uint32_t generation = 0;
    Key96 prefix{0ull, 0u};
    uint32_t remaining = k;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    const int64_t t0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;

    for (int pass = 0; pass < kFusedPasses; ++pass) {
        const int shift = kFusedShift[pass], bits = kFusedBits[pass];
        for (int b = threadIdx.x; b < kFusedBins; b += blockDim.x) s_hist[b] = 0;
        __syncthreads();
        for (int64_t i = t0; i < n; i += stride) {
            if (flags[i] & kFlagLeaf) {
                const Key96 key{f64_to_ordered(gain[i]), ~(uint32_t)i};
                if (key96_prefix_equal(key, prefix, shift + bits)) atomicAdd(&s_hist[key96_digit(key, shift, bits)], 1u);
            }
        }
        __syncthreads();
        for (int b = threadIdx.x; b < (1 << bits); b += blockDim.x)
            if (s_hist[b]) atomicAdd(&st->hist[pass][b], s_hist[b]);
        fused_grid_barrier(&st->barrier, generation);
        // every CTA finds the digit of the remaining-th largest key from the same global histogram
        if (threadIdx.x < 32) {
            // warp scan from the top bin down
            const int nb = 1 << bits;
            const int per = nb / 32;
            const volatile uint32_t* h = st->hist[pass];
            uint32_t mine = 0;
            const int hi_bin = nb - 1 - (int)threadIdx.x * per;       // lane 0 owns the top `per` bins
            for (int j = 0; j < per; ++j) mine += h[hi_bin - j];
            uint32_t incl = mine;
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t v = __shfl_up_sync(0xffffffffu, incl, o);
                if ((int)threadIdx.x >= o) incl += v;
            }
            const uint32_t excl = incl - mine;                          // keys in the lanes above mine
            if (remaining > excl && remaining <= incl) {
                uint32_t rem = remaining - excl;
                int digit = hi_bin;
                for (int j = 0; j < per; ++j) {
                    const uint32_t c = h[hi_bin - j];
                    if (rem <= c) { digit = hi_bin - j; break; }
                    rem -= c;
                }
                s_digit = (uint32_t)digit;
                s_rem = rem;
                s_cnt = h[digit];
            }
        }
        __syncthreads();
        const uint32_t digit = s_digit;
        remaining = s_rem;
        const uint32_t bucket = s_cnt;
        if (shift >= 32) prefix.hi |= (uint64_t)digit << (shift - 32);
        else prefix.lo |= digit << shift;
        __syncthreads();
        // Early finish: k - remaining keys lie above the chosen bucket and `bucket` keys in it. Once that many fit the
        // shared-memory sort, the remaining digits need no histogram passes (and no grid barriers): collect them all
        // and let the sort find the k largest. With continuous gains this happens after the second pass.
        final_shift = shift;
        n_cand = (k - remaining) + bucket;
        if (sort_in_kernel && n_cand <= max_candidates) break;
    }
    // every key whose digits down to `final_shift` are >= those of the prefix is a candidate (n_cand of them; exactly the
    // k winners when all passes ran)
    for (int64_t i = t0; i < n; i += stride) {
        if (flags[i] & kFlagLeaf) {
            const Key96 key{f64_to_ordered(gain[i]), ~(uint32_t)i};
            if (key96_top_ge(key, prefix, final_shift)) {
                const uint32_t pos = atomicAdd(&st->n_out, 1u);
                if (pos < n_cand) { win_key[pos] = key.hi; win_idx[pos] = (uint32_t)i; }
            }
        }
    }
    if (!sort_in_kernel) return;
    fused_grid_barrier(&st->barrier, generation);
    if (blockIdx.x != 0) return;
    // bitonic sort of the candidates, descending composite key = (gain descending, index ascending); the first k win
    uint32_t p2 = 1;
    while (p2 < n_cand) p2 <<= 1;
    uint64_t* s_hi = reinterpret_cast<uint64_t*>(fused_smem);
    uint32_t* s_lo = reinterpret_cast<uint32_t*>(s_hi + p2);
    for (uint32_t i = threadIdx.x; i < p2; i += blockDim.x) {
        // __ldcg: written by other CTAs in this launch
        s_hi[i] = i < n_cand ? __ldcg(win_key + i) : 0ull;
        s_lo[i] = i < n_cand ? ~__ldcg(win_idx + i) : 0u;
    }
    __syncthreads();
    for (uint32_t size = 2; size <= p2; size <<= 1) {
        for (uint32_t strd = size >> 1; strd > 0; strd >>= 1) {
            for (uint32_t i = threadIdx.x; i < p2 / 2; i += blockDim.x) {
                const uint32_t lo = 2 * i - (i & (strd - 1));
                const uint32_t hi = lo + strd;
                const bool desc = ((lo & size) == 0);
                const Key96 a{s_hi[lo], s_lo[lo]}, b{s_hi[hi], s_lo[hi]};
                if (key96_gt(b, a) == desc) {
                    s_hi[lo] = b.hi; s_lo[lo] = b.lo;
                    s_hi[hi] = a.hi; s_lo[hi] = a.lo;
                }
            }
            __syncthreads();
        }
    }
    for (uint32_t i = threadIdx.x; i < k; i += blockDim.x) out[i] = (int64_t)(~s_lo[i]);
}

// ---------------------------------------------------------------- captured metric (s_cube.py:317-336)
// sum of metric^2 over the leaves; fixed reduction tree -> deterministic
__global__ void __launch_bounds__(256)
leaf_sumsq_partial_kernel(const double* __restrict__ metric, const uint8_t* __restrict__ flags, int64_t n,
                          double* __restrict__ partial) {
    __shared__ double sw[8];
    double acc = 0.0;
    const int64_t base = (int64_t)blockIdx.x * 4096;
    for (int j = threadIdx.x; j < 4096; j += 256) {
        const int64_t i = base + j;
        if (i < n && (flags[i] & kFlagLeaf)) acc = __fma_rn(metric[i], metric[i], acc);
    }
    for (int o = 16; o > 0; o >>= 1) acc = __dadd_rn(acc, shfl_xor_d(acc, o));
    if ((threadIdx.x & 31) == 0) sw[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        double s = 0.0;
        for (int w = 0; w < 8; ++w) s = __dadd_rn(s, sw[w]);
        partial[blockIdx.x] = s;
    }
}

__global__ void __launch_bounds__(256)
sum_partials_kernel(const double* __restrict__ partial, int64_t n, double* __restrict__ out) {
    __shared__ double sw[8];
    double acc = 0.0;
    for (int64_t i = threadIdx.x; i < n; i += 256) acc = __dadd_rn(acc, partial[i]);
    for (int o = 16; o > 0; o >>= 1) acc = __dadd_rn(acc, shfl_xor_d(acc, o));
    if ((threadIdx.x & 31) == 0) sw[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        double s = 0.0;
        for (int w = 0; w < 8; ++w) s = __dadd_rn(s, sw[w]);
        out[0] = s;
    }
}

__global__ void __launch_bounds__(256)
sumsq_partial_kernel(const double* __restrict__ x, int64_t n, double* __restrict__ partial) {
    __shared__ double sw[8];
    double acc = 0.0;
    const int64_t base = (int64_t)blockIdx.x * 4096;
    for (int j = threadIdx.x; j < 4096; j += 256) {
        const int64_t i = base + j;
        if (i < n) acc = __fma_rn(x[i], x[i], acc);
    }
    for (int o = 16; o > 0; o >>= 1) acc = __dadd_rn(acc, shfl_xor_d(acc, o));
    if ((threadIdx.x & 31) == 0) sw[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        double s = 0.0;
        for (int w = 0; w < 8; ++w) s = __dadd_rn(s, sw[w]);
        partial[blockIdx.x] = s;
    }
}

}  // namespace s3

using namespace s3;

extern "C" {

int s3_cells_refine(double* d_center, int32_t* d_level, uint8_t* d_flags, const int64_t* d_parents, int64_t n_parents,
                    int64_t first_child, int dim, double width, void* stream) {
    S3_REQUIRE(d_center && d_level && d_flags && d_parents, "s3_cells_refine: NULL argument");
    S3_REQUIRE(dim == 2 || dim == 3, "s3_cells_refine: dim must be 2 or 3");
    if (n_parents == 0) return S3_OK;
    const int64_t threads = n_parents << dim;
    cells_refine_kernel<<<(unsigned)ceil_div(threads, 256), 256, 0, (cudaStream_t)stream>>>(
        d_center, d_level, d_flags, d_parents, n_parents, first_child, dim, width);
    S3_LAUNCH_CHECK();
    note_launch(1);
    return S3_OK;
}

int s3_cells_gain(const s3_knn_t* knn, const double* d_center, const int32_t* d_level, const int64_t* d_cells,
                  int64_t first, int64_t n, int k, double width, double gain0, int sdm_order, double* d_metric,
                  double* d_gain, void* stream) {
    S3_REQUIRE(knn && d_center && d_level && d_metric && d_gain, "s3_cells_gain: NULL argument");
    const KnnIndex* ix = knn_index_of(knn);
    S3_REQUIRE(ix->values != nullptr, "s3_cells_gain: KNN index has no values (metric)");
    S3_REQUIRE(k >= 1 && k <= kKnnMaxK && k <= ix->n, "s3_cells_gain: k=%d out of range", k);
    if (n == 0) return S3_OK;
    S3_REQUIRE(n < ((int64_t)1 << 31), "s3_cells_gain: too many cells in one call");
    KnnView v = make_view(*ix);
    if (ix->dim == 2)
        cells_gain_kernel<2><<<(unsigned)n, 32 * 5, 0, (cudaStream_t)stream>>>(v, d_center, d_level, d_cells, first, n, k,
                                                                             width, gain0, sdm_order, d_metric, d_gain);
    else
        cells_gain_kernel<3><<<(unsigned)n, 32 * 9, 0, (cudaStream_t)stream>>>(v, d_center, d_level, d_cells, first, n, k,
                                                                             width, gain0, sdm_order, d_metric, d_gain);
    S3_LAUNCH_CHECK();
    note_launch(1);
    return S3_OK;
}

// Pre-pass of the mask entry points: the geometries named by the bit mask `stl_geoms` are closed triangulated surfaces
// (GEOM_STL); their per-node inside flags are computed by the tiled kernel of stl.cuh into stream-ordered scratch.
// n_tri of each geometry is read from the (host-visible copy of the) header the caller passes in `stl_ntri`.
static int stl_prepass(Scratch& scratch, const StlPoints& src, int64_t n_pts, const int32_t* d_geom_hdr,
                       const double* d_geom_par, int n_geoms, int only_geom, int stl_geoms, const int32_t* stl_meta,
                       StlPre* pre, cudaStream_t st) {
    pre->n = 0;
    for (int g = 0; g < n_geoms && g < 31; ++g) {
        if (!((stl_geoms >> g) & 1) || (only_geom >= 0 && g != only_geom)) continue;
        if (pre->n == kMaxStlPre) break;                                 // further STL surfaces take the per-thread path
        uint8_t* flags = nullptr;
        S3_TRY(scratch.alloc(&flags, (size_t)n_pts));
        // stl_meta (host): {parameter offset, n_tri} per geometry, the same numbers as in the device header
        const int offset = stl_meta[2 * g], n_tri = stl_meta[2 * g + 1];
        stl_inside_kernel<<<(unsigned)ceil_div(n_pts, kStlThreads), kStlThreads, 0, st>>>(src, n_pts, d_geom_par + offset,
                                                                                        n_tri, flags);
        S3_LAUNCH_CHECK();
        note_launch(1);
        pre->inside[pre->n] = flags;
        pre->geom[pre->n] = g;
        ++pre->n;
    }
    return S3_OK;
}

int s3_cells_mask(const double* d_center, const int32_t* d_level, const int64_t* d_cells, int64_t first, int64_t n,
                  int dim, double width, const int32_t* d_geom_hdr, const double* d_geom_par, int n_geoms,
                  int only_geom, int refine_mode, int apply, uint8_t* d_invalid, uint8_t* d_flags, double* d_gain,
                  int stl_geoms, const int32_t* stl_meta, void* stream) {
    S3_REQUIRE(d_center && d_level && d_invalid, "s3_cells_mask: NULL argument");
    S3_REQUIRE(n_geoms == 0 || (d_geom_hdr && d_geom_par), "s3_cells_mask: geometry tables missing");
    S3_REQUIRE(!apply || (d_flags && d_gain), "s3_cells_mask: apply needs flags and gain");
    S3_REQUIRE(stl_geoms == 0 || stl_meta, "s3_cells_mask: stl_geoms needs stl_meta");
    if (n == 0) return S3_OK;
    cudaStream_t st = (cudaStream_t)stream;
    Scratch scratch(st);
    StlPre pre{};
    if (stl_geoms && dim == 3) {
        StlPoints src{};
        src.mode = 0; src.center = d_center; src.level = d_level; src.cells = d_cells; src.first = first; src.width = width;
        S3_TRY(stl_prepass(scratch, src, n * 8, d_geom_hdr, d_geom_par, n_geoms, only_geom, stl_geoms, stl_meta, &pre, st));
    }
    cells_mask_kernel<<<(unsigned)ceil_div(n, 128), 128, 0, st>>>(
        d_center, d_level, d_cells, first, n, dim, width, d_geom_hdr, d_geom_par, n_geoms, only_geom, refine_mode,
        apply, d_invalid, d_flags, d_gain, pre);
    S3_LAUNCH_CHECK();
    note_launch(1);
    return S3_OK;
}

int s3_nodes_mask(const double* d_nodes, int64_t n, int n_nodes, int dim, const int32_t* d_geom_hdr,
                  const double* d_geom_par, int n_geoms, int only_geom, int refine_mode, uint8_t* d_invalid,
                  int stl_geoms, const int32_t* stl_meta, void* stream) {
    S3_REQUIRE(d_nodes && d_invalid && d_geom_hdr && d_geom_par, "s3_nodes_mask: NULL argument");
    S3_REQUIRE(dim == 2 || dim == 3, "s3_nodes_mask: dim must be 2 or 3");
    S3_REQUIRE(n_nodes >= 1 && n_nodes <= 64, "s3_nodes_mask: n_nodes out of range");
    S3_REQUIRE(stl_geoms == 0 || stl_meta, "s3_nodes_mask: stl_geoms needs stl_meta");
    if (n == 0) return S3_OK;
    cudaStream_t st = (cudaStream_t)stream;
    Scratch scratch(st);
    StlPre pre{};
    if (stl_geoms && dim == 3) {
        StlPoints src{};
        src.mode = 1; src.points = d_nodes;
        S3_TRY(stl_prepass(scratch, src, n * n_nodes, d_geom_hdr, d_geom_par, n_geoms, only_geom, stl_geoms, stl_meta, &pre, st));
    }
    nodes_mask_kernel<<<(unsigned)ceil_div(n, 128), 128, 0, st>>>(
        d_nodes, n, n_nodes, dim, d_geom_hdr, d_geom_par, n_geoms, only_geom, refine_mode, d_invalid, pre);
    S3_LAUNCH_CHECK();
    note_launch(1);
    return S3_OK;
}

int s3_points_inside(const double* d_points, int64_t n, int dim, const int32_t* d_geom_hdr, const double* d_geom_par,
                     int geom, uint8_t* d_inside, int stl_geoms, const int32_t* stl_meta, void* stream) {
    S3_REQUIRE(d_points && d_inside && d_geom_hdr && d_geom_par, "s3_points_inside: NULL argument");
    S3_REQUIRE(dim == 2 || dim == 3, "s3_points_inside: dim must be 2 or 3");
    S3_REQUIRE(stl_geoms == 0 || stl_meta, "s3_points_inside: stl_geoms needs stl_meta");
    if (n == 0) return S3_OK;
    cudaStream_t st = (cudaStream_t)stream;
    if (dim == 3 && geom >= 0 && geom < 31 && ((stl_geoms >> geom) & 1)) {
        StlPoints src{};
        src.mode = 1; src.points = d_points;
        stl_inside_kernel<<<(unsigned)ceil_div(n, kStlThreads), kStlThreads, 0, st>>>(
            src, n, d_geom_par + stl_meta[2 * geom], stl_meta[2 * geom + 1], d_inside);
        S3_LAUNCH_CHECK();
        note_launch(1);
        return S3_OK;
    }
    points_inside_kernel<<<(unsigned)ceil_div(n, 128), 128, 0, st>>>(d_points, n, dim, d_geom_hdr, d_geom_par, geom,
                                                                    d_inside);
    S3_LAUNCH_CHECK();
    note_launch(1);
    return S3_OK;
}

static int g_select_fused = 1;     // 1 = one cooperative launch (default), 0 = multi-kernel radix select
extern "C" int s3_select_set_fused(int on) { g_select_fused = on != 0; return S3_OK; }

static int select_topk_multi(const double* d_gain, const uint8_t* d_flags, int64_t n_cells, int64_t k, int64_t* d_out,
                             cudaStream_t st_) {
    Scratch scratch(st_);
    const int nblocks = (int)ceil_div(n_cells, kSelTile);
    SelectState* st = nullptr;
    uint32_t *cnt_gt = nullptr, *cnt_eq = nullptr, *totals = nullptr, *ia = nullptr, *ib = nullptr;
    uint64_t *ka = nullptr, *kb = nullptr;
    S3_TRY(scratch.alloc(&st, 1));
    S3_TRY(scratch.alloc(&cnt_gt, nblocks));
    S3_TRY(scratch.alloc(&cnt_eq, nblocks));
    S3_TRY(scratch.alloc(&totals, 2));
    S3_TRY(scratch.alloc(&ka, k));
    S3_TRY(scratch.alloc(&kb, k));
    S3_TRY(scratch.alloc(&ia, k));
    S3_TRY(scratch.alloc(&ib, k));
    select_init_kernel<<<1, 256, 0, st_>>>(st, (uint64_t)k);
    for (int pass = 7; pass >= 0; --pass) select_pass_kernel<<<nblocks, 256, 0, st_>>>(d_gain, d_flags, n_cells, pass, st);
    select_count_kernel<<<nblocks, 256, 0, st_>>>(d_gain, d_flags, n_cells, st, cnt_gt, cnt_eq);
    select_scan_kernel<<<1, 1024, 0, st_>>>(cnt_gt, cnt_eq, nblocks, totals);
    select_scatter_kernel<<<nblocks, 256, 0, st_>>>(d_gain, d_flags, n_cells, st, cnt_gt, cnt_eq, totals, ka, ia);
    S3_LAUNCH_CHECK();
    note_launch(12);
    bool in_a = true;
    S3_TRY(radix_sort_pairs(ka, ia, kb, ib, k, 0, 64, st_, &in_a));
    note_launch(24);
    widen_idx_kernel<<<(unsigned)ceil_div(k, 256), 256, 0, st_>>>(in_a ? ia : ib, k, d_out);
    S3_LAUNCH_CHECK();
    note_launch(1);
    return S3_OK;
}

int s3_select_topk(const double* d_gain, const uint8_t* d_flags, int64_t n_cells, int64_t k, int64_t* d_out,
                   void* stream) {
    S3_REQUIRE(d_gain && d_flags && d_out, "s3_select_topk: NULL argument");
    S3_REQUIRE(k >= 0 && k <= n_cells, "s3_select_topk: k out of range");
    S3_REQUIRE(n_cells < ((int64_t)1 << 31), "s3_select_topk: too many cells");
    if (k == 0) return S3_OK;
    cudaStream_t st_ = (cudaStream_t)stream;
    if (!g_select_fused || k > kFusedMaxSortK) return select_topk_multi(d_gain, d_flags, n_cells, k, d_out, st_);

    Scratch scratch(st_);
    FusedSelectState* st = nullptr;
    uint64_t* win_key = nullptr;
    uint32_t* win_idx = nullptr;
    // candidates the in-kernel sort accepts before all digits are resolved (early finish of the radix select)
    uint32_t max_cand = (uint32_t)(2 * k > 1024 ? 2 * k : 1024);
    if (max_cand > (uint32_t)kFusedMaxSortK) max_cand = kFusedMaxSortK;
    S3_TRY(scratch.alloc(&st, 1));
    S3_TRY(scratch.alloc(&win_key, max_cand));
    S3_TRY(scratch.alloc(&win_idx, max_cand));
    S3_CUDA(cudaMemsetAsync(st, 0, sizeof(FusedSelectState), st_));
    uint32_t p2 = 1;
    while (p2 < max_cand) p2 <<= 1;
    size_t smem = (size_t)p2 * 12;
    if (smem < kFusedBins * sizeof(uint32_t)) smem = kFusedBins * sizeof(uint32_t);
    // function attributes are per device: set it on every call (cheap) instead of once per process
    S3_CUDA(cudaFuncSetAttribute(select_fused_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kFusedMaxSortK * 12));
    // enough CTAs to stream the cell arrays, never more than one per SM of THIS device (co-residency of the grid barrier)
    int dev = 0, sms = kNumSMs;
    S3_CUDA(cudaGetDevice(&dev));
    S3_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    int grid = (int)ceil_div(n_cells, (int64_t)kFusedThreads * 8);
    if (grid > sms) grid = sms;
    if (grid < 1) grid = 1;
    uint32_t k32 = (uint32_t)k;
    int sort_in_kernel = 1;
    void* args[] = {(void*)&d_gain, (void*)&d_flags, (void*)&n_cells, (void*)&k32, (void*)&st, (void*)&win_key,
                    (void*)&win_idx, (void*)&d_out, (void*)&sort_in_kernel, (void*)&max_cand};
    if (cudaLaunchCooperativeKernel((const void*)select_fused_kernel, dim3((unsigned)grid), dim3(kFusedThreads), args,
                                    smem, st_) != cudaSuccess) {
        (void)cudaGetLastError();                       // e.g. a MIG slice that cannot co-schedule the grid: multi-kernel path
        return select_topk_multi(d_gain, d_flags, n_cells, k, d_out, st_);
    }
    note_launch(1);
    return S3_OK;
}

int s3_leaf_sumsq(const double* d_metric, const uint8_t* d_flags, int64_t n_cells, double* d_out, void* stream) {
    S3_REQUIRE(d_metric && d_flags && d_out, "s3_leaf_sumsq: NULL argument");
    cudaStream_t st_ = (cudaStream_t)stream;
    Scratch scratch(st_);
    const int64_t nb = ceil_div(n_cells > 0 ? n_cells : 1, 4096);
    double* partial = nullptr;
    S3_TRY(scratch.alloc(&partial, nb));
    leaf_sumsq_partial_kernel<<<(unsigned)nb, 256, 0, st_>>>(d_metric, d_flags, n_cells, partial);
    sum_partials_kernel<<<1, 256, 0, st_>>>(partial, nb, d_out);
    S3_LAUNCH_CHECK();
    note_launch(2);
    return S3_OK;
}

int s3_sumsq(const double* d_x, int64_t n, double* d_out, void* stream) {
    S3_REQUIRE(d_x && d_out, "s3_sumsq: NULL argument");
    cudaStream_t st_ = (cudaStream_t)stream;
    Scratch scratch(st_);
    const int64_t nb = ceil_div(n > 0 ? n : 1, 4096);
    double* partial = nullptr;
    S3_TRY(scratch.alloc(&partial, nb));
    sumsq_partial_kernel<<<(unsigned)nb, 256, 0, st_>>>(d_x, n, partial);
    sum_partials_kernel<<<1, 256, 0, st_>>>(partial, nb, d_out);
    S3_LAUNCH_CHECK();
    note_launch(2);
    return S3_OK;
}

}  // extern "C"
