// The inline-PTX layer of the tensor-core kernels (sm_100a): mbarriers, TMA tensor loads and the host-side encoding of
// their tensor maps, cluster helpers, tcgen05 (UMMA descriptors, MMA, commit, fences, TMEM allocation and loads) and the
// TF32 hi / lo split of the 3xTF32 products.
#pragma once
#include <cuda.h>
#include <initializer_list>
#include "common.cuh"

namespace s3 {

// ---------------------------------------------------------------- mbarriers
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive_cta(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
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
__device__ __forceinline__ void named_bar(int id, int n) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(n) : "memory"); }

// ---------------------------------------------------------------- TMA tensor loads
__device__ __forceinline__ void tma_prefetch(const CUtensorMap* map) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, int c0, int c1, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::
            "r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* map, int c0, int c1, int c2, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::
            "r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
        : "memory");
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

// Tensor map of a dense fp32 array at `base` (host side): `dims` innermost first, rows packed (the stride of each
// dimension is the product of the ones inside it), `box` in elements. `name` goes into the error message.
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static int tma_map_f32(CUtensorMap* map, const char* name, void* base, std::initializer_list<int64_t> dims,
                       std::initializer_list<int> box, CUtensorMapSwizzle swizzle) {
    static PFN_encodeTiled encode = nullptr;
    if (!encode) {
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult qres;
        S3_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
        S3_REQUIRE(fn != nullptr && qres == cudaDriverEntryPointSuccess, "tensor map encoder not available");
        encode = (PFN_encodeTiled)fn;
    }
    const int rank = (int)dims.size();
    S3_REQUIRE(rank >= 1 && rank <= 3 && (int)box.size() == rank, "tensor map %s: bad rank", name);
    cuuint64_t gdim[3], gstride[3];
    cuuint32_t gbox[3], estride[3] = {1, 1, 1};
    cuuint64_t bytes = 4;
    for (int i = 0; i < rank; ++i) {
        gdim[i] = (cuuint64_t)dims.begin()[i];
        gbox[i] = (cuuint32_t)box.begin()[i];
        bytes *= gdim[i];
        gstride[i] = bytes;                                  // gstride[i] is the stride of dimension i + 1
    }
    memset(map, 0, sizeof(*map));
    const CUresult cr = encode(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, (cuuint32_t)rank, base, gdim, gstride, gbox, estride,
                               CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                               CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    S3_REQUIRE(cr == CUDA_SUCCESS, "tensor map %s: encoding failed with code %d", name, (int)cr);
    return S3_OK;
}

// ---------------------------------------------------------------- clusters
__device__ __forceinline__ uint32_t cluster_rank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\nbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// ---------------------------------------------------------------- tcgen05: TF32 operands, MMA, TMEM
// hi = tf32_rna(x), lo = x - hi (exact in fp32; the tensor core drops lo's low bits): the operands of 3xTF32
__device__ __forceinline__ void tf32_split(float x, float& hi, float& lo) {
    uint32_t hbits;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(hbits) : "f"(x));
    hi = __uint_as_float(hbits);
    lo = x - hi;
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
// One stage of K-major operands, 32 floats of K (4 UMMA K-steps of 8) at shared addresses a_hi / a_lo / b_hi / b_lo:
// D (+)= A_lo B_hi + A_hi B_lo + A_hi B_hi (passes == 3, 3xTF32) or A_hi B_hi. The first MMA overwrites D unless
// `accumulate`.
__device__ __forceinline__ void umma_stage_k(uint32_t d_tmem, uint32_t a_hi, uint32_t a_lo, uint32_t b_hi, uint32_t b_lo,
                                             uint32_t idesc, int passes, uint32_t accumulate) {
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) {
        const uint32_t koff = (uint32_t)ks * 32u;
        const uint64_t ah = umma_desc_k_sw128(a_hi + koff);
        const uint64_t bh = umma_desc_k_sw128(b_hi + koff);
        if (passes == 3) {
            const uint64_t al = umma_desc_k_sw128(a_lo + koff);
            const uint64_t bl = umma_desc_k_sw128(b_lo + koff);
            umma_tf32(d_tmem, al, bh, idesc, accumulate);
            umma_tf32(d_tmem, ah, bl, idesc, 1u);
            umma_tf32(d_tmem, ah, bh, idesc, 1u);
        } else {
            umma_tf32(d_tmem, ah, bh, idesc, accumulate);
        }
        accumulate = 1u;
    }
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

// Warp-collective: allocate `cols` TMEM columns, write their base address to the shared `slot` and give up the right to
// allocate more (so that another CTA on the SM can take the rest).
__device__ __forceinline__ void tmem_alloc(uint32_t* slot, uint32_t cols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot)), "r"(cols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
// warp-collective, by the warp that allocated
__device__ __forceinline__ void tmem_dealloc(uint32_t base, uint32_t cols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(base), "r"(cols) : "memory");
}
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

}  // namespace s3
