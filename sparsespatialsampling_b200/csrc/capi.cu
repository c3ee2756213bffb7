// Library-level entry points: error reporting, version, launch accounting.
#include <atomic>
#include <stdarg.h>
#include "common.cuh"
#include "../../include/s3b200.h"

namespace s3 {

static thread_local char g_error[1024] = "";
static std::atomic<int64_t> g_launches{0};

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_error, sizeof(g_error), fmt, ap);
    va_end(ap);
}

void configure_mempool_once() {
    static std::atomic<uint32_t> done_mask{0};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 32) return;
    const uint32_t bit = 1u << dev;
    if (done_mask.load(std::memory_order_acquire) & bit) return;
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, dev) == cudaSuccess) {
        uint64_t threshold = ~0ull;
        cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &threshold);
    }
    done_mask.fetch_or(bit, std::memory_order_release);
}

void note_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

}  // namespace s3

namespace s3 {

// Copies the window [col0, col0 + width) of the rows `rows[0..n_rows)` of a pitched fp32 matrix into a dense buffer.
// The source may be pinned host memory (UVA: the kernel then reads it over PCIe, 512 contiguous bytes per warp
// request), which moves only the rows the sampled grid references instead of the whole snapshot batch.
__global__ void __launch_bounds__(256)
gather_rows_kernel(const float* __restrict__ src, int64_t src_pitch, const int32_t* __restrict__ rows, int64_t n_rows,
                   int64_t width, float* __restrict__ dst, int64_t dst_pitch, int vec) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int64_t chunks = (width + 127) / 128;                  // 128 floats = 512 bytes per warp step
    const int64_t items = n_rows * chunks;
    for (int64_t it = warp; it < items; it += n_warps) {
        const int64_t r = it / chunks, c = it - r * chunks;
        const int64_t col = c * 128 + lane * 4;
        const float* s = src + (int64_t)rows[r] * src_pitch + col;
        float* d = dst + r * dst_pitch + col;
        if (vec && col + 4 <= width) {
            *reinterpret_cast<float4*>(d) = *reinterpret_cast<const float4*>(s);
        } else {
            for (int e = 0; e < 4; ++e)
                if (col + e < width) d[e] = s[e];
        }
    }
}

}  // namespace s3

extern "C" {

int s3_gather_rows(const float* src, int64_t src_pitch, const int32_t* d_rows, int64_t n_rows, int64_t width,
                   float* d_dst, int64_t dst_pitch, int n_ctas, void* stream) {
    S3_REQUIRE(n_rows >= 0 && width >= 0, "s3_gather_rows: bad sizes");
    if (n_rows == 0 || width == 0) return S3_OK;
    S3_REQUIRE(src && d_rows && d_dst, "s3_gather_rows: NULL argument");
    S3_REQUIRE(src_pitch >= width && dst_pitch >= width, "s3_gather_rows: pitch smaller than the window");
    const int vec = (((uintptr_t)src | (uintptr_t)d_dst) % 16 == 0) && (src_pitch % 4 == 0) && (dst_pitch % 4 == 0);
    int grid = n_ctas > 0 ? n_ctas : 2 * s3::kNumSMs;
    s3::gather_rows_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(src, src_pitch, d_rows, n_rows, width, d_dst,
                                                                  dst_pitch, vec);
    S3_LAUNCH_CHECK();
    s3::note_launch(1);
    return S3_OK;
}

const char* s3_last_error(void) { return s3::g_error; }

int s3_version(void) { return 102; }

int64_t s3_launch_count(void) { return s3::g_launches.load(std::memory_order_relaxed); }

int s3_copy2d_async(void* dst, int64_t dst_pitch, const void* src, int64_t src_pitch, int64_t width, int64_t height,
                    int kind, void* stream) {
    S3_REQUIRE(dst && src, "s3_copy2d_async: NULL argument");
    S3_REQUIRE(width >= 0 && height >= 0 && dst_pitch >= width && src_pitch >= width, "s3_copy2d_async: bad geometry");
    S3_REQUIRE(kind == 0 || kind == 1, "s3_copy2d_async: kind must be 0 (host to device) or 1 (device to host)");
    if (width == 0 || height == 0) return S3_OK;
    const cudaMemcpyKind k = kind == 0 ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToHost;
    if (width == dst_pitch && width == src_pitch) {
        // dense on both sides: one linear copy (a 2-D host-to-device copy whose width equals the pitch measured
        // 31.5 GB/s instead of 55, scripts/pitch_probe.py)
        S3_CUDA(cudaMemcpyAsync(dst, src, (size_t)width * (size_t)height, k, (cudaStream_t)stream));
        return S3_OK;
    }
    S3_CUDA(cudaMemcpy2DAsync(dst, (size_t)dst_pitch, src, (size_t)src_pitch, (size_t)width, (size_t)height,
                              k, (cudaStream_t)stream));
    return S3_OK;
}

}  // extern "C"
