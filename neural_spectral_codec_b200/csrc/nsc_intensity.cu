// RangeImageProjector.project(points, keep_intensity=True) (reference
// src/encoding/range_image.py:129-232): the range image plus, per pixel, the intensity of the
// closest point -- the largest intensity when several points tie on the range (:217-226), never
// below the 0 the image is initialised with. This branch is NOT on the encoding path
// (spectral_encoder.py:217 passes keep_intensity=False); it completes the projector's surface.
//
// One packed 64-bit atomicMin per point on (range bits, ~intensity bits): the minimum key holds
// the minimum range and, among equal ranges, the maximum intensity -- deterministic whatever the
// point order. The range must be the ROUNDED sqrt here (the reference ties on range, and two
// different sums of squares can round to the same range), so this kernel pays one sqrt per point.
#include "nsc_point.h"

namespace nsc {

namespace {

constexpr int kIThreads = 512;

__global__ void __launch_bounds__(kIThreads)
project_intensity_kernel(const float* __restrict__ points, const long long* __restrict__ offsets,
                         long long origin, int n_scans, const __grid_constant__ DeviceParams dp,
                         float* __restrict__ range_out, float* __restrict__ intensity_out) {
    extern __shared__ unsigned long long img64[];
    const int n_pix = dp.E * kPitch;
    for (int scan = blockIdx.x; scan < n_scans; scan += gridDim.x) {
        __syncthreads();
        for (int i = threadIdx.x; i < n_pix; i += kIThreads) img64[i] = ~0ull;
        __syncthreads();
        const float4* p4 = reinterpret_cast<const float4*>(points) + (offsets[scan] - origin);
        const int n = (int)(offsets[scan + 1] - offsets[scan]);
        for (int i = threadIdx.x; i < n; i += kIThreads) {
            const float4 v = __ldcs(p4 + i);
            uint32_t row_b, col_b;
            const uint32_t key = classify(v.x, v.y, v.z, dp, dp.row_mode, row_b, col_b);
            if (key == 0xffffffffu || key_is_empty(key, dp)) continue;
            const uint32_t rbits = __float_as_uint(__fsqrt_rn(__uint_as_float(key)));
            // max(0, intensity); a NaN intensity propagates like np.maximum (NaN sorts above +Inf)
            const uint32_t ibits = v.w > 0.0f ? __float_as_uint(v.w) : (v.w != v.w ? 0x7fc00000u : 0u);
            const uint32_t pix = (row_b - kFloorBias) * kPitch + (col_b - kFloorBias);
            atomicMin(&img64[pix], ((unsigned long long)rbits << 32) | (0xffffffffu - ibits));
        }
        __syncthreads();
        for (int i = threadIdx.x; i < dp.E * kAz; i += kIThreads) {
            const int r = i / kAz, c = i - r * kAz;
            unsigned long long k = img64[r * kPitch + c];
            if (c == 0) k = min(k, img64[r * kPitch + kAz]);        // azimuth == 2 pi wraps to column 0
            const bool empty = k == ~0ull;
            const long long o = (long long)scan * dp.E * kAz + i;
            range_out[o] = empty ? 0.0f : __uint_as_float((uint32_t)(k >> 32));
            intensity_out[o] = empty ? 0.0f : __uint_as_float(0xffffffffu - (uint32_t)(k & 0xffffffffu));
        }
    }
}

// More than 64 rows: 128 x 361 64-bit keys do not fit one CTA's shared memory, so each scan takes
// two passes over its points, each owning half of the rows (the first (E + 1) / 2, then the rest).
__global__ void __launch_bounds__(kIThreads)
project_intensity_tall_kernel(const float* __restrict__ points, const long long* __restrict__ offsets,
                              long long origin, int n_scans, const __grid_constant__ DeviceParams dp,
                              float* __restrict__ range_out, float* __restrict__ intensity_out) {
    extern __shared__ unsigned long long img64[];
    const int half = (dp.E + 1) / 2;
    for (int scan = blockIdx.x; scan < n_scans; scan += gridDim.x) {
        const float4* p4 = reinterpret_cast<const float4*>(points) + (offsets[scan] - origin);
        const int n = (int)(offsets[scan + 1] - offsets[scan]);
        for (int row0 = 0; row0 < dp.E; row0 += half) {
            const int rows = min(half, dp.E - row0);
            __syncthreads();
            for (int i = threadIdx.x; i < rows * kPitch; i += kIThreads) img64[i] = ~0ull;
            __syncthreads();
            for (int i = threadIdx.x; i < n; i += kIThreads) {
                const float4 v = __ldcs(p4 + i);
                uint32_t row_b, col_b;
                const uint32_t key = classify<NSC_MAX_ELEVATION>(v.x, v.y, v.z, dp, dp.row_mode, row_b, col_b);
                const int row = (int)(row_b - kFloorBias) - row0;
                if (key == 0xffffffffu || key_is_empty(key, dp) || row < 0 || row >= rows) continue;
                const uint32_t rbits = __float_as_uint(__fsqrt_rn(__uint_as_float(key)));
                const uint32_t ibits = v.w > 0.0f ? __float_as_uint(v.w) : (v.w != v.w ? 0x7fc00000u : 0u);
                const uint32_t pix = row * kPitch + (col_b - kFloorBias);
                atomicMin(&img64[pix], ((unsigned long long)rbits << 32) | (0xffffffffu - ibits));
            }
            __syncthreads();
            for (int i = threadIdx.x; i < rows * kAz; i += kIThreads) {
                const int r = i / kAz, c = i - r * kAz;
                unsigned long long k = img64[r * kPitch + c];
                if (c == 0) k = min(k, img64[r * kPitch + kAz]);
                const bool empty = k == ~0ull;
                const long long o = ((long long)scan * dp.E + row0) * kAz + i;
                range_out[o] = empty ? 0.0f : __uint_as_float((uint32_t)(k >> 32));
                intensity_out[o] = empty ? 0.0f : __uint_as_float(0xffffffffu - (uint32_t)(k & 0xffffffffu));
            }
        }
    }
}

}  // namespace

}  // namespace nsc

using namespace nsc;

extern "C" int nsc_project_intensity_batch(const float* d_points, const int64_t* d_offsets,
                                           int64_t point_origin, int n_scans, const nsc_params* p,
                                           float* d_range_images, float* d_intensity_images,
                                           void* stream) {
    int32_t lut[NSC_N_FREQS] = {0};
    DeviceParams dp;
    int st = make_device_params(p, lut, &dp);
    if (st != NSC_OK) return st;
    if (n_scans < 0) return NSC_ERR_BAD_COUNT;
    if (!d_offsets) return NSC_ERR_NULL_POINTER;
    if (reinterpret_cast<uintptr_t>(d_points) & 15u) return NSC_ERR_ALIGNMENT;
    if (n_scans == 0) return NSC_OK;
    if (!d_range_images || !d_intensity_images) return NSC_ERR_NULL_POINTER;
    int dev = 0, sms = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return record_cuda(e);
    e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (e != cudaSuccess) return record_cuda(e);
    const bool tall = dp.E > kShortRows;
    const auto kernel = tall ? project_intensity_tall_kernel : project_intensity_kernel;
    const int smem = (tall ? (dp.E + 1) / 2 : dp.E) * kPitch * 8;
    e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e != cudaSuccess) return record_cuda(e);
    const int grid = n_scans < sms ? n_scans : sms;
    kernel<<<grid, kIThreads, smem, (cudaStream_t)stream>>>(
        d_points, (const long long*)d_offsets, point_origin, n_scans, dp, d_range_images, d_intensity_images);
    return record_cuda(cudaGetLastError());
}
