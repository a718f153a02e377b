// uint16 quantisation of descriptor rows (SURVEY.md 8(f) rank 4): HistogramQuantizer.quantize /
// dequantize of reference src/encoding/quantization.py:131-192, batched over rows and generalised
// from 50 bins to any row length (the 800-D descriptor -> 1600-byte records). The pairwise-sum plan,
// the hoisted divisor and the rounding are in nsc_quantize.cuh, shared with the encoder's uint16
// epilogue.
#include "nsc_quantize.cuh"

namespace nsc {

namespace {

constexpr int kQThreads = 256;
constexpr int kQWarps = kQThreads / 32;
#ifndef NSC_Q_BATCH
#define NSC_Q_BATCH 4
#endif
#ifndef NSC_Q_MIN_BLOCKS
#define NSC_Q_MIN_BLOCKS 5
#endif
#ifndef NSC_DQ_MIN_BLOCKS
#define NSC_DQ_MIN_BLOCKS 5
#endif
constexpr int kVecBatch = NSC_Q_BATCH;   // 16-byte loads in flight per lane

__device__ __forceinline__ unsigned bits_or(float4 v) {
    return __float_as_uint(v.x) | __float_as_uint(v.y) | __float_as_uint(v.z) | __float_as_uint(v.w);
}

// One row per warp. VEC (n_bins % 8 == 0, 16-byte aligned bases, so every row of both arrays starts
// on a 16-byte boundary): the row moves with 16-byte accesses; rows whose elements are all
// non-negative and whose denominator is of moderate size (every descriptor row) take the hoisted
// division, are packed to uint16 in place and leave with 16-byte stores.
template <bool VEC>
__global__ void __launch_bounds__(kQThreads, NSC_Q_MIN_BLOCKS)
quantize_kernel(const float* __restrict__ hist, long long n_rows, int n_bins, float eps,
                const __grid_constant__ SumPlan plan, unsigned short* __restrict__ q_out) {
    extern __shared__ __align__(16) float smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float* row_s = smem + warp * (n_bins + kSumSlots);
    float* slot_s = row_s + n_bins;
    const long long n_warps = (long long)gridDim.x * kQWarps;
    for (long long r = (long long)blockIdx.x * kQWarps + warp; r < n_rows; r += n_warps) {
        unsigned sign_or = 0x80000000u;                     // scalar rows: always the general path
        if (VEC) {
            sign_or = 0;
            const float4* src = reinterpret_cast<const float4*>(hist + r * n_bins);
            float4* dst = reinterpret_cast<float4*>(row_s);
            const int n_vec = n_bins >> 2;
            for (int v0 = 0; v0 < n_vec; v0 += 32 * kVecBatch) {
                float4 t[kVecBatch];
#pragma unroll
                for (int k = 0; k < kVecBatch; ++k) {
                    const int v = v0 + k * 32 + lane;
                    if (v < n_vec) t[k] = __ldg(src + v);
                }
#pragma unroll
                for (int k = 0; k < kVecBatch; ++k) {
                    const int v = v0 + k * 32 + lane;
                    if (v < n_vec) {
                        dst[v] = t[k];
                        sign_or |= bits_or(t[k]);
                    }
                }
            }
        } else {
            for (int e = lane; e < n_bins; e += 32) row_s[e] = hist[r * n_bins + e];
        }
        __syncwarp();
        const float sum = numpy_sum(row_s, plan, slot_s, lane);
        const bool norm = sum > eps;                       // quantization.py:144-146
        const float denom = __fadd_rn(sum, eps);
        int qsum = 0;
        unsigned best = 0;                                  // (q << 16) | (0xffff - index): first max
        // eps >= 0 and no negative element: every element <= sum <= denom, so 0 <= quotient <= 1 and
        // the scaled value needs no clamp
        const bool packed = VEC && norm && eps >= 0.0f && moderate(denom) &&
                            (__reduce_or_sync(0xffffffffu, sign_or) >> 31) == 0;
        if (packed) {
            const RowDivisor div(denom);
            const float4* in4 = reinterpret_cast<const float4*>(row_s);
            uint2* out2 = reinterpret_cast<uint2*>(row_s);
            const int n_vec = n_bins >> 2;
            // x + 2^23 rounds 0 <= x <= 65535 to an integer, ties to even like np.round, and leaves it in
            // the low bits: 0x4B000000 + q. Sums and shifts below work on those bits modulo 2^32.
            unsigned bits_sum = 0;
            // the packed values of elements [4v, 4v + 4) land on bytes [8v, 8v + 8) of the row: behind
            // everything still to be read, once the lanes of this pass have read theirs (the barrier)
            for (int v0 = 0; v0 < n_vec; v0 += 32) {
                const int v = v0 + lane;
                float4 h = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
                if (v < n_vec) h = in4[v];
                __syncwarp();
                if (v < n_vec) {
                    const unsigned b0 = __float_as_uint(__fadd_rn(__fmul_rn(div(h.x), 65535.0f), 8388608.0f));
                    const unsigned b1 = __float_as_uint(__fadd_rn(__fmul_rn(div(h.y), 65535.0f), 8388608.0f));
                    const unsigned b2 = __float_as_uint(__fadd_rn(__fmul_rn(div(h.z), 65535.0f), 8388608.0f));
                    const unsigned b3 = __float_as_uint(__fadd_rn(__fmul_rn(div(h.w), 65535.0f), 8388608.0f));
                    const unsigned c = 0xffffu - 4u * (unsigned)v;
                    bits_sum += (b0 + b1) + (b2 + b3);
                    best = max(max(best, (b0 << 16) + c), (b1 << 16) + (c - 1u));
                    best = max(max(best, (b2 << 16) + (c - 2u)), (b3 << 16) + (c - 3u));
                    out2[v] = make_uint2(__byte_perm(b0, b1, 0x5410), __byte_perm(b2, b3, 0x5410));
                }
            }
            qsum = (int)bits_sum;                          // biased by 0x4B000000 per element, removed below
        } else {
            for (int e = lane; e < n_bins; e += 32) {
                const int q = quantise_value(norm ? __fdiv_rn(row_s[e], denom) : row_s[e]);
                row_s[e] = __int_as_float(q);
                qsum += q;
                best = max(best, ((unsigned)q << 16) | (0xffffu - (unsigned)e));
            }
        }
        qsum = (int)__reduce_add_sync(0xffffffffu, (unsigned)qsum);
        if (packed) qsum = (int)((unsigned)qsum - (unsigned)n_bins * 0x4B000000u);
        best = __reduce_max_sync(0xffffffffu, best);
        __syncwarp();
        if (lane == 0 && qsum > 0 && qsum != 65535) {      // :154-167: rounding error into the largest bin
            const int idx = 0xffff - (int)(best & 0xffffu);
            int v = (int)(best >> 16) + (65535 - qsum);
            v = v < 0 ? 0 : (v > 65535 ? 65535 : v);
            if (packed) reinterpret_cast<unsigned short*>(row_s)[idx] = (unsigned short)v;
            else row_s[idx] = __int_as_float(v);
        }
        __syncwarp();
        if (packed) {
            uint4* dst = reinterpret_cast<uint4*>(q_out + r * n_bins);
            const uint4* src = reinterpret_cast<const uint4*>(row_s);
            for (int v = lane; v < (n_bins >> 3); v += 32) dst[v] = src[v];
        } else if (VEC) {
            uint4* dst = reinterpret_cast<uint4*>(q_out + r * n_bins);
            const int4* src = reinterpret_cast<const int4*>(row_s);
            for (int v = lane; v < (n_bins >> 3); v += 32) {
                const int4 a = src[2 * v], b = src[2 * v + 1];     // eight integers, each 0..65535
                dst[v] = make_uint4((unsigned)a.x | ((unsigned)a.y << 16), (unsigned)a.z | ((unsigned)a.w << 16),
                                    (unsigned)b.x | ((unsigned)b.y << 16), (unsigned)b.z | ((unsigned)b.w << 16));
            }
        } else {
            for (int e = lane; e < n_bins; e += 32)
                q_out[r * n_bins + e] = (unsigned short)__float_as_int(row_s[e]);
        }
        __syncwarp();
    }
}

// The inverse: uint16 row -> float32 row / (sum + eps). The elements are integers 0..65535 and a
// positive sum is an integer 1..n_bins x 65535, so the hoisted division applies to every row with
// an ordinary eps (a zero element gives an exact 0).
template <bool VEC>
__global__ void __launch_bounds__(kQThreads, NSC_DQ_MIN_BLOCKS)
dequantize_kernel(const unsigned short* __restrict__ q_in, long long n_rows, int n_bins, float eps,
                  const __grid_constant__ SumPlan plan, float* __restrict__ hist) {
    extern __shared__ __align__(16) float smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float* row_s = smem + warp * (n_bins + kSumSlots);
    float* slot_s = row_s + n_bins;
    const float uniform = __fdiv_rn(1.0f, (float)n_bins);
    const long long n_warps = (long long)gridDim.x * kQWarps;
    for (long long r = (long long)blockIdx.x * kQWarps + warp; r < n_rows; r += n_warps) {
        if (VEC) {
            // four uint16 (8 bytes) per lane -> one float4 per lane: consecutive lanes, consecutive
            // 16-byte slots of the row (no shared-memory bank conflicts)
            const uint2* src = reinterpret_cast<const uint2*>(q_in + r * n_bins);
            float4* dst = reinterpret_cast<float4*>(row_s);
            const int n_vec = n_bins >> 2;
            for (int v0 = 0; v0 < n_vec; v0 += 32 * kVecBatch) {
                uint2 t[kVecBatch];
#pragma unroll
                for (int k = 0; k < kVecBatch; ++k) {
                    const int v = v0 + k * 32 + lane;
                    if (v < n_vec) t[k] = __ldg(src + v);
                }
#pragma unroll
                for (int k = 0; k < kVecBatch; ++k) {
                    const int v = v0 + k * 32 + lane;
                    if (v < n_vec)
                        dst[v] = make_float4((float)(t[k].x & 0xffffu), (float)(t[k].x >> 16),
                                             (float)(t[k].y & 0xffffu), (float)(t[k].y >> 16));
                }
            }
        } else {
            for (int e = lane; e < n_bins; e += 32) row_s[e] = (float)q_in[r * n_bins + e];
        }
        __syncwarp();
        const float sum = numpy_sum(row_s, plan, slot_s, lane);
        const bool norm = sum > eps;                       // quantization.py:184-190
        const float denom = __fadd_rn(sum, eps);
        const bool hoisted = norm && denom >= 0.5f && moderate(denom);
        const RowDivisor div(hoisted ? denom : 1.0f);
        if (VEC) {
            float4* dst = reinterpret_cast<float4*>(hist + r * n_bins);
            const float4* src = reinterpret_cast<const float4*>(row_s);
            for (int v = lane; v < (n_bins >> 2); v += 32) {
                float4 h = src[v];
                if (hoisted) {
                    h = make_float4(div(h.x), div(h.y), div(h.z), div(h.w));
                } else {
                    h.x = norm ? __fdiv_rn(h.x, denom) : uniform;
                    h.y = norm ? __fdiv_rn(h.y, denom) : uniform;
                    h.z = norm ? __fdiv_rn(h.z, denom) : uniform;
                    h.w = norm ? __fdiv_rn(h.w, denom) : uniform;
                }
                dst[v] = h;
            }
        } else {
            for (int e = lane; e < n_bins; e += 32)
                hist[r * n_bins + e] = hoisted ? div(row_s[e]) : (norm ? __fdiv_rn(row_s[e], denom) : uniform);
        }
        __syncwarp();
    }
}

bool rows_vectorisable(const void* a, const void* b, int n_bins) {
    return n_bins % 8 == 0 && (reinterpret_cast<uintptr_t>(a) & 15) == 0 && (reinterpret_cast<uintptr_t>(b) & 15) == 0;
}

int launch_cfg(long long n_rows, int n_bins, int* n_sms, size_t* smem, SumPlan* plan) {
    if (n_rows < 0) return NSC_ERR_BAD_COUNT;
    const int st = build_plan(n_bins, plan);
    if (st != NSC_OK) return st;
    int dev = 0, sms = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return record_cuda(e);
    e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (e != cudaSuccess) return record_cuda(e);
    *n_sms = sms;
    *smem = (size_t)kQWarps * (n_bins + kSumSlots) * 4;
    return NSC_OK;
}

// One wave of CTAs, all resident: the rows are dealt round-robin to the warps of the grid, so a grid
// larger than what fits would run its surplus CTAs as a second, mostly empty wave.
template <typename K, typename... Args>
int launch_rows(K kernel, int sms, size_t smem, long long n_rows, cudaStream_t stream, Args... args) {
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return record_cuda(e);
    int resident = 0;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&resident, kernel, kQThreads, smem);
    if (e != cudaSuccess) return record_cuda(e);
    if (resident < 1) return NSC_ERR_BAD_PARAMS;
    long long g = (n_rows + kQWarps - 1) / kQWarps;
    if (g > (long long)sms * resident) g = (long long)sms * resident;
    kernel<<<(int)g, kQThreads, smem, stream>>>(args...);
    return record_cuda(cudaGetLastError());
}

}  // namespace

}  // namespace nsc

using namespace nsc;

extern "C" {

int nsc_quantize_histograms(const float* d_hist, int64_t n_rows, int n_bins, float epsilon,
                            uint16_t* d_quantized, void* stream) {
    int sms = 0;
    size_t smem = 0;
    SumPlan plan;
    int st = launch_cfg(n_rows, n_bins, &sms, &smem, &plan);
    if (st != NSC_OK) return st;
    if (n_rows == 0) return NSC_OK;
    if (!d_hist || !d_quantized) return NSC_ERR_NULL_POINTER;
    auto kernel = rows_vectorisable(d_hist, d_quantized, n_bins) ? quantize_kernel<true> : quantize_kernel<false>;
    return launch_rows(kernel, sms, smem, n_rows, (cudaStream_t)stream, d_hist, (long long)n_rows, n_bins, epsilon,
                       plan, d_quantized);
}

int nsc_dequantize_histograms(const uint16_t* d_quantized, int64_t n_rows, int n_bins, float epsilon,
                              float* d_hist, void* stream) {
    int sms = 0;
    size_t smem = 0;
    SumPlan plan;
    int st = launch_cfg(n_rows, n_bins, &sms, &smem, &plan);
    if (st != NSC_OK) return st;
    if (n_rows == 0) return NSC_OK;
    if (!d_hist || !d_quantized) return NSC_ERR_NULL_POINTER;
    auto kernel = rows_vectorisable(d_hist, d_quantized, n_bins) ? dequantize_kernel<true> : dequantize_kernel<false>;
    return launch_rows(kernel, sms, smem, n_rows, (cudaStream_t)stream, d_quantized, (long long)n_rows, n_bins,
                       epsilon, plan, d_hist);
}

int nsc_test_pairwise_sum_plan(int n_bins, int32_t* n_leaves, int32_t* n_adds, int32_t* result_slot,
                               uint16_t* leaf_start, uint16_t* leaf_len, uint8_t* add_a, uint8_t* add_b) {
    if (!n_leaves || !n_adds || !result_slot || !leaf_start || !leaf_len || !add_a || !add_b)
        return NSC_ERR_NULL_POINTER;
    SumPlan plan;
    const int st = build_plan(n_bins, &plan);
    if (st != NSC_OK) return st;
    *n_leaves = plan.n_leaves;
    *n_adds = plan.n_adds;
    *result_slot = plan.result_slot;
    for (int l = 0; l < plan.n_leaves; ++l) {
        leaf_start[l] = plan.leaf_start[l];
        leaf_len[l] = plan.leaf_len[l];
    }
    for (int t = 0; t < plan.n_adds; ++t) {
        add_a[t] = plan.add_a[t];
        add_b[t] = plan.add_b[t];
    }
    return NSC_OK;
}

}  // extern "C"
