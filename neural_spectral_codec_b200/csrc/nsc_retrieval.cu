// Stage-1 retrieval over the descriptor database (SURVEY.md 8(f) rank 1): 1-D Wasserstein
// distance = sum |CDF_db - CDF_query| (reference src/retrieval/wasserstein.py:134-172), the
// spatial exclusion of src/retrieval/two_stage_retrieval.py:158-166 and the top-K of
// wasserstein.py:358-364, as three kernels:
//   cdf_rows_kernel        histogram rows -> normalised CDF rows, once per database insert
//   wasserstein_kernel     streams the CDF rows once per group of <= kMaxQueries queries (HBM bound:
//                          4*n_bins bytes per row), writes the (Q, N) distances, +inf where excluded
//                          and every warp's smallest (distance, index) key per query
//   select_kernel          k <= 128: many CTAs per query. The k-th smallest of 256 group minima
//                          (groups of warp minima = disjoint row sets) bounds the k-th smallest key
//                          from above; each CTA collects the keys of its slice under the bound (a
//                          few more than k in all), the last CTA of a query sorts them. ~5 us
//                          instead of one CTA re-reading all N distances.
//                          (a candidate overflow -- fewer than k finite group minima -- is
//                          resolved by that CTA with an exact 8-pass radix select of the 64-bit keys)
//   topk_kernel            128 < k <= 1024: one CTA per query, per-thread-minimum bound + candidate
//                          sort, 4-pass radix select as the last resort
// and, for nsc_wasserstein_rank (any k), a stable segmented radix sort of each query's distances:
// rank_hist_kernel, rank_scan_kernel, rank_scatter_kernel (see "rank" below).
#include <math.h>

#include "nsc_internal.h"

namespace nsc {

namespace {

constexpr int kRThreads = 256;
constexpr int kRWarps = kRThreads / 32;
constexpr int kMaxQueries = 8;      // query CDFs resident in shared memory per launch
constexpr int kMaxPerLane = 32;     // n_bins <= 1024
constexpr int kTopThreads = 1024;

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
    return v;
}

// A warp turns one histogram row, staged in shared memory, into its normalised CDF held in
// registers: lane l owns the contiguous elements [l*per, (l+1)*per). mode 0: database row,
// h / (sum + eps) if sum > eps else h (wasserstein.py:157-162); mode 1: query, h / sum if
// sum > eps (wasserstein.py:152-154).
template <int MODE>
__device__ __forceinline__ void row_cdf(const float* row_s, int n_bins, int per, float eps, int lane,
                                        float* c /* kMaxPerLane */) {
    float s = 0.0f;
#pragma unroll
    for (int i = 0; i < kMaxPerLane; ++i) {
        const int e = lane * per + i;
        c[i] = (i < per && e < n_bins) ? row_s[e] : 0.0f;
        s += c[i];
    }
    const float total = warp_sum(s);
    const bool norm = total > eps;
    const float denom = MODE == 0 ? total + eps : total;
    float run = 0.0f;
#pragma unroll
    for (int i = 0; i < kMaxPerLane; ++i) {
        if (i < per) {
            const float h = norm ? __fdiv_rn(c[i], denom) : c[i];
            run += h;
            c[i] = run;
        }
    }
    // exclusive scan of the lane totals
    float incl = run;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const float o = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += o;
    }
    const float offset = incl - run;
#pragma unroll
    for (int i = 0; i < kMaxPerLane; ++i)
        if (i < per) c[i] += offset;
}

__global__ void __launch_bounds__(kRThreads)
cdf_rows_kernel(const float* __restrict__ hists, long long n, int n_bins, float eps,
                float* __restrict__ cdfs) {
    extern __shared__ float smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int per = (n_bins + 31) / 32;
    float* row_s = smem + warp * (per * 32);
    const long long n_warps = (long long)gridDim.x * kRWarps;
    for (long long r = (long long)blockIdx.x * kRWarps + warp; r < n; r += n_warps) {
        const float* src = hists + r * n_bins;
        for (int e = lane; e < per * 32; e += 32) row_s[e] = e < n_bins ? __ldcs(src + e) : 0.0f;
        __syncwarp();
        float c[kMaxPerLane];
        row_cdf<0>(row_s, n_bins, per, eps, lane, c);
        __syncwarp();
#pragma unroll
        for (int i = 0; i < kMaxPerLane; ++i)
            if (i < per) row_s[lane * per + i] = c[i];
        __syncwarp();
        float* dst = cdfs + r * n_bins;
        for (int e = lane; e < n_bins; e += 32) dst[e] = row_s[e];
        __syncwarp();
    }
}

// uint16 rows -> uint16 CDF rows in units of 1/65535, one warp per row: an integer prefix scan S
// (lane l owns the contiguous elements [l*per, (l+1)*per), like row_cdf) and the total T = S[n-1].
// T = 65535 (every quantised row): S itself, exact. T = 0: zeros (the distance pass reads them as
// the uniform CDF). Any other T: round-half-even(65535 S / T) in 64-bit integers.
__global__ void __launch_bounds__(kRThreads)
cdf16_rows_kernel(const unsigned short* __restrict__ rows, long long n, int n_bins,
                  unsigned short* __restrict__ cdfs) {
    extern __shared__ unsigned short smem16[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int per = (n_bins + 31) / 32;
    unsigned short* row_s = smem16 + warp * (per * 32);
    const long long n_warps = (long long)gridDim.x * kRWarps;
    for (long long r = (long long)blockIdx.x * kRWarps + warp; r < n; r += n_warps) {
        const unsigned short* src = rows + r * n_bins;
        for (int e = lane; e < per * 32; e += 32) row_s[e] = e < n_bins ? __ldcs(src + e) : 0;
        __syncwarp();
        unsigned s[kMaxPerLane];
        unsigned run = 0;
#pragma unroll
        for (int i = 0; i < kMaxPerLane; ++i)
            if (i < per) {
                run += row_s[lane * per + i];
                s[i] = run;
            }
        unsigned incl = run;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const unsigned o = __shfl_up_sync(0xffffffffu, incl, d);
            if (lane >= d) incl += o;
        }
        const unsigned offset = incl - run;
        const unsigned total = __shfl_sync(0xffffffffu, incl, 31);
        __syncwarp();
#pragma unroll
        for (int i = 0; i < kMaxPerLane; ++i)
            if (i < per) {
                unsigned v = s[i] + offset;
                if (total == 0) {
                    v = 0;
                } else if (total != 65535u) {
                    const unsigned long long num = 65535ull * v;
                    unsigned long long qt = num / total;
                    const unsigned long long rem = num - qt * total;
                    if (2 * rem > total || (2 * rem == total && (qt & 1))) ++qt;
                    v = (unsigned)qt;
                }
                row_s[lane * per + i] = (unsigned short)v;
            }
        __syncwarp();
        unsigned short* dst = cdfs + r * n_bins;
        for (int e = lane; e < n_bins; e += 32) dst[e] = row_s[e];
        __syncwarp();
    }
}

struct QueryArgs {
    const float* queries;     // Q x n_bins histograms
    const void* db_cdfs;      // N x n_bins: float32 CDF rows, or uint16 rows in units of 1/65535
    const double* db_xyz;     // N x 3 or null
    const double* query_xyz;  // Q x 3 or null
    double min_dist;
    float* distances;         // Q x N
    unsigned long long* warp_min;   // Q x (gridDim.x * kRWarps) smallest (distance bits, row) per warp, or null
    long long n_db;
    int n_queries, n_bins;
    float eps;
};

// CDF rows per warp ring (one fewer in flight): 4 when two CTAs per SM still fit, else 3

__device__ __forceinline__ void cp_async4(void* dst, const void* src) {
    const unsigned d = (unsigned)__cvta_generic_to_shared(dst);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(d), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async16(void* dst, const void* src) {
    const unsigned d = (unsigned)__cvta_generic_to_shared(dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(src) : "memory");
}

// PER = elements per lane (n_bins <= 32 * PER); PER = 25 is the 800-D descriptor.
// T = float: CDF rows of nsc_wasserstein_cdf. T = unsigned short: rows of nsc_wasserstein_cdf_u16 in
// units of 1/65535 (counts). The uint16 instantiation works in counts: each query CDF is scaled by
// 65535 once when it is staged, each database element converts to float exactly, and the sum of a
// row is scaled back by 1/65535 once.
template <typename T, int PER, int kRowStages>
__global__ void __launch_bounds__(kRThreads)
wasserstein_kernel(const __grid_constant__ QueryArgs a) {
    constexpr bool kCounts = sizeof(T) == 2;
    extern __shared__ __align__(16) float smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    constexpr int padded = PER * 32;
    float* qcdf = smem;                                           // Q x padded
    T* ring = reinterpret_cast<T*>(smem + a.n_queries * padded) + warp * (kRowStages * padded);
    const long long n_warps = (long long)gridDim.x * kRWarps;
    const long long r0 = (long long)blockIdx.x * kRWarps + warp;
    // 16-byte copies where every row starts on a 16-byte boundary. uint16 rows: 4-byte copies of
    // element pairs where rows start on 4-byte boundaries; an odd n_bins (or an unaligned base) has
    // no cp.async size, so those rows go through plain loads (synchronous, still in ring order).
    const bool vec = kCounts ? (a.n_bins & 7) == 0 && (reinterpret_cast<uintptr_t>(a.db_cdfs) & 15) == 0
                             : (a.n_bins & 3) == 0;
    const bool pairs = kCounts && (a.n_bins & 1) == 0 && (reinterpret_cast<uintptr_t>(a.db_cdfs) & 3) == 0;
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");   // the selection may become resident now
    if (a.n_bins < padded)
        for (int s = 0; s < kRowStages; ++s)
            for (int e = a.n_bins + lane; e < padded; e += 32) ring[s * padded + e] = T(0);
    __syncwarp();
    auto issue = [&](long long r, int slot) {
        if (r < a.n_db) {
            const T* src = static_cast<const T*>(a.db_cdfs) + r * a.n_bins;
            T* dst = ring + slot * padded;
            constexpr int kVec = 16 / sizeof(T);
            if (vec) {
                for (int e = lane * kVec; e < a.n_bins; e += 32 * kVec) cp_async16(dst + e, src + e);
            } else if (!kCounts) {
                for (int e = lane; e < a.n_bins; e += 32) cp_async4(dst + e, src + e);
            } else if (pairs) {
                for (int e = lane * 2; e < a.n_bins; e += 64) cp_async4(dst + e, src + e);
            } else {
                for (int e = lane; e < a.n_bins; e += 32) dst[e] = src[e];
            }
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    // the first rows are on their way while the query CDFs are built
#pragma unroll
    for (int s = 0; s < kRowStages - 1; ++s) issue(r0 + s * n_warps, s);
    // query CDFs (wasserstein.py:152-154,165), one warp per query, staged through the ring slot
    // the prologue above left free (its padding lanes stay zero). A uint16 ring slot is too small
    // for a float row, so there the query is staged in its own qcdf row: row_cdf reads the whole row
    // into registers before the warp overwrites it.
    {
        float* stage = reinterpret_cast<float*>(ring + (kRowStages - 1) * padded);
        for (int q = warp; q < a.n_queries; q += kRWarps) {
            if (kCounts) stage = qcdf + q * padded;
            for (int e = lane; e < padded; e += 32) stage[e] = e < a.n_bins ? a.queries[(long long)q * a.n_bins + e] : 0.0f;
            __syncwarp();
            float c[kMaxPerLane];
            row_cdf<1>(stage, a.n_bins, PER, a.eps, lane, c);
            if (kCounts) __syncwarp();
#pragma unroll
            for (int i = 0; i < PER; ++i)      // padding lanes hold 0, like the padding of the database rows
                qcdf[q * padded + lane * PER + i] = lane * PER + i < a.n_bins ? (kCounts ? c[i] * 65535.0f : c[i]) : 0.0f;
            __syncwarp();
        }
    }
    // an all-zero uint16 row (an empty scan's wire row) stands for the uniform CDF (i + 1) / n_bins,
    // which dequantize yields for it: 65535 (i + 1) / n_bins counts, rounded once
    const double uniform_step = kCounts ? 65535.0 / a.n_bins : 0.0;
    __syncthreads();
    const bool spatial = a.db_xyz != nullptr && a.query_xyz != nullptr;
    int slot = 0;
    unsigned long long best[kMaxQueries];       // lane 0: smallest key of this warp's rows, per query
#pragma unroll
    for (int q = 0; q < kMaxQueries; ++q) best[q] = ~0ull;
    for (long long r = r0; r < a.n_db; r += n_warps) {
        issue(r + (kRowStages - 1) * n_warps, (slot + kRowStages - 1) % kRowStages);
        asm volatile("cp.async.wait_group %0;" ::"n"(kRowStages - 1) : "memory");
        __syncwarp();
        const T* row_s = ring + slot * padded + lane * PER;
        float c[PER];
#pragma unroll
        for (int i = 0; i < PER; ++i) {
            if (kCounts)      // 2^23 + c as float bits, minus 2^23: exact for 0 <= c <= 65535
                c[i] = __uint_as_float(0x4B000000u | (unsigned)row_s[i]) - 8388608.0f;
            else
                c[i] = row_s[i];
        }
        if (kCounts && ring[slot * padded + a.n_bins - 1] == T(0)) {   // CDF rows end on 0 only when all zero
#pragma unroll
            for (int i = 0; i < PER; ++i) {
                const int e = lane * PER + i;
                c[i] = e < a.n_bins ? (float)((e + 1) * uniform_step) : 0.0f;
            }
        }
        double px = 0, py = 0, pz = 0;
        if (spatial && lane == 0) { px = a.db_xyz[3 * r]; py = a.db_xyz[3 * r + 1]; pz = a.db_xyz[3 * r + 2]; }
#pragma unroll
        for (int q = 0; q < kMaxQueries; ++q) {
            if (q >= a.n_queries) break;
            const float* qc = qcdf + q * padded + lane * PER;
            float d0 = 0.0f, d1 = 0.0f;
#pragma unroll
            for (int i = 0; i + 1 < PER; i += 2) {
                d0 += fabsf(c[i] - qc[i]);
                d1 += fabsf(c[i + 1] - qc[i + 1]);
            }
            if (PER & 1) d0 += fabsf(c[PER - 1] - qc[PER - 1]);
            float d = warp_sum(d0 + d1);
            if (kCounts) d *= 1.0f / 65535.0f;
            if (lane == 0) {
                if (spatial) {   // two_stage_retrieval.py:160-164: skip keyframes closer than the threshold
                    const double dx = px - a.query_xyz[3 * q], dy = py - a.query_xyz[3 * q + 1],
                                 dz = pz - a.query_xyz[3 * q + 2];
                    if (sqrt(dx * dx + dy * dy + dz * dz) < a.min_dist) d = INFINITY;
                }
                a.distances[(long long)q * a.n_db + r] = d;
                const unsigned long long key = ((unsigned long long)__float_as_uint(d) << 32) | (unsigned)r;
                best[q] = key < best[q] ? key : best[q];
            }
        }
        __syncwarp();
        slot = (slot + 1) % kRowStages;
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    if (a.warp_min && lane == 0) {
#pragma unroll
        for (int q = 0; q < kMaxQueries; ++q)
            if (q < a.n_queries)
                a.warp_min[(long long)q * n_warps + (long long)blockIdx.x * kRWarps + warp] = best[q];
    }
}

// ---- top-K ----------------------------------------------------------------------------------
struct TopkArgs {
    const float* distances;   // Q x N, >= 0 or +inf (excluded)
    long long n_db;
    int k;
    long long* top_idx;       // Q x k, -1 padded
    float* top_dist;          // Q x k, +inf padded
    int* top_count;           // Q
};

// Workspace of the selection, per query: counters {candidates, CTAs done, overflow, pad}, then
// kSelCap candidate keys, then the warp minima of the distance pass. Zero before the first call;
// every call leaves the counters zero again.
constexpr int kSelThreads = 256;      // == the radix of the fallback select
#ifndef NSC_SEL_CAP
#define NSC_SEL_CAP 1024               // the tuning build uses 128 so that the tests reach the overflow path
#endif
constexpr int kSelCap = NSC_SEL_CAP;
constexpr int kSelMaxK = 128;
static_assert(kSelCap >= kSelMaxK && kSelCap <= 1024 && (kSelCap & (kSelCap - 1)) == 0, "candidate list");
constexpr int kSelCtas = 128;         // CTAs per query, at most
struct SelectArgs {
    const float* distances;
    const unsigned long long* warp_min;   // Q x n_min
    int n_min;
    long long n_db;
    int k;
    int* counters;                        // Q x 4
    unsigned long long* cand;             // Q x kSelCap
    long long* top_idx;
    float* top_dist;
    int* top_count;
};

// ascending bitonic sort of n (power of two, <= 1024) 64-bit keys in shared memory
template <int NT>
__device__ __forceinline__ void bitonic_sort_keys(unsigned long long* sel, unsigned n) {
    for (unsigned size = 2; size <= n; size <<= 1) {
        for (unsigned stride = size >> 1; stride > 0; stride >>= 1) {
            for (unsigned t = threadIdx.x; t < n; t += NT) {
                const unsigned j = t ^ stride;
                if (j > t) {
                    const unsigned long long x = sel[t], y = sel[j];
                    const bool up = (t & size) == 0;
                    if ((x > y) == up) { sel[t] = y; sel[j] = x; }
                }
            }
            __syncthreads();
        }
    }
}

__global__ void __launch_bounds__(kSelThreads)
select_kernel(const __grid_constant__ SelectArgs a) {
    __shared__ unsigned long long sel[kSelCap];
    __shared__ int s_last, s_count, s_valid;
    const int q = blockIdx.y, g = blockIdx.x, tid = threadIdx.x;
    const unsigned kInf = 0x7f800000u;
    // launched as a programmatic dependent of the distance pass: resident early, released when that
    // grid has completed and its writes are visible
    asm volatile("griddepcontrol.wait;" ::: "memory");
    // 1. bound: k-th smallest of 256 group minima (each group = the rows of some warps)
    unsigned long long m = ~0ull;
    {
        const unsigned long long* wm = a.warp_min + (long long)q * a.n_min;
        int i = tid;
        for (; i + 3 * kSelThreads < a.n_min; i += 4 * kSelThreads) {        // four loads in flight
            const unsigned long long v0 = __ldcg(wm + i), v1 = __ldcg(wm + i + kSelThreads),
                                     v2 = __ldcg(wm + i + 2 * kSelThreads), v3 = __ldcg(wm + i + 3 * kSelThreads);
            const unsigned long long a01 = v0 < v1 ? v0 : v1, a23 = v2 < v3 ? v2 : v3;
            const unsigned long long a03 = a01 < a23 ? a01 : a23;
            m = a03 < m ? a03 : m;
        }
        for (; i < a.n_min; i += kSelThreads) {
            const unsigned long long v = __ldcg(wm + i);
            m = v < m ? v : m;
        }
    }
    sel[tid] = m;
    __syncthreads();
    bitonic_sort_keys<kSelThreads>(sel, kSelThreads);
    unsigned long long bound = sel[a.k - 1];
    const unsigned long long finite_max = ((unsigned long long)(kInf - 1u) << 32) | 0xffffffffull;
    if (bound > finite_max) bound = finite_max;            // fewer than k finite minima: take every finite key
    __syncthreads();
    // 2. this CTA's slice of the row: keys under the bound go to the query's candidate list
    const long long per = (a.n_db + gridDim.x - 1) / gridDim.x;
    const long long lo = (long long)g * per, hi = lo + per < a.n_db ? lo + per : a.n_db;
    const unsigned* keys = reinterpret_cast<const unsigned*>(a.distances + (long long)q * a.n_db);
    int* cnt = a.counters + 4 * q;
    auto consider = [&](unsigned bits, long long i) {
        const unsigned long long key = ((unsigned long long)bits << 32) | (unsigned)i;
        if (key <= bound) {
            const int pos = atomicAdd(&cnt[0], 1);
            if (pos < kSelCap) a.cand[(long long)q * kSelCap + pos] = key;
        }
    };
    {
        long long i = lo + tid;
        for (; i + 3 * kSelThreads < hi; i += 4 * kSelThreads) {               // four loads in flight
            const unsigned k0 = __ldcg(keys + i), k1 = __ldcg(keys + i + kSelThreads),
                           k2 = __ldcg(keys + i + 2 * kSelThreads), k3 = __ldcg(keys + i + 3 * kSelThreads);
            consider(k0, i);
            consider(k1, i + kSelThreads);
            consider(k2, i + 2 * kSelThreads);
            consider(k3, i + 3 * kSelThreads);
        }
        for (; i < hi; i += kSelThreads) consider(__ldcg(keys + i), i);
    }
    // 3. the last CTA of the query sorts the candidates
    __threadfence();
    __syncthreads();
    if (tid == 0) {
        const int ticket = atomicAdd(&cnt[1], 1);
        s_last = ticket == (int)gridDim.x - 1;
        s_valid = 0;
        if (s_last) {
            __threadfence();
            s_count = atomicAdd(&cnt[0], 0);
        }
    }
    __syncthreads();
    if (!s_last) return;
    const int n_cand = s_count;
    if (tid == 0) { cnt[0] = 0; cnt[1] = 0; }              // leave the workspace clean for the next call
    int n_have = n_cand;
    if (n_cand > kSelCap) {
        // More keys under the bound than the candidate list holds (fewer than k finite group
        // minima, or rows clustered in few groups). Rare, so this CTA alone finds the exact k-th
        // smallest key by an 8-pass radix select over all N keys -- they are distinct 64-bit
        // values (distance bits, row), so there are no ties to order -- and collects the keys
        // up to it.
        __shared__ unsigned hist[256];
        __shared__ unsigned long long s_prefix;
        __shared__ unsigned s_need;
        unsigned long long prefix = 0;
        unsigned need = (unsigned)a.k;
        for (int shift = 56; shift >= 0; shift -= 8) {
            hist[tid] = 0;                                   // kSelThreads == 256
            __syncthreads();
            for (long long i = tid; i < a.n_db; i += kSelThreads) {
                const unsigned long long key = ((unsigned long long)__ldcg(keys + i) << 32) | (unsigned)i;
                if (key <= finite_max && (shift == 56 || (key >> (shift + 8)) == (prefix >> (shift + 8))))
                    atomicAdd(&hist[(unsigned)(key >> shift) & 255u], 1u);
            }
            __syncthreads();
            if (tid == 0) {
                unsigned acc = 0, b = 0;
                for (; b < 255; ++b) {
                    if (acc + hist[b] >= need) break;
                    acc += hist[b];
                }
                s_prefix = prefix | ((unsigned long long)b << shift);
                s_need = need - acc;                         // fewer than k finite keys: ends on the largest one
            }
            __syncthreads();
            prefix = s_prefix;
            need = s_need;
        }
        if (tid == 0) s_count = 0;
        for (int i = tid; i < kSelCap; i += kSelThreads) sel[i] = ~0ull;
        __syncthreads();
        for (long long i = tid; i < a.n_db; i += kSelThreads) {
            const unsigned long long key = ((unsigned long long)__ldcg(keys + i) << 32) | (unsigned)i;
            if (key <= prefix && key <= finite_max) {
                const int pos = atomicAdd(&s_count, 1);
                if (pos < kSelCap) sel[pos] = key;
            }
        }
        __syncthreads();
        n_have = s_count < kSelCap ? s_count : kSelCap;
    } else {
        for (int i = tid; i < kSelCap; i += kSelThreads)
            sel[i] = i < n_cand ? __ldcg(a.cand + (long long)q * kSelCap + i) : ~0ull;
        __syncthreads();
    }
    unsigned n_sort = 32;
    while ((int)n_sort < n_have) n_sort <<= 1;
    bitonic_sort_keys<kSelThreads>(sel, n_sort);
    int valid = 0;                                          // finite candidates among the first k
    for (int i = tid; i < a.k; i += kSelThreads) {
        const bool ok = i < n_have && (unsigned)(sel[i] >> 32) < kInf;
        a.top_idx[(long long)q * a.k + i] = ok ? (long long)(unsigned)(sel[i] & 0xffffffffull) : -1;
        a.top_dist[(long long)q * a.k + i] = ok ? __uint_as_float((unsigned)(sel[i] >> 32)) : INFINITY;
        valid += ok;
    }
    valid = __reduce_add_sync(0xffffffffu, valid);
    if ((tid & 31) == 0 && valid) atomicAdd(&s_valid, valid);
    __syncthreads();
    if (tid == 0) a.top_count[q] = s_valid;
}

__device__ __forceinline__ unsigned block_excl_scan(unsigned v, unsigned* warp_tot, unsigned* total) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    unsigned incl = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const unsigned o = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += o;
    }
    if (lane == 31) warp_tot[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        unsigned t = warp_tot[lane];
        unsigned ti = t;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const unsigned o = __shfl_up_sync(0xffffffffu, ti, d);
            if (lane >= d) ti += o;
        }
        warp_tot[lane] = ti - t;
        if (lane == 31) *total = ti;
    }
    __syncthreads();
    const unsigned r = warp_tot[warp] + incl - v;
    __syncthreads();
    return r;
}

__device__ __forceinline__ void bitonic_sort_1024(unsigned long long* sel) {
    const unsigned tid = threadIdx.x;
    for (unsigned size = 2; size <= kTopThreads; size <<= 1) {
        for (unsigned stride = size >> 1; stride > 0; stride >>= 1) {
            const unsigned j = tid ^ stride;
            if (j > tid) {
                const unsigned long long x = sel[tid], y = sel[j];
                const bool up = (tid & size) == 0;
                if ((x > y) == up) { sel[tid] = y; sel[j] = x; }
            }
            __syncthreads();
        }
    }
}

// One CTA per query. Fast path: the k-th smallest of the 1024 per-thread minima bounds the k-th
// smallest distance from above, and (unless the distances are massively tied) only a few more
// than k keys lie under that bound: collect them, sort, done -- two passes over the keys.
// Fallback (more than 1024 keys under the bound): 4-pass radix select of the k-th smallest
// key with warp-aggregated histogram updates, then gather (ordered for surplus ties).
__global__ void __launch_bounds__(kTopThreads)
topk_kernel(const __grid_constant__ TopkArgs a) {
    __shared__ unsigned hist[256];
    __shared__ unsigned warp_tot[32];
    __shared__ unsigned s_total, s_prefix, s_need, s_nvalid, s_eq_total, s_fill;
    __shared__ unsigned long long sel[kTopThreads];
    const int q = blockIdx.x, tid = threadIdx.x, lane = tid & 31;
    const unsigned* keys = reinterpret_cast<const unsigned*>(a.distances + (long long)q * a.n_db);
    const unsigned kInf = 0x7f800000u;
    const long long n_round = (a.n_db + kTopThreads - 1) / kTopThreads * kTopThreads;

    // pass A: per-thread minimum and the number of candidates (finite distances)
    unsigned lmin = 0xffffffffu, valid = 0;
    {
        long long i = tid;
        for (; i + 3 * kTopThreads < a.n_db; i += 4 * kTopThreads) {
            const unsigned k0 = keys[i], k1 = keys[i + kTopThreads], k2 = keys[i + 2 * kTopThreads],
                           k3 = keys[i + 3 * kTopThreads];
            lmin = min(min(lmin, k0), min(k1, min(k2, k3)));
            valid += (k0 < kInf) + (k1 < kInf) + (k2 < kInf) + (k3 < kInf);
        }
        for (; i < a.n_db; i += kTopThreads) {
            const unsigned k0 = keys[i];
            lmin = min(lmin, k0);
            valid += k0 < kInf;
        }
    }
    if (tid == 0) { s_nvalid = 0; s_fill = 0; }
    sel[tid] = (unsigned long long)lmin << 32;
    __syncthreads();
    valid = (unsigned)__reduce_add_sync(0xffffffffu, valid);
    if (lane == 0) atomicAdd(&s_nvalid, valid);
    bitonic_sort_1024(sel);                       // ends with a barrier
    const unsigned k = min((unsigned)a.k, s_nvalid);
    const unsigned bound = k > 0 ? min((unsigned)(sel[k - 1] >> 32), kInf - 1u) : 0u;
    __syncthreads();
    sel[tid] = ~0ull;
    __syncthreads();
    // pass B: collect every key <= bound
    if (k > 0) {
        long long i = tid;
        for (; i + 3 * kTopThreads < a.n_db; i += 4 * kTopThreads) {
            unsigned kk[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) kk[u] = keys[i + u * kTopThreads];
#pragma unroll
            for (int u = 0; u < 4; ++u)
                if (kk[u] <= bound) {
                    const unsigned pos = atomicAdd(&s_fill, 1u);
                    if (pos < kTopThreads) sel[pos] = ((unsigned long long)kk[u] << 32) | (unsigned)(i + u * kTopThreads);
                }
        }
        for (; i < a.n_db; i += kTopThreads) {
            const unsigned k0 = keys[i];
            if (k0 <= bound) {
                const unsigned pos = atomicAdd(&s_fill, 1u);
                if (pos < kTopThreads) sel[pos] = ((unsigned long long)k0 << 32) | (unsigned)i;
            }
        }
    }
    __syncthreads();
    const bool overflow = s_fill > kTopThreads;
    __syncthreads();

    if (overflow) {
        unsigned prefix = 0, need = k;
        for (int shift = 24; shift >= 0; shift -= 8) {
            if (tid < 256) hist[tid] = 0;
            __syncthreads();
            const unsigned mask_hi = shift == 24 ? 0u : (0xffffffffu << (shift + 8));
            for (long long i = tid; i < n_round; i += kTopThreads) {
                const unsigned key = i < a.n_db ? keys[i] : 0xffffffffu;
                const bool act = i < a.n_db && (key & mask_hi) == prefix;
                const unsigned amask = __ballot_sync(0xffffffffu, act);
                if (act) {
                    const unsigned bin = (key >> shift) & 255u;
                    const unsigned peers = __match_any_sync(amask, bin);
                    if (lane == __ffs(peers) - 1) atomicAdd(&hist[bin], (unsigned)__popc(peers));
                }
            }
            __syncthreads();
            if (tid == 0) {
                unsigned acc = 0, b = 0;
                for (; b < 256; ++b) {
                    if (acc + hist[b] >= need) break;
                    acc += hist[b];
                }
                s_prefix = prefix | (b << shift);
                s_need = need - acc;
                s_eq_total = hist[b];      // after the last pass: keys equal to the k-th smallest
            }
            __syncthreads();
            prefix = s_prefix;
            need = s_need;
        }
        // every key < prefix and `need` keys == prefix; with surplus ties the lowest indices win
        const unsigned n_less = k - need;
        sel[tid] = ~0ull;
        if (tid == 0) s_fill = 0;
        __syncthreads();
        const bool all_eq = s_eq_total == need;
        for (long long i = tid; i < a.n_db; i += kTopThreads) {
            const unsigned key = keys[i];
            if (key < prefix || (all_eq && key == prefix))
                sel[atomicAdd(&s_fill, 1u)] = ((unsigned long long)key << 32) | (unsigned)i;
        }
        if (!all_eq) {
            unsigned base_eq = 0;
            for (long long i0 = 0; i0 < a.n_db && base_eq < need; i0 += kTopThreads) {
                const long long i = i0 + tid;
                const unsigned eq = i < a.n_db && keys[i] == prefix;
                const unsigned pe = block_excl_scan(eq, warp_tot, &s_total);
                if (eq && base_eq + pe < need)
                    sel[n_less + base_eq + pe] = ((unsigned long long)prefix << 32) | (unsigned)i;
                base_eq += s_total;
                __syncthreads();
            }
        }
        __syncthreads();
    }
    bitonic_sort_1024(sel);   // packed (distance bits, index) ascending; unused slots = ~0
    if (tid < a.k) {
        const bool ok = (unsigned)tid < k;
        a.top_idx[(long long)q * a.k + tid] = ok ? (long long)(unsigned)(sel[tid] & 0xffffffffull) : -1;
        a.top_dist[(long long)q * a.k + tid] = ok ? __uint_as_float((unsigned)(sel[tid] >> 32)) : INFINITY;
    }
    if (tid == 0) a.top_count[q] = (int)k;
}

// ---- rank: every row of the database in order -----------------------------------------------
// nsc_wasserstein_rank orders each query's distances with a stable LSD radix sort of the 32-bit
// patterns, the row index riding along as payload (distances are >= 0, +inf or NaN, so unsigned
// order is numeric order with NaN last). A tile of kRankTile keys never straddles two queries.
// Every pass is three launches:
//   rank_hist_kernel     digit counts of each tile
//   rank_scan_kernel     one CTA per query: exclusive scan of its counts, digit-major, which gives
//                        every (digit, tile) its first output position
//   rank_scatter_kernel  stable rank inside the tile (per-warp digit counters, match_any within a
//                        round of 32 keys), then the scatter of keys and rows
// The first pass reads the keys straight from the distances (row = position); rows enter in index
// order and every pass is stable, so equal distances stay in row order. The last pass writes only
// the ranks below min(top_k, finite keys) into the outputs, its scan the padding and the count.
#ifndef NSC_RANK_BITS
#define NSC_RANK_BITS 8                // 8 or 11: DESIGN.md §7 has the measurement
#endif
constexpr int kRankBits = NSC_RANK_BITS;
static_assert(kRankBits == 8 || kRankBits == 11, "digit width");
constexpr int kRadix = 1 << kRankBits;
constexpr int kRankPasses = (32 + kRankBits - 1) / kRankBits;
constexpr int kRankThreads = 256;
constexpr int kRankWarps = kRankThreads / 32;
constexpr int kRankItems = 16;                          // keys per thread
constexpr long long kRankTile = kRankThreads * kRankItems;
constexpr int kScanThreads = 1024;
constexpr int kScanItems = 8;
constexpr unsigned kInfBits = 0x7f800000u;
constexpr int kMaxGridY = 65535;                        // queries per launch

struct RankArgs {
    const unsigned* src_keys;   // Q x N; the first pass reads the distances' bits
    const unsigned* src_rows;   // Q x N; null on the first pass (row = position)
    unsigned* dst_keys;         // Q x N; unused on the last pass
    unsigned* dst_rows;
    unsigned* hist;             // Q x kRadix x n_tiles: counts, then first output positions
    unsigned* finite;           // Q x n_tiles: finite keys per tile (first pass)
    unsigned* n_finite;         // Q
    long long n_db;
    long long k;
    long long* top_idx;         // Q x k
    float* top_dist;
    int* top_count;
    int q0;                     // first query of the launch
    int n_tiles;
    int shift;
    int first, last;
};

__global__ void __launch_bounds__(kRankThreads)
rank_hist_kernel(const __grid_constant__ RankArgs a) {
    __shared__ unsigned h[kRadix];
    __shared__ unsigned s_fin;
    const int lane = threadIdx.x & 31;
    const long long q = a.q0 + (long long)blockIdx.y, lo = (long long)blockIdx.x * kRankTile;
    const int n = (int)(a.n_db - lo < kRankTile ? a.n_db - lo : kRankTile);
    for (int i = threadIdx.x; i < kRadix; i += kRankThreads) h[i] = 0;
    if (threadIdx.x == 0) s_fin = 0;
    const unsigned* keys = a.src_keys + q * a.n_db + lo;
    unsigned key[kRankItems];
#pragma unroll
    for (int i = 0; i < kRankItems; ++i) {
        const int e = i * kRankThreads + threadIdx.x;
        key[i] = e < n ? keys[e] : 0u;
    }
    __syncthreads();
    unsigned fin = 0;
#pragma unroll
    for (int i = 0; i < kRankItems; ++i) {
        const bool act = i * kRankThreads + (int)threadIdx.x < n;
        const unsigned amask = __ballot_sync(0xffffffffu, act);
        if (act) {
            const unsigned d = (key[i] >> a.shift) & (kRadix - 1);
            const unsigned peers = __match_any_sync(amask, d);      // ties share digits: one atomic per digit
            if (lane == __ffs(peers) - 1) atomicAdd(&h[d], (unsigned)__popc(peers));
            fin += key[i] < kInfBits;
        }
    }
    if (a.first) {
        fin = __reduce_add_sync(0xffffffffu, fin);
        if (lane == 0 && fin) atomicAdd(&s_fin, fin);
    }
    __syncthreads();
    unsigned* out = a.hist + q * kRadix * a.n_tiles + blockIdx.x;
    for (int d = threadIdx.x; d < kRadix; d += kRankThreads) out[(long long)d * a.n_tiles] = h[d];
    if (a.first && threadIdx.x == 0) a.finite[q * a.n_tiles + blockIdx.x] = s_fin;
}

__global__ void __launch_bounds__(kScanThreads)
rank_scan_kernel(const __grid_constant__ RankArgs a) {
    __shared__ __align__(16) unsigned s[kScanThreads * kScanItems];
    __shared__ unsigned warp_tot[32];
    __shared__ unsigned s_total, s_fin;
    const int tid = threadIdx.x;
    const long long q = a.q0 + (long long)blockIdx.x;
    const long long n = (long long)kRadix * a.n_tiles;
    unsigned* h = a.hist + q * n;
    unsigned carry = 0;
    for (long long base = 0; base < n; base += kScanThreads * kScanItems) {
        for (int i = tid; i < kScanThreads * kScanItems; i += kScanThreads) s[i] = base + i < n ? h[base + i] : 0u;
        __syncthreads();
        uint4* s4 = reinterpret_cast<uint4*>(s) + tid * (kScanItems / 4);
        const uint4 v0 = s4[0], v1 = s4[1];
        const unsigned v[kScanItems] = {v0.x, v0.y, v0.z, v0.w, v1.x, v1.y, v1.z, v1.w};
        unsigned sum = 0;
#pragma unroll
        for (int j = 0; j < kScanItems; ++j) sum += v[j];
        unsigned run = block_excl_scan(sum, warp_tot, &s_total) + carry;     // ends with a barrier
        unsigned o[kScanItems];
#pragma unroll
        for (int j = 0; j < kScanItems; ++j) { o[j] = run; run += v[j]; }
        s4[0] = make_uint4(o[0], o[1], o[2], o[3]);
        s4[1] = make_uint4(o[4], o[5], o[6], o[7]);
        carry += s_total;
        __syncthreads();
        for (int i = tid; i < kScanThreads * kScanItems; i += kScanThreads)
            if (base + i < n) h[base + i] = s[i];
        __syncthreads();
    }
    if (a.first) {
        unsigned f = 0;
        for (int t = tid; t < a.n_tiles; t += kScanThreads) f += a.finite[q * a.n_tiles + t];
        f = block_excl_scan(f, warp_tot, &s_total);
        if (tid == 0) { s_fin = s_total; a.n_finite[q] = s_total; }
        __syncthreads();
    }
    if (a.last) {
        const long long nf = a.first ? s_fin : a.n_finite[q];
        const long long c = a.k < nf ? a.k : nf;
        for (long long r = c + tid; r < a.k; r += kScanThreads) {
            a.top_idx[q * a.k + r] = -1;
            a.top_dist[q * a.k + r] = INFINITY;
        }
        if (tid == 0) a.top_count[q] = (int)c;
    }
}

__global__ void __launch_bounds__(kRankThreads)
rank_scatter_kernel(const __grid_constant__ RankArgs a) {
    extern __shared__ unsigned rank_cnt[];              // kRankWarps x kRadix
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long long q = a.q0 + (long long)blockIdx.y, lo = (long long)blockIdx.x * kRankTile;
    const int n = (int)(a.n_db - lo < kRankTile ? a.n_db - lo : kRankTile);
    unsigned* wc = rank_cnt + warp * kRadix;
    for (int i = lane; i < kRadix; i += 32) wc[i] = 0;
    // warp w owns the tile's keys [w0, w0 + 32 * kRankItems), 32 consecutive ones per round
    const int w0 = warp * 32 * kRankItems;
    const unsigned* keys = a.src_keys + q * a.n_db + lo;
    const unsigned* rows = a.src_rows ? a.src_rows + q * a.n_db + lo : nullptr;
    unsigned key[kRankItems], row[kRankItems], pos[kRankItems];
#pragma unroll
    for (int i = 0; i < kRankItems; ++i) {
        const int e = w0 + i * 32 + lane;
        key[i] = e < n ? keys[e] : 0u;
        row[i] = e < n ? (rows ? rows[e] : (unsigned)(lo + e)) : 0u;
    }
    __syncwarp();
    // rank among the warp's keys of the same digit, in position order
#pragma unroll
    for (int i = 0; i < kRankItems; ++i) {
        const bool act = w0 + i * 32 + lane < n;
        const unsigned amask = __ballot_sync(0xffffffffu, act);
        if (act) {
            const unsigned d = (key[i] >> a.shift) & (kRadix - 1);
            const unsigned peers = __match_any_sync(amask, d);
            const int leader = __ffs(peers) - 1;
            unsigned base = 0;
            if (lane == leader) {
                base = wc[d];
                wc[d] = base + __popc(peers);
            }
            pos[i] = __shfl_sync(amask, base, leader) + __popc(peers & ((1u << lane) - 1));
        }
        __syncwarp();
    }
    __syncthreads();
    // each warp's first output position per digit: the tile's (rank_scan_kernel), then the lower warps'
    const unsigned* start = a.hist + q * kRadix * a.n_tiles + blockIdx.x;
    for (int d = threadIdx.x; d < kRadix; d += kRankThreads) {
        unsigned run = start[(long long)d * a.n_tiles];
#pragma unroll
        for (int w = 0; w < kRankWarps; ++w) {
            const unsigned c = rank_cnt[w * kRadix + d];
            rank_cnt[w * kRadix + d] = run;
            run += c;
        }
    }
    __syncthreads();
    if (!a.last) {
#pragma unroll
        for (int i = 0; i < kRankItems; ++i)
            if (w0 + i * 32 + lane < n) {
                const long long p = q * a.n_db + wc[(key[i] >> a.shift) & (kRadix - 1)] + pos[i];
                a.dst_keys[p] = key[i];
                a.dst_rows[p] = row[i];
            }
    } else {
        const long long nf = a.n_finite[q];
        const long long c = a.k < nf ? a.k : nf;
#pragma unroll
        for (int i = 0; i < kRankItems; ++i)
            if (w0 + i * 32 + lane < n) {
                const long long p = (long long)wc[(key[i] >> a.shift) & (kRadix - 1)] + pos[i];
                if (p < c) {
                    a.top_idx[q * a.k + p] = row[i];
                    a.top_dist[q * a.k + p] = __uint_as_float(key[i]);
                }
            }
    }
}

int sm_count(int* sms) {
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return record_cuda(e);
    e = cudaDeviceGetAttribute(sms, cudaDevAttrMultiProcessorCount, dev);
    return e == cudaSuccess ? NSC_OK : record_cuda(e);
}

// Workspace of the rank, in 256-byte aligned regions: keys and rows twice (ping-pong), the tile
// counts, the finite keys per tile and per query. size = SIZE_MAX where that does not fit a size_t.
struct RankLayout {
    size_t keys[2], rows[2], hist, finite, n_finite, size;
};

RankLayout rank_layout(long long n_queries, long long n_db) {
    RankLayout l{};
    const unsigned __int128 tiles = (n_db + kRankTile - 1) / kRankTile;
    const unsigned __int128 sizes[7] = {(unsigned __int128)n_queries * n_db * 4, (unsigned __int128)n_queries * n_db * 4,
                                        (unsigned __int128)n_queries * n_db * 4, (unsigned __int128)n_queries * n_db * 4,
                                        (unsigned __int128)n_queries * kRadix * tiles * 4,
                                        (unsigned __int128)n_queries * tiles * 4, (unsigned __int128)n_queries * 4};
    size_t* at[7] = {&l.keys[0], &l.rows[0], &l.keys[1], &l.rows[1], &l.hist, &l.finite, &l.n_finite};
    unsigned __int128 off = 0;
    for (int i = 0; i < 7; ++i) {
        *at[i] = (size_t)off;
        off += (sizes[i] + 255) / 256 * 256;
    }
    l.size = off > (unsigned __int128)SIZE_MAX ? SIZE_MAX : (size_t)off;
    return l;
}

}  // namespace

}  // namespace nsc

using namespace nsc;

extern "C" {

int nsc_wasserstein_cdf(const float* d_hists, int64_t n_rows, int n_bins, float epsilon,
                        float* d_cdfs, void* stream) {
    if (n_rows < 0) return NSC_ERR_BAD_COUNT;
    if (n_bins < 1 || n_bins > 32 * kMaxPerLane) return NSC_ERR_BAD_PARAMS;
    if (n_rows == 0) return NSC_OK;
    if (!d_hists || !d_cdfs) return NSC_ERR_NULL_POINTER;
    int sms = 0;
    int st = sm_count(&sms);
    if (st != NSC_OK) return st;
    const int padded = ((n_bins + 31) / 32) * 32;
    const size_t smem = (size_t)kRWarps * padded * 4;
    long long grid = (n_rows + kRWarps - 1) / kRWarps;
    if (grid > (long long)sms * 8) grid = (long long)sms * 8;
    cdf_rows_kernel<<<(int)grid, kRThreads, smem, (cudaStream_t)stream>>>(d_hists, n_rows, n_bins,
                                                                         epsilon, d_cdfs);
    return record_cuda(cudaGetLastError());
}

int nsc_wasserstein_cdf_u16(const uint16_t* d_rows, int64_t n_rows, int n_bins, uint16_t* d_cdf16, void* stream) {
    if (n_rows < 0) return NSC_ERR_BAD_COUNT;
    if (n_bins < 1 || n_bins > 32 * kMaxPerLane) return NSC_ERR_BAD_PARAMS;
    if (n_rows == 0) return NSC_OK;
    if (!d_rows || !d_cdf16) return NSC_ERR_NULL_POINTER;
    int sms = 0;
    int st = sm_count(&sms);
    if (st != NSC_OK) return st;
    const int padded = ((n_bins + 31) / 32) * 32;
    const size_t smem = (size_t)kRWarps * padded * 2;
    long long grid = (n_rows + kRWarps - 1) / kRWarps;
    if (grid > (long long)sms * 8) grid = (long long)sms * 8;
    cdf16_rows_kernel<<<(int)grid, kRThreads, smem, (cudaStream_t)stream>>>(
        reinterpret_cast<const unsigned short*>(d_rows), n_rows, n_bins, reinterpret_cast<unsigned short*>(d_cdf16));
    return record_cuda(cudaGetLastError());
}

constexpr int kMaxDistGrid = 1024;     // CTAs of the distance pass (bounds the warp-minima rows of the workspace)

size_t nsc_wasserstein_workspace_bytes(int n_queries) {
    if (n_queries < 0) return 0;
    const size_t per_query = 16 + (size_t)kSelCap * 8 + (size_t)kMaxDistGrid * kRWarps * 8;
    return (size_t)n_queries * per_query + 256;
}

size_t nsc_wasserstein_rank_workspace_bytes(int n_queries, int64_t n_db) {
    if (n_queries < 0 || n_db < 0 || n_db >= (1ll << 32)) return 0;
    return rank_layout(n_queries, n_db).size;
}

}  // extern "C"

namespace {

// nsc_wasserstein_query and nsc_wasserstein_query_u16: T is the element type of the database rows
template <typename T>
int wasserstein_query(const float* d_query_hists, int n_queries, const T* d_db_cdfs,
                      int64_t n_db, int n_bins, float epsilon, const double* d_db_xyz,
                      const double* d_query_xyz, double min_spatial_distance,
                      float* d_distances, int top_k, int64_t* d_top_idx, float* d_top_dist,
                      int32_t* d_top_count, void* d_workspace, size_t workspace_bytes, void* stream) {
    if (n_queries < 0 || n_db < 0 || top_k < 0) return NSC_ERR_BAD_COUNT;
    if (n_bins < 1 || n_bins > 32 * kMaxPerLane || top_k > kTopThreads) return NSC_ERR_BAD_PARAMS;
    if (n_db >= (1ll << 32)) return NSC_ERR_BAD_COUNT;
    if (n_queries == 0) return NSC_OK;
    if (!d_query_hists || !d_distances) return NSC_ERR_NULL_POINTER;
    if (n_db > 0 && !d_db_cdfs) return NSC_ERR_NULL_POINTER;
    if (top_k > 0 && (!d_top_idx || !d_top_dist || !d_top_count)) return NSC_ERR_NULL_POINTER;
    if ((d_db_xyz == nullptr) != (d_query_xyz == nullptr)) return NSC_ERR_NULL_POINTER;
    // the many-CTA selection needs the workspace; without one (or for large k) one CTA per query selects
    const bool fused_select = top_k > 0 && top_k <= kSelMaxK && n_db > 0 && d_workspace &&
                              workspace_bytes >= nsc_wasserstein_workspace_bytes(n_queries);
    int* counters = (int*)d_workspace;
    unsigned long long* cand = (unsigned long long*)((char*)d_workspace + (((size_t)n_queries * 16 + 255) & ~(size_t)255));
    unsigned long long* warp_min = cand + (size_t)n_queries * kSelCap;
    cudaStream_t s = (cudaStream_t)stream;
    int sms = 0;
    int st = sm_count(&sms);
    if (st != NSC_OK) return st;
    int n_min = 0;
    if (n_db > 0) {
        void (*kern)(const QueryArgs) = nullptr;
        int per = (n_bins + 31) / 32;
        per = per <= 8 ? 8 : per <= 16 ? 16 : per <= 25 ? 25 : 32;
        // one grid for every group of queries (sized for the largest group), so that the rows of
        // warp minima have one length
        const int q_max = n_queries < kMaxQueries ? n_queries : kMaxQueries;
        int smem_optin = 0, dev = 0;
        cudaError_t e = cudaGetDevice(&dev);
        if (e == cudaSuccess) e = cudaDeviceGetAttribute(&smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
        if (e != cudaSuccess) return record_cuda(e);
        auto smem_for = [&](int nq, int stages) {
            return (size_t)nq * per * 32 * 4 + (size_t)kRWarps * stages * per * 32 * sizeof(T);
        };
        const int stages = 2 * (smem_for(q_max, 4) + 1024) <= (size_t)smem_optin ? 4 : 3;   // keep two CTAs per SM
        if (stages == 4)
            kern = per == 8 ? wasserstein_kernel<T, 8, 4> : per == 16 ? wasserstein_kernel<T, 16, 4>
                   : per == 25 ? wasserstein_kernel<T, 25, 4> : wasserstein_kernel<T, 32, 4>;
        else
            kern = per == 8 ? wasserstein_kernel<T, 8, 3> : per == 16 ? wasserstein_kernel<T, 16, 3>
                   : per == 25 ? wasserstein_kernel<T, 25, 3> : wasserstein_kernel<T, 32, 3>;
        const size_t smem_max = smem_for(q_max, stages);
        e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_max);
        if (e != cudaSuccess) return record_cuda(e);
        int per_sm = 0;
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kRThreads, smem_max);
        if (e != cudaSuccess) return record_cuda(e);
        if (per_sm < 1) return NSC_ERR_BAD_PARAMS;
        long long grid = (n_db + kRWarps - 1) / kRWarps;
        if (grid > (long long)sms * per_sm) grid = (long long)sms * per_sm;
        if (grid > kMaxDistGrid) grid = kMaxDistGrid;
        n_min = (int)grid * kRWarps;
        for (int q0 = 0; q0 < n_queries; q0 += kMaxQueries) {
            QueryArgs a;
            a.n_queries = n_queries - q0 < kMaxQueries ? n_queries - q0 : kMaxQueries;
            a.queries = d_query_hists + (size_t)q0 * n_bins;
            a.db_cdfs = d_db_cdfs;
            a.db_xyz = d_db_xyz;
            a.query_xyz = d_query_xyz ? d_query_xyz + 3 * (size_t)q0 : nullptr;
            a.min_dist = min_spatial_distance;
            a.distances = d_distances + (size_t)q0 * n_db;
            a.warp_min = fused_select ? warp_min + (size_t)q0 * n_min : nullptr;
            a.n_db = n_db;
            a.n_bins = n_bins;
            a.eps = epsilon;
            kern<<<(int)grid, kRThreads, smem_for(a.n_queries, stages), s>>>(a);
            e = cudaGetLastError();
            if (e != cudaSuccess) return record_cuda(e);
        }
    }
    if (top_k > 0) {
        TopkArgs t;
        t.distances = d_distances;
        t.n_db = n_db;
        t.k = top_k;
        t.top_idx = (long long*)d_top_idx;
        t.top_dist = d_top_dist;
        t.top_count = d_top_count;
        if (fused_select) {
            SelectArgs sa;
            sa.distances = d_distances;
            sa.warp_min = warp_min;
            sa.n_min = n_min;
            sa.n_db = n_db;
            sa.k = top_k;
            sa.counters = counters;
            sa.cand = cand;
            sa.top_idx = (long long*)d_top_idx;
            sa.top_dist = d_top_dist;
            sa.top_count = d_top_count;
            long long per_q = (n_db + 4 * kSelThreads - 1) / (4 * kSelThreads);      // ~1024 rows per CTA
            const int ctas = (int)(per_q < 1 ? 1 : per_q > kSelCtas ? kSelCtas : per_q);
            // programmatic dependent launch: the grid is set up while the distance pass drains
            cudaLaunchConfig_t cfg = {};
            cfg.gridDim = dim3(ctas, n_queries);
            cfg.blockDim = dim3(kSelThreads);
            cfg.dynamicSmemBytes = 0;
            cfg.stream = s;
            cudaLaunchAttribute attr[1];
            attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
            attr[0].val.programmaticStreamSerializationAllowed = 1;
            cfg.attrs = attr;
            cfg.numAttrs = 1;
            return record_cuda(cudaLaunchKernelEx(&cfg, select_kernel, sa));
        }
        topk_kernel<<<n_queries, kTopThreads, 0, s>>>(t);
        return record_cuda(cudaGetLastError());
    }
    return NSC_OK;
}

// nsc_wasserstein_rank and nsc_wasserstein_rank_u16: the distance pass of wasserstein_query, then
// the radix sort of every query's distances
template <typename T>
int wasserstein_rank(const float* d_query_hists, int n_queries, const T* d_db_cdfs, int64_t n_db, int n_bins,
                     float epsilon, const double* d_db_xyz, const double* d_query_xyz, double min_spatial_distance,
                     float* d_distances, int64_t top_k, int64_t* d_top_idx, float* d_top_dist, int32_t* d_top_count,
                     void* d_workspace, size_t workspace_bytes, void* stream) {
    if (n_queries < 0 || n_db < 0 || n_db >= (1ll << 32) || top_k < 0) return NSC_ERR_BAD_COUNT;
    if (n_bins < 1 || n_bins > 32 * kMaxPerLane) return NSC_ERR_BAD_PARAMS;
    if (n_queries == 0) return NSC_OK;
    if (!d_query_hists || !d_distances) return NSC_ERR_NULL_POINTER;
    if (n_db > 0 && !d_db_cdfs) return NSC_ERR_NULL_POINTER;
    if (top_k > 0 && (!d_top_idx || !d_top_dist || !d_top_count)) return NSC_ERR_NULL_POINTER;
    if ((d_db_xyz == nullptr) != (d_query_xyz == nullptr)) return NSC_ERR_NULL_POINTER;
    const RankLayout l = rank_layout(n_queries, n_db);
    if (top_k > 0 && (!d_workspace || workspace_bytes < l.size)) return NSC_ERR_WORKSPACE;
    int st = wasserstein_query(d_query_hists, n_queries, d_db_cdfs, n_db, n_bins, epsilon, d_db_xyz, d_query_xyz,
                               min_spatial_distance, d_distances, 0, nullptr, nullptr, nullptr, nullptr, 0, stream);
    if (st != NSC_OK || top_k == 0) return st;
    cudaStream_t s = (cudaStream_t)stream;
    char* ws = static_cast<char*>(d_workspace);
    const size_t scatter_smem = (size_t)kRankWarps * kRadix * 4;
    if (scatter_smem > 48 * 1024) {
        const cudaError_t e = cudaFuncSetAttribute(rank_scatter_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                   (int)scatter_smem);
        if (e != cudaSuccess) return record_cuda(e);
    }
    RankArgs a{};
    a.hist = reinterpret_cast<unsigned*>(ws + l.hist);
    a.finite = reinterpret_cast<unsigned*>(ws + l.finite);
    a.n_finite = reinterpret_cast<unsigned*>(ws + l.n_finite);
    a.n_db = n_db;
    a.k = top_k;
    a.top_idx = (long long*)d_top_idx;
    a.top_dist = d_top_dist;
    a.top_count = d_top_count;
    a.n_tiles = (int)((n_db + kRankTile - 1) / kRankTile);
    // no rows (n_db = 0): one scan launch, which writes the padding and the counts
    const int passes = n_db > 0 ? kRankPasses : 1;
    for (int q0 = 0; q0 < n_queries; q0 += kMaxGridY) {
        const int nq = n_queries - q0 < kMaxGridY ? n_queries - q0 : kMaxGridY;
        a.q0 = q0;
        for (int p = 0; p < passes; ++p) {
            a.shift = p * kRankBits;
            a.first = p == 0;
            a.last = p == passes - 1;
            a.src_keys = p == 0 ? reinterpret_cast<const unsigned*>(d_distances)
                                : reinterpret_cast<const unsigned*>(ws + l.keys[(p - 1) & 1]);
            a.src_rows = p == 0 ? nullptr : reinterpret_cast<const unsigned*>(ws + l.rows[(p - 1) & 1]);
            a.dst_keys = reinterpret_cast<unsigned*>(ws + l.keys[p & 1]);
            a.dst_rows = reinterpret_cast<unsigned*>(ws + l.rows[p & 1]);
            const dim3 tiles(a.n_tiles, nq);
            if (n_db > 0) rank_hist_kernel<<<tiles, kRankThreads, 0, s>>>(a);
            rank_scan_kernel<<<nq, kScanThreads, 0, s>>>(a);
            if (n_db > 0) rank_scatter_kernel<<<tiles, kRankThreads, scatter_smem, s>>>(a);
            const cudaError_t e = cudaGetLastError();
            if (e != cudaSuccess) return record_cuda(e);
        }
    }
    return NSC_OK;
}

}  // namespace

extern "C" {

int nsc_wasserstein_query(const float* d_query_hists, int n_queries, const float* d_db_cdfs,
                          int64_t n_db, int n_bins, float epsilon, const double* d_db_xyz,
                          const double* d_query_xyz, double min_spatial_distance,
                          float* d_distances, int top_k, int64_t* d_top_idx, float* d_top_dist,
                          int32_t* d_top_count, void* d_workspace, size_t workspace_bytes, void* stream) {
    return wasserstein_query(d_query_hists, n_queries, d_db_cdfs, n_db, n_bins, epsilon, d_db_xyz, d_query_xyz,
                             min_spatial_distance, d_distances, top_k, d_top_idx, d_top_dist, d_top_count,
                             d_workspace, workspace_bytes, stream);
}

int nsc_wasserstein_query_u16(const float* d_query_hists, int n_queries, const uint16_t* d_db_cdf16,
                              int64_t n_db, int n_bins, float epsilon, const double* d_db_xyz,
                              const double* d_query_xyz, double min_spatial_distance,
                              float* d_distances, int top_k, int64_t* d_top_idx, float* d_top_dist,
                              int32_t* d_top_count, void* d_workspace, size_t workspace_bytes, void* stream) {
    return wasserstein_query(d_query_hists, n_queries, reinterpret_cast<const unsigned short*>(d_db_cdf16), n_db,
                             n_bins, epsilon, d_db_xyz, d_query_xyz, min_spatial_distance, d_distances, top_k,
                             d_top_idx, d_top_dist, d_top_count, d_workspace, workspace_bytes, stream);
}

int nsc_wasserstein_rank(const float* d_query_hists, int n_queries, const float* d_db_cdfs, int64_t n_db,
                         int n_bins, float epsilon, const double* d_db_xyz, const double* d_query_xyz,
                         double min_spatial_distance, float* d_distances, int64_t top_k, int64_t* d_top_idx,
                         float* d_top_dist, int32_t* d_top_count, void* d_workspace, size_t workspace_bytes,
                         void* stream) {
    return wasserstein_rank(d_query_hists, n_queries, d_db_cdfs, n_db, n_bins, epsilon, d_db_xyz, d_query_xyz,
                            min_spatial_distance, d_distances, top_k, d_top_idx, d_top_dist, d_top_count,
                            d_workspace, workspace_bytes, stream);
}

int nsc_wasserstein_rank_u16(const float* d_query_hists, int n_queries, const uint16_t* d_db_cdf16, int64_t n_db,
                             int n_bins, float epsilon, const double* d_db_xyz, const double* d_query_xyz,
                             double min_spatial_distance, float* d_distances, int64_t top_k, int64_t* d_top_idx,
                             float* d_top_dist, int32_t* d_top_count, void* d_workspace, size_t workspace_bytes,
                             void* stream) {
    return wasserstein_rank(d_query_hists, n_queries, reinterpret_cast<const unsigned short*>(d_db_cdf16), n_db,
                            n_bins, epsilon, d_db_xyz, d_query_xyz, min_spatial_distance, d_distances, top_k,
                            d_top_idx, d_top_dist, d_top_count, d_workspace, workspace_bytes, stream);
}

}  // extern "C"
