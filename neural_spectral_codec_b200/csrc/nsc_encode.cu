// Fused encode kernels: points -> min-range image (shared memory) -> interpolation -> spectrum
// -> descriptor. Persistent CTAs pull whole scans from a work counter, so the range image, its
// interpolation and the spectrum never leave shared memory: HBM traffic is the 16 B per point
// and the descriptor. The kernels share the per-point and the tail code:
//   encode_points_ws_kernel     the hot one (large batches of 16-byte points): one 1024-thread CTA
//                               per SM, a TMA producer thread, 24 stream warps, 7 tail warps, two
//                               images; see the comment above it
//   encode_points_kernel        generic: 2 x 512-thread CTAs per SM, every warp streams and then runs
//                               the tail (12-byte points, images too large to keep twice)
//   encode_points_split_kernel  small batches: one thread-block cluster per scan
//   encode_points_tall_kernel, encode_points_tall_split_kernel
//                               the generic and the cluster kernel for images of 65..128 rows: one
//                               image per SM, points straight into registers, pooled before the FFT
#include <stdlib.h>

#include <mutex>
#include <utility>
#include <vector>

#include <cooperative_groups.h>

#include "nsc_point.h"
#include "nsc_tail.cuh"

namespace nsc {

namespace {

constexpr int kUnroll = 4;   // points in flight per thread (12-byte points, plain loads)
#ifndef NSC_TALL_PTS
#define NSC_TALL_PTS 12
#endif
constexpr int kTallPts = NSC_TALL_PTS;   // 16-byte points in flight per thread of a tall kernel (even)
static_assert(kTallPts % 2 == 0, "the tall feed classifies points in pairs");

// EncodeOutputs as the kernels read it: the peer pointers by value, and with rows_q the quantiser's
// pairwise-sum plan for rows of D elements (nsc_quantize.cuh), built once per launch on the host.
struct KernelOutputs {
    float* rows;
    unsigned short* rows_q;
    float q_eps;
    SumPlan q_plan;
    float* images;
    int stage;
    PeerOut peers;
    __device__ bool descriptors() const { return rows || rows_q || peers.n > 0; }
    __device__ RowDest row(int scan, int D) const {
        RowDest d;
        d.out = rows ? rows + (long long)scan * D : nullptr;
        d.peers = &peers;
        d.peer_row = peers.row0 + scan;
        d.out_q = rows_q ? rows_q + (long long)scan * D : nullptr;
        d.q_eps = q_eps;
        d.plan = &q_plan;
        return d;
    }
};

struct EncodeArgs {
    const float* points;
    const long long* offsets;
    long long origin;
    int n_scans;
    KernelOutputs out;
    unsigned* counter;
    // warp-specialised kernel: the last n_scans - n_whole scans are handed out in `parts` pieces
    // each, so that the final, partial wave of the grid is spread over all CTAs (see launch_encode)
    int n_whole, parts, n_units;
    unsigned* part_arrive;       // one counter per split scan (zero before the launch)
    unsigned* part_image;        // one E x 361 key image per split scan (0xffffffff before the launch)
};

// The point layout picks the feed of the generic and cluster kernels: 16-byte points stream through
// the per-thread cp.async ring, 12-byte points take plain loads (cp.async needs 16-byte sources).
// The warp-specialised kernel has its own whole-stage TMA ring. Feeds measured and dropped: DESIGN.md §4.
__host__ __device__ constexpr int ring_bytes(int stride) { return stride == 4 ? kCpRingBytes : 0; }

// ---- mbarrier / bulk-copy (TMA) primitives ------------------------------------------------
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(bar), "r"(parity)
        : "memory");
}
// The same with an L2 cache policy: the points are read exactly once, so they are marked
// evict-first and do not push the (dirty) descriptor lines of this and the peer GPUs out of L2
// while the kernel runs -- write-backs trickling into the read stream cost far more DRAM time
// than their bytes (tools/peer_store_cost.py).
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ void bulk_copy_g2s_hint(uint32_t dst, const void* src, uint32_t bytes,
                                                   uint32_t bar, uint64_t pol) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;"
        ::"r"(dst), "l"(src), "r"(bytes), "r"(bar), "l"(pol)
        : "memory");
}
// global -> shared bulk copy, completion counted in bytes on an mbarrier.
__device__ __forceinline__ void bulk_copy_g2s(uint32_t dst, const void* src, uint32_t bytes,
                                              uint32_t bar) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
        ::"r"(dst), "l"(src), "r"(bytes), "r"(bar)
        : "memory");
}
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return (uint32_t)__cvta_generic_to_shared(p);
}
// 16-byte asynchronous global -> shared copy (SASS LDGSTS), L2-only caching.
__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() {
    asm volatile("cp.async.commit_group;" ::: "memory");
}
template <int N>
__device__ __forceinline__ void cp_async_wait() {
    asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ float4 lds128(uint32_t addr) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
                 : "r"(addr)
                 : "memory");
    return v;
}

// Per-pixel min of the key (bits of s). img_biased = shared address of the image minus the
// floor bias of row and column (nsc_point.h), so the address is two integer ops. A plain read
// first: after the first few hits most points are not a new minimum, and a stale read can only
// cause a redundant atomic, never a missed one. No branch: the atomic is predicated.
__device__ __forceinline__ void scatter_min(uint32_t img_biased, uint32_t row_b, uint32_t col_b,
                                            uint32_t key) {
    const uint32_t addr = row_b * (uint32_t)(kPitch * 4) + (col_b * 4u + img_biased);
#ifdef NSC_DEBUG_BOUNDS
    // self-check build (compute-sanitizer is closed on this pool): the pixel must lie inside the image
    {
        const uint32_t r = row_b - kFloorBias, c = col_b - kFloorBias;
        if (r >= (uint32_t)NSC_MAX_ELEVATION || c > (uint32_t)kAz ||
            addr - (img_biased + kFloorBias * (uint32_t)(kPitch * 4 + 4)) != (r * kPitch + c) * 4u)
            __trap();
    }
#endif
    uint32_t cur;
    asm("ld.shared.u32 %0, [%1];" : "=r"(cur) : "r"(addr));
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.lt.u32 p, %1, %2;\n"
        "@p red.shared.min.u32 [%0], %1;\n"
        "}\n" ::"r"(addr), "r"(key), "r"(cur)
        : "memory");
}

template <int ROWMODE, int ROWS = kShortRows>
__device__ __forceinline__ void project_point(float x, float y, float z, const DeviceParams& dp,
                                              uint32_t img_biased, bool in_range = true) {
    uint32_t row_b, col_b;
    uint32_t key = classify<ROWS>(x, y, z, dp, ROWMODE, row_b, col_b);
    if (!in_range) key = 0xffffffffu;
    scatter_min(img_biased, row_b, col_b, key);
}

// Two points through the packed FP32 pipe (classify2, nsc_point.h); same bits as two project_point calls.
template <int ROWMODE, int ROWS = kShortRows>
__device__ __forceinline__ void project_pair(const float4& a, const float4& b, const DeviceParams& dp,
                                             uint32_t img_biased, bool in_a = true, bool in_b = true) {
    uint32_t ka, ra, ca, kb, rb, cb;
    classify2<ROWS>(a.x, a.y, a.z, b.x, b.y, b.z, dp, ROWMODE, ka, ra, ca, kb, rb, cb);
    if (!in_a) ka = 0xffffffffu;
    if (!in_b) kb = 0xffffffffu;
    scatter_min(img_biased, ra, ca, ka);
    scatter_min(img_biased, rb, cb, kb);
}

// Point pass over points [beg, beg + n) of the concatenated buffer: every kept point lowers the
// key of its pixel in the shared-memory min image. CTA-collective (no barrier inside). ROWS: the
// row capacity of the kernel; the tall kernels (ROWS > kShortRows) keep no ring.
template <int STRIDE, int ROWMODE, int ROWS = kShortRows>
__device__ __forceinline__ void point_pass(const float* __restrict__ points, long long beg, int n,
                                           const DeviceParams& dp, uint32_t img_biased,
                                           unsigned char* ring) {
    const int tid = threadIdx.x;
    if (STRIDE == 4 && ROWS > kShortRows) {
        // Tall kernels: the image leaves no room for a ring, so each thread keeps kTallPts
        // 16-byte points in flight in registers (LDG.128, evict-first); points past the end are
        // NaN, which never lowers a key (classify). 12 points: 1.13 x the rate of 8, 1.53 x that of 4
        // (profiles/r3d_tall_image_cost.txt); 16 would not fit 128 registers.
        const float4* gp = reinterpret_cast<const float4*>(points) + beg + tid;
        const float4 nan4 = make_float4(NAN, NAN, NAN, NAN);
        for (int base = 0; base < n; base += kThreads * kTallPts) {
            float4 v[kTallPts];
#pragma unroll
            for (int u = 0; u < kTallPts; ++u) v[u] = base + u * kThreads + tid < n ? __ldcs(gp + base + u * kThreads) : nan4;
#pragma unroll
            for (int u = 0; u < kTallPts; u += 2) project_pair<ROWMODE, ROWS>(v[u], v[u + 1], dp, img_biased);
        }
    } else if (STRIDE == 4) {
        // Each thread streams its own points through a private kCpDepth-deep shared-memory
        // ring of 16-byte cp.async copies. No cross-thread barrier is needed: a thread only
        // reads what it copied itself. Stage `it` holds points it*kStagePoints +
        // u*kThreads + tid, u < kCpPts; stage it + kCpDepth - 1 is issued before stage it
        // is consumed.
        constexpr int kStagePoints = kCpPts * kThreads;
        constexpr int kSlotBytes = kCpPts * kThreads * 16;
        const float4* gp = reinterpret_cast<const float4*>(points) + beg + tid;
        const uint32_t ring_t = smem_u32(ring) + tid * 16;
        const int n_full = n / kStagePoints;              // stages with every point in range
        const int n_iter = (n + kStagePoints - 1) / kStagePoints;
        auto issue_checked = [&](int it) {
            if (it < n_iter) {
#pragma unroll
                for (int u = 0; u < kCpPts; ++u) {
                    const int i = it * kStagePoints + u * kThreads;
                    if (i + tid < n)
                        cp_async16(ring_t + (it % kCpDepth) * kSlotBytes + u * (kThreads * 16), gp + i);
                }
            }
            cp_async_commit();
        };
#pragma unroll
        for (int d = 0; d < kCpDepth - 1; ++d) issue_checked(d);
        int it = 0;
        // Main trips: kCpDepth stages per trip so every ring slot is a compile-time offset and
        // no bounds checks remain (all stages touched are full).
        for (; it + 2 * kCpDepth - 2 < n_full; it += kCpDepth) {
            const float4* g = gp + (long long)it * kStagePoints;
#pragma unroll
            for (int s = 0; s < kCpDepth; ++s) {
#pragma unroll
                for (int u = 0; u < kCpPts; ++u)
                    cp_async16(ring_t + ((s + kCpDepth - 1) % kCpDepth) * kSlotBytes + u * (kThreads * 16),
                               g + (s + kCpDepth - 1) * kStagePoints + u * kThreads);
                cp_async_commit();
                cp_async_wait<kCpDepth - 1>();
                float4 v[kCpPts];
#pragma unroll
                for (int u = 0; u < kCpPts; ++u) v[u] = lds128(ring_t + s * kSlotBytes + u * (kThreads * 16));
#pragma unroll
                for (int u = 0; u < kCpPts; ++u)
                    project_point<ROWMODE>(v[u].x, v[u].y, v[u].z, dp, img_biased);
            }
        }
        // Remaining stages (the last few full ones and the partial one), bounds-checked.
        for (; it < n_iter; ++it) {
            issue_checked(it + kCpDepth - 1);
            cp_async_wait<kCpDepth - 1>();
#pragma unroll
            for (int u = 0; u < kCpPts; ++u) {
                const int i = it * kStagePoints + u * kThreads + tid;
                const float4 v = lds128(ring_t + (it % kCpDepth) * kSlotBytes + u * (kThreads * 16));
                project_point<ROWMODE>(v.x, v.y, v.z, dp, img_biased, i < n);
            }
        }
        cp_async_wait<0>();
    } else {
        const float* p = points + beg * 3;
        for (int base = 0; base < n; base += kThreads * kUnroll) {
            float x[kUnroll], y[kUnroll], z[kUnroll];
#pragma unroll
            for (int u = 0; u < kUnroll; ++u) {
                const int i = base + u * kThreads + tid;
                const bool in = i < n;
                x[u] = in ? __ldcs(p + 3 * (long long)i) : NAN;
                y[u] = in ? __ldcs(p + 3 * (long long)i + 1) : NAN;
                z[u] = in ? __ldcs(p + 3 * (long long)i + 2) : NAN;
            }
#pragma unroll
            for (int u = 0; u < kUnroll; ++u)
                project_point<ROWMODE, ROWS>(x[u], y[u], z[u], dp, img_biased);
        }
    }
}

#ifdef NSC_PHASE_TIMING
// Tuning build: thread 0 of every CTA accumulates the cycles it spends in each phase of a scan
// into counter[4 + 2*phase] (64-bit), phases: 0 init, 1 point pass, 2 rows_to_filled,
// 3 spectrum_and_bins, 4 normalise, 5..9 the sub-phases of spectrum_and_bins. Read back by
// tools/phase_timing.py.
#define NSC_PHASE(p)                                                                         \
    do {                                                                                     \
        if (threadIdx.x == 0) {                                                              \
            const long long now_ = clock64();                                                \
            atomicAdd(reinterpret_cast<unsigned long long*>(a.counter) + 2 + (p),            \
                      (unsigned long long)(now_ - phase_t0));                                \
            phase_t0 = now_;                                                                 \
        }                                                                                    \
    } while (0)
#else
#define NSC_PHASE(p) do { (void)phase_t0; } while (0)
#endif

// Everything after the scatter for one scan, run by the thread group G: keys -> ranges,
// interpolation, (optional) image output, spectrum, bins, normalisation, descriptor store.
// `mark(p)` is called between the phases: 2, 3 and 4 here, 5..9 inside spectrum_and_bins (9: the
// image is read for the last time). Returns false, right after the image output, when the launch
// writes no descriptors. ROWS > kShortRows (tall kernels): the image is pooled in place to its
// first T rows before the spectrum (pool_rows_in_place).
template <typename G, int ROWS = kShortRows, typename Mark>
__device__ __forceinline__ bool finish_scan(const EncodeArgs& a, const DeviceParams& dp,
                                            const TailSmem& S, int scan, Mark mark) {
    const KernelOutputs& o = a.out;
    const int D = dp.T * dp.n_bins;
    // bits of min s -> range = sqrt_rn(s); empty -> 0 (range_image.py:162,:214); masks; hole
    // interpolation; empty-row indirection
    float* stage0 = (o.images && o.stage == NSC_STAGE_PROJECTED) ? o.images + (long long)scan * dp.E * kAz : nullptr;
    rows_to_filled<true, G>(S, dp.E, dp.interpolate != 0, stage0, [&dp](uint32_t key) {
        return key_is_empty(key, dp) ? 0.0f : __fsqrt_rn(__uint_as_float(key));
    });
    if (o.images && o.stage == NSC_STAGE_INTERPOLATED) {
        for (int i = G::tid(); i < dp.E * kAz; i += G::kSize) {
            const int r = i / kAz, c = i - r * kAz;
            o.images[(long long)scan * dp.E * kAz + i] = S.img[S.src[r] * kPitch + c];
        }
    }
    mark(2);
    if (!o.descriptors()) return false;
    int rows = dp.E;
    if (ROWS > kShortRows) {
        pool_rows_in_place<G>(S, dp.E, dp.T);
        rows = dp.T;
    }
    spectrum_and_bins(S, dp, rows, mark, G());
    mark(3);
    normalise_and_store(S, dp, o.row(scan, D), G());
    mark(4);
    return true;
}

// The persistent loop of encode_points_kernel and encode_points_tall_kernel: every warp streams
// the scan's points and then runs its tail.
template <int STRIDE, int ROWMODE, int ROWS>
__device__ __forceinline__ void persistent_scans(const EncodeArgs& a, const DeviceParams& dp) {
    constexpr bool tall = ROWS > kShortRows;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ int s_scan;
    const SmemLayout L(dp.E, dp.T, dp.n_bins, tall ? 0 : ring_bytes(STRIDE), tall);
    const TailSmem S(smem_raw, L);
    uint32_t* img = reinterpret_cast<uint32_t*>(S.img);
    const uint32_t img_biased = smem_u32(img) - kFloorBias * (uint32_t)(kPitch * 4 + 4);
    const int tid = threadIdx.x;
    const int n_pix = dp.E * kPitch;

    init_tail_tables(S, dp);
    long long phase_t0 = clock64();
    // Thread 0 always holds the NEXT scan index: the atomic's round trip (~1 us) is issued at the
    // top of a scan and only consumed at the top of the following one.
    int next_scan = tid == 0 ? (int)atomicAdd(a.counter, 1u) : 0;

    for (;;) {
        __syncthreads();
        if (tid == 0) {
            s_scan = next_scan;
            if (next_scan < a.n_scans) next_scan = (int)atomicAdd(a.counter, 1u);
        }
        for (int i = tid; i < n_pix; i += kThreads) img[i] = kInfBits;
        __syncthreads();
        const int scan = s_scan;
        if (scan >= a.n_scans) break;
        const long long beg = a.offsets[scan] - a.origin;
        const int n = (int)(a.offsets[scan + 1] - a.offsets[scan]);
        NSC_PHASE(0);
        point_pass<STRIDE, ROWMODE, ROWS>(a.points, beg, n, dp, img_biased, smem_raw + L.ring_off);
        __syncthreads();
        NSC_PHASE(1);
        finish_scan<CtaGroup, ROWS>(a, dp, S, scan, [&](int p) { NSC_PHASE(p); });
    }
    if (tid == 0) wait_bulk_stores_done();      // descriptors leave shared memory before the CTA does
}

template <int STRIDE, int ROWMODE>
__global__ void __launch_bounds__(kThreads, kMinBlocks)
encode_points_kernel(const __grid_constant__ EncodeArgs a, const __grid_constant__ DeviceParams dp) {
    persistent_scans<STRIDE, ROWMODE, kShortRows>(a, dp);
}

// Images of more than 64 rows (up to NSC_MAX_ELEVATION): a 128 x 361 key image is 184 832 B, so
// one CTA per SM holds one image and no ring; the points come straight from global memory into
// registers (point_pass) and the tail pools the image before the spectrum (finish_scan).
template <int STRIDE, int ROWMODE>
__global__ void __launch_bounds__(kThreads, 1)
encode_points_tall_kernel(const __grid_constant__ EncodeArgs a, const __grid_constant__ DeviceParams dp) {
    persistent_scans<STRIDE, ROWMODE, NSC_MAX_ELEVATION>(a, dp);
}

// ---- warp-specialised persistent kernel ---------------------------------------------------
// One CTA of 1024 threads per SM, three roles:
//   producer  (1 thread of the last warp) walks the CTA's scans and keeps kWsDepth whole stages
//             of kWsStagePoints points in flight with cp.async.bulk (TMA, SASS UBLKCP), one copy
//             per stage, straight across scan boundaries. Measured with no arithmetic at all
//             (tools/feedbw.cu, profiles/r2c_feedbw.txt): 7.39 TB/s, against 6.93 TB/s for the
//             per-thread cp.async ring and 7.28 TB/s for plain LDG.128.
//   stream    (kWsStreamWarps warps) wait for a stage, read their points of it with LDS.128,
//             classify and scatter into one of two shared-memory images, hand the slot back.
//   tail      (kWsTailWarps warps) run ranges, interpolation, FFT, bins and normalisation of the
//             scan the stream warps finished before, from the other image.
// Synchronisation is by mbarriers only (plus the named barrier of the tail group):
//   slot_full[s]   the producer's expect_tx + the copy's bytes            -> stream warps wait
//   slot_empty[s]  one arrival per stream warp                            -> producer waits
//   img_full[b]    one arrival per stream warp when scan k is in image b  -> tail warps wait
//   img_empty[b]   one arrival per tail warp when image b is reset        -> stream warps wait
// Scan indices: the producer takes the CTA's k-th scan (block index for k = 0, the work counter
// afterwards) and publishes (k, scan, n_points) in mail[k & 3]; the other roles spin until the
// sequence number matches. It reuses an entry only when the tail has finished scan k - 4
// (tail_done), which every reader of that entry precedes. scan >= n_scans ends every role.
#ifndef NSC_WS_STREAM_WARPS
#define NSC_WS_STREAM_WARPS 24
#endif
#ifndef NSC_WS_TAIL_WARPS
#define NSC_WS_TAIL_WARPS 7
#endif
// Stage = 3 points per stream thread (36 KB per bulk copy), 4 stages: 144 KB ring. Measured
// (profiles/r2g_ab_*.txt): 3 x 4 beats 2 x 6 by 1 %, 4 x 3 by 0.4 %, 6 x 2 by 4 %; 1 x 12 loses 15 %.
#ifndef NSC_WS_DEPTH
#define NSC_WS_DEPTH 4
#endif
#ifndef NSC_WS_PTS
#define NSC_WS_PTS 3
#endif
constexpr int kWsStreamWarps = NSC_WS_STREAM_WARPS;
constexpr int kWsTailWarps = NSC_WS_TAIL_WARPS;
constexpr int kWsStreamThreads = kWsStreamWarps * 32;
constexpr int kWsTailThreads = kWsTailWarps * 32;
constexpr int kWsThreads = kWsStreamThreads + kWsTailThreads + 32;     // + the producer's warp
constexpr int kWsDepth = NSC_WS_DEPTH;
constexpr int kWsPts = NSC_WS_PTS;                                     // points per stream thread per stage
constexpr int kWsStagePoints = kWsPts * kWsStreamThreads;
constexpr int kWsSlotBytes = kWsStagePoints * 16;
constexpr int kBarTail = 1, kBarInit = 2;
using TailGroup = ThreadGroup<kWsTailThreads, kBarTail, kWsStreamThreads>;
static_assert(kWsThreads <= 1024 && kWsTailWarps <= kWarps, "warp split");

struct WsLayout {
    int img_off[2], tw_off, fa_off, hist_off, mask_off, nvalid_off, src_off, red_off, bins_off;
    int mail_off, mbar_off, ring_off, total, img_words;
    bool ok;       // false: this geometry needs the generic kernel
    __host__ __device__ WsLayout(int rows, int T, int n_bins) {
        int o = 0;
        auto take = [&o](int bytes) { int r = o; o += (bytes + 127) & ~127; return r; };
        const int n_sig = (T + 1) / 2;
        ok = n_sig <= kMaxSignals;
        const int sig_bytes = (n_sig < kMaxSignals ? n_sig : kMaxSignals) * kAz * 8;
        // an image doubles as the second FFT buffer of its own tail
        const int img_bytes = rows * kPitch * 4 > sig_bytes ? rows * kPitch * 4 : sig_bytes;
        img_words = rows * kPitch;
        ring_off = take(kWsDepth * kWsSlotBytes);
        img_off[0] = take(img_bytes);
        img_off[1] = take(img_bytes);
        tw_off = take(kAz * 8);
        fa_off = take(sig_bytes);
        hist_off = take(T * n_bins * 4);
        mask_off = take(rows * kMaskWords * 4);
        nvalid_off = take(rows * 4);
        src_off = take(rows * 4);
        red_off = take(kWarps * 8 + 16);
        bins_off = take(NSC_MAX_BINS + 3);
        mail_off = take(4 * 16 + 16);                    // 4 entries + tail_done + the arrival ticket of a split scan
        mbar_off = take((2 * kWsDepth + 4) * 8);
        total = o;
    }
};

// mbarrier addresses behind L.mbar_off
struct WsBars {
    uint32_t base;
    __device__ explicit WsBars(uint32_t b) : base(b) {}
    __device__ uint32_t slot_full(uint32_t s) const { return base + 8 * s; }
    __device__ uint32_t slot_empty(uint32_t s) const { return base + 8 * (kWsDepth + s); }
    __device__ uint32_t img_full(int b) const { return base + 8 * (2 * kWsDepth + b); }
    __device__ uint32_t img_empty(int b) const { return base + 8 * (2 * kWsDepth + 2 + b); }
};

// mail entry k & 3: int4 {sequence k, scan index, points of the scan, unused}
__device__ __forceinline__ void mail_read(const volatile int* mail, int k, int& scan, int& n) {
    const volatile int* e = mail + 4 * (k & 3);
    while (e[0] != k) { }
    __threadfence_block();
    scan = e[1];
    n = e[2];
}

__device__ __forceinline__ void ws_producer_role(const EncodeArgs& a, unsigned char* smem, const WsLayout& L) {
    volatile int* mail = reinterpret_cast<volatile int*>(smem + L.mail_off);
    const volatile int* tail_done = mail + 16;
    const WsBars bars(smem_u32(smem + L.mbar_off));
    const uint32_t ring = smem_u32(smem + L.ring_off);
    const float4* p4 = reinterpret_cast<const float4*>(a.points);
    int unit = blockIdx.x;
    int next = (int)gridDim.x + (int)atomicAdd(a.counter, 1u);
    const uint64_t pol = l2_policy_evict_first();
    // Evict-first only when the kernel has no peers (single-GPU encode: +1 %, the points no longer
    // push the descriptor lines out of L2); when descriptors of 7 peers are landing in this GPU's
    // memory it costs 3.5 % (profiles/r2o_*), so the copies stay plain there.
    const bool hint = a.out.peers.n == 0;
    uint32_t slot = 0, phase = 0;                     // phase = (stage counter / kWsDepth) & 1
    bool wrapped = false;
    for (int k = 0;; ++k) {
        int n = 0, scan = a.n_scans;
        const float4* src = p4;
        if (unit < a.n_units) {
            // units 0 .. n_whole-1 are whole scans; the rest are the `parts` pieces of the last scans
            const int j = unit - a.n_whole;
            scan = j < 0 ? unit : a.n_whole + j / a.parts;
            const long long o0 = a.offsets[scan];
            const long long n_tot = a.offsets[scan + 1] - o0;
            long long lo = 0, hi = n_tot;
            if (j >= 0) {
                const int part = j % a.parts;
                lo = n_tot * part / a.parts;
                hi = n_tot * (part + 1) / a.parts;
            }
            n = (int)(hi - lo);
            src += o0 - a.origin + lo;
        }
        while (*tail_done < k - 3) { }                // entry k & 3 is free: scan k - 4 is finished
        volatile int* e = mail + 4 * (k & 3);
        e[1] = scan;
        e[2] = n;
        __threadfence_block();
        e[0] = k;
        if (scan >= a.n_scans) break;
        for (int base = 0; base < n; base += kWsStagePoints) {
            if (wrapped) mbar_wait(bars.slot_empty(slot), phase ^ 1);
            const uint32_t bytes = (uint32_t)min(kWsStagePoints, n - base) * 16u;
            mbar_expect_tx(bars.slot_full(slot), bytes);
            if (hint) bulk_copy_g2s_hint(ring + slot * kWsSlotBytes, src + base, bytes, bars.slot_full(slot), pol);
            else bulk_copy_g2s(ring + slot * kWsSlotBytes, src + base, bytes, bars.slot_full(slot));
            if (++slot == kWsDepth) { slot = 0; phase ^= 1; wrapped = true; }
        }
        unit = next;
        if (unit < a.n_units) next = (int)gridDim.x + (int)atomicAdd(a.counter, 1u);
    }
}

template <int ROWMODE>
__device__ __forceinline__ void ws_stream_role(const EncodeArgs& a, const DeviceParams& dp,
                                               unsigned char* smem, const WsLayout& L) {
    const int tid = threadIdx.x;
    const volatile int* mail = reinterpret_cast<const volatile int*>(smem + L.mail_off);
    const WsBars bars(smem_u32(smem + L.mbar_off));
    const uint32_t ring_t = smem_u32(smem + L.ring_off) + tid * 16;
    const uint32_t bias = kFloorBias * (uint32_t)(kPitch * 4 + 4);
    const uint32_t img_b0 = smem_u32(smem + L.img_off[0]) - bias, img_b1 = smem_u32(smem + L.img_off[1]) - bias;
    uint32_t slot = 0, phase = 0;
    for (int k = 0;; ++k) {
        const int b = k & 1;
        int scan, n;
        mail_read(mail, k, scan, n);
        if (scan >= a.n_scans) break;
        if (k >= 2) mbar_wait(bars.img_empty(b), ((k >> 1) - 1) & 1);      // image b is free again
        const uint32_t img_biased = b ? img_b1 : img_b0;
        for (int base = 0; base < n; base += kWsStagePoints) {
            mbar_wait(bars.slot_full(slot), phase);
            const uint32_t src = ring_t + slot * kWsSlotBytes;
            float4 v[kWsPts];
#pragma unroll
            for (int u = 0; u < kWsPts; ++u) v[u] = lds128(src + u * (kWsStreamThreads * 16));
            if (base + kWsStagePoints <= n) {
#pragma unroll
                for (int u = 0; u + 1 < kWsPts; u += 2) project_pair<ROWMODE>(v[u], v[u + 1], dp, img_biased);
                if (kWsPts & 1)
                    project_point<ROWMODE>(v[kWsPts - 1].x, v[kWsPts - 1].y, v[kWsPts - 1].z, dp, img_biased);
            } else {
#pragma unroll
                for (int u = 0; u + 1 < kWsPts; u += 2)
                    project_pair<ROWMODE>(v[u], v[u + 1], dp, img_biased, base + u * kWsStreamThreads + tid < n,
                                          base + (u + 1) * kWsStreamThreads + tid < n);
                if (kWsPts & 1)
                    project_point<ROWMODE>(v[kWsPts - 1].x, v[kWsPts - 1].y, v[kWsPts - 1].z, dp, img_biased,
                                           base + (kWsPts - 1) * kWsStreamThreads + tid < n);
            }
            __syncwarp();
            if ((tid & 31) == 0) mbar_arrive(bars.slot_empty(slot));
            if (++slot == kWsDepth) { slot = 0; phase ^= 1; }
        }
        __syncwarp();
        if ((tid & 31) == 0) mbar_arrive(bars.img_full(b));
    }
}

__device__ __forceinline__ void ws_tail_role(const EncodeArgs& a, const DeviceParams& dp,
                                             unsigned char* smem, const WsLayout& L) {
    using G = TailGroup;
    const int gt = G::tid();
    volatile int* mail = reinterpret_cast<volatile int*>(smem + L.mail_off);
    const WsBars bars(smem_u32(smem + L.mbar_off));
    TailSmem S;
    S.tw = (float2*)(smem + L.tw_off);
    S.fa = (float2*)(smem + L.fa_off);
    S.hist = (float*)(smem + L.hist_off);
    S.mask = (uint32_t*)(smem + L.mask_off);
    S.nvalid = (int*)(smem + L.nvalid_off);
    S.src = (int*)(smem + L.src_off);
    S.red = (double*)(smem + L.red_off);
    S.bin_start = smem + L.bins_off;
    for (int k = 0;; ++k) {
        const int b = k & 1;
        int scan, n_unused;
        mail_read(mail, k, scan, n_unused);
        if (scan >= a.n_scans) break;
        mbar_wait(bars.img_full(b), (k >> 1) & 1);        // every stream warp is done with image b
        S.img = (float*)(smem + (b ? L.img_off[1] : L.img_off[0]));
        S.fb = (float2*)S.img;
        uint32_t* img = reinterpret_cast<uint32_t*>(S.img);
        // the image is dead once the magnitudes are out of it: hand it back to the stream warps
        auto release = [&]() {
            for (int i = gt; i < L.img_words; i += G::kSize) img[i] = kInfBits;
            __syncwarp();
            if ((gt & 31) == 0) mbar_arrive(bars.img_empty(b));
        };
        if (scan >= a.n_whole) {
            // One piece of a split scan: min-merge this image into the scan's image in global
            // memory; the CTA that brings the last piece takes the merged image back and runs the
            // tail, the others hand their image back and move on.
            unsigned* g = a.part_image + (size_t)(scan - a.n_whole) * L.img_words;
            for (int i = gt; i < L.img_words; i += G::kSize)
                if (img[i] != kInfBits) atomicMin(g + i, img[i]);
            __threadfence();
            G::sync();
            if (gt == 0) mail[17] = (int)atomicAdd(a.part_arrive + (scan - a.n_whole), 1u);
            G::sync();
            if (mail[17] != a.parts - 1) {
                release();
                G::sync();
                if (gt == 0) mail[16] = k + 1;            // tail_done
                continue;
            }
            __threadfence();
            for (int i = gt; i < L.img_words; i += G::kSize) img[i] = __ldcg(g + i);
            G::sync();
        }
        if (!finish_scan<G>(a, dp, S, scan, [&](int p) { if (p == 9) release(); })) {
            G::sync();     // projection only: every thread is done reading the image
            release();
        }
        G::sync();         // S.red / S.hist / S.src are rewritten by the next scan's tail
        if (gt == 0) mail[16] = k + 1;                    // tail_done
    }
    if (gt == 0) wait_bulk_stores_done();                 // descriptors leave shared memory before the CTA does
}

template <int ROWMODE>
__global__ void __launch_bounds__(kWsThreads, 1)
encode_points_ws_kernel(const __grid_constant__ EncodeArgs a, const __grid_constant__ DeviceParams dp) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const WsLayout L(dp.E, dp.T, dp.n_bins);
    const int tid = threadIdx.x;
    // a kernel enqueued as a programmatic dependent (the signal-and-wait of a multi-GPU step) may
    // be set up from now on; it still waits for this grid to complete before it does anything
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    if (tid == 0) {
        volatile int* mail = reinterpret_cast<volatile int*>(smem_raw + L.mail_off);
        const WsBars bars(smem_u32(smem_raw + L.mbar_off));
        for (int s = 0; s < kWsDepth; ++s) {
            mbar_init(bars.slot_full(s), 1);
            mbar_init(bars.slot_empty(s), kWsStreamWarps);
        }
        for (int b = 0; b < 2; ++b) {
            mbar_init(bars.img_full(b), kWsStreamWarps);
            mbar_init(bars.img_empty(b), kWsTailWarps);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        for (int i = 0; i < 4; ++i) mail[4 * i] = -1;      // sequence numbers that match no k
        mail[16] = 0;                                       // tail_done
    }
    __syncthreads();
    if (tid >= kWsStreamThreads + kWsTailThreads) {
        // the producer starts copying at once; the tables below are built under its first loads
        if (tid == kWsStreamThreads + kWsTailThreads) ws_producer_role(a, smem_raw, L);
        return;
    }
    {
        TailSmem S;
        S.tw = (float2*)(smem_raw + L.tw_off);
        S.bin_start = smem_raw + L.bins_off;
        constexpr int kWorkers = kWsStreamThreads + kWsTailThreads;
        for (int m = tid; m < kAz; m += kWorkers) {
            float sn, cs;
            sincospif((float)m * (1.0f / 180.0f), &sn, &cs);
            S.tw[m] = make_float2(cs, -sn);
        }
        for (int i = tid; i <= dp.n_bins; i += kWorkers) S.bin_start[i] = dp.bin_start[i];
        uint32_t* i0 = reinterpret_cast<uint32_t*>(smem_raw + L.img_off[0]);
        uint32_t* i1 = reinterpret_cast<uint32_t*>(smem_raw + L.img_off[1]);
        for (int i = tid; i < L.img_words; i += kWorkers) {
            i0[i] = kInfBits;
            i1[i] = kInfBits;
        }
        asm volatile("bar.sync %0, %1;" ::"n"(kBarInit), "n"(kWorkers) : "memory");
    }
    if (tid < kWsStreamThreads) ws_stream_role<ROWMODE>(a, dp, smem_raw, L);
    else ws_tail_role(a, dp, smem_raw, L);
}

// Small batches (fewer scans than SMs / cluster size): one thread-block CLUSTER per scan. The
// CTAs of a cluster each scatter a contiguous slice of the scan into their own shared-memory
// image; after a cluster barrier the leader min-reduces the other images through distributed
// shared memory and runs the tail. Cuts the latency of a single 120 k-point scan from one SM's
// worth of time to roughly 1/cluster_size of it plus the tail.
template <int STRIDE, int ROWMODE, int ROWS>
__device__ __forceinline__ void cluster_scan(const EncodeArgs& a, const DeviceParams& dp) {
    constexpr bool tall = ROWS > kShortRows;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    namespace cg = cooperative_groups;
    cg::cluster_group cluster = cg::this_cluster();
    const unsigned rank = cluster.block_rank(), csize = cluster.num_blocks();
    const SmemLayout L(dp.E, dp.T, dp.n_bins, tall ? 0 : ring_bytes(STRIDE), tall);
    const TailSmem S(smem_raw, L);
    uint32_t* img = reinterpret_cast<uint32_t*>(S.img);
    const uint32_t img_biased = smem_u32(img) - kFloorBias * (uint32_t)(kPitch * 4 + 4);
    const int tid = threadIdx.x;
    const int n_pix = dp.E * kPitch;
    const int scan = blockIdx.x / csize;      // grid = n_scans * cluster size

    if (rank == 0) init_tail_tables(S, dp);
    for (int i = tid; i < n_pix; i += kThreads) img[i] = kInfBits;
    __syncthreads();
    const long long beg = a.offsets[scan] - a.origin;
    const int n = (int)(a.offsets[scan + 1] - a.offsets[scan]);
    const int per = (n + (int)csize - 1) / (int)csize;
    const int lo = min(n, (int)rank * per), hi = min(n, lo + per);
    point_pass<STRIDE, ROWMODE, ROWS>(a.points, beg + lo, hi - lo, dp, img_biased, smem_raw + L.ring_off);
    cluster.sync();                           // every partial image is complete
    if (rank == 0) {
        for (int i = tid; i < n_pix; i += kThreads) {
            uint32_t m = img[i];
            for (unsigned r = 1; r < csize; ++r) m = min(m, cluster.map_shared_rank(img, r)[i]);
            img[i] = m;
        }
    }
    cluster.sync();                           // peers may exit only after the leader has read them
    if (rank == 0) {
        __syncthreads();
        long long phase_t0 = 0;
        finish_scan<CtaGroup, ROWS>(a, dp, S, scan, [&](int p) { NSC_PHASE(p); });
        if (tid == 0) wait_bulk_stores_done();
    }
}

template <int STRIDE, int ROWMODE>
__global__ void __launch_bounds__(kThreads, 1)
encode_points_split_kernel(const __grid_constant__ EncodeArgs a, const __grid_constant__ DeviceParams dp) {
    cluster_scan<STRIDE, ROWMODE, kShortRows>(a, dp);
}

// The same for images of more than 64 rows: every CTA of the cluster holds a whole tall image.
template <int STRIDE, int ROWMODE>
__global__ void __launch_bounds__(kThreads, 1)
encode_points_tall_split_kernel(const __grid_constant__ EncodeArgs a, const __grid_constant__ DeviceParams dp) {
    cluster_scan<STRIDE, ROWMODE, NSC_MAX_ELEVATION>(a, dp);
}

// Range images in, descriptors out: SpectralEncoder.forward / encode_range_image
// (spectral_encoder.py:160-204, :231-261). No projection, no interpolation.
__global__ void __launch_bounds__(kThreads, kMinBlocks)
encode_images_kernel(const float* __restrict__ images, int n_images, int rows,
                     const __grid_constant__ DeviceParams dp, float* __restrict__ out) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const SmemLayout L(rows, dp.T, dp.n_bins);
    const TailSmem S(smem_raw, L);
    const int D = dp.T * dp.n_bins;
    init_tail_tables(S, dp);
    if (threadIdx.x < rows) S.src[threadIdx.x] = threadIdx.x;
    for (int im = blockIdx.x; im < n_images; im += gridDim.x) {
        __syncthreads();
        const float* src = images + (long long)im * rows * kAz;
        for (int i = threadIdx.x; i < rows * kAz; i += kThreads) {
            const int r = i / kAz, c = i - r * kAz;
            S.img[r * kPitch + c] = src[i];
        }
        __syncthreads();
        spectrum_and_bins(S, dp, rows);
        RowDest dst;
        dst.out = out + (long long)im * D;
        normalise_and_store(S, dp, dst);
    }
    if (threadIdx.x == 0) wait_bulk_stores_done();
}

// The same for images of more than 64 rows: pooled to T rows while they are read from global
// memory (pooled_value's arithmetic; forward() has no empty-row fill), so shared memory holds the
// T-row image only.
__global__ void __launch_bounds__(kThreads, kMinBlocks)
encode_tall_images_kernel(const float* __restrict__ images, int n_images, int rows,
                          const __grid_constant__ DeviceParams dp, float* __restrict__ out) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int T = dp.T;
    const SmemLayout L(T, T, dp.n_bins);
    const TailSmem S(smem_raw, L);
    const int D = T * dp.n_bins;
    init_tail_tables(S, dp);
    if (threadIdx.x < T) S.src[threadIdx.x] = threadIdx.x;
    for (int im = blockIdx.x; im < n_images; im += gridDim.x) {
        __syncthreads();
        const float* src = images + (long long)im * rows * kAz;
        for (int i = threadIdx.x; i < T * kAz; i += kThreads) {
            const int t = i / kAz, c = i - t * kAz;
            const int r0 = (t * rows) / T, r1 = ((t + 1) * rows + T - 1) / T;
            float sum = 0.0f;
            for (int r = r0; r < r1; ++r) sum += src[r * kAz + c];
            S.img[t * kPitch + c] = sum / (float)(r1 - r0);
        }
        __syncthreads();
        spectrum_and_bins(S, dp, T);
        RowDest dst;
        dst.out = out + (long long)im * D;
        normalise_and_store(S, dp, dst);
    }
    if (threadIdx.x == 0) wait_bulk_stores_done();
}

// interpolate_range_image on device images (range_image.py:15-89).
__global__ void __launch_bounds__(kThreads, kMinBlocks)
interpolate_kernel(const float* __restrict__ in, int n_images, int rows, int nearest, float* __restrict__ out) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const SmemLayout L(rows, 1, 1);
    const TailSmem S(smem_raw, L);
    for (int im = blockIdx.x; im < n_images; im += gridDim.x) {
        __syncthreads();
        const float* src = in + (long long)im * rows * kAz;
        for (int i = threadIdx.x; i < rows * kAz; i += kThreads) {
            const int r = i / kAz, c = i - r * kAz;
            S.img[r * kPitch + c] = src[i];
        }
        __syncthreads();
        rows_to_filled<false>(S, rows, true, nullptr, [](uint32_t) { return 0.0f; }, nearest != 0);
        float* dst = out + (long long)im * rows * kAz;
        for (int i = threadIdx.x; i < rows * kAz; i += kThreads) {
            const int r = i / kAz, c = i - r * kAz;
            dst[i] = S.img[S.src[r] * kPitch + c];
        }
    }
}

struct DeviceInfo {
    int sms = 0;
    int max_smem_optin = 0;
};

int device_info(DeviceInfo* out) {
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return record_cuda(e);
    static std::mutex mu;
    static DeviceInfo cache[64];
    std::lock_guard<std::mutex> lk(mu);
    if (dev >= 0 && dev < 64 && cache[dev].sms > 0) { *out = cache[dev]; return NSC_OK; }
    DeviceInfo di;
    e = cudaDeviceGetAttribute(&di.sms, cudaDevAttrMultiProcessorCount, dev);
    if (e != cudaSuccess) return record_cuda(e);
    e = cudaDeviceGetAttribute(&di.max_smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
    if (e != cudaSuccess) return record_cuda(e);
    if (dev >= 0 && dev < 64) cache[dev] = di;
    *out = di;
    return NSC_OK;
}

// Raises the kernel's dynamic shared-memory limit when needed and returns its occupancy; both are
// remembered per (kernel, device) so a steady-state launch makes no runtime query.
struct KernelState {
    const void* fn;
    int device;
    int smem_limit;                 // largest cudaFuncAttributeMaxDynamicSharedMemorySize set so far
    std::vector<std::pair<int, int>> occupancy;   // (smem, blocks per SM)
};

template <typename K>
int configure(K kernel, int smem, const DeviceInfo& di, int* blocks_per_sm) {
    if (smem > di.max_smem_optin) return NSC_ERR_BAD_PARAMS;
    static std::mutex mu;
    static std::vector<KernelState> states;
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return record_cuda(e);
    std::lock_guard<std::mutex> lk(mu);
    KernelState* ks = nullptr;
    for (KernelState& s : states)
        if (s.fn == (const void*)kernel && s.device == dev) ks = &s;
    if (!ks) {
        states.push_back(KernelState{(const void*)kernel, dev, 0, {}});
        ks = &states.back();
    }
    if (smem > ks->smem_limit) {
        e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        if (e != cudaSuccess) return record_cuda(e);
        ks->smem_limit = smem;
    }
    if (blocks_per_sm) {
        for (const auto& o : ks->occupancy)
            if (o.first == smem) { *blocks_per_sm = o.second; return NSC_OK; }
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(blocks_per_sm, kernel, kThreads, smem);
        if (e != cudaSuccess) return record_cuda(e);
        if (*blocks_per_sm < 1) return NSC_ERR_BAD_PARAMS;
        ks->occupancy.emplace_back(smem, *blocks_per_sm);
    }
    return NSC_OK;
}

using PointKernel = void (*)(const EncodeArgs, const DeviceParams);

// The instantiation of the cluster (split) or the generic point kernel, for images of up to 64
// rows or taller ones, for a point stride and a row mode.
#define NSC_POINT_KERNELS(K) {{K<3, kRowPoly>, K<3, kRowSearch>}, {K<4, kRowPoly>, K<4, kRowSearch>}}
PointKernel point_kernel(bool split, bool tall, int stride, int row_mode) {
    static const PointKernel generic[2][2] = NSC_POINT_KERNELS(encode_points_kernel);
    static const PointKernel cluster[2][2] = NSC_POINT_KERNELS(encode_points_split_kernel);
    static const PointKernel generic_tall[2][2] = NSC_POINT_KERNELS(encode_points_tall_kernel);
    static const PointKernel cluster_tall[2][2] = NSC_POINT_KERNELS(encode_points_tall_split_kernel);
    const PointKernel(*k)[2] = split ? (tall ? cluster_tall : cluster) : (tall ? generic_tall : generic);
    return k[stride == 4 ? 1 : 0][row_mode == kRowPoly ? 0 : 1];
}
#undef NSC_POINT_KERNELS

}  // namespace

// Workspace: [0, 256) work counter; [256, 256 + 4 * kMaxSplitScans) arrival counters and then one
// E x 361 key image per split scan (launch_encode splits the scans of the last, partial wave of the
// grid when the workspace has room for it; kMinWorkspace is enough for everything else).
constexpr int kMaxSplitScans = 256;
constexpr size_t kMinWorkspace = 256;
static size_t split_workspace(int n_split, int E) {
    return kMinWorkspace + (size_t)kMaxSplitScans * 4 + (size_t)n_split * E * kPitch * 4;
}
size_t workspace_bytes_for(int n_scans, int E) {
    (void)n_scans;
    return E > kShortRows ? kMinWorkspace : split_workspace(kMaxSplitScans - 1, E);   // tall kernels split no scan
}
size_t workspace_bytes_min() { return kMinWorkspace; }

int launch_encode(const PointBatch& in, const DeviceParams& dp, const EncodeOutputs& out,
                  unsigned* d_workspace, size_t workspace_bytes, cudaStream_t stream) {
    const int n_scans = in.n_scans;
    if (n_scans == 0) return NSC_OK;
    if (out.n_peers < 0 || out.n_peers > NSC_MAX_PEERS) return NSC_ERR_BAD_COUNT;
    // uint16 rows are packed over the float32 row in shared memory: they are written alone
    if (out.rows_q && (out.rows || out.n_peers > 0)) return NSC_ERR_BAD_PARAMS;
    DeviceInfo di;
    int st = device_info(&di);
    if (st != NSC_OK) return st;
    EncodeArgs a = {};
    a.points = in.points;
    a.offsets = in.offsets;
    a.origin = in.origin;
    a.n_scans = n_scans;
    a.out.rows = out.rows;
    a.out.rows_q = out.rows_q;
    a.out.q_eps = out.q_eps;
    if (out.rows_q) {
        st = build_plan(dp.T * dp.n_bins, &a.out.q_plan);    // D <= NSC_MAX_DESCRIPTOR: always fits
        if (st != NSC_OK) return st;
    }
    a.out.images = out.images;
    a.out.stage = out.stage;
    for (int i = 0; i < out.n_peers; ++i) a.out.peers.ptr[i] = out.peers[i];
    a.out.peers.n = out.n_peers;
    a.out.peers.row0 = out.peer_row0;
    a.counter = d_workspace;
    a.n_whole = n_scans;
    a.parts = 1;
    a.n_units = n_scans;

    // Kernel choice. Product builds take no switches; tuning builds (-DNSC_TUNING, csrc/Makefile
    // VARIANT=tune) read NSC_SPLIT=0, NSC_WS=0 and NSC_TAILSPLIT=0 from the environment, once, so
    // that A/B runs and the bit-identity tests can route a batch around the cluster kernel, the
    // warp-specialised kernel or the split of its last wave.
#ifdef NSC_TUNING
    static const bool env_split = [] { const char* e = getenv("NSC_SPLIT"); return !(e && e[0] == '0'); }();
    static const bool env_ws = [] { const char* e = getenv("NSC_WS"); return !(e && e[0] == '0'); }();
    static const bool env_ts = [] { const char* e = getenv("NSC_TAILSPLIT"); return !(e && e[0] == '0'); }();
#else
    constexpr bool env_split = true, env_ws = true, env_ts = true;
#endif
    // Images of more than 64 rows take the tall kernels (one image per SM, no ring, no
    // warp-specialised variant): by the row count alone.
    const bool tall = dp.E > kShortRows;
    const SmemLayout L(dp.E, dp.T, dp.n_bins, tall ? 0 : ring_bytes(in.stride), tall);
    int csize = 1;
    if (env_split) {
        if (n_scans * 8 <= di.sms) csize = 8;
        else if (n_scans * 4 <= di.sms) csize = 4;
        else if (n_scans * 2 <= di.sms) csize = 2;
    }
    PointKernel kernel = nullptr;
    if (csize > 1) {
        kernel = point_kernel(true, tall, in.stride, dp.row_mode);
        st = configure(kernel, L.total, di, nullptr);
        if (st != NSC_OK) return st;
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3((unsigned)(n_scans * csize));
        cfg.blockDim = dim3(kThreads);
        cfg.dynamicSmemBytes = (size_t)L.total;
        cfg.stream = stream;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = (unsigned)csize;
        attr[0].val.clusterDim.y = 1;
        attr[0].val.clusterDim.z = 1;
        cfg.attrs = attr;
        cfg.numAttrs = 1;
        return record_cuda(cudaLaunchKernelEx(&cfg, kernel, a, dp));
    }
    // Large batches of 16-byte points: the warp-specialised kernel, when two images, the FFT
    // scratch and the ring fit one SM's shared memory; other geometries take the generic kernel.
    const WsLayout W(dp.E, dp.T, dp.n_bins);
    if (!tall && env_ws && in.stride == 4 && W.ok && W.total <= di.max_smem_optin) {
        kernel = dp.row_mode == kRowPoly ? encode_points_ws_kernel<kRowPoly> : encode_points_ws_kernel<kRowSearch>;
        st = configure(kernel, W.total, di, nullptr);
        if (st != NSC_OK) return st;
        const int grid = di.sms < n_scans ? di.sms : n_scans;
        // The scans are handed out dynamically, one per CTA at a time, so the last R = n_scans mod
        // grid of them keep only part of the GPU busy for a whole scan time. When R <= grid / 2 each
        // of them is split into P = floor(grid / R) pieces (merged through a key image in global
        // memory by the tail warps), one piece per CTA: that wave then lasts 1 / P of a scan time
        // (600 scans: +5 %, profiles/r2s_ab_hdl64_600.txt). More pieces than CTAs do not pay: a
        // piece streams faster than its tail -- the merge, and for the last piece the whole FFT --
        // runs, and the tail warps become the bottleneck (4541 scans as 4 pieces each: -3 %).
        const int R = n_scans > grid ? n_scans % grid : 0;
        if (env_ts && R > 0 && 2 * R <= grid) {
            int P = grid / R;
            if (P > 8) P = 8;
            if (workspace_bytes >= split_workspace(R, dp.E)) {
                a.n_whole = n_scans - R;
                a.parts = P;
                a.n_units = a.n_whole + R * P;
                a.part_arrive = d_workspace + kMinWorkspace / 4;
                a.part_image = a.part_arrive + kMaxSplitScans;
            }
        }
        cudaError_t e = cudaMemsetAsync(d_workspace, 0, a.parts > 1 ? kMinWorkspace + (size_t)kMaxSplitScans * 4 : 8, stream);
        if (e != cudaSuccess) return record_cuda(e);
        if (a.parts > 1) {
            e = cudaMemsetAsync(a.part_image, 0xff, (size_t)R * dp.E * kPitch * 4, stream);
            if (e != cudaSuccess) return record_cuda(e);
        }
        kernel<<<grid, kWsThreads, W.total, stream>>>(a, dp);
        return record_cuda(cudaGetLastError());
    }
    kernel = point_kernel(false, tall, in.stride, dp.row_mode);
    int per_sm = 0;
    st = configure(kernel, L.total, di, &per_sm);
    if (st != NSC_OK) return st;
#ifdef NSC_PHASE_TIMING
    cudaError_t e = cudaMemsetAsync(d_workspace, 0, 128, stream);
#else
    cudaError_t e = cudaMemsetAsync(d_workspace, 0, 2 * sizeof(unsigned), stream);
#endif
    if (e != cudaSuccess) return record_cuda(e);
    int grid = di.sms * per_sm;
    if (grid > n_scans) grid = n_scans;
    kernel<<<grid, kThreads, L.total, stream>>>(a, dp);
    return record_cuda(cudaGetLastError());
}

int launch_encode_images(const float* d_images, int n_images, int rows, const DeviceParams& dp,
                         float* d_out, cudaStream_t stream) {
    if (n_images == 0) return NSC_OK;
    DeviceInfo di;
    int st = device_info(&di);
    if (st != NSC_OK) return st;
    // more than 64 rows: pooled while loaded, so the kernel holds T <= 64 rows
    const bool tall = rows > kShortRows;
    const SmemLayout L(tall ? dp.T : rows, dp.T, dp.n_bins);
    const auto kernel = tall ? encode_tall_images_kernel : encode_images_kernel;
    int per_sm = 0;
    st = configure(kernel, L.total, di, &per_sm);
    if (st != NSC_OK) return st;
    int grid = di.sms * per_sm;
    if (grid > n_images) grid = n_images;
    kernel<<<grid, kThreads, L.total, stream>>>(d_images, n_images, rows, dp, d_out);
    return record_cuda(cudaGetLastError());
}

int launch_interpolate(const float* d_in, int n_images, int rows, int nearest, float* d_out, cudaStream_t stream) {
    if (n_images == 0) return NSC_OK;
    DeviceInfo di;
    int st = device_info(&di);
    if (st != NSC_OK) return st;
    const SmemLayout L(rows, 1, 1);
    int per_sm = 0;
    st = configure(interpolate_kernel, L.total, di, &per_sm);
    if (st != NSC_OK) return st;
    int grid = di.sms * per_sm;
    if (grid > n_images) grid = n_images;
    interpolate_kernel<<<grid, kThreads, L.total, stream>>>(d_in, n_images, rows, nearest, d_out);
    return record_cuda(cudaGetLastError());
}

}  // namespace nsc
