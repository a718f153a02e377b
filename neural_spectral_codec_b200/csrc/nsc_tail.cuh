// Shared-memory tail of the encoder: everything after the per-pixel min scatter.
//   validity masks -> circular linear hole interpolation + empty-row fill
//   (reference src/encoding/range_image.py:15-89) -> optional row pooling
//   (spectral_encoder.py:171-176) -> 360-point FFT magnitude per row (:180-186) ->
//   contiguous-frequency bin sums (:118-158) -> L1 normalisation (:197-202) -> optionally the
//   uint16 wire format (HistogramQuantizer.quantize, quantization.py:131-167).
// All functions are CTA-collective: every thread of the block must call them.
#pragma once
#include "nsc_fft.cuh"
#include "nsc_internal.h"
#include "nsc_quantize.cuh"

namespace nsc {

#ifndef NSC_THREADS
#define NSC_THREADS 512
#endif
#ifndef NSC_MIN_BLOCKS
#define NSC_MIN_BLOCKS 2
#endif
constexpr int kThreads = NSC_THREADS;
constexpr int kWarps = kThreads / 32;
constexpr int kMinBlocks = NSC_MIN_BLOCKS;   // resident CTAs per SM the kernels are compiled for

// The threads that run the tail together: the whole CTA (BAR = 0, __syncthreads), or a warp
// group of a warp-specialised CTA meeting on its own named barrier (encode_points_ws_kernel).
template <int SIZE, int BAR, int TID0>
struct ThreadGroup {
    static constexpr int kSize = SIZE;
    static constexpr int kGroupWarps = SIZE / 32;
    __device__ static __forceinline__ int tid() { return (int)threadIdx.x - TID0; }
    __device__ static __forceinline__ void sync() {
        if (BAR == 0) __syncthreads();
        else asm volatile("bar.sync %0, %1;" ::"n"(BAR), "n"(SIZE) : "memory");
    }
};
using CtaGroup = ThreadGroup<kThreads, 0, 0>;

// Per-thread cp.async ring (LDGSTS feed): kCpDepth stages of kCpPts 16-byte points per thread.
#ifndef NSC_CP_PTS
#define NSC_CP_PTS 2
#endif
#ifndef NSC_CP_DEPTH
#define NSC_CP_DEPTH 4
#endif
constexpr int kCpPts = NSC_CP_PTS;
constexpr int kCpDepth = NSC_CP_DEPTH;
constexpr int kCpRingBytes = kCpDepth * kCpPts * kThreads * 16;   // 65 536 B per CTA

// Shared-memory carve-up, identical on host (size) and device (pointers). With a ring the two
// FFT buffers alias it: the ring is idle (fully consumed) while the tail runs.
// pooled: the layout of the tall kernels (rows > kShortRows), whose tail pools the image in place
// to its first T rows (pool_rows_in_place) before the spectrum; both FFT buffers then lie in the
// image's dead rows above them, and no ring is kept.
struct SmemLayout {
    int img_off, tw_off, fa_off, fb_off, hist_off, mask_off, nvalid_off, src_off, red_off;
    int ring_off, bins_off, total;
    int n_sig;  // complex FFTs per batch
    __host__ __device__ SmemLayout(int rows, int T, int n_bins, int ring_bytes = 0, bool pooled = false) {
        const bool ring = ring_bytes > 0;
        int o = 0;
        auto take = [&o](int bytes) { int r = o; o += (bytes + 127) & ~127; return r; };
        n_sig = (T + 1) / 2 < kMaxSignals ? (T + 1) / 2 : kMaxSignals;
        const int sig_bytes = n_sig * kAz * 8;
        if (pooled) {
            const int pooled_bytes = (T * kPitch * 4 + 127) & ~127;
            const int img_bytes = rows * kPitch * 4;
            img_off = take(img_bytes > pooled_bytes + 2 * sig_bytes ? img_bytes : pooled_bytes + 2 * sig_bytes);
            tw_off = take(kAz * 8);
            ring_off = fa_off = img_off + pooled_bytes;
            fb_off = fa_off + sig_bytes;
        } else {
            img_off = take(rows * kPitch * 4);
            tw_off = take(kAz * 8);
            // The second FFT buffer may reuse the image: once the (single) batch of signals has
            // been loaded from the image into fa, the image is dead.
            const bool fb_on_img = (T + 1) / 2 <= kMaxSignals && rows * kPitch * 4 >= sig_bytes;
            const int scratch = fb_on_img ? sig_bytes : 2 * sig_bytes;
            ring_off = take(ring && ring_bytes > scratch ? ring_bytes : scratch);
            fa_off = ring_off;
            fb_off = fb_on_img ? img_off : ring_off + sig_bytes;
        }
        hist_off = take(T * n_bins * 4);
        mask_off = take(rows * kMaskWords * 4);
        nvalid_off = take(rows * 4);
        src_off = take(rows * 4);
        red_off = take(kWarps * 8 + 16);
        bins_off = take(NSC_MAX_BINS + 3);
        total = o;
    }
};

struct TailSmem {
    float* img;        // rows x kPitch
    float2* tw;        // exp(-2 pi i m / 360)
    float2* fa;
    float2* fb;
    float* hist;
    uint32_t* mask;    // rows x kMaskWords validity bits (value > 0)
    int* nvalid;
    int* src;          // row r of the filled image is stored row src[r]
    double* red;
    uint8_t* bin_start;  // copy of DeviceParams::bin_start: per-thread indices would serialise in the constant bank
    __device__ TailSmem() {}
    __device__ TailSmem(unsigned char* base, const SmemLayout& L)
        : img((float*)(base + L.img_off)), tw((float2*)(base + L.tw_off)),
          fa((float2*)(base + L.fa_off)), fb((float2*)(base + L.fb_off)),
          hist((float*)(base + L.hist_off)), mask((uint32_t*)(base + L.mask_off)),
          nvalid((int*)(base + L.nvalid_off)), src((int*)(base + L.src_off)),
          red((double*)(base + L.red_off)), bin_start(base + L.bins_off) {}
};

// Per-CTA constants of the tail: FFT twiddles and the bin boundaries.
template <typename P>
__device__ __forceinline__ void init_tail_tables(const TailSmem& S, const P& dp) {
    const int n_thr = (int)blockDim.x;
    for (int m = threadIdx.x; m < kAz; m += n_thr) {
        float s, c;
        sincospif((float)m * (1.0f / 180.0f), &s, &c);   // angle = 2 pi m / 360
        S.tw[m] = make_float2(c, -s);
    }
    for (int b = threadIdx.x; b <= dp.n_bins; b += n_thr) S.bin_start[b] = dp.bin_start[b];
}

// Nearest valid column strictly left / right of x on the circular row; the returned position
// is unwrapped (left in (x-360, x), right in (x, x+360)), as np.interp sees it on the tiled
// abscissa (range_image.py:55-64). Requires at least one valid bit in the row.
__device__ __forceinline__ int prev_valid(const uint32_t* m, int x) {
    int w = x >> 5, off = 0;
    uint32_t bits = m[w] & ((1u << (x & 31)) - 1u);
    while (bits == 0) {
        if (--w < 0) { w = kMaskWords - 1; off -= kAz; }
        bits = m[w];
    }
    return off + w * 32 + 31 - __clz(bits);
}
__device__ __forceinline__ int next_valid(const uint32_t* m, int x) {
    int w = x >> 5, off = 0;
    uint32_t bits = m[w] & ~((2u << (x & 31)) - 1u);
    while (bits == 0) {
        if (++w >= kMaskWords) { w = 0; off += kAz; }
        bits = m[w];
    }
    return off + w * 32 + __ffs(bits) - 1;
}

// One warp per row: (optionally) turn the scattered keys into ranges, build the validity mask
// (valid <=> value > 0, range_image.py:35) and fill the holes of the row by circular linear
// interpolation (range_image.py:33-64). Everything a row needs was produced by the same warp,
// so no block barrier separates the three steps. FROM_KEYS: the row holds the bits of the min
// of s per pixel (plus the 361st column for azimuth == 2 pi); `to_value(key)` maps them to ranges.
// `stage0`, if not null, receives the un-interpolated rows (rows x 360, global memory).
// `nearest` selects interpolate_range_image(method='nearest') (range_image.py:66-75): a hole takes
// the value of the valid pixel at the smallest circular distance, the lower column on a tie
// (np.argmin over ascending valid indices).
template <bool FROM_KEYS, typename G = CtaGroup, typename ToValue>
__device__ __forceinline__ void rows_to_filled(const TailSmem& S, int rows, bool interpolate,
                                               float* __restrict__ stage0, ToValue to_value,
                                               bool nearest = false) {
    const int warp = G::tid() >> 5, lane = G::tid() & 31;
    for (int r = warp; r < rows; r += G::kGroupWarps) {
        float* row = S.img + r * kPitch;
        uint32_t* m = S.mask + r * kMaskWords;
        int cnt = 0;
#pragma unroll
        for (int w = 0; w < kMaskWords; ++w) {
            const int c = w * 32 + lane;
            float v = 0.0f;
            if (c < kAz) {
                if (FROM_KEYS) {
                    uint32_t key = __float_as_uint(row[c]);
                    if (c == 0) key = min(key, __float_as_uint(row[kAz]));   // azimuth == 2 pi -> column 0
                    v = to_value(key);
                    row[c] = v;
                } else {
                    v = row[c];
                }
                if (stage0) stage0[r * kAz + c] = v;
            }
            const uint32_t bits = __ballot_sync(0xffffffffu, v > 0.0f);
            cnt += __popc(bits);
            if (lane == 0) m[w] = bits;
        }
        if (lane == 0) S.nvalid[r] = cnt;
        __syncwarp();
        if (interpolate && cnt != 0 && cnt != kAz) {
            // writes only hole pixels and reads only valid ones: race-free in place
            for (int x = lane; x < kAz; x += 32) {
                if ((m[x >> 5] >> (x & 31)) & 1u) continue;
                const int xl = prev_valid(m, x), xr = next_valid(m, x);
                const int il = xl < 0 ? xl + kAz : xl, ir = xr >= kAz ? xr - kAz : xr;
                if (nearest) {
                    const int dl = x - xl, dr = xr - x;
                    row[x] = row[dl < dr || (dl == dr && il < ir) ? il : ir];
                    continue;
                }
                const double fl = (double)row[il];
                const double fr = (double)row[ir];
                // np.interp: slope = (fp[j+1]-fp[j])/(xp[j+1]-xp[j]); slope*(x-xp[j]) + fp[j], float64
                const double slope = __ddiv_rn(__dsub_rn(fr, fl), (double)(xr - xl));
                row[x] = __double2float_rn(__dadd_rn(__dmul_rn(slope, (double)(x - xl)), fl));
            }
        }
    }
    G::sync();
    // Empty-row fill (range_image.py:77-87) as a row indirection src[] instead of copies: rows with
    // no pixel > 0 take the nearest filled row below, leading ones the first non-empty row above;
    // an all-empty image stays zero (the sequential in-place semantics of the reference).
    if (G::tid() < rows) {
        const int r = G::tid();
        int s = r;
        if (interpolate && S.nvalid[r] == 0) {
            int k = r - 1;
            while (k >= 0 && S.nvalid[k] == 0) --k;
            if (k < 0) {
                k = r + 1;
                while (k < rows && S.nvalid[k] == 0) ++k;
            }
            if (k >= 0 && k < rows) s = k;
        }
        S.src[r] = s;
    }
    G::sync();
}

// Descriptor stores as bulk copies shared -> global (TMA, SASS UBLKCP.G.S): the normalised
// descriptor is written in place over S.hist and ONE thread sends the 3.2 KB to the local output
// and to every peer's database -- over NVLink for the remote ones -- instead of every thread
// storing every element 1 + n_peers times. wait_bulk_stores_read() must precede the next write to
// S.hist by any thread (called by the issuing thread before a group barrier that all pass).
__device__ __forceinline__ void bulk_store_s2g(void* dst, const void* src_smem, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst),
                 "r"((uint32_t)__cvta_generic_to_shared(src_smem)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void wait_bulk_stores_read() {
    asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
}
__device__ __forceinline__ void wait_bulk_stores_done() {
    asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
}

// Value of target row i at column n: the stored row, or the mean of its source rows when the
// image height differs from T (adaptive_avg_pool2d on (1,1,rows,360) -> (T,360)).
__device__ __forceinline__ float pooled_value(const TailSmem& S, int rows, int T, int i, int n) {
    if (rows == T) return S.img[S.src[i] * kPitch + n];
    const int r0 = (i * rows) / T, r1 = ((i + 1) * rows + T - 1) / T;
    float sum = 0.0f;
    for (int r = r0; r < r1; ++r) sum += S.img[S.src[r] * kPitch + n];
    return sum / (float)(r1 - r0);
}

// The tall kernels' pooling (rows > T): rows 0..T-1 of S.img become the pooled rows, with
// pooled_value's arithmetic, and S.src the identity, so that spectrum_and_bins(S, dp, T) reads
// them and the FFT buffers may take the rows above (SmemLayout's `pooled` layout). First the
// empty-row fill is written out (an empty row takes its source row's values; sources are never
// empty, so no copy reads a copied row), then every thread pools one column upwards: target row i
// reads rows >= floor(i * rows / T) >= i, none of which a smaller target has overwritten.
template <typename G>
__device__ __forceinline__ void pool_rows_in_place(const TailSmem& S, int rows, int T) {
    for (int i = G::tid(); i < rows * kAz; i += G::kSize) {
        const int r = i / kAz, c = i - r * kAz;
        if (S.src[r] != r) S.img[r * kPitch + c] = S.img[S.src[r] * kPitch + c];
    }
    G::sync();
    for (int r = G::tid(); r < rows; r += G::kSize) S.src[r] = r;
    G::sync();
    for (int n = G::tid(); n < kAz; n += G::kSize)
        for (int i = 0; i < T; ++i) S.img[i * kPitch + n] = pooled_value(S, rows, T, i, n);
    G::sync();
}

// One Stockham pass of radix R over n_sig complex signals of length 360: one thread per
// butterfly (nsc_fft.cuh), R inputs and outputs in registers.
template <int R, int NS, typename G = CtaGroup>
__device__ __forceinline__ void fft_pass(const float2* __restrict__ x, float2* __restrict__ y,
                                         const float2* __restrict__ tw, int n_sig) {
    constexpr int kBfly = kAz / R;
    for (int t = G::tid(); t < n_sig * kBfly; t += G::kSize) {
        const int g = t / kBfly, j = t - g * kBfly;
        stockham_butterfly<R, NS>(x + g * kAz, y + g * kAz, tw, j);
    }
}

// Rows of the (pooled) image, two per complex signal -> spectra -> magnitudes -> bin sums in
// S.hist (un-normalised). The mapping hist index -> thread (i = tid + k * kThreads) is the one
// normalise_and_store() uses, so no barrier is needed between the two for S.hist.
struct NoMark {
    __device__ __forceinline__ void operator()(int) const {}
};
// `mark(p)` is a tuning hook called by thread-uniform code between the sub-phases (5 = signals
// loaded, 6..8 = after each FFT pass, 9 = magnitudes); a no-op in product builds.
template <typename P, typename Mark = NoMark, typename G = CtaGroup>
__device__ __forceinline__ void spectrum_and_bins(const TailSmem& S, const P& dp, int rows,
                                                  Mark mark = Mark(), G = G()) {
    const int T = dp.T, nb = dp.n_bins;
    const int n_sig_total = (T + 1) / 2;
    const int cap = n_sig_total < kMaxSignals ? n_sig_total : kMaxSignals;
    // the previous descriptor may still be on its way out of S.hist (bulk stores of
    // normalise_and_store): the thread that issued them waits here; every other thread passes at
    // least one group barrier below before S.hist is written again
    if (G::tid() == 0) wait_bulk_stores_read();
    float* mag = reinterpret_cast<float*>(S.fa);           // 2 * n_sig x 181, valid after the last pass
    for (int g0 = 0; g0 < n_sig_total; g0 += cap) {
        const int n_sig = min(cap, n_sig_total - g0);
        for (int t = G::tid(); t < n_sig * kAz; t += G::kSize) {
            const int g = t / kAz, n = t - g * kAz;
            const int ra = 2 * (g0 + g), rb = ra + 1;
            const float a = pooled_value(S, rows, T, ra, n);
            const float b = rb < T ? pooled_value(S, rows, T, rb, n) : 0.0f;
            S.fa[t] = make_float2(a, b);
        }
        G::sync();
        mark(5);
        fft_pass<8, 1, G>(S.fa, S.fb, S.tw, n_sig);
        G::sync();
        mark(6);
        fft_pass<9, 8, G>(S.fb, S.fa, S.tw, n_sig);
        G::sync();
        mark(7);
        fft_pass<5, 72, G>(S.fa, S.fb, S.tw, n_sig);
        G::sync();
        mark(8);
        // Z = FFT(a + i b): A[k] = (Z[k] + conj Z[-k]) / 2, B[k] = (Z[k] - conj Z[-k]) / 2i; one
        // thread per (signal, frequency), both magnitudes (fa is free again: the spectrum is in fb)
        for (int t = G::tid(); t < n_sig * kFreqs; t += G::kSize) {
            const int g = t / kFreqs, k = t - g * kFreqs;
            const float2* z = S.fb + g * kAz;
            const float2 p = z[k], m = z[k == 0 ? 0 : kAz - k];
            const float ar = p.x + m.x, ai = p.y - m.y;
            const float br = p.y + m.y, bi = p.x - m.x;
            mag[(2 * g) * kFreqs + k] = 0.5f * __fsqrt_rn(fmaf(ar, ar, ai * ai));
            mag[(2 * g + 1) * kFreqs + k] = 0.5f * __fsqrt_rn(fmaf(br, br, bi * bi));
        }
        G::sync();
        mark(9);
        // contiguous-frequency bin sums in ascending k: the CPU order of scatter_add_
        const int row0 = 2 * g0, row1 = min(T, 2 * (g0 + n_sig));
        for (int i = G::tid(); i < T * nb; i += G::kSize) {
            const int r = i / nb, b = i - r * nb;
            if (r < row0 || r >= row1) continue;
            const float* mr = mag + (r - row0) * kFreqs;
            float h = 0.0f;
            for (int k = S.bin_start[b], k1 = S.bin_start[b + 1]; k < k1; ++k) h += mr[k];
            S.hist[i] = h;
        }
        if (g0 + cap < n_sig_total) G::sync();   // the next batch overwrites fa / fb
    }
}

// The peer databases a launch copies every float32 descriptor row to (row row0 + scan).
struct PeerOut {
    float* ptr[NSC_MAX_PEERS];
    int n;
    long long row0;
};

// Where normalise_and_store sends one descriptor row: float32 to `out` (if set) and to row
// `peer_row` of every database in `peers` (if set), or, with out_q set (nothing else), the uint16
// wire format of quantise_and_store to out_q (q_eps, plan: the quantiser's epsilon and the
// pairwise-sum plan for D).
struct RowDest {
    float* out = nullptr;
    const PeerOut* peers = nullptr;
    long long peer_row = 0;
    unsigned short* out_q = nullptr;
    float q_eps = 0.0f;
    const SumPlan* plan = nullptr;
    __device__ int n_peers() const { return peers ? peers->n : 0; }
};

// The uint16 epilogue of normalise_and_store: the normalised row -- the float32 values the float
// path stores -- goes through HistogramQuantizer.quantize as nsc_quantize_histograms would take it
// from global memory (NumPy-order row sum, one division, half-to-even rounding, the rounding error
// added to the first largest bin) and leaves as 2 D bytes. Shared memory: the row stays in S.hist
// (integers in place, then packed to uint16 at its front), the pairwise-sum slots use S.fa (dead
// once the bin sums are in S.hist; the next scan writes it only after a group barrier), the
// per-warp partials and the row sum use S.red.
template <typename G>
__device__ __forceinline__ void quantise_and_store(const TailSmem& S, int D, bool ok, float denom, float uniform,
                                                   unsigned short* out_q, float q_eps, const SumPlan& plan) {
    const int warp = G::tid() >> 5, lane = G::tid() & 31;
    unsigned* part = reinterpret_cast<unsigned*>(S.red);          // [0, 2 warps): integer sums, first maxima
    float* sum_s = reinterpret_cast<float*>(S.red) + 2 * G::kGroupWarps;
    static_assert(4 * (2 * G::kGroupWarps + 1) <= kWarps * 8 + 16, "S.red holds the partials");
    for (int i = G::tid(); i < D; i += G::kSize) S.hist[i] = ok ? __fdiv_rn(S.hist[i], denom) : uniform;
    G::sync();                     // also: every thread has read the float path's partials in S.red
    if (warp == 0) {
        const float s = numpy_sum(S.hist, plan, reinterpret_cast<float*>(S.fa), lane);
        if (lane == 0) *sum_s = s;
    }
    G::sync();
    const float sum = *sum_s;
    const bool norm = sum > q_eps;                                 // quantization.py:144-146
    const float qden = __fadd_rn(sum, q_eps);
    // the hoisted division gives __fdiv_rn's bits for a denominator of moderate size (RowDivisor)
    const bool hoisted = norm && moderate(qden);
    const RowDivisor div(hoisted ? qden : 1.0f);
    unsigned qsum = 0, best = 0;                                   // best: (q << 16) | (0xffff - index)
    for (int i = G::tid(); i < D; i += G::kSize) {
        const float h = S.hist[i];
        const int q = quantise_value(norm ? (hoisted ? div(h) : __fdiv_rn(h, qden)) : h);
        S.hist[i] = __int_as_float(q);                             // own entry: no barrier needed
        qsum += (unsigned)q;
        best = max(best, ((unsigned)q << 16) | (0xffffu - (unsigned)i));
    }
    qsum = __reduce_add_sync(0xffffffffu, qsum);
    best = __reduce_max_sync(0xffffffffu, best);
    if (lane == 0) {
        part[warp] = qsum;
        part[G::kGroupWarps + warp] = best;
    }
    G::sync();
    qsum = 0;
    best = 0;
    for (int w = 0; w < G::kGroupWarps; ++w) {
        qsum += part[w];
        best = max(best, part[G::kGroupWarps + w]);
    }
    // quantization.py:154-167: the rounding error goes into the first largest bin
    int fix_idx = -1, fix_val = 0;
    if ((int)qsum > 0 && qsum != 65535u) {
        fix_idx = 0xffff - (int)(best & 0xffffu);
        const int v = (int)(best >> 16) + (65535 - (int)qsum);
        fix_val = v < 0 ? 0 : (v > 65535 ? 65535 : v);
    }
    const int* qs = reinterpret_cast<const int*>(S.hist);
    if ((D & 7) == 0 && (reinterpret_cast<uintptr_t>(out_q) & 15) == 0) {
        // pack in place, 8 integers (32 bytes) -> 16 bytes: unit u lands on bytes [16 u, 16 u + 16).
        // A pass writes below everything later passes read; its barrier orders its own reads (and
        // those of every earlier pass) before its writes.
        const int n_units = D >> 3;
        for (int u0 = 0; u0 < n_units; u0 += G::kSize) {
            const int u = u0 + G::tid();
            uint4 w = make_uint4(0u, 0u, 0u, 0u);
            if (u < n_units) {
                const int4 a = reinterpret_cast<const int4*>(qs)[2 * u];
                const int4 b = reinterpret_cast<const int4*>(qs)[2 * u + 1];
                const int e = 8 * u;
                auto f = [&](int q, int k) { return (unsigned)(e + k == fix_idx ? fix_val : q); };
                w = make_uint4(f(a.x, 0) | (f(a.y, 1) << 16), f(a.z, 2) | (f(a.w, 3) << 16),
                               f(b.x, 4) | (f(b.y, 5) << 16), f(b.z, 6) | (f(b.w, 7) << 16));
            }
            G::sync();
            if (u < n_units) reinterpret_cast<uint4*>(S.hist)[u] = w;
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic writes -> async-proxy reads
        G::sync();
        if (G::tid() == 0) {
            bulk_store_s2g(out_q, S.hist, (uint32_t)D * 2u);
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        }
        return;
    }
    for (int i = G::tid(); i < D; i += G::kSize) out_q[i] = (unsigned short)(i == fix_idx ? fix_val : qs[i]);
    // S.red / S.hist / S.fa are next written after the barriers at the top of the next scan
}

// h / (sum h + eps), or the uniform descriptor when sum h <= eps (spectral_encoder.py:197-202), to
// the destinations of `dst`.
template <typename P, typename G = CtaGroup>
__device__ __forceinline__ void normalise_and_store(const TailSmem& S, const P& dp, RowDest dst,
                                                    G = G()) {
    const int D = dp.T * dp.n_bins;
    const int warp = G::tid() >> 5, lane = G::tid() & 31;
    double acc = 0.0;
    for (int i = G::tid(); i < D; i += G::kSize) acc += (double)S.hist[i];   // own entries only
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, d);
    if (lane == 0) S.red[warp] = acc;
    G::sync();
    double tot = 0.0;
#pragma unroll
    for (int w = 0; w < G::kGroupWarps; ++w) tot += S.red[w];
    const float total = (float)tot;
    const bool ok = total > dp.eps;
    const float denom = __fadd_rn(total, dp.eps);
    if (dst.out_q) {
        quantise_and_store<G>(S, D, ok, denom, dp.uniform, dst.out_q, dst.q_eps, *dst.plan);
        return;
    }
    // bulk path: 16-byte granularity of size and of every destination row
    bool bulk = ((D * 4) & 15) == 0 && (dst.out == nullptr || (reinterpret_cast<uintptr_t>(dst.out) & 15) == 0);
    for (int p = 0; p < dst.n_peers(); ++p) bulk = bulk && (reinterpret_cast<uintptr_t>(dst.peers->ptr[p]) & 15) == 0;
    if (bulk) {
        for (int i = G::tid(); i < D; i += G::kSize) S.hist[i] = ok ? __fdiv_rn(S.hist[i], denom) : dp.uniform;
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic writes -> async-proxy reads
        G::sync();
        if (G::tid() == 0) {
            if (dst.out) bulk_store_s2g(dst.out, S.hist, (uint32_t)D * 4u);
            for (int p = 0; p < dst.n_peers(); ++p)
                bulk_store_s2g(dst.peers->ptr[p] + dst.peer_row * D, S.hist, (uint32_t)D * 4u);
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        }
        return;
    }
    for (int i = G::tid(); i < D; i += G::kSize) {
        const float v = ok ? __fdiv_rn(S.hist[i], denom) : dp.uniform;
        if (dst.out) dst.out[i] = v;
        for (int p = 0; p < dst.n_peers(); ++p) dst.peers->ptr[p][dst.peer_row * D + i] = v;
    }
    // S.red / S.hist are next written after the barriers at the top of the next scan
}

}  // namespace nsc
