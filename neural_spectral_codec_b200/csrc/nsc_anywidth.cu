// The encoder for image widths other than 360 columns. The reference accepts any n_azimuth
// (src/encoding/spectral_encoder.py:35-47, range_image.py:102-127); every shipped config uses 360,
// which is what the fused kernels of nsc_encode.cu are specialised to (8*9*5 FFT plan, column
// polynomial in units of 1 degree). This file keeps the class a drop-in for the other widths with
// two kernels behind nsc_anywidth_points / nsc_anywidth_images.
//
// The GENERAL kernel favours being obviously right over being fast, and serves every call:
//   * projection with the reference's own float32 / float64 operation order (range_image.py:146-198)
//     and CUDA's atan2f, per-pixel min by a 32-bit atomicMin on the bits of the range
//     (project_point_ref, nsc_anywidth.cuh);
//   * hole interpolation ('linear' in float64 like np.interp, or 'nearest') and the empty-row fill
//     (range_image.py:15-89) on a validity snapshot;
//   * adaptive row pooling (spectral_encoder.py:171-176), a direct O(W^2) DFT per row in float64
//     with an exact-index twiddle table (any W, no plan), magnitudes, contiguous bin sums in
//     ascending frequency, L1 normalisation (spectral_encoder.py:180-202).
// One CTA per scan / image, grid-stride; images and spectra live in a per-CTA global scratch
// (L2-resident), the histogram in shared memory. ~0.1-0.3 ms per scan for W <= 1024.
//
// The FUSED kernel takes every call that computes descriptors when W has no prime factor above 13
// and its shared-memory layout fits one block (choose_fused): the image, the FFT buffers, the
// twiddles and the histogram live in shared memory, one 512-thread CTA per SM loops over the
// scans. It projects with the same project_point_ref (shared-memory atomicMin), interpolates,
// fills and pools with the general kernel's arithmetic (images and pooled rows bit-identical), and
// takes the spectrum with an fp32 mixed-radix Stockham FFT, two pooled rows per complex transform,
// bin sums straight from the spectrum and the general kernel's normalisation. The descriptors
// agree with the general kernel's to the suite's tolerances.
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include <vector>

#include "nsc_anywidth.cuh"
#include "nsc_fft.cuh"
#include "nsc_internal.h"
#include "nsc_quantize.cuh"

namespace nsc {

namespace {

constexpr int kGThreads = 256;
constexpr int kMaxWidth = 4096;

struct Scratch {
    float* img;          // E x W (key bits during the scatter)
    float* pooled;       // T x W
    float* mag;          // T x F
    double2* tw;         // W
    unsigned char* valid;  // E x W
    __host__ __device__ static size_t bytes(int E, int W, int T, int F) {
        size_t b = 0;
        b += ((size_t)E * W * 4 + 255) & ~(size_t)255;
        b += ((size_t)T * W * 4 + 255) & ~(size_t)255;
        b += ((size_t)T * F * 4 + 255) & ~(size_t)255;
        b += ((size_t)W * 16 + 255) & ~(size_t)255;
        b += ((size_t)E * W + 255) & ~(size_t)255;
        return b;
    }
    __device__ Scratch(unsigned char* base, int E, int W, int T, int F) {
        size_t o = 0;
        img = (float*)(base + o);
        o += ((size_t)E * W * 4 + 255) & ~(size_t)255;
        pooled = (float*)(base + o);
        o += ((size_t)T * W * 4 + 255) & ~(size_t)255;
        mag = (float*)(base + o);
        o += ((size_t)T * F * 4 + 255) & ~(size_t)255;
        tw = (double2*)(base + o);
        o += ((size_t)W * 16 + 255) & ~(size_t)255;
        valid = base + o;
    }
};

// The uint16 rows of nsc_anywidth_points_u16 (the kernels' Q instantiations): the quantiser's epsilon
// and NumPy's pairwise-sum plan for D = T * n_bins, built on the host once per launch.
struct QuantOut {
    unsigned short* out;       // n x T x n_bins
    float eps;
    SumPlan plan;
};

// The uint16 epilogue of both kernels: the normalised row -- the float32 values the float path
// stores -- goes through HistogramQuantizer.quantize as nsc_quantize_histograms would take it from
// global memory (NumPy-order row sum, one division, half-to-even rounding, the rounding error added
// to the first largest bin), the arithmetic of quantise_and_store (nsc_tail.cuh) with the CTA's own
// barriers. hist: the D bin sums, normalised in place and then replaced by the integers; slot:
// kSumSlots floats for warp 0's pairwise sum; part: 2 x NT / 32 words. Both lie in shared memory
// that is dead at this point; the caller's next writes to them follow its barrier at the top of the
// next scan. Every thread has read the float path's partials before the first barrier here.
// Not inlined: it runs once per scan, and inlined into the general kernel it made that kernel spill.
template <int NT>
__device__ __noinline__ void quantise_row(float* hist, int D, bool ok, float denom, float uniform,
                                             const QuantOut& q, float* slot, unsigned* part, unsigned short* out) {
    constexpr int kWarps = NT / 32;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    for (int i = tid; i < D; i += NT) hist[i] = ok ? __fdiv_rn(hist[i], denom) : uniform;
    __syncthreads();
    if (warp == 0) numpy_sum(hist, q.plan, slot, lane);
    __syncthreads();
    const float sum = slot[q.plan.result_slot];
    const bool norm = sum > q.eps;                                 // quantization.py:144-146
    const float qden = __fadd_rn(sum, q.eps);
    const bool hoisted = norm && moderate(qden);                   // __fdiv_rn's bits (RowDivisor)
    const RowDivisor div(hoisted ? qden : 1.0f);
    unsigned qsum = 0, best = 0;                                   // best: (q << 16) | (0xffff - index)
    for (int i = tid; i < D; i += NT) {
        const float h = hist[i];
        const int v = quantise_value(norm ? (hoisted ? div(h) : __fdiv_rn(h, qden)) : h);
        hist[i] = __int_as_float(v);
        qsum += (unsigned)v;
        best = max(best, ((unsigned)v << 16) | (0xffffu - (unsigned)i));
    }
    qsum = __reduce_add_sync(0xffffffffu, qsum);
    best = __reduce_max_sync(0xffffffffu, best);
    if (lane == 0) {
        part[warp] = qsum;
        part[kWarps + warp] = best;
    }
    __syncthreads();
    qsum = 0;
    best = 0;
    for (int w = 0; w < kWarps; ++w) {
        qsum += part[w];
        best = max(best, part[kWarps + w]);
    }
    int fix_idx = -1, fix_val = 0;                                 // quantization.py:154-167
    if ((int)qsum > 0 && qsum != 65535u) {
        fix_idx = 0xffff - (int)(best & 0xffffu);
        const int v = (int)(best >> 16) + (65535 - (int)qsum);
        fix_val = v < 0 ? 0 : (v > 65535 ? 65535 : v);
    }
    for (int i = tid; i < D; i += NT) out[i] = (unsigned short)(i == fix_idx ? fix_val : __float_as_int(hist[i]));
}

// ROWS: the capacity of the per-row arrays (kShortRows, or NSC_MAX_ELEVATION for taller images).
// Q: uint16 rows to q.out (and no images) instead of float32 rows to a.out; the dynamic shared
// memory then holds kSumSlots more floats after the histogram.
template <int ROWS, bool Q>
__global__ void __launch_bounds__(kGThreads)
anywidth_kernel(const __grid_constant__ AnyArgs a, const __grid_constant__ QuantOut q) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float* hist = reinterpret_cast<float*>(smem_raw);                  // T x n_bins
    __shared__ int s_nvalid[ROWS], s_src[ROWS];
    __shared__ double s_red[kGThreads / 32];
    const int tid = threadIdx.x, E = a.E, W = a.W, T = a.T, F = a.F;
    const Scratch S(a.scratch + (size_t)blockIdx.x * a.scratch_per_cta, E, W, T, F);
    unsigned* keys = reinterpret_cast<unsigned*>(S.img);
    const int D = T * a.n_bins;
    for (int m = tid; m < W; m += kGThreads) {                         // exp(-2 pi i m / W), m reduced exactly
        double s, c;
        sincospi(2.0 * (double)m / (double)W, &s, &c);
        S.tw[m] = make_double2(c, -s);
    }
    for (int item = blockIdx.x; item < a.n; item += gridDim.x) {
        __syncthreads();
        // ---- the range image
        if (a.images_in) {
            const float* src = a.images_in + (size_t)item * E * W;
            for (int i = tid; i < E * W; i += kGThreads) S.img[i] = src[i];
        } else {
            for (int i = tid; i < E * W; i += kGThreads) keys[i] = kInfBits;
            __syncthreads();
            const long long beg = a.offsets[item] - a.origin;
            const int n = (int)(a.offsets[item + 1] - a.offsets[item]);
            const float* p = a.points + beg * a.stride;
            for (int i = tid; i < n; i += kGThreads) {
                int pix;
                unsigned key;
                if (project_point_ref(p[(size_t)i * a.stride], p[(size_t)i * a.stride + 1], p[(size_t)i * a.stride + 2],
                                      a, pix, key))
                    atomicMin(keys + pix, key);                                          // np.minimum.at, :208
            }
            __syncthreads();
            for (int i = tid; i < E * W; i += kGThreads) {                              // empty -> 0, :214
                const unsigned k = keys[i];
                S.img[i] = k == kInfBits ? 0.0f : __uint_as_float(k);
            }
        }
        __syncthreads();
        if (a.images_out && a.stage == NSC_STAGE_PROJECTED)
            for (int i = tid; i < E * W; i += kGThreads) a.images_out[(size_t)item * E * W + i] = S.img[i];
        // ---- hole interpolation + empty-row fill (range_image.py:15-89)
        if (tid < E) { s_nvalid[tid] = 0; s_src[tid] = tid; }
        __syncthreads();
        if (a.interpolate) {
            for (int i = tid; i < E * W; i += kGThreads) {
                const bool v = S.img[i] > 0.0f;                                          // :35
                S.valid[i] = v;
                if (v) atomicAdd(&s_nvalid[i / W], 1);
            }
            __syncthreads();
            for (int i = tid; i < E * W; i += kGThreads) {
                const int r = i / W, x = i - r * W;
                const int cnt = s_nvalid[r];
                if (cnt == 0 || cnt == W || S.valid[i]) continue;
                const unsigned char* vr = S.valid + (size_t)r * W;
                int dl = 1, dr = 1;                       // distances to the nearest valid pixel on each side
                while (!vr[(x - dl + W) % W]) ++dl;
                while (!vr[(x + dr) % W]) ++dr;
                const int il = (x - dl + W) % W, ir = (x + dr) % W;
                const float* row = S.img + (size_t)r * W;
                if (a.interpolate == 2) {                 // 'nearest': the lower column on a tie (np.argmin)
                    S.img[i] = row[dl < dr || (dl == dr && il < ir) ? il : ir];
                } else {                                  // np.interp on the tiled abscissa, float64 (:55-64)
                    const double fl = (double)row[il], fr = (double)row[ir];
                    const double slope = __ddiv_rn(__dsub_rn(fr, fl), (double)(dl + dr));
                    S.img[i] = __double2float_rn(__dadd_rn(__dmul_rn(slope, (double)dl), fl));
                }
            }
            __syncthreads();
            if (tid < E && s_nvalid[tid] == 0) {          // :77-87, sequential in-place semantics
                int k = tid - 1;
                while (k >= 0 && s_nvalid[k] == 0) --k;
                if (k < 0) {
                    k = tid + 1;
                    while (k < E && s_nvalid[k] == 0) ++k;
                }
                if (k >= 0 && k < E) s_src[tid] = k;
            }
            __syncthreads();
        }
        if (a.images_out && a.stage == NSC_STAGE_INTERPOLATED)
            for (int i = tid; i < E * W; i += kGThreads) {
                const int r = i / W, x = i - r * W;
                a.images_out[(size_t)item * E * W + i] = S.img[(size_t)s_src[r] * W + x];
            }
        if (!Q && !a.out) continue;
        // ---- row pooling (adaptive_avg_pool2d over rows, spectral_encoder.py:171-176)
        for (int i = tid; i < T * W; i += kGThreads) {
            const int t = i / W, x = i - t * W;
            float v;
            if (E == T) {
                v = S.img[(size_t)s_src[t] * W + x];
            } else {
                const int r0 = (t * E) / T, r1 = ((t + 1) * E + T - 1) / T;
                float sum = 0.0f;
                for (int r = r0; r < r1; ++r) sum += S.img[(size_t)s_src[r] * W + x];
                v = sum / (float)(r1 - r0);
            }
            S.pooled[i] = v;
        }
        __syncthreads();
        // ---- |rfft| by a direct DFT in float64 (spectral_encoder.py:180-186)
        for (int i = tid; i < T * F; i += kGThreads) {
            const int t = i / F, k = i - t * F;
            const float* row = S.pooled + (size_t)t * W;
            double re = 0.0, im = 0.0;
            int m = 0;
            for (int x = 0; x < W; ++x) {
                const double2 w = S.tw[m];
                const double v = (double)row[x];
                re = fma(v, w.x, re);
                im = fma(v, w.y, im);
                m += k;
                if (m >= W) m -= W;
            }
            S.mag[i] = (float)sqrt(re * re + im * im);
        }
        __syncthreads();
        // ---- bin sums in ascending frequency (spectral_encoder.py:118-158), normalisation (:197-202)
        double acc = 0.0;
        for (int i = tid; i < D; i += kGThreads) {
            const int t = i / a.n_bins, b = i - t * a.n_bins;
            float h = 0.0f;
            for (int k = a.bin_start[b], k1 = a.bin_start[b + 1]; k < k1; ++k) h += S.mag[(size_t)t * F + k];
            hist[i] = h;
            acc += (double)h;
        }
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, d);
        if ((tid & 31) == 0) s_red[tid >> 5] = acc;
        __syncthreads();
        double tot = 0.0;
        for (int w = 0; w < kGThreads / 32; ++w) tot += s_red[w];
        const float total = (float)tot;
        const bool ok = total > a.eps;
        const float denom = __fadd_rn(total, a.eps);
        if (Q)
            quantise_row<kGThreads>(hist, D, ok, denom, a.uniform, q, hist + D, reinterpret_cast<unsigned*>(s_red),
                                    q.out + (size_t)item * D);
        else
            for (int i = tid; i < D; i += kGThreads)
                a.out[(size_t)item * D + i] = ok ? __fdiv_rn(hist[i], denom) : a.uniform;
    }
}

// ================================================================================================
// The fused kernel: the same stages with the image in shared memory and an fp32 FFT.
//
// A mixed-radix Stockham FFT of W points: pass p of radix R reads butterfly j's inputs
// x[j + r * W / R], r < R, multiplies input r by exp(-2 pi i k r / (NS R)) with NS the product of
// the earlier radices and k = j mod NS, takes an R-point DFT and writes output q to
// y[(j / NS) * NS * R + k + q * NS]. Radices 8, 4, 2, 3, 5 have register butterflies
// (nsc_fft.cuh); 7, 11 and 13 take the generic odd-prime butterfly. The pass code is
// __host__ __device__ so that nsc_test_anywidth_fft runs it on the CPU.
constexpr int kMaxPasses = 12;           // 4096 = 2^12

struct FftPlan {
    int n_pass;
    int radix[kMaxPasses];
};

// Radices in pass order: 8s, then a 4 or a 2 for what remains of the power of two, then the odd
// primes. False when W has a prime factor above 13.
__host__ __device__ inline bool plan_fft(int W, FftPlan* p) {
    p->n_pass = 0;
    int w = W;
    const int order[] = {8, 4, 2, 3, 5, 7, 11, 13};
    for (int r : order)
        while (w % r == 0 && p->n_pass < kMaxPasses) {
            p->radix[p->n_pass++] = r;
            w /= r;
        }
    return w == 1;
}

// exp(-2 pi i m / W) with m / W reduced exactly (as the general kernel's table), rounded to float2.
__host__ __device__ inline float2 any_twiddle(int m, int W) {
    double s, c;
#ifdef __CUDA_ARCH__
    sincospi(2.0 * (double)m / (double)W, &s, &c);
#else
    const double x = 2.0 * (double)m / (double)W;
    s = sin(M_PI * x);
    c = cos(M_PI * x);
#endif
    return make_float2((float)c, (float)-s);
}

// X[q] = sum_r a[r] w^(q r) for an odd prime R, w = exp(-2 pi i / R) = tw[W / R]: inputs paired as
// t = a[r] + a[R-r], d = a[r] - a[R-r], outputs q and R - q from one cosine and one sine sum.
template <int R>
NSC_FFT_HD void dft_odd_prime_store(float2* a, const float2* tw, int m, float2* out, int ns) {
    constexpr int H = (R - 1) / 2;
    float2 x0 = a[0];
#pragma unroll
    for (int r = 1; r <= H; ++r) {
        const float2 t = cadd(a[r], a[R - r]), d = csub(a[r], a[R - r]);
        a[r] = t;
        a[R - r] = d;
        x0 = cadd(x0, t);
    }
    out[0] = x0;
#pragma unroll 1
    for (int q = 1; q <= H; ++q) {
        float2 s = a[0], u = make_float2(0.0f, 0.0f);
        int e = 0;                                            // q r mod R
#pragma unroll
        for (int r = 1; r <= H; ++r) {
            e += q;
            if (e >= R) e -= R;
            const float2 w = tw[e * m];                       // (cos th, -sin th), th = 2 pi q r / R
            s = make_float2(fmaf(a[r].x, w.x, s.x), fmaf(a[r].y, w.x, s.y));
            u = make_float2(fmaf(-a[R - r].y, w.y, u.x), fmaf(a[R - r].x, w.y, u.y));   // -i d sin th
        }
        out[q * ns] = cadd(s, u);
        out[(R - q) * ns] = csub(s, u);
    }
}

template <int R>
NSC_FFT_HD void any_butterfly(const float2* __restrict__ x, float2* __restrict__ y, const float2* __restrict__ tw,
                              int W, int ns, int j) {
    const int m = W / R;                      // butterflies per signal
    const int blk = j / ns, k = j - blk * ns;
    const int step = k * (m / ns);            // k * W / (ns * R)
    float2 a[R];
#pragma unroll
    for (int r = 0; r < R; ++r) a[r] = x[j + r * m];
    if (k) {
#pragma unroll
        for (int r = 1; r < R; ++r) a[r] = cmul(a[r], tw[r * step]);
    }
    float2* out = y + blk * ns * R + k;
    if (R == 2) {
        out[0] = cadd(a[0], a[1]);
        out[ns] = csub(a[0], a[1]);
        return;
    }
    if (R == 7 || R == 11 || R == 13) {
        dft_odd_prime_store<R>(a, tw, m, out, ns);
        return;
    }
    if (R == 3) dft3(a[0], a[1], a[2]);
    else if (R == 4) dft4(a[0], a[1], a[2], a[3]);
    else if (R == 5) dft5(a);
    else dft8(a);
#pragma unroll
    for (int q = 0; q < R; ++q) out[q * ns] = a[q];
}

// Butterflies t0, t0 + step, ... of one pass over n_sig signals of W points each.
template <int R>
NSC_FFT_HD void any_pass(const float2* x, float2* y, const float2* tw, int W, int ns, int n_sig, int t0, int step) {
    const int m = W / R;
    for (int t = t0; t < n_sig * m; t += step) {
        const int g = t / m, j = t - g * m;
        any_butterfly<R>(x + g * W, y + g * W, tw, W, ns, j);
    }
}

__host__ __device__ inline void fft_pass(int R, const float2* x, float2* y, const float2* tw, int W, int ns, int n_sig,
                                         int t0, int step) {
    switch (R) {
        case 8: any_pass<8>(x, y, tw, W, ns, n_sig, t0, step); break;
        case 4: any_pass<4>(x, y, tw, W, ns, n_sig, t0, step); break;
        case 2: any_pass<2>(x, y, tw, W, ns, n_sig, t0, step); break;
        case 3: any_pass<3>(x, y, tw, W, ns, n_sig, t0, step); break;
        case 5: any_pass<5>(x, y, tw, W, ns, n_sig, t0, step); break;
        case 7: any_pass<7>(x, y, tw, W, ns, n_sig, t0, step); break;
        case 11: any_pass<11>(x, y, tw, W, ns, n_sig, t0, step); break;
        default: any_pass<13>(x, y, tw, W, ns, n_sig, t0, step); break;
    }
}

constexpr int kFThreads = 512;
constexpr size_t kSmemOptIn = 227 * 1024;      // one block's opt-in shared memory on sm_100
constexpr int kMaxFusedSignals = 8;            // row pairs transformed at once
constexpr int kPtsInFlight = 4;                // point loads per thread before the first projection

// Byte offsets of the fused kernel's shared memory.
struct FusedLayout {
    int n_sig;                  // complex signals (row pairs) per FFT batch
    unsigned img;               // E x W range image (key bits during the scatter)
    unsigned bits;              // E x ceil(W / 32) validity words (interpolation)
    unsigned tw;                // W float2 twiddles
    unsigned fa, fb;            // n_sig x W float2 each: the Stockham ping-pong
    unsigned hist;              // T x n_bins bin sums
    unsigned bstart;            // n_bins + 1 first frequencies
    unsigned nvalid, src;       // E ints each: valid pixels per row, source row of the empty-row fill
    unsigned red;               // kFThreads / 32 doubles
    unsigned total;
};

inline FusedLayout fused_layout(int E, int W, int T, int n_bins, int n_sig) {
    FusedLayout L;
    size_t o = 0;
    auto take = [&o](size_t bytes) {
        const unsigned at = (unsigned)o;
        o += (bytes + 15) & ~(size_t)15;
        return at;
    };
    L.n_sig = n_sig;
    L.red = take((kFThreads / 32) * 8);
    L.img = take((size_t)E * W * 4);
    L.bits = take((size_t)E * ((W + 31) / 32) * 4);
    L.tw = take((size_t)W * 8);
    L.fa = take((size_t)n_sig * W * 8);
    L.fb = take((size_t)n_sig * W * 8);
    L.hist = take((size_t)T * n_bins * 4);
    L.bstart = take(((size_t)n_bins + 1) * 4);
    L.nvalid = take((size_t)E * 4);
    L.src = take((size_t)E * 4);
    L.total = (unsigned)o;
    return L;
}

// The choice between the kernels, from the arguments alone: the fused kernel needs a descriptor
// to compute, a width whose prime factors are at most 13 and a layout with one row pair
// that fits one block's shared memory (as many row pairs per batch as fit, up to
// kMaxFusedSignals). Tuning builds (-DNSC_TUNING) take NSC_ANYWIDTH=0 to force the general kernel.
bool choose_fused(const nsc_params* p, int rows, bool want_descriptor, FusedLayout* L, FftPlan* plan) {
#ifdef NSC_TUNING
    static const bool env_fused = [] { const char* e = getenv("NSC_ANYWIDTH"); return !(e && e[0] == '0'); }();
    if (!env_fused) return false;
#endif
    if (!want_descriptor || !plan_fft(p->n_azimuth, plan)) return false;
    const int T = p->target_rows, n_sig_total = (T + 1) / 2;
    for (int s = n_sig_total < kMaxFusedSignals ? n_sig_total : kMaxFusedSignals; s >= 1; --s) {
        *L = fused_layout(rows, p->n_azimuth, T, p->n_bins, s);
        if (L->total <= kSmemOptIn) return true;
    }
    return false;
}

struct FusedArgs {
    AnyArgs a;
    FusedLayout L;
    FftPlan plan;
    QuantOut q;                 // the Q instantiation's output
};

// One scan's points into the key image: kPtsInFlight loads per thread in flight, then the
// projections and shared-memory atomicMin on the range bits. VEC4: stride 4 from a 16-byte
// aligned base, one float4 per point.
template <bool VEC4>
__device__ __forceinline__ void scatter_points(const AnyArgs& a, int item, unsigned* keys) {
    const long long beg = a.offsets[item] - a.origin;
    const int n = (int)(a.offsets[item + 1] - a.offsets[item]);
    const float* p = a.points + beg * a.stride;
    for (int i0 = threadIdx.x; i0 < n; i0 += kPtsInFlight * kFThreads) {
        float x[kPtsInFlight], y[kPtsInFlight], z[kPtsInFlight];
#pragma unroll
        for (int u = 0; u < kPtsInFlight; ++u) {
            const int i = i0 + u * kFThreads;
            if (i < n) {
                if (VEC4) {
                    const float4 v = reinterpret_cast<const float4*>(p)[i];
                    x[u] = v.x, y[u] = v.y, z[u] = v.z;
                } else {
                    const float* q = p + (size_t)i * a.stride;
                    x[u] = q[0], y[u] = q[1], z[u] = q[2];
                }
            }
        }
#pragma unroll
        for (int u = 0; u < kPtsInFlight; ++u) {
            int pix;
            unsigned key;
            if (i0 + u * kFThreads < n && project_point_ref(x[u], y[u], z[u], a, pix, key)) atomicMin(keys + pix, key);
        }
    }
}

// The general kernel's pooling arithmetic (row t of the pooled image at column x).
__device__ __forceinline__ float pooled_at(const float* img, const int* src, int E, int T, int W, int t, int x) {
    if (E == T) return img[src[t] * W + x];
    const int r0 = (t * E) / T, r1 = ((t + 1) * E + T - 1) / T;
    float sum = 0.0f;
    for (int r = r0; r < r1; ++r) sum += img[src[r] * W + x];
    return sum / (float)(r1 - r0);
}

// Nearest set bit strictly left / right of column x in a circular row of W bits with at least one
// set bit other than x's: the column the general kernel's pixel-by-pixel walk stops at.
__device__ __forceinline__ int valid_left(const unsigned* row, int W, int x) {
    int c = x == 0 ? W - 1 : x - 1;
    for (;;) {
        const unsigned v = row[c >> 5] & (0xffffffffu >> (31 - (c & 31)));
        if (v) return (c & ~31) + 31 - __clz(v);
        c = (c & ~31) - 1;
        if (c < 0) c = W - 1;
    }
}
__device__ __forceinline__ int valid_right(const unsigned* row, int W, int x) {
    int c = x == W - 1 ? 0 : x + 1;
    for (;;) {
        const unsigned v = row[c >> 5] & (0xffffffffu << (c & 31));
        if (v) return (c & ~31) + __ffs(v) - 1;
        c = (c & ~31) + 32;
        if (c >= W) c = 0;
    }
}

// Q: uint16 rows to f.q.out instead of float32 rows to a.out. The epilogue's pairwise-sum slots go
// in fa, dead once the bin sums are in hist: a row of D <= T (W / 2 + 1) elements, T <= 64, needs at
// most 2 ceil(D / 57) - 1 slots (leaves of more than 57 elements), fewer bytes than fa's W x 8.
template <bool VEC4, bool Q>
__global__ void __launch_bounds__(kFThreads, 1)
anywidth_fused_kernel(const __grid_constant__ FusedArgs f) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const AnyArgs& a = f.a;
    const FusedLayout& L = f.L;
    float* img = reinterpret_cast<float*>(smem_raw + L.img);
    unsigned* keys = reinterpret_cast<unsigned*>(img);
    unsigned* bits = reinterpret_cast<unsigned*>(smem_raw + L.bits);
    float2* tw = reinterpret_cast<float2*>(smem_raw + L.tw);
    float2* fa = reinterpret_cast<float2*>(smem_raw + L.fa);
    float2* fb = reinterpret_cast<float2*>(smem_raw + L.fb);
    float* hist = reinterpret_cast<float*>(smem_raw + L.hist);
    int* bstart = reinterpret_cast<int*>(smem_raw + L.bstart);
    int* s_nvalid = reinterpret_cast<int*>(smem_raw + L.nvalid);
    int* s_src = reinterpret_cast<int*>(smem_raw + L.src);
    double* s_red = reinterpret_cast<double*>(smem_raw + L.red);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int E = a.E, W = a.W, T = a.T, nb = a.n_bins, D = T * nb, EW = E * W;
    const int words = (W + 31) >> 5;
    for (int m = tid; m < W; m += kFThreads) tw[m] = any_twiddle(m, W);
    for (int b = tid; b <= nb; b += kFThreads) bstart[b] = a.bin_start[b];
    for (int item = blockIdx.x; item < a.n; item += gridDim.x) {
        __syncthreads();
        // ---- the range image
        if (a.images_in) {
            const float* src = a.images_in + (size_t)item * EW;
            for (int i = tid; i < EW; i += kFThreads) img[i] = src[i];
        } else {
            for (int i = tid; i < EW; i += kFThreads) keys[i] = kInfBits;
            __syncthreads();
            scatter_points<VEC4>(a, item, keys);
            __syncthreads();
            for (int i = tid; i < EW; i += kFThreads) {                                // empty -> 0
                const unsigned k = keys[i];
                img[i] = k == kInfBits ? 0.0f : __uint_as_float(k);
            }
        }
        if (tid < E) { s_nvalid[tid] = 0; s_src[tid] = tid; }
        __syncthreads();
        if (a.images_out && a.stage == NSC_STAGE_PROJECTED)
            for (int i = tid; i < EW; i += kFThreads) a.images_out[(size_t)item * EW + i] = img[i];
        // ---- hole interpolation + empty-row fill: the general kernel's arithmetic on a bit snapshot
        if (a.interpolate) {
            for (int w = warp; w < E * words; w += kFThreads / 32) {
                const int r = w / words, x = (w - r * words) * 32 + lane;
                const unsigned v = __ballot_sync(0xffffffffu, x < W && img[r * W + x] > 0.0f);
                if (lane == 0) {
                    bits[w] = v;
                    if (v) atomicAdd(&s_nvalid[r], __popc(v));
                }
            }
            __syncthreads();
            for (int i = tid; i < EW; i += kFThreads) {
                const int r = i / W, x = i - r * W;
                const int cnt = s_nvalid[r];
                const unsigned* vr = bits + r * words;
                if (cnt == 0 || cnt == W || ((vr[x >> 5] >> (x & 31)) & 1u)) continue;
                const int il = valid_left(vr, W, x), ir = valid_right(vr, W, x);
                const int dl = x - il + (il > x ? W : 0), dr = ir - x + (ir < x ? W : 0);
                const float* row = img + r * W;
                if (a.interpolate == 2) {
                    img[i] = row[dl < dr || (dl == dr && il < ir) ? il : ir];
                } else {
                    const double fl = (double)row[il], fr = (double)row[ir];
                    const double slope = __ddiv_rn(__dsub_rn(fr, fl), (double)(dl + dr));
                    img[i] = __double2float_rn(__dadd_rn(__dmul_rn(slope, (double)dl), fl));
                }
            }
            __syncthreads();
            if (tid < E && s_nvalid[tid] == 0) {
                int k = tid - 1;
                while (k >= 0 && s_nvalid[k] == 0) --k;
                if (k < 0) {
                    k = tid + 1;
                    while (k < E && s_nvalid[k] == 0) ++k;
                }
                if (k >= 0 && k < E) s_src[tid] = k;
            }
            __syncthreads();
        }
        if (a.images_out && a.stage == NSC_STAGE_INTERPOLATED)
            for (int i = tid; i < EW; i += kFThreads) {
                const int r = i / W, x = i - r * W;
                a.images_out[(size_t)item * EW + i] = img[s_src[r] * W + x];
            }
        // ---- pooled rows 2g, 2g + 1 -> one complex FFT -> split by conjugate symmetry -> bin sums
        const int n_sig_total = (T + 1) / 2;
        for (int g0 = 0; g0 < n_sig_total; g0 += L.n_sig) {
            const int n_sig = min(L.n_sig, n_sig_total - g0);
            for (int t = tid; t < n_sig * W; t += kFThreads) {
                const int g = t / W, x = t - g * W;
                const int ra = 2 * (g0 + g), rb = ra + 1;
                fa[t] = make_float2(pooled_at(img, s_src, E, T, W, ra, x),
                                    rb < T ? pooled_at(img, s_src, E, T, W, rb, x) : 0.0f);
            }
            __syncthreads();
            float2 *x = fa, *y = fb;
            for (int p = 0, ns = 1; p < f.plan.n_pass; ++p) {
                const int R = f.plan.radix[p];
                fft_pass(R, x, y, tw, W, ns, n_sig, tid, kFThreads);
                __syncthreads();
                float2* t = x;
                x = y;
                y = t;
                ns *= R;
            }
            // Z = FFT(a + i b): |A[k]| = |Z[k] + conj Z[-k]| / 2, |B[k]| = |Z[k] - conj Z[-k]| / 2,
            // summed over each bin's frequencies in ascending k as they are computed
            for (int i = tid; i < n_sig * 2 * nb; i += kFThreads) {
                const int g = i / (2 * nb), rem = i - g * 2 * nb, h = rem >= nb, b = rem - h * nb;
                const int row = 2 * (g0 + g) + h;
                if (row >= T) continue;
                const float2* z = x + g * W;
                float s = 0.0f;
                for (int k = bstart[b], k1 = bstart[b + 1]; k < k1; ++k) {
                    const float2 p = z[k], m = z[k == 0 ? 0 : W - k];
                    const float re = h ? p.y + m.y : p.x + m.x, im = h ? p.x - m.x : p.y - m.y;
                    s += 0.5f * __fsqrt_rn(fmaf(re, re, im * im));
                }
                hist[row * nb + b] = s;
            }
            __syncthreads();
        }
        // ---- normalisation: the general kernel's rule (float64 total, __fdiv_rn by total + eps)
        double acc = 0.0;
        for (int i = tid; i < D; i += kFThreads) acc += (double)hist[i];
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, d);
        if (lane == 0) s_red[warp] = acc;
        __syncthreads();
        double tot = 0.0;
        for (int w = 0; w < kFThreads / 32; ++w) tot += s_red[w];
        const float total = (float)tot;
        const bool ok = total > a.eps;
        const float denom = __fadd_rn(total, a.eps);
        if (Q)
            quantise_row<kFThreads>(hist, D, ok, denom, a.uniform, f.q, reinterpret_cast<float*>(fa),
                                    reinterpret_cast<unsigned*>(s_red), f.q.out + (size_t)item * D);
        else
            for (int i = tid; i < D; i += kFThreads)
                a.out[(size_t)item * D + i] = ok ? __fdiv_rn(hist[i], denom) : a.uniform;
    }
}

int validate_any(const nsc_params* p) {
    if (!p) return NSC_ERR_NULL_POINTER;
    if (p->struct_size != (int32_t)sizeof(nsc_params)) return NSC_ERR_BAD_STRUCT;
    if (p->n_azimuth < 2 || p->n_azimuth > kMaxWidth) return NSC_ERR_BAD_PARAMS;
    if (p->n_elevation < 1 || p->n_elevation > max_rows(p)) return NSC_ERR_BAD_PARAMS;
    if (p->target_rows < 1 || p->target_rows > NSC_MAX_TARGET_ROWS) return NSC_ERR_BAD_PARAMS;
    if (p->n_bins < 1 || p->n_bins > p->n_azimuth / 2 + 1) return NSC_ERR_BAD_PARAMS;
    if ((long long)p->target_rows * p->n_bins > NSC_MAX_DESCRIPTOR) return NSC_ERR_BAD_PARAMS;
    if (!(p->min_range >= 0.0f) || !(p->max_range >= p->min_range) || !isfinite(p->max_range)) return NSC_ERR_BAD_PARAMS;
    if (!isfinite(p->el_min_rad) || !isfinite(p->el_max_rad) || !(p->el_max_rad > p->el_min_rad)) return NSC_ERR_BAD_PARAMS;
    if (!(p->epsilon >= 0.0f) || !isfinite(p->epsilon)) return NSC_ERR_BAD_PARAMS;
    return NSC_OK;
}

int grid_for(int n, int* grid, int* sms_out = nullptr) {
    int dev = 0, sms = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (e != cudaSuccess) return record_cuda(e);
    *grid = n < 2 * sms ? n : 2 * sms;
    if (sms_out) *sms_out = sms;
    return NSC_OK;
}
constexpr int kMaxGrid = 1024;     // bounds the workspace without asking the device

size_t table_bytes(const nsc_params* p) { return (((size_t)p->n_bins + 1) * 4 + 255) & ~(size_t)255; }

// The first frequency of every bin from the host table (n_azimuth / 2 + 1 entries), into start if
// given: NSC_ERR_BAD_LUT for a table that decreases or leaves [0, n_bins).
int bin_starts(const nsc_params* p, const int32_t* h_lut, int* start) {
    const int F = p->n_azimuth / 2 + 1;
    int prev = 0, b = 0;
    for (int k = 0; k < F; ++k) {
        if (h_lut[k] < prev || h_lut[k] >= p->n_bins) return NSC_ERR_BAD_LUT;
        prev = h_lut[k];
        if (start)
            while (b <= h_lut[k]) start[b++] = k;
    }
    if (start)
        while (b <= p->n_bins) start[b++] = F;
    return NSC_OK;
}

// q: the uint16 rows of nsc_anywidth_points_u16 (a.out null), or null.
int run(AnyArgs& a, const nsc_params* p, int rows, const int32_t* h_lut, QuantOut* q, void* ws, size_t ws_bytes,
        cudaStream_t s) {
    a.E = rows;
    a.W = p->n_azimuth;
    a.T = p->target_rows;
    a.F = p->n_azimuth / 2 + 1;
    a.n_bins = p->n_bins;
    a.min_range = p->min_range;
    a.max_range = p->max_range;
    a.eps = p->epsilon;
    a.uniform = 1.0f / (float)(a.T * a.n_bins);
    a.el_min = p->el_min_rad;
    a.el_max = p->el_max_rad;
    int grid = 0, sms = 0;
    int st = grid_for(a.n, &grid, &sms);
    if (st != NSC_OK) return st;
    if (grid > kMaxGrid) grid = kMaxGrid;
    const size_t per = Scratch::bytes(a.E, a.W, a.T, a.F);
    if (!ws || ws_bytes < table_bytes(p) + per * (size_t)grid) return NSC_ERR_WORKSPACE;
    a.scratch = (unsigned char*)ws + table_bytes(p);
    a.scratch_per_cta = per;
    a.bin_start = (const int*)ws;
    const bool want = a.out || q;
    if (want) {
        if (!h_lut) return NSC_ERR_NULL_POINTER;
        std::vector<int> start(a.n_bins + 1);
        const int st_lut = bin_starts(p, h_lut, start.data());
        if (st_lut != NSC_OK) return st_lut;
        // pageable source: the runtime stages it before returning, so the vector may go away
        cudaError_t e = cudaMemcpyAsync(ws, start.data(), start.size() * 4, cudaMemcpyHostToDevice, s);
        if (e != cudaSuccess) return record_cuda(e);
    }
    QuantOut qo;
    memset(&qo, 0, sizeof(qo));
    if (q) {
        qo = *q;
        st = build_plan(a.T * a.n_bins, &qo.plan);        // D <= NSC_MAX_DESCRIPTOR: always fits
        if (st != NSC_OK) return st;
    }
    // the same kernel for both output types: the uint16 rows quantise the floats the float call writes
    FusedArgs f;
    if (choose_fused(p, rows, want, &f.L, &f.plan)) {
        // as many CTAs as fit on every SM, each looping over scans / images
        f.a = a;
        f.q = qo;
        const bool vec4 = a.points && a.stride == 4 && ((uintptr_t)a.points & 15) == 0;
        const auto kernel = q ? (vec4 ? anywidth_fused_kernel<true, true> : anywidth_fused_kernel<false, true>)
                              : (vec4 ? anywidth_fused_kernel<true, false> : anywidth_fused_kernel<false, false>);
        cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)f.L.total);
        int per_sm = 0;
        if (e == cudaSuccess) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, kFThreads, f.L.total);
        if (e != cudaSuccess) return record_cuda(e);
        const long long fgrid = (long long)sms * (per_sm > 0 ? per_sm : 1);
        kernel<<<(int)(a.n < fgrid ? a.n : fgrid), kFThreads, f.L.total, s>>>(f);
        return record_cuda(cudaGetLastError());
    }
    const size_t smem = ((size_t)a.T * a.n_bins + (q ? kSumSlots : 0)) * 4;
    const auto kernel = q ? (a.E > kShortRows ? anywidth_kernel<NSC_MAX_ELEVATION, true> : anywidth_kernel<kShortRows, true>)
                          : (a.E > kShortRows ? anywidth_kernel<NSC_MAX_ELEVATION, false>
                                              : anywidth_kernel<kShortRows, false>);
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return record_cuda(e);
    kernel<<<grid, kGThreads, smem, s>>>(a, qo);
    return record_cuda(cudaGetLastError());
}

}  // namespace

int check_anywidth(const nsc_params* p, const int32_t* h_lut) {
    const int st = validate_any(p);
    if (st != NSC_OK) return st;
    if (!h_lut) return NSC_ERR_NULL_POINTER;
    return bin_starts(p, h_lut, nullptr);
}

}  // namespace nsc

using namespace nsc;

extern "C" {

size_t nsc_anywidth_workspace_bytes(int n, int rows, const nsc_params* p) {
    if (n < 0 || validate_any(p) != NSC_OK || rows < 1 || rows > max_rows(p)) return 0;
    const int grid = n < kMaxGrid ? (n < 1 ? 1 : n) : kMaxGrid;
    return table_bytes(p) + Scratch::bytes(rows, p->n_azimuth, p->target_rows, p->n_azimuth / 2 + 1) * (size_t)grid;
}

int nsc_test_anywidth_path(const nsc_params* p, int rows, int want_descriptor) {
    const int st = validate_any(p);
    if (st != NSC_OK) return st;
    if (rows < 1 || rows > max_rows(p)) return NSC_ERR_BAD_PARAMS;
    FusedLayout L;
    FftPlan plan;
    return choose_fused(p, rows, want_descriptor != 0, &L, &plan) ? 1 : 0;
}

int nsc_test_anywidth_fft(int W, const float* h_in, float* h_out) {
    FftPlan plan;
    if (W < 2 || W > kMaxWidth || !plan_fft(W, &plan)) return NSC_ERR_BAD_PARAMS;
    if (!h_in || !h_out) return NSC_ERR_NULL_POINTER;
    std::vector<float2> tw(W), x(W), y(W);
    for (int m = 0; m < W; ++m) tw[m] = any_twiddle(m, W);
    for (int i = 0; i < W; ++i) x[i] = make_float2(h_in[2 * i], h_in[2 * i + 1]);
    for (int p = 0, ns = 1; p < plan.n_pass; ++p) {
        fft_pass(plan.radix[p], x.data(), y.data(), tw.data(), W, ns, 1, 0, 1);
        x.swap(y);
        ns *= plan.radix[p];
    }
    for (int i = 0; i < W; ++i) {
        h_out[2 * i] = x[i].x;
        h_out[2 * i + 1] = x[i].y;
    }
    return NSC_OK;
}

int nsc_anywidth_points(const float* d_points, int point_stride, const int64_t* d_offsets, int64_t point_origin,
                        int n_scans, const nsc_params* p, const int32_t* h_lut, float* d_out, float* d_images,
                        int stage, void* d_workspace, size_t workspace_bytes, void* stream) {
    int st = validate_any(p);
    if (st != NSC_OK) return st;
    if (n_scans < 0) return NSC_ERR_BAD_COUNT;
    if (point_stride != 3 && point_stride != 4) return NSC_ERR_BAD_STRIDE;
    if (stage != NSC_STAGE_PROJECTED && stage != NSC_STAGE_INTERPOLATED) return NSC_ERR_BAD_PARAMS;
    if (n_scans == 0) return NSC_OK;
    if (!d_offsets || (!d_out && !d_images)) return NSC_ERR_NULL_POINTER;
    AnyArgs a;
    memset(&a, 0, sizeof(a));
    a.points = d_points;
    a.stride = point_stride;
    a.offsets = (const long long*)d_offsets;
    a.origin = point_origin;
    a.n = n_scans;
    a.interpolate = (d_out ? p->interpolate_empty != 0 : stage == NSC_STAGE_INTERPOLATED) ? 1 : 0;
    if (d_out && d_images && stage == NSC_STAGE_INTERPOLATED && !a.interpolate) return NSC_ERR_BAD_PARAMS;
    a.out = d_out;
    a.images_out = d_images;
    a.stage = stage;
    return run(a, p, p->n_elevation, h_lut, nullptr, d_workspace, workspace_bytes, (cudaStream_t)stream);
}

int nsc_anywidth_points_u16(const float* d_points, int point_stride, const int64_t* d_offsets, int64_t point_origin,
                            int n_scans, const nsc_params* p, const int32_t* h_lut, float q_epsilon, uint16_t* d_out,
                            void* d_workspace, size_t workspace_bytes, void* stream) {
    int st = validate_any(p);
    if (st != NSC_OK) return st;
    if (n_scans < 0) return NSC_ERR_BAD_COUNT;
    if (point_stride != 3 && point_stride != 4) return NSC_ERR_BAD_STRIDE;
    if (n_scans == 0) return NSC_OK;
    if (!d_offsets || !d_out) return NSC_ERR_NULL_POINTER;
    AnyArgs a;
    memset(&a, 0, sizeof(a));
    a.points = d_points;
    a.stride = point_stride;
    a.offsets = (const long long*)d_offsets;
    a.origin = point_origin;
    a.n = n_scans;
    a.interpolate = p->interpolate_empty != 0 ? 1 : 0;
    a.stage = NSC_STAGE_INTERPOLATED;
    QuantOut q;
    q.out = d_out;
    q.eps = q_epsilon;
    return run(a, p, p->n_elevation, h_lut, &q, d_workspace, workspace_bytes, (cudaStream_t)stream);
}

int nsc_anywidth_images(const float* d_images_in, int n_images, int rows, const nsc_params* p, const int32_t* h_lut,
                        int interp_method, float* d_out, float* d_images_out, void* d_workspace,
                        size_t workspace_bytes, void* stream) {
    int st = validate_any(p);
    if (st != NSC_OK) return st;
    if (n_images < 0) return NSC_ERR_BAD_COUNT;
    if (rows < 1 || rows > max_rows(p)) return NSC_ERR_BAD_PARAMS;
    if (interp_method != -1 && interp_method != NSC_INTERP_LINEAR && interp_method != NSC_INTERP_NEAREST)
        return NSC_ERR_BAD_PARAMS;
    if (n_images == 0) return NSC_OK;
    if (!d_images_in || (!d_out && !d_images_out)) return NSC_ERR_NULL_POINTER;
    AnyArgs a;
    memset(&a, 0, sizeof(a));
    a.images_in = d_images_in;
    a.n = n_images;
    a.interpolate = interp_method == -1 ? 0 : interp_method == NSC_INTERP_NEAREST ? 2 : 1;
    a.out = d_out;
    a.images_out = d_images_out;
    a.stage = NSC_STAGE_INTERPOLATED;
    return run(a, p, rows, h_lut, nullptr, d_workspace, workspace_bytes, (cudaStream_t)stream);
}

}  // extern "C"
