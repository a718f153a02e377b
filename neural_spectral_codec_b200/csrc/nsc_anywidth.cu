// The encoder for image widths other than 360 columns. The reference accepts any n_azimuth
// (src/encoding/spectral_encoder.py:35-47, range_image.py:102-127); every shipped config uses 360,
// which is what the fused kernels of nsc_encode.cu are specialised to (8*9*5 FFT plan, column
// polynomial in units of 1 degree). This file keeps the class a drop-in for the other widths with
// ONE general kernel that favours being obviously right over being fast:
//   * projection with the reference's own float32 / float64 operation order (range_image.py:146-198)
//     and CUDA's atan2f, per-pixel min by a 32-bit atomicMin on the bits of the range;
//   * hole interpolation ('linear' in float64 like np.interp, or 'nearest') and the empty-row fill
//     (range_image.py:15-89) on a validity snapshot;
//   * adaptive row pooling (spectral_encoder.py:171-176), a direct O(W^2) DFT per row in float64
//     with an exact-index twiddle table (any W, no plan), magnitudes, contiguous bin sums in
//     ascending frequency, L1 normalisation (spectral_encoder.py:180-202).
// One CTA per scan / image, grid-stride; images and spectra live in a per-CTA global scratch
// (L2-resident), the histogram in shared memory. ~0.1-0.3 ms per scan for W <= 1024.
#include <math.h>
#include <string.h>

#include <vector>

#include "nsc_internal.h"

namespace nsc {

namespace {

constexpr int kGThreads = 256;
constexpr int kMaxWidth = 4096;

struct AnyArgs {
    // input: points (CSR) or images
    const float* points;
    int stride;
    const long long* offsets;
    long long origin;
    const float* images_in;    // n x rows x W, or null
    int n;                     // scans or images
    int E, W, T, F, n_bins;
    int interpolate;           // 0 none, 1 linear, 2 nearest
    float min_range, max_range, eps, uniform;
    double el_min, el_max;
    const int* bin_start;      // n_bins + 1 first frequencies (device)
    float* out;                // n x T x n_bins, or null
    float* images_out;         // n x E x W, or null
    int stage;                 // NSC_STAGE_PROJECTED / NSC_STAGE_INTERPOLATED for images_out
    unsigned char* scratch;    // per-CTA regions
    size_t scratch_per_cta;
};

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

// One point -> (pixel, range bits), range_image.py:146-198 in the reference's arithmetic:
// float32 for range / azimuth / elevation / column, float64 for the row.
__device__ __forceinline__ bool project_point_ref(float x, float y, float z, const AnyArgs& a, int& pix,
                                                  unsigned& key) {
    if (!(isfinite(x) && isfinite(y) && isfinite(z))) return false;                       // :151
    const float x2 = fminf(fmaxf(__fmul_rn(x, x), 0.0f), 1e10f), y2 = fminf(fmaxf(__fmul_rn(y, y), 0.0f), 1e10f),
                z2 = fminf(fmaxf(__fmul_rn(z, z), 0.0f), 1e10f);                          // :159-161
    const float rho2 = __fadd_rn(x2, y2);
    const float rng = __fsqrt_rn(__fadd_rn(rho2, z2));                                    // :162
    if (!(rng >= a.min_range && rng <= a.max_range) || !isfinite(rng)) return false;      // :174
    const float pi_f = 3.14159265358979323846f, two_pi_f = 6.28318530717958647692f;
    float az = __fadd_rn(atan2f(y, x), pi_f);                                             // :166-167
    if (az >= two_pi_f) az = __fsub_rn(az, two_pi_f);                                     // (az + pi) % 2 pi
    const float el = atan2f(z, __fsqrt_rn(rho2));                                         // :170-171
    const double frac = ((double)el - a.el_min) / (a.el_max - a.el_min);                  // :186 (float64)
    double rowd = floor(frac * (double)a.E);
    int row = rowd < 0.0 ? 0 : rowd > (double)(a.E - 1) ? a.E - 1 : (int)rowd;            // :187-191
    const float cold = floorf(__fmul_rn(__fdiv_rn(az, two_pi_f), (float)a.W));            // :194
    int col = cold < 0.0f ? 0 : cold > (float)(a.W - 1) ? a.W - 1 : (int)cold;            // :195-198
    pix = row * a.W + col;
    key = __float_as_uint(rng);
    return true;
}

// ROWS: the capacity of the per-row arrays (kShortRows, or NSC_MAX_ELEVATION for taller images).
template <int ROWS>
__global__ void __launch_bounds__(kGThreads)
anywidth_kernel(const __grid_constant__ AnyArgs a) {
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
        if (!a.out) continue;
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
        for (int i = tid; i < D; i += kGThreads)
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

int grid_for(int n, int* grid) {
    int dev = 0, sms = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (e != cudaSuccess) return record_cuda(e);
    *grid = n < 2 * sms ? n : 2 * sms;
    return NSC_OK;
}
constexpr int kMaxGrid = 1024;     // bounds the workspace without asking the device

size_t table_bytes(const nsc_params* p) { return (((size_t)p->n_bins + 1) * 4 + 255) & ~(size_t)255; }

int run(AnyArgs& a, const nsc_params* p, int rows, const int32_t* h_lut, void* ws, size_t ws_bytes, cudaStream_t s) {
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
    int grid = 0;
    int st = grid_for(a.n, &grid);
    if (st != NSC_OK) return st;
    if (grid > kMaxGrid) grid = kMaxGrid;
    const size_t per = Scratch::bytes(a.E, a.W, a.T, a.F);
    if (!ws || ws_bytes < table_bytes(p) + per * (size_t)grid) return NSC_ERR_WORKSPACE;
    a.scratch = (unsigned char*)ws + table_bytes(p);
    a.scratch_per_cta = per;
    a.bin_start = (const int*)ws;
    if (a.out) {
        if (!h_lut) return NSC_ERR_NULL_POINTER;
        std::vector<int> start(a.n_bins + 1);
        int prev = 0, b = 0;
        for (int k = 0; k < a.F; ++k) {
            if (h_lut[k] < prev || h_lut[k] >= a.n_bins) return NSC_ERR_BAD_LUT;
            prev = h_lut[k];
            while (b <= h_lut[k]) start[b++] = k;
        }
        while (b <= a.n_bins) start[b++] = a.F;
        // pageable source: the runtime stages it before returning, so the vector may go away
        cudaError_t e = cudaMemcpyAsync(ws, start.data(), start.size() * 4, cudaMemcpyHostToDevice, s);
        if (e != cudaSuccess) return record_cuda(e);
    }
    const size_t smem = (size_t)a.T * a.n_bins * 4;
    const auto kernel = a.E > kShortRows ? anywidth_kernel<NSC_MAX_ELEVATION> : anywidth_kernel<kShortRows>;
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return record_cuda(e);
    kernel<<<grid, kGThreads, smem, s>>>(a);
    return record_cuda(cudaGetLastError());
}

}  // namespace

}  // namespace nsc

using namespace nsc;

extern "C" {

size_t nsc_anywidth_workspace_bytes(int n, int rows, const nsc_params* p) {
    if (n < 0 || validate_any(p) != NSC_OK || rows < 1 || rows > max_rows(p)) return 0;
    const int grid = n < kMaxGrid ? (n < 1 ? 1 : n) : kMaxGrid;
    return table_bytes(p) + Scratch::bytes(rows, p->n_azimuth, p->target_rows, p->n_azimuth / 2 + 1) * (size_t)grid;
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
    return run(a, p, p->n_elevation, h_lut, d_workspace, workspace_bytes, (cudaStream_t)stream);
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
    return run(a, p, rows, h_lut, d_workspace, workspace_bytes, (cudaStream_t)stream);
}

}  // extern "C"
