// What both kernels of nsc_anywidth.cu share: their launch arguments and the per-point projection,
// so that the general and the fused kernel assign every point to the same pixel with the same range
// bits, and their images are bit-identical.
#pragma once
#include <math.h>

#include "nsc_internal.h"

namespace nsc {

namespace {

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

}  // namespace

}  // namespace nsc
