// Host-side constants of the encoder: parameter validation, the float32 range-filter
// thresholds, the atan polynomials, the row thresholds and the bin table. Everything here
// runs once per distinct (nsc_params, lut) and is memoised.
#include <math.h>
#include <string.h>

#include <mutex>
#include <vector>

#include "nsc_point.h"

namespace nsc {

int validate_params(const nsc_params* p) {
    if (!p) return NSC_ERR_NULL_POINTER;
    if (p->struct_size != (int32_t)sizeof(nsc_params)) return NSC_ERR_BAD_STRUCT;
    if (p->n_azimuth != NSC_N_AZIMUTH) return NSC_ERR_BAD_PARAMS;
    if (p->n_elevation < 1 || p->n_elevation > max_rows(p)) return NSC_ERR_BAD_PARAMS;
    if (p->target_rows < 1 || p->target_rows > NSC_MAX_TARGET_ROWS) return NSC_ERR_BAD_PARAMS;
    if (p->n_bins < 1 || p->n_bins > NSC_MAX_BINS) return NSC_ERR_BAD_PARAMS;
    if ((long long)p->target_rows * p->n_bins > NSC_MAX_DESCRIPTOR) return NSC_ERR_BAD_PARAMS;
    if (!(p->min_range >= 0.0f) || !(p->max_range >= p->min_range) || !isfinite(p->max_range))
        return NSC_ERR_BAD_PARAMS;
    if (!isfinite(p->el_min_rad) || !isfinite(p->el_max_rad) || !(p->el_max_rad > p->el_min_rad))
        return NSC_ERR_BAD_PARAMS;
    if (!(p->epsilon >= 0.0f) || !isfinite(p->epsilon)) return NSC_ERR_BAD_PARAMS;
    return NSC_OK;
}

namespace {

float bits_to_float(uint32_t b) {
    float f;
    memcpy(&f, &b, 4);
    return f;
}

// Smallest float32 s >= 0 with sqrtf(s) >= r (sqrtf is correctly rounded and monotone).
float sqrt_preimage_lo(float r) {
    uint32_t lo = 0, hi = kInfBits;  // answer in [lo, hi]
    while (lo < hi) {
        uint32_t mid = lo + (hi - lo) / 2;
        if (sqrtf(bits_to_float(mid)) >= r) hi = mid; else lo = mid + 1;
    }
    return bits_to_float(lo);
}
// Largest finite float32 s with sqrtf(s) <= r.
float sqrt_preimage_hi(float r) {
    uint32_t lo = 0, hi = kInfBits - 1;
    while (lo < hi) {
        uint32_t mid = lo + (hi - lo + 1) / 2;
        if (sqrtf(bits_to_float(mid)) <= r) lo = mid; else hi = mid - 1;
    }
    return bits_to_float(lo);
}

// Weighted least squares by modified Gram-Schmidt in long double: min sum w_i (A c - b)_i^2.
void wls(const std::vector<long double>& A, const std::vector<long double>& b,
         const std::vector<long double>& w, int m, int n, long double* c) {
    std::vector<long double> Q(A.size()), R(n * n, 0.0L), qtb(n);
    for (int i = 0; i < m; ++i)
        for (int j = 0; j < n; ++j) Q[i * n + j] = A[i * n + j] * w[i];
    std::vector<long double> rhs(m);
    for (int i = 0; i < m; ++i) rhs[i] = b[i] * w[i];
    for (int j = 0; j < n; ++j) {
        for (int k = 0; k < j; ++k) {
            long double d = 0;
            for (int i = 0; i < m; ++i) d += Q[i * n + k] * Q[i * n + j];
            R[k * n + j] = d;
            for (int i = 0; i < m; ++i) Q[i * n + j] -= d * Q[i * n + k];
        }
        long double nrm = 0;
        for (int i = 0; i < m; ++i) nrm += Q[i * n + j] * Q[i * n + j];
        nrm = sqrtl(nrm);
        R[j * n + j] = nrm;
        for (int i = 0; i < m; ++i) Q[i * n + j] /= nrm;
    }
    for (int j = 0; j < n; ++j) {
        long double d = 0;
        for (int i = 0; i < m; ++i) d += Q[i * n + j] * rhs[i];
        qtb[j] = d;
    }
    for (int j = n - 1; j >= 0; --j) {
        long double v = qtb[j];
        for (int k = j + 1; k < n; ++k) v -= R[j * n + k] * c[k];
        c[j] = v / R[j * n + j];
    }
}

// Near-minimax odd polynomial: scale * atan(u) ~= u * P(u^2) on [0, umax] (Lawson-style
// reweighted least squares on Chebyshev nodes). Returns the max error in radians of the
// float32 Horner/FMA evaluation the kernel performs.
double fit_atan(double umax, int n, double scale, float* coef) {
    const int m = 768;
    std::vector<long double> A(m * n), b(m), w(m, 1.0L);
    for (int i = 0; i < m; ++i) {
        long double v = 0.5L - 0.5L * cosl(3.14159265358979323846264338327950288L * (i + 0.5L) / m);
        if (v < 1e-9L) v = 1e-9L;
        long double pw = v, v2 = v * v;
        for (int j = 0; j < n; ++j) { A[i * n + j] = pw; pw *= v2; }
        b[i] = atanl(v * umax);
    }
    std::vector<long double> c(n);
    for (int it = 0; it < 40; ++it) {
        wls(A, b, w, m, n, c.data());
        long double emax = 0;
        std::vector<long double> e(m);
        for (int i = 0; i < m; ++i) {
            long double s = 0;
            for (int j = 0; j < n; ++j) s += A[i * n + j] * c[j];
            e[i] = fabsl(s - b[i]);
            if (e[i] > emax) emax = e[i];
        }
        if (emax == 0) break;
        long double mean = 0;
        for (int i = 0; i < m; ++i) { w[i] *= 1.0L + 8.0L * e[i] / emax; mean += w[i]; }
        mean /= m;
        for (int i = 0; i < m; ++i) w[i] /= mean;
    }
    long double pw = 1.0L / umax, inv2 = 1.0L / (umax * umax);
    for (int j = 0; j < n; ++j) { coef[j] = (float)(c[j] * pw * scale); pw *= inv2; }
    double worst = 0;
    const int grid = 200000;
    for (int i = 0; i <= grid; ++i) {
        float u = (float)(umax * i / grid);
        float u2 = u * u;
        float p = coef[n - 1];
        for (int j = n - 2; j >= 0; --j) p = fmaf(p, u2, coef[j]);
        double got = (double)p * (double)u;  // the final multiply / fma rounds once more: <= 1 ulp
        double err = fabs(got / scale - atan((double)u));
        if (err > worst) worst = err;
    }
    return worst;
}

float eval_row(const DeviceParams& d, float u) {
    float u2 = u * u;
    float p = d.row_p[kRowTerms - 1];
    for (int i = kRowTerms - 2; i >= 0; --i) p = fmaf(p, u2, d.row_p[i]);
    return fmaf(p, u, d.row_off);
}

struct Memo {
    nsc_params p;
    int32_t lut[NSC_N_FREQS];
    DeviceParams d;
};
std::mutex g_mu;
std::vector<Memo> g_memo;

// Max error (radians) of the literal column polynomial of nsc_point.h, evaluated as the
// kernel evaluates it (float32 Horner with FMA).
double col_poly_error() {
    static const double err = [] {
        const float c[kColTerms] = {NSC_COL_C0, NSC_COL_C1, NSC_COL_C2, NSC_COL_C3,
                                    NSC_COL_C4, NSC_COL_C5, NSC_COL_C6};
        const double scale = 360.0 / (2.0 * 3.14159265358979323846);
        double worst = 0;
        const int grid = 400000;
        for (int i = 0; i <= grid; ++i) {
            const float t = (float)((double)i / grid);
            const float t2 = t * t;
            float p = c[kColTerms - 1];
            for (int j = kColTerms - 2; j >= 0; --j) p = fmaf(p, t2, c[j]);
            const float r = p * t;
            worst = fmax(worst, fabs((double)r / scale - atan((double)t)));
        }
        return worst;
    }();
    return err;
}

}  // namespace

int make_device_params(const nsc_params* p, const int32_t* h_lut, DeviceParams* out) {
    int st = validate_params(p);
    if (st != NSC_OK) return st;
    if (!h_lut || !out) return NSC_ERR_NULL_POINTER;
    int prev = 0;
    for (int k = 0; k < NSC_N_FREQS; ++k) {
        if (h_lut[k] < prev || h_lut[k] >= p->n_bins) return NSC_ERR_BAD_LUT;
        prev = h_lut[k];
    }
    {
        std::lock_guard<std::mutex> lk(g_mu);
        for (const Memo& m : g_memo)
            if (memcmp(&m.p, p, sizeof(nsc_params)) == 0 && memcmp(m.lut, h_lut, sizeof(m.lut)) == 0) {
                *out = m.d;
                return NSC_OK;
            }
    }
    DeviceParams d;
    memset(&d, 0, sizeof(d));
    d.E = p->n_elevation;
    d.T = p->target_rows;
    d.n_bins = p->n_bins;
    d.interpolate = p->interpolate_empty ? 1 : 0;
    d.s_lo = sqrt_preimage_lo(p->min_range);
    d.s_hi = sqrt_preimage_hi(p->max_range);
    d.eps = p->epsilon;
    d.uniform = 1.0f / (float)(d.T * d.n_bins);

    if (!(col_poly_error() < 1e-6)) return NSC_ERR_BAD_PARAMS;

    // Rows. Edges are el_min + k * width, k = 0..E (range_image.py:186-188, float64).
    const double width = (p->el_max_rad - p->el_min_rad) / d.E;
    for (int k = 0; k < NSC_MAX_ELEVATION; ++k) {
        double edge = p->el_min_rad + k * width;
        float c;
        if (k == 0 || k >= d.E) c = INFINITY;
        else if (edge >= 1.5707963) c = INFINITY;
        else if (edge <= -1.5707963) c = -INFINITY;
        else { double t = tan(edge); c = (float)(t * fabs(t)); }
        d.row_c[k] = c;
    }
    d.row_mode = kRowSearch;
    // Any u below tan(el_min + width/4) is row 0 and any u above tan(el_max - width/4) is row
    // E-1, so u is clamped there and the polynomial only has to cover the field of view.
    const double lo_ang = p->el_min_rad + 0.25 * width, hi_ang = p->el_max_rad - 0.25 * width;
    if (lo_ang > -0.65 && hi_ang < 0.65) {
        const double umax = fmax(fabs(tan(lo_ang)), fabs(tan(hi_ang))) * 1.0001 + 1e-6;
        double err = fit_atan(umax, kRowTerms, 1.0 / width, d.row_p);
        d.row_off = (float)(-p->el_min_rad / width);
        d.u_lo = (float)tan(lo_ang);
        d.u_hi = (float)tan(hi_ang);
        float r_lo = eval_row(d, d.u_lo), r_hi = eval_row(d, d.u_hi);
        if (err < 2e-7 && r_lo > 0.05f && r_lo < 0.45f && r_hi > d.E - 0.45f && r_hi < d.E - 0.05f)
            d.row_mode = kRowPoly;
    }

    int b = 0;
    for (int k = 0; k < NSC_N_FREQS; ++k)
        while (b <= h_lut[k]) d.bin_start[b++] = (uint8_t)k;
    while (b <= d.n_bins) d.bin_start[b++] = (uint8_t)NSC_N_FREQS;

    {
        std::lock_guard<std::mutex> lk(g_mu);
        if (g_memo.size() >= 64) g_memo.erase(g_memo.begin());
        Memo m;
        m.p = *p;
        memcpy(m.lut, h_lut, sizeof(m.lut));
        m.d = d;
        g_memo.push_back(m);
    }
    *out = d;
    return NSC_OK;
}

}  // namespace nsc

extern "C" {

int nsc_abi_version(void) { return NSC_ABI_VERSION; }

const char* nsc_strerror(int status) {
    switch (status) {
        case NSC_OK: return "ok";
        case NSC_ERR_NULL_POINTER: return "null pointer";
        case NSC_ERR_BAD_STRIDE: return "point stride must be 3 or 4 floats";
        case NSC_ERR_BAD_COUNT: return "negative scan / image count";
        case NSC_ERR_BAD_PARAMS: return "nsc_params outside the supported envelope";
        case NSC_ERR_BAD_LUT: return "freq->bin table not monotone or out of range";
        case NSC_ERR_WORKSPACE: return "workspace missing or too small";
        case NSC_ERR_ALIGNMENT: return "4-float points must be 16-byte aligned";
        case NSC_ERR_BAD_OFFSETS: return "scan offsets not monotone";
        case NSC_ERR_CUDA: return "CUDA runtime error (see nsc_last_cuda_error)";
        case NSC_ERR_BAD_STRUCT: return "nsc_params.struct_size does not match this ABI";
        default: return "unknown status";
    }
}

void nsc_default_params(nsc_params* p) {
    if (!p) return;
    memset(p, 0, sizeof(*p));
    p->struct_size = (int32_t)sizeof(nsc_params);
    p->n_elevation = 16;
    p->n_azimuth = NSC_N_AZIMUTH;
    p->n_bins = 50;
    p->target_rows = 16;
    p->interpolate_empty = 1;
    p->min_range = 1.0f;
    p->max_range = 80.0f;
    p->el_min_rad = -24.8 * (3.14159265358979323846 / 180.0);   // np.deg2rad(-24.8)
    p->el_max_rad = 2.0 * (3.14159265358979323846 / 180.0);     // np.deg2rad(2.0)
    p->epsilon = 1e-8f;
}

int nsc_freq_to_bin(float alpha, const nsc_params* p, int32_t* h_lut) {
    int st = nsc::validate_params(p);
    if (st != NSC_OK) return st;
    if (!h_lut) return NSC_ERR_NULL_POINTER;
    const int nb = p->n_bins, steps = nb + 1;
    std::vector<float> edges(steps);
    const float step = 1.0f / (float)nb;   // torch.linspace(0, 1, nb + 1), float32
    const float denom = expf(alpha) - 1.0f + p->epsilon;
    for (int i = 0; i < steps; ++i) {
        // torch fills the lower half from the start and the upper half from the end
        float t = (i < steps / 2) ? (0.0f + step * (float)i) : (1.0f - step * (float)(steps - 1 - i));
        edges[i] = (expf(alpha * t) - 1.0f) / denom * (float)NSC_N_FREQS;
    }
    for (int k = 0; k < NSC_N_FREQS; ++k) {
        int ub = 0;  // searchsorted(edges, k, right=True): first index with edges[idx] > k
        while (ub < steps && edges[ub] <= (float)k) ++ub;
        int b = ub - 1;
        h_lut[k] = b < 0 ? 0 : (b > nb - 1 ? nb - 1 : b);
    }
    return NSC_OK;
}

}  // extern "C"
