// Internal declarations shared by the translation units of libnsc_b200.so.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "nsc_b200.h"

namespace nsc {

constexpr int kAz = NSC_N_AZIMUTH;      // 360 columns
constexpr int kFreqs = NSC_N_FREQS;     // 181
constexpr int kPitch = kAz + 1;         // smem row pitch of the min-image: column 360 catches az == 2*pi
constexpr int kMaskWords = 12;          // 360 validity bits per row
constexpr uint32_t kInfBits = 0x7f800000u;
constexpr int kColTerms = 7;            // odd polynomial for atan on [0,1] (azimuth)
constexpr int kRowTerms = 5;            // odd polynomial for atan on the elevation FOV
constexpr int kMaxSignals = 8;          // complex 360-point FFTs in flight per CTA (two rows each)
// Row capacity of the encode kernels for images of up to 64 rows; taller images (up to
// NSC_MAX_ELEVATION) take the tall kernels, whose row search reaches row NSC_MAX_ELEVATION - 1.
constexpr int kShortRows = NSC_MAX_ELEVATION_SHORT;
// The row envelope of a parameter block: NSC_MAX_ELEVATION with NSC_FLAG_TALL_IMAGES, else 64.
inline int max_rows(const nsc_params* p) {
    return (p->flags & NSC_FLAG_TALL_IMAGES) ? NSC_MAX_ELEVATION : NSC_MAX_ELEVATION_SHORT;
}

enum RowMode { kRowPoly = 0, kRowSearch = 1 };

// Kernel arguments derived on the host from nsc_params (+ the freq->bin table). Passed by
// value as a __grid_constant__ so every field is a constant-bank operand.
struct DeviceParams {
    int E;                 // projected rows
    int T;                 // target rows after pooling
    int n_bins;
    int interpolate;
    int row_mode;          // RowMode
    float s_lo, s_hi;      // keep a point iff s_lo <= (x*x + y*y) + z*z <= s_hi (host_tables.cu)
    float eps;
    float uniform;         // 1 / (T * n_bins) in float32
    float row_p[kRowTerms];   // (atan(u) - el_min) / row_width = row_off + u * P(u^2)
    float row_off;
    float u_lo, u_hi;      // clamp of u = z / rho that keeps the row value inside (0, E)
    float row_c[NSC_MAX_ELEVATION];  // kRowSearch: row_c[k] = tan(edge_k)*|tan(edge_k)|, k = 1..E-1
    uint8_t bin_start[NSC_MAX_BINS + 3];  // first frequency of bin b; bin_start[n_bins] = 181
};

// Fills DeviceParams; returns an nsc_status. Results are memoised per (params, lut).
int make_device_params(const nsc_params* p, const int32_t* h_lut, DeviceParams* out);
int validate_params(const nsc_params* p);

// thread-local CUDA error text for nsc_last_cuda_error().
int record_cuda(cudaError_t e);

// The points of an encode launch: scan i is points [offsets[i] - origin, offsets[i + 1] - origin)
// of `points`, `stride` floats (3 or 4) per point.
struct PointBatch {
    const float* points;
    int stride;
    const long long* offsets;    // n_scans + 1 entries, device memory
    long long origin;
    int n_scans;
};

// What an encode launch writes; every output left null is not written. Descriptor rows are
// n_scans x D (D = T * n_bins): float32 to `rows` and to rows peer_row0 + scan of the n_peers
// databases in `peers` (a host array of device pointers), or the uint16 wire format alone to
// `rows_q` (HistogramQuantizer.quantize with epsilon q_eps). Range images are n_scans x E x 360,
// taken at `stage` (NSC_STAGE_*).
struct EncodeOutputs {
    float* rows = nullptr;
    unsigned short* rows_q = nullptr;
    float q_eps = 0.0f;
    float* images = nullptr;
    int stage = NSC_STAGE_PROJECTED;
    float* const* peers = nullptr;
    int n_peers = 0;
    long long peer_row0 = 0;
};

// Launchers (nsc_encode.cu)
int launch_encode(const PointBatch& in, const DeviceParams& dp, const EncodeOutputs& out,
                  unsigned* d_workspace, size_t workspace_bytes, cudaStream_t stream);
int launch_encode_images(const float* d_images, int n_images, int rows, const DeviceParams& dp,
                         float* d_out, cudaStream_t stream);
int launch_interpolate(const float* d_in, int n_images, int rows, int nearest, float* d_out, cudaStream_t stream);
size_t workspace_bytes_for(int n_scans, int E);   // recommended: room to split the last wave's scans
size_t workspace_bytes_min();                      // enough for every launch (no splitting)

// The parameter and freq->bin table checks of nsc_anywidth_points, in its order (nsc_anywidth.cu)
int check_anywidth(const nsc_params* p, const int32_t* h_lut);

}  // namespace nsc
