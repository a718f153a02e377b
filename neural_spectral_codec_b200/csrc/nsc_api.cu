// extern "C" entry points of libnsc_b200.so (declared in include/nsc_b200.h).
#include <string.h>

#include <string>

#include "nsc_point.h"

namespace nsc {

static thread_local std::string t_cuda_error;

int record_cuda(cudaError_t e) {
    if (e == cudaSuccess) return NSC_OK;
    t_cuda_error = std::string(cudaGetErrorName(e)) + ": " + cudaGetErrorString(e);
    return NSC_ERR_CUDA;
}

static int check_points(const float* d_points, int stride, const int64_t* d_offsets, int n_scans) {
    if (n_scans < 0) return NSC_ERR_BAD_COUNT;
    if (stride != 3 && stride != 4) return NSC_ERR_BAD_STRIDE;
    if (!d_offsets) return NSC_ERR_NULL_POINTER;
    if (stride == 4 && (reinterpret_cast<uintptr_t>(d_points) & 15u)) return NSC_ERR_ALIGNMENT;
    return NSC_OK;
}

}  // namespace nsc

using namespace nsc;

extern "C" {

const char* nsc_last_cuda_error(void) { return t_cuda_error.c_str(); }

size_t nsc_workspace_bytes(int n_scans, const nsc_params* p) {
    if (n_scans < 0 || validate_params(p) != NSC_OK) return 0;
    return workspace_bytes_for(n_scans, p->n_elevation);
}

}  // extern "C"

namespace {
// nsc_encode_batch (d_out_q null) and nsc_encode_batch_u16 (d_out null): one validation order
int encode_batch(const float* d_points, int point_stride, const int64_t* d_offsets, int64_t point_origin,
                 int n_scans, const nsc_params* p, const int32_t* h_lut, float* d_out, uint16_t* d_out_q,
                 float q_epsilon, void* d_workspace, size_t workspace_bytes, void* stream) {
    DeviceParams dp;
    int st = make_device_params(p, h_lut, &dp);
    if (st != NSC_OK) return st;
    st = check_points(d_points, point_stride, d_offsets, n_scans);
    if (st != NSC_OK) return st;
    if (n_scans == 0) return NSC_OK;
    if (!d_out && !d_out_q) return NSC_ERR_NULL_POINTER;
    if (!d_workspace || workspace_bytes < workspace_bytes_min()) return NSC_ERR_WORKSPACE;
    EncodeOutputs out;
    out.rows = d_out;
    out.rows_q = d_out_q;
    out.q_eps = q_epsilon;
    return launch_encode({d_points, point_stride, (const long long*)d_offsets, point_origin, n_scans}, dp, out,
                         (unsigned*)d_workspace, workspace_bytes, (cudaStream_t)stream);
}
}  // namespace

extern "C" {

int nsc_encode_batch(const float* d_points, int point_stride, const int64_t* d_offsets,
                     int64_t point_origin, int n_scans, const nsc_params* p, const int32_t* h_lut,
                     float* d_out, void* d_workspace, size_t workspace_bytes, void* stream) {
    return encode_batch(d_points, point_stride, d_offsets, point_origin, n_scans, p, h_lut, d_out, nullptr, 0.0f,
                        d_workspace, workspace_bytes, stream);
}

int nsc_encode_batch_u16(const float* d_points, int point_stride, const int64_t* d_offsets,
                         int64_t point_origin, int n_scans, const nsc_params* p, const int32_t* h_lut,
                         float q_epsilon, uint16_t* d_out, void* d_workspace, size_t workspace_bytes,
                         void* stream) {
    return encode_batch(d_points, point_stride, d_offsets, point_origin, n_scans, p, h_lut, nullptr, d_out,
                        q_epsilon, d_workspace, workspace_bytes, stream);
}

int nsc_encode_batch_peers(const float* d_points, int point_stride, const int64_t* d_offsets,
                           int64_t point_origin, int n_scans, const nsc_params* p,
                           const int32_t* h_lut, float* const* h_peer_db, int n_peers,
                           int64_t db_row0, void* d_workspace, size_t workspace_bytes, void* stream) {
    DeviceParams dp;
    int st = make_device_params(p, h_lut, &dp);
    if (st != NSC_OK) return st;
    st = check_points(d_points, point_stride, d_offsets, n_scans);
    if (st != NSC_OK) return st;
    if (n_peers < 1 || n_peers > NSC_MAX_PEERS) return NSC_ERR_BAD_COUNT;
    if (!h_peer_db) return NSC_ERR_NULL_POINTER;
    for (int i = 0; i < n_peers; ++i)
        if (!h_peer_db[i]) return NSC_ERR_NULL_POINTER;
    if (n_scans == 0) return NSC_OK;
    if (!d_workspace || workspace_bytes < workspace_bytes_min()) return NSC_ERR_WORKSPACE;
    EncodeOutputs out;
    out.peers = h_peer_db;
    out.n_peers = n_peers;
    out.peer_row0 = db_row0;
    return launch_encode({d_points, point_stride, (const long long*)d_offsets, point_origin, n_scans}, dp, out,
                         (unsigned*)d_workspace, workspace_bytes, (cudaStream_t)stream);
}

namespace {
struct PeerFlags {
    uint32_t* ptr[NSC_MAX_PEERS];
};
// Thread p: release-store `value` into peer p's flag of this rank, then acquire-poll this rank's
// flag of peer p. Everything enqueued before this kernel on the stream (the encode kernel's peer
// stores) is complete, and made visible system-wide by the fence, before any flag is raised.
__global__ void peer_signal_wait_kernel(PeerFlags f, int n_peers, int rank, uint32_t signal_value,
                                        uint32_t wait_value) {
    const int p = threadIdx.x;
    // programmatic dependent of the encode kernel: set up while that grid drains, released when
    // it has completed and its (peer) stores are flushed
    asm volatile("griddepcontrol.wait;" ::: "memory");
    if (p >= n_peers) return;
    __threadfence_system();
    uint32_t* theirs = f.ptr[p] + rank;
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(theirs), "r"(signal_value) : "memory");
    const uint32_t* mine = f.ptr[rank] + p;
    uint32_t seen;
    do {
        asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(seen) : "l"(mine) : "memory");
    } while ((int32_t)(seen - wait_value) < 0);      // wrap-safe "seen < wait_value"
}
}  // namespace

int nsc_peer_signal_wait(uint32_t* const* h_peer_flags, int n_peers, int rank, uint32_t signal_value,
                         uint32_t wait_value, void* stream) {
    if (n_peers < 1 || n_peers > NSC_MAX_PEERS || rank < 0 || rank >= n_peers) return NSC_ERR_BAD_COUNT;
    if (!h_peer_flags) return NSC_ERR_NULL_POINTER;
    PeerFlags f;
    for (int i = 0; i < NSC_MAX_PEERS; ++i) {
        f.ptr[i] = i < n_peers ? h_peer_flags[i] : nullptr;
        if (i < n_peers && !f.ptr[i]) return NSC_ERR_NULL_POINTER;
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(1);
    cfg.blockDim = dim3(32);
    cfg.stream = (cudaStream_t)stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return record_cuda(cudaLaunchKernelEx(&cfg, peer_signal_wait_kernel, f, n_peers, rank, signal_value, wait_value));
}

int nsc_project_batch(const float* d_points, int point_stride, const int64_t* d_offsets,
                      int64_t point_origin, int n_scans, const nsc_params* p, int stage,
                      float* d_images, void* d_workspace, size_t workspace_bytes, void* stream) {
    // The projection does not depend on the bin table: use the identity-to-zero table.
    int32_t lut[NSC_N_FREQS];
    memset(lut, 0, sizeof(lut));
    DeviceParams dp;
    int st = make_device_params(p, lut, &dp);
    if (st != NSC_OK) return st;
    st = check_points(d_points, point_stride, d_offsets, n_scans);
    if (st != NSC_OK) return st;
    if (stage != NSC_STAGE_PROJECTED && stage != NSC_STAGE_INTERPOLATED) return NSC_ERR_BAD_PARAMS;
    if (n_scans == 0) return NSC_OK;
    if (!d_images) return NSC_ERR_NULL_POINTER;
    if (!d_workspace || workspace_bytes < workspace_bytes_min()) return NSC_ERR_WORKSPACE;
    EncodeOutputs out;
    out.images = d_images;
    out.stage = stage;
    return launch_encode({d_points, point_stride, (const long long*)d_offsets, point_origin, n_scans}, dp, out,
                         (unsigned*)d_workspace, workspace_bytes, (cudaStream_t)stream);
}

int nsc_encode_range_images(const float* d_images, int n_images, int rows, const nsc_params* p,
                            const int32_t* h_lut, float* d_out, void* stream) {
    DeviceParams dp;
    int st = make_device_params(p, h_lut, &dp);
    if (st != NSC_OK) return st;
    if (n_images < 0) return NSC_ERR_BAD_COUNT;
    if (rows < 1 || rows > max_rows(p)) return NSC_ERR_BAD_PARAMS;
    if (n_images == 0) return NSC_OK;
    if (!d_images || !d_out) return NSC_ERR_NULL_POINTER;
    return launch_encode_images(d_images, n_images, rows, dp, d_out, (cudaStream_t)stream);
}

int nsc_interpolate_range_images(const float* d_images_in, int n_images, int rows, int method,
                                 float* d_images_out, void* stream) {
    if (n_images < 0) return NSC_ERR_BAD_COUNT;
    if (rows < 1 || rows > NSC_MAX_ELEVATION) return NSC_ERR_BAD_PARAMS;
    if (method != NSC_INTERP_LINEAR && method != NSC_INTERP_NEAREST) return NSC_ERR_BAD_PARAMS;
    if (n_images == 0) return NSC_OK;
    if (!d_images_in || !d_images_out) return NSC_ERR_NULL_POINTER;
    return launch_interpolate(d_images_in, n_images, rows, method == NSC_INTERP_NEAREST, d_images_out,
                              (cudaStream_t)stream);
}

/* ---- test hook: the kernel's per-point function evaluated on the host ------------------ */
int nsc_test_host_classify(const float* h_points, int point_stride, int64_t n_points,
                           const nsc_params* p, int32_t* h_row, int32_t* h_col, uint8_t* h_keep) {
    int32_t lut[NSC_N_FREQS];
    memset(lut, 0, sizeof(lut));
    DeviceParams dp;
    int st = make_device_params(p, lut, &dp);
    if (st != NSC_OK) return st;
    if (point_stride != 3 && point_stride != 4) return NSC_ERR_BAD_STRIDE;
    if (n_points < 0) return NSC_ERR_BAD_COUNT;
    if (n_points && (!h_points || !h_row || !h_col || !h_keep)) return NSC_ERR_NULL_POINTER;
    for (int64_t i = 0; i < n_points; ++i) {
        const float* q = h_points + i * point_stride;
        uint32_t row_b = 0, col_b = 0;
        // the row search of the tall kernels: the same rows as the short one's for E <= 64
        const uint32_t key = classify<NSC_MAX_ELEVATION>(q[0], q[1], q[2], dp, dp.row_mode, row_b, col_b);
        const bool keep = key != 0xffffffffu && !key_is_empty(key, dp);
        h_keep[i] = keep ? 1 : 0;
        h_row[i] = keep ? (int32_t)(row_b - kFloorBias) : -1;
        int32_t c = keep ? (int32_t)(col_b - kFloorBias) : -1;
        h_col[i] = c == kAz ? 0 : c;
    }
    return NSC_OK;
}

int nsc_test_row_mode(const nsc_params* p) {
    int32_t lut[NSC_N_FREQS];
    memset(lut, 0, sizeof(lut));
    DeviceParams dp;
    int st = make_device_params(p, lut, &dp);
    return st != NSC_OK ? st : dp.row_mode;
}

}  // extern "C"
