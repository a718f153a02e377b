// extern "C" entry points of libnsc_b200.so (declared in include/nsc_b200.h).
#include <string.h>

#include <atomic>
#include <condition_variable>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

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
    if (rows < 1 || rows > NSC_MAX_ELEVATION) return NSC_ERR_BAD_PARAMS;
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

/* ---- host-buffer pipeline ------------------------------------------------------------- */
// A few persistent host threads that copy one pageable buffer into pinned staging piece by piece,
// each piece handed to the copy engine by the thread that staged it. One CPU core moves ~10 GB/s
// out of pageable memory, a quarter of what PCIe 5 takes; four of them keep up with it.
struct StagePool {
    std::vector<std::thread> workers;
    std::mutex mu;
    std::condition_variable cv_work, cv_done;
    unsigned long long generation = 0;
    int active = 0;
    bool stop = false;
    // the current job
    const char* src = nullptr;
    char* stage = nullptr;
    char* d_dst = nullptr;
    size_t bytes = 0, piece = 0;
    std::atomic<size_t> next{0};
    std::atomic<int> err{0};
    cudaStream_t stream = nullptr;
    int device = 0;

    void pieces() {
        for (;;) {
            const size_t off = next.fetch_add(1) * piece;
            if (off >= bytes) return;
            const size_t len = bytes - off < piece ? bytes - off : piece;
            memcpy(stage + off, src + off, len);
            const cudaError_t e = cudaMemcpyAsync(d_dst + off, stage + off, len, cudaMemcpyHostToDevice, stream);
            if (e != cudaSuccess) err.store((int)e);
        }
    }
    void worker() {
        cudaSetDevice(device);
        unsigned long long seen = 0;
        for (;;) {
            {
                std::unique_lock<std::mutex> lk(mu);
                cv_work.wait(lk, [&] { return stop || generation != seen; });
                if (stop) return;
                seen = generation;
            }
            pieces();
            std::lock_guard<std::mutex> lk(mu);
            if (--active == 0) cv_done.notify_one();
        }
    }
    void start(int n, int dev) {
        device = dev;
        for (int i = 0; i < n; ++i) workers.emplace_back([this] { worker(); });
    }
    // copies [src, src + n) through `stage` into d_dst on `stream`; returns when all of it is staged
    cudaError_t run(const void* s, void* st, void* d, size_t n, size_t piece_bytes, cudaStream_t cs) {
        src = (const char*)s;
        stage = (char*)st;
        d_dst = (char*)d;
        bytes = n;
        piece = piece_bytes;
        stream = cs;
        next.store(0);
        err.store(0);
        const bool fan_out = !workers.empty() && n > 2 * piece_bytes;
        if (fan_out) {
            std::lock_guard<std::mutex> lk(mu);
            active = (int)workers.size();
            ++generation;
        }
        if (fan_out) cv_work.notify_all();
        pieces();
        if (fan_out) {
            std::unique_lock<std::mutex> lk(mu);
            cv_done.wait(lk, [&] { return active == 0; });
        }
        return (cudaError_t)err.load();
    }
    ~StagePool() {
        {
            std::lock_guard<std::mutex> lk(mu);
            stop = true;
        }
        cv_work.notify_all();
        for (auto& t : workers) t.join();
    }
};

struct nsc_pipeline {
    int device;
    int n_buffers;
    int64_t max_chunk_points;
    int max_chunk_scans;
    struct Slot {
        cudaStream_t stream;
        cudaEvent_t done;
        float* d_points;
        long long* d_offsets;
        float* d_out;
        unsigned* d_ws;
        float* h_stage;        // pinned staging of one chunk (nsc_pipeline_encode_scans), lazy
        long long* h_offsets;  // pinned chunk offsets
        float* h_out;          // pinned chunk descriptors
        bool busy;
    } slot[4];
    unsigned next_single;      // rotation of nsc_pipeline_encode_scan over the slots
    StagePool* pool;           // lazily started by nsc_pipeline_encode_scan
};

static const int kMaxChunkScans = 1024;
static const int kMaxDescriptor = NSC_MAX_DESCRIPTOR;

void nsc_pipeline_destroy(nsc_pipeline* pl) {
    if (!pl) return;
    int prev = 0;
    cudaGetDevice(&prev);
    cudaSetDevice(pl->device);
    for (int i = 0; i < pl->n_buffers; ++i) {
        nsc_pipeline::Slot& s = pl->slot[i];
        if (s.stream) cudaStreamSynchronize(s.stream);
        if (s.d_points) cudaFree(s.d_points);
        if (s.d_offsets) cudaFree(s.d_offsets);
        if (s.d_out) cudaFree(s.d_out);
        if (s.d_ws) cudaFree(s.d_ws);
        if (s.h_stage) cudaFreeHost(s.h_stage);
        if (s.h_offsets) cudaFreeHost(s.h_offsets);
        if (s.h_out) cudaFreeHost(s.h_out);
        if (s.done) cudaEventDestroy(s.done);
        if (s.stream) cudaStreamDestroy(s.stream);
    }
    delete pl->pool;
    cudaSetDevice(prev);
    delete pl;
}

int nsc_pipeline_create(int64_t max_chunk_points, int n_buffers, int device, nsc_pipeline** out) {
    if (!out) return NSC_ERR_NULL_POINTER;
    *out = nullptr;
    if (max_chunk_points < 1 || n_buffers < 1 || n_buffers > 4) return NSC_ERR_BAD_COUNT;
    int prev = 0;
    cudaError_t e = cudaGetDevice(&prev);
    if (e != cudaSuccess) return record_cuda(e);
    e = cudaSetDevice(device);
    if (e != cudaSuccess) return record_cuda(e);
    nsc_pipeline* pl = new nsc_pipeline();
    memset(pl, 0, sizeof(*pl));
    pl->device = device;
    pl->n_buffers = n_buffers;
    pl->max_chunk_points = max_chunk_points;
    pl->max_chunk_scans = kMaxChunkScans;
    int st = NSC_OK;
    for (int i = 0; i < n_buffers && st == NSC_OK; ++i) {
        nsc_pipeline::Slot& s = pl->slot[i];
        if ((e = cudaStreamCreateWithFlags(&s.stream, cudaStreamNonBlocking)) != cudaSuccess ||
            (e = cudaEventCreateWithFlags(&s.done, cudaEventDisableTiming)) != cudaSuccess ||
            (e = cudaMalloc(&s.d_points, (size_t)max_chunk_points * 16)) != cudaSuccess ||
            (e = cudaMalloc(&s.d_offsets, (size_t)(kMaxChunkScans + 1) * 8)) != cudaSuccess ||
            (e = cudaMalloc(&s.d_out, (size_t)kMaxChunkScans * kMaxDescriptor * 4)) != cudaSuccess ||
            (e = cudaMalloc(&s.d_ws, 256)) != cudaSuccess)
            st = record_cuda(e);
    }
    cudaSetDevice(prev);
    if (st != NSC_OK) {
        nsc_pipeline_destroy(pl);
        return st;
    }
    *out = pl;
    return NSC_OK;
}

}  // extern "C"

// nsc_pipeline_encode / nsc_pipeline_encode_u16: descriptors of out_bytes (4 or 2) per element,
// the uint16 ones in the first half of the slot's float32 descriptor buffer.
static int pipeline_encode(nsc_pipeline* pl, const float* h_points, int point_stride, int64_t n_points,
                           const int64_t* h_offsets, int n_scans, const nsc_params* p, const int32_t* h_lut,
                           void* h_out, size_t out_bytes, float q_eps) {
    if (!pl) return NSC_ERR_NULL_POINTER;
    DeviceParams dp;
    int st = make_device_params(p, h_lut, &dp);
    if (st != NSC_OK) return st;
    if (n_scans < 0) return NSC_ERR_BAD_COUNT;
    if (point_stride != 3 && point_stride != 4) return NSC_ERR_BAD_STRIDE;
    if (n_scans == 0) return NSC_OK;
    if (!h_points || !h_offsets || !h_out) return NSC_ERR_NULL_POINTER;
    if (n_points < 0) return NSC_ERR_BAD_COUNT;
    if (h_offsets[0] < 0 || h_offsets[n_scans] > n_points) return NSC_ERR_BAD_OFFSETS;
    for (int i = 0; i < n_scans; ++i)
        if (h_offsets[i + 1] < h_offsets[i]) return NSC_ERR_BAD_OFFSETS;
    const int D = dp.T * dp.n_bins;
    int prev = 0;
    cudaError_t e = cudaGetDevice(&prev);
    if (e != cudaSuccess) return record_cuda(e);
    e = cudaSetDevice(pl->device);
    if (e != cudaSuccess) return record_cuda(e);
    EncodeOutputs out;
    out.q_eps = q_eps;

    int first = 0, k = 0;
    while (first < n_scans && st == NSC_OK) {
        // chunk = as many whole scans as fit the staging buffer
        int last = first;
        while (last < n_scans && last - first < pl->max_chunk_scans &&
               h_offsets[last + 1] - h_offsets[first] <= pl->max_chunk_points)
            ++last;
        if (last == first) { st = NSC_ERR_WORKSPACE; break; }
        nsc_pipeline::Slot& s = pl->slot[k % pl->n_buffers];
        if (s.busy) {   // host offsets / output of the previous use must be complete
            if ((e = cudaEventSynchronize(s.done)) != cudaSuccess) { st = record_cuda(e); break; }
            s.busy = false;
        }
        const int64_t p0 = h_offsets[first], np = h_offsets[last] - p0;
        const int ns = last - first;
        const size_t pbytes = (size_t)np * point_stride * 4;
        if ((e = cudaMemcpyAsync(s.d_points, h_points + p0 * point_stride, pbytes,
                                 cudaMemcpyHostToDevice, s.stream)) != cudaSuccess ||
            (e = cudaMemcpyAsync(s.d_offsets, h_offsets + first, (size_t)(ns + 1) * 8,
                                 cudaMemcpyHostToDevice, s.stream)) != cudaSuccess) {
            st = record_cuda(e);
            break;
        }
        if (out_bytes == 4) out.rows = s.d_out;
        else out.rows_q = reinterpret_cast<unsigned short*>(s.d_out);
        st = launch_encode({s.d_points, point_stride, s.d_offsets, p0, ns}, dp, out, s.d_ws, 256, s.stream);
        if (st != NSC_OK) break;
        if ((e = cudaMemcpyAsync((char*)h_out + (size_t)first * D * out_bytes, s.d_out, (size_t)ns * D * out_bytes,
                                 cudaMemcpyDeviceToHost, s.stream)) != cudaSuccess ||
            (e = cudaEventRecord(s.done, s.stream)) != cudaSuccess) {
            st = record_cuda(e);
            break;
        }
        s.busy = true;
        first = last;
        ++k;
    }
    for (int i = 0; i < pl->n_buffers; ++i) {
        nsc_pipeline::Slot& s = pl->slot[i];
        if ((e = cudaStreamSynchronize(s.stream)) != cudaSuccess && st == NSC_OK) st = record_cuda(e);
        s.busy = false;
    }
    cudaSetDevice(prev);
    return st;
}

// Copies scans [first, last) into the pinned staging buffer with a few host threads (a single
// memcpy stream cannot keep up with PCIe 5 from pageable memory).
static void stage_scans(float* dst, const float* const* h_scans, const int64_t* h_counts, int first,
                        int last, int stride, long long* offs_out) {
    std::vector<size_t> start(last - first + 1, 0);
    for (int i = first; i < last; ++i) start[i - first + 1] = start[i - first] + (size_t)h_counts[i];
    for (int i = first; i <= last; ++i) offs_out[i - first] = (long long)start[i - first];
    const size_t total_bytes = start[last - first] * stride * 4;
    unsigned hw = std::thread::hardware_concurrency();
    int n_thr = (int)(total_bytes >> 22);                 // one thread per 4 MiB, at most 12
    if (n_thr > 12) n_thr = 12;
    if (hw && n_thr > (int)hw) n_thr = (int)hw;
    if (n_thr < 1) n_thr = 1;
    auto work = [&](int t) {
        // thread t copies the byte range [t, t+1) * total / n_thr, walking the scans it overlaps
        const size_t lo = total_bytes * t / n_thr, hi = total_bytes * (t + 1) / n_thr;
        for (int i = first; i < last; ++i) {
            const size_t b0 = start[i - first] * stride * 4, b1 = start[i - first + 1] * stride * 4;
            const size_t c0 = b0 > lo ? b0 : lo, c1 = b1 < hi ? b1 : hi;
            if (c0 < c1)
                memcpy((char*)dst + c0, (const char*)h_scans[i] + (c0 - b0), c1 - c0);
        }
    };
    if (n_thr == 1) { work(0); return; }
    std::vector<std::thread> pool;
    for (int t = 1; t < n_thr; ++t) pool.emplace_back(work, t);
    work(0);
    for (auto& th : pool) th.join();
}

// nsc_pipeline_encode_scans / nsc_pipeline_encode_scans_u16: descriptors as in pipeline_encode.
static int pipeline_encode_scans(nsc_pipeline* pl, const float* const* h_scans, const int64_t* h_counts,
                                 int point_stride, int n_scans, const nsc_params* p, const int32_t* h_lut,
                                 void* h_out, size_t out_bytes, float q_eps) {
    if (!pl) return NSC_ERR_NULL_POINTER;
    DeviceParams dp;
    int st = make_device_params(p, h_lut, &dp);
    if (st != NSC_OK) return st;
    if (n_scans < 0) return NSC_ERR_BAD_COUNT;
    if (point_stride != 3 && point_stride != 4) return NSC_ERR_BAD_STRIDE;
    if (n_scans == 0) return NSC_OK;
    if (!h_scans || !h_counts || !h_out) return NSC_ERR_NULL_POINTER;
    for (int i = 0; i < n_scans; ++i) {
        if (h_counts[i] < 0) return NSC_ERR_BAD_OFFSETS;
        if (h_counts[i] > 0 && !h_scans[i]) return NSC_ERR_NULL_POINTER;
        if (h_counts[i] > pl->max_chunk_points) return NSC_ERR_WORKSPACE;
    }
    const int D = dp.T * dp.n_bins;
    int prev = 0;
    cudaError_t e = cudaGetDevice(&prev);
    if (e != cudaSuccess) return record_cuda(e);
    e = cudaSetDevice(pl->device);
    if (e != cudaSuccess) return record_cuda(e);

    EncodeOutputs out;
    out.q_eps = q_eps;
    // pinned staging for every slot, allocated on the first call of this entry point
    for (int i = 0; i < pl->n_buffers; ++i) {
        nsc_pipeline::Slot& s = pl->slot[i];
        if ((!s.h_stage && (e = cudaHostAlloc(&s.h_stage, (size_t)pl->max_chunk_points * 16, cudaHostAllocDefault)) != cudaSuccess) ||
            (!s.h_offsets && (e = cudaHostAlloc(&s.h_offsets, (size_t)(kMaxChunkScans + 1) * 8, cudaHostAllocDefault)) != cudaSuccess) ||
            (!s.h_out && (e = cudaHostAlloc(&s.h_out, (size_t)kMaxChunkScans * kMaxDescriptor * 4, cudaHostAllocDefault)) != cudaSuccess)) {
            cudaSetDevice(prev);
            return record_cuda(e);
        }
    }
    struct Pending { int first, count; };
    Pending pending[4] = {};
    auto retire = [&](int k) -> int {      // wait for slot k and hand its descriptors to the caller
        nsc_pipeline::Slot& s = pl->slot[k];
        if (!s.busy) return NSC_OK;
        cudaError_t er = cudaEventSynchronize(s.done);
        if (er != cudaSuccess) return record_cuda(er);
        memcpy((char*)h_out + (size_t)pending[k].first * D * out_bytes, s.h_out, (size_t)pending[k].count * D * out_bytes);
        s.busy = false;
        return NSC_OK;
    };
    int first = 0, k = 0;
    while (first < n_scans && st == NSC_OK) {
        int last = first;
        int64_t np = 0;
        while (last < n_scans && last - first < pl->max_chunk_scans && np + h_counts[last] <= pl->max_chunk_points)
            np += h_counts[last++];
        const int slot_i = k % pl->n_buffers;
        nsc_pipeline::Slot& s = pl->slot[slot_i];
        if ((st = retire(slot_i)) != NSC_OK) break;
        const int ns = last - first;
        stage_scans(s.h_stage, h_scans, h_counts, first, last, point_stride, s.h_offsets);
        if ((e = cudaMemcpyAsync(s.d_points, s.h_stage, (size_t)np * point_stride * 4,
                                 cudaMemcpyHostToDevice, s.stream)) != cudaSuccess ||
            (e = cudaMemcpyAsync(s.d_offsets, s.h_offsets, (size_t)(ns + 1) * 8, cudaMemcpyHostToDevice,
                                 s.stream)) != cudaSuccess) {
            st = record_cuda(e);
            break;
        }
        if (out_bytes == 4) out.rows = s.d_out;
        else out.rows_q = reinterpret_cast<unsigned short*>(s.d_out);
        st = launch_encode({s.d_points, point_stride, s.d_offsets, 0, ns}, dp, out, s.d_ws, 256, s.stream);
        if (st != NSC_OK) break;
        if ((e = cudaMemcpyAsync(s.h_out, s.d_out, (size_t)ns * D * out_bytes, cudaMemcpyDeviceToHost, s.stream)) != cudaSuccess ||
            (e = cudaEventRecord(s.done, s.stream)) != cudaSuccess) {
            st = record_cuda(e);
            break;
        }
        s.busy = true;
        pending[slot_i].first = first;
        pending[slot_i].count = ns;
        first = last;
        ++k;
    }
    for (int i = 0; i < pl->n_buffers; ++i) {
        if (st == NSC_OK) st = retire(i);
        else { cudaStreamSynchronize(pl->slot[i].stream); pl->slot[i].busy = false; }
    }
    cudaSetDevice(prev);
    return st;
}

extern "C" {

int nsc_pipeline_encode(nsc_pipeline* pl, const float* h_points, int point_stride,
                        int64_t n_points, const int64_t* h_offsets, int n_scans,
                        const nsc_params* p, const int32_t* h_lut, float* h_out) {
    return pipeline_encode(pl, h_points, point_stride, n_points, h_offsets, n_scans, p, h_lut, h_out, 4, 0.0f);
}

int nsc_pipeline_encode_u16(nsc_pipeline* pl, const float* h_points, int point_stride,
                            int64_t n_points, const int64_t* h_offsets, int n_scans,
                            const nsc_params* p, const int32_t* h_lut, float q_epsilon, uint16_t* h_out) {
    return pipeline_encode(pl, h_points, point_stride, n_points, h_offsets, n_scans, p, h_lut, h_out, 2, q_epsilon);
}

int nsc_pipeline_encode_scans(nsc_pipeline* pl, const float* const* h_scans, const int64_t* h_counts,
                              int point_stride, int n_scans, const nsc_params* p,
                              const int32_t* h_lut, float* h_out) {
    return pipeline_encode_scans(pl, h_scans, h_counts, point_stride, n_scans, p, h_lut, h_out, 4, 0.0f);
}

int nsc_pipeline_encode_scans_u16(nsc_pipeline* pl, const float* const* h_scans, const int64_t* h_counts,
                                  int point_stride, int n_scans, const nsc_params* p,
                                  const int32_t* h_lut, float q_epsilon, uint16_t* h_out) {
    return pipeline_encode_scans(pl, h_scans, h_counts, point_stride, n_scans, p, h_lut, h_out, 2, q_epsilon);
}

// One scan from pageable host memory to a descriptor ON THE DEVICE, on the caller's stream: the
// reference's call shape (one encode_points(numpy) per scan, pipeline.py:336-354). The scan is
// copied into pinned staging in 256 KB pieces by the calling thread and up to three pool threads,
// each piece handed to the copy engine as soon as it is staged, so staging and DMA overlap; the
// kernel follows on the same stream. Returns when the source array may be reused; nothing else is synchronised (a slot
// is reused only after the work that read its staging has finished).
int nsc_pipeline_encode_scan(nsc_pipeline* pl, const float* h_points, int point_stride, int64_t n_points,
                             const nsc_params* p, const int32_t* h_lut, float* d_out, void* stream) {
    if (!pl) return NSC_ERR_NULL_POINTER;
    DeviceParams dp;
    int st = make_device_params(p, h_lut, &dp);
    if (st != NSC_OK) return st;
    if (point_stride != 3 && point_stride != 4) return NSC_ERR_BAD_STRIDE;
    if (n_points < 0) return NSC_ERR_BAD_COUNT;
    if (n_points > pl->max_chunk_points) return NSC_ERR_WORKSPACE;
    if ((n_points && !h_points) || !d_out) return NSC_ERR_NULL_POINTER;
    int prev = 0;
    cudaError_t e = cudaGetDevice(&prev);
    if (e != cudaSuccess) return record_cuda(e);
    if ((e = cudaSetDevice(pl->device)) != cudaSuccess) return record_cuda(e);
    nsc_pipeline::Slot& s = pl->slot[pl->next_single++ % pl->n_buffers];
    cudaStream_t cs = (cudaStream_t)stream;
    auto fail = [&](cudaError_t err) { cudaSetDevice(prev); return record_cuda(err); };
    if (!s.h_stage && (e = cudaHostAlloc(&s.h_stage, (size_t)pl->max_chunk_points * 16, cudaHostAllocDefault)) != cudaSuccess)
        return fail(e);
    if (!s.h_offsets && (e = cudaHostAlloc(&s.h_offsets, (size_t)(kMaxChunkScans + 1) * 8, cudaHostAllocDefault)) != cudaSuccess)
        return fail(e);
    if (s.busy) {           // the previous use of this slot's staging and device buffers
        if ((e = cudaEventSynchronize(s.done)) != cudaSuccess) return fail(e);
        s.busy = false;
    }
    s.h_offsets[0] = 0;
    s.h_offsets[1] = n_points;
    if ((e = cudaMemcpyAsync(s.d_offsets, s.h_offsets, 16, cudaMemcpyHostToDevice, cs)) != cudaSuccess) return fail(e);
    if (!pl->pool) {
        unsigned hw = std::thread::hardware_concurrency();
        pl->pool = new StagePool();
        pl->pool->start(hw >= 8 ? 3 : hw >= 4 ? 1 : 0, pl->device);
    }
    const size_t bytes = (size_t)n_points * point_stride * 4;
    if (bytes && (e = pl->pool->run(h_points, s.h_stage, s.d_points, bytes, 256 << 10, cs)) != cudaSuccess) return fail(e);
    EncodeOutputs out;
    out.rows = d_out;
    st = launch_encode({s.d_points, point_stride, s.d_offsets, 0, 1}, dp, out, s.d_ws, 256, cs);
    if (st == NSC_OK) {
        if ((e = cudaEventRecord(s.done, cs)) != cudaSuccess) return fail(e);
        s.busy = true;
    }
    cudaSetDevice(prev);
    return st;
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
        const uint32_t key = classify(q[0], q[1], q[2], dp, dp.row_mode, row_b, col_b);
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
