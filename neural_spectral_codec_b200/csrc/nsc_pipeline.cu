// Host-buffer pipeline of libnsc_b200.so (nsc_pipeline_*, declared in include/nsc_b200.h): scans in
// host memory go to the device in chunks through per-slot buffers and streams, are encoded there,
// and their rows come back, the copies of one chunk overlapping the kernel of another. Width 360
// runs the kernels of nsc_encode.cu, every other width those of nsc_anywidth.cu.
#include <string.h>

#include <atomic>
#include <condition_variable>
#include <mutex>
#include <thread>
#include <vector>

#include "nsc_internal.h"

using namespace nsc;

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

// Makes `device` current for the scope and gives the caller its device back on every return.
struct DeviceScope {
    int prev = 0;
    cudaError_t err;
    explicit DeviceScope(int device) : err(cudaGetDevice(&prev)) {
        if (err == cudaSuccess) err = cudaSetDevice(device);
    }
    ~DeviceScope() {
        if (err == cudaSuccess) cudaSetDevice(prev);
    }
};

static const int kMaxChunkScans = 1024;
static const int kMaxDescriptor = NSC_MAX_DESCRIPTOR;

struct nsc_pipeline {
    int device;
    int n_buffers;
    int sms;
    int64_t max_chunk_points;
    // A slot's buffers may be reused only when it is not busy. busy: `done` was recorded after the
    // last enqueued work that reads or writes these buffers, on whichever stream that work went
    // to. wait() and mark() below are the only code that reads or sets it.
    struct Slot {
        cudaStream_t stream;
        cudaEvent_t done;
        float* d_points;
        long long* d_offsets;
        float* d_out;
        unsigned* d_ws;
        void* d_any_ws;        // workspace of the other widths' kernels, lazy, grown on demand
        size_t any_ws_bytes;
        float* h_stage;        // pinned staging of one chunk (list path, single scans), lazy
        long long* h_offsets;  // pinned chunk offsets, lazy
        float* h_out;          // pinned chunk descriptors (list path), lazy
        bool busy;
    } slot[4];
    unsigned next_single;      // rotation of nsc_pipeline_encode_scan over the slots
    StagePool* pool;           // lazily started by nsc_pipeline_encode_scan
};

using Slot = nsc_pipeline::Slot;

// Waits until the work that last used the slot's buffers has finished.
static cudaError_t wait(Slot& s) {
    if (!s.busy) return cudaSuccess;
    const cudaError_t e = cudaEventSynchronize(s.done);
    if (e == cudaSuccess) s.busy = false;
    return e;
}

// Called on every return path after work that uses the slot's buffers was enqueued on `stream`. If
// the event cannot be recorded, the stream is synchronised instead and the record's error returned.
static cudaError_t mark(Slot& s, cudaStream_t stream) {
    const cudaError_t e = cudaEventRecord(s.done, stream);
    s.busy = e == cudaSuccess;
    if (!s.busy) cudaStreamSynchronize(stream);
    return e;
}

// Pinned staging of points and offsets (and of the rows if need_out), allocated on first use.
static cudaError_t ensure_pinned(const nsc_pipeline* pl, Slot& s, bool need_out) {
    cudaError_t e = cudaSuccess;
    if (!s.h_stage) e = cudaHostAlloc(&s.h_stage, (size_t)pl->max_chunk_points * 16, cudaHostAllocDefault);
    if (e == cudaSuccess && !s.h_offsets)
        e = cudaHostAlloc(&s.h_offsets, (size_t)(kMaxChunkScans + 1) * 8, cudaHostAllocDefault);
    if (e == cudaSuccess && need_out && !s.h_out)
        e = cudaHostAlloc(&s.h_out, (size_t)kMaxChunkScans * kMaxDescriptor * 4, cudaHostAllocDefault);
    return e;
}

// What a call encodes with: at 360 columns the kernels of nsc_encode.cu with `dp`, at any other
// width those of nsc_anywidth.cu with p and h_lut.
struct Encoder {
    const nsc_params* p;
    const int32_t* h_lut;
    bool any_width;
    DeviceParams dp;
};

// The parameter and table checks of the entry point each width's kernels have: nsc_encode_batch's
// at 360 columns (and for a null or foreign parameter block), nsc_anywidth_points' at the others.
static int prepare(const nsc_params* p, const int32_t* h_lut, Encoder* enc) {
    enc->p = p;
    enc->h_lut = h_lut;
    enc->any_width = p && p->struct_size == (int32_t)sizeof(nsc_params) && p->n_azimuth != NSC_N_AZIMUTH;
    return enc->any_width ? check_anywidth(p, h_lut) : make_device_params(p, h_lut, &enc->dp);
}

// The one encode launch of every entry point: scans `in` of the slot's buffers, rows to out.rows or
// out.rows_q, on `stream`. The other widths' workspace (the bin table and the general kernel's
// per-CTA scratch for the grid of this launch) is allocated on first use and grown when a later call
// needs more; the caller has waited for the slot, so nothing in flight still uses it.
static int encode(const nsc_pipeline* pl, Slot& s, const Encoder& enc, const PointBatch& in,
                  const EncodeOutputs& out, cudaStream_t stream) {
    if (!enc.any_width) return launch_encode(in, enc.dp, out, s.d_ws, 256, stream);
    const int grid = in.n_scans < 2 * pl->sms ? in.n_scans : 2 * pl->sms;
    const size_t need = nsc_anywidth_workspace_bytes(grid, enc.p->n_elevation, enc.p);
    if (s.any_ws_bytes < need) {
        if (s.d_any_ws) cudaFree(s.d_any_ws);
        s.d_any_ws = nullptr;
        s.any_ws_bytes = 0;
        const cudaError_t e = cudaMalloc(&s.d_any_ws, need);
        if (e != cudaSuccess) return record_cuda(e);
        s.any_ws_bytes = need;
    }
    const int64_t* offsets = (const int64_t*)in.offsets;
    if (out.rows_q)
        return nsc_anywidth_points_u16(in.points, in.stride, offsets, in.origin, in.n_scans, enc.p, enc.h_lut,
                                       out.q_eps, out.rows_q, s.d_any_ws, s.any_ws_bytes, stream);
    return nsc_anywidth_points(in.points, in.stride, offsets, in.origin, in.n_scans, enc.p, enc.h_lut, out.rows,
                               nullptr, NSC_STAGE_INTERPOLATED, s.d_any_ws, s.any_ws_bytes, stream);
}

// The checks both batch entry points make first, in this order. NSC_OK with n_scans == 0 means
// there is nothing to do.
static int check_batch(const nsc_pipeline* pl, const nsc_params* p, const int32_t* h_lut, int n_scans,
                       int stride, const void* h_points, const void* h_index, const void* h_out, Encoder* enc) {
    if (!pl) return NSC_ERR_NULL_POINTER;
    const int st = prepare(p, h_lut, enc);
    if (st != NSC_OK) return st;
    if (n_scans < 0) return NSC_ERR_BAD_COUNT;
    if (stride != 3 && stride != 4) return NSC_ERR_BAD_STRIDE;
    if (n_scans > 0 && (!h_points || !h_index || !h_out)) return NSC_ERR_NULL_POINTER;
    return NSC_OK;
}

// The chunk loop of both batch entry points, on pl->device. The scans [first, chunk_end(first)) go
// to the next slot: put(slot, first, last, &origin) enqueues their points and offsets (relative to
// `origin`) on slot.stream, and their rows come back on that stream straight into h_out or, with
// `bounce`, through the slot's pinned h_out. Returns when every slot is free and h_out complete.
template <class ChunkEnd, class Put>
static int run_chunks(nsc_pipeline* pl, int n_scans, int stride, const Encoder& enc, void* h_out,
                      size_t out_bytes, float q_eps, bool bounce, ChunkEnd chunk_end, Put put) {
    const size_t row_bytes = (size_t)enc.p->target_rows * enc.p->n_bins * out_bytes;
    EncodeOutputs out;
    out.q_eps = q_eps;
    // bounced rows of THIS call still in a slot's h_out; a slot that another call left busy has none
    struct Pending { int first, count; };
    Pending pending[4] = {};
    auto retire = [&](int i) -> int {
        const cudaError_t e = wait(pl->slot[i]);
        if (e != cudaSuccess) return record_cuda(e);
        if (pending[i].count)
            memcpy((char*)h_out + pending[i].first * row_bytes, pl->slot[i].h_out, pending[i].count * row_bytes);
        pending[i].count = 0;
        return NSC_OK;
    };
    int st = NSC_OK;
    for (int first = 0, k = 0; first < n_scans && st == NSC_OK; ++k) {
        const int i = k % pl->n_buffers, last = chunk_end(first), ns = last - first;
        Slot& s = pl->slot[i];
        if ((st = retire(i)) != NSC_OK) break;
        long long origin = 0;
        st = record_cuda(put(s, first, last, &origin));
        if (out_bytes == 4) out.rows = s.d_out;
        else out.rows_q = reinterpret_cast<unsigned short*>(s.d_out);
        if (st == NSC_OK)
            st = encode(pl, s, enc, {s.d_points, stride, s.d_offsets, origin, ns}, out, s.stream);
        if (st == NSC_OK)
            st = record_cuda(cudaMemcpyAsync(bounce ? (void*)s.h_out : (char*)h_out + first * row_bytes, s.d_out,
                                             ns * row_bytes, cudaMemcpyDeviceToHost, s.stream));
        const cudaError_t e = mark(s, s.stream);      // after a failure too: the copies may be queued
        if (st == NSC_OK) st = record_cuda(e);
        if (bounce) pending[i] = {first, ns};
        first = last;
    }
    for (int i = 0; i < pl->n_buffers; ++i) {
        if (st == NSC_OK) st = retire(i);
        else wait(pl->slot[i]);
    }
    return st;
}

// Descriptors of out_bytes (4 or 2) per element, the uint16 ones in the first half of the slot's
// float32 descriptor buffer. Points go to the device straight from the caller's buffer.
static int pipeline_encode(nsc_pipeline* pl, const float* h_points, int point_stride, int64_t n_points,
                           const int64_t* h_offsets, int n_scans, const nsc_params* p, const int32_t* h_lut,
                           void* h_out, size_t out_bytes, float q_eps) {
    Encoder enc;
    const int st = check_batch(pl, p, h_lut, n_scans, point_stride, h_points, h_offsets, h_out, &enc);
    if (st != NSC_OK || n_scans == 0) return st;
    if (n_points < 0) return NSC_ERR_BAD_COUNT;
    if (h_offsets[0] < 0 || h_offsets[n_scans] > n_points) return NSC_ERR_BAD_OFFSETS;
    for (int i = 0; i < n_scans; ++i)
        if (h_offsets[i + 1] < h_offsets[i]) return NSC_ERR_BAD_OFFSETS;
    for (int i = 0; i < n_scans; ++i)
        if (h_offsets[i + 1] - h_offsets[i] > pl->max_chunk_points) return NSC_ERR_WORKSPACE;
    DeviceScope on(pl->device);
    if (on.err != cudaSuccess) return record_cuda(on.err);
    // as many whole scans as fit the staging buffer
    auto chunk_end = [&](int first) {
        int last = first;
        while (last < n_scans && last - first < kMaxChunkScans &&
               h_offsets[last + 1] - h_offsets[first] <= pl->max_chunk_points)
            ++last;
        return last;
    };
    auto put = [&](Slot& s, int first, int last, long long* origin) {
        *origin = h_offsets[first];
        cudaError_t e = cudaMemcpyAsync(s.d_points, h_points + *origin * point_stride,
                                        (size_t)(h_offsets[last] - *origin) * point_stride * 4,
                                        cudaMemcpyHostToDevice, s.stream);
        if (e == cudaSuccess)
            e = cudaMemcpyAsync(s.d_offsets, h_offsets + first, (size_t)(last - first + 1) * 8,
                                cudaMemcpyHostToDevice, s.stream);
        return e;
    };
    return run_chunks(pl, n_scans, point_stride, enc, h_out, out_bytes, q_eps, false, chunk_end, put);
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

// Descriptors as in pipeline_encode. Scans are gathered into the slot's pinned staging, and rows
// come back through its pinned h_out.
static int pipeline_encode_scans(nsc_pipeline* pl, const float* const* h_scans, const int64_t* h_counts,
                                 int point_stride, int n_scans, const nsc_params* p, const int32_t* h_lut,
                                 void* h_out, size_t out_bytes, float q_eps) {
    Encoder enc;
    const int st = check_batch(pl, p, h_lut, n_scans, point_stride, h_scans, h_counts, h_out, &enc);
    if (st != NSC_OK || n_scans == 0) return st;
    for (int i = 0; i < n_scans; ++i) {
        if (h_counts[i] < 0) return NSC_ERR_BAD_OFFSETS;
        if (h_counts[i] > 0 && !h_scans[i]) return NSC_ERR_NULL_POINTER;
        if (h_counts[i] > pl->max_chunk_points) return NSC_ERR_WORKSPACE;
    }
    DeviceScope on(pl->device);
    if (on.err != cudaSuccess) return record_cuda(on.err);
    for (int i = 0; i < pl->n_buffers; ++i) {
        const cudaError_t e = ensure_pinned(pl, pl->slot[i], true);
        if (e != cudaSuccess) return record_cuda(e);
    }
    auto chunk_end = [&](int first) {
        int last = first;
        int64_t np = 0;
        while (last < n_scans && last - first < kMaxChunkScans && np + h_counts[last] <= pl->max_chunk_points)
            np += h_counts[last++];
        return last;
    };
    auto put = [&](Slot& s, int first, int last, long long* origin) {
        *origin = 0;
        stage_scans(s.h_stage, h_scans, h_counts, first, last, point_stride, s.h_offsets);
        cudaError_t e = cudaMemcpyAsync(s.d_points, s.h_stage, (size_t)s.h_offsets[last - first] * point_stride * 4,
                                        cudaMemcpyHostToDevice, s.stream);
        if (e == cudaSuccess)
            e = cudaMemcpyAsync(s.d_offsets, s.h_offsets, (size_t)(last - first + 1) * 8, cudaMemcpyHostToDevice,
                                s.stream);
        return e;
    };
    return run_chunks(pl, n_scans, point_stride, enc, h_out, out_bytes, q_eps, true, chunk_end, put);
}

extern "C" {

void nsc_pipeline_destroy(nsc_pipeline* pl) {
    if (!pl) return;
    DeviceScope on(pl->device);
    for (int i = 0; i < pl->n_buffers; ++i) {
        Slot& s = pl->slot[i];
        wait(s);
        if (s.d_points) cudaFree(s.d_points);
        if (s.d_offsets) cudaFree(s.d_offsets);
        if (s.d_out) cudaFree(s.d_out);
        if (s.d_ws) cudaFree(s.d_ws);
        if (s.d_any_ws) cudaFree(s.d_any_ws);
        if (s.h_stage) cudaFreeHost(s.h_stage);
        if (s.h_offsets) cudaFreeHost(s.h_offsets);
        if (s.h_out) cudaFreeHost(s.h_out);
        if (s.done) cudaEventDestroy(s.done);
        if (s.stream) cudaStreamDestroy(s.stream);
    }
    delete pl->pool;
    delete pl;
}

int nsc_pipeline_create(int64_t max_chunk_points, int n_buffers, int device, nsc_pipeline** out) {
    if (!out) return NSC_ERR_NULL_POINTER;
    *out = nullptr;
    if (max_chunk_points < 1 || n_buffers < 1 || n_buffers > 4) return NSC_ERR_BAD_COUNT;
    DeviceScope on(device);
    if (on.err != cudaSuccess) return record_cuda(on.err);
    nsc_pipeline* pl = new nsc_pipeline();
    memset(pl, 0, sizeof(*pl));
    pl->device = device;
    pl->n_buffers = n_buffers;
    pl->max_chunk_points = max_chunk_points;
    const cudaError_t e_sms = cudaDeviceGetAttribute(&pl->sms, cudaDevAttrMultiProcessorCount, device);
    if (e_sms != cudaSuccess) {
        nsc_pipeline_destroy(pl);
        return record_cuda(e_sms);
    }
    for (int i = 0; i < n_buffers; ++i) {
        Slot& s = pl->slot[i];
        cudaError_t e;
        if ((e = cudaStreamCreateWithFlags(&s.stream, cudaStreamNonBlocking)) != cudaSuccess ||
            (e = cudaEventCreateWithFlags(&s.done, cudaEventDisableTiming)) != cudaSuccess ||
            (e = cudaMalloc(&s.d_points, (size_t)max_chunk_points * 16)) != cudaSuccess ||
            (e = cudaMalloc(&s.d_offsets, (size_t)(kMaxChunkScans + 1) * 8)) != cudaSuccess ||
            (e = cudaMalloc(&s.d_out, (size_t)kMaxChunkScans * kMaxDescriptor * 4)) != cudaSuccess ||
            (e = cudaMalloc(&s.d_ws, 256)) != cudaSuccess) {
            nsc_pipeline_destroy(pl);
            return record_cuda(e);
        }
    }
    *out = pl;
    return NSC_OK;
}

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
// kernel follows on the same stream. Returns when the source array may be reused; nothing is
// synchronised but the slot's previous use.
int nsc_pipeline_encode_scan(nsc_pipeline* pl, const float* h_points, int point_stride, int64_t n_points,
                             const nsc_params* p, const int32_t* h_lut, float* d_out, void* stream) {
    if (!pl) return NSC_ERR_NULL_POINTER;
    Encoder enc;
    int st = prepare(p, h_lut, &enc);
    if (st != NSC_OK) return st;
    if (point_stride != 3 && point_stride != 4) return NSC_ERR_BAD_STRIDE;
    if (n_points < 0) return NSC_ERR_BAD_COUNT;
    if (n_points > pl->max_chunk_points) return NSC_ERR_WORKSPACE;
    if ((n_points && !h_points) || !d_out) return NSC_ERR_NULL_POINTER;
    DeviceScope on(pl->device);
    if (on.err != cudaSuccess) return record_cuda(on.err);
    Slot& s = pl->slot[pl->next_single++ % pl->n_buffers];
    cudaStream_t cs = (cudaStream_t)stream;
    cudaError_t e = ensure_pinned(pl, s, false);
    if (e == cudaSuccess) e = wait(s);
    if (e != cudaSuccess) return record_cuda(e);
    s.h_offsets[0] = 0;
    s.h_offsets[1] = n_points;
    if (!pl->pool) {
        unsigned hw = std::thread::hardware_concurrency();
        pl->pool = new StagePool();
        pl->pool->start(hw >= 8 ? 3 : hw >= 4 ? 1 : 0, pl->device);
    }
    e = cudaMemcpyAsync(s.d_offsets, s.h_offsets, 16, cudaMemcpyHostToDevice, cs);
    const size_t bytes = (size_t)n_points * point_stride * 4;
    if (e == cudaSuccess && bytes) e = pl->pool->run(h_points, s.h_stage, s.d_points, bytes, 256 << 10, cs);
    st = record_cuda(e);
    if (st == NSC_OK) {
        EncodeOutputs out;
        out.rows = d_out;
        st = encode(pl, s, enc, {s.d_points, point_stride, s.d_offsets, 0, 1}, out, cs);
    }
    e = mark(s, cs);
    return st != NSC_OK ? st : record_cuda(e);
}

}  // extern "C"
