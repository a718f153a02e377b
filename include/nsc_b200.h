/*
 * nsc_b200.h -- C ABI of the B200-native spectral encoding front end.
 *
 * Drop-in boundary for ONE path of Kimun-Park/Neural-Spectral-Codec:
 *     points -> E x 360 min-range image -> hole interpolation -> row-wise 360-pt
 *     rFFT magnitude -> n_bins exponential histogram per row -> L1-normalised
 *     (target_rows * n_bins)-D descriptor.
 *
 * The reference has no FFI layer for this path; its boundary is the Python class
 * SpectralEncoder (reference src/encoding/spectral_encoder.py:24-261) calling
 * RangeImageProjector.project / interpolate_range_image
 * (reference src/encoding/range_image.py:129-232, :15-89). Each entry point below
 * names the reference interface it replaces. The Python host mirror that binds this
 * header with ctypes is neural_spectral_codec_b200/encoder.py; INTEGRATION.md shows the
 * stub a maintainer of the reference would add.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes; no C++ or torch types cross this boundary.
 *   - d_* pointers are CUDA device pointers, h_* pointers are host pointers.
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream). All
 *     device work is enqueued on it; entry points taking d_* pointers never synchronise.
 *   - The caller owns every buffer. The library keeps no mutable global state; the only
 *     per-process caches are immutable device attributes (SM count, occupancy).
 *   - Every function returns NSC_OK (0) or a negative nsc_status; nothing throws.
 *   - There is no CPU fallback: without a CUDA device every compute entry point returns
 *     NSC_ERR_CUDA.
 */
#ifndef NSC_B200_H
#define NSC_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NSC_ABI_VERSION 2
#define NSC_N_AZIMUTH 360        /* the in-kernel FFT is a 360-point transform            */
#define NSC_N_FREQS 181          /* n_azimuth/2 + 1, spectral_encoder.py:88               */
/* Rows of the projected image, held whole in one CTA's shared memory: up to 64 rows for every
 * parameter block, up to 128 (one row per beam of a 128-beam sensor) for one that sets
 * NSC_FLAG_TALL_IMAGES in nsc_params.flags. Images of more than 64 rows take their own kernels (one
 * image per SM) and are pooled to target_rows <= 64 before the spectrum. A parameter block without
 * the flag -- e.g. one filled for a library that stopped at 64 rows -- is refused above 64 rows with
 * NSC_ERR_BAD_PARAMS, as before; libraries older than the flag ignore it and refuse 65..128 rows the
 * same way. */
#define NSC_MAX_ELEVATION 128
#define NSC_MAX_ELEVATION_SHORT 64
#define NSC_FLAG_TALL_IMAGES 1   /* nsc_params.flags: accept rows up to NSC_MAX_ELEVATION */
#define NSC_MAX_TARGET_ROWS 64
#define NSC_MAX_BINS 181
#define NSC_MAX_DESCRIPTOR 4096  /* target_rows * n_bins held in shared memory             */
#define NSC_MAX_PEERS 8          /* GPUs of one NVSwitch box written by the fused all-gather */

typedef enum nsc_status {
    NSC_OK = 0,
    NSC_ERR_NULL_POINTER = -1,
    NSC_ERR_BAD_STRIDE = -2,       /* point stride must be 3 or 4 floats                  */
    NSC_ERR_BAD_COUNT = -3,        /* negative n_scans / n_images                          */
    NSC_ERR_BAD_PARAMS = -4,       /* nsc_params outside the supported envelope            */
    NSC_ERR_BAD_LUT = -5,          /* freq->bin table not monotone / out of range          */
    NSC_ERR_WORKSPACE = -6,        /* workspace missing or too small                       */
    NSC_ERR_ALIGNMENT = -7,        /* stride-4 points must be 16-byte aligned              */
    NSC_ERR_BAD_OFFSETS = -8,      /* host offsets not monotone / outside the point buffer */
    NSC_ERR_CUDA = -9,             /* CUDA runtime error (see nsc_last_cuda_error)         */
    NSC_ERR_BAD_STRUCT = -10       /* struct_size does not match this ABI                  */
} nsc_status;

/* Encoder constants. Mirrors the constructor of the reference encoder
 * (spectral_encoder.py:35-47) and the projector defaults it never forwards
 * (range_image.py:102-109). POD; set struct_size = sizeof(nsc_params). */
typedef struct nsc_params {
    int32_t struct_size;
    int32_t n_elevation;        /* rows of the projected image, 1..NSC_MAX_ELEVATION_SHORT,
                                   1..NSC_MAX_ELEVATION with NSC_FLAG_TALL_IMAGES               */
    int32_t n_azimuth;          /* NSC_N_AZIMUTH for the fused kernels; nsc_anywidth_* take others */
    int32_t n_bins;             /* histogram bins per row, 1..NSC_MAX_BINS                  */
    int32_t target_rows;        /* target_elevation_bins; rows are average-pooled to this   */
    int32_t interpolate_empty;  /* 1 = fill empty pixels before the FFT (reference default) */
    float min_range;            /* 1.0  (range_image.py:108)                                */
    float max_range;            /* 80.0 (range_image.py:107)                                */
    double el_min_rad;          /* np.deg2rad(elevation_range[0]) (range_image.py:126)      */
    double el_max_rad;          /* np.deg2rad(elevation_range[1]) (range_image.py:127)      */
    float epsilon;              /* 1e-8 (spectral_encoder.py:42)                            */
    int32_t flags;              /* NSC_FLAG_*; 0 from nsc_default_params (formerly reserved) */
} nsc_params;

/* Which image nsc_project_batch writes out. */
#define NSC_STAGE_PROJECTED 0      /* RangeImageProjector.project output (range_image.py:129-214) */
#define NSC_STAGE_INTERPOLATED 1   /* after interpolate_range_image (range_image.py:15-89)        */

int nsc_abi_version(void);
const char* nsc_strerror(int status);
/* Text of the last CUDA error seen by the calling thread ("" if none). */
const char* nsc_last_cuda_error(void);
/* Fills defaults of the reference constructor for a 16-row encoder. */
void nsc_default_params(nsc_params* p);

/* freq -> bin table of SpectralEncoder._bin_fft_magnitudes (spectral_encoder.py:136-145)
 * computed in float32 C arithmetic: edges[i] = (exp(a*i/n_bins)-1)/(exp(a)-1+eps)*n_freqs
 * (spectral_encoder.py:107-114), bin[k] = clamp(upper_bound(edges, k) - 1, 0, n_bins-1).
 * The Python host passes the table it computed with the reference's own torch calls; this
 * function serves non-Python callers and is tested equal to it. h_lut has NSC_N_FREQS ints. */
int nsc_freq_to_bin(float alpha, const nsc_params* p, int32_t* h_lut);

/* Device workspace of nsc_encode_batch / nsc_encode_batch_peers / nsc_project_batch. 256 bytes (the
 * work counter) are enough for every call and smaller workspaces are refused; the RECOMMENDED size
 * returned here (a few MB) also holds one key image per scan of the grid's last, partial wave,
 * which lets a batch whose last wave fills at most half of the SMs split those scans over all
 * of them (+5 % on 600 scans); images of more than 64 rows split no scan and get the 256 bytes.
 * The result does not depend on the workspace size. Contents need no initialisation. */
size_t nsc_workspace_bytes(int n_scans, const nsc_params* p);

/* Replaces a loop of SpectralEncoder.encode_points (spectral_encoder.py:206-229; callers
 * src/pipeline.py:245,351, train_multi_dataset.py:182) over n_scans scans.
 *   d_points   concatenated scans, float32, point_stride (3 or 4) floats per point, AoS
 *              xyz[i] exactly as the reference loaders produce (kitti_loader.py:100-115)
 *   d_offsets  int64[n_scans+1] CSR offsets in POINTS; scan i = [offsets[i]-point_origin,
 *              offsets[i+1]-point_origin) relative to d_points
 *   h_lut      int32[NSC_N_FREQS] freq->bin table on the HOST (monotone non-decreasing)
 *   d_out      float32[n_scans * target_rows * n_bins], row-major (scan, row, bin) -- the
 *              layout of histograms.flatten() (spectral_encoder.py:158)
 * One fused kernel launch; the range image, its interpolation and the spectrum live in
 * shared memory only. */
int nsc_encode_batch(const float* d_points, int point_stride, const int64_t* d_offsets,
                     int64_t point_origin, int n_scans, const nsc_params* p,
                     const int32_t* h_lut, float* d_out, void* d_workspace,
                     size_t workspace_bytes, void* stream);

/* nsc_encode_batch straight to the descriptor wire format: each row is normalised as above and
 * quantised in the same kernel's epilogue exactly as nsc_quantize_histograms (below) would quantise
 * the float32 row nsc_encode_batch writes -- the same integers for every row, empty scans included --
 * without the float32 round trip through device memory.
 *   q_epsilon  the quantiser's epsilon (HistogramQuantizer default 1e-8; independent of p->epsilon)
 *   d_out      uint16[n_scans * target_rows * n_bins], each row summing to 65535 (a row whose
 *              rounded total is 0 stays all zero, as in the reference)
 * Arguments are validated in the order of nsc_encode_batch, with the same status codes. */
int nsc_encode_batch_u16(const float* d_points, int point_stride, const int64_t* d_offsets,
                         int64_t point_origin, int n_scans, const nsc_params* p,
                         const int32_t* h_lut, float q_epsilon, uint16_t* d_out, void* d_workspace,
                         size_t workspace_bytes, void* stream);

/* nsc_encode_batch fused with the all-gather that follows it in a multi-GPU encode
 * (SURVEY.md 8(e): the replicated descriptor database that
 * WassersteinRetriever.add_to_database, reference src/retrieval/wasserstein.py:300-326, would
 * hold). Each descriptor is stored by the encode kernel's epilogue straight into row
 * db_row0 + i of EVERY database in h_peer_db[0..n_peers): host array of device pointers, one
 * per GPU of the box, peer-mapped into this process (CUDA IPC / symmetric memory), the local
 * database included. No separate collective pass; the caller synchronises all ranks
 * afterwards (nsc_peer_signal_wait below, or any barrier), exactly as after an NCCL all-gather. */
int nsc_encode_batch_peers(const float* d_points, int point_stride, const int64_t* d_offsets,
                           int64_t point_origin, int n_scans, const nsc_params* p,
                           const int32_t* h_lut, float* const* h_peer_db, int n_peers,
                           int64_t db_row0, void* d_workspace, size_t workspace_bytes, void* stream);

/* The synchronisation of a fused multi-GPU step, as ONE small kernel on `stream` (after the
 * nsc_encode_batch_peers launch): tells every peer "rank `rank` has stored step signal_value" by a
 * system-scope release store into the peer's flag array, then spins with system-scope acquire
 * loads until every peer has announced at least wait_value. h_peer_flags[p]: device pointer
 * (peer-mapped) to rank p's array of n_peers uint32 flags, zero before the first step;
 * signal_value must grow by one per step.
 *   wait_value == signal_value      the step's database is complete when the kernel ends. With the
 *       database double-buffered by the caller (step s writes buffer s & 1) no barrier is needed
 *       BEFORE the encode: a rank that returns from the wait of step s-1 knows every peer has
 *       passed, in stream order, everything it enqueued before its own step s-1 -- including
 *       whatever read buffer s & 1 after step s-2.
 *   wait_value == signal_value - 1  a rank may run one step ahead of the slowest peer (the wait
 *       practically never blocks); step s-1 is complete when the kernel ends. Needs FOUR buffers
 *       (step s writes buffer s & 3): leaving the wait for s-2 means every peer has finished its
 *       own step s-2, which it started after consuming step s-4. */
int nsc_peer_signal_wait(uint32_t* const* h_peer_flags, int n_peers, int rank, uint32_t signal_value,
                         uint32_t wait_value, void* stream);

/* Replaces RangeImageProjector.project(points, keep_intensity=False)[0]
 * (stage = NSC_STAGE_PROJECTED) optionally followed by interpolate_range_image
 * (stage = NSC_STAGE_INTERPOLATED). d_images: float32[n_scans * n_elevation * 360].
 * Used by the parity tests and by the projector attribute of the Python mirror. */
int nsc_project_batch(const float* d_points, int point_stride, const int64_t* d_offsets,
                      int64_t point_origin, int n_scans, const nsc_params* p, int stage,
                      float* d_images, void* d_workspace, size_t workspace_bytes, void* stream);

/* Replaces RangeImageProjector.project(points, keep_intensity=True) (range_image.py:129-232):
 * the range image and the intensity image (intensity of the closest point per pixel; the largest
 * one when several points tie on the range, :217-226). 4-float points only. Not on the encoding
 * path (spectral_encoder.py:217 passes keep_intensity=False); one packed 64-bit atomicMin on
 * (range bits, ~intensity bits) per point. Both outputs: float32[n_scans * n_elevation * 360]. */
int nsc_project_intensity_batch(const float* d_points, const int64_t* d_offsets,
                                int64_t point_origin, int n_scans, const nsc_params* p,
                                float* d_range_images, float* d_intensity_images, void* stream);

/* Replaces SpectralEncoder.forward / encode_batch / encode_range_image
 * (spectral_encoder.py:160-204, :231-261): range images in, no projection and no
 * interpolation; rows are average-pooled to target_rows when they differ
 * (spectral_encoder.py:171-176). d_images: float32[n_images * rows * 360]. */
int nsc_encode_range_images(const float* d_images, int n_images, int rows, const nsc_params* p,
                            const int32_t* h_lut, float* d_out, void* stream);

/* Replaces interpolate_range_image(img, method) (range_image.py:15-89) on a batch of images
 * already on the device: method NSC_INTERP_LINEAR = circular linear interpolation along azimuth
 * (the encoder's path), NSC_INTERP_NEAREST = nearest valid pixel (:66-75, the lower column on a
 * tie); both followed by the empty-row fill (:77-87). In and out may alias. */
#define NSC_INTERP_LINEAR 0
#define NSC_INTERP_NEAREST 1
int nsc_interpolate_range_images(const float* d_images_in, int n_images, int rows, int method,
                                 float* d_images_out, void* stream);

/* ---- image widths other than 360 columns ----------------------------------------------------
 * The reference accepts any n_azimuth (spectral_encoder.py:35-47, range_image.py:102-127); every
 * shipped config uses 360, which the entry points above are specialised to (they refuse other
 * widths with NSC_ERR_BAD_PARAMS). These two cover 2 <= n_azimuth <= 4096 with two kernels and the
 * same results to the same tolerances. A call with d_out set, a width whose prime factors are all at
 * most 13 and an image that fits one block's shared memory (nsc_test_anywidth_path) runs a fused
 * kernel: image, fp32 mixed-radix FFT and histogram in shared memory, ~1.5 us per scan on a whole
 * B200 (about a fifth of the 360-column rate). Every other call runs a general kernel (the
 * reference's own operation order for the projection, a direct float64 DFT per row), ~0.1-0.3 ms
 * per scan per CTA. Both give bit-identical range images. h_lut has
 * n_azimuth / 2 + 1 entries. Workspace: nsc_anywidth_workspace_bytes(n, rows, p), enough for both
 * kernels, needs no initialisation.
 *   nsc_anywidth_points  encode_points / project [+ interpolate_range_image] for n_scans scans:
 *       d_out (descriptors, float32[n_scans * target_rows * n_bins]) and / or d_images
 *       (float32[n_scans * n_elevation * n_azimuth], the image named by `stage`); either may be NULL
 *   nsc_anywidth_points_u16  nsc_anywidth_points straight to the wire format of nsc_encode_batch_u16:
 *       d_out uint16[n_scans * target_rows * n_bins], each row the integers nsc_quantize_histograms
 *       (q_epsilon) gives for the float32 row nsc_anywidth_points writes for the same call (empty and
 *       fully filtered scans included), quantised in the same kernel's epilogue. No images. The call
 *       runs the kernel the float32 call runs, with the same workspace; arguments are validated in
 *       nsc_anywidth_points' order, with the same status codes
 *   nsc_anywidth_images  forward / encode_range_image (interp_method = -1: no interpolation, as the
 *       reference's forward) and interpolate_range_image (d_out NULL, d_images_out set,
 *       interp_method NSC_INTERP_LINEAR | NSC_INTERP_NEAREST) on images already on the device */
size_t nsc_anywidth_workspace_bytes(int n, int rows, const nsc_params* p);
int nsc_anywidth_points(const float* d_points, int point_stride, const int64_t* d_offsets, int64_t point_origin,
                        int n_scans, const nsc_params* p, const int32_t* h_lut, float* d_out, float* d_images,
                        int stage, void* d_workspace, size_t workspace_bytes, void* stream);
int nsc_anywidth_points_u16(const float* d_points, int point_stride, const int64_t* d_offsets, int64_t point_origin,
                            int n_scans, const nsc_params* p, const int32_t* h_lut, float q_epsilon, uint16_t* d_out,
                            void* d_workspace, size_t workspace_bytes, void* stream);
int nsc_anywidth_images(const float* d_images_in, int n_images, int rows, const nsc_params* p, const int32_t* h_lut,
                        int interp_method, float* d_out, float* d_images_out, void* d_workspace,
                        size_t workspace_bytes, void* stream);

/* ---- host-buffer pipeline (the end-to-end call: H2D, encode, D2H inside) -------------- */
/* Every encode entry point of the pipeline accepts every image width the entry points above
 * accept: n_azimuth = 360 runs the kernels of nsc_encode_batch / nsc_encode_batch_u16 and is
 * validated as they validate; any other n_azimuth (2..4096) runs those of nsc_anywidth_points /
 * nsc_anywidth_points_u16 and is validated by their rules (h_lut then has n_azimuth / 2 + 1
 * entries). The rows are those the device entry points give for the same scans, however the scans
 * are chunked. At other widths each buffer also keeps the workspace of those kernels (for the
 * general kernel, per-CTA scratch of up to a few MB times the CTAs of one chunk): it is
 * allocated by the first call that needs it and grown by a later call that needs more. */
typedef struct nsc_pipeline nsc_pipeline;

/* Creates a pipeline that stages at most max_chunk_points points per chunk through
 * n_buffers (1..4) device staging buffers with one stream each. A pipeline serves one call at a
 * time (calls from several threads must not overlap on it). Its encode entry points may be mixed on
 * one pipeline: a buffer is reused only after the work that last used it, on whichever stream
 * (nsc_pipeline_encode_scan's included), has finished. */
int nsc_pipeline_create(int64_t max_chunk_points, int n_buffers, int device, nsc_pipeline** out);
void nsc_pipeline_destroy(nsc_pipeline* pl);

/* Same contract as nsc_encode_batch with HOST buffers: h_points (pinned memory gives full
 * PCIe rate; pageable works), h_offsets int64[n_scans+1] starting at 0, h_out
 * float32[n_scans * target_rows * n_bins]. Chunks of whole scans are copied H2D, encoded
 * and copied back D2H on rotating streams so copies overlap compute. Synchronous: returns
 * when h_out is complete. Offsets that decrease, start below 0 or end beyond n_points (the
 * length of h_points in points) return NSC_ERR_BAD_OFFSETS, and a scan larger than
 * max_chunk_points returns NSC_ERR_WORKSPACE, both before anything is copied. */
int nsc_pipeline_encode(nsc_pipeline* pl, const float* h_points, int point_stride,
                        int64_t n_points, const int64_t* h_offsets, int n_scans,
                        const nsc_params* p, const int32_t* h_lut, float* h_out);
/* The same with the wire format of nsc_encode_batch_u16 in h_out (uint16[n_scans * target_rows *
 * n_bins]): the rows a keyframe store keeps, in one call; 2 bytes per element cross PCIe instead of 4. */
int nsc_pipeline_encode_u16(nsc_pipeline* pl, const float* h_points, int point_stride,
                            int64_t n_points, const int64_t* h_offsets, int n_scans,
                            const nsc_params* p, const int32_t* h_lut, float q_epsilon, uint16_t* h_out);

/* ONE scan from pageable host memory to a descriptor on the DEVICE, on the caller's stream -- the
 * reference's own call shape: encoder.encode_points(numpy_scan) per scan (pipeline.py:245,
 * :336-354, train_multi_dataset.py:182), whose result lives on alpha.device. The scan is staged
 * through pinned memory in 256 KB pieces by the calling thread and up to three threads the
 * pipeline keeps for this, each piece going to the copy engine as soon as it is staged; the fused
 * kernel follows on `stream`. Returns as soon as h_points may be reused; d_out (float32[target_rows * n_bins]) is
 * complete in stream order. n_points <= max_chunk_points of the pipeline. */
int nsc_pipeline_encode_scan(nsc_pipeline* pl, const float* h_points, int point_stride, int64_t n_points,
                             const nsc_params* p, const int32_t* h_lut, float* d_out, void* stream);

/* The same for scans that live in SEPARATE host arrays, as the reference's loaders hand them
 * out one np.fromfile() at a time (kitti_loader.py:100-115) -- the loop of pipeline.py:336-354
 * without concatenating first. h_scans[i] points to h_counts[i] points of point_stride floats
 * (pageable memory is fine: chunks are gathered into pinned staging by a few host threads while
 * the previous chunk is on the wire). h_out: float32[n_scans * target_rows * n_bins]. */
int nsc_pipeline_encode_scans(nsc_pipeline* pl, const float* const* h_scans, const int64_t* h_counts,
                              int point_stride, int n_scans, const nsc_params* p,
                              const int32_t* h_lut, float* h_out);
/* ... and with uint16 rows of nsc_encode_batch_u16 in h_out (uint16[n_scans * target_rows * n_bins]). */
int nsc_pipeline_encode_scans_u16(nsc_pipeline* pl, const float* const* h_scans, const int64_t* h_counts,
                                  int point_stride, int n_scans, const nsc_params* p,
                                  const int32_t* h_lut, float q_epsilon, uint16_t* h_out);

/* ---- keyframe gate geometry (SURVEY.md 8(f), third "next" row) ------------------------------ */
/* Voxel-set IoU of n_pairs cloud pairs in one launch: the geometric-novelty criterion of the
 * reference's keyframe gate, compute_overlap (reference src/data/pose_utils.py:323-389) as called
 * by KeyframeSelectionCriteria.check_geometric_novelty (src/keyframe/criteria.py:96-131), AFTER
 * its random subsample (the caller draws it; the host mirror does so with the reference's NumPy
 * calls, so equal seeds give equal results).
 *   d_points   all clouds concatenated, float32 or float64 (points_are_f64), point_stride 3 | 4;
 *              with stride 4 a non-finite 4th column drops the point, as in the reference
 *   d_offsets  int64[2 * n_pairs + 1]: cloud A of pair i is points [off[2i], off[2i+1]), cloud B is
 *              [off[2i+1], off[2i+2])
 *   d_T        float64[n_pairs * 16], row-major 4x4 that maps A into B's frame (T_12)
 *   d_counts   int32[n_pairs * 3]: voxels of A, voxels of B, voxels in both
 *   d_iou      float64[n_pairs]: both / union, 0.0 for an empty union
 * total_points = off[2 * n_pairs]; max_pair_points >= the largest |A| + |B| (pairs of up to
 * 16384 points keep their hash set in shared memory). Workspace from
 * nsc_voxel_overlap_workspace_bytes(total_points, max_pair_points, n_pairs). */
size_t nsc_voxel_overlap_workspace_bytes(int64_t total_points, int64_t max_pair_points, int n_pairs);
int nsc_voxel_overlap_batch(const void* d_points, int point_stride, int points_are_f64,
                            const int64_t* d_offsets, int64_t total_points, int64_t max_pair_points,
                            const double* d_T, int n_pairs, double voxel_size, int32_t* d_counts,
                            double* d_iou, void* d_workspace, size_t workspace_bytes, void* stream);

/* ---- stage-1 retrieval over the descriptor database (SURVEY.md 8(f), first "next" row) ---- */
/* Normalised CDF rows of a block of database histograms: cdf = cumsum(h / (sum h + eps)) where
 * sum h > eps, cumsum(h) otherwise -- the database half of wasserstein_distance_batch_torch
 * (reference src/retrieval/wasserstein.py:157-166), computed once when rows are inserted
 * (WassersteinRetriever.add_to_database, :300-326) instead of on every query.
 * d_hists, d_cdfs: float32[n_rows * n_bins]; n_bins <= 1024. */
int nsc_wasserstein_cdf(const float* d_hists, int64_t n_rows, int n_bins, float epsilon,
                        float* d_cdfs, void* stream);

/* Replaces WassersteinRetriever.query (wasserstein.py:328-367) for n_queries queries at once,
 * with the spatial exclusion of TwoStageRetrieval._global_retrieval
 * (src/retrieval/two_stage_retrieval.py:158-166) folded in.
 *   d_query_hists  float32[n_queries * n_bins] raw query histograms (normalised in-kernel:
 *                  h / sum h where sum h > eps, wasserstein.py:152-154)
 *   d_db_cdfs      float32[n_db * n_bins] from nsc_wasserstein_cdf
 *   d_db_xyz, d_query_xyz  float64 positions (pose[:3, 3]); both NULL = no spatial filter;
 *                  database rows closer than min_spatial_distance (strict <) get distance +inf
 *   d_distances    float32[n_queries * n_db] OUT: sum_i |cdf_db[i] - cdf_q[i]| (also scratch
 *                  for the selection; always written)
 *   top_k          0 = distances only; else <= 1024: d_top_idx int64[n_queries * top_k] (-1
 *                  padded), d_top_dist float32 (ascending, +inf padded), d_top_count
 *                  int32[n_queries] = min(top_k, rows not excluded). Ties are broken by the
 *                  lower database index (deterministic). Larger top_k (up to the whole database):
 *                  nsc_wasserstein_rank below, which returns the same results for top_k <= 1024.
 *   d_workspace    nsc_wasserstein_workspace_bytes(n_queries) bytes, ZERO before the first call
 *                  (every call leaves it zero where it matters). With it, top_k <= 128 is selected
 *                  by many CTAs per query from per-warp minima kept by the distance pass; NULL or
 *                  larger top_k: one CTA per query re-reads the distances. Same result. */
size_t nsc_wasserstein_workspace_bytes(int n_queries);
int nsc_wasserstein_query(const float* d_query_hists, int n_queries, const float* d_db_cdfs,
                          int64_t n_db, int n_bins, float epsilon, const double* d_db_xyz,
                          const double* d_query_xyz, double min_spatial_distance,
                          float* d_distances, int top_k, int64_t* d_top_idx, float* d_top_dist,
                          int32_t* d_top_count, void* d_workspace, size_t workspace_bytes, void* stream);

/* The same database kept as uint16 rows: a quarter of the float32 database's bytes, and half the
 * bytes the distance pass streams per row.
 * nsc_wasserstein_cdf_u16 turns uint16 histogram rows (the wire format of nsc_quantize_histograms /
 * nsc_encode_batch_u16) into uint16 CDF rows in units of 1/65535. With S_i the integer prefix sums of
 * a row and T = S_{n_bins-1}:
 *   T = 65535 (every row the quantiser or the encoder writes): the stored row is S_i, exact.
 *   T = 0 (an empty scan's row): the stored row is all zero. The query reads a stored row whose last
 *         element is 0 as the uniform CDF (i + 1) / n_bins -- what dequantize yields for a zero row --
 *         computed in the kernel, not rounded into storage.
 *   any other T: round-half-even(65535 * S_i / T) in 64-bit integers, at most 0.5 / 65535 per CDF
 *         element from the CDF of the dequantised float row.
 * d_rows, d_cdf16: uint16[n_rows * n_bins]; n_bins <= 1024. Status codes and their order are those of
 * nsc_wasserstein_cdf.
 * nsc_wasserstein_query_u16 is nsc_wasserstein_query over d_db_cdf16 from nsc_wasserstein_cdf_u16
 * (queries stay float32 histograms): the same validation order and codes, the same workspace, top-K
 * selection and spatial filter. Its distances equal those of the float32 database of the dequantised
 * rows to float32 rounding (the sums run in counts and are scaled by 1/65535 once per row). */
int nsc_wasserstein_cdf_u16(const uint16_t* d_rows, int64_t n_rows, int n_bins, uint16_t* d_cdf16, void* stream);
int nsc_wasserstein_query_u16(const float* d_query_hists, int n_queries, const uint16_t* d_db_cdf16,
                              int64_t n_db, int n_bins, float epsilon, const double* d_db_xyz,
                              const double* d_query_xyz, double min_spatial_distance,
                              float* d_distances, int top_k, int64_t* d_top_idx, float* d_top_dist,
                              int32_t* d_top_count, void* d_workspace, size_t workspace_bytes, void* stream);

/* Any top_k, up to the whole database and beyond: the reference's TwoStageRetrieval._global_retrieval
 * asks for every keyframe (top_k = len(keyframes), two_stage_retrieval.py:181-185).
 * nsc_wasserstein_rank / nsc_wasserstein_rank_u16 take the arguments of nsc_wasserstein_query /
 * nsc_wasserstein_query_u16 with a 64-bit top_k, run the same distance pass (d_distances bit-identical)
 * and then rank each query's rows with a stable radix sort. Results, for every top_k:
 *   - the order is that of the key (distance bit pattern as uint32, row index), ascending: equal
 *     distances go to the lower row, +inf (excluded rows) and NaN last; the selection of
 *     nsc_wasserstein_query follows the same rule;
 *   - d_top_count[q] = min(top_k, finite distances of query q); entries at or past it are -1 / +inf,
 *     including those past n_db when top_k > n_db;
 *   - top_k = 0: distances only; n_queries = 0: nothing.
 * Validation, before any CUDA call: n_queries < 0, n_db < 0 or >= 2^32, top_k < 0 -> NSC_ERR_BAD_COUNT;
 * n_bins outside 1..1024 -> NSC_ERR_BAD_PARAMS; then the pointers of nsc_wasserstein_query ->
 * NSC_ERR_NULL_POINTER; then, when top_k > 0, a workspace that is NULL or smaller than
 * nsc_wasserstein_rank_workspace_bytes(n_queries, n_db) -> NSC_ERR_WORKSPACE.
 * The workspace (O(n_queries * n_db): keys and rows twice plus per-tile counts) needs no
 * initialisation and carries nothing between calls. nsc_wasserstein_rank_workspace_bytes returns 0
 * for negative arguments and n_db >= 2^32, SIZE_MAX where the size does not fit a size_t. All work is
 * queued on `stream`: no synchronisation, no allocation. */
size_t nsc_wasserstein_rank_workspace_bytes(int n_queries, int64_t n_db);
int nsc_wasserstein_rank(const float* d_query_hists, int n_queries, const float* d_db_cdfs,
                         int64_t n_db, int n_bins, float epsilon, const double* d_db_xyz,
                         const double* d_query_xyz, double min_spatial_distance,
                         float* d_distances, int64_t top_k, int64_t* d_top_idx, float* d_top_dist,
                         int32_t* d_top_count, void* d_workspace, size_t workspace_bytes, void* stream);
int nsc_wasserstein_rank_u16(const float* d_query_hists, int n_queries, const uint16_t* d_db_cdf16,
                             int64_t n_db, int n_bins, float epsilon, const double* d_db_xyz,
                             const double* d_query_xyz, double min_spatial_distance,
                             float* d_distances, int64_t top_k, int64_t* d_top_idx, float* d_top_dist,
                             int32_t* d_top_count, void* d_workspace, size_t workspace_bytes, void* stream);

/* ---- descriptor wire format (SURVEY.md 8(f), fourth "next" row) --------------------------- */
/* Replaces HistogramQuantizer.quantize / dequantize (reference src/encoding/quantization.py
 * :131-167, :169-192) for n_rows rows at once and any row length <= 4096 (the reference class is
 * instantiated for 50 bins; the 800-D descriptor quantises to 1600 bytes). Integers are
 * bit-identical to the reference's: the row sum follows NumPy's pairwise float32 order.
 *   quantize:   h / (sum h + eps) where sum h > eps, round-half-even(h * 65535), rounding error
 *               added to the first largest bin so that the row sums to 65535
 *   dequantize: q / (sum q + eps), or 1 / n_bins where sum q <= eps */
int nsc_quantize_histograms(const float* d_hist, int64_t n_rows, int n_bins, float epsilon,
                            uint16_t* d_quantized, void* stream);
int nsc_dequantize_histograms(const uint16_t* d_quantized, int64_t n_rows, int n_bins, float epsilon,
                              float* d_hist, void* stream);

/* ---- test hooks (not part of the product path) ----------------------------------------- */
/* Evaluates the kernel's per-point inline function (csrc/nsc_point.h) on the HOST for
 * n_points points: row / col (or -1) and keep flag per point. It exists so that the CPU-only
 * test suite can compare the pixel assignment with the oracle without a GPU; it computes no
 * image and no descriptor, and nothing in the encoder calls it. */
int nsc_test_host_classify(const float* h_points, int point_stride, int64_t n_points,
                           const nsc_params* p, int32_t* h_row, int32_t* h_col, uint8_t* h_keep);
/* 0 = polynomial row assignment, 1 = threshold search (wide fields of view); < 0 = status. */
int nsc_test_row_mode(const nsc_params* p);
/* Which kernel nsc_anywidth_points / nsc_anywidth_images run for images of `rows` rows under p,
 * with (want_descriptor != 0) or without a descriptor output: 1 = the fused shared-memory kernel,
 * 0 = the general kernel, < 0 = status (the entry points' parameter checks). Host only. */
int nsc_test_anywidth_path(const nsc_params* p, int rows, int want_descriptor);
/* The fused kernel's W-point complex forward FFT (its plan and radix passes, twiddles in float32)
 * run on the host: h_in and h_out hold W interleaved (re, im) float pairs. NSC_ERR_BAD_PARAMS for W
 * outside 2..4096 or with a prime factor above 13. */
int nsc_test_anywidth_fft(int W, const float* h_in, float* h_out);
/* The summation plan the quantiser kernels follow for rows of n_bins elements (host only, no CUDA
 * call): leaves [leaf_start[l], leaf_start[l] + leaf_len[l]) for l < *n_leaves, each summed with
 * NumPy's 8 strided accumulators, then *n_adds additions in single-assignment form -- addition t
 * writes slot *n_leaves + t = slot add_a[t] + slot add_b[t], a leaf's slot being its index -- and the
 * row sum is slot *result_slot. The arrays hold 64 entries. Lets the CPU-only suite check, for every
 * row length, that the plan reproduces NumPy's pairwise float32 sum bit for bit. */
int nsc_test_pairwise_sum_plan(int n_bins, int32_t* n_leaves, int32_t* n_adds, int32_t* result_slot,
                               uint16_t* leaf_start, uint16_t* leaf_len, uint8_t* add_a, uint8_t* add_b);

#ifdef __cplusplus
}
#endif
#endif /* NSC_B200_H */
