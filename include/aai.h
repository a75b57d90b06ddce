/*
 * aai.h -- C ABI of the B200-native area-average interpolation hot path.
 *
 * This is the drop-in boundary for the ONE operator of Ishikawa-lab/Area_average_interpolation that this
 * repository accelerates:
 *
 *     pair<bool,string> AreaAverageInterpolation::areaAverageInterpolation(
 *         IMG src, IMG &dst, dP srcResolution, dP dstResolution,
 *         dP srcIsocenter, dP &dstIsocenter, double rotationAngle)            (Source.cpp:55-583)
 *
 * (and, as the "next" row f1, its unweighted sibling fastAreaAverageInterpolation, Source.cpp:584-911).
 * A C caller cannot receive a callee-sized std::vector, so the reference call is split into
 *   1. aai_plan_create()  -- everything the reference decides before its main loop
 *                            (validation 112-132, expansion/quadrant 139-176, canvas geometry 177-200),
 *                            i.e. the output size, the returned dstIsocenter and the error string;
 *   2. aai_run_host() / aai_run_device() -- the main loop 411-579 on the GPU(s).
 * The C++ host mirror with the reference's exact signature lives in
 * area_average_interpolation_b200/csrc/aai.hpp; the Python mirror in area_average_interpolation_b200/.
 *
 * Plain C types only; no STL, no torch types.  Every function is thread-safe for distinct plans/buffers.
 * There is NO CPU fallback: the run functions fail with AAI_ERR_CUDA when no sm_100a device is usable.
 */
#ifndef AAI_H_
#define AAI_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AAI_VERSION 100

/* Status codes.  1..4 are the reference's four validation failures, in the order it tests them
 * (Source.cpp:112, 118, 123, 128); aai_status_string() returns the reference's message verbatim. */
enum {
    AAI_OK = 0,
    AAI_ERR_RESOLUTION_XY = 1,  /* "Assumed X & Y resolution are same."                          (115) */
    AAI_ERR_RESOLUTION_NONPOS = 2, /* "0 or negative resolution is not acceptable."              (120) */
    AAI_ERR_NO_ROWS = 3,        /* "There is no data in src array."                              (125) */
    AAI_ERR_NO_COLUMNS = 4,     /* "There is no data in the second dimension of src array."      (130) */
    /* beyond the reference (it loops forever / reads out of bounds on these): */
    AAI_ERR_ANGLE = 5,          /* rotation angle is NaN or infinite (reference: endless loop at 141-142) */
    AAI_ERR_ARGUMENT = 6,       /* null pointer, bad dtype / channel count / band, image too large */
    AAI_ERR_CUDA = 7,           /* CUDA runtime / driver failure; see aai_last_error() */
    AAI_ERR_NO_DEVICE = 8       /* no usable CUDA device (there is no CPU fallback) */
};

/* Element types of pitched images.  AAI_U16 is unsigned 16-bit (film scans, CT slices).
 * Supported (source, canvas) pairs: F64 / F32 / U8 sources write F64, F32 or U8 canvases; a U16 source writes F64, F32
 * or U16 canvases, and a U16 canvas takes a U16 source only.  The run functions refuse the other four pairs
 * (F64 / F32 / U8 -> U16, U16 -> U8) with AAI_ERR_ARGUMENT before any CUDA call.
 * Integer canvases (the reference only knows doubles): the real-valued result is rounded half up and saturated,
 * to [0, 255] for U8 and to [0, 65535] for U16.  Integer sources take the same kernels as float sources, FP32 ones
 * with AAI_ARITH_F32 (16-bit values are exact in FP32). */
enum { AAI_F64 = 0, AAI_F32 = 1, AAI_U8 = 2, AAI_U16 = 3 };

/* Interpolation mode = the reference's `interpolationMode` user setting (Source.cpp:1534). */
enum {
    AAI_MODE_AREA_AVERAGE = 1, /* areaAverageInterpolation      (Source.cpp:55)  -- the north-star path */
    AAI_MODE_FAST = 2,         /* fastAreaAverageInterpolation  (Source.cpp:584) */
    /* beyond the reference (SURVEY 8f row f4): geometrically exact overlap areas, i.e. area averaging WITHOUT the
     * reference's shape-2/4 leg quirk (Source.cpp:1055-1062); opt-in, never the default, checked against its own
     * exact polygon-clipping oracle */
    AAI_MODE_AREA_AVERAGE_EXACT = 3
};

/* Arithmetic of the overlap kernel. */
enum {
    AAI_ARITH_F64 = 0, /* geometry, areas and accumulation in double (<= 1e-9 relative vs the reference) */
    AAI_ARITH_F32 = 1, /* geometry + shape decisions in double, area polynomials + accumulation in float */
    /* AAI_ARITH_F32 with the overlap kernel's source window staged through shared memory by a 2-D TMA tensor map (the
     * lay-out BASELINE.json's north star describes).  Same results; measured slower / faster per shape in
     * profiles/README.md -- the default FP32 kernel reads through L1.  Identity addressing only (scale 1, quadrant 0);
     * otherwise identical to AAI_ARITH_F32. */
    AAI_ARITH_F32_STAGED = 2,
    /* AAI_ARITH_F32 with fast mode computed from the SOURCE side where that applies (float single-channel images, scale 1,
     * quadrant 0, footprint box up to 5 pixels): every source pixel is read once, coalesced, and binned into the one
     * footprint it lies in (aai_kernels_bin.cu).  Same inside decisions as the default canvas-side gather kernel, a
     * different FP32 summation order; bitwise reproducible across band partitions.  Measured slower than the gather
     * kernel on B200 (profiles/README.md), so it is not the default.  Identical to AAI_ARITH_F32 in the other modes. */
    AAI_ARITH_F32_BINNED = 3,
    /* AAI_ARITH_F32 with fast mode computed by the staged gather kernel made persistent: CTAs walk over the canvas tiles
     * with two shared-memory window buffers, the TMA load of the next tile in flight while the current one is evaluated.
     * Same arithmetic as AAI_ARITH_F32_STAGED.  Identical to AAI_ARITH_F32 in the other modes. */
    AAI_ARITH_F32_RING = 4
};

/*
 * The geometry plan: the ~30 scalars the reference derives before its main loop.  POD, immutable after
 * aai_plan_create(), shared by every band / device so that N-GPU results are bitwise identical to 1 GPU.
 */
typedef struct aai_plan {
    int32_t status;     /* AAI_OK or 1..5 */
    uint32_t scale;     /* integer source expansion S (Source.cpp:139) */
    int32_t quadrant;   /* beforehandRotationMode k in 0..3 (140-146) */
    int32_t axis_aligned; /* 1 when the reduced angle is exactly axis-aligned (separable path) */
    int64_t src_w, src_h; /* original source size */
    int64_t mod_w, mod_h; /* expanded + quadrant-rotated source size (150-156) */
    int64_t dst_w, dst_h; /* canvas size (179-180) */
    double theta_deg;   /* reduced angle in [0,90) */
    double sin_t, cos_t; /* (147-148) */
    double iso_x, iso_y; /* isocentre in expanded coordinates (173-174) */
    double ratio;       /* expansionRatio (177) */
    double side;        /* dstSideLength L: footprint side in expanded pixels (178) */
    double dst_iso_x, dst_iso_y; /* the reference's OUT parameter dstIsocenter (185-186) */
    double off_ix, off_iy; /* dstIsocenterOffset (183-184) */
    double off_x, off_y;   /* canvas offset (187-200) */
    double reach;       /* L*sqrt(2)/2: half-diagonal used by the search window (426-429) */
} aai_plan;

/* A pitched image (or a horizontal band of one) in host or device memory.
 * Row y of the full image, y0 <= y < y0+rows, starts at (char*)data + (y - y0)*pitch_bytes and holds
 * width*channels interleaved elements of `dtype`.  Full images have y0 = 0, rows = height. */
typedef struct aai_image {
    void *data;
    int64_t pitch_bytes;
    int64_t width, height; /* of the FULL image */
    int64_t y0, rows;      /* rows present in `data` */
    int32_t dtype;         /* AAI_F64 / AAI_F32 / AAI_U8 / AAI_U16 */
    int32_t channels;      /* 1..4 interleaved channels sharing one geometry */
} aai_image;

/* ---- plan ---------------------------------------------------------------------------------------------- */

/* Replaces Source.cpp:112-200.  Arguments are the reference's (src.front().size(), src.size(),
 * srcResolution, dstResolution, srcIsocenter, rotationAngle).  Returns plan->status. */
int aai_plan_create(int64_t src_w, int64_t src_h, double src_res_x, double src_res_y, double dst_res_x,
                    double dst_res_y, double src_iso_x, double src_iso_y, double angle_deg, aai_plan *plan);

/* The reference's ret.second for status 0..4 ("" for AAI_OK); a description for the other codes. */
const char *aai_status_string(int status);

/* Message of the last AAI_ERR_CUDA / AAI_ERR_ARGUMENT on the calling thread. */
const char *aai_last_error(void);

/* ---- row-band partitioner (SURVEY 8e; host logic, no GPU needed) ---------------------------------------- */

/* Splits canvas rows [0, dst_h) into n_parts contiguous bands balanced by kernel cost: covered pixels plus a fraction
 * of the EMPTY ones (canvas corners of a rotated image are empty, but an empty pixel still costs its set-up and its zero
 * store).  bounds[0..n_parts] receives the band limits.  aai_partition_rows() uses the fraction of the FP32 overlap
 * kernel; aai_partition_rows_weighted() takes it from the caller, and aai_band_empty_weight() returns the fraction
 * measured on B200 for the kernel that (mode, arith) selects on this plan (the FP64 kernel's covered pixels cost more,
 * fast mode's less).  aai_run_host() partitions with the weight of its own (mode, arith). */
int aai_partition_rows(const aai_plan *plan, int n_parts, int64_t *bounds);
int aai_partition_rows_weighted(const aai_plan *plan, int n_parts, double empty_weight, int64_t *bounds);
double aai_band_empty_weight(const aai_plan *plan, int mode, int arith);

/* Source rows/columns (in ORIGINAL source coordinates, half-open) that canvas rows [row0,row1) can touch:
 * the band's halo. */
int aai_band_source_window(const aai_plan *plan, int64_t row0, int64_t row1, int64_t *src_x0, int64_t *src_x1,
                           int64_t *src_y0, int64_t *src_y1);

/* Number of canvas pixels in rows [row0,row1) whose search window meets the source (the rest are written as 0). */
int64_t aai_covered_pixels(const aai_plan *plan, int64_t row0, int64_t row1);

/* ---- pitched device images ----------------------------------------------------------------------------- */

int aai_device_count(void);

/* Allocates rows [y0, y0+rows) of a width x height x channels image on `device` (cudaMallocPitch layout,
 * pitch a multiple of 512 bytes so that every row is TMA- and 128-bit aligned). */
int aai_image_alloc(aai_image *img, int device, int64_t width, int64_t height, int64_t y0, int64_t rows,
                    int32_t dtype, int32_t channels);
int aai_image_free(aai_image *img, int device);
/* Copies the rows the device image holds from / to a host image that holds at least those rows. */
int aai_image_upload(const aai_image *device_img, const aai_image *host_img, int device, void *stream);
int aai_image_download(const aai_image *host_img, const aai_image *device_img, int device, void *stream);

/* Copies rows [y0,y1) of a device image into another device image of the same shape (same or PEER device: with
 * peer access enabled the copy goes over NVLink).  Both must hold those rows.  Asynchronous on `stream`. */
int aai_image_copy_rows(const aai_image *dst_device_img, const aai_image *src_device_img, int64_t y0, int64_t y1,
                        int device, void *stream);

/* Cross-process sharing of a device image for one-process-per-GPU launches (CUDA IPC): the owner exports the
 * allocation that `device_ptr` points to (it must be the base of an aai_image_alloc / cudaMalloc allocation), a peer
 * process opens it on its own device and can then read it with aai_image_copy_rows (NVLink peer copy, no NCCL). */
#define AAI_IPC_HANDLE_BYTES 64
int aai_ipc_export(const void *device_ptr, unsigned char handle[AAI_IPC_HANDLE_BYTES]);
int aai_ipc_open(const unsigned char handle[AAI_IPC_HANDLE_BYTES], int device, void **device_ptr);
int aai_ipc_close(void *device_ptr, int device);

/* Row f3 of SURVEY 8f: the reference's expansion + quadrant pre-rotation (Source.cpp:157-172) as a stand-alone device
 * op, for callers that want `modSrc` itself: dst_mod (plan->mod_w x plan->mod_h, same dtype / channels as src) receives
 * the source replicated `scale` times and rotated quadrant*90 degrees clockwise.  (The resampling kernels never
 * materialise it; they index the source through the same map.) */
int aai_expand_device(const aai_plan *plan, const aai_image *src, const aai_image *dst_mod, int device, void *stream);

/* Measurement helper (bench.py): sustained FP32 FMA rate of `device` in TFLOP/s, measured with a register-only FFMA
 * kernel (16 independent chains per thread).  The rotated-clip kernels are FP32-pipe bound by contract (SURVEY 8d) and
 * MEASURED_PEAKS.json holds no FP32 figure, so the roofline denominator is measured here.  Nothing in the reference
 * corresponds to it. */
int aai_measure_fp32_tflops(int device, double *tflops);

/* ---- the hot path --------------------------------------------------------------------------------------- */

/* Main loop of the reference (Source.cpp:411-579 / 866-907) for canvas rows [row0,row1) on one device.
 * `src` must hold the rows reported by aai_band_source_window() (or the whole image); `dst` must hold rows
 * [row0,row1) (or the whole canvas).  Both are DEVICE images on `device`.  Asynchronous on `stream`
 * (a cudaStream_t; NULL = the default stream); returns after enqueueing. */
int aai_run_device(const aai_plan *plan, int mode, int arith, const aai_image *src, const aai_image *dst,
                   int64_t row0, int64_t row1, int device, void *stream);

/* A batch of images that share one plan (BASELINE config 5: 256 slices; the slices of a CT volume under one rotation).
 * When the images are whole and equally strided in memory (srcs[k].data = srcs[0].data + k*stride, same for dsts;
 * same pitch, dtype and channel count) the whole batch is ONE kernel launch: the TMA-staged separable kernel takes the
 * stack as a rank-3 tensor map (one grid row per image), every other kernel of the path (FP32 / FP64 overlap kernels,
 * fast mode, direct-tap separable) runs with grid.z = image.  Otherwise the images are enqueued one after the other.
 * Results are bitwise identical to per-image aai_run_device calls.  Device images, asynchronous on `stream`. */
int aai_run_device_batch(const aai_plan *plan, int mode, int arith, const aai_image *srcs, const aai_image *dsts,
                         int n_images, int device, void *stream);

/* Adjoint (transpose) of what aai_run_device computes for `plan` and `mode`, FP64 weights: src_grads[k] receives
 * G = F^T canvas_grads[k].  Whole device images; F32 or F64, the same type and channel count on both sides.  Equally
 * strided stacks are one launch of each kernel (the rule of aai_run_device_batch), other lists run image by image.
 * Deterministic: bitwise the same for a stack and for per-image calls.  Asynchronous on `stream`.
 *
 * The forward is out[p] = sum_q A_pq v[src(q)] / S_p (S_p = sum_q A_pq, out = 0 where S_p <= DBL_EPSILON; fast mode:
 * A_pq = 1 for the cells whose centre lies in the closed footprint).  The adjoint is
 * G[s] = sum over the expanded cells q of s of sum_p (A_pq / S_p) g[p], with the weights of the FP64 forward; the
 * gradient of an AAI_ARITH_F32 forward is exact only to that arithmetic's tolerance.  F^T applied to a canvas of ones
 * is the coverage of each source pixel.  Scratch (8 bytes per canvas pixel) is allocated and freed in stream order. */
int aai_run_device_adjoint(const aai_plan *plan, int mode, const aai_image *canvas_grads, const aai_image *src_grads,
                           int n_images, int device, void *stream);

/* The reference call end to end with HOST buffers: upload (each device gets its band's halo), kernels on
 * per-device streams, download.  `devices` = NULL / n_devices = 0 means device 0.  No NCCL: bands are
 * independent.  Blocks until dst is complete. */
int aai_run_host(const aai_plan *plan, int mode, int arith, const aai_image *src, const aai_image *dst,
                 const int *devices, int n_devices);

/* One band of the host-buffer call on one device: uploads the band's source halo, runs the kernels, downloads
 * canvas rows [row0,row1) into `dst` (host images; each may hold just the band's halo / the band itself).  With `stream` = NULL an internal per-device stream
 * is used and the call blocks; otherwise the work is enqueued on `stream` (a cudaStream_t) and the call returns
 * without waiting unless `synchronize` is non-zero (use pinned host memory for truly asynchronous copies).
 * This is what one rank of a one-process-per-GPU launch calls. */
int aai_run_host_band(const aai_plan *plan, int mode, int arith, const aai_image *src, const aai_image *dst,
                      int64_t row0, int64_t row1, int device, void *stream, int synchronize);

/* A batch of HOST images that share one plan (BASELINE config 5 end to end; a CT volume): the slices are uploaded,
 * resampled and downloaded in a pipeline of three streams -- groups of slices go through a ring of device buffers, each
 * group is ONE batched kernel launch (aai_run_device_batch), and group g's upload / kernel / download overlap the
 * neighbouring groups' (PCIe is full duplex).  Whole images; srcs[k] / dsts[k] may be any host buffers (use pinned
 * memory for truly asynchronous copies).  `stream` / `synchronize` as in aai_run_host_band. */
int aai_run_host_batch(const aai_plan *plan, int mode, int arith, const aai_image *srcs, const aai_image *dsts,
                       int n_images, int device, void *stream, int synchronize);

/* ---- peer group: ONE large image over one process per GPU, end to end (SURVEY 8e, NVLink halo option) ------------
 *
 * With plain row bands every rank would upload its whole source halo from the host -- about half of the image per rank
 * for a rotated canvas, i.e. N/2 images over PCIe in total.  In a peer group every source row crosses PCIe exactly once:
 * rank r owns source rows [H r/N, H (r+1)/N), uploads them in chunks into its own full-size device image, and every
 * rank pulls the rows of its halo that it does not own out of the owners' device images with peer copies over NVLink
 * (CUDA IPC memory mappings) AS THE CHUNKS LAND.  There is no NCCL and no barrier; the ranks synchronise through two
 * monotonic counters per rank in a small POSIX shared-memory segment ("upload chunks landed", "steps whose pulls are
 * complete"), driven by the calling host thread: it polls its own upload events and publishes them, polls the owners'
 * counters and enqueues each pull the moment its chunk has landed.  Kernel and download of the band are chunk-pipelined
 * behind the pulls on the caller's stream, so a step costs about the slowest upload plus a short tail.
 *
 * Set-up (once per plan / image type): every rank calls aai_peer_create, exchanges the AAI_PEER_BLOB_BYTES blob of
 * aai_peer_export with all ranks through ANY out-of-band channel (MPI, a torch.distributed object gather, files), and
 * calls aai_peer_connect with the world_size blobs in rank order.  Then aai_peer_run per step.  Results are bitwise
 * identical to one GPU (all ranks share the plan). */
typedef struct aai_peer aai_peer;
#define AAI_PEER_BLOB_BYTES 2048
/* Tuning knob (process-wide, read by aai_peer_create; every rank must use the same value): into how many chunks an
 * owner cuts its upload, 1..8, default 4 (more chunks let the NVLink pulls start earlier).  Returns the value in force
 * (n outside 1..8 only queries). */
int aai_peer_upload_chunks(int n);
int aai_peer_create(const aai_plan *plan, int32_t dtype, int32_t channels, int rank, int world_size, int device,
                    aai_peer **out);
int aai_peer_export(aai_peer *peer, unsigned char blob[AAI_PEER_BLOB_BYTES]);
int aai_peer_connect(aai_peer *peer, const unsigned char *blobs_of_all_ranks);
/* Source rows [*y0, *y1) this rank uploads; canvas rows [*row0, *row1) it computes (aai_partition_rows). */
int aai_peer_owned_rows(const aai_peer *peer, int64_t *y0, int64_t *y1);
int aai_peer_band(const aai_peer *peer, int64_t *row0, int64_t *row1);
/* One step: `host_src` holds (at least) the owned source rows, `host_dst` receives the band's canvas rows (each may be
 * a band view: y0/rows).  The host buffers are read / written when the copies execute: `host_src` must be ready when the
 * call is made (a step's uploads overlap the previous step's downloads), `host_dst` is complete when `stream` is.  Enqueued on `stream` (NULL = an internal stream, blocking); returns without waiting unless
 * `synchronize`; it does return only after this rank's uploads have landed and its halo pulls have been enqueued and
 * completed (the host drives that exchange), while its kernels and downloads may still be in flight on `stream`.  All
 * ranks must call it the same number of times; waiting for a rank that never arrives fails after 60 s. */
int aai_peer_run(aai_peer *peer, int mode, int arith, const aai_image *host_src, const aai_image *host_dst,
                 void *stream, int synchronize);
/* The rank's full-size device source image (rows of the band's halo are valid after a step) -- for device-resident
 * follow-up work (aai_run_device). */
int aai_peer_device_source(const aai_peer *peer, aai_image *out);
/* Device-side phase times [ms] of this rank's LAST step, measured from the start of its upload: own upload complete, last
 * halo pull complete, last kernel complete, last download complete (waits for the step to finish). */
int aai_peer_last_timing(aai_peer *peer, float ms[4]);
/* Frees the group's device memory and IPC mappings.  Call it once every rank has completed its last step (any barrier
 * of the launcher): peers read this rank's device image. */
int aai_peer_destroy(aai_peer *peer);

/* Kernel-launch counter of this process (every overlap / separable / fast kernel launch increments it). */
int64_t aai_launch_count(void);

/* Device-side breakdown [ms] of the last aai_run_host() on this thread, from CUDA events on the per-device
 * streams (max over devices): host->device copies, kernels, device->host copies.  Large bands are pipelined
 * (chunked upload / kernel / download on three streams): the phases overlap, so the whole call is reported in
 * *h2d_ms and the other two are 0.  Returns AAI_OK or AAI_ERR_ARGUMENT if no run has completed. */
int aai_last_host_timing(float *h2d_ms, float *kernel_ms, float *d2h_ms);

#ifdef __cplusplus
}
#endif
#endif /* AAI_H_ */
