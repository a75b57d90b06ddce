// Internal declarations shared by the host plan, the C ABI glue and the CUDA kernels.
#ifndef AAI_INTERNAL_H_
#define AAI_INTERNAL_H_

#include <cuda_runtime.h>

#include <cstdint>
#include <vector>

#include "../../include/aai.h"
#include "aai_cell.cuh"

// canvas pixels per CTA of the one-thread-per-pixel kernels (see aai_device.cuh); rows go on grid.y, which CUDA limits
// to 65535 blocks, so the C ABI cuts taller row ranges into several launches
#ifndef AAI_TILE_W
#define AAI_TILE_W 16
#endif
#ifndef AAI_TILE_H
#define AAI_TILE_H 8
#endif
#define AAI_MAX_ROWS_PER_LAUNCH (65535LL * AAI_TILE_H)

// Everything a kernel needs, passed by value (__grid_constant__).  Built on the host in FP64 from the plan.
struct AaiKernelParams {
    // canvas-pixel centre expression of Source.cpp:212-219
    double side, off_ix, off_iy, iso_x, iso_y, off_x, off_y;
    // the same centre as an affine map of the canvas pixel (x, y): cx = aff_x0 + x aff_xx + y aff_xy, cy likewise
    double aff_x0, aff_xx, aff_xy, aff_y0, aff_yx, aff_yy;
    float ext32;      // hb + 1/2 + 2e-6: half extent of the cell range in the FP32 kernel
    AaiShape shape;   // cos/sin, h = L/2 and the derived footprint constants (aai_cell.cuh)
    AaiShapeF shapef; // the same in FP32 (+ guard band) for the FP32 kernel
    int32_t f32_ok;   // FP32 kernel admissible (angle not within ~3 degrees of an axis)
    int32_t quirk;    // 1: reproduce the reference's shape-2/4 leg quirk (default), 0: geometrically exact areas
    int32_t staged;   // FP32 kernels: 1 = source window staged through shared memory by TMA (A/B variant),
                      // 2 = fast mode binned from the source side where aai_kernels_bin.cu applies (A/B variant),
                      // 3 = fast mode by the persistent, double-buffered staged kernel (A/B variant)
    int32_t reverse_rows;  // host side only: the launcher of short FP32 overlap launches picks the bottom-up instantiation
    int32_t tip_window;    // host side only: aai_tip_window_ok for the plan's shape and aai_f32_maxn (FP32 overlap kernel)
    double reach;     // L*sqrt(2)/2 (search window, 426-429)
    double hb;        // h*(c+s): half extent of the footprint's axis-aligned bounding box
    int32_t mod_w, mod_h, dst_w, dst_h;
    int32_t scale, quadrant;
    // expanded + quadrant-rotated pixel (i,j) -> expanded pixel (ex,ey) = (axi*i + axj*j + ax0, ayi*i + ayj*j + ay0)
    // (inverse of Source.cpp:163-168), then source pixel = (ex/scale, ey/scale) via a multiply-high
    int32_t e_axi, e_axj, e_ax0, e_ayi, e_ayj, e_ay0;
    uint32_t div_magic;  // floor(2^32/scale)+1: exact for ex*scale < 2^32
    // source view (original frame): rows [src_y0, src_y0+src_rows) are present
    const void *src;
    int64_t src_pitch;
    int32_t src_w, src_h, src_y0, src_rows;
    int32_t channels;
    // destination band view: rows [dst_y0, dst_y0+dst_rows) are present; rows [row0,row1) are computed
    void *dst;
    int64_t dst_pitch;
    int32_t dst_y0, row0, row1;
    // batch of equally strided images sharing one plan (0/1 = single image): blockIdx.y of the separable TMA kernel,
    // blockIdx.z of every other kernel selects the image
    int32_t batch;
    int64_t src_batch_stride, dst_batch_stride;  // bytes between consecutive images
    int32_t src_batch_rows, dst_batch_rows;      // the same in rows of the pitch (grid.z kernels; strides are whole rows)
};

// Cells per axis of the FP32 overlap kernel's translation unit (4, 5, 6 or 8) for footprint boxes of half extent ext32:
// at most floor(2 ext32) + 1 cells per axis have non-zero overlap; 0 when no unit holds them
inline int aai_f32_maxn(float ext32) {
    const int n = (int)floor(2.0 * (double)ext32 + 1e-6) + 1;  // = floor(2 hb + 1 + ~4e-6) + 1
    return n <= 4 ? 4 : n <= 5 ? 5 : n <= 6 ? 6 : n <= 8 ? 8 : 0;
}

// Bytes per element of an AAI_* element type, 0 for an unknown type: the one table every buffer size is taken from.
inline size_t aai_elem_size(int dtype) {
    switch (dtype) {
        case AAI_F64: return 8;
        case AAI_F32: return 4;
        case AAI_U16: return 2;
        case AAI_U8: return 1;
        default: return 0;
    }
}
// Row pitch of the library's device images: rows start on 512-byte boundaries, which satisfies TMA's 16-byte global
// stride rule and 128-bit accesses.
inline int64_t aai_device_pitch(int64_t width, int32_t channels, int dtype) {
    return (width * channels * (int64_t)aai_elem_size(dtype) + 511) / 512 * 512;
}
inline const char *aai_dtype_name(int dtype) {
    switch (dtype) {
        case AAI_F64: return "float64";
        case AAI_F32: return "float32";
        case AAI_U16: return "uint16";
        case AAI_U8: return "uint8";
        default: return "unknown";
    }
}
// The (source, canvas) element-type pairs the kernels are compiled for (include/aai.h): a 16-bit canvas takes a 16-bit
// source only, a 16-bit source writes float or 16-bit canvases.  Keeps the number of instantiations bounded.
inline constexpr bool aai_dtype_pair_ok(int src_dtype, int dst_dtype) {
    if (dst_dtype == AAI_U16) return src_dtype == AAI_U16;
    if (src_dtype == AAI_U16) return dst_dtype != AAI_U8;
    return true;
}
// AAI_OK, or AAI_ERR_ARGUMENT with a message naming the refused pair (aai_last_error); no CUDA call
int aai_check_dtype_pair(const char *who, int src_dtype, int dst_dtype);

AaiKernelParams aai_make_kernel_params(const aai_plan &plan, const aai_image &src, const aai_image &dst,
                                       int64_t row0, int64_t row1);

// kernel launchers (aai_kernels.cu); return the cudaError_t of the launch as int
int aai_launch_overlap(const AaiKernelParams &kp, int arith, int src_dtype, int dst_dtype, void *stream);
int aai_launch_separable(const AaiKernelParams &kp, int arith, int src_dtype, int dst_dtype, void *stream);
int aai_launch_fast(const AaiKernelParams &kp, int arith, int src_dtype, int dst_dtype, void *stream);
int aai_launch_expand(const AaiKernelParams &kp, int elem_bytes, void *stream);
// measurement helper: launches the FP32 FMA probe, returns the flop it performs
int aai_probe_fp32(int blocks, int iters, float *scratch, double *flop, void *stream);
// aai_kernels_sep.cu: TMA-staged separable kernel; returns cudaErrorNotSupported when its fast path does not apply
int aai_launch_separable_tma(const AaiKernelParams &kp, int arith, int src_dtype, int dst_dtype, void *stream);
// aai_kernels_sep.cu: FP32 direct-tap kernel for axis-aligned cases outside the TMA kernel's preconditions
int aai_launch_separable_direct_f32(const AaiKernelParams &kp, int src_dtype, int dst_dtype, void *stream);
// aai_kernels_f32.cu, one translation unit per maximum cell count per axis
int aai_launch_overlap_f32_n4(const AaiKernelParams &kp, int src_dtype, int dst_dtype, void *stream);
int aai_launch_overlap_f32_n5(const AaiKernelParams &kp, int src_dtype, int dst_dtype, void *stream);
int aai_launch_overlap_f32_n6(const AaiKernelParams &kp, int src_dtype, int dst_dtype, void *stream);
int aai_launch_overlap_f32_n8(const AaiKernelParams &kp, int src_dtype, int dst_dtype, void *stream);
// fast mode, FP32 arithmetic, unrolled (same translation units): float / 8-bit images with 1 or 3 channels
int aai_launch_fast_f32_n4(const AaiKernelParams &kp, int src_dtype, int dst_dtype, void *stream);
int aai_launch_fast_f32_n5(const AaiKernelParams &kp, int src_dtype, int dst_dtype, void *stream);
int aai_launch_fast_f32_n6(const AaiKernelParams &kp, int src_dtype, int dst_dtype, void *stream);
int aai_launch_fast_f32_n8(const AaiKernelParams &kp, int src_dtype, int dst_dtype, void *stream);
// aai_kernels_bin.cu: fast mode by source-side binning; cudaErrorNotSupported when its preconditions do not hold
int aai_launch_fast_bin(const AaiKernelParams &kp, int src_dtype, int dst_dtype, void *stream);
// aai_kernels_f64.cu, likewise (unrolled FP64 kernel; cudaErrorNotSupported -> the rolled kernel in aai_kernels.cu)
int aai_launch_overlap_f64_n4(const AaiKernelParams &kp, int src_dtype, int dst_dtype, void *stream);
int aai_launch_overlap_f64_n5(const AaiKernelParams &kp, int src_dtype, int dst_dtype, void *stream);
int aai_launch_overlap_f64_n6(const AaiKernelParams &kp, int src_dtype, int dst_dtype, void *stream);
int aai_launch_overlap_f64_n8(const AaiKernelParams &kp, int src_dtype, int dst_dtype, void *stream);

// aai_kernels_adj.cu: adjoint of the resampling operator (aai_run_device_adjoint).  `kp` carries the plan's geometry
// (built with the source gradients as `src` and the canvas gradients as `dst`); the pointers below are what the kernels
// read and write.
struct AaiAdjointParams {
    AaiKernelParams kp;
    double *rcp;                 // [dst_h][dst_w]: 1/S_p of the forward, 0 where it writes 0
    double inv_side;             // 1/L (the gather's inverse centre map; no FP64 division in the kernel)
    const void *canvas;          // canvas gradients of image 0; image k at canvas + k * canvas_stride bytes
    int64_t canvas_pitch, canvas_stride;
    void *out;                   // source gradients, likewise
    int64_t out_pitch, out_stride;
    int32_t row0, row1;          // rows of this launch: canvas rows (normaliser) or source rows (gather)
};
// one launch each over rows [ap.row0, ap.row1) (at most AAI_MAX_ROWS_PER_LAUNCH); return the cudaError_t as int
int aai_launch_adjoint_norm(const AaiAdjointParams &ap, int mode, int axis_aligned, void *stream);
int aai_launch_adjoint_gather(const AaiAdjointParams &ap, int mode, int axis_aligned, int dtype, int n_images,
                              void *stream);

void aai_set_error(const char *fmt, ...);
// aai_launch_count() bookkeeping for launchers that start more than the one kernel the C ABI glue counts per call
void aai_count_extra_launches(int n);

// Enqueues the copy of `rows` rows of `row_bytes` bytes between two pitched buffers; nothing for rows <= 0.
cudaError_t aai_copy_pitched(void *dst, int64_t dst_pitch, const void *src, int64_t src_pitch, size_t row_bytes,
                             int64_t rows, cudaMemcpyKind kind, cudaStream_t stream);
// Creates timing-free events until `events` holds at least n (grow-only per-run event pools).
cudaError_t aai_grow_events(std::vector<cudaEvent_t> &events, size_t n);

#endif  // AAI_INTERNAL_H_
