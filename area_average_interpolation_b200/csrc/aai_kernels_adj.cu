// Adjoint (transpose) of the resampling operator, FP64 weights (aai_run_device_adjoint, include/aai.h).
//
// The forward is out[p] = sum_q A_pq v[src(q)] / S_p over the expanded, quadrant-rotated cells q, with S_p = sum_q A_pq
// and out = 0 where S_p <= DBL_EPSILON (fast mode: A_pq = 1 when the centre of q lies in the closed footprint, S_p the
// count, out = 0 where it is 0).  Its transpose is
//     G[s] = sum over the scale^2 cells q of source pixel s of  sum_p (A_pq / S_p) g[p].
// Two kernels:
//   * adjoint_norm_kernel: 1/S_p per canvas pixel (0 where the forward writes 0), once per call -- it depends on the
//     plan only, so every image of a batch shares it;
//   * adjoint_gather_kernel: one thread per ORIGINAL source pixel.  For each of its expanded cells it inverts the affine
//     footprint-centre map, which bounds the canvas pixels whose footprint can meet the cell (at most 2 per axis: the
//     cell's extent across a footprint row is c + s <= sqrt(2) < L), evaluates the forward's weight for each and
//     accumulates sum w r_p g[p] in FP64.  Every output is written by one thread in an order fixed by the geometry:
//     no atomics, bitwise reproducible across calls and batches.
// The weights are the FP64 forward's: aai_pair_area (rotated; reference operand order of the centre), the wx * wy of
// separable_kernel_f64 (axis-aligned), the closed point-in-square test of pixel_fast_f64 (fast mode), each over the
// forward's own cell range, so that the pairs evaluated are exactly the forward's.
#include <cuda_runtime.h>

#include <cfloat>
#include <cstdint>

#include "aai_device.cuh"

using namespace aai_dev;

namespace {

enum AdjKind { ADJ_ROTATED = 0, ADJ_SEPARABLE = 1, ADJ_FAST = 2 };

// Weight of the pair (canvas pixel (x, y), expanded cell (i, j)) as the FP64 forward evaluates it; 0 for a pair the
// forward does not visit.  Rotated plans and fast mode (axis-aligned area modes: separable_axis_weight).
template <int KIND>
__device__ __forceinline__ double pair_weight(const AaiKernelParams &kp, int x, int y, int i, int j) {
    double cx, cy;
    pixel_centre(kp, x, y, cx, cy);
    if (KIND == ADJ_ROTATED) {
        int ix0, ix1, jy0, jy1;
        cell_range(kp, cx, cy, ix0, ix1, jy0, jy1);
        if (i < ix0 || i > ix1 || j < jy0 || j > jy1) return 0.0;
        return aai_pair_area(kp.shape, cx, cy, i, j, kp.quirk != 0);
    } else {
        int wx0, wx1, wy0, wy1;
        search_window(kp, cx, cy, wx0, wx1, wy0, wy1);
        const double ext = kp.hb + 1e-6;
        if (i < max(wx0, __double2int_ru(cx - ext)) || i > min(wx1, __double2int_rd(cx + ext)) ||
            j < max(wy0, __double2int_ru(cy - ext)) || j > min(wy1, __double2int_rd(cy + ext)))
            return 0.0;
        const double ry = (double)j - cy;
        const double rx = (double)i - cx;
        const double u0 = rx * kp.shape.cs - ry * kp.shape.sn;
        const double v0 = rx * kp.shape.sn + ry * kp.shape.cs;
        return (fabs(u0) <= kp.shape.half && fabs(v0) <= kp.shape.half) ? 1.0 : 0.0;
    }
}

// One axis of separable_kernel_f64's weight: footprint centre coordinate c (pixel_centre; on an axis-aligned plan cx
// depends on x only and cy on y only), cell index i, image extent n -- the same window, range and overlap expressions,
// so that wx * wy is bitwise the forward's area
__device__ __forceinline__ double separable_axis_weight(const AaiKernelParams &kp, double c, int i, int n) {
    const int w0 = max(0, __double2int_rd(__dsub_rn(__dsub_rn(c, kp.reach), 1.0)));
    const int w1 = min(__double2int_ru(__dadd_rn(__dadd_rn(c, kp.reach), 1.0)), n - 1);
    const double ext = kp.shape.half + 0.5 + 1e-9;
    if (i < max(w0, __double2int_ru(c - ext)) || i > min(w1, __double2int_rd(c + ext))) return 0.0;
    return fmax(fmin(c + kp.shape.half, (double)i + 0.5) - fmax(c - kp.shape.half, (double)i - 0.5), 0.0);
}

// S_p of the forward over the same cells, summed in the forward's row-major order
template <int KIND>
__device__ __forceinline__ double weight_sum(const AaiKernelParams &kp, int x, int y) {
    double cx, cy;
    pixel_centre(kp, x, y, cx, cy);
    int ix0, ix1, jy0, jy1;
    if (KIND == ADJ_ROTATED) {
        cell_range(kp, cx, cy, ix0, ix1, jy0, jy1);
    } else {
        int wx0, wx1, wy0, wy1;
        search_window(kp, cx, cy, wx0, wx1, wy0, wy1);
        const double ext = KIND == ADJ_SEPARABLE ? kp.shape.half + 0.5 + 1e-9 : kp.hb + 1e-6;
        ix0 = max(wx0, __double2int_ru(cx - ext));
        ix1 = min(wx1, __double2int_rd(cx + ext));
        jy0 = max(wy0, __double2int_ru(cy - ext));
        jy1 = min(wy1, __double2int_rd(cy + ext));
    }
    double s = 0.0;
    for (int j = jy0; j <= jy1; ++j) {
        const double ry = (double)j - cy;
        for (int i = ix0; i <= ix1; ++i) {
            if (KIND == ADJ_ROTATED) {
                s += aai_pair_area(kp.shape, cx, cy, i, j, kp.quirk != 0);
            } else if (KIND == ADJ_SEPARABLE) {
                const double xl = cx - kp.shape.half, xr = cx + kp.shape.half;
                const double yt = cy - kp.shape.half, yb = cy + kp.shape.half;
                const double wy = fmax(fmin(yb, (double)j + 0.5) - fmax(yt, (double)j - 0.5), 0.0);
                const double wx = fmax(fmin(xr, (double)i + 0.5) - fmax(xl, (double)i - 0.5), 0.0);
                s += wx * wy;
            } else {
                const double rx = (double)i - cx;
                const double u0 = rx * kp.shape.cs - ry * kp.shape.sn;
                const double v0 = rx * kp.shape.sn + ry * kp.shape.cs;
                if (fabs(u0) <= kp.shape.half && fabs(v0) <= kp.shape.half) s += 1.0;
            }
        }
    }
    return s;
}

// 1/S_p per canvas pixel of rows [row0, row1); 0 where the forward writes 0 (Source.cpp:577; fast mode: count 0)
template <int KIND>
__global__ void __launch_bounds__(TILE_W *TILE_H) adjoint_norm_kernel(const __grid_constant__ AaiAdjointParams ap) {
    const AaiKernelParams &kp = ap.kp;
    const int x = blockIdx.x * TILE_W + threadIdx.x;
    const int y = ap.row0 + blockIdx.y * TILE_H + threadIdx.y;
    if (x >= kp.dst_w || y >= ap.row1) return;
    const double s = weight_sum<KIND>(kp, x, y);
    const bool ok = KIND == ADJ_FAST ? s > 0.0 : DBL_EPSILON < fabs(s);
    ap.rcp[(int64_t)y * kp.dst_w + x] = ok ? 1.0 / s : 0.0;
}

// One thread per original source pixel of rows [row0, row1); blockIdx.z = image of an equally strided stack.
// (ptxas holds the rotated and fast-mode instantiations to 64-72 registers with small spills; a minimum of 4 CTAs per SM
// removes the spills at 76-117 registers but measured slower on B200 -- config 4: 15.4 against 14.1 ms, fast mode 3.49
// against 2.96 ms -- the lost occupancy costs more than the spills, profiles/README.md)
template <int KIND, typename T, int NC>
__global__ void __launch_bounds__(TILE_W *TILE_H) adjoint_gather_kernel(const __grid_constant__ AaiAdjointParams ap) {
    const AaiKernelParams &kp = ap.kp;
    const int sx = blockIdx.x * TILE_W + threadIdx.x;
    const int sy = ap.row0 + blockIdx.y * TILE_H + threadIdx.y;
    if (sx >= kp.src_w || sy >= ap.row1) return;
    const char *g = (const char *)ap.canvas + (int64_t)blockIdx.z * ap.canvas_stride;
    // inverse of the affine centre map cx = aff_x0 + x L c + y L s, cy = aff_y0 - x L s + y L c
    const double c = kp.shape.cs, s = kp.shape.sn, inv_l = ap.inv_side;
    // a cell meets footprint x only if its centre is within 1/2 + (c+s)/(2L) of x across the footprint rows (fast mode:
    // within 1/2); the margin absorbs the rounding of this inverse map -- the weight decides, not the range
    const double reach = (KIND == ADJ_FAST ? 0.5 : 0.5 + kp.shape.m * inv_l) + 1e-6;
    double acc[NC];
#pragma unroll
    for (int ch = 0; ch < NC; ++ch) acc[ch] = 0.0;
    const int sc = kp.scale;
    for (int ey = sy * sc; ey < (sy + 1) * sc; ++ey) {
        for (int ex = sx * sc; ex < (sx + 1) * sc; ++ex) {
            // expanded pixel -> expanded + quadrant-rotated cell (Source.cpp:163-168; mod_to_src is its inverse)
            int i, j;
            switch (kp.quadrant) {
                case 0: i = ex; j = ey; break;
                case 1: i = kp.mod_w - 1 - ey; j = ex; break;
                case 2: i = kp.mod_w - 1 - ex; j = kp.mod_h - 1 - ey; break;
                default: i = ey; j = kp.mod_h - 1 - ex; break;
            }
            const double dx = (double)i - kp.aff_x0, dy = (double)j - kp.aff_y0;
            const double px = (dx * c - dy * s) * inv_l, py = (dx * s + dy * c) * inv_l;
            int x0 = max(0, (int)ceil(px - reach)), x1 = min(kp.dst_w - 1, (int)floor(px + reach));
            int y0 = max(0, (int)ceil(py - reach)), y1 = min(kp.dst_h - 1, (int)floor(py + reach));
            // axis-aligned: the weight factorises, each axis is evaluated once per candidate (the candidate range spans
            // 1 + 1/L + 2e-6 < 2 canvas pixels per axis: at most 2 candidates)
            double wx0 = 0.0, wx1 = 0.0, wy0 = 0.0, wy1 = 0.0;
            if (KIND == ADJ_SEPARABLE) {
                x1 = min(x1, x0 + 1);
                y1 = min(y1, y0 + 1);
                double cx0, cy0, cx1, cy1;
                pixel_centre(kp, x0, y0, cx0, cy0);
                pixel_centre(kp, x0 + 1, y0 + 1, cx1, cy1);
                wx0 = separable_axis_weight(kp, cx0, i, kp.mod_w);
                wy0 = separable_axis_weight(kp, cy0, j, kp.mod_h);
                wx1 = x1 > x0 ? separable_axis_weight(kp, cx1, i, kp.mod_w) : 0.0;
                wy1 = y1 > y0 ? separable_axis_weight(kp, cy1, j, kp.mod_h) : 0.0;
            }
            for (int y = y0; y <= y1; ++y) {
                const char *grow = g + (int64_t)y * ap.canvas_pitch;
                for (int x = x0; x <= x1; ++x) {
                    double w;
                    if constexpr (KIND == ADJ_SEPARABLE)
                        w = (x == x0 ? wx0 : wx1) * (y == y0 ? wy0 : wy1);
                    else
                        w = pair_weight<KIND>(kp, x, y, i, j);
                    if (w == 0.0) continue;
                    const double wr = w * __ldg(ap.rcp + (int64_t)y * kp.dst_w + x);
#pragma unroll
                    for (int ch = 0; ch < NC; ++ch) acc[ch] += wr * SrcLoad<T>::get(grow, x * NC + ch);
                }
            }
        }
    }
    char *orow = (char *)ap.out + (int64_t)blockIdx.z * ap.out_stride + (int64_t)sy * ap.out_pitch;
#pragma unroll
    for (int ch = 0; ch < NC; ++ch) store_dst<T>(orow, sx * NC + ch, acc[ch]);
}

template <int KIND, typename T>
cudaError_t gather_channels(const AaiAdjointParams &ap, dim3 grid, cudaStream_t st) {
    const dim3 block(TILE_W, TILE_H);
    switch (ap.kp.channels) {
        case 1: adjoint_gather_kernel<KIND, T, 1><<<grid, block, 0, st>>>(ap); break;
        case 2: adjoint_gather_kernel<KIND, T, 2><<<grid, block, 0, st>>>(ap); break;
        case 3: adjoint_gather_kernel<KIND, T, 3><<<grid, block, 0, st>>>(ap); break;
        case 4: adjoint_gather_kernel<KIND, T, 4><<<grid, block, 0, st>>>(ap); break;
        default: return cudaErrorInvalidValue;
    }
    return cudaGetLastError();
}

template <int KIND>
cudaError_t gather_typed(const AaiAdjointParams &ap, int dtype, dim3 grid, cudaStream_t st) {
    switch (dtype) {
        case AAI_F64: return gather_channels<KIND, double>(ap, grid, st);
        case AAI_F32: return gather_channels<KIND, float>(ap, grid, st);
        default: return cudaErrorInvalidValue;
    }
}

int adj_kind(int mode, int axis_aligned) {
    return mode == AAI_MODE_FAST ? ADJ_FAST : axis_aligned ? ADJ_SEPARABLE : ADJ_ROTATED;
}

}  // namespace

int aai_launch_adjoint_norm(const AaiAdjointParams &ap, int mode, int axis_aligned, void *stream) {
    const int rows = ap.row1 - ap.row0;
    if (rows <= 0 || ap.kp.dst_w <= 0) return (int)cudaSuccess;
    const dim3 grid((ap.kp.dst_w + TILE_W - 1) / TILE_W, (rows + TILE_H - 1) / TILE_H), block(TILE_W, TILE_H);
    cudaStream_t st = (cudaStream_t)stream;
    switch (adj_kind(mode, axis_aligned)) {
        case ADJ_ROTATED: adjoint_norm_kernel<ADJ_ROTATED><<<grid, block, 0, st>>>(ap); break;
        case ADJ_SEPARABLE: adjoint_norm_kernel<ADJ_SEPARABLE><<<grid, block, 0, st>>>(ap); break;
        default: adjoint_norm_kernel<ADJ_FAST><<<grid, block, 0, st>>>(ap); break;
    }
    return (int)cudaGetLastError();
}

int aai_launch_adjoint_gather(const AaiAdjointParams &ap, int mode, int axis_aligned, int dtype, int n_images,
                              void *stream) {
    const int rows = ap.row1 - ap.row0;
    if (rows <= 0 || ap.kp.src_w <= 0 || n_images <= 0) return (int)cudaSuccess;
    const dim3 grid((ap.kp.src_w + TILE_W - 1) / TILE_W, (rows + TILE_H - 1) / TILE_H, n_images);
    cudaStream_t st = (cudaStream_t)stream;
    switch (adj_kind(mode, axis_aligned)) {
        case ADJ_ROTATED: return (int)gather_typed<ADJ_ROTATED>(ap, dtype, grid, st);
        case ADJ_SEPARABLE: return (int)gather_typed<ADJ_SEPARABLE>(ap, dtype, grid, st);
        default: return (int)gather_typed<ADJ_FAST>(ap, dtype, grid, st);
    }
}
