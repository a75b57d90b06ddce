// CUDA kernels (sm_100a) of the area-average hot path: the main loop of
// AreaAverageInterpolation::areaAverageInterpolation (Source.cpp:411-579).
//
// Formulation (NOT the reference's 16-segment-test classifier; see DESIGN.md §3):
//   * canvas pixel (x,y) -> footprint centre C in expanded-source coordinates (same FP64 expression as 212-219);
//     the footprint is the square |u|<=h, |v|<=h with u = (p-C).(c,-s), v = (p-C).(s,c), h = L/2.
//   * for every expanded source pixel (unit cell) in the footprint's bounding box, the overlap area is
//         A = 1/2 * sum over the 4 cell sides of  dist(V, side) * |side ∩ footprint|
//     (Green's theorem with the origin at the footprint vertex V nearest to the cell: the two footprint edges
//     through V contribute nothing, the two far edges cannot reach the cell because L > sqrt(2)).
//     |side ∩ footprint| comes from the footprint's chord on the grid line, computed once per grid line.
//     This single closed form reproduces all nine shapes of Source.cpp:1052-1401 in general position.
//   * the reference's shape 2 / shape 4 leg quirk (1055-1062, SURVEY.md §0.2) is then substituted: when the only
//     footprint edge crossing the cell is a left/right edge (direction (s,c)) that passes completely through it
//     and isolates exactly one cell corner at distance d, the triangle is 1/2 (1-d/c)(1-d/s).
//     Decisions are made in FP64 from FP64 geometry.
#include <cuda_runtime.h>

#include <cfloat>
#include <cstdint>
#include <cstdlib>

#include "aai_device.cuh"

using namespace aai_dev;

namespace {

// ------------------------------------------------------------------------------------------------------------
// Overlap kernel, FP64 arithmetic: one thread per canvas pixel, global (read-only path) source loads.
// ------------------------------------------------------------------------------------------------------------
template <typename TI, typename TO, int NC>
__global__ void __launch_bounds__(TILE_W *TILE_H)
    overlap_kernel_f64(const __grid_constant__ AaiKernelParams kp) {
    const int x = blockIdx.x * TILE_W + threadIdx.x;
    const int y = kp.row0 + blockIdx.y * TILE_H + threadIdx.y;
    if (x >= kp.dst_w || y >= kp.row1) return;
    double cx, cy;
    pixel_centre(kp, x, y, cx, cy);
    int ix0, ix1, jy0, jy1;
    cell_range(kp, cx, cy, ix0, ix1, jy0, jy1);
    double sumA, acc[NC];
    pixel_f64<TI, NC>(kp, cx, cy, ix0, ix1, jy0, jy1, sumA, acc);
    char *drow = (char *)kp.dst + (int64_t)(y - dst_row0(kp)) * kp.dst_pitch;
    const bool ok = DBL_EPSILON < fabs(sumA);  // Source.cpp:577
#pragma unroll
    for (int ch = 0; ch < NC; ++ch) store_dst<TO>(drow, x * NC + ch, ok ? acc[ch] / sumA : 0.0);
}

// ------------------------------------------------------------------------------------------------------------
// Separable kernel v1 (reduced angle exactly 0): footprint = axis-aligned square, overlap = wx(i) * wy(j).
// ------------------------------------------------------------------------------------------------------------
template <typename TI, typename TO, int NC>
__global__ void __launch_bounds__(TILE_W *TILE_H)
    separable_kernel_f64(const __grid_constant__ AaiKernelParams kp) {
    const int x = blockIdx.x * TILE_W + threadIdx.x;
    const int y = kp.row0 + blockIdx.y * TILE_H + threadIdx.y;
    if (x >= kp.dst_w || y >= kp.row1) return;
    double cx, cy;
    pixel_centre(kp, x, y, cx, cy);
    int wx0, wx1, wy0, wy1;
    search_window(kp, cx, cy, wx0, wx1, wy0, wy1);
    const double ext = kp.shape.half + 0.5 + 1e-9;
    const int ix0 = max(wx0, __double2int_ru(cx - ext)), ix1 = min(wx1, __double2int_rd(cx + ext));
    const int jy0 = max(wy0, __double2int_ru(cy - ext)), jy1 = min(wy1, __double2int_rd(cy + ext));
    const double xl = cx - kp.shape.half, xr = cx + kp.shape.half, yt = cy - kp.shape.half, yb = cy + kp.shape.half;
    double sumA = 0.0;
    double acc[NC];
#pragma unroll
    for (int ch = 0; ch < NC; ++ch) acc[ch] = 0.0;
    for (int j = jy0; j <= jy1; ++j) {
        const double wy = fmax(fmin(yb, (double)j + 0.5) - fmax(yt, (double)j - 0.5), 0.0);
        for (int i = ix0; i <= ix1; ++i) {
            const double wx = fmax(fmin(xr, (double)i + 0.5) - fmax(xl, (double)i - 0.5), 0.0);
            const double area = wx * wy;
            if (area != 0.0) {
                int sx, sy;
                mod_to_src(kp, i, j, sx, sy);
                const char *row = (const char *)kp.src + (int64_t)(sy - src_row0(kp)) * kp.src_pitch;
                sumA += area;
#pragma unroll
                for (int ch = 0; ch < NC; ++ch) acc[ch] += SrcLoad<TI>::get(row, sx * NC + ch) * area;
            }
        }
    }
    char *drow = (char *)kp.dst + (int64_t)(y - dst_row0(kp)) * kp.dst_pitch;
    const bool ok = DBL_EPSILON < fabs(sumA);
#pragma unroll
    for (int ch = 0; ch < NC; ++ch) store_dst<TO>(drow, x * NC + ch, ok ? acc[ch] / sumA : 0.0);
}

// ------------------------------------------------------------------------------------------------------------
// Fast mode (Source.cpp:866-907): unweighted mean of the expanded pixels whose CENTRE lies in the footprint.
// ------------------------------------------------------------------------------------------------------------
template <typename TI, typename TO, int NC>
__global__ void __launch_bounds__(TILE_W *TILE_H) fast_kernel(const __grid_constant__ AaiKernelParams kp) {
    const int x = blockIdx.x * TILE_W + threadIdx.x;
    const int y = kp.row0 + blockIdx.y * TILE_H + threadIdx.y;
    if (x >= kp.dst_w || y >= kp.row1) return;
    int count;
    double acc[NC];
    pixel_fast_f64<TI, NC>(kp, x, y, count, acc);
    char *drow = (char *)kp.dst + (int64_t)(y - dst_row0(kp)) * kp.dst_pitch;
#pragma unroll
    for (int ch = 0; ch < NC; ++ch) store_dst<TO>(drow, x * NC + ch, count > 0 ? acc[ch] / (double)count : 0.0);
}

// FP32 arithmetic for float / integer images.  The inside test is a discontinuous decision, so -- as in the FP32 overlap
// kernel -- the footprint centre is split into a lattice point and an FP32 fraction, the smallest margin of the decisive
// comparisons is tracked, and a pixel with a margin inside the guard band is redone in FP64 (pixel_fast_f64).
template <typename TI, typename TO, int NC>
__global__ void __launch_bounds__(TILE_W *TILE_H) fast_kernel_f32(const __grid_constant__ AaiKernelParams kp) {
    const int x = blockIdx.x * TILE_W + threadIdx.x;
    const int y = kp.row0 + blockIdx.y * TILE_H + threadIdx.y;
    if (x >= kp.dst_w || y >= kp.row1) return;
    const double cx = fma((double)x, kp.aff_xx, fma((double)y, kp.aff_xy, kp.aff_x0));
    const double cy = fma((double)x, kp.aff_yx, fma((double)y, kp.aff_yy, kp.aff_y0));
    const int irx = __double2int_rn(cx), iry = __double2int_rn(cy);
    const float fx = (float)(cx - (double)irx), fy = (float)(cy - (double)iry);
    // cells whose centre can lie in the footprint: |i - cx| <= h(c+s) (with an FP32 safety margin), inside the image
    const float ext = kp.shapef.hb + 4e-6f;
    const int ix0 = max(0, irx + __float2int_ru(fx - ext)), ix1 = min(kp.mod_w - 1, irx + __float2int_rd(fx + ext));
    const int jy0 = max(0, iry + __float2int_ru(fy - ext)), jy1 = min(kp.mod_h - 1, iry + __float2int_rd(fy + ext));
    const AaiShapeF &g = kp.shapef;
    const float tau = 4e-6f;
    float count = 0.0f, acc[NC], worst = 1.0f;
#pragma unroll
    for (int ch = 0; ch < NC; ++ch) acc[ch] = 0.0f;
    const bool ident = kp.scale == 1 && kp.quadrant == 0;
    constexpr int ESZ = (int)sizeof(TI) * NC;
    const float rx0 = (float)(ix0 - irx) - fx;
    for (int j = jy0; j <= jy1; ++j) {
        const float ry = (float)(j - iry) - fy;
        const float ur = -ry * g.sn, vr = ry * g.cs;
        const char *rowp = (const char *)kp.src + (int64_t)(j - src_row0(kp)) * kp.src_pitch + (int64_t)ix0 * ESZ;  // ident only
        float rx = rx0;
        for (int i = ix0; i <= ix1; ++i, rx += 1.0f, rowp += ESZ) {
            const float mu = g.half - fabsf(fmaf(rx, g.cs, ur));
            const float mv = g.half - fabsf(fmaf(rx, g.sn, vr));
            // margins of the comparisons that decide (the other coordinate is not clearly outside)
            if (mv > -tau) worst = fminf(worst, fabsf(mu));
            if (mu > -tau) worst = fminf(worst, fabsf(mv));
            if (mu >= 0.0f && mv >= 0.0f) {  // closed point-in-square (837-864)
                const char *p = rowp;
                if (!ident) {
                    int sx, sy;
                    mod_to_src(kp, i, j, sx, sy);
                    p = (const char *)kp.src + (int64_t)(sy - src_row0(kp)) * kp.src_pitch + (int64_t)sx * ESZ;
                }
                count += 1.0f;
#pragma unroll
                for (int ch = 0; ch < NC; ++ch) acc[ch] += LoadF<TI>::get(p + ch * (int)sizeof(TI));
            }
        }
    }
    char *drow = (char *)kp.dst + (int64_t)(y - dst_row0(kp)) * kp.dst_pitch;
    if (worst < tau) {  // a centre within the guard band of a footprint edge: FP64 decides
        int c64;
        double a64[NC];
        pixel_fast_f64<TI, NC>(kp, x, y, c64, a64);
#pragma unroll
        for (int ch = 0; ch < NC; ++ch) store_dst<TO>(drow, x * NC + ch, c64 > 0 ? a64[ch] / (double)c64 : 0.0);
    } else {
        const float inv = count > 0.0f ? 1.0f / count : 0.0f;
#pragma unroll
        for (int ch = 0; ch < NC; ++ch) store_dst<TO>(drow, x * NC + ch, (double)(acc[ch] * inv));
    }
}

// ------------------------------------------------------------------------------------------------------------
// Stand-alone expansion + quadrant pre-rotation (Source.cpp:157-172): modSrc[my][mx] = src[sy][sx].
// ------------------------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256) expand_kernel(const __grid_constant__ AaiKernelParams kp) {
    const int mx = blockIdx.x * 64 + (threadIdx.x & 63);
    const int my = kp.row0 + blockIdx.y * 4 + (threadIdx.x >> 6);  // row0: first expanded row of this launch
    if (mx >= kp.mod_w || my >= kp.mod_h) return;
    int sx, sy;
    mod_to_src(kp, mx, my, sx, sy);
    const T *srow = (const T *)((const char *)kp.src + (int64_t)(sy - kp.src_y0) * kp.src_pitch);
    T *drow = (T *)((char *)kp.dst + (int64_t)my * kp.dst_pitch);
    for (int ch = 0; ch < kp.channels; ++ch) drow[mx * kp.channels + ch] = srow[sx * kp.channels + ch];
}

// ------------------------------------------------------------------------------------------------------------
// Measurement helper (bench.py roofline denominator): sustained FP32 FMA rate of the device, 16 independent FFMA
// chains per thread, 2 flop per FFMA.  Not part of the resampling path.
// ------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) fp32_peak_kernel(float *out, int iters, float a, float b) {
    float v[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) v[k] = (float)(threadIdx.x + k);
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int k = 0; k < 16; ++k) v[k] = fmaf(v[k], a, b);
    }
    float sum = 0.0f;
#pragma unroll
    for (int k = 0; k < 16; ++k) sum += v[k];
    if (sum == 123.456f) out[0] = sum;  // never true: keeps the chains alive
}

enum KernelKind { K_OVERLAP, K_SEPARABLE, K_FAST, K_FAST_F32 };

template <KernelKind KIND, typename TI, typename TO, int NC>
cudaError_t launch_typed(const AaiKernelParams &kp, cudaStream_t stream) {
    if (kp.row1 <= kp.row0 || kp.dst_w <= 0) return cudaSuccess;
    const dim3 grid = canvas_grid(kp), block(TILE_W, TILE_H);
    if constexpr (KIND == K_OVERLAP) overlap_kernel_f64<TI, TO, NC><<<grid, block, 0, stream>>>(kp);
    if constexpr (KIND == K_SEPARABLE) separable_kernel_f64<TI, TO, NC><<<grid, block, 0, stream>>>(kp);
    if constexpr (KIND == K_FAST) fast_kernel<TI, TO, NC><<<grid, block, 0, stream>>>(kp);
    if constexpr (KIND == K_FAST_F32) fast_kernel_f32<TI, TO, NC><<<grid, block, 0, stream>>>(kp);
    return cudaGetLastError();
}

// the rolled kernels: every instantiated (source, canvas) pair of Srcs x Dsts, 1-4 channels
template <KernelKind KIND, typename Srcs, typename Dsts>
cudaError_t launch_any(const AaiKernelParams &kp, int src_dtype, int dst_dtype, cudaStream_t stream) {
    return with_pair<Srcs, Dsts>(src_dtype, dst_dtype, cudaErrorInvalidValue, [&](auto ti, auto to) {
        using TI = typename decltype(ti)::type;
        using TO = typename decltype(to)::type;
        return with_channels<1, 2, 3, 4>(kp.channels, cudaErrorInvalidValue, [&](auto nc) {
            return launch_typed<KIND, TI, TO, decltype(nc)::value>(kp, stream);
        });
    });
}

}  // namespace

int aai_launch_overlap(const AaiKernelParams &kp, int arith, int src_dtype, int dst_dtype, void *stream) {
    if (arith == AAI_ARITH_F32 && kp.f32_ok && (kp.channels == 1 || kp.channels == 3)) {
        switch (aai_f32_maxn(kp.ext32)) {
            case 4: return aai_launch_overlap_f32_n4(kp, src_dtype, dst_dtype, stream);
            case 5: return aai_launch_overlap_f32_n5(kp, src_dtype, dst_dtype, stream);
            case 6: return aai_launch_overlap_f32_n6(kp, src_dtype, dst_dtype, stream);
            case 8: return aai_launch_overlap_f32_n8(kp, src_dtype, dst_dtype, stream);
            default: break;
        }
    }
    // FP64 arithmetic: the unrolled kernel when the footprint fits its register arrays, else the rolled one
    // (its general-frame addressing divides by the scale with a multiply-high, exact below 2^32 / scale)
    const uint64_t max_e = (uint64_t)(kp.mod_w > kp.mod_h ? kp.mod_w : kp.mod_h);
    bool unrolled = kp.shape.sn > 0.0 && kp.shape.cs > 0.0 && max_e * (uint64_t)kp.scale < 0x100000000ULL;
#ifdef AAI_DEV_KNOBS  // developer builds only; the shipped library reads no environment
    if (getenv("AAI_F64_ROLLED")) unrolled = false;
#endif
    if (unrolled) {
        const int n = (int)floor(2.0 * kp.hb + 1.0 + 2e-9) + 1;  // cells per axis within hb + 1/2 + 1e-9 of the centre
        int e = (int)cudaErrorNotSupported;
        if (n <= 4) e = aai_launch_overlap_f64_n4(kp, src_dtype, dst_dtype, stream);
        else if (n <= 5) e = aai_launch_overlap_f64_n5(kp, src_dtype, dst_dtype, stream);
        else if (n <= 6) e = aai_launch_overlap_f64_n6(kp, src_dtype, dst_dtype, stream);
        else if (n <= 8) e = aai_launch_overlap_f64_n8(kp, src_dtype, dst_dtype, stream);
        if (e != (int)cudaErrorNotSupported) return e;
    }
    return (int)launch_any<K_OVERLAP, AnyElem, AnyElem>(kp, src_dtype, dst_dtype, (cudaStream_t)stream);
}
int aai_probe_fp32(int blocks, int iters, float *scratch, double *flop, void *stream) {
    fp32_peak_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(scratch, iters, 0.999f, 0.001f);
    *flop = (double)blocks * 256.0 * 16.0 * 2.0 * (double)iters;
    return (int)cudaGetLastError();
}
int aai_launch_separable(const AaiKernelParams &kp, int arith, int src_dtype, int dst_dtype, void *stream) {
    // TMA-staged two-pass kernel when its preconditions hold, else direct taps
    int e = aai_launch_separable_tma(kp, arith, src_dtype, dst_dtype, stream);
    if (e != (int)cudaErrorNotSupported) return e;
    if (arith == AAI_ARITH_F32) {  // quadrants 1-3, scale > 1, RGB: FP32 direct taps
        e = aai_launch_separable_direct_f32(kp, src_dtype, dst_dtype, stream);
        if (e != (int)cudaErrorNotSupported) return e;
    }
    return (int)launch_any<K_SEPARABLE, AnyElem, AnyElem>(kp, src_dtype, dst_dtype, (cudaStream_t)stream);
}
int aai_launch_expand(const AaiKernelParams &kp, int elem_bytes, void *stream) {
    if (kp.mod_w <= 0 || kp.mod_h <= 0) return (int)cudaSuccess;
    cudaStream_t st = (cudaStream_t)stream;
    AaiKernelParams k = kp;
    constexpr int kSlab = 65535 * 4;  // expanded rows per launch (grid.y limit)
    for (int r0 = 0; r0 < kp.mod_h; r0 += kSlab) {
        const int rows = kp.mod_h - r0 < kSlab ? kp.mod_h - r0 : kSlab;
        const dim3 grid((kp.mod_w + 63) / 64, (rows + 3) / 4);
        k.row0 = r0;
        switch (elem_bytes) {
            case 1: expand_kernel<uint8_t><<<grid, 256, 0, st>>>(k); break;
            case 2: expand_kernel<uint16_t><<<grid, 256, 0, st>>>(k); break;
            case 4: expand_kernel<float><<<grid, 256, 0, st>>>(k); break;
            case 8: expand_kernel<double><<<grid, 256, 0, st>>>(k); break;
            default: return (int)cudaErrorInvalidValue;
        }
        const cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) return (int)e;
    }
    return (int)cudaSuccess;
}

int aai_launch_fast(const AaiKernelParams &kp, int arith, int src_dtype, int dst_dtype, void *stream) {
    // FP32 arithmetic on request for float / integer sources (the mean of 8-byte doubles stays in FP64)
    const uint64_t max_e = (uint64_t)(kp.mod_w > kp.mod_h ? kp.mod_w : kp.mod_h);
    const bool f32 = arith == AAI_ARITH_F32 && src_dtype != AAI_F64 && dst_dtype != AAI_F64 && max_e < (1u << 30);
    // unrolled kernel: at most floor(2 hb + ~1e-5) + 1 lattice points per axis lie within hb of a footprint centre
    if (f32 && kp.staged == 2) {  // AAI_ARITH_F32_BINNED: float single-channel images in the source frame
        const int e = aai_launch_fast_bin(kp, src_dtype, dst_dtype, stream);
        if (e != (int)cudaErrorNotSupported) return e;
    }
    if (f32 && (kp.channels == 1 || kp.channels == 3) && max_e * (uint64_t)kp.scale < 0x100000000ULL) {
        const int nf = (int)floor(2.0 * ((double)kp.shapef.hb + 4e-6) + 1e-6) + 1;
        if (nf <= 3) return aai_launch_fast_f32_n4(kp, src_dtype, dst_dtype, stream);
        if (nf <= 4) return aai_launch_fast_f32_n5(kp, src_dtype, dst_dtype, stream);
        if (nf <= 5) return aai_launch_fast_f32_n6(kp, src_dtype, dst_dtype, stream);
        if (nf <= 7) return aai_launch_fast_f32_n8(kp, src_dtype, dst_dtype, stream);
    }
    if (f32) return (int)launch_any<K_FAST_F32, NarrowElem, NarrowElem>(kp, src_dtype, dst_dtype, (cudaStream_t)stream);
    return (int)launch_any<K_FAST, AnyElem, AnyElem>(kp, src_dtype, dst_dtype, (cudaStream_t)stream);
}
