// Device helpers shared by the kernel translation units (aai_kernels.cu, aai_kernels_f32.cu, ...).
#ifndef AAI_DEVICE_CUH_
#define AAI_DEVICE_CUH_

#include <cuda.h>
#include <cuda_runtime.h>

#include <cfloat>
#include <cstdint>
#include <type_traits>

#include "aai_cell.cuh"
#include "aai_internal.h"

namespace aai_dev {

// canvas pixels per CTA (one thread each); a warp covers 32/TILE_W rows.  16x8 (128 threads, 6-7 CTAs/SM for the FP32
// kernel) measured 3.7 % faster than 16x16 on config 4: same warps per SM, finer-grained CTA turnover; 32x4 and 8x16
// re-measured on the final kernel: 1.478 / 1.463 ms against 1.466 ms (profiles/r1_v17_ab_occupancy_tiles.txt).
constexpr int TILE_W = AAI_TILE_W;
constexpr int TILE_H = AAI_TILE_H;

// Element types: the AAI_* code of a C++ element type and the element type of its TMA tensor maps (the separable TMA
// kernel, the STAGED / RING overlap and fast-mode kernels).
template <typename T>
struct Elem;
template <>
struct Elem<double> {
    static constexpr int dtype = AAI_F64;
    static constexpr CUtensorMapDataType tmap = CU_TENSOR_MAP_DATA_TYPE_FLOAT64;
};
template <>
struct Elem<float> {
    static constexpr int dtype = AAI_F32;
    static constexpr CUtensorMapDataType tmap = CU_TENSOR_MAP_DATA_TYPE_FLOAT32;
};
template <>
struct Elem<uint16_t> {
    static constexpr int dtype = AAI_U16;
    static constexpr CUtensorMapDataType tmap = CU_TENSOR_MAP_DATA_TYPE_UINT16;
};
template <>
struct Elem<uint8_t> {
    static constexpr int dtype = AAI_U8;
    static constexpr CUtensorMapDataType tmap = CU_TENSOR_MAP_DATA_TYPE_UINT8;
};
// (source, canvas) pairs that are instantiated: the dispatchers skip the others at compile time (the C ABI refuses them)
template <typename TI, typename TO>
constexpr bool pair_ok() {
    return aai_dtype_pair_ok(Elem<TI>::dtype, Elem<TO>::dtype);
}

// Host-side dispatch from run-time AAI_* codes and channel counts to template arguments.  Each kernel family names the
// element types and channel counts it is compiled for; nothing outside those lists is instantiated.
template <typename T>
struct Tag {
    using type = T;
};
template <typename... Ts>
struct Types {};
using AnyElem = Types<double, float, uint8_t, uint16_t>;
using NarrowElem = Types<float, uint8_t, uint16_t>;  // FP32-only kernels: no double side

// f(Tag<T>{}) for the T among Ts whose Elem<T>::dtype is `dtype`; `otherwise` when there is none
template <typename... Ts, typename F>
cudaError_t with_elem(Types<Ts...>, int dtype, cudaError_t otherwise, F &&f) {
    cudaError_t e = otherwise;
    ((dtype == Elem<Ts>::dtype && (e = f(Tag<Ts>{}), true)) || ...);
    return e;
}
// f(Tag<TI>{}, Tag<TO>{}) for an instantiated pair (pair_ok) of Srcs x Dsts; `otherwise` for any other pair
// (nested generic lambdas: decltype of a captured parameter is a reference, so the type is taken in the outer one)
template <typename Srcs, typename Dsts, typename F>
cudaError_t with_pair(int src_dtype, int dst_dtype, cudaError_t otherwise, F &&f) {
    return with_elem(Srcs{}, src_dtype, otherwise, [&](auto ti) {
        using TI = typename decltype(ti)::type;
        return with_elem(Dsts{}, dst_dtype, otherwise, [&](auto to) {
            using TO = typename decltype(to)::type;
            if constexpr (pair_ok<TI, TO>())
                return f(Tag<TI>{}, Tag<TO>{});
            else
                return otherwise;
        });
    });
}
// f(std::integral_constant<int, NC>{}) for nc among NCs; `otherwise` when it is not listed
template <int... NCs, typename F>
cudaError_t with_channels(int nc, cudaError_t otherwise, F &&f) {
    cudaError_t e = otherwise;
    ((nc == NCs && (e = f(std::integral_constant<int, NCs>{}), true)) || ...);
    return e;
}

// grid of the one-thread-per-canvas-pixel kernels over rows [row0, row1): TILE_W x TILE_H pixels per CTA, one z slice
// per image of a batch
inline dim3 canvas_grid(const AaiKernelParams &kp) {
    const int rows = kp.row1 - kp.row0;
    return dim3((kp.dst_w + TILE_W - 1) / TILE_W, (rows + TILE_H - 1) / TILE_H, kp.batch > 1 ? kp.batch : 1);
}

template <typename T>
struct SrcLoad;
template <>
struct SrcLoad<double> {
    static __device__ __forceinline__ double get(const void *row, int idx) { return __ldg((const double *)row + idx); }
};
template <>
struct SrcLoad<float> {
    static __device__ __forceinline__ double get(const void *row, int idx) {
        return (double)__ldg((const float *)row + idx);
    }
};
template <>
struct SrcLoad<uint8_t> {
    static __device__ __forceinline__ double get(const void *row, int idx) {
        return (double)__ldg((const uint8_t *)row + idx);
    }
};
template <>
struct SrcLoad<uint16_t> {
    static __device__ __forceinline__ double get(const void *row, int idx) {
        return (double)__ldg((const uint16_t *)row + idx);
    }
};

// 16-bit value -> float without the conversion unit: the value placed in the mantissa of 2^23, minus 2^23 (exact below
// 2^23; one LOP3 + one FADD instead of an I2F, which issues at a quarter of the FP32 rate)
#ifndef AAI_U16_CVT_MAGIC
#define AAI_U16_CVT_MAGIC 1  // 0: I2F (A/B in profiles/)
#endif
__device__ __forceinline__ float u16_to_float(uint32_t v) {
#if AAI_U16_CVT_MAGIC
    return __int_as_float(0x4B000000u | v) - 8388608.0f;
#else
    return (float)v;
#endif
}
template <typename TA, typename T>
__device__ __forceinline__ TA to_arith(T v) {
    return (TA)v;
}
template <>
__device__ __forceinline__ float to_arith<float, uint16_t>(uint16_t v) {
    return u16_to_float(v);
}

// FP32 kernels: one source element at a byte address, as float (exact for 8- and 16-bit values)
template <typename T>
struct LoadF;
template <>
struct LoadF<double> {
    static __device__ __forceinline__ float get(const char *p) { return (float)__ldg((const double *)p); }
};
template <>
struct LoadF<float> {
    static __device__ __forceinline__ float get(const char *p) { return __ldg((const float *)p); }
};
template <>
struct LoadF<uint8_t> {
    static __device__ __forceinline__ float get(const char *p) { return (float)__ldg((const uint8_t *)p); }
};
template <>
struct LoadF<uint16_t> {
    static __device__ __forceinline__ float get(const char *p) { return u16_to_float(__ldg((const uint16_t *)p)); }
};

template <typename T>
__device__ __forceinline__ void store_dst(void *row, int idx, double v);
template <>
__device__ __forceinline__ void store_dst<double>(void *row, int idx, double v) {
    ((double *)row)[idx] = v;
}
template <>
__device__ __forceinline__ void store_dst<float>(void *row, int idx, double v) {
    ((float *)row)[idx] = (float)v;
}
template <>
__device__ __forceinline__ void store_dst<uint8_t>(void *row, int idx, double v) {
    // the reference defines no 8-bit store; documented rule: round half up, saturate to [0,255]
    double r = floor(v + 0.5);
    r = fmin(fmax(r, 0.0), 255.0);
    ((uint8_t *)row)[idx] = (uint8_t)(int)r;
}
template <>
__device__ __forceinline__ void store_dst<uint16_t>(void *row, int idx, double v) {
    // the 8-bit rule with the 16-bit bound: round half up, saturate to [0,65535]
    double r = floor(v + 0.5);
    r = fmin(fmax(r, 0.0), 65535.0);
    ((uint16_t *)row)[idx] = (uint16_t)(int)r;
}

// The same stores from an FP32 result (FP32 kernels).  Integer canvases: v + 0.5f is exact below 2^23 and larger values
// saturate, so the result is the one store_dst gives for (double)v.
template <typename T>
__device__ __forceinline__ void store_f(void *row, int idx, float v);
template <>
__device__ __forceinline__ void store_f<double>(void *row, int idx, float v) {
    ((double *)row)[idx] = (double)v;
}
template <>
__device__ __forceinline__ void store_f<float>(void *row, int idx, float v) {
    ((float *)row)[idx] = v;
}
template <>
__device__ __forceinline__ void store_f<uint8_t>(void *row, int idx, float v) {
    ((uint8_t *)row)[idx] = (uint8_t)__float2int_rd(fminf(fmaxf(v + 0.5f, 0.0f), 255.0f));  // round half up, saturate
}
template <>
__device__ __forceinline__ void store_f<uint16_t>(void *row, int idx, float v) {
    ((uint16_t *)row)[idx] = (uint16_t)__float2int_rd(fminf(fmaxf(v + 0.5f, 0.0f), 65535.0f));  // round half up, saturate
}

// Batched launches: gridDim.z = the images of an equally strided stack that share one plan (aai_run_device_batch);
// blockIdx.z selects this CTA's image.  The stack is addressed as ONE tall image -- image k's row r is row
// r + k * batch_rows of the stack -- so the batch costs one integer multiply-add per base row instead of 64-bit pointer
// arithmetic (the FP32 overlap kernel is issue-bound: every instruction per pixel shows).  Single-image launches have
// gridDim.z = 1 and batch_rows = 0.
__device__ __forceinline__ int src_row0(const AaiKernelParams &kp) {
    return kp.src_y0 - (int)blockIdx.z * kp.src_batch_rows;
}
__device__ __forceinline__ int dst_row0(const AaiKernelParams &kp) {
    return kp.dst_y0 - (int)blockIdx.z * kp.dst_batch_rows;
}

// expanded + quadrant-rotated pixel (mx,my) -> original source pixel (inverse of Source.cpp:163-168)
__device__ __forceinline__ void mod_to_src(const AaiKernelParams &kp, int mx, int my, int &sx, int &sy) {
    int ex, ey;
    switch (kp.quadrant) {
        case 0: ex = mx; ey = my; break;
        case 1: ex = my; ey = kp.mod_w - 1 - mx; break;
        case 2: ex = kp.mod_w - 1 - mx; ey = kp.mod_h - 1 - my; break;
        default: ex = kp.mod_h - 1 - my; ey = mx; break;
    }
    if (kp.scale == 1) {
        sx = ex;
        sy = ey;
    } else {
        sx = ex / kp.scale;
        sy = ey / kp.scale;
    }
}

// canvas pixel centre, evaluated with the reference's operand order and no FMA contraction (212-219)
__device__ __forceinline__ void pixel_centre(const AaiKernelParams &kp, int x, int y, double &cx, double &cy) {
    const double u = __dadd_rn(__dsub_rn(__dmul_rn(__dadd_rn((double)x, kp.off_ix), kp.side), kp.iso_x), kp.off_x);
    const double v = __dadd_rn(__dsub_rn(__dmul_rn(__dadd_rn((double)y, kp.off_iy), kp.side), kp.iso_y), kp.off_y);
    cx = __dadd_rn(__dadd_rn(__dmul_rn(u, kp.shape.cs), __dmul_rn(v, kp.shape.sn)), kp.iso_x);
    cy = __dadd_rn(__dadd_rn(__dmul_rn(-u, kp.shape.sn), __dmul_rn(v, kp.shape.cs)), kp.iso_y);
}

// the reference's clamped search window (426-429)
__device__ __forceinline__ void search_window(const AaiKernelParams &kp, double cx, double cy, int &x0, int &x1,
                                              int &y0, int &y1) {
    x0 = max(0, __double2int_rd(__dsub_rn(__dsub_rn(cx, kp.reach), 1.0)));
    x1 = min(__double2int_ru(__dadd_rn(__dadd_rn(cx, kp.reach), 1.0)), kp.mod_w - 1);
    y0 = max(0, __double2int_rd(__dsub_rn(__dsub_rn(cy, kp.reach), 1.0)));
    y1 = min(__double2int_ru(__dadd_rn(__dadd_rn(cy, kp.reach), 1.0)), kp.mod_h - 1);
}

// ------------------------------------------------------------------------------------------------------------
// FP64 evaluation of one canvas pixel over the cells [ix0,ix1] x [jy0,jy1] (also the precision fallback of the
// FP32 kernel).
// ------------------------------------------------------------------------------------------------------------
template <typename TI, int NC>
__device__ __forceinline__ void pixel_f64(const AaiKernelParams &kp, double cx, double cy, int ix0, int ix1, int jy0,
                                          int jy1, double &sumA, double (&acc)[NC]) {
    sumA = 0.0;
#pragma unroll
    for (int ch = 0; ch < NC; ++ch) acc[ch] = 0.0;
    if (ix0 > ix1 || jy0 > jy1) return;
    const AaiShape &g = kp.shape;
    // chord of the footprint on the horizontal grid line through the top of row jy0 (relative to C)
    double xlT, xrT;
    aai_chord_h(g, ((double)jy0 - 0.5) - cy, xlT, xrT);
    for (int j = jy0; j <= jy1; ++j) {
        const double ry = (double)j - cy;
        double xlB, xrB;
        aai_chord_h(g, ry + 0.5, xlB, xrB);
        // chord on the vertical grid line through the left of column ix0
        double yt, yb;
        aai_chord_v(g, ((double)ix0 - 0.5) - cx, yt, yb);
        double lenL = aai_overlap1(yt, yb, ry);
        for (int i = ix0; i <= ix1; ++i) {
            const double rx = (double)i - cx;
            aai_chord_v(g, rx + 0.5, yt, yb);
            const double lenR = aai_overlap1(yt, yb, ry);
            const double lenT = aai_overlap1(xlT, xrT, rx);
            const double lenB = aai_overlap1(xlB, xrB, rx);
            const double area = aai_cell_area(g, rx, ry, lenT, lenB, lenL, lenR, kp.quirk != 0);
            lenL = lenR;
            if (area != 0.0) {
                int sx, sy;
                mod_to_src(kp, i, j, sx, sy);
                const char *row = (const char *)kp.src + (int64_t)(sy - src_row0(kp)) * kp.src_pitch;
                sumA += area;
#pragma unroll
                for (int ch = 0; ch < NC; ++ch) acc[ch] += SrcLoad<TI>::get(row, sx * NC + ch) * area;
            }
        }
        xlT = xlB;
        xrT = xrB;
    }
}

// ------------------------------------------------------------------------------------------------------------
// Fast mode (Source.cpp:866-907): unweighted mean of the expanded pixels whose CENTRE lies in the footprint.
// ------------------------------------------------------------------------------------------------------------
// FP64 evaluation of one canvas pixel (also the precision fallback of the FP32 fast kernel)
template <typename TI, int NC>
__device__ __forceinline__ void pixel_fast_f64(const AaiKernelParams &kp, int x, int y, int &count, double (&acc)[NC]) {
    double cx, cy;
    pixel_centre(kp, x, y, cx, cy);
    int wx0, wx1, wy0, wy1;
    search_window(kp, cx, cy, wx0, wx1, wy0, wy1);
    const double ext = kp.hb + 1e-6;
    const int ix0 = max(wx0, __double2int_ru(cx - ext)), ix1 = min(wx1, __double2int_rd(cx + ext));
    const int jy0 = max(wy0, __double2int_ru(cy - ext)), jy1 = min(wy1, __double2int_rd(cy + ext));
    count = 0;
#pragma unroll
    for (int ch = 0; ch < NC; ++ch) acc[ch] = 0.0;
    for (int j = jy0; j <= jy1; ++j) {
        const double ry = (double)j - cy;
        for (int i = ix0; i <= ix1; ++i) {
            const double rx = (double)i - cx;
            const double u0 = rx * kp.shape.cs - ry * kp.shape.sn;
            const double v0 = rx * kp.shape.sn + ry * kp.shape.cs;
            if (fabs(u0) <= kp.shape.half && fabs(v0) <= kp.shape.half) {  // closed point-in-square (837-864)
                int sx, sy;
                mod_to_src(kp, i, j, sx, sy);
                const char *row = (const char *)kp.src + (int64_t)(sy - src_row0(kp)) * kp.src_pitch;
                count += 1;
#pragma unroll
                for (int ch = 0; ch < NC; ++ch) acc[ch] += SrcLoad<TI>::get(row, sx * NC + ch);
            }
        }
    }
}

// Cells that can have non-zero overlap: |i - cx| < hb + 1/2, clamped to the image.  The reference's search window
// (Source.cpp:426-429, search_window() above) always contains this range -- its half width L*sqrt(2)/2 + 1 is at
// least hb + 1/2 = L(c+s)/2 + 1/2 and it is clamped to the same image bounds -- so intersecting with it is a no-op and
// the cells it adds all have zero overlap.  Returns true when the image border cut the range (a border pixel: some
// of its footprint lies outside the image).
__device__ __forceinline__ bool cell_range(const AaiKernelParams &kp, double cx, double cy, int &ix0, int &ix1,
                                           int &jy0, int &jy1) {
    const double ext = kp.hb + 0.5 + 1e-9;
    const int bx0 = __double2int_ru(cx - ext), bx1 = __double2int_rd(cx + ext);
    const int by0 = __double2int_ru(cy - ext), by1 = __double2int_rd(cy + ext);
    ix0 = max(0, bx0);
    ix1 = min(kp.mod_w - 1, bx1);
    jy0 = max(0, by0);
    jy1 = min(kp.mod_h - 1, by1);
    return bx0 < 0 || by0 < 0 || bx1 > kp.mod_w - 1 || by1 > kp.mod_h - 1;
}


// ------------------------------------------------------------------------------------------------------------
// Warp-cooperative FP64 evaluation of the few canvas pixels of a warp that need it (border pixels: the footprint
// leaves the image and the total area is partial; FP32 guard-band hits).  One lane evaluating its 25-49 cells alone keeps
// the other 31 lanes of its warp waiting -- for a small image (BASELINE config 2) or the end bands of a multi-GPU
// partition, whose share of border pixels is high, that was most of the kernel's tail.  Here the 32 lanes take one
// CELL each of the flagged pixel (exact Green area + the per-cell quirk decision, aai_pair_area; the cell's source
// value), and the weighted sum and the total area are reduced with warp shuffles.
// EVERY lane of the warp must call this (no early returns before it); lanes with `need` set receive their pixel's sums.
// ------------------------------------------------------------------------------------------------------------
template <typename TI, int NC>
__device__ __forceinline__ void warp_pixels_f64(const AaiKernelParams &kp, bool need, int x, int y, double &sumA,
                                                double (&acc)[NC]) {
    constexpr unsigned FULL = 0xffffffffu;
    const int lane = (threadIdx.y * TILE_W + threadIdx.x) & 31;
    unsigned todo = __ballot_sync(FULL, need);
    while (todo) {
        const int src_lane = __ffs(todo) - 1;
        todo &= todo - 1;
        const int px = __shfl_sync(FULL, x, src_lane), py = __shfl_sync(FULL, y, src_lane);
        double cx, cy;
        pixel_centre(kp, px, py, cx, cy);
        int i0, i1, j0, j1;
        cell_range(kp, cx, cy, i0, i1, j0, j1);
        const int nc = i1 - i0 + 1, ncell = nc > 0 && j1 >= j0 ? nc * (j1 - j0 + 1) : 0;
        double s = 0.0, a[NC];
#pragma unroll
        for (int ch = 0; ch < NC; ++ch) a[ch] = 0.0;
        for (int c = lane; c < ncell; c += 32) {
            const int j = j0 + c / nc, i = i0 + c % nc;
            const double area = aai_pair_area(kp.shape, cx, cy, i, j, kp.quirk != 0);
            if (area != 0.0) {
                int sx, sy;
                mod_to_src(kp, i, j, sx, sy);
                const char *row = (const char *)kp.src + (int64_t)(sy - src_row0(kp)) * kp.src_pitch;
                s += area;
#pragma unroll
                for (int ch = 0; ch < NC; ++ch) a[ch] += SrcLoad<TI>::get(row, sx * NC + ch) * area;
            }
        }
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
            s += __shfl_xor_sync(FULL, s, off);
#pragma unroll
            for (int ch = 0; ch < NC; ++ch) a[ch] += __shfl_xor_sync(FULL, a[ch], off);
        }
        if (lane == src_lane) {
            sumA = s;
#pragma unroll
            for (int ch = 0; ch < NC; ++ch) acc[ch] = a[ch];
        }
    }
}

}  // namespace aai_dev

#endif  // AAI_DEVICE_CUH_
