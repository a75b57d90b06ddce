// Overlap kernel, FP64 arithmetic, unrolled form (the north star's "FP64 kernel", <= 1e-9 relative to the reference) --
// main loop of AreaAverageInterpolation::areaAverageInterpolation (Source.cpp:411-579) for double images, for every
// image when FP64 arithmetic is requested, and for angles within ~3 degrees of an axis (which the FP32 kernel declines).
//
// Same formulation as the FP32 kernel (aai_kernels_f32.cu) without its FP32-specific parts: compiled once per AAI_MAXN
// (maximum number of cells per axis one footprint can touch) so that the column loop is unrolled and the MAXN+1
// vertical-line chords live in registers; every cell gets its exact overlap (Green form), the total area of a footprint
// inside the image is L^2, and the reference's shape-2/4 quirk is one pair of corrected cells per minor-axis grid line
// that a left/right edge crosses (aai_edge_quirk_f64).  Decisions are made directly on FP64 margins computed from the
// reference's own expression of the footprint centre (pixel_centre): no guard band, no redo.  Border pixels (footprint
// partly outside the image: partial total area) and footprints wider than MAXN take the per-cell routine, evaluated
// warp-cooperatively (warp_pixels_f64 in aai_device.cuh: one cell per lane, shuffle reduction); the rolled kernel
// overlap_kernel_f64 in aai_kernels.cu runs the per-cell routine for every pixel (pixel_f64).
#include "aai_device.cuh"

#ifndef AAI_MAXN
#error "compile with -DAAI_MAXN=4|5|6|8"
#endif

using namespace aai_dev;

namespace {

constexpr int MAXN = AAI_MAXN;
#ifndef AAI_F64_COOP
#define AAI_F64_COOP 0  // 1: border pixels warp-cooperative as in the FP32 kernel.  Measured on BASELINE config 4: 3.603 ms against 3.351 ms for each lane alone (profiles/README.md) -- the FP64 kernel keeps the round-1 form
#endif

#ifndef AAI_F64_MIN_CTAS
#define AAI_F64_MIN_CTAS (512 / (AAI_TILE_W * AAI_TILE_H))  // 4 CTAs of 128 threads per SM: 128 registers
#endif
template <typename TI, typename TO, int NC, bool IDENT>
__global__ void __launch_bounds__(TILE_W *TILE_H, AAI_F64_MIN_CTAS)
    overlap_kernel_f64u(const __grid_constant__ AaiKernelParams kp) {
    // (no early return: every lane of a warp reaches the cooperative section below)
    const int x = blockIdx.x * TILE_W + threadIdx.x;
    const int y = kp.row0 + blockIdx.y * TILE_H + threadIdx.y;
#if AAI_F64_COOP
    const bool valid = x < kp.dst_w && y < kp.row1;
#else
    if (x >= kp.dst_w || y >= kp.row1) return;
    constexpr bool valid = true;
#endif
    double cx, cy;
    pixel_centre(kp, x, y, cx, cy);
    int ix0, ix1, jy0, jy1;
    const bool border = cell_range(kp, cx, cy, ix0, ix1, jy0, jy1);
    const int ncols = ix1 - ix0 + 1, nrows = jy1 - jy0 + 1;
    char *drow = (char *)kp.dst + (int64_t)(y - dst_row0(kp)) * kp.dst_pitch;
    const bool work = valid && ncols > 0 && nrows > 0;
    if (valid && !work) {  // footprint bounding box misses the image: the reference writes 0 (577)
#pragma unroll
        for (int ch = 0; ch < NC; ++ch) store_dst<TO>(drow, x * NC + ch, 0.0);
#if !AAI_F64_COOP
        return;
#endif
    }
    double sumA = 0.0, acc[NC];
    // border pixels (partial total area) and footprints wider than MAXN: per-cell routine, one cell per lane of the warp
    const bool coop = work && (border || ncols > MAXN || nrows > MAXN);
    if (work && !coop) {
        const AaiShape &g = kp.shape;
#pragma unroll
        for (int ch = 0; ch < NC; ++ch) acc[ch] = 0.0;
        const double rx0 = (double)ix0 - cx, ry0 = (double)jy0 - cy;
        const double e0 = rx0 - 0.5, t0 = ry0 - 0.5;  // left boundary of column 0, top of row 0
        double yt[MAXN + 1], yb[MAXN + 1];
#pragma unroll
        for (int k = 0; k <= MAXN; ++k) aai_chord_v(g, e0 + (double)k, yt[k], yb[k]);
        double xlT, xrT;
        aai_chord_h(g, t0, xlT, xrT);
        double lenTop[MAXN];  // the cells' top sides inside the footprint: the previous row's bottom sides
        {
            double prev = aai_clamp_chord(e0, xlT, xrT);
#pragma unroll
            for (int k = 0; k < MAXN; ++k) {
                const double next = aai_clamp_chord(e0 + (double)(k + 1), xlT, xrT);
                lenTop[k] = next - prev;
                prev = next;
            }
        }
        double cv[MAXN + 1];  // vertical chords clamped at the top of the current row
#pragma unroll
        for (int k = 0; k <= MAXN; ++k) cv[k] = aai_clamp_chord(t0, yt[k], yb[k]);
        constexpr int ESZ = (int)sizeof(TI) * NC;
        const char *rowp0 = (const char *)kp.src + (int64_t)(jy0 - src_row0(kp)) * kp.src_pitch + (int64_t)ix0 * ESZ;
        // General frame: expanded pixel (i,j) -> source pixel is separable (one source coordinate depends on the column
        // only, the other on the row only; swapped for quadrants 1/3): byte offset = col_off(i) + row_off(j), the column
        // parts hoisted out of the row loop (as in the FP32 kernel).
        const bool swapped = kp.e_axi == 0;
        auto div_s = [&](int e) -> int64_t {
            return (int64_t)(kp.scale != 1 ? __umulhi((unsigned)e, kp.div_magic) : (unsigned)e);
        };
        auto col_off = [&](int i) -> int64_t {
            return swapped ? (div_s(kp.e_ayi * i + kp.e_ay0) - src_row0(kp)) * kp.src_pitch
                           : div_s(kp.e_axi * i + kp.e_ax0) * ESZ;
        };
        auto row_off = [&](int j) -> int64_t {
            return swapped ? div_s(kp.e_axj * j + kp.e_ax0) * ESZ
                           : (div_s(kp.e_ayj * j + kp.e_ay0) - src_row0(kp)) * kp.src_pitch;
        };
        int64_t coff[MAXN];
        if (!IDENT) {
#pragma unroll
            for (int k = 0; k < MAXN; ++k) coff[k] = col_off(ix0 + min(k, ncols - 1));
        }
        auto cell_ptr = [&](int k, int r) -> const char * {  // source element of cell (column k, row r), any k
            if (IDENT) return rowp0 + (int64_t)r * kp.src_pitch + (int64_t)k * ESZ;
            return (const char *)kp.src + row_off(jy0 + r) + col_off(ix0 + k);
        };
        for (int r = 0; r < nrows; ++r) {
            const char *rowp = IDENT ? rowp0 + (int64_t)r * kp.src_pitch : (const char *)kp.src + row_off(jy0 + r);
            const double ry = ry0 + (double)r;
            double xlB, xrB;
            aai_chord_h(g, ry + 0.5, xlB, xrB);
            const double yb1 = ry + 0.5;  // bottom of this row
            double cnext = aai_clamp_chord(yb1, yt[0], yb[0]);
            double lenL = cnext - cv[0];
            cv[0] = cnext;
            double hprev = aai_clamp_chord(e0, xlB, xrB);
#pragma unroll
            for (int k = 0; k < MAXN; ++k) {
                const double rx = rx0 + (double)k;
                cnext = aai_clamp_chord(yb1, yt[k + 1], yb[k + 1]);
                const double lenR = cnext - cv[k + 1];
                cv[k + 1] = cnext;
                const double hnext = aai_clamp_chord(e0 + (double)(k + 1), xlB, xrB);
                const double lenB = hnext - hprev;
                hprev = hnext;
                const double area = aai_cell_exact_f64(g, rx, ry, lenTop[k], lenB, lenL, lenR);
                lenTop[k] = lenB;
                lenL = lenR;
                if (k < ncols) {  // columns beyond the footprint box are never read (their area is exactly 0)
                    const char *p = IDENT ? rowp + k * ESZ : rowp + coff[k];
#pragma unroll
                    for (int ch = 0; ch < NC; ++ch) acc[ch] = fma(SrcLoad<TI>::get(p, ch), area, acc[ch]);
                }
            }
        }
        // total overlap: the exact areas of a footprint inside the image add up to L^2
        sumA = g.area_total;
        if (kp.quirk) {
            const double g0m = g.steep ? e0 : t0, g0M = g.steep ? t0 : e0;
            auto fix = [&](int mi, int Mi, double d) {  // cell (minor index, major index) += d
                const int k = g.steep ? mi : Mi, r = g.steep ? Mi : mi;
                if (d != 0.0 && (unsigned)k < (unsigned)ncols && (unsigned)r < (unsigned)nrows) {
                    const char *p = cell_ptr(k, r);
                    sumA += d;
#pragma unroll
                    for (int ch = 0; ch < NC; ++ch) acc[ch] = fma(SrcLoad<TI>::get(p, ch), d, acc[ch]);
                }
            };
            for (int q = 0; q < g.ncross; ++q) {
                int mi, Mi;
                double db, da;
                aai_edge_quirk_f64<true>(g, g0m, g0M, q, mi, Mi, db, da);
                fix(mi, Mi, db);
                fix(mi + 1, Mi, da);
                aai_edge_quirk_f64<false>(g, g0m, g0M, q, mi, Mi, db, da);
                fix(mi, Mi, db);
                fix(mi + 1, Mi, da);
            }
        }
    }
#if AAI_F64_COOP
    if (__any_sync(0xffffffffu, coop)) warp_pixels_f64<TI, NC>(kp, coop, x, y, sumA, acc);
#else
    if (coop) pixel_f64<TI, NC>(kp, cx, cy, ix0, ix1, jy0, jy1, sumA, acc);
#endif
    if (work) {
        const bool ok = DBL_EPSILON < fabs(sumA);  // Source.cpp:577
#pragma unroll
        for (int ch = 0; ch < NC; ++ch) store_dst<TO>(drow, x * NC + ch, ok ? acc[ch] / sumA : 0.0);
    }
}

template <typename TI, typename TO, int NC>
cudaError_t launch3(const AaiKernelParams &kp, cudaStream_t stream) {
    const int rows = kp.row1 - kp.row0;
    if (rows <= 0 || kp.dst_w <= 0) return cudaSuccess;
    dim3 block(TILE_W, TILE_H);
    dim3 grid((kp.dst_w + TILE_W - 1) / TILE_W, (rows + TILE_H - 1) / TILE_H, kp.batch > 1 ? kp.batch : 1);
    if (kp.scale == 1 && kp.quadrant == 0)
        overlap_kernel_f64u<TI, TO, NC, true><<<grid, block, 0, stream>>>(kp);
    else
        overlap_kernel_f64u<TI, TO, NC, false><<<grid, block, 0, stream>>>(kp);
    return cudaGetLastError();
}
template <typename TI, typename TO>
cudaError_t launch2(const AaiKernelParams &kp, cudaStream_t stream) {
    switch (kp.channels) {
        case 1: return launch3<TI, TO, 1>(kp, stream);
        case 3: return launch3<TI, TO, 3>(kp, stream);
        default: return cudaErrorNotSupported;  // the caller falls back to the rolled kernel
    }
}
template <typename TI>
cudaError_t launch1(const AaiKernelParams &kp, int dst_dtype, cudaStream_t stream) {
    switch (dst_dtype) {
        case AAI_F64: return launch2<TI, double>(kp, stream);
        case AAI_F32: return launch2<TI, float>(kp, stream);
        case AAI_U8: if constexpr (pair_ok<TI, uint8_t>()) return launch2<TI, uint8_t>(kp, stream); break;
        case AAI_U16: if constexpr (pair_ok<TI, uint16_t>()) return launch2<TI, uint16_t>(kp, stream); break;
    }
    return cudaErrorInvalidValue;
}

}  // namespace

#define AAI_CAT2(a, b) a##b
#define AAI_CAT(a, b) AAI_CAT2(a, b)

int AAI_CAT(aai_launch_overlap_f64_n, AAI_MAXN)(const AaiKernelParams &kp, int src_dtype, int dst_dtype, void *stream) {
    cudaStream_t st = (cudaStream_t)stream;
    switch (src_dtype) {
        case AAI_F64: return (int)launch1<double>(kp, dst_dtype, st);
        case AAI_F32: return (int)launch1<float>(kp, dst_dtype, st);
        case AAI_U8: return (int)launch1<uint8_t>(kp, dst_dtype, st);
        case AAI_U16: return (int)launch1<uint16_t>(kp, dst_dtype, st);
        default: return (int)cudaErrorInvalidValue;
    }
}
