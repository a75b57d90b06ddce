// Overlap kernel, FP32 arithmetic (the north star's "FP32 kernel") -- main loop of
// AreaAverageInterpolation::areaAverageInterpolation (Source.cpp:411-579) for float / 8-bit / 16-bit images.
//
// Compiled once per AAI_MAXN (4, 5, 6, 8 = maximum number of source cells per axis that one footprint can
// touch; the host picks the smallest that fits L(cos+sin)+1), so that the column loop is fully unrolled and the
// MAXN+1 vertical-line chords of the footprint live in registers.
//
// Same formulation as the FP64 kernel (aai_kernels.cu), on footprint-local coordinates:
//   * the footprint centre is computed in FP64 exactly like the reference (212-219) and split into the nearest
//     lattice point + an FP32 fraction, so every FP32 quantity is O(L) with ~1e-7 absolute error;
//   * side lengths |side ∩ footprint| are differences of FADD.SAT (no min/max on the half-rate ALU pipe);
//   * the kernel is instruction-issue bound, so horizontally adjacent cells are evaluated two at a time on
//     Blackwell's packed FP32 instructions (FFMA2 / FMUL2 / FADD2 = fma.rn.f32x2, sm_100a);
//   * every cell gets its exact overlap (Green form, no decision), so the total area of a footprint inside the image
//     is L^2 and is not accumulated; the reference's shape-2/4 quirk is then applied as one pair of corrected cells
//     per minor-axis grid line that a left/right footprint edge crosses (aai_edge_quirk_f32 in aai_cell.cuh: at most
//     2 (floor(L min(s,c)) + 1) events per canvas pixel instead of a search in every row);
//     the smallest decision margin of the pixel is tracked and, when it falls inside the FP32 guard band, or when
//     the image border clips the footprint (border pixels need relative accuracy), the pixel is redone in FP64
//     (pixel_f64) -- FP32 rounding can never flip one of the reference's discontinuous decisions.
#include <cuda.h>

#include <algorithm>
#include <cmath>

#include "aai_device.cuh"

#ifndef AAI_MAXN
#error "compile with -DAAI_MAXN=4|5|6|8"
#endif

using namespace aai_dev;

namespace {

constexpr int MAXN = AAI_MAXN;
#ifndef AAI_ROW_UNROLL
#define AAI_ROW_UNROLL 1
#endif
constexpr int kRowUnroll = AAI_ROW_UNROLL;
#ifndef AAI_WIN_ROW_UNROLL
// rows of the cell window (WIN below) per loop iteration: all of them.  Measured on config 4 (MAXN 5, B200 at 1000 W,
// 1965 MHz): 1.314 ms with 1 row, 1.307 ms with 2, 1.156 ms with 4 (the row-to-row register moves of the prefetch and the
// chords vanish; profiles/r3_tip_window_ab.json)
#define AAI_WIN_ROW_UNROLL (AAI_MAXN - 1)
#endif
constexpr int kWinRowUnroll = AAI_WIN_ROW_UNROLL;
// Columns that every interior footprint of this translation unit touches: a footprint box of side 2 ext holds at least
// floor(2 ext) lattice columns, and the host picks the smallest MAXN >= floor(2 ext) + 1 (MAXN = 8 also serves
// floor(2 ext) = 6, MAXN = 4 also floor(2 ext) = 2: L(c+s) < 2).  Their loads need no predicate; a pixel whose FP32 cell
// range comes out narrower (2 ext within rounding of an integer) takes the FP64 path.
#ifndef AAI_MINC
#define AAI_MINC (AAI_MAXN == 8 ? 6 : AAI_MAXN == 4 ? 2 : AAI_MAXN - 1)
#endif
constexpr int MINC = AAI_MINC;


// ------------------------------------------------------------------------------------------------------------
// STAGED variants (the north star's lay-out, selected with AAI_ARITH_F32_STAGED): the source window of a CTA's 16 x 8
// canvas pixels is brought into shared memory by ONE 2-D TMA tile load (cp.async.bulk.tensor.2d through a CUtensorMap,
// completion on an mbarrier) and the cells are read with LDS instead of LDG.  Footprints of a rotated canvas row step
// through the source diagonally, so a warp's 32 loads of "cell k" hit ~28 different 32-byte sectors -- 28 L1 tag
// wavefronts per LDG -- while the same 32 addresses in shared memory cost ~2.6 bank-conflict wavefronts.  Measured
// (profiles/README.md, round 2): that relief does not pay for the per-CTA load latency -- overlap kernel 1.475 ms staged
// against 1.386 ms through L1 on BASELINE config 4, fast mode 0.658 against 0.616 ms -- so both default to LDG.
// Identity addressing only (scale 1, quadrant 0); the window origin is rounded down to a 16-byte boundary (TMA
// requirement); out-of-image parts of the box are zero-filled by the hardware and never read (pixels whose footprint
// box leaves the image take the FP64 path, which reads global memory).
// ------------------------------------------------------------------------------------------------------------
struct StageParams {
    int bw, bh;  // TMA box = source window of one CTA: elements (pixels x channels) per row, rows
};

__device__ __forceinline__ uint32_t st_smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

// Loads the CTA's source window; every thread of the CTA must call it (it synchronises).  Returns the window origin
// (sox in ELEMENTS of the interleaved row, soy in rows of the whole image) -- valid also when nothing was loaded
// because the window misses the image.
template <int EB, int NC>  // EB = bytes per element, NC = interleaved channels
__device__ __forceinline__ void stage_window(const CUtensorMap *tmap, const AaiKernelParams &kp, const StageParams &sp,
                                             unsigned char *smem, uint64_t *bar, int *origin, float ext, int &sox,
                                             int &soy) {
    const int tid = threadIdx.y * TILE_W + threadIdx.x;
    if (tid == 0) {  // one thread: window origin (FP64, the centre map is affine: extremes at the tile's corners), TMA
        const int x0 = blockIdx.x * TILE_W, y0 = kp.row0 + blockIdx.y * TILE_H;
        double lox = 1e300, loy = 1e300;
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            const double xx = (double)(x0 + (c & 1) * (TILE_W - 1)), yy = (double)(y0 + (c >> 1) * (TILE_H - 1));
            lox = fmin(lox, fma(xx, kp.aff_xx, fma(yy, kp.aff_xy, kp.aff_x0)));
            loy = fmin(loy, fma(xx, kp.aff_yx, fma(yy, kp.aff_yy, kp.aff_y0)));
        }
        constexpr int EAL = 16 / EB;  // elements per 16 bytes: the TMA start coordinate must be a multiple of it
        int ex = (__double2int_rd(lox - (double)ext) - 1) * NC;
        ex = (ex >= 0 ? ex / EAL : -((-ex + EAL - 1) / EAL)) * EAL;
        const int ey = __double2int_rd(loy - (double)ext) - 1;
        origin[0] = ex;
        origin[1] = ey;
        asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(st_smem_u32(bar)), "r"(1));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        const uint32_t bytes = (uint32_t)(sp.bw * sp.bh * EB);
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(st_smem_u32(bar)), "r"(bytes) : "memory");
        asm volatile(
            "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::
                "r"(st_smem_u32(smem)),
            "l"(tmap), "r"(st_smem_u32(bar)), "r"(ex), "r"(ey - src_row0(kp))
            : "memory");
    }
    __syncthreads();  // barrier initialised, origin visible
    sox = origin[0];
    soy = origin[1];
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "ST_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra.uni ST_DONE;\n"
        "bra.uni ST_WAIT;\n"
        "ST_DONE:\n"
        "}\n" ::"r"(st_smem_u32(bar)),
        "r"(0)
        : "memory");
}

template <typename TI, bool STAGED>
struct LoadS {
    static __device__ __forceinline__ float get(const char *p) {
        if constexpr (STAGED)
            return to_arith<float>(*reinterpret_cast<const TI *>(p));  // shared memory (the pointer derives from the staged tile)
        else
            return LoadF<TI>::get(p);
    }
};

// ---- host side of the staged variants: tensor map over the (band of the / stack of) source image(s) + box size ------
typedef CUresult (*StEncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                    const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
StEncodeTiledFn st_encode_fn() {
    static const StEncodeTiledFn fn = [] {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            return (StEncodeTiledFn)p;
        cudaGetLastError();
        return (StEncodeTiledFn) nullptr;
    }();
    return fn;
}

struct StageHost {
    CUtensorMap map;
    StageParams sp;
    size_t smem;
};
// false: the staged variant does not apply (the caller launches the LDG kernel)
template <typename TI, int NC>
bool stage_prepare(const AaiKernelParams &kp, double ext, StageHost &h) {
    StEncodeTiledFn enc = st_encode_fn();
    if (!enc || kp.scale != 1 || kp.quadrant != 0 || sizeof(TI) == 8) return false;
    if ((kp.src_pitch % 16) != 0 || (reinterpret_cast<uintptr_t>(kp.src) % 16) != 0) return false;
    constexpr int EB = (int)sizeof(TI), EAL = 16 / EB;
    // extent of the footprint centres over one tile (the centre map is affine), plus the cell range on both sides, plus
    // the slack of stage_window() (one pixel, alignment of the origin)
    const double sx = (TILE_W - 1) * std::fabs(kp.aff_xx) + (TILE_H - 1) * std::fabs(kp.aff_xy);
    const double sy = (TILE_W - 1) * std::fabs(kp.aff_yx) + (TILE_H - 1) * std::fabs(kp.aff_yy);
    const int wpx = (int)std::ceil(sx + 2.0 * ext) + 4;
    h.sp.bw = (wpx * NC + (EAL - 1) + EAL - 1) / EAL * EAL;
    h.sp.bh = (int)std::ceil(sy + 2.0 * ext) + 4;
    h.smem = (size_t)h.sp.bw * h.sp.bh * EB;
    if (h.sp.bw > 256 || h.sp.bh > 256 || h.smem > 30 * 1024) return false;
    // one tall 2-D tensor: a stack of equally strided slices is addressed through its row index (src_batch_rows)
    const int64_t rows = kp.batch > 1 ? (int64_t)kp.src_batch_rows * kp.batch : (int64_t)kp.src_rows;
    const cuuint64_t gdim[2] = {(cuuint64_t)kp.src_w * NC, (cuuint64_t)rows};
    const cuuint64_t gstride[1] = {(cuuint64_t)kp.src_pitch};
    const cuuint32_t box[2] = {(cuuint32_t)h.sp.bw, (cuuint32_t)h.sp.bh};
    const cuuint32_t estr[2] = {1, 1};
    return enc(&h.map, Elem<TI>::tmap, 2, const_cast<void *>(kp.src), gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
               CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
               CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}


// IDENT: scale 1, quadrant 0 (expanded pixel (i,j) IS source pixel (i,j)): constant element stride, offsets fold
// into the load instruction.  Otherwise the general expanded-frame affine map + division by the scale.
#ifndef AAI_F32_MIN_BLOCKS
// resident threads per SM the register allocation is bounded for: 28 warps (72 registers) for MAXN = 4, 24 warps (80
// registers) for MAXN = 5 (measured on config 4 with the final row body: 5/6/7/8 CTAs per SM = 1.562/1.455/1.466/1.529 ms;
// config 3, MAXN = 4: 6 CTAs 8.19 ms vs 7 CTAs 8.14 ms), 16 warps for the wide footprints
#define AAI_F32_MIN_BLOCKS ((AAI_MAXN <= 4 ? 896 : AAI_MAXN == 5 ? 768 : 512) / (AAI_TILE_W * AAI_TILE_H))
#endif
// ADDR: how a cell finds its source value.
//   ADDR_GENERAL  expanded + quadrant-rotated frame, separable byte offset col_off(i) + row_off(j)
//   ADDR_IDENT    scale 1, quadrant 0: expanded pixel (i,j) IS source pixel (i,j), offsets fold into the loads
//   ADDR_GROUPED  general frame with scale >= MAXN-1 (upscaling): the <= MAXN x MAXN cells of a footprint fall into at
//                 most 2 x 2 source pixels, so the four weights are computed DIRECTLY (aai_quadrant_areas_f32: Green form
//                 about the corner of the source-pixel boundaries, no loop over cells), the quirk corrections are added
//                 per source pixel, and each source pixel is loaded ONCE per canvas pixel
enum { ADDR_GENERAL = 0, ADDR_IDENT = 1, ADDR_GROUPED = 2 };
// stage / spitch / sox / soy: the CTA's staged source window (STAGED only): row pitch in bytes, origin in elements / rows
// PDL: the instantiation for SHORT launches (row bands of a multi-GPU partition, pipeline chunks, small images), launched
// with the programmatic-stream-serialization attribute: it releases its dependents at once (the next launch's CTAs become
// resident while this grid's last wave drains) and touches no global memory before griddepcontrol.wait, which returns
// once the preceding grid has completed and flushed -- so any data dependence between consecutive launches is still
// honoured.  Measured (profiles/r2_z_pdl_ab.txt): the 8 bands of config 4 0.1844 -> 0.1824 ms, config 2 38 -> 36 us; the
// two instructions cost ~80 ns per CTA on long launches, and even behind a run-time flag 0.7 % of the whole-canvas
// launch -- hence a separate instantiation, used below kPdlMaxCtas CTAs only.
// WIN (identity addressing, one channel, plans that pass aai_tip_window_ok): a fixed window of MAXN-1 rows x MAXN-1
// columns from the footprint's first cell row and column, then the two tips of the footprint outside it in closed form
// (aai_tip_strips_f32).  A box of D = L(c+s) < MAXN - 1 cells holds MAXN - 1 or MAXN cells per axis, but the
// row loop runs to the warp's largest count and the columns are unrolled to MAXN, so every pixel paid for MAXN^2 cells.
template <typename TI, typename TO, int NC, int ADDR, bool STAGED, bool PDL = false, bool REV = false, bool WIN = false>
__device__ __forceinline__ void overlap_body(const AaiKernelParams &kp, const char *stage, int spitch, int sox, int soy) {
    constexpr bool IDENT = ADDR == ADDR_IDENT, GROUPED = ADDR == ADDR_GROUPED;
    static_assert(!STAGED || IDENT, "staging is implemented for identity addressing");
    static_assert(!WIN || (IDENT && NC == 1), "the cell window is implemented for identity addressing, one channel");
    constexpr int NCOL = WIN ? MAXN - 1 : MAXN;  // cell columns evaluated per row
    if constexpr (PDL) asm volatile("griddepcontrol.launch_dependents;");
    // (no early return: every lane of a warp reaches the cooperative FP64 section at the end)
    const int x = blockIdx.x * TILE_W + threadIdx.x;
    // REV (short-launch instantiation only): CTA rows bottom-up.  A row band whose covered span narrows downwards -- the
    // lower half of a rotated canvas -- measured 2 % slower top-down than bottom-up (config 4, 8 bands: 0.1824 vs 0.1787 ms,
    // profiles/r2_zz_band_order.txt), so the launcher picks the direction in which the covered rows get wider.  A compile-
    // time choice: as a run-time select the same arithmetic cost every launch 3.4 %.
    const int by = REV ? (int)gridDim.y - 1 - (int)blockIdx.y : (int)blockIdx.y;
    const int y = kp.row0 + by * TILE_H + threadIdx.y;
    const bool valid = x < kp.dst_w && y < kp.row1;
    // Footprint centre from the affine form of Source.cpp:212-219 (two FP64 FMAs per coordinate; within ~1e-12 of
    // the reference's own expression, pixel_centre(), which the FP64 redo path below evaluates), split into the nearest
    // lattice point and an FP32 fraction.
    const double cx = fma((double)x, kp.aff_xx, fma((double)y, kp.aff_xy, kp.aff_x0));
    const double cy = fma((double)x, kp.aff_yx, fma((double)y, kp.aff_yy, kp.aff_y0));
    const int irx = __double2int_rn(cx), iry = __double2int_rn(cy);
    const float fx = (float)(cx - (double)irx), fy = (float)(cy - (double)iry);
    // cells that can have non-zero overlap (|i - cx| < hb + 1/2, FP32 with a safety margin: the cells it may add have
    // exactly zero area), clamped to the image; border = some of the footprint's box lies outside the image
    const int bx0 = irx + __float2int_ru(fx - kp.ext32), bx1 = irx + __float2int_rd(fx + kp.ext32);
    const int by0 = iry + __float2int_ru(fy - kp.ext32), by1 = iry + __float2int_rd(fy + kp.ext32);
    const int ix0 = max(0, bx0), ix1 = min(kp.mod_w - 1, bx1), jy0 = max(0, by0), jy1 = min(kp.mod_h - 1, by1);
    const bool border = bx0 < 0 || by0 < 0 || bx1 > kp.mod_w - 1 || by1 > kp.mod_h - 1;
    const int ncols = ix1 - ix0 + 1, nrows = jy1 - jy0 + 1;
    char *drow = (char *)kp.dst + (int64_t)(y - dst_row0(kp)) * kp.dst_pitch;
    const bool work = valid && ncols > 0 && nrows > 0;
    if constexpr (PDL) asm volatile("griddepcontrol.wait;" ::: "memory");  // above: address arithmetic only
    if (valid && !work) {  // footprint bounding box misses the image: the reference writes 0 (577)
#pragma unroll
        for (int ch = 0; ch < NC; ++ch) store_f<TO>(drow, x * NC + ch, 0.0f);
    }
    float sumA = 0.0f, acc[NC];
#pragma unroll
    for (int ch = 0; ch < NC; ++ch) acc[ch] = 0.0f;
    float worst = 1.0f;
    // Border pixels (footprint partly outside the image) are normalised by a partial, possibly tiny, total area:
    // they need relative accuracy, so they take the FP64 path (~0.1% of a large canvas).
    bool redo = work && (border || ncols > MAXN || nrows > MAXN || ncols < MINC);  // (the MAXN test cannot fire for the MAXN the host picked)
    if (WIN) redo = redo || (work && nrows < MAXN - 1);  // the window's cells are read without predicates
    if (work && !redo) {
        const AaiShapeF &g = kp.shapef;
        const int dj0 = jy0 - iry;
        const float rx0 = (float)(ix0 - irx) - fx;
        float yt[NCOL + 1], yb[NCOL + 1];
        if (!GROUPED) {
#pragma unroll
            for (int k = 0; k + 1 <= NCOL; k += 2) {  // two grid lines per packed instruction
                AaiF2 t2, b2;
                aai_chord_v_f32x2(g, aai_f2(rx0 + ((float)k - 0.5f), rx0 + ((float)k + 0.5f)), t2, b2);
                yt[k] = t2.x;
                yt[k + 1] = t2.y;
                yb[k] = b2.x;
                yb[k + 1] = b2.y;
            }
            if ((NCOL + 1) & 1) aai_chord_v_f32(g, rx0 + ((float)NCOL - 0.5f), yt[NCOL], yb[NCOL]);
        }
        float xlT = 0.0f, xrT = 0.0f;  // chord of the footprint on the row's top grid line
        const float t0 = ((float)dj0 - fy) - 0.5f;  // top of row 0
        if (!GROUPED) aai_chord_h_f32(g, t0, xlT, xrT);
        const float e0 = rx0 - 0.5f;  // left boundary of column 0
        constexpr int ESZ = (int)sizeof(TI) * NC;
        // row pitch and first cell of the footprint: in the source image, or (STAGED) in the CTA's shared-memory window
        const int64_t pitch = STAGED ? (int64_t)spitch : kp.src_pitch;
        const char *rowp0 = STAGED ? stage + (jy0 - soy) * spitch + (ix0 * NC - sox) * (int)sizeof(TI)
                                   : (const char *)kp.src + (int64_t)(jy0 - src_row0(kp)) * kp.src_pitch + (int64_t)ix0 * ESZ;
        const char *rowp = rowp0;
        // General path: expanded pixel (i,j) -> source pixel is separable (one source coordinate depends on the
        // column only, the other on the row only; which one is swapped for quadrants 1/3), so the byte offset is
        // col_off(i) + row_off(j); the column parts are hoisted out of the row loop.
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
        if (!IDENT && !GROUPED) {
#pragma unroll
            for (int k = 0; k < MAXN; ++k) coff[k] = col_off(ix0 + min(k, ncols - 1));
        }
        // GROUPED: the first nA columns of the cell range belong to the first source column, the rest to the second one;
        // rows likewise (nT); W[row group][column group] = total weight of the source pixel.  Along an axis the
        // expanded coordinate e moves by +-1 per cell, so the first group holds S - e mod S (resp. e mod S + 1) cells.
        int nA = MAXN, nT = MAXN;
        float W00 = 0.0f, W01 = 0.0f, W10 = 0.0f, W11 = 0.0f;
        if (GROUPED) {
            auto first_group = [&](int e, int step) -> int {  // cells sharing the first cell's source pixel
                const int rem = e - (int)div_s(e) * kp.scale;
                return step > 0 ? kp.scale - rem : rem + 1;
            };
            const int ac = swapped ? kp.e_ayi : kp.e_axi, ec0 = swapped ? kp.e_ay0 : kp.e_ax0;
            const int ar = swapped ? kp.e_axj : kp.e_ayj, er0 = swapped ? kp.e_ax0 : kp.e_ay0;
            nA = first_group(ac * ix0 + ec0, ac);
            nT = first_group(ar * jy0 + er0, ar);
            // the source-pixel boundaries inside the cell range (at most one per axis: the range holds <= scale + 1
            // cells), relative to the footprint centre; none -> beyond the footprint
            aai_quadrant_areas_f32(g, e0 + (float)nA, t0 + (float)nT, nA < ncols, nT < nrows, W00, W01, W10, W11);
        }
        // lengths of the cells' top sides inside the footprint: the previous row's bottom sides
        float lenTop[NCOL];
        if (!GROUPED) {
#pragma unroll
            for (int k = 0; k < NCOL; ++k) lenTop[k] = aai_overlap1_f32(xlT, xrT, e0 + (float)k);
        }
        // Source values are fetched one row ahead of their use (the loads of row r+1 are in flight while the areas of
        // row r are computed): the accumulate at the end of a row never waits for its own row's loads.
        // (Single-channel kernels only: three channels would need 30 staging registers.)
        constexpr bool PREFETCH = NC == 1 && !GROUPED;
        float buf[NCOL][NC];
        auto fetch = [&](int r, float (&v)[NCOL][NC]) {
            if (IDENT)
                rowp = rowp0 + (int64_t)r * pitch;
            else
                rowp = (const char *)kp.src + row_off(jy0 + r);
#pragma unroll
            for (int k = 0; k < NCOL; ++k) {
#pragma unroll
                for (int ch = 0; ch < NC; ++ch) v[k][ch] = 0.0f;
                if (k < MINC || k < ncols) {  // columns beyond the footprint box are never read (their area is exactly 0)
                    const char *p = IDENT ? rowp + k * ESZ : rowp + coff[k];
#pragma unroll
                    for (int ch = 0; ch < NC; ++ch) v[k][ch] = LoadS<TI, STAGED>::get(p + ch * (int)sizeof(TI));
                }
            }
        };
        if (PREFETCH) fetch(0, buf);
        // one row of cells: `cur` holds this row's source values (PREFETCH), `nxt` receives the next row's
        const int nr = WIN ? MAXN - 1 : nrows;  // rows evaluated
        auto row = [&](int r, float (&cur)[NCOL][NC], float (&nxt)[NCOL][NC]) {
            if (PREFETCH) {
                if (r + 1 < nr) fetch(r + 1, nxt);
            } else {
                rowp = IDENT ? rowp0 + (int64_t)r * pitch : (const char *)kp.src + row_off(jy0 + r);
            }
            const float ry = (float)(dj0 + r) - fy;
            float xlB, xrB;
            aai_chord_h_f32(g, ry + 0.5f, xlB, xrB);
            const float ey = ry - 0.5f;
            float lenL = aai_overlap1_f32(yt[0], yb[0], ey);
            const float ur = -ry * g.sn, vr = ry * g.cs;
            auto take = [&](int k, float area) {
                if (PREFETCH) {
#pragma unroll
                    for (int ch = 0; ch < NC; ++ch) acc[ch] = fmaf(cur[k][ch], area, acc[ch]);
                } else if (k < MINC || k < ncols) {  // load at the point of use
                    const char *p = IDENT ? rowp + k * ESZ : rowp + coff[k];
#pragma unroll
                    for (int ch = 0; ch < NC; ++ch)
                        acc[ch] = fmaf(LoadS<TI, STAGED>::get(p + ch * (int)sizeof(TI)), area, acc[ch]);
                }
            };
            // cells two at a time on the packed FP32 pipe (FFMA2/FMUL2/FADD2), a last odd cell on the scalar one
#pragma unroll
            for (int k = 0; k + 1 < NCOL; k += 2) {
                const float rxa = rx0 + (float)k, rxb = rx0 + (float)(k + 1);
                const float exa = rxa - 0.5f, exb = rxb - 0.5f;
                // side lengths of the two cells: saturated ends on the scalar pipe, their differences packed
                const AaiF2 lMR = aai_sub2(aai_f2(aai_sat(yb[k + 1] - ey), aai_sat(yb[k + 2] - ey)),
                                           aai_f2(aai_sat(yt[k + 1] - ey), aai_sat(yt[k + 2] - ey)));
                const float lenM = lMR.x, lenR = lMR.y;
                const AaiF2 lT = aai_f2(lenTop[k], lenTop[k + 1]);
                const AaiF2 lB = aai_sub2(aai_f2(aai_sat(xrB - exa), aai_sat(xrB - exb)),
                                          aai_f2(aai_sat(xlB - exa), aai_sat(xlB - exb)));
                lenTop[k] = lB.x;
                lenTop[k + 1] = lB.y;
                const AaiF2 rx2 = aai_f2(rxa, rxb);
                const AaiF2 u0 = aai_fma2(rx2, aai_f2(g.cs), aai_f2(ur)), v0 = aai_fma2(rx2, aai_f2(g.sn), aai_f2(vr));
                const AaiF2 area = aai_cell_exact_f32x2(g, u0, v0, lT, lB, aai_f2(lenL, lenM), aai_f2(lenM, lenR));
                lenL = lenR;
                take(k, area.x);
                take(k + 1, area.y);
            }
            if (NCOL & 1) {
                constexpr int k = NCOL - 1;
                const float rx = rx0 + (float)k;
                const float ex = rx - 0.5f;
                const float lenR = aai_overlap1_f32(yt[k + 1], yb[k + 1], ey);
                const float lenT = lenTop[k];
                const float lenB = aai_overlap1_f32(xlB, xrB, ex);
                lenTop[k] = lenB;
                const float u0 = fmaf(rx, g.cs, ur), v0 = fmaf(rx, g.sn, vr);
                const float area = aai_cell_exact_f32(g, u0, v0, lenT, lenB, lenL, lenR);
                take(k, area);
            }
        };
        auto row_step = [&](int r) {
            float nxt[NCOL][NC];
            row(r, buf, nxt);
            if (PREFETCH) {
#pragma unroll
                for (int k = 0; k < NCOL; ++k)
#pragma unroll
                    for (int ch = 0; ch < NC; ++ch) buf[k][ch] = nxt[k][ch];
            }
        };
        if (WIN) {
#pragma unroll kWinRowUnroll
            for (int r = 0; r < MAXN - 1; ++r) row_step(r);
        } else if (!GROUPED) {
#pragma unroll kRowUnroll
            for (int r = 0; r < nrows; ++r) row_step(r);
        }
        if constexpr (WIN) {  // the right tip in column MAXN-1, the bottom tip in row MAXN-1
            int first[2];
            AaiF2 tip[3];
            aai_tip_strips_f32<MAXN - 1>(g, e0, t0, first, tip);
            // strips beyond the box have area 0: their loads are clamped into it
            const char *colp = rowp0 + min(MAXN - 1, ncols - 1) * ESZ, *rowpb = rowp0 + min(MAXN - 1, nrows - 1) * pitch;
#pragma unroll
            for (int j = 0; j < 3; ++j) {
                acc[0] = fmaf(LoadS<TI, STAGED>::get(colp + min(first[0] + j, nrows - 1) * pitch), tip[j].x, acc[0]);
                acc[0] = fmaf(LoadS<TI, STAGED>::get(rowpb + min(first[1] + j, ncols - 1) * ESZ), tip[j].y, acc[0]);
            }
        }
        // Total overlap: the exact areas of a footprint inside the image add up to L^2 (border pixels never get here).
        sumA = g.area_total;
        // The reference's shape-2/4 quirk: one pair of corrected cells per minor-axis grid line crossed by a left/right
        // edge (DESIGN.md 3.3).
        if (kp.quirk) {
            const float g0m = g.steep ? e0 : t0, g0M = g.steep ? t0 : e0;
            // the two cells of a crossing are neighbours along the minor axis: one address, one stride.  Branch-free: an
            // event that does not apply has d = 0 (its cells are clamped into the footprint's range and contribute 0).
            const int64_t minor_stride = IDENT ? (g.steep ? (int64_t)ESZ : pitch) : 0;
            auto fix2 = [&](int mi, int Mi, float d_before, float d_after) {
                const int mlim = (g.steep ? ncols : nrows) - 2, Mlim = (g.steep ? nrows : ncols) - 1;
                mi = max(0, min(mi, mlim));
                Mi = max(0, min(Mi, Mlim));
                const int k = g.steep ? mi : Mi, r = g.steep ? Mi : mi;
                if (GROUPED) {  // corrections go to the weights of the cells' source pixels: no loads here
                    // the two cells are neighbours along the minor axis and share the major index
                    const int k1 = k + (g.steep ? 1 : 0), r1 = r + (g.steep ? 0 : 1);
                    const float both = d_before + d_after;
                    if (g.steep) {  // same row: split by column group, then one row group
                        const float dA = (k < nA ? d_before : 0.0f) + (k1 < nA ? d_after : 0.0f), dB = both - dA;
                        const bool top = r < nT;
                        W00 += top ? dA : 0.0f;
                        W01 += top ? dB : 0.0f;
                        W10 += top ? 0.0f : dA;
                        W11 += top ? 0.0f : dB;
                    } else {  // same column: split by row group, then one column group
                        const float dT = (r < nT ? d_before : 0.0f) + (r1 < nT ? d_after : 0.0f), dBt = both - dT;
                        const bool left = k < nA;
                        W00 += left ? dT : 0.0f;
                        W10 += left ? dBt : 0.0f;
                        W01 += left ? 0.0f : dT;
                        W11 += left ? 0.0f : dBt;
                    }
                    sumA += both;
                    return;
                }
                const char *p0, *p1;
                if (IDENT) {
                    p0 = rowp0 + (int64_t)r * pitch + (int64_t)k * ESZ;
                    p1 = p0 + minor_stride;
                } else {
                    p0 = (const char *)kp.src + row_off(jy0 + r) + col_off(ix0 + k);
                    p1 = (const char *)kp.src + row_off(jy0 + r + (g.steep ? 0 : 1)) + col_off(ix0 + k + (g.steep ? 1 : 0));
                }
                sumA += d_before + d_after;
#pragma unroll
                for (int ch = 0; ch < NC; ++ch) {
                    acc[ch] = fmaf(LoadS<TI, STAGED>::get(p0 + ch * (int)sizeof(TI)), d_before, acc[ch]);
                    acc[ch] = fmaf(LoadS<TI, STAGED>::get(p1 + ch * (int)sizeof(TI)), d_after, acc[ch]);
                }
            };
            for (int q = 0; q < g.ncross; ++q) {  // both left/right edges per packed instruction
                int mi[2], Mi[2];
                float db[2], da[2];
                aai_edge_quirk_pair_f32(g, g0m, g0M, q, mi, Mi, db, da, worst);
                fix2(mi[0], Mi[0], db[0], da[0]);
                fix2(mi[1], Mi[1], db[1], da[1]);
            }

        }
        if (GROUPED) {  // the (at most) four source pixels, once each
            const int64_t roff0 = row_off(jy0), roffL = row_off(jy1), coff0 = col_off(ix0), coffL = col_off(ix1);
            const char *base = (const char *)kp.src;
            const char *p00 = base + roff0 + coff0, *p01 = base + roff0 + coffL;
            const char *p10 = base + roffL + coff0, *p11 = base + roffL + coffL;
#pragma unroll
            for (int ch = 0; ch < NC; ++ch) {
                const int o = ch * (int)sizeof(TI);
                acc[ch] = fmaf(LoadS<TI, STAGED>::get(p00 + o), W00,
                               fmaf(LoadS<TI, STAGED>::get(p01 + o), W01,
                                    fmaf(LoadS<TI, STAGED>::get(p10 + o), W10, LoadS<TI, STAGED>::get(p11 + o) * W11)));
            }
        }
        // guard band of the quirk decision -> FP64
        redo = worst < g.tau || sumA < 0.25f;
    }
    // rare path, warp-cooperative: the flagged pixels of this warp one after the other, one CELL per lane
    double s64 = 0.0, a64[NC];
    if (__any_sync(0xffffffffu, redo)) warp_pixels_f64<TI, NC>(kp, redo, x, y, s64, a64);
    if (redo) {
        const bool ok = DBL_EPSILON < fabs(s64);
#pragma unroll
        for (int ch = 0; ch < NC; ++ch) store_dst<TO>(drow, x * NC + ch, ok ? a64[ch] / s64 : 0.0);
    } else if (work) {
        const float inv = 1.0f / sumA;
#pragma unroll
        for (int ch = 0; ch < NC; ++ch) store_f<TO>(drow, x * NC + ch, acc[ch] * inv);
    }
}

template <typename TI, typename TO, int NC, int ADDR, bool PDL = false, bool REV = false, bool WIN = false>
__global__ void __launch_bounds__(TILE_W *TILE_H, AAI_F32_MIN_BLOCKS)
    overlap_kernel_f32(const __grid_constant__ AaiKernelParams kp) {
    overlap_body<TI, TO, NC, ADDR, false, PDL, REV, WIN>(kp, nullptr, 0, 0, 0);
}
#ifndef AAI_PDL
#define AAI_PDL 1
#endif
constexpr long long kPdlMaxCtas = 150000;
template <typename TI, typename TO, int NC, bool WIN>
cudaError_t launch_short_pdl(const AaiKernelParams &kp, dim3 grid, dim3 block, cudaStream_t stream) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = 0;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    if (kp.reverse_rows) return cudaLaunchKernelEx(&cfg, overlap_kernel_f32<TI, TO, NC, ADDR_IDENT, true, true, WIN>, kp);
    return cudaLaunchKernelEx(&cfg, overlap_kernel_f32<TI, TO, NC, ADDR_IDENT, true, false, WIN>, kp);
}

// the same kernel with the CTA's source window staged through shared memory by TMA (see "STAGED variants" above)
template <typename TI, typename TO, int NC, bool WIN>
__global__ void __launch_bounds__(TILE_W *TILE_H, AAI_F32_MIN_BLOCKS)
    overlap_kernel_f32_tma(const __grid_constant__ CUtensorMap tmap, const __grid_constant__ AaiKernelParams kp,
                           const StageParams sp) {
    extern __shared__ __align__(128) unsigned char stage_raw[];
    __shared__ uint64_t bar;
    __shared__ int origin[2];
    int sox, soy;
    stage_window<(int)sizeof(TI), NC>(&tmap, kp, sp, stage_raw, &bar, origin, kp.ext32, sox, soy);
    overlap_body<TI, TO, NC, ADDR_IDENT, true, false, false, WIN>(kp, (const char *)stage_raw, sp.bw * (int)sizeof(TI), sox,
                                                             soy);
}

// identity addressing: staged (A/B variant), short launches with PDL, or the whole-canvas kernel
template <typename TI, typename TO, int NC, bool WIN>
cudaError_t launch_ident(const AaiKernelParams &kp, dim3 grid, dim3 block, cudaStream_t stream) {
    StageHost h;
    if (kp.staged == 1 && stage_prepare<TI, NC>(kp, (double)kp.ext32, h)) {
        overlap_kernel_f32_tma<TI, TO, NC, WIN><<<grid, block, h.smem, stream>>>(h.map, kp, h.sp);
        return cudaGetLastError();
    }
    if (AAI_PDL && (long long)grid.x * grid.y * grid.z <= kPdlMaxCtas) return launch_short_pdl<TI, TO, NC, WIN>(kp, grid, block, stream);
    overlap_kernel_f32<TI, TO, NC, ADDR_IDENT, false, false, WIN><<<grid, block, 0, stream>>>(kp);
    return cudaGetLastError();
}

#ifndef AAI_TIP_WINDOW
#define AAI_TIP_WINDOW 1  // 0: every plan takes the full MAXN x MAXN body (A/B builds)
#endif

template <typename TI, typename TO, int NC>
cudaError_t launch3(const AaiKernelParams &kp, cudaStream_t stream) {
    if (kp.row1 <= kp.row0 || kp.dst_w <= 0) return cudaSuccess;
    const dim3 grid = canvas_grid(kp), block(TILE_W, TILE_H);
    if (kp.scale == 1 && kp.quadrant == 0) {
        if constexpr (AAI_TIP_WINDOW && NC == 1) {
            if (kp.tip_window) return launch_ident<TI, TO, NC, true>(kp, grid, block, stream);
        }
        return launch_ident<TI, TO, NC, false>(kp, grid, block, stream);
    } else if (MAXN == 4 && kp.scale >= MAXN - 1)
        overlap_kernel_f32<TI, TO, NC, (MAXN == 4 ? ADDR_GROUPED : ADDR_GENERAL)><<<grid, block, 0, stream>>>(kp);
    else
        overlap_kernel_f32<TI, TO, NC, ADDR_GENERAL><<<grid, block, 0, stream>>>(kp);
    return cudaGetLastError();
}


// ------------------------------------------------------------------------------------------------------------
// Fast mode (fastAreaAverageInterpolation, Source.cpp:866-907), FP32 arithmetic, unrolled: the unweighted mean of the
// expanded pixels whose CENTRE lies in the footprint (closed point-in-square test, 837-864).
//
// HBM-bound by contract (each source byte once + each canvas byte once), so the kernel only has to stay out of the
// way: at most NF = MAXN - 1 lattice points per axis can lie within h(c+s) of the footprint centre, all NF x NF
// candidates are loaded unconditionally up front (independent loads in flight together; the footprints of a warp's
// 16 x 2 canvas pixels overlap, L1 serves most of them) and tested branch-free -- two FFMAs for the footprint-local
// coordinates, margin m = min(h - |u|, h - |v|), predicated adds.  The inside test is a discontinuous decision: as in
// the overlap kernel the centre is split into lattice point + FP32 fraction, the smallest |m| of the pixel is tracked,
// and a pixel with a margin inside the guard band -- or whose candidate box the image border clips -- is redone in FP64
// (pixel_fast_f64, the reference's own centre expression).
// ------------------------------------------------------------------------------------------------------------
constexpr int NF = MAXN - 1;
#ifndef AAI_FAST_VEC_LOADS
#define AAI_FAST_VEC_LOADS 1  // float, 1 channel, identity addressing: 128-bit loads (0: scalar loads; A/B in profiles/)
#endif
#ifndef AAI_FAST_PRED_LOADS
#define AAI_FAST_PRED_LOADS 1  // multi-channel images: load only the inside cells (0: always load all candidates up front)
#endif
#ifndef AAI_FAST_SKIP_LOADS
#define AAI_FAST_SKIP_LOADS 1  // 128-bit-load kernel: do not request rows / vectors beyond the last lattice row / column of the box
#endif
// VEC (float images, one channel, identity addressing, 16-byte aligned rows): the NF candidates of a row are read as
// aligned 128-bit vectors (the 4 NV floats from the 16-byte boundary below the first candidate) and shifted into place
// with selects -- 8 instead of 16 loads per pixel.  A rotated warp-wide load touches one 32-byte sector per lane whatever
// its width, and the L1 tag stage is what bounds this kernel (l1tex 77 % with scalar loads).
template <typename TI, typename TO, int NC, bool IDENT, bool STAGED, bool VEC = false>
__device__ __forceinline__ void fast_body(const AaiKernelParams &kp, const char *stage, int spitch, int sox, int soy,
                                          int tile_x, int tile_y) {
    static_assert(!STAGED || IDENT, "staging is implemented for identity addressing");
    static_assert(!VEC || (IDENT && !STAGED && NC == 1 && sizeof(TI) == 4), "vector loads: float, 1 channel, identity");
    constexpr int NV = (NF + 3 + 3) / 4;  // aligned float4 vectors that cover NF floats from any offset 0..3
    const int x = tile_x * TILE_W + threadIdx.x;
    const int y = kp.row0 + tile_y * TILE_H + threadIdx.y;
    if (x >= kp.dst_w || y >= kp.row1) return;
    const double cx = fma((double)x, kp.aff_xx, fma((double)y, kp.aff_xy, kp.aff_x0));
    const double cy = fma((double)x, kp.aff_yx, fma((double)y, kp.aff_yy, kp.aff_y0));
    const int irx = __double2int_rn(cx), iry = __double2int_rn(cy);
    const float fx = (float)(cx - (double)irx), fy = (float)(cy - (double)iry);
    const AaiShapeF &g = kp.shapef;
    constexpr float tau = 4e-6f;
    // lattice points whose centre can lie in the footprint: |i - cx| <= h(c+s) (FP32 with a safety margin)
    const float ext = g.hb + tau;
    const int bx0 = irx + __float2int_ru(fx - ext), bx1 = irx + __float2int_rd(fx + ext);
    const int by0 = iry + __float2int_ru(fy - ext), by1 = iry + __float2int_rd(fy + ext);
    char *drow = (char *)kp.dst + (int64_t)(y - dst_row0(kp)) * kp.dst_pitch;
    if (bx1 < 0 || by1 < 0 || bx0 > kp.mod_w - 1 || by0 > kp.mod_h - 1) {  // no candidate in the image: count 0 -> 0
#pragma unroll
        for (int ch = 0; ch < NC; ++ch) store_f<TO>(drow, x * NC + ch, 0.0f);
        return;
    }
    // the unrolled NF x NF block starts at (bx0, by0); it must lie inside the image (else: FP64 path below)
    // (VEC: the aligned vectors must end inside the row as well)
    const bool inside_img = bx0 >= 0 && by0 >= 0 && bx0 + NF - 1 <= kp.mod_w - 1 && by0 + NF - 1 <= kp.mod_h - 1 &&
                            bx1 - bx0 < NF && by1 - by0 < NF && (!VEC || (bx0 & ~3) + 4 * NV <= kp.mod_w);
    float count = 0.0f, acc[NC], worst = 1.0f;
#pragma unroll
    for (int ch = 0; ch < NC; ++ch) acc[ch] = 0.0f;
    if (inside_img) {
        constexpr int ESZ = (int)sizeof(TI) * NC;
        const bool swapped = kp.e_axi == 0;
        auto div_s = [&](int e) -> int64_t {
            return (int64_t)(kp.scale != 1 ? __umulhi((unsigned)e, kp.div_magic) : (unsigned)e);
        };
        int64_t coff[NF], roff[NF];
        if (STAGED) {  // offsets inside the CTA's shared-memory window
#pragma unroll
            for (int k = 0; k < NF; ++k) {
                coff[k] = ((bx0 + k) * NC - sox) * (int)sizeof(TI);
                roff[k] = (by0 + k - soy) * spitch;
            }
        } else if (IDENT) {
#pragma unroll
            for (int k = 0; k < NF; ++k) {
                coff[k] = (int64_t)(bx0 + k) * ESZ;
                roff[k] = (int64_t)(by0 + k - src_row0(kp)) * kp.src_pitch;
            }
        } else {
#pragma unroll
            for (int k = 0; k < NF; ++k) {
                const int i = bx0 + k, j = by0 + k;
                coff[k] = swapped ? (div_s(kp.e_ayi * i + kp.e_ay0) - src_row0(kp)) * kp.src_pitch
                                  : div_s(kp.e_axi * i + kp.e_ax0) * ESZ;
                roff[k] = swapped ? div_s(kp.e_axj * j + kp.e_ax0) * ESZ
                                  : (div_s(kp.e_ayj * j + kp.e_ay0) - src_row0(kp)) * kp.src_pitch;
            }
        }
        const float rx0 = (float)(bx0 - irx) - fx, ry0 = (float)(by0 - iry) - fy;
        if constexpr (VEC) {
            const int o = bx0 & 3;
            const char *rowp = (const char *)kp.src + (int64_t)(by0 - src_row0(kp)) * kp.src_pitch + (int64_t)(bx0 - o) * 4;
            float v[NF][NF];
            // the lattice points of the box are columns bx0 .. bx1 and rows by0 .. by1 (often one fewer than NF): vectors
            // and rows beyond them hold no inside cell and are not requested -- the kernel is bound by the L1 tag stage, and
            // the predicates are known before the first load (config 4: 5.4 instead of 8 requests per pixel, 0.588 -> 0.540 ms;
            // the scalar-load kernel of 8-bit images does not gain from the same predicates: config 2 17 -> 19 us)
            const int last_col = o + (bx1 - bx0), last_row = by1 - by0;
#pragma unroll
            for (int r = 0; r < NF; ++r) {  // all vector loads first: up to NF * NV independent 128-bit loads in flight
                float w[4 * NV];
#pragma unroll
                for (int q = 0; q < NV; ++q) {
                    const bool need = AAI_FAST_SKIP_LOADS ? (r <= last_row && 4 * q <= last_col) : true;
                    const float4 t = need ? __ldg(reinterpret_cast<const float4 *>(rowp) + q) : make_float4(0.f, 0.f, 0.f, 0.f);
                    w[4 * q] = t.x;
                    w[4 * q + 1] = t.y;
                    w[4 * q + 2] = t.z;
                    w[4 * q + 3] = t.w;
                }
                rowp += kp.src_pitch;
                // shift by o = 0..3 in two select stages (o & 1, then o & 2)
                float t1[NF + 2];
#pragma unroll
                for (int i = 0; i < NF + 2; ++i) t1[i] = (o & 1) ? w[i + 1] : w[i];
#pragma unroll
                for (int k = 0; k < NF; ++k) v[r][k] = (o & 2) ? t1[k + 2] : t1[k];
            }
#pragma unroll
            for (int r = 0; r < NF; ++r) {
                const float ry = ry0 + (float)r;
                const float2 uvr = make_float2(-ry * g.sn, ry * g.cs), cssn = make_float2(g.cs, g.sn);
#pragma unroll
                for (int k = 0; k < NF; ++k) {
                    const float rx = rx0 + (float)k;
                    // (u, v) in one packed FFMA2; min(h - |u|, h - |v|) = h - max(|u|, |v|) exactly (same subtraction)
                    const float2 uv = __ffma2_rn(make_float2(rx, rx), cssn, uvr);
                    const float m = g.half - fmaxf(fabsf(uv.x), fabsf(uv.y));
                    worst = fminf(worst, fabsf(m));
                    if (m >= 0.0f) {  // closed point-in-square (837-864); predicated adds, no branch
                        count += 1.0f;
                        acc[0] += v[r][k];
                    }
                }
            }
        } else
        // Single channel: all NF x NF candidates are loaded up front (loads in flight while the margins are computed).
        // Several channels: margins of all candidates first, then ONLY the inside cells are loaded (predicated LDG; less
        // than half of the candidates lie inside, and three loads per candidate weigh more than their latency).  Measured
        // (profiles/r2_n_fast_ab.txt): config 4 (1 channel) 0.615 ms up front vs 0.697 ms predicated; config 3 (RGB)
        // 3.73 ms up front vs 3.21 ms predicated.
        if constexpr (AAI_FAST_PRED_LOADS && NC > 1) {
        float mm[NF][NF];
#pragma unroll
        for (int r = 0; r < NF; ++r) {
            const float ry = ry0 + (float)r;
            const float ur = -ry * g.sn, vr = ry * g.cs;
#pragma unroll
            for (int k = 0; k < NF; ++k) {
                const float rx = rx0 + (float)k;
                const float mu = g.half - fabsf(fmaf(rx, g.cs, ur));
                const float mv = g.half - fabsf(fmaf(rx, g.sn, vr));
                const float m = fminf(mu, mv);
                worst = fminf(worst, fabsf(m));
                mm[r][k] = m;
            }
        }
#pragma unroll
        for (int r = 0; r < NF; ++r) {
            const char *rowp = (STAGED ? stage : (const char *)kp.src) + roff[r];
#pragma unroll
            for (int k = 0; k < NF; ++k) {
                if (mm[r][k] >= 0.0f) {  // closed point-in-square (837-864)
                    count += 1.0f;
#pragma unroll
                    for (int ch = 0; ch < NC; ++ch)
                        acc[ch] += LoadS<TI, STAGED>::get(rowp + coff[k] + ch * (int)sizeof(TI));
                }
            }
        }
        } else {
#pragma unroll
        for (int r = 0; r < NF; ++r) {
            float v[NF][NC];
            const char *rowp = (STAGED ? stage : (const char *)kp.src) + roff[r];
#pragma unroll
            for (int k = 0; k < NF; ++k)
#pragma unroll
                for (int ch = 0; ch < NC; ++ch) v[k][ch] = LoadS<TI, STAGED>::get(rowp + coff[k] + ch * (int)sizeof(TI));
            const float ry = ry0 + (float)r;
            const float ur = -ry * g.sn, vr = ry * g.cs;
#pragma unroll
            for (int k = 0; k < NF; ++k) {
                const float rx = rx0 + (float)k;
                const float mu = g.half - fabsf(fmaf(rx, g.cs, ur));
                const float mv = g.half - fabsf(fmaf(rx, g.sn, vr));
                const float m = fminf(mu, mv);
                worst = fminf(worst, fabsf(m));
                if (m >= 0.0f) {  // closed point-in-square (837-864); predicated adds, no branch
                    count += 1.0f;
#pragma unroll
                    for (int ch = 0; ch < NC; ++ch) acc[ch] += v[k][ch];
                }
            }
        }
        }
    }
    if (!inside_img || worst < tau) {  // border pixel, or a centre within the guard band of a footprint edge: FP64 decides
        int c64;
        double a64[NC];
        pixel_fast_f64<TI, NC>(kp, x, y, c64, a64);
#pragma unroll
        for (int ch = 0; ch < NC; ++ch) store_dst<TO>(drow, x * NC + ch, c64 > 0 ? a64[ch] / (double)c64 : 0.0);
    } else {
        const float inv = count > 0.0f ? 1.0f / count : 0.0f;
#pragma unroll
        for (int ch = 0; ch < NC; ++ch) store_f<TO>(drow, x * NC + ch, acc[ch] * inv);
    }
}

template <typename TI, typename TO, int NC, bool IDENT>
__global__ void __launch_bounds__(TILE_W *TILE_H, 1024 / (TILE_W * TILE_H))
    fast_kernel_f32u(const __grid_constant__ AaiKernelParams kp) {
    fast_body<TI, TO, NC, IDENT, false>(kp, nullptr, 0, 0, 0, blockIdx.x, blockIdx.y);
}
// float images, one channel, identity addressing, 16-byte aligned rows: 128-bit loads (see fast_body)
template <typename TO>
__global__ void __launch_bounds__(TILE_W *TILE_H, 1024 / (TILE_W * TILE_H))
    fast_kernel_f32u_vec(const __grid_constant__ AaiKernelParams kp) {
    fast_body<float, TO, 1, true, false, true>(kp, nullptr, 0, 0, 0, blockIdx.x, blockIdx.y);
}

// the same kernel with the CTA's source window staged through shared memory by TMA (AAI_ARITH_F32_STAGED).  Measured on
// BASELINE config 4: 0.658 ms against 0.616 ms for the LDG kernel -- the L1 tag stage is relieved (77 % -> 42 %), but every
// CTA now waits for its own TMA load before its ~250 instructions per thread (stalls: long_scoreboard 36 %, barrier 17 %)
template <typename TI, typename TO, int NC>
__global__ void __launch_bounds__(TILE_W *TILE_H, 1024 / (TILE_W * TILE_H))
    fast_kernel_f32u_tma(const __grid_constant__ CUtensorMap tmap, const __grid_constant__ AaiKernelParams kp,
                         const StageParams sp) {
    extern __shared__ __align__(128) unsigned char stage_raw[];
    __shared__ uint64_t bar;
    __shared__ int origin[2];
    int sox, soy;
    stage_window<(int)sizeof(TI), NC>(&tmap, kp, sp, stage_raw, &bar, origin, kp.shapef.hb + 4e-6f, sox, soy);
    fast_body<TI, TO, NC, true, true>(kp, (const char *)stage_raw, sp.bw * (int)sizeof(TI), sox, soy, blockIdx.x, blockIdx.y);
}

// The staged kernel made PERSISTENT (AAI_ARITH_F32_RING): a CTA walks over the canvas tiles blockIdx.x, + gridDim.x, ...
// with TWO window buffers -- while the 128 threads evaluate tile k out of one buffer, the TMA load of tile k + 1 is in
// flight into the other (one elected thread computes the next window origin and issues it; completion on one mbarrier per
// buffer, phase = use count).  That removes what sank the one-shot staged kernel (every CTA waiting for its own load in
// front of ~250 instructions per thread) and keeps its relief of the L1 tag stage (LDS instead of rotated LDGs).
constexpr int RING_STAGES = 2;
template <typename TI, typename TO, int NC>
__global__ void __launch_bounds__(TILE_W *TILE_H, 1024 / (TILE_W * TILE_H))
    fast_kernel_f32u_ring(const __grid_constant__ CUtensorMap tmap, const __grid_constant__ AaiKernelParams kp,
                          const StageParams sp, const int tiles_x, const int ntiles) {
    extern __shared__ __align__(128) unsigned char stage_raw[];
    __shared__ uint64_t full[RING_STAGES];
    __shared__ int origin[RING_STAGES][2];
    constexpr int EB = (int)sizeof(TI), EAL = 16 / EB;
    const int tid = threadIdx.y * TILE_W + threadIdx.x;
    const uint32_t stage_bytes = (uint32_t)(sp.bw * sp.bh * EB);
    const uint32_t stage_stride = (stage_bytes + 127u) & ~127u;
    const float ext = kp.shapef.hb + 4e-6f;
    auto issue = [&](int t, int s) {  // one thread: window origin of tile t (FP64, extremes at the tile's corners), TMA
        const int ty = t / tiles_x, tx = t - ty * tiles_x;
        const int x0 = tx * TILE_W, y0 = kp.row0 + ty * TILE_H;
        double lox = 1e300, loy = 1e300;
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            const double xx = (double)(x0 + (c & 1) * (TILE_W - 1)), yy = (double)(y0 + (c >> 1) * (TILE_H - 1));
            lox = fmin(lox, fma(xx, kp.aff_xx, fma(yy, kp.aff_xy, kp.aff_x0)));
            loy = fmin(loy, fma(xx, kp.aff_yx, fma(yy, kp.aff_yy, kp.aff_y0)));
        }
        int ex = (__double2int_rd(lox - (double)ext) - 1) * NC;
        ex = (ex >= 0 ? ex / EAL : -((-ex + EAL - 1) / EAL)) * EAL;
        const int ey = __double2int_rd(loy - (double)ext) - 1;
        origin[s][0] = ex;
        origin[s][1] = ey;
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(st_smem_u32(&full[s])), "r"(stage_bytes)
                     : "memory");
        asm volatile(
            "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::
                "r"(st_smem_u32(stage_raw + (size_t)s * stage_stride)),
            "l"(&tmap), "r"(st_smem_u32(&full[s])), "r"(ex), "r"(ey - src_row0(kp))
            : "memory");
    };
    if (tid == 0) {
#pragma unroll
        for (int s = 0; s < RING_STAGES; ++s)
            asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(st_smem_u32(&full[s])), "r"(1));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        if ((int)blockIdx.x < ntiles) issue((int)blockIdx.x, 0);
    }
    int k = 0;
    for (int t = (int)blockIdx.x; t < ntiles; t += (int)gridDim.x, ++k) {
        const int s = k & 1;
        __syncthreads();  // every thread is done with the other buffer (tile k - 1); origin[s] of this tile is visible
        if (tid == 0 && t + (int)gridDim.x < ntiles) issue(t + (int)gridDim.x, s ^ 1);
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "RG_WAIT:\n"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
            "@p bra.uni RG_DONE;\n"
            "bra.uni RG_WAIT;\n"
            "RG_DONE:\n"
            "}\n" ::"r"(st_smem_u32(&full[s])),
            "r"((k >> 1) & 1)
            : "memory");
        const int ty = t / tiles_x, tx = t - ty * tiles_x;
        fast_body<TI, TO, NC, true, true>(kp, (const char *)stage_raw + (size_t)s * stage_stride, sp.bw * EB, origin[s][0],
                                          origin[s][1], tx, ty);
    }
}

template <typename TI, typename TO, int NC>
cudaError_t launch_fast3(const AaiKernelParams &kp, cudaStream_t stream) {
    if (kp.row1 <= kp.row0 || kp.dst_w <= 0) return cudaSuccess;
    const dim3 grid = canvas_grid(kp), block(TILE_W, TILE_H);
    if (kp.scale == 1 && kp.quadrant == 0) {
        StageHost h;
        if ((kp.staged == 1 || kp.staged == 3) && stage_prepare<TI, NC>(kp, (double)kp.shapef.hb + 1e-5, h)) {
            if (kp.staged == 3) {  // AAI_ARITH_F32_RING: persistent CTAs, two window buffers
                int dev = 0, sms = 0;
                cudaGetDevice(&dev);
                cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
                const int tiles_x = (int)grid.x, ntiles = (int)(grid.x * grid.y);
                const size_t smem = RING_STAGES * ((h.smem + 127) & ~(size_t)127);
                const int per_sm = 1024 / (TILE_W * TILE_H);
                const dim3 pgrid((unsigned)std::min(ntiles, sms * per_sm), 1, grid.z);
                static thread_local int attr_dev = -1;  // two buffers of a wide window exceed the 48 KB default
                if (attr_dev != dev) {
                    const cudaError_t e = cudaFuncSetAttribute(fast_kernel_f32u_ring<TI, TO, NC>,
                                                               cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024);
                    if (e != cudaSuccess) return e;
                    attr_dev = dev;
                }
                fast_kernel_f32u_ring<TI, TO, NC><<<pgrid, block, smem, stream>>>(h.map, kp, h.sp, tiles_x, ntiles);
                return cudaGetLastError();
            }
            fast_kernel_f32u_tma<TI, TO, NC><<<grid, block, h.smem, stream>>>(h.map, kp, h.sp);  // AAI_ARITH_F32_STAGED
            return cudaGetLastError();
        }
        if constexpr (sizeof(TI) == 4 && NC == 1) {
            if ((kp.src_pitch % 16) == 0 && (reinterpret_cast<uintptr_t>(kp.src) % 16) == 0 && AAI_FAST_VEC_LOADS) {
                fast_kernel_f32u_vec<TO><<<grid, block, 0, stream>>>(kp);
                return cudaGetLastError();
            }
        }
        fast_kernel_f32u<TI, TO, NC, true><<<grid, block, 0, stream>>>(kp);
    } else {
        fast_kernel_f32u<TI, TO, NC, false><<<grid, block, 0, stream>>>(kp);
    }
    return cudaGetLastError();
}

}  // namespace

#define AAI_CAT2(a, b) a##b
#define AAI_CAT(a, b) AAI_CAT2(a, b)

int AAI_CAT(aai_launch_overlap_f32_n, AAI_MAXN)(const AaiKernelParams &kp, int src_dtype, int dst_dtype, void *stream) {
    return (int)with_pair<AnyElem, AnyElem>(src_dtype, dst_dtype, cudaErrorInvalidValue, [&](auto ti, auto to) {
        using TI = typename decltype(ti)::type;
        using TO = typename decltype(to)::type;
        return with_channels<1, 3>(kp.channels, cudaErrorInvalidValue, [&](auto nc) {
            return launch3<TI, TO, decltype(nc)::value>(kp, (cudaStream_t)stream);
        });
    });
}

// fast mode, FP32 arithmetic: float / 8-bit / 16-bit sources, float or integer destinations (double destinations take
// the FP64 fast kernel), 1 or 3 channels
int AAI_CAT(aai_launch_fast_f32_n, AAI_MAXN)(const AaiKernelParams &kp, int src_dtype, int dst_dtype, void *stream) {
    return (int)with_pair<NarrowElem, NarrowElem>(src_dtype, dst_dtype, cudaErrorInvalidValue, [&](auto ti, auto to) {
        using TI = typename decltype(ti)::type;
        using TO = typename decltype(to)::type;
        return with_channels<1, 3>(kp.channels, cudaErrorInvalidValue, [&](auto nc) {
            return launch_fast3<TI, TO, decltype(nc)::value>(kp, (cudaStream_t)stream);
        });
    });
}
