// Separable kernel for axis-aligned reduced angles (0/90/180/270 degrees): the main loop of
// AreaAverageInterpolation::areaAverageInterpolation (Source.cpp:411-579) when every footprint is an axis-aligned
// square, so that the overlap area factorises, A_ij = wx(i) * wy(j) (SURVEY.md §7.6, DESIGN.md §3.5), and
//     dst = sum_j wy(j) sum_i wx(i) src[j][i] / (sum wx * sum wy)        (sums over in-image cells, Source.cpp:577).
//
// HBM-bound by contract (each source byte read once, each canvas byte written once).  One CTA = one canvas tile
// TW x TH.  Its source window is staged into shared memory by ONE 2-D TMA tile load (cp.async.bulk.tensor.2d through
// a CUtensorMap, completion on an mbarrier; out-of-image parts of the box are zero-filled by the hardware and carry
// weight 0).  The two banded 1-D passes run out of that tile with the intermediate in registers: for every canvas pixel
// the horizontal taps of each of its source rows (weights in registers, taps read as aligned vectors so that the
// stride-L accesses of a warp do not collide on shared-memory banks), then the vertical taps (weights broadcast from
// shared memory), then the coalesced store.  (A first version wrote the horizontal pass to a shared-memory tile and
// synchronised: 3x the instructions, issue-bound at 64 %; see profiles/.)  Several CTAs are resident per SM, so one
// CTA's TMA load overlaps the other CTAs' arithmetic.
//
// A batch of equally strided images is ONE launch: the tensor map is rank 3 (x, y, image), blockIdx.y = image.
//
// Fast path preconditions (checked by the host launcher, otherwise the direct-tap kernel in aai_kernels.cu runs):
// scale 1, quadrant 0, one channel, 16-byte aligned rows, footprint side small enough for a <=256-wide TMA box.
// TMA tile coordinates must be 16-byte aligned in the innermost dimension: the window origin is rounded down.
#include <cuda.h>

#include <atomic>
#include <cstdio>
#include <cstdlib>
#include <type_traits>

#include "aai_device.cuh"

using namespace aai_dev;

namespace {

constexpr int SEP_THREADS = 256;   // consumer threads (canvas pixels); one more warp produces (TMA + row weights)
constexpr int SEP_BLOCK = SEP_THREADS + 32;

struct SepParams {
    int tw, th;  // canvas tile
    int bw, bh;  // TMA box = source window of one tile (elements, rows)
    int tiles_x, tiles_y;
    int tiles_per_cta;  // consecutive tile rows one CTA walks through
    int stages;         // source windows in the shared-memory ring (stages - 1 loads in flight while one is evaluated)
};

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra.uni WAIT_DONE;\n"
        "bra.uni WAIT_LOOP;\n"
        "WAIT_DONE:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
// (x, y, image) box of a rank-3 tensor map: a batch of equally strided images is one tensor
__device__ __forceinline__ void tma_load_3d(void *dst, const CUtensorMap *map, uint64_t *bar, int c0, int c1, int c2) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::
            "r"(smem_u32(dst)),
        "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
        : "memory");
}

template <typename TA>
__device__ __forceinline__ TA sat01(TA x) {
    return x < (TA)0 ? (TA)0 : (x > (TA)1 ? (TA)1 : x);
}
template <>
__device__ __forceinline__ float sat01<float>(float x) {
    return __saturatef(x);
}

// taps of one canvas coordinate: cells [first, first+MAXT) around the footprint interval [c-h, c+h], weight of tap t =
// |[first+t-1/2, first+t+1/2] ∩ [c-h, c+h]| for in-image cells, 0 otherwise
template <typename TA, int MAXT>
__device__ __forceinline__ void axis_taps(double c, double h, int limit, int &first, TA (&w)[MAXT], TA &sum) {
    first = __double2int_rd(c - h - 0.5) + 1;
    const double e = (double)first - 0.5;
    const TA lo = (TA)((c - h) - e), hi = (TA)((c + h) - e);
    sum = (TA)0;
#pragma unroll
    for (int t = 0; t < MAXT; ++t) {
        TA v = sat01<TA>(hi - (TA)t) - sat01<TA>(lo - (TA)t);
        const int i = first + t;
        v = (i >= 0 && i < limit) ? v : (TA)0;
        w[t] = v;
        sum += v;
    }
}

// aligned vector of source elements in shared memory: 8 bytes for 4-byte elements, otherwise one element
template <typename TI>
struct TapVec {
    static constexpr int N = 1;
    static __device__ __forceinline__ void load(const TI *p, TI (&v)[1]) { v[0] = *p; }
};
template <>
struct TapVec<float> {
    static constexpr int N = 2;
    static __device__ __forceinline__ void load(const float *p, float (&v)[2]) {
        const float2 t = *reinterpret_cast<const float2 *>(p);
        v[0] = t.x;
        v[1] = t.y;
    }
};

template <typename TA, int MAXT>
__host__ __device__ constexpr size_t sep_weight_bytes(int th) {
    return ((size_t)th * ((MAXT + 1 + 3) / 4 * 4) * sizeof(TA) + (size_t)th * sizeof(int) + 15) / 16 * 16;
}

template <typename TA>
__device__ __forceinline__ TA sep_normalise(TA acc, TA total) {  // Source.cpp:577
    return ((double)total > DBL_EPSILON) ? acc / total : (TA)0;
}
template <>
__device__ __forceinline__ float sep_normalise<float>(float acc, float total) {
    const float q = __fdividef(acc, total);  // branch-free (<= 2 ulp); the select discards inf/NaN of an empty footprint
    return total > (float)DBL_EPSILON ? q : 0.0f;
}

// per-canvas-row record in shared memory: MAXT vertical weights followed by their sum, padded to a multiple of four
// elements so that a float record is read with 16-byte loads
template <typename TA, int N>
__device__ __forceinline__ void load_record(const TA *rec, TA (&w)[N]) {
#pragma unroll
    for (int k = 0; k < N; ++k) w[k] = rec[k];
}
template <int N>
__device__ __forceinline__ void load_record(const float *rec, float (&w)[N]) {
#pragma unroll
    for (int k = 0; k < N; k += 4) {
        const float4 t = *reinterpret_cast<const float4 *>(rec + k);
        w[k] = t.x;
        if (k + 1 < N) w[k + 1] = t.y;
        if (k + 2 < N) w[k + 2] = t.z;
        if (k + 3 < N) w[k + 3] = t.w;
    }
}

// One CTA walks DOWN a strip of canvas tiles (same canvas columns, consecutive tile rows): the column weights and
// their vector layout are computed once per CTA; the source windows go through a ring of shared-memory buffers that a
// dedicated producer warp keeps full (TMA load of tile t+S-1 and its row weights while the eight consumer warps
// evaluate tile t), so HBM never waits for the arithmetic and no consumer warp carries the FP64 weight set-up.
template <typename TI, typename TO, typename TA, int TW, int MAXT>
__global__ void __launch_bounds__(SEP_BLOCK)
    separable_tma_kernel(const __grid_constant__ CUtensorMap tmap, const __grid_constant__ AaiKernelParams kp,
                         const SepParams sp) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    constexpr int RG = SEP_THREADS / TW;  // row groups
    constexpr int VEC = TapVec<TI>::N;
    constexpr int NV = (MAXT + 2 * (VEC - 1)) / VEC;  // aligned vectors that cover MAXT taps from any start offset
    constexpr int RS = (MAXT + 1 + 3) / 4 * 4;  // record stride (elements)
    const size_t tile_bytes = ((size_t)sp.bw * sp.bh * sizeof(TI) + 127) / 128 * 128;
    const size_t wgt_bytes = sep_weight_bytes<TA, MAXT>(sp.th);
    // layout: tile[stages], weights[stages] (records [th][RS], then element offsets [th]), barriers[stages]
    const int S = sp.stages;
    unsigned char *wgt_raw = smem_raw + (size_t)S * tile_bytes;
    uint64_t *bar = reinterpret_cast<uint64_t *>(wgt_raw + (size_t)S * wgt_bytes);

    const int tid = threadIdx.x;
    const int tx = blockIdx.x % sp.tiles_x, seg = blockIdx.x / sp.tiles_x;
    const int ty0 = seg * sp.tiles_per_cta, ntile = min(sp.tiles_per_cta, sp.tiles_y - ty0);
    const int x0 = tx * TW;
    const double h = kp.shape.half;

    // source window origin of tile row t of this strip (expanded frame == source frame on this path).
    // TMA needs the box to start on a 16-byte boundary of the innermost dimension (measured on B200: a misaligned
    // start coordinate raises cudaErrorIllegalInstruction), so the window's x origin is rounded down to ALIGN elements
    constexpr int ALIGN = 16 / (int)sizeof(TI);
    double c0x, c0y;
    pixel_centre(kp, x0, kp.row0 + ty0 * sp.th, c0x, c0y);
    const int ox_raw = __double2int_rd(c0x - h - 0.5);
    const int ox = (ox_raw >= 0 ? ox_raw / ALIGN : -((-ox_raw + ALIGN - 1) / ALIGN)) * ALIGN;
    auto origin_y = [&](int t) {
        double ax, ay;
        pixel_centre(kp, x0, kp.row0 + (ty0 + t) * sp.th, ax, ay);
        return __double2int_rd(ay - h - 0.5);
    };
    auto issue = [&](int t) {  // one thread: TMA load of tile t's window into buffer t % S
        uint64_t *bb = bar + (t % S);
        mbar_expect_tx(bb, (uint32_t)(sp.bw * sp.bh * sizeof(TI)));
        tma_load_3d(smem_raw + (size_t)(t % S) * tile_bytes, &tmap, bb, ox, origin_y(t) - kp.src_y0, (int)blockIdx.y);
    };
    auto row_weights = [&](int t, int lane) {  // producer warp: vertical taps of tile t's canvas rows into weights[t % S]
        TA *rec = reinterpret_cast<TA *>(wgt_raw + (size_t)(t % S) * wgt_bytes);  // [th][RS]: weights, sum
        int *off = reinterpret_cast<int *>(rec + (size_t)sp.th * RS);               // [th] element offset of the first row
        const int oy = origin_y(t);
        for (int r = lane; r < sp.th; r += 32) {
            const int y = kp.row0 + (ty0 + t) * sp.th + r;
            TA w[MAXT], sy = (TA)0;
            int first = oy;
            if (y < kp.row1) {
                double cx, cy;
                pixel_centre(kp, x0, y, cx, cy);
                axis_taps<TA, MAXT>(cy, h, kp.mod_h, first, w, sy);
            } else {
#pragma unroll
                for (int k = 0; k < MAXT; ++k) w[k] = (TA)0;
            }
#pragma unroll
            for (int k = 0; k < MAXT; ++k) rec[r * RS + k] = w[k];
            rec[r * RS + MAXT] = sy;
            // clamp the tap rows into the box (rows beyond it have weight 0 by construction of the box size)
            off[r] = max(0, min(first - oy, sp.bh - MAXT)) * sp.bw;
        }
    };
    const bool producer = tid >= SEP_THREADS;
    const int lane = tid & 31;

    if (tid == 0) {
        for (int k = 0; k < S; ++k) mbar_init(bar + k, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (producer) {
        for (int t = 0; t < S - 1 && t < ntile; ++t) {
            if (lane == 0) issue(t);
            row_weights(t, lane);
        }
    }

    // per-column weights (registers), once per strip, while the first load is in flight
    const int xo = tid % TW, rg = tid / TW;
    const int x = x0 + xo;
    int cfirst = 0;
    TA wx[MAXT], sumx = (TA)0;
    if (!producer && x < kp.dst_w) {
        double cx, cy;
        pixel_centre(kp, x, kp.row0, cx, cy);
        axis_taps<TA, MAXT>(cx, h, kp.mod_w, cfirst, wx, sumx);
        cfirst -= ox;
    } else {
#pragma unroll
        for (int t = 0; t < MAXT; ++t) wx[t] = (TA)0;
    }
    // clamp the tap window into the box (taps beyond it have weight 0 by construction of the box size), then widen it
    // to whole aligned vectors: weights wv[] = wx[] shifted by the start offset inside the first vector, zero elsewhere
    cfirst = max(0, min(cfirst, sp.bw - MAXT - 2 * (VEC - 1)));
    const int cbase = cfirst / VEC * VEC, shift = cfirst - cbase;
    TA wv[NV * VEC];
#pragma unroll
    for (int q = 0; q < NV * VEC; ++q) {
        TA v = (TA)0;
#pragma unroll
        for (int t = 0; t < MAXT; ++t) v = (q - shift == t) ? wx[t] : v;
        wv[q] = v;
    }
    __syncthreads();  // row weights of the first tiles visible

    for (int t = 0; t < ntile; ++t) {
        if (producer) {
            // tile t+S-1: load + row weights (its buffers were last read in iteration t-1, which ended with a barrier)
            if (t + S - 1 < ntile) {
                if (lane == 0) issue(t + S - 1);
                row_weights(t + S - 1, lane);
            }
            __syncthreads();
            continue;
        }
        const int b = t % S;
        const TI *tile = reinterpret_cast<const TI *>(smem_raw + (size_t)b * tile_bytes) + cbase;
        const TA *rec = reinterpret_cast<const TA *>(wgt_raw + (size_t)b * wgt_bytes);
        const int *off = reinterpret_cast<const int *>(rec + (size_t)sp.th * RS);
        const int y0 = kp.row0 + (ty0 + t) * sp.th;
        const int ylim = min(sp.th, kp.row1 - y0);  // canvas rows of this tile that exist
        mbar_wait(bar + b, (uint32_t)((t / S) & 1));
        if (x < kp.dst_w) {
            // U independent canvas rows at a time, stage by stage, so that the shared-memory loads of U pixels are in
            // flight together (one dependent chain per pixel is latency-bound: few resident warps per SM)
            constexpr int U = 4;
            char *out_row = (char *)kp.dst + (int64_t)blockIdx.y * kp.dst_batch_stride +
                            (int64_t)(y0 + rg - kp.dst_y0) * kp.dst_pitch;
            for (int yb = rg; yb < sp.th; yb += RG * U) {
                const TI *row[U];
                TA w[U][MAXT + 1], acc[U];
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    const int yo = min(yb + u * RG, sp.th - 1);
                    row[u] = tile + off[yo];
                    load_record(rec + yo * RS, w[u]);
                    acc[u] = (TA)0;
                }
#pragma unroll
                for (int k = 0; k < MAXT; ++k) {
                    TI v[U][NV][VEC];
#pragma unroll
                    for (int u = 0; u < U; ++u)  // all loads of this source row first ...
#pragma unroll
                        for (int q = 0; q < NV; ++q) TapVec<TI>::load(row[u] + k * sp.bw + q * VEC, v[u][q]);
#pragma unroll
                    for (int u = 0; u < U; ++u) {  // ... then its horizontal taps and its vertical tap
                        TA hs = (TA)0;
#pragma unroll
                        for (int q = 0; q < NV; ++q)
#pragma unroll
                            for (int e = 0; e < VEC; ++e) hs += wv[q * VEC + e] * to_arith<TA>(v[u][q][e]);
                        acc[u] += w[u][k] * hs;
                    }
                }
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    const TA out = sep_normalise<TA>(acc[u], sumx * w[u][MAXT]);
                    if (yb + u * RG < ylim) {
                        if constexpr (std::is_same<TA, float>::value) store_f<TO>(out_row, x, out);
                        else store_dst<TO>(out_row, x, out);
                    }
                    out_row += (int64_t)RG * kp.dst_pitch;
                }
            }
        }
        __syncthreads();  // tile t's buffers are free, the row weights just written are visible
    }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                  const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// driver entry point, resolved once (thread-safe: aai_run_host drives one host thread per device)
EncodeTiledFn encode_tiled_fn() {
    static const EncodeTiledFn fn = [] {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            return (EncodeTiledFn)p;
        cudaGetLastError();
        return (EncodeTiledFn) nullptr;
    }();
    return fn;
}

constexpr int kSepMaxDevices = 64;
// SM count of the current device (cached per device; 0 = not yet queried)
int sm_count_of(int dev) {
    static std::atomic<int> cache[kSepMaxDevices];
    if (dev < 0 || dev >= kSepMaxDevices) return 148;
    int n = cache[dev].load(std::memory_order_relaxed);
    if (n <= 0) {
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) {
            cudaGetLastError();
            n = 148;
        }
        cache[dev].store(n, std::memory_order_relaxed);
    }
    return n;
}

// The encoded tensor map of the last launch of this thread, reused while the source view is the same (a cfg-1 sized
// image is launch-latency bound: re-encoding the map and re-setting the kernel attribute was most of its host cost).
struct TmapKey {
    const void *src;
    int64_t pitch, batch_stride;
    int32_t w, rows, batch, bw, bh, dtype;
    bool operator==(const TmapKey &o) const {
        return src == o.src && pitch == o.pitch && batch_stride == o.batch_stride && w == o.w && rows == o.rows &&
               batch == o.batch && bw == o.bw && bh == o.bh && dtype == o.dtype;
    }
};
struct TmapCache {
    bool valid = false;
    TmapKey key;
    CUtensorMap map;
};

// returns cudaErrorNotSupported when the fast path does not apply (the caller then uses the direct-tap kernel)
template <typename TI, typename TO, typename TA, int TW, int MAXT>
cudaError_t launch_sep(const AaiKernelParams &kp, cudaStream_t stream) {
    EncodeTiledFn enc = encode_tiled_fn();
    if (!enc) return cudaErrorNotSupported;
    const double L = 2.0 * kp.shape.half;
    const int esz = (int)sizeof(TI), align = 16 / esz;
    SepParams sp;
    sp.tw = TW;
    sp.stages = 2;
#ifdef AAI_DEV_KNOBS  // developer builds only (sweeps in profiles/); the shipped library reads no environment
    if (const char *e = getenv("AAI_SEP_STAGES")) sp.stages = atoi(e);
    if (sp.stages < 2 || sp.stages > 8) return cudaErrorNotSupported;
#endif
    const int batch = kp.batch > 0 ? kp.batch : 1;
    const int rows = kp.row1 - kp.row0;
    // tile height: the tallest of 48 / 32 / 16 canvas rows whose ring of source windows leaves room for two CTAs per SM
    // (measured on config 5: 48 rows x 2 stages, 2 CTAs/SM is the fastest -- fewer halo rows, 54 KB per TMA load)
    size_t tile_bytes = 0, wgt_bytes = 0, smem = 0;
    bool found = false;
    for (int th : {48, 32, 16}) {
#ifdef AAI_DEV_KNOBS
        if (const char *e = getenv("AAI_SEP_TH")) th = atoi(e);
        if (th < 8 || th > 256 || th % (SEP_THREADS / TW) != 0) return cudaErrorNotSupported;
#endif
        sp.th = th;
        // the window must hold MAXT taps starting at the first cell of the LAST column / row of the tile
        // (+ align-1 columns because the window origin is rounded down to a 16-byte boundary)
        // (+ 2(VEC-1) so that the taps can be read as whole aligned vectors)
        sp.bw = ((int)ceil((TW - 1) * L) + MAXT + 3 + 2 * (TapVec<TI>::N - 1) + (align - 1) + align - 1) / align * align;
        sp.bh = (int)ceil((sp.th - 1) * L) + MAXT + 3;
        tile_bytes = ((size_t)sp.bw * sp.bh * esz + 127) / 128 * 128;
        wgt_bytes = sep_weight_bytes<TA, MAXT>(sp.th);
        smem = sp.stages * (tile_bytes + wgt_bytes) + 8 * sp.stages + 16;
        if (sp.bw <= 256 && sp.bh <= 256 && sp.bw >= MAXT && sp.bh >= MAXT && smem <= 112 * 1024) {
            found = true;
            break;
        }
#ifdef AAI_DEV_KNOBS
        if (getenv("AAI_SEP_TH")) break;
#endif
    }
    if (!found && (sp.bw > 256 || sp.bh > 256 || sp.bw < MAXT || sp.bh < MAXT || smem > 220 * 1024))
        return cudaErrorNotSupported;
    sp.tiles_x = (kp.dst_w + TW - 1) / TW;
    sp.tiles_y = (rows + sp.th - 1) / sp.th;
    // strips are cut into segments so that the grid still fills the device (~4 CTAs per SM) when the batch is small
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return cudaGetLastError();
    const int want_ctas = 4 * sm_count_of(dev);
    int segs = (want_ctas + sp.tiles_x * batch - 1) / (sp.tiles_x * batch);
    segs = segs < 1 ? 1 : (segs > sp.tiles_y ? sp.tiles_y : segs);
    sp.tiles_per_cta = (sp.tiles_y + segs - 1) / segs;
    segs = (sp.tiles_y + sp.tiles_per_cta - 1) / sp.tiles_per_cta;

    const int64_t batch_stride = batch > 1 ? kp.src_batch_stride : kp.src_pitch * (int64_t)kp.src_rows;
    if (batch_stride % 16 != 0) return cudaErrorNotSupported;
    static thread_local TmapCache cache;  // per kernel instantiation and host thread
    const TmapKey key = {kp.src, kp.src_pitch, batch_stride, kp.src_w, kp.src_rows, batch, sp.bw, sp.bh, (int32_t)Elem<TI>::tmap};
    if (!cache.valid || !(cache.key == key)) {
        const cuuint64_t gdim[3] = {(cuuint64_t)kp.src_w, (cuuint64_t)kp.src_rows, (cuuint64_t)batch};
        const cuuint64_t gstride[2] = {(cuuint64_t)kp.src_pitch, (cuuint64_t)batch_stride};
        const cuuint32_t box[3] = {(cuuint32_t)sp.bw, (cuuint32_t)sp.bh, 1};
        const cuuint32_t estr[3] = {1, 1, 1};
        const CUresult r = enc(&cache.map, Elem<TI>::tmap, 3, const_cast<void *>(kp.src), gdim, gstride, box, estr,
                               CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                               CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) {
            cache.valid = false;
            return cudaErrorNotSupported;
        }
        cache.key = key;
        cache.valid = true;
    }
    const CUtensorMap &tmap = cache.map;
#ifdef AAI_DEV_KNOBS
    if (getenv("AAI_DEBUG"))
        fprintf(stderr, "[aai] separable TMA: TI=%d bytes TA=%d bytes TW=%d MAXT=%d box %dx%d tiles %dx%d smem %zu src %p pitch %lld "
                "w %d rows %d\n", esz, (int)sizeof(TA), TW, MAXT, sp.bw, sp.bh, sp.tiles_x, sp.tiles_y, smem, kp.src,
                (long long)kp.src_pitch, kp.src_w, kp.src_rows);
#endif
    auto kernel = separable_tma_kernel<TI, TO, TA, TW, MAXT>;
    // dynamic shared-memory limit of this instantiation: raised once per device (grow-only)
    static std::atomic<int> smem_set[kSepMaxDevices];
    if (dev < 0 || dev >= kSepMaxDevices || smem_set[dev].load(std::memory_order_relaxed) < (int)smem) {
        cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        if (dev >= 0 && dev < kSepMaxDevices) smem_set[dev].store((int)smem, std::memory_order_relaxed);
    }
    kernel<<<dim3(sp.tiles_x * segs, batch), SEP_BLOCK, smem, stream>>>(tmap, kp, sp);
    return cudaGetLastError();
}

template <typename TI, typename TO, typename TA>
cudaError_t launch_sep_shape(const AaiKernelParams &kp, cudaStream_t stream) {
    const double L = 2.0 * kp.shape.half;
    // an interval of length L meets at most ceil(L)+1 unit cells with positive length
    const int taps = (int)ceil(L - 1e-12) + 1;
    cudaError_t e = cudaErrorNotSupported;
    if (taps <= 3) e = launch_sep<TI, TO, TA, 64, 3>(kp, stream);
    if (e == cudaErrorNotSupported && taps <= 4) e = launch_sep<TI, TO, TA, 64, 4>(kp, stream);
    if (e == cudaErrorNotSupported && taps <= 6) e = launch_sep<TI, TO, TA, 64, 6>(kp, stream);
    if (e == cudaErrorNotSupported && taps <= 10) e = launch_sep<TI, TO, TA, 32, 10>(kp, stream);
    return e;
}

// taps in TA arithmetic for the sources Srcs, every canvas type
template <typename TA, typename Srcs>
cudaError_t launch_sep_pair(const AaiKernelParams &kp, int src_dtype, int dst_dtype, cudaStream_t stream) {
    return with_pair<Srcs, AnyElem>(src_dtype, dst_dtype, cudaErrorInvalidValue, [&](auto ti, auto to) {
        return launch_sep_shape<typename decltype(ti)::type, typename decltype(to)::type, TA>(kp, stream);
    });
}


// ------------------------------------------------------------------------------------------------------------
// Axis-aligned cases OUTSIDE the TMA kernel's preconditions -- a quadrant pre-rotation (90 / 180 / 270 degrees,
// Source.cpp:163-168), an integer expansion (scale > 1), interleaved RGB -- in FP32 arithmetic: direct taps, fully
// unrolled.  Same weights as the TMA kernel (axis_taps<float>: the footprint interval against the unit cells of the
// expanded frame, in-image cells only), the cells found through the separable byte offset col_off(i) + row_off(j) of
// the expanded-frame index map (as in the FP32 overlap kernel), MAXT x MAXT loads per canvas pixel through L1.
// (Before round 2 these cases ran on the FP64 direct-tap kernel with a division per tap.)
// ------------------------------------------------------------------------------------------------------------
// TRANSPOSED (quadrants 1 / 3: canvas y runs along source x): the lanes of a warp step along canvas y, so that the
// MAXT x MAXT loads of a pixel stay coalesced and the one store per pixel takes the stride instead.
template <typename TI, typename TO, int NC, int MAXT, bool TRANSPOSED>
__global__ void __launch_bounds__(TILE_W *TILE_H)
    separable_direct_f32(const __grid_constant__ AaiKernelParams kp) {
    const int x = TRANSPOSED ? blockIdx.x * TILE_H + threadIdx.y : blockIdx.x * TILE_W + threadIdx.x;
    const int y = kp.row0 + (TRANSPOSED ? blockIdx.y * TILE_W + threadIdx.x : blockIdx.y * TILE_H + threadIdx.y);
    if (x >= kp.dst_w || y >= kp.row1) return;
    double cx, cy;
    pixel_centre(kp, x, y, cx, cy);
    const double h = kp.shape.half;
    float wx[MAXT], wy[MAXT], sumx, sumy;
    int fx0, fy0;
    axis_taps<float, MAXT>(cx, h, kp.mod_w, fx0, wx, sumx);
    axis_taps<float, MAXT>(cy, h, kp.mod_h, fy0, wy, sumy);
    constexpr int ESZ = (int)sizeof(TI) * NC;
    const bool swapped = kp.e_axi == 0;
    auto div_s = [&](int e) -> int64_t {
        return (int64_t)(kp.scale != 1 ? __umulhi((unsigned)e, kp.div_magic) : (unsigned)e);
    };
    int64_t coff[MAXT], roff[MAXT];
#pragma unroll
    for (int k = 0; k < MAXT; ++k) {  // out-of-image taps carry weight 0: clamp their address into the image
        const int i = min(max(fx0 + k, 0), kp.mod_w - 1), j = min(max(fy0 + k, 0), kp.mod_h - 1);
        coff[k] = swapped ? (div_s(kp.e_ayi * i + kp.e_ay0) - src_row0(kp)) * kp.src_pitch
                          : div_s(kp.e_axi * i + kp.e_ax0) * ESZ;
        roff[k] = swapped ? div_s(kp.e_axj * j + kp.e_ax0) * ESZ
                          : (div_s(kp.e_ayj * j + kp.e_ay0) - src_row0(kp)) * kp.src_pitch;
    }
    float acc[NC];
#pragma unroll
    for (int ch = 0; ch < NC; ++ch) acc[ch] = 0.0f;
#pragma unroll
    for (int r = 0; r < MAXT; ++r) {
        const char *rowp = (const char *)kp.src + roff[r];
        float hs[NC];
#pragma unroll
        for (int ch = 0; ch < NC; ++ch) hs[ch] = 0.0f;
#pragma unroll
        for (int k = 0; k < MAXT; ++k)
#pragma unroll
            for (int ch = 0; ch < NC; ++ch)
                hs[ch] += wx[k] * to_arith<float>(__ldg(reinterpret_cast<const TI *>(rowp + coff[k]) + ch));
#pragma unroll
        for (int ch = 0; ch < NC; ++ch) acc[ch] += wy[r] * hs[ch];
    }
    char *drow = (char *)kp.dst + (int64_t)(y - dst_row0(kp)) * kp.dst_pitch;
    const float total = sumx * sumy;
#pragma unroll
    for (int ch = 0; ch < NC; ++ch) store_f<TO>(drow, x * NC + ch, sep_normalise<float>(acc[ch], total));
}

template <typename TI, typename TO, int NC>
cudaError_t launch_direct_taps(const AaiKernelParams &kp, cudaStream_t stream) {
    const double L = 2.0 * kp.shape.half;
    const int taps = (int)ceil(L - 1e-12) + 1;
    const int rows = kp.row1 - kp.row0;
    dim3 block(TILE_W, TILE_H);
    const bool tr = kp.e_axi == 0;  // quadrants 1 / 3
    const int tw = tr ? TILE_H : TILE_W, th = tr ? TILE_W : TILE_H;
    if ((rows + th - 1) / th > 65535) return cudaErrorNotSupported;
    dim3 grid((kp.dst_w + tw - 1) / tw, (rows + th - 1) / th, kp.batch > 1 ? kp.batch : 1);
    if (taps <= 3) {
        if (tr) separable_direct_f32<TI, TO, NC, 3, true><<<grid, block, 0, stream>>>(kp);
        else separable_direct_f32<TI, TO, NC, 3, false><<<grid, block, 0, stream>>>(kp);
    } else if (taps <= 4) {
        if (tr) separable_direct_f32<TI, TO, NC, 4, true><<<grid, block, 0, stream>>>(kp);
        else separable_direct_f32<TI, TO, NC, 4, false><<<grid, block, 0, stream>>>(kp);
    } else if (taps <= 6) {
        if (tr) separable_direct_f32<TI, TO, NC, 6, true><<<grid, block, 0, stream>>>(kp);
        else separable_direct_f32<TI, TO, NC, 6, false><<<grid, block, 0, stream>>>(kp);
    } else {
        return cudaErrorNotSupported;
    }
    return cudaGetLastError();
}

}  // namespace

// Returns cudaErrorNotSupported (as int) when the TMA fast path does not apply.
int aai_launch_separable_tma(const AaiKernelParams &kp, int arith, int src_dtype, int dst_dtype, void *stream) {
    if (kp.scale != 1 || kp.quadrant != 0 || kp.channels != 1) return (int)cudaErrorNotSupported;
    if ((kp.src_pitch % 16) != 0 || (reinterpret_cast<uintptr_t>(kp.src) % 16) != 0) return (int)cudaErrorNotSupported;
    if (kp.row1 <= kp.row0 || kp.dst_w <= 0) return (int)cudaSuccess;
    cudaStream_t st = (cudaStream_t)stream;
    if (arith == AAI_ARITH_F32 && src_dtype != AAI_F64)
        return (int)launch_sep_pair<float, NarrowElem>(kp, src_dtype, dst_dtype, st);
    return (int)launch_sep_pair<double, AnyElem>(kp, src_dtype, dst_dtype, st);
}

// FP32 direct-tap kernel for the axis-aligned cases the TMA kernel does not take (quadrants 1-3, scale > 1, RGB);
// cudaErrorNotSupported -> the caller falls back to the FP64 direct-tap kernel (also for double images, which keep FP64
// arithmetic).
int aai_launch_separable_direct_f32(const AaiKernelParams &kp, int src_dtype, int dst_dtype, void *stream) {
    const uint64_t max_e = (uint64_t)(kp.mod_w > kp.mod_h ? kp.mod_w : kp.mod_h);
    if (max_e * (uint64_t)kp.scale >= 0x100000000ULL) return (int)cudaErrorNotSupported;  // multiply-high division range
    if (kp.row1 <= kp.row0 || kp.dst_w <= 0) return (int)cudaSuccess;
    return (int)with_pair<NarrowElem, NarrowElem>(src_dtype, dst_dtype, cudaErrorNotSupported, [&](auto ti, auto to) {
        using TI = typename decltype(ti)::type;
        using TO = typename decltype(to)::type;
        return with_channels<1, 3>(kp.channels, cudaErrorNotSupported, [&](auto nc) {
            return launch_direct_taps<TI, TO, decltype(nc)::value>(kp, (cudaStream_t)stream);
        });
    });
}
