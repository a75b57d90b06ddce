// C ABI glue (include/aai.h): pitched device images, kernel dispatch, the host-buffer entry point with its
// row-band partitioner over per-device streams.  CUDA runtime only -- no torch, no NCCL (bands are independent,
// SURVEY.md §8e), no CPU fallback.
#include <cuda_runtime.h>

#include <atomic>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "aai_internal.h"

namespace {

thread_local char g_error[512] = "";
std::atomic<int64_t> g_launches{0};
thread_local float g_h2d_ms = -1.f, g_kernel_ms = -1.f, g_d2h_ms = -1.f;

int cuda_fail(cudaError_t e, const char *what) {
    aai_set_error("%s: %s (%s)", what, cudaGetErrorString(e), cudaGetErrorName(e));
    return (e == cudaErrorNoDevice || e == cudaErrorInsufficientDriver) ? AAI_ERR_NO_DEVICE : AAI_ERR_CUDA;
}
#define AAI_CUDA(call)                                   \
    do {                                                 \
        cudaError_t e_ = (call);                         \
        if (e_ != cudaSuccess) return cuda_fail(e_, #call); \
    } while (0)

bool image_ok(const aai_image *im) {
    return im && im->data && aai_elem_size(im->dtype) && im->channels >= 1 && im->channels <= 4 && im->width > 0 &&
           im->height > 0 && im->rows >= 0 && im->y0 >= 0 && im->y0 + im->rows <= im->height &&
           im->pitch_bytes >= (int64_t)(im->width * im->channels * (int64_t)aai_elem_size(im->dtype));
}

// well-formed source and canvas images of the plan's sizes with one channel count (rows are the caller's business)
bool images_match_plan(const aai_plan *plan, const aai_image *src, const aai_image *dst) {
    return image_ok(src) && image_ok(dst) && src->width == plan->src_w && src->height == plan->src_h &&
           dst->width == plan->dst_w && dst->height == plan->dst_h && src->channels == dst->channels;
}
bool mode_ok(int mode) { return mode >= AAI_MODE_AREA_AVERAGE && mode <= AAI_MODE_AREA_AVERAGE_EXACT; }
bool arith_ok(int arith) { return arith >= AAI_ARITH_F64 && arith <= AAI_ARITH_F32_RING; }

int check_plan(const char *who, const aai_plan *plan) {
    if (plan) return plan->status;
    aai_set_error("%s: null plan", who);
    return AAI_ERR_ARGUMENT;
}

int check_device(const char *who, int device) {
    if (aai_device_count() > device && device >= 0) return AAI_OK;
    aai_set_error("%s: device %d not present; this library has no CPU fallback", who, device);
    return aai_device_count() <= 0 ? AAI_ERR_NO_DEVICE : AAI_ERR_ARGUMENT;
}

// Launches fn(a, b) for each slab [a, b) of at most AAI_MAX_ROWS_PER_LAUNCH rows of [row0, row1), counting each
// launch in aai_launch_count(): the kernels put rows on grid.y (<= 65535 CTAs), so taller row ranges (line scans, large
// upscales) take several launches.  Returns the first launch error (cudaError_t as int).
template <class Fn>
int launch_slabs(int64_t row0, int64_t row1, Fn fn) {
    for (int64_t a = row0; a < row1; a += AAI_MAX_ROWS_PER_LAUNCH) {
        const int e = fn(a, a + AAI_MAX_ROWS_PER_LAUNCH < row1 ? a + AAI_MAX_ROWS_PER_LAUNCH : row1);
        if (e != (int)cudaSuccess) return e;
        g_launches.fetch_add(1);
    }
    return (int)cudaSuccess;
}

// grow-only per-device scratch images used by aai_run_host (avoids cudaMalloc/cudaFree per call)
struct Workspace {
    void *ptr[2] = {nullptr, nullptr};
    size_t cap[2] = {0, 0};
    cudaStream_t stream = nullptr;          // compute stream (also the only stream of unpipelined runs)
    cudaStream_t up = nullptr, dn = nullptr;  // copy streams of the pipelined host path
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
    std::vector<cudaEvent_t> chunk_ev;        // 2 per chunk: upload done, kernel done
    cudaEvent_t fork = nullptr, join_up = nullptr, join_dn = nullptr;
    cudaEvent_t done = nullptr;  // end of the last band run that used this workspace (asynchronous callers may
    bool done_valid = false;     // use different streams: the next run waits for it before touching the buffers)
    std::mutex busy;  // held for the duration of one band run on this device
};
constexpr int kMaxDevices = 64;
std::mutex g_ws_mutex;
Workspace g_ws[kMaxDevices];

int workspace_get(int device, size_t bytes0, size_t bytes1, Workspace **out) {
    if (device < 0 || device >= kMaxDevices) {
        aai_set_error("device index %d out of range", device);
        return AAI_ERR_ARGUMENT;
    }
    std::lock_guard<std::mutex> lock(g_ws_mutex);
    Workspace &w = g_ws[device];
    AAI_CUDA(cudaSetDevice(device));
    if (!w.stream) {
        AAI_CUDA(cudaStreamCreateWithFlags(&w.stream, cudaStreamNonBlocking));
        AAI_CUDA(cudaStreamCreateWithFlags(&w.up, cudaStreamNonBlocking));
        AAI_CUDA(cudaStreamCreateWithFlags(&w.dn, cudaStreamNonBlocking));
        for (auto &e : w.ev) AAI_CUDA(cudaEventCreate(&e));
        AAI_CUDA(cudaEventCreateWithFlags(&w.fork, cudaEventDisableTiming));
        AAI_CUDA(cudaEventCreateWithFlags(&w.join_up, cudaEventDisableTiming));
        AAI_CUDA(cudaEventCreateWithFlags(&w.join_dn, cudaEventDisableTiming));
        AAI_CUDA(cudaEventCreateWithFlags(&w.done, cudaEventDisableTiming));
    }
    const size_t need[2] = {bytes0, bytes1};
    for (int k = 0; k < 2; ++k) {
        if (w.cap[k] < need[k]) {
            if (w.ptr[k]) AAI_CUDA(cudaFree(w.ptr[k]));
            w.ptr[k] = nullptr;
            w.cap[k] = 0;
            AAI_CUDA(cudaMalloc(&w.ptr[k], need[k]));
            w.cap[k] = need[k];
        }
    }
    *out = &w;
    return AAI_OK;
}

// Head of a host-buffer run on `device`'s workspace: holds the workspace's busy lock in `busy` for the rest of the
// run, sizes its buffers, picks the stream (the caller's, else the workspace's own) and records ev[0], the start of the
// run.  A pipelined run asks for chunk_events > 0 chunk events and gets its copy streams forked off `st` at ev[0].
int pipeline_head(std::unique_lock<std::mutex> &busy, int device, size_t bytes0, size_t bytes1, void *stream,
                  int chunk_events, Workspace **out, cudaStream_t *st_out) {
    busy = std::unique_lock<std::mutex>(g_ws[device < kMaxDevices ? device : 0].busy);
    if (const int r = workspace_get(device, bytes0, bytes1, out)) return r;
    Workspace *w = *out;
    const cudaStream_t st = *st_out = stream ? (cudaStream_t)stream : w->stream;
    // the workspace is shared by every run on this device: order this run after the previous one even when an
    // asynchronous caller switched streams in between
    if (w->done_valid) AAI_CUDA(cudaStreamWaitEvent(st, w->done, 0));
    AAI_CUDA(aai_grow_events(w->chunk_ev, (size_t)chunk_events));
    AAI_CUDA(cudaEventRecord(w->ev[0], st));
    if (chunk_events > 0) {
        AAI_CUDA(cudaStreamWaitEvent(w->up, w->ev[0], 0));
        AAI_CUDA(cudaStreamWaitEvent(w->dn, w->ev[0], 0));
    }
    return AAI_OK;
}

// Tail of a host-buffer run: a pipelined run joins its copy streams back onto `st`; then ev[3] and `done` mark the end.
// A synchronous call waits and stores aai_last_host_timing(): the three phases of an unpipelined run (ev[1] and ev[2]
// between them), or the whole call of a pipelined one, whose overlapped phases cannot be separated.
int pipeline_tail(Workspace *w, cudaStream_t st, bool pipelined, bool synchronize) {
    if (pipelined) {
        AAI_CUDA(cudaEventRecord(w->join_up, w->up));
        AAI_CUDA(cudaEventRecord(w->join_dn, w->dn));
        AAI_CUDA(cudaStreamWaitEvent(st, w->join_up, 0));
        AAI_CUDA(cudaStreamWaitEvent(st, w->join_dn, 0));
    }
    AAI_CUDA(cudaEventRecord(w->ev[3], st));
    AAI_CUDA(cudaEventRecord(w->done, st));
    w->done_valid = true;
    if (!synchronize) return AAI_OK;
    AAI_CUDA(cudaStreamSynchronize(st));
    if (!pipelined) {
        AAI_CUDA(cudaEventElapsedTime(&g_h2d_ms, w->ev[0], w->ev[1]));
        AAI_CUDA(cudaEventElapsedTime(&g_kernel_ms, w->ev[1], w->ev[2]));
        AAI_CUDA(cudaEventElapsedTime(&g_d2h_ms, w->ev[2], w->ev[3]));
        return AAI_OK;
    }
    float total = 0.f;
    AAI_CUDA(cudaEventElapsedTime(&total, w->ev[0], w->ev[3]));
    g_h2d_ms = total;
    g_kernel_ms = 0.f;
    g_d2h_ms = 0.f;
    return AAI_OK;
}

}  // namespace

cudaError_t aai_copy_pitched(void *dst, int64_t dst_pitch, const void *src, int64_t src_pitch, size_t row_bytes,
                             int64_t rows, cudaMemcpyKind kind, cudaStream_t stream) {
    if (rows <= 0) return cudaSuccess;
    // Both sides dense (no padding between rows): one linear copy (faster DMA than a strided 2-D copy).  With padded
    // rows the copy must not touch the bytes between rows -- a host image may be a column view of a wider array.
    if ((size_t)dst_pitch == row_bytes && (size_t)src_pitch == row_bytes)
        return cudaMemcpyAsync(dst, src, row_bytes * (size_t)rows, kind, stream);
    return cudaMemcpy2DAsync(dst, (size_t)dst_pitch, src, (size_t)src_pitch, row_bytes, (size_t)rows, kind, stream);
}

cudaError_t aai_grow_events(std::vector<cudaEvent_t> &events, size_t n) {
    while (events.size() < n) {
        cudaEvent_t e;
        if (const cudaError_t r = cudaEventCreateWithFlags(&e, cudaEventDisableTiming)) return r;
        events.push_back(e);
    }
    return cudaSuccess;
}

void aai_count_extra_launches(int n) { g_launches.fetch_add(n); }

int aai_check_dtype_pair(const char *who, int src_dtype, int dst_dtype) {
    if (aai_dtype_pair_ok(src_dtype, dst_dtype)) return AAI_OK;
    aai_set_error("%s: a %s source cannot write a %s canvas (a uint16 canvas takes a uint16 source; a uint16 source "
                  "writes float64, float32 or uint16 canvases)",
                  who, aai_dtype_name(src_dtype), aai_dtype_name(dst_dtype));
    return AAI_ERR_ARGUMENT;
}

void aai_set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_error, sizeof g_error, fmt, ap);
    va_end(ap);
}

AaiKernelParams aai_make_kernel_params(const aai_plan &p, const aai_image &src, const aai_image &dst, int64_t row0,
                                       int64_t row1) {
    AaiKernelParams k;
    std::memset(&k, 0, sizeof k);
    k.side = p.side;
    k.off_ix = p.off_ix;
    k.off_iy = p.off_iy;
    k.iso_x = p.iso_x;
    k.iso_y = p.iso_y;
    k.off_x = p.off_x;
    k.off_y = p.off_y;
    const double c = p.cos_t, s = p.sin_t, h = p.side / 2;
    {
        const double u0 = (p.off_ix * p.side - p.iso_x) + p.off_x, v0 = (p.off_iy * p.side - p.iso_y) + p.off_y;
        k.aff_x0 = (u0 * c + v0 * s) + p.iso_x;
        k.aff_y0 = (-u0 * s + v0 * c) + p.iso_y;
        k.aff_xx = p.side * c;
        k.aff_xy = p.side * s;
        k.aff_yx = -p.side * s;
        k.aff_yy = p.side * c;
        k.ext32 = (float)(h * (c + s) + 0.5 + 2e-6);
    }
    k.shape = aai_make_shape(c, s, p.side);
    const AaiShape &g = k.shape;
    // FP32 constants incl. the guard band of the FP32 shape decisions; near-axis angles (1/sin or 1/cos > 20) use the
    // FP64 kernel
    k.shapef = aai_make_shape_f(c, s, p.side);
    const double amp = std::fmax(1.0, std::fmax(g.inv_c, g.inv_s));
    const uint64_t max_e = (uint64_t)(p.mod_w > p.mod_h ? p.mod_w : p.mod_h);
    k.f32_ok = (s > 0.0 && c > 0.0 && amp <= 20.0 && max_e * p.scale < 0x100000000ULL) ? 1 : 0;
    {
        const int nmax = aai_f32_maxn(k.ext32);
        k.tip_window = nmax > 0 && aai_tip_window_ok(c, s, p.side, nmax) ? 1 : 0;
    }
    k.quirk = 1;
    k.reach = p.reach;
    k.hb = h * (c + s);
    k.mod_w = (int32_t)p.mod_w;
    k.mod_h = (int32_t)p.mod_h;
    k.dst_w = (int32_t)p.dst_w;
    k.dst_h = (int32_t)p.dst_h;
    k.scale = (int32_t)p.scale;
    k.quadrant = p.quadrant;
    const int32_t mw1 = (int32_t)p.mod_w - 1, mh1 = (int32_t)p.mod_h - 1;
    switch (p.quadrant) {
        case 0: k.e_axi = 1; k.e_axj = 0; k.e_ax0 = 0; k.e_ayi = 0; k.e_ayj = 1; k.e_ay0 = 0; break;
        case 1: k.e_axi = 0; k.e_axj = 1; k.e_ax0 = 0; k.e_ayi = -1; k.e_ayj = 0; k.e_ay0 = mw1; break;
        case 2: k.e_axi = -1; k.e_axj = 0; k.e_ax0 = mw1; k.e_ayi = 0; k.e_ayj = -1; k.e_ay0 = mh1; break;
        default: k.e_axi = 0; k.e_axj = -1; k.e_ax0 = mh1; k.e_ayi = 1; k.e_ayj = 0; k.e_ay0 = 0; break;
    }
    k.div_magic = p.scale > 1 ? (uint32_t)(0x100000000ULL / p.scale) + 1u : 0u;
    k.src = src.data;
    k.src_pitch = src.pitch_bytes;
    k.src_w = (int32_t)src.width;
    k.src_h = (int32_t)src.height;
    k.src_y0 = (int32_t)src.y0;
    k.src_rows = (int32_t)src.rows;
    k.channels = src.channels;
    k.dst = dst.data;
    k.dst_pitch = dst.pitch_bytes;
    k.dst_y0 = (int32_t)dst.y0;
    k.row0 = (int32_t)row0;
    k.row1 = (int32_t)row1;
    return k;
}

// One kernel of the path over canvas rows [kp.row0, kp.row1), slab by slab (bands are independent: the same result)
static int launch_rows(const aai_plan &plan, int mode, int arith, AaiKernelParams kp, int src_dtype, int dst_dtype,
                       void *stream) {
    kp.staged = arith == AAI_ARITH_F32_STAGED ? 1 : arith == AAI_ARITH_F32_BINNED ? 2 : arith == AAI_ARITH_F32_RING ? 3 : 0;
    if (kp.staged) arith = AAI_ARITH_F32;
    return launch_slabs(kp.row0, kp.row1, [&](int64_t a, int64_t b) {
        kp.row0 = (int32_t)a;
        kp.row1 = (int32_t)b;
        {  // CTA row order: towards the end of the launch where the rotated image covers more of the canvas rows
            const int64_t n = kp.row1 - kp.row0, e = n / 8 > 64 ? 64 : (n / 8 > 0 ? n / 8 : 1);
            kp.reverse_rows = aai_covered_pixels(&plan, kp.row0, kp.row0 + e) > aai_covered_pixels(&plan, kp.row1 - e, kp.row1) ? 1 : 0;
        }
        if (mode == AAI_MODE_FAST) return aai_launch_fast(kp, arith, src_dtype, dst_dtype, stream);
        if (plan.axis_aligned) return aai_launch_separable(kp, arith, src_dtype, dst_dtype, stream);
        return aai_launch_overlap(kp, arith, src_dtype, dst_dtype, stream);
    });
}

extern "C" {

const char *aai_last_error(void) { return g_error; }

int64_t aai_launch_count(void) { return g_launches.load(); }

int aai_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

int aai_image_alloc(aai_image *img, int device, int64_t width, int64_t height, int64_t y0, int64_t rows,
                    int32_t dtype, int32_t channels) {
    if (!img || !aai_elem_size(dtype) || channels < 1 || channels > 4 || width <= 0 || height <= 0 || rows < 0 ||
        y0 < 0 || y0 + rows > height) {
        aai_set_error("aai_image_alloc: bad argument");
        return AAI_ERR_ARGUMENT;
    }
    AAI_CUDA(cudaSetDevice(device));
    std::memset(img, 0, sizeof *img);
    img->width = width;
    img->height = height;
    img->y0 = y0;
    img->rows = rows;
    img->dtype = dtype;
    img->channels = channels;
    img->pitch_bytes = aai_device_pitch(width, channels, dtype);
    const size_t bytes = (size_t)img->pitch_bytes * (size_t)(rows > 0 ? rows : 1);
    AAI_CUDA(cudaMalloc(&img->data, bytes));
    return AAI_OK;
}

int aai_image_free(aai_image *img, int device) {
    if (!img) return AAI_ERR_ARGUMENT;
    if (img->data) {
        AAI_CUDA(cudaSetDevice(device));
        AAI_CUDA(cudaFree(img->data));
    }
    img->data = nullptr;
    return AAI_OK;
}

static int copy_rows(const aai_image *dst, const aai_image *src, cudaMemcpyKind kind, int device, void *stream) {
    // copies the rows of the image that holds FEWER rows (the device band) from/to the other one
    if (!image_ok(dst) || !image_ok(src) || dst->width != src->width || dst->height != src->height ||
        dst->dtype != src->dtype || dst->channels != src->channels) {
        aai_set_error("aai_image copy: incompatible images");
        return AAI_ERR_ARGUMENT;
    }
    const aai_image *band = (kind == cudaMemcpyHostToDevice) ? dst : src;
    const aai_image *full = (kind == cudaMemcpyHostToDevice) ? src : dst;
    if (band->y0 < full->y0 || band->y0 + band->rows > full->y0 + full->rows) {
        aai_set_error("aai_image copy: band rows [%lld,%lld) not inside [%lld,%lld)", (long long)band->y0,
                      (long long)(band->y0 + band->rows), (long long)full->y0, (long long)(full->y0 + full->rows));
        return AAI_ERR_ARGUMENT;
    }
    if (band->rows == 0) return AAI_OK;
    AAI_CUDA(cudaSetDevice(device));
    const size_t row_bytes = (size_t)(band->width * band->channels) * aai_elem_size(band->dtype);
    const char *s = (const char *)src->data + (kind == cudaMemcpyHostToDevice ? (band->y0 - src->y0) * src->pitch_bytes : 0);
    char *d = (char *)dst->data + (kind == cudaMemcpyDeviceToHost ? (band->y0 - dst->y0) * dst->pitch_bytes : 0);
    AAI_CUDA(aai_copy_pitched(d, dst->pitch_bytes, s, src->pitch_bytes, row_bytes, band->rows, kind, (cudaStream_t)stream));
    return AAI_OK;
}

int aai_image_upload(const aai_image *device_img, const aai_image *host_img, int device, void *stream) {
    return copy_rows(device_img, host_img, cudaMemcpyHostToDevice, device, stream);
}
int aai_image_download(const aai_image *host_img, const aai_image *device_img, int device, void *stream) {
    return copy_rows(host_img, device_img, cudaMemcpyDeviceToHost, device, stream);
}

int aai_image_copy_rows(const aai_image *dst, const aai_image *src, int64_t y0, int64_t y1, int device, void *stream) {
    if (!image_ok(dst) || !image_ok(src) || dst->width != src->width || dst->height != src->height ||
        dst->dtype != src->dtype || dst->channels != src->channels || y0 < 0 || y1 < y0 || y0 < dst->y0 ||
        y1 > dst->y0 + dst->rows || y0 < src->y0 || y1 > src->y0 + src->rows) {
        aai_set_error("aai_image_copy_rows: incompatible images or rows [%lld,%lld) not present", (long long)y0,
                      (long long)y1);
        return AAI_ERR_ARGUMENT;
    }
    if (y1 == y0) return AAI_OK;
    AAI_CUDA(cudaSetDevice(device));
    const size_t row_bytes = (size_t)(src->width * src->channels) * aai_elem_size(src->dtype);
    char *d = (char *)dst->data + (y0 - dst->y0) * dst->pitch_bytes;
    const char *s = (const char *)src->data + (y0 - src->y0) * src->pitch_bytes;
    AAI_CUDA(aai_copy_pitched(d, dst->pitch_bytes, s, src->pitch_bytes, row_bytes, y1 - y0, cudaMemcpyDefault,
                              (cudaStream_t)stream));
    return AAI_OK;
}

int aai_ipc_export(const void *device_ptr, unsigned char handle[AAI_IPC_HANDLE_BYTES]) {
    static_assert(sizeof(cudaIpcMemHandle_t) == AAI_IPC_HANDLE_BYTES, "IPC handle size");
    if (!device_ptr || !handle) return AAI_ERR_ARGUMENT;
    cudaIpcMemHandle_t h;
    AAI_CUDA(cudaIpcGetMemHandle(&h, const_cast<void *>(device_ptr)));
    std::memcpy(handle, &h, sizeof h);
    return AAI_OK;
}

int aai_ipc_open(const unsigned char handle[AAI_IPC_HANDLE_BYTES], int device, void **device_ptr) {
    if (!handle || !device_ptr) return AAI_ERR_ARGUMENT;
    AAI_CUDA(cudaSetDevice(device));
    cudaIpcMemHandle_t h;
    std::memcpy(&h, handle, sizeof h);
    AAI_CUDA(cudaIpcOpenMemHandle(device_ptr, h, cudaIpcMemLazyEnablePeerAccess));
    return AAI_OK;
}

int aai_ipc_close(void *device_ptr, int device) {
    if (!device_ptr) return AAI_OK;
    AAI_CUDA(cudaSetDevice(device));
    AAI_CUDA(cudaIpcCloseMemHandle(device_ptr));
    return AAI_OK;
}

int aai_run_device(const aai_plan *plan, int mode, int arith, const aai_image *src, const aai_image *dst,
                   int64_t row0, int64_t row1, int device, void *stream) {
    if (const int r = check_plan("aai_run_device", plan)) return r;
    if (!images_match_plan(plan, src, dst)) {
        aai_set_error("aai_run_device: images do not match the plan (src %lldx%lld, canvas %lldx%lld)",
                      (long long)plan->src_w, (long long)plan->src_h, (long long)plan->dst_w, (long long)plan->dst_h);
        return AAI_ERR_ARGUMENT;
    }
    if (const int r = aai_check_dtype_pair("aai_run_device", src->dtype, dst->dtype)) return r;
    if (!mode_ok(mode)) {
        aai_set_error("aai_run_device: interpolation mode must be 1, 2 or 3");
        return AAI_ERR_ARGUMENT;
    }
    if (!arith_ok(arith)) {
        aai_set_error("aai_run_device: unknown arithmetic %d", arith);
        return AAI_ERR_ARGUMENT;
    }
    if (row0 < 0 || row1 > plan->dst_h || row0 > row1 || row0 < dst->y0 || row1 > dst->y0 + dst->rows) {
        aai_set_error("aai_run_device: rows [%lld,%lld) outside the destination band", (long long)row0, (long long)row1);
        return AAI_ERR_ARGUMENT;
    }
    if (row0 == row1) return AAI_OK;
    int64_t sx0, sx1, sy0, sy1;
    aai_band_source_window(plan, row0, row1, &sx0, &sx1, &sy0, &sy1);
    if (sy1 > sy0 && (sy0 < src->y0 || sy1 > src->y0 + src->rows)) {
        aai_set_error("aai_run_device: source rows [%lld,%lld) needed, [%lld,%lld) present", (long long)sy0,
                      (long long)sy1, (long long)src->y0, (long long)(src->y0 + src->rows));
        return AAI_ERR_ARGUMENT;
    }
    AAI_CUDA(cudaSetDevice(device));
    AaiKernelParams kp = aai_make_kernel_params(*plan, *src, *dst, row0, row1);
    kp.quirk = mode == AAI_MODE_AREA_AVERAGE_EXACT ? 0 : 1;
    const int e = launch_rows(*plan, mode, arith, kp, src->dtype, dst->dtype, stream);
    if (e != (int)cudaSuccess) return cuda_fail((cudaError_t)e, "kernel launch");
    return AAI_OK;
}

static int check_host_images(const char *who, const aai_plan *plan, const aai_image *src, const aai_image *dst,
                             bool whole) {
    if (const int r = check_plan(who, plan)) return r;
    if (!images_match_plan(plan, src, dst)) {
        aai_set_error("%s: host images do not match the plan", who);
        return AAI_ERR_ARGUMENT;
    }
    if (const int r = aai_check_dtype_pair(who, src->dtype, dst->dtype)) return r;
    if (whole && (src->y0 != 0 || src->rows != src->height || dst->y0 != 0 || dst->rows != dst->height)) {
        aai_set_error("%s: whole host images expected", who);
        return AAI_ERR_ARGUMENT;
    }
    return AAI_OK;
}

int aai_expand_device(const aai_plan *plan, const aai_image *src, const aai_image *dst_mod, int device, void *stream) {
    if (const int r = check_plan("aai_expand_device", plan)) return r;
    if (!image_ok(src) || !image_ok(dst_mod) || src->width != plan->src_w || src->height != plan->src_h ||
        src->y0 != 0 || src->rows != src->height || dst_mod->width != plan->mod_w || dst_mod->height != plan->mod_h ||
        dst_mod->y0 != 0 || dst_mod->rows != dst_mod->height || src->dtype != dst_mod->dtype ||
        src->channels != dst_mod->channels) {
        aai_set_error("aai_expand_device: need a whole source image and a whole %lld x %lld image of the same type",
                      (long long)plan->mod_w, (long long)plan->mod_h);
        return AAI_ERR_ARGUMENT;
    }
    AAI_CUDA(cudaSetDevice(device));
    // the kernel-parameter builder takes canvas-shaped destinations; only the source view and the index map are used
    aai_image canvas = *dst_mod;
    canvas.width = plan->dst_w;
    canvas.height = plan->dst_h;
    AaiKernelParams kp = aai_make_kernel_params(*plan, *src, canvas, 0, 0);
    kp.dst = dst_mod->data;
    kp.dst_pitch = dst_mod->pitch_bytes;
    const int e = aai_launch_expand(kp, (int)aai_elem_size(src->dtype), stream);
    if (e != (int)cudaSuccess) return cuda_fail((cudaError_t)e, "expand kernel launch");
    g_launches.fetch_add(1);
    return AAI_OK;
}

int aai_measure_fp32_tflops(int device, double *tflops) {
    if (!tflops) {
        aai_set_error("aai_measure_fp32_tflops: null result");
        return AAI_ERR_ARGUMENT;
    }
    AAI_CUDA(cudaSetDevice(device));
    int sms = 0;
    AAI_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
    float *scratch = nullptr;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    double flop = 0.0, best = 0.0;
    int rc = AAI_OK;
    cudaError_t ce = cudaMalloc(&scratch, 256);
    if (ce == cudaSuccess) ce = cudaEventCreate(&e0);
    if (ce == cudaSuccess) ce = cudaEventCreate(&e1);
    if (ce != cudaSuccess) rc = cuda_fail(ce, "FP32 probe set-up");
    for (int rep = 0; rep < 4 && rc == AAI_OK; ++rep) {  // first repetition warms up
        cudaEventRecord(e0, 0);
        const int e = aai_probe_fp32(sms * 8, 1 << 16, scratch, &flop, nullptr);
        cudaEventRecord(e1, 0);
        if (e != (int)cudaSuccess || cudaEventSynchronize(e1) != cudaSuccess) {
            rc = cuda_fail((cudaError_t)(e != (int)cudaSuccess ? e : (int)cudaGetLastError()), "FP32 probe");
            break;
        }
        float ms = 0.f;
        cudaEventElapsedTime(&ms, e0, e1);
        if (rep > 0 && ms > 0.f && flop / (ms * 1e-3) / 1e12 > best) best = flop / (ms * 1e-3) / 1e12;
    }
    if (e0) cudaEventDestroy(e0);
    if (e1) cudaEventDestroy(e1);
    if (scratch) cudaFree(scratch);
    *tflops = best;
    return rc;
}

// Equally strided stack of whole images that match the plan: srcs[k].data = srcs[0].data + k * sstride, dsts likewise,
// same pitch, dtype and channel count, strides positive whole rows (the grid.z kernels address the stack as one tall
// image) below 2^30 rows.  Shared by aai_run_device_batch and aai_run_device_adjoint.
static bool whole_image_stack(const aai_plan *plan, const aai_image *srcs, const aai_image *dsts, int n_images,
                              int64_t *sstride_out, int64_t *dstride_out) {
    const aai_image &s0 = srcs[0], &d0 = dsts[0];
    bool stack = n_images > 1 && images_match_plan(plan, &s0, &d0) && s0.y0 == 0 && s0.rows == s0.height &&
                 d0.y0 == 0 && d0.rows == d0.height;
    const int64_t sstride = stack ? (const char *)srcs[1].data - (const char *)s0.data : 0;
    const int64_t dstride = stack ? (const char *)dsts[1].data - (const char *)d0.data : 0;
    for (int k = 1; stack && k < n_images; ++k) {
        const aai_image &a = srcs[k], &b = dsts[k];
        stack = a.data == (const char *)s0.data + k * sstride && b.data == (char *)d0.data + k * dstride &&
                a.pitch_bytes == s0.pitch_bytes && b.pitch_bytes == d0.pitch_bytes && a.dtype == s0.dtype &&
                b.dtype == d0.dtype && a.width == s0.width && a.height == s0.height && a.y0 == 0 &&
                a.rows == a.height && b.width == d0.width && b.height == d0.height && b.y0 == 0 &&
                b.rows == b.height && a.channels == s0.channels && b.channels == d0.channels;
    }
    *sstride_out = sstride;
    *dstride_out = dstride;
    return stack && sstride > 0 && dstride > 0 && sstride % s0.pitch_bytes == 0 && dstride % d0.pitch_bytes == 0 &&
           sstride / s0.pitch_bytes < (1 << 30) && dstride / d0.pitch_bytes < (1 << 30);
}

int aai_run_device_batch(const aai_plan *plan, int mode, int arith, const aai_image *srcs, const aai_image *dsts,
                         int n_images, int device, void *stream) {
    if (!plan || !srcs || !dsts || n_images <= 0) {
        aai_set_error("aai_run_device_batch: bad argument");
        return AAI_ERR_ARGUMENT;
    }
    if (plan->status != AAI_OK) return plan->status;
    for (int k = 0; k < n_images; ++k)
        if (const int r = aai_check_dtype_pair("aai_run_device_batch", srcs[k].dtype, dsts[k].dtype)) return r;
    // One launch for the whole batch when the images form an equally strided stack of whole images: the separable TMA
    // kernel takes the stack as a rank-3 tensor (grid.y = image), every other kernel as grid.z = image.
    // (An unknown mode or arithmetic takes the per-image path, where aai_run_device refuses it.)
    const aai_image &s0 = srcs[0], &d0 = dsts[0];
    int64_t sstride = 0, dstride = 0;
    if (mode_ok(mode) && arith_ok(arith) && whole_image_stack(plan, srcs, dsts, n_images, &sstride, &dstride)) {
        AAI_CUDA(cudaSetDevice(device));
        const int64_t srows = sstride / s0.pitch_bytes, drows = dstride / d0.pitch_bytes;
        // images per launch: grid.y / grid.z limit, and row indices of the stack must stay below 2^31
        int64_t per_launch = 65535;
        const int64_t most_rows = srows > drows ? srows : drows;
        if (per_launch * most_rows > 0x7fffffffLL) per_launch = 0x7fffffffLL / most_rows;
        if (per_launch < 1) per_launch = 1;
        for (int first = 0; first < n_images; first += (int)per_launch) {
            const int n = n_images - first < per_launch ? n_images - first : (int)per_launch;
            AaiKernelParams kp = aai_make_kernel_params(*plan, srcs[first], dsts[first], 0, plan->dst_h);
            kp.quirk = mode == AAI_MODE_AREA_AVERAGE_EXACT ? 0 : 1;
            kp.batch = n;
            kp.src_batch_stride = sstride;
            kp.dst_batch_stride = dstride;
            kp.src_batch_rows = (int32_t)srows;
            kp.dst_batch_rows = (int32_t)drows;
            const int e = launch_rows(*plan, mode, arith, kp, s0.dtype, d0.dtype, stream);
            if (e != (int)cudaSuccess) return cuda_fail((cudaError_t)e, "batched kernel launch");
        }
        return AAI_OK;
    }
    for (int k = 0; k < n_images; ++k) {
        const int r = aai_run_device(plan, mode, arith, &srcs[k], &dsts[k], 0, plan->dst_h, device, stream);
        if (r != AAI_OK) return r;
    }
    return AAI_OK;
}

// Host-side argument checks of aai_run_device_adjoint, in the order the header lists them; no CUDA call
static int check_adjoint_args(const aai_plan *plan, int mode, const aai_image *canvas_grads, const aai_image *src_grads,
                              int n_images) {
    const char *who = "aai_run_device_adjoint";
    if (!plan || !canvas_grads || !src_grads || n_images <= 0) {
        aai_set_error("%s: null pointer or no images", who);
        return AAI_ERR_ARGUMENT;
    }
    if (plan->status != AAI_OK) return plan->status;
    if (!mode_ok(mode)) {
        aai_set_error("%s: interpolation mode must be 1, 2 or 3", who);
        return AAI_ERR_ARGUMENT;
    }
    for (int k = 0; k < n_images; ++k) {
        const aai_image &g = canvas_grads[k], &s = src_grads[k];
        if (!g.data || !s.data) {
            aai_set_error("%s: image %d has no data", who, k);
            return AAI_ERR_ARGUMENT;
        }
        if ((g.dtype != AAI_F32 && g.dtype != AAI_F64) || (s.dtype != AAI_F32 && s.dtype != AAI_F64) ||
            g.dtype != s.dtype) {
            aai_set_error("%s: gradients are float32 or float64, the same on both sides (image %d: canvas %s, source %s)",
                          who, k, aai_dtype_name(g.dtype), aai_dtype_name(s.dtype));
            return AAI_ERR_ARGUMENT;
        }
        if (g.channels != s.channels) {
            aai_set_error("%s: image %d: the canvas has %d channels, the source %d", who, k, (int)g.channels,
                          (int)s.channels);
            return AAI_ERR_ARGUMENT;
        }
        if (g.y0 != 0 || g.rows != g.height || s.y0 != 0 || s.rows != s.height) {
            aai_set_error("%s: image %d: whole images expected (y0 = 0, rows = height)", who, k);
            return AAI_ERR_ARGUMENT;
        }
        if (!images_match_plan(plan, &s, &g)) {
            aai_set_error("%s: image %d does not match the plan (source %lldx%lld, canvas %lldx%lld, 1-4 channels, "
                          "pitch >= row bytes)",
                          who, k, (long long)plan->src_w, (long long)plan->src_h, (long long)plan->dst_w,
                          (long long)plan->dst_h);
            return AAI_ERR_ARGUMENT;
        }
    }
    return AAI_OK;
}

int aai_run_device_adjoint(const aai_plan *plan, int mode, const aai_image *canvas_grads, const aai_image *src_grads,
                           int n_images, int device, void *stream) {
    if (const int r = check_adjoint_args(plan, mode, canvas_grads, src_grads, n_images)) return r;
    AAI_CUDA(cudaSetDevice(device));
    cudaStream_t st = (cudaStream_t)stream;
    const aai_image &s0 = src_grads[0], &g0 = canvas_grads[0];
    AaiAdjointParams ap;
    std::memset(&ap, 0, sizeof ap);
    ap.kp = aai_make_kernel_params(*plan, s0, g0, 0, plan->dst_h);
    ap.kp.quirk = mode == AAI_MODE_AREA_AVERAGE_EXACT ? 0 : 1;
    // 1/S_p in stream-ordered scratch: two calls in flight on different streams never share it
    const size_t rcp_bytes = (size_t)plan->dst_w * (size_t)plan->dst_h * sizeof(double);
    AAI_CUDA(cudaMallocAsync((void **)&ap.rcp, rcp_bytes, st));
    const char *what = "adjoint normaliser launch";
    int e = launch_slabs(0, plan->dst_h, [&](int64_t a, int64_t b) {
        ap.row0 = (int32_t)a;
        ap.row1 = (int32_t)b;
        return aai_launch_adjoint_norm(ap, mode, plan->axis_aligned, st);
    });
    ap.inv_side = 1.0 / plan->side;
    // gather over source rows, slab by slab; an equally strided stack is one launch per slab (grid.z = image).  Element
    // type and channel count are those of image `first`: a stack shares them (whole_image_stack), a list may mix them.
    auto gather = [&](int first, int n, int64_t canvas_stride, int64_t out_stride) {
        ap.kp.channels = src_grads[first].channels;
        ap.canvas = canvas_grads[first].data;
        ap.canvas_pitch = canvas_grads[first].pitch_bytes;
        ap.canvas_stride = canvas_stride;
        ap.out = src_grads[first].data;
        ap.out_pitch = src_grads[first].pitch_bytes;
        ap.out_stride = out_stride;
        return launch_slabs(0, plan->src_h, [&](int64_t a, int64_t b) {
            ap.row0 = (int32_t)a;
            ap.row1 = (int32_t)b;
            return aai_launch_adjoint_gather(ap, mode, plan->axis_aligned, src_grads[first].dtype, n, st);
        });
    };
    if (e == (int)cudaSuccess) {
        what = "adjoint gather launch";
        int64_t sstride = 0, cstride = 0;
        if (whole_image_stack(plan, src_grads, canvas_grads, n_images, &sstride, &cstride)) {
            for (int first = 0; first < n_images && e == (int)cudaSuccess; first += 65535)  // grid.z limit
                e = gather(first, n_images - first < 65535 ? n_images - first : 65535, cstride, sstride);
        } else {
            for (int k = 0; k < n_images && e == (int)cudaSuccess; ++k) e = gather(k, 1, 0, 0);
        }
    }
    const cudaError_t ef = cudaFreeAsync(ap.rcp, st);
    if (e != (int)cudaSuccess) return cuda_fail((cudaError_t)e, what);
    AAI_CUDA(ef);
    return AAI_OK;
}

int aai_run_host_band(const aai_plan *plan, int mode, int arith, const aai_image *src, const aai_image *dst,
                      int64_t row0, int64_t row1, int device, void *stream, int synchronize) {
    int r = check_host_images("aai_run_host_band", plan, src, dst, false);
    if (r != AAI_OK) return r;
    if (row0 < 0 || row1 > plan->dst_h || row0 > row1) {
        aai_set_error("aai_run_host_band: bad rows [%lld,%lld)", (long long)row0, (long long)row1);
        return AAI_ERR_ARGUMENT;
    }
    if (row1 == row0) return AAI_OK;
    if ((r = check_device("aai_run_host_band", device)) != AAI_OK) return r;
    int64_t sx0, sx1, sy0, sy1;
    aai_band_source_window(plan, row0, row1, &sx0, &sx1, &sy0, &sy1);
    aai_image dsrc = *src, ddst = *dst;
    dsrc.y0 = sy0;
    dsrc.rows = sy1 - sy0;
    dsrc.pitch_bytes = aai_device_pitch(src->width, src->channels, src->dtype);
    ddst.y0 = row0;
    ddst.rows = row1 - row0;
    ddst.pitch_bytes = aai_device_pitch(dst->width, dst->channels, dst->dtype);
    // Pipelined path for large bands: the canvas band is cut into chunks of rows; the source halo is uploaded
    // progressively (each source row once), chunk c's kernel starts as soon as its own halo has arrived and its rows
    // are downloaded while later chunks are still uploading / computing (PCIe is full duplex).  Three streams,
    // fork/joined on the caller's stream.  Needs page-locked host buffers to overlap; with pageable memory the copies
    // serialise but the result is the same.
    const size_t total_bytes = (size_t)dsrc.pitch_bytes * (size_t)dsrc.rows + (size_t)ddst.pitch_bytes * (size_t)ddst.rows;
    const int64_t band_rows = row1 - row0;
    int chunks = 1;
    if (total_bytes >= ((size_t)48 << 20) && band_rows >= 64) chunks = (int)(band_rows < 32 * 16 ? band_rows / 16 : 32);
#ifdef AAI_DEV_KNOBS  // developer builds only; the shipped library reads no environment
    if (const char *e = getenv("AAI_HOST_CHUNKS")) chunks = atoi(e) > 0 ? atoi(e) : chunks;
#endif
    if (chunks > band_rows) chunks = (int)band_rows;
    std::unique_lock<std::mutex> busy;
    Workspace *w = nullptr;
    cudaStream_t st = nullptr;
    r = pipeline_head(busy, device, (size_t)dsrc.pitch_bytes * (size_t)(dsrc.rows > 0 ? dsrc.rows : 1),
                      (size_t)ddst.pitch_bytes * (size_t)ddst.rows, stream, chunks > 1 ? 2 * chunks : 0, &w, &st);
    if (r != AAI_OK) return r;
    dsrc.data = w->ptr[0];
    ddst.data = w->ptr[1];
    if (chunks <= 1) {
        if (dsrc.rows > 0) {
            r = aai_image_upload(&dsrc, src, device, st);
            if (r != AAI_OK) return r;
        }
        AAI_CUDA(cudaEventRecord(w->ev[1], st));
        r = aai_run_device(plan, mode, arith, &dsrc, &ddst, row0, row1, device, st);
        if (r != AAI_OK) return r;
        AAI_CUDA(cudaEventRecord(w->ev[2], st));
        r = aai_image_download(dst, &ddst, device, st);
        if (r != AAI_OK) return r;
        return pipeline_tail(w, st, false, synchronize || !stream);
    }
    cudaStream_t s_k = st;  // kernels run on the caller's stream itself
    int64_t have_lo = 0, have_hi = 0;  // source rows [have_lo, have_hi) already queued for upload
    bool have_any = false;
    auto upload_rows = [&](int64_t a, int64_t b) -> int {
        if (b <= a) return AAI_OK;
        aai_image part = dsrc;
        part.data = (char *)dsrc.data + (a - dsrc.y0) * dsrc.pitch_bytes;
        part.y0 = a;
        part.rows = b - a;
        return aai_image_upload(&part, src, device, w->up);
    };
    for (int c = 0; c < chunks; ++c) {
        const int64_t r0 = row0 + band_rows * c / chunks, r1 = row0 + band_rows * (c + 1) / chunks;
        int64_t cx0, cx1, a, b;
        aai_band_source_window(plan, r0, r1, &cx0, &cx1, &a, &b);
        if (b > a) {
            if (!have_any) {
                r = upload_rows(a, b);
                have_lo = a;
                have_hi = b;
                have_any = true;
            } else {
                r = AAI_OK;
                if (a < have_lo) {
                    r = upload_rows(a, have_lo);
                    have_lo = a;
                }
                if (r == AAI_OK && b > have_hi) {
                    r = upload_rows(have_hi, b);
                    have_hi = b;
                }
            }
            if (r != AAI_OK) return r;
        }
        AAI_CUDA(cudaEventRecord(w->chunk_ev[2 * c], w->up));
        AAI_CUDA(cudaStreamWaitEvent(s_k, w->chunk_ev[2 * c], 0));
        r = aai_run_device(plan, mode, arith, &dsrc, &ddst, r0, r1, device, s_k);
        if (r != AAI_OK) return r;
        AAI_CUDA(cudaEventRecord(w->chunk_ev[2 * c + 1], s_k));
        AAI_CUDA(cudaStreamWaitEvent(w->dn, w->chunk_ev[2 * c + 1], 0));
        aai_image part = ddst;
        part.data = (char *)ddst.data + (r0 - ddst.y0) * ddst.pitch_bytes;
        part.y0 = r0;
        part.rows = r1 - r0;
        r = aai_image_download(dst, &part, device, w->dn);
        if (r != AAI_OK) return r;
    }
    return pipeline_tail(w, st, true, synchronize || !stream);
}

int aai_run_host_batch(const aai_plan *plan, int mode, int arith, const aai_image *srcs, const aai_image *dsts,
                       int n_images, int device, void *stream, int synchronize) {
    if (!plan || !srcs || !dsts || n_images <= 0) {
        aai_set_error("aai_run_host_batch: bad argument");
        return AAI_ERR_ARGUMENT;
    }
    for (int k = 0; k < n_images; ++k) {
        const int r = check_host_images("aai_run_host_batch", plan, &srcs[k], &dsts[k], true);
        if (r != AAI_OK) return r;
        if (srcs[k].dtype != srcs[0].dtype || dsts[k].dtype != dsts[0].dtype || srcs[k].channels != srcs[0].channels) {
            aai_set_error("aai_run_host_batch: the images of a batch must share element types and channel count");
            return AAI_ERR_ARGUMENT;
        }
    }
    if (const int r = check_device("aai_run_host_batch", device)) return r;
    // Ring of kRing groups of `per` slices each in the device workspace: group i is uploaded (one copy per slice),
    // resampled with ONE batched launch and downloaded, on three streams; its buffers are reused by group i + kRing
    // once its kernel (source buffers) resp. its download (canvas buffers) has finished.
    constexpr int kRing = 3;
    aai_image ds = srcs[0], dd = dsts[0];
    ds.pitch_bytes = aai_device_pitch(ds.width, ds.channels, ds.dtype);
    dd.pitch_bytes = aai_device_pitch(dd.width, dd.channels, dd.dtype);
    const size_t s_bytes = (size_t)ds.pitch_bytes * (size_t)ds.height, d_bytes = (size_t)dd.pitch_bytes * (size_t)dd.height;
    int per = (int)(((size_t)192 << 20) / (s_bytes + d_bytes));
    per = per < 1 ? 1 : (per > 16 ? 16 : per);
    if (per > n_images) per = n_images;
    const int groups = (n_images + per - 1) / per;
    std::unique_lock<std::mutex> busy;
    Workspace *w = nullptr;
    cudaStream_t st = nullptr;
    int r = pipeline_head(busy, device, s_bytes * (size_t)per * kRing, d_bytes * (size_t)per * kRing, stream,
                          3 * kRing, &w, &st);
    if (r != AAI_OK) return r;
    std::vector<aai_image> gs((size_t)per), gd((size_t)per);
    for (int g = 0; g < groups; ++g) {
        const int slot = g % kRing, first = g * per, n = n_images - first < per ? n_images - first : per;
        cudaEvent_t up_done = w->chunk_ev[3 * slot], k_done = w->chunk_ev[3 * slot + 1], dn_done = w->chunk_ev[3 * slot + 2];
        if (g >= kRing) {  // the slot's previous occupant: its kernel has read the sources, its download the canvases
            AAI_CUDA(cudaStreamWaitEvent(w->up, k_done, 0));
            AAI_CUDA(cudaStreamWaitEvent(st, dn_done, 0));
        }
        for (int k = 0; k < n; ++k) {
            gs[(size_t)k] = ds;
            gs[(size_t)k].data = (char *)w->ptr[0] + ((size_t)slot * per + k) * s_bytes;
            gd[(size_t)k] = dd;
            gd[(size_t)k].data = (char *)w->ptr[1] + ((size_t)slot * per + k) * d_bytes;
            r = aai_image_upload(&gs[(size_t)k], &srcs[first + k], device, w->up);
            if (r != AAI_OK) return r;
        }
        AAI_CUDA(cudaEventRecord(up_done, w->up));
        AAI_CUDA(cudaStreamWaitEvent(st, up_done, 0));
        r = aai_run_device_batch(plan, mode, arith, gs.data(), gd.data(), n, device, st);
        if (r != AAI_OK) return r;
        AAI_CUDA(cudaEventRecord(k_done, st));
        AAI_CUDA(cudaStreamWaitEvent(w->dn, k_done, 0));
        for (int k = 0; k < n; ++k) {
            r = aai_image_download(&dsts[first + k], &gd[(size_t)k], device, w->dn);
            if (r != AAI_OK) return r;
        }
        AAI_CUDA(cudaEventRecord(dn_done, w->dn));
    }
    return pipeline_tail(w, st, true, synchronize || !stream);
}

int aai_run_host(const aai_plan *plan, int mode, int arith, const aai_image *src, const aai_image *dst,
                 const int *devices, int n_devices) {
    int rc = check_host_images("aai_run_host", plan, src, dst, true);
    if (rc != AAI_OK) return rc;
    const int dev0 = 0;
    if (!devices || n_devices <= 0) {
        devices = &dev0;
        n_devices = 1;
    }
    const int have = aai_device_count();
    if (have <= 0) {
        aai_set_error("aai_run_host: no CUDA device; this library has no CPU fallback");
        return AAI_ERR_NO_DEVICE;
    }
    for (int k = 0; k < n_devices; ++k)
        if (devices[k] < 0 || devices[k] >= have) {
            aai_set_error("aai_run_host: device %d not present (%d devices)", devices[k], have);
            return AAI_ERR_ARGUMENT;
        }
    std::vector<int64_t> bounds((size_t)n_devices + 1);
    rc = aai_partition_rows_weighted(plan, n_devices, aai_band_empty_weight(plan, mode, arith), bounds.data());
    if (rc != AAI_OK) return rc;
    if (n_devices == 1) return aai_run_host_band(plan, mode, arith, src, dst, 0, plan->dst_h, devices[0], nullptr, 1);

    // one host thread per device: pageable-memory copies block their issuing thread
    std::vector<int> status((size_t)n_devices, AAI_OK);
    std::vector<std::string> messages((size_t)n_devices);
    std::vector<float> t_h2d((size_t)n_devices, 0.f), t_k((size_t)n_devices, 0.f), t_d2h((size_t)n_devices, 0.f);
    std::vector<std::thread> pool;
    for (int k = 0; k < n_devices; ++k)
        pool.emplace_back([&, k]() {
            status[(size_t)k] = aai_run_host_band(plan, mode, arith, src, dst, bounds[(size_t)k],
                                                  bounds[(size_t)k + 1], devices[k], nullptr, 1);
            if (status[(size_t)k] != AAI_OK) messages[(size_t)k] = g_error;
            t_h2d[(size_t)k] = g_h2d_ms;
            t_k[(size_t)k] = g_kernel_ms;
            t_d2h[(size_t)k] = g_d2h_ms;
        });
    for (auto &t : pool) t.join();
    for (int k = 0; k < n_devices; ++k)
        if (status[(size_t)k] != AAI_OK) {
            aai_set_error("device %d: %s", devices[k], messages[(size_t)k].c_str());
            return status[(size_t)k];
        }
    g_h2d_ms = g_kernel_ms = g_d2h_ms = 0.f;
    for (int k = 0; k < n_devices; ++k) {
        g_h2d_ms = std::fmax(g_h2d_ms, t_h2d[(size_t)k]);
        g_kernel_ms = std::fmax(g_kernel_ms, t_k[(size_t)k]);
        g_d2h_ms = std::fmax(g_d2h_ms, t_d2h[(size_t)k]);
    }
    return AAI_OK;
}

int aai_last_host_timing(float *h2d_ms, float *kernel_ms, float *d2h_ms) {
    if (g_kernel_ms < 0.f) return AAI_ERR_ARGUMENT;
    if (h2d_ms) *h2d_ms = g_h2d_ms;
    if (kernel_ms) *kernel_ms = g_kernel_ms;
    if (d2h_ms) *d2h_ms = g_d2h_ms;
    return AAI_OK;
}

}  // extern "C"
