// Peer group (include/aai.h): ONE large image resampled by one process per GPU, end to end from host buffers.
//
// Every source row crosses PCIe once (its owner rank uploads it, in chunks, into the owner's full-size device image);
// the rows of a band's halo that the rank does not own are pulled out of the owners' device images over NVLink (CUDA IPC
// memory mappings) as the chunks land.  The ranks synchronise through two monotonic counters per rank in a POSIX
// shared-memory page -- "upload chunks landed" and "steps whose pulls are complete" -- driven by the host: the calling
// thread polls its own upload events (cudaEventQuery) and publishes them, polls the owners' counters and enqueues each
// pull the moment its chunk has landed.  (A first version expressed the same dependencies with interprocess CUDA
// events waited on by the copy streams; measured on 8 B200s every such wait cost milliseconds -- 13.3 ms per step
// against 9.0 ms for round 1's barrier scheme -- so the device-side waits were dropped; profiles/README.md.)
// No NCCL, no barrier: the bands are independent (SURVEY.md §8e; the reference's loop nest Source.cpp:413-415 has no
// cross-pixel dependency).
#include <cuda_runtime.h>
#include <fcntl.h>
#include <sched.h>
#include <sys/mman.h>
#include <unistd.h>

#include <atomic>
#include <chrono>
#include <cstdio>
#include <cstring>
#include <new>
#include <vector>

#include "aai_internal.h"

namespace {

constexpr int kMaxChunks = 8;         // upload chunks per owner (an IPC event each)
constexpr uint32_t kMagic = 0x41414950;  // "AAIP"
constexpr double kHostWaitSeconds = 60.0;

struct PeerShm {  // one page of POSIX shared memory per rank
    std::atomic<uint64_t> landed;  // upload chunks of this rank that have arrived in its device image, over all steps
    std::atomic<uint64_t> pulled;  // last step whose halo pulls this rank has completed (its peers' rows may be reused)
};

#pragma pack(push, 1)
struct Blob {
    uint32_t magic;
    int32_t rank, world, n_chunks;
    int64_t pitch;
    cudaIpcMemHandle_t mem;
    char shm_name[64];
};
#pragma pack(pop)
static_assert(sizeof(Blob) <= AAI_PEER_BLOB_BYTES, "blob size");

struct Remote {  // what this rank knows about rank p
    void *full = nullptr;                 // p's device image, mapped here (nullptr for p == rank)
    PeerShm *shm = nullptr;
    int n_chunks = 0;
    int64_t y0 = 0, y1 = 0;               // rows p owns
};

}  // namespace

struct aai_peer {
    aai_plan plan;
    int32_t dtype = 0, channels = 0;
    int rank = 0, world = 1, device = 0;
    int64_t row0 = 0, row1 = 0;          // canvas band of this rank
    int64_t halo_y0 = 0, halo_y1 = 0;    // source rows the band can touch
    aai_image full{};                    // own device image (all rows allocated)
    aai_image band{};                    // device canvas band (allocated by the first step)
    cudaStream_t own = nullptr, up = nullptr, pl = nullptr, dn = nullptr;
    cudaEvent_t fork = nullptr, join_up = nullptr, join_pl = nullptr, join_dn = nullptr, k_last = nullptr;
    cudaEvent_t t_fork = nullptr, t_up = nullptr, t_pl = nullptr, t_k = nullptr, t_dn = nullptr;  // phase timing of the last step
    bool timed = false;
    cudaEvent_t landed[kMaxChunks] = {};  // own upload chunks
    cudaEvent_t pulled = nullptr;         // own "pulls of this step are done"
    std::vector<cudaEvent_t> op_ev, k_ev;  // local: after each pull op / each kernel chunk
    PeerShm *shm = nullptr;
    char shm_name[64] = "";
    std::vector<Remote> remote;
    uint64_t step = 0;
    bool connected = false;
};

namespace {

int fail(cudaError_t e, const char *what) {
    aai_set_error("%s: %s (%s)", what, cudaGetErrorString(e), cudaGetErrorName(e));
    return AAI_ERR_CUDA;
}
#define PEER_CUDA(call)                                \
    do {                                               \
        cudaError_t e_ = (call);                       \
        if (e_ != cudaSuccess) return fail(e_, #call); \
    } while (0)

void owned_rows(int64_t h, int world, int p, int64_t &y0, int64_t &y1) {
    y0 = h * p / world;
    y1 = h * (p + 1) / world;
}

// upload chunks of an owner: four (so that the pulls of the first quarters overlap the upload of the later ones), fewer
// when that would make them smaller than 8 MB -- every chunk costs an interprocess event wait per reader, and at 8 ranks
// the uploads of all owners run concurrently anyway; every rank computes the same split
std::atomic<int> g_upload_chunks{4};
int chunk_count(int64_t rows, int64_t row_bytes) {
    if (rows <= 0) return 0;
    int64_t n = rows * row_bytes / (8 << 20);
    if (n < 1) n = 1;
    if (n > g_upload_chunks.load()) n = g_upload_chunks.load();
    if (n > kMaxChunks) n = kMaxChunks;
    if (n > rows) n = rows;
    return (int)n;
}
void chunk_rows(int64_t y0, int64_t y1, int n, int c, int64_t &a, int64_t &b) {
    a = y0 + (y1 - y0) * c / n;
    b = y0 + (y1 - y0) * (c + 1) / n;
}

bool host_wait(const std::atomic<uint64_t> &v, uint64_t want) {
    const auto t0 = std::chrono::steady_clock::now();
    for (int spin = 0; v.load(std::memory_order_acquire) < want; ++spin) {
        if ((spin & 1023) == 1023) {
            sched_yield();
            if (std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count() > kHostWaitSeconds)
                return false;
        }
    }
    return true;
}

}  // namespace

extern "C" {

int aai_peer_upload_chunks(int n) {
    if (n >= 1 && n <= kMaxChunks) g_upload_chunks.store(n);
    return g_upload_chunks.load();
}

int aai_peer_create(const aai_plan *plan, int32_t dtype, int32_t channels, int rank, int world_size, int device,
                    aai_peer **out) {
    if (!plan || !out || !aai_elem_size(dtype) || channels < 1 || channels > 4 || world_size < 1 || rank < 0 ||
        rank >= world_size) {
        aai_set_error("aai_peer_create: bad argument");
        return AAI_ERR_ARGUMENT;
    }
    if (plan->status != AAI_OK) return plan->status;
    PEER_CUDA(cudaSetDevice(device));
    aai_peer *g = new (std::nothrow) aai_peer();
    if (!g) return AAI_ERR_ARGUMENT;
    g->plan = *plan;
    g->dtype = dtype;
    g->channels = channels;
    g->rank = rank;
    g->world = world_size;
    g->device = device;
    std::vector<int64_t> bounds((size_t)world_size + 1);
    int rc = aai_partition_rows(plan, world_size, bounds.data());
    if (rc != AAI_OK) {
        delete g;
        return rc;
    }
    g->row0 = bounds[(size_t)rank];
    g->row1 = bounds[(size_t)rank + 1];
    int64_t sx0, sx1;
    aai_band_source_window(plan, g->row0, g->row1, &sx0, &sx1, &g->halo_y0, &g->halo_y1);
    rc = aai_image_alloc(&g->full, device, plan->src_w, plan->src_h, 0, plan->src_h, dtype, channels);
    if (rc != AAI_OK) {
        aai_peer_destroy(g);
        return rc;
    }
    cudaError_t e = cudaSuccess;
    auto ok = [&](cudaError_t r) {
        if (e == cudaSuccess) e = r;
    };
    ok(cudaStreamCreateWithFlags(&g->own, cudaStreamNonBlocking));
    ok(cudaStreamCreateWithFlags(&g->up, cudaStreamNonBlocking));
    ok(cudaStreamCreateWithFlags(&g->pl, cudaStreamNonBlocking));
    ok(cudaStreamCreateWithFlags(&g->dn, cudaStreamNonBlocking));
    for (cudaEvent_t *ev : {&g->fork, &g->join_up, &g->join_pl, &g->join_dn, &g->k_last})
        ok(cudaEventCreateWithFlags(ev, cudaEventDisableTiming));
    for (cudaEvent_t *ev : {&g->t_fork, &g->t_up, &g->t_pl, &g->t_k, &g->t_dn}) ok(cudaEventCreate(ev));
    for (int c = 0; c < kMaxChunks; ++c) ok(cudaEventCreateWithFlags(&g->landed[c], cudaEventDisableTiming));
    ok(cudaEventCreateWithFlags(&g->pulled, cudaEventDisableTiming));
    if (e != cudaSuccess) {
        aai_peer_destroy(g);
        return fail(e, "aai_peer_create: streams / events");
    }
    // the page of host counters the other ranks poll
    static std::atomic<unsigned> serial{0};
    std::snprintf(g->shm_name, sizeof g->shm_name, "/aai_peer_%d_%d_%u", (int)getpid(), rank, serial.fetch_add(1));
    const int fd = shm_open(g->shm_name, O_CREAT | O_EXCL | O_RDWR, 0600);
    if (fd < 0 || ftruncate(fd, 4096) != 0) {
        if (fd >= 0) close(fd);
        aai_set_error("aai_peer_create: cannot create the shared-memory page %s", g->shm_name);
        g->shm_name[0] = 0;
        aai_peer_destroy(g);
        return AAI_ERR_CUDA;
    }
    void *m = mmap(nullptr, 4096, PROT_READ | PROT_WRITE, MAP_SHARED, fd, 0);
    close(fd);
    if (m == MAP_FAILED) {
        aai_set_error("aai_peer_create: mmap of %s failed", g->shm_name);
        aai_peer_destroy(g);
        return AAI_ERR_CUDA;
    }
    g->shm = new (m) PeerShm();
    g->shm->landed.store(0);
    g->shm->pulled.store(0);
    *out = g;
    return AAI_OK;
}

int aai_peer_export(aai_peer *g, unsigned char blob[AAI_PEER_BLOB_BYTES]) {
    if (!g || !blob) return AAI_ERR_ARGUMENT;
    PEER_CUDA(cudaSetDevice(g->device));
    Blob b;
    std::memset(&b, 0, sizeof b);
    b.magic = kMagic;
    b.rank = g->rank;
    b.world = g->world;
    int64_t y0, y1;
    owned_rows(g->plan.src_h, g->world, g->rank, y0, y1);
    b.n_chunks = chunk_count(y1 - y0, g->plan.src_w * g->channels * (int64_t)aai_elem_size(g->dtype));
    b.pitch = g->full.pitch_bytes;
    PEER_CUDA(cudaIpcGetMemHandle(&b.mem, g->full.data));
    std::memcpy(b.shm_name, g->shm_name, sizeof b.shm_name);
    std::memset(blob, 0, AAI_PEER_BLOB_BYTES);
    std::memcpy(blob, &b, sizeof b);
    return AAI_OK;
}

int aai_peer_connect(aai_peer *g, const unsigned char *blobs) {
    if (!g || !blobs || g->connected) {
        aai_set_error("aai_peer_connect: bad argument or already connected");
        return AAI_ERR_ARGUMENT;
    }
    PEER_CUDA(cudaSetDevice(g->device));
    g->remote.assign((size_t)g->world, Remote());
    const int64_t row_bytes = g->plan.src_w * g->channels * (int64_t)aai_elem_size(g->dtype);
    for (int p = 0; p < g->world; ++p) {
        Blob b;
        std::memcpy(&b, blobs + (size_t)p * AAI_PEER_BLOB_BYTES, sizeof b);
        Remote &r = g->remote[(size_t)p];
        owned_rows(g->plan.src_h, g->world, p, r.y0, r.y1);
        r.n_chunks = chunk_count(r.y1 - r.y0, row_bytes);
        if (b.magic != kMagic || b.rank != p || b.world != g->world || b.n_chunks != r.n_chunks ||
            b.pitch != g->full.pitch_bytes) {
            aai_set_error("aai_peer_connect: blob %d does not belong to this group (rank %d of %d, %d chunks, pitch %lld)",
                          p, b.rank, b.world, b.n_chunks, (long long)b.pitch);
            return AAI_ERR_ARGUMENT;
        }
        if (p == g->rank) {
            r.shm = g->shm;
            continue;
        }
        PEER_CUDA(cudaIpcOpenMemHandle(&r.full, b.mem, cudaIpcMemLazyEnablePeerAccess));
        const int fd = shm_open(b.shm_name, O_RDWR, 0600);
        void *m = fd >= 0 ? mmap(nullptr, 4096, PROT_READ | PROT_WRITE, MAP_SHARED, fd, 0) : MAP_FAILED;
        if (fd >= 0) close(fd);
        if (m == MAP_FAILED) {
            aai_set_error("aai_peer_connect: cannot map the shared-memory page %s of rank %d", b.shm_name, p);
            return AAI_ERR_CUDA;
        }
        r.shm = reinterpret_cast<PeerShm *>(m);
    }
    g->connected = true;
    return AAI_OK;
}

int aai_peer_owned_rows(const aai_peer *g, int64_t *y0, int64_t *y1) {
    if (!g) return AAI_ERR_ARGUMENT;
    int64_t a, b;
    owned_rows(g->plan.src_h, g->world, g->rank, a, b);
    if (y0) *y0 = a;
    if (y1) *y1 = b;
    return AAI_OK;
}

int aai_peer_band(const aai_peer *g, int64_t *row0, int64_t *row1) {
    if (!g) return AAI_ERR_ARGUMENT;
    if (row0) *row0 = g->row0;
    if (row1) *row1 = g->row1;
    return AAI_OK;
}

int aai_peer_device_source(const aai_peer *g, aai_image *out) {
    if (!g || !out) return AAI_ERR_ARGUMENT;
    *out = g->full;
    return AAI_OK;
}

int aai_peer_run(aai_peer *g, int mode, int arith, const aai_image *hsrc, const aai_image *hdst, void *stream,
                 int synchronize) {
    // (the element-type pair first: refused alike on every rank, whatever the state of its group)
    if (hsrc && hdst)
        if (const int r = aai_check_dtype_pair("aai_peer_run", hsrc->dtype, hdst->dtype)) return r;
    if (!g || !g->connected || !hsrc || !hdst || !hsrc->data || !hdst->data) {
        aai_set_error("aai_peer_run: group not connected or null image");
        return AAI_ERR_ARGUMENT;
    }
    const aai_plan &plan = g->plan;
    int64_t oy0, oy1;
    owned_rows(plan.src_h, g->world, g->rank, oy0, oy1);
    const int64_t row_bytes = plan.src_w * g->channels * (int64_t)aai_elem_size(g->dtype);
    const int64_t dst_row_bytes = plan.dst_w * g->channels * (int64_t)aai_elem_size(hdst->dtype);
    if (hsrc->width != plan.src_w || hsrc->height != plan.src_h || hsrc->dtype != g->dtype ||
        hsrc->channels != g->channels || hsrc->y0 > oy0 || hsrc->y0 + hsrc->rows < oy1 ||
        hsrc->pitch_bytes < row_bytes || hdst->width != plan.dst_w || hdst->height != plan.dst_h ||
        !aai_elem_size(hdst->dtype) || hdst->channels != g->channels || hdst->y0 > g->row0 ||
        hdst->y0 + hdst->rows < g->row1 || hdst->pitch_bytes < dst_row_bytes) {
        aai_set_error("aai_peer_run: host images must hold the owned source rows [%lld,%lld) and the canvas band [%lld,%lld)",
                      (long long)oy0, (long long)oy1, (long long)g->row0, (long long)g->row1);
        return AAI_ERR_ARGUMENT;
    }
    PEER_CUDA(cudaSetDevice(g->device));
    if (g->row1 > g->row0 && (!g->band.data || g->band.dtype != hdst->dtype)) {  // device canvas band, (re)allocated lazily
        if (g->band.data) {
            PEER_CUDA(cudaDeviceSynchronize());
            PEER_CUDA(cudaFree(g->band.data));
            g->band.data = nullptr;
        }
        const int rc = aai_image_alloc(&g->band, g->device, plan.dst_w, plan.dst_h, g->row0, g->row1 - g->row0,
                                       hdst->dtype, g->channels);
        if (rc != AAI_OK) return rc;
    }
    const uint64_t s = ++g->step;
    cudaStream_t st = stream ? (cudaStream_t)stream : g->own;
    // The copy streams start as soon as the previous step's KERNELS have finished (they were the last readers of the
    // device image) -- not after its downloads: PCIe is full duplex, so this step's uploads overlap the previous step's
    // device-to-host copies.  (Host buffers are read / written when the copies execute; the caller's stream orders only
    // the kernels and the completion of `host_dst`.)  The first step starts after everything queued on the caller's stream.
    if (s == 1) {
        PEER_CUDA(cudaEventRecord(g->fork, st));
        for (cudaStream_t q : {g->up, g->pl}) PEER_CUDA(cudaStreamWaitEvent(q, g->fork, 0));
    } else {
        for (cudaStream_t q : {g->up, g->pl}) PEER_CUDA(cudaStreamWaitEvent(q, g->k_last, 0));
    }
    PEER_CUDA(cudaEventRecord(g->t_fork, g->up));  // phase times count from the moment this step's upload may start

    // 1. my rows may be overwritten once every reader has finished pulling them in the previous step
    if (s > 1)
        for (int p = 0; p < g->world; ++p) {
            if (p == g->rank) continue;
            if (!host_wait(g->remote[(size_t)p].shm->pulled, s - 1)) {
                aai_set_error("aai_peer_run: rank %d did not complete step %llu", p, (unsigned long long)(s - 1));
                return AAI_ERR_CUDA;
            }
        }
    // 2. upload my rows, chunk by chunk, an event after each
    const Remote &me = g->remote[(size_t)g->rank];
    for (int c = 0; c < me.n_chunks; ++c) {
        int64_t a, b;
        chunk_rows(oy0, oy1, me.n_chunks, c, a, b);
        PEER_CUDA(aai_copy_pitched((char *)g->full.data + a * g->full.pitch_bytes, g->full.pitch_bytes,
                                   (const char *)hsrc->data + (a - hsrc->y0) * hsrc->pitch_bytes, hsrc->pitch_bytes,
                                   (size_t)row_bytes, b - a, cudaMemcpyHostToDevice, g->up));
        PEER_CUDA(cudaEventRecord(g->landed[c], g->up));
    }
    PEER_CUDA(cudaEventRecord(g->t_up, g->up));

    // 3. progress loop (host driven): publish my chunks as they land; enqueue the pull of every chunk of my halo that
    //    other ranks own the moment its owner has published it.  Remember after which op each source row range is complete.
    struct Op {
        int64_t a, b;   // source rows this op completes
        int own_chunk;  // >= 0: one of my own upload chunks (no copy, the kernel waits on its event); < 0: pull -1 - index
    };
    std::vector<Op> ops;
    std::vector<int> next((size_t)g->world, 0);  // next chunk of owner p to pull
    for (int c = 0; c < me.n_chunks; ++c) {      // my own rows inside my halo: the kernels wait on the upload events
        int64_t a, b;
        chunk_rows(oy0, oy1, me.n_chunks, c, a, b);
        a = std::max(a, g->halo_y0);
        b = std::min(b, g->halo_y1);
        if (b > a) ops.push_back({a, b, c});
    }
    size_t n_pull = 0;
    int published = 0, remaining = 0;
    for (int p = 0; p < g->world; ++p) {
        const Remote &r = g->remote[(size_t)p];
        if (p == g->rank || std::max(r.y0, g->halo_y0) >= std::min(r.y1, g->halo_y1)) next[(size_t)p] = r.n_chunks;
        remaining += r.n_chunks - next[(size_t)p];
    }
    const auto t0 = std::chrono::steady_clock::now();
    for (unsigned spin = 0; published < me.n_chunks || remaining > 0; ++spin) {
        bool progressed = false;
        while (published < me.n_chunks) {
            const cudaError_t q = cudaEventQuery(g->landed[published]);
            if (q == cudaErrorNotReady) break;
            if (q != cudaSuccess) return fail(q, "aai_peer_run: upload");
            ++published;
            g->shm->landed.store((s - 1) * (uint64_t)me.n_chunks + (uint64_t)published, std::memory_order_release);
            progressed = true;
        }
        for (int p = 0; p < g->world; ++p) {
            const Remote &r = g->remote[(size_t)p];
            while (next[(size_t)p] < r.n_chunks &&
                   r.shm->landed.load(std::memory_order_acquire) >= (s - 1) * (uint64_t)r.n_chunks + (uint64_t)next[(size_t)p] + 1) {
                const int c = next[(size_t)p]++;
                --remaining;
                progressed = true;
                int64_t a, b;
                chunk_rows(r.y0, r.y1, r.n_chunks, c, a, b);
                a = std::max(a, g->halo_y0);
                b = std::min(b, g->halo_y1);
                if (b <= a) continue;
                PEER_CUDA(aai_copy_pitched((char *)g->full.data + a * g->full.pitch_bytes, g->full.pitch_bytes,
                                           (const char *)r.full + a * g->full.pitch_bytes, g->full.pitch_bytes,
                                           (size_t)row_bytes, b - a, cudaMemcpyDefault, g->pl));
                PEER_CUDA(aai_grow_events(g->op_ev, n_pull + 1));
                PEER_CUDA(cudaEventRecord(g->op_ev[n_pull], g->pl));
                ops.push_back({a, b, -1 - (int)n_pull});
                ++n_pull;
            }
        }
        if (!progressed && (spin & 63) == 63) {
            sched_yield();
            if (std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count() > kHostWaitSeconds) {
                aai_set_error("aai_peer_run: step %llu timed out waiting for the uploads of the other ranks",
                              (unsigned long long)s);
                return AAI_ERR_CUDA;
            }
        }
    }
    PEER_CUDA(cudaEventRecord(g->pulled, g->pl));
    PEER_CUDA(cudaEventRecord(g->t_pl, g->pl));

    // 4. kernels + downloads, chunk by chunk, each kernel after the last op that completes a row range it reads
    const int64_t band_rows = g->row1 - g->row0;
    int chunks = band_rows >= 64 ? (int)std::min<int64_t>(8, band_rows / 16) : 1;
    if (band_rows <= 0) chunks = 0;
    PEER_CUDA(aai_grow_events(g->k_ev, (size_t)chunks));
    std::vector<char> waited(ops.size(), 0);
    for (int j = 0; j < chunks; ++j) {
        const int64_t r0 = g->row0 + band_rows * j / chunks, r1 = g->row0 + band_rows * (j + 1) / chunks;
        int64_t cx0, cx1, a, b;
        aai_band_source_window(&plan, r0, r1, &cx0, &cx1, &a, &b);
        for (size_t k = 0; k < ops.size(); ++k) {
            if (waited[k] || std::max(ops[k].a, a) >= std::min(ops[k].b, b)) continue;
            waited[k] = 1;  // (stream order: later kernel chunks inherit the wait)
            cudaEvent_t e = ops[k].own_chunk >= 0 ? g->landed[ops[k].own_chunk] : g->op_ev[(size_t)(-1 - ops[k].own_chunk)];
            PEER_CUDA(cudaStreamWaitEvent(st, e, 0));
        }
        const int rc = aai_run_device(&plan, mode, arith, &g->full, &g->band, r0, r1, g->device, st);
        if (rc != AAI_OK) return rc;
        PEER_CUDA(cudaEventRecord(g->k_ev[(size_t)j], st));
        PEER_CUDA(cudaStreamWaitEvent(g->dn, g->k_ev[(size_t)j], 0));
        PEER_CUDA(aai_copy_pitched((char *)hdst->data + (r0 - hdst->y0) * hdst->pitch_bytes, hdst->pitch_bytes,
                                   (const char *)g->band.data + (r0 - g->row0) * g->band.pitch_bytes,
                                   g->band.pitch_bytes, (size_t)dst_row_bytes, r1 - r0, cudaMemcpyDeviceToHost, g->dn));
    }
    PEER_CUDA(cudaEventRecord(g->t_k, st));
    PEER_CUDA(cudaEventRecord(g->k_last, st));
    PEER_CUDA(cudaEventRecord(g->t_dn, g->dn));
    g->timed = true;
    // my pulls are complete: the owners may overwrite their rows (their next step waits for this counter)
    PEER_CUDA(cudaEventSynchronize(g->pulled));
    g->shm->pulled.store(s, std::memory_order_release);
    // join: the caller's stream continues after the uploads, the pulls and the downloads
    PEER_CUDA(cudaEventRecord(g->join_up, g->up));
    PEER_CUDA(cudaEventRecord(g->join_pl, g->pl));
    PEER_CUDA(cudaEventRecord(g->join_dn, g->dn));
    PEER_CUDA(cudaStreamWaitEvent(st, g->join_up, 0));
    PEER_CUDA(cudaStreamWaitEvent(st, g->join_pl, 0));
    PEER_CUDA(cudaStreamWaitEvent(st, g->join_dn, 0));
    if (synchronize || !stream) PEER_CUDA(cudaStreamSynchronize(st));
    return AAI_OK;
}

int aai_peer_last_timing(aai_peer *g, float ms[4]) {
    if (!g || !ms || !g->timed) return AAI_ERR_ARGUMENT;
    PEER_CUDA(cudaSetDevice(g->device));
    cudaEvent_t ev[4] = {g->t_up, g->t_pl, g->t_k, g->t_dn};
    for (int k = 0; k < 4; ++k) {
        PEER_CUDA(cudaEventSynchronize(ev[k]));
        PEER_CUDA(cudaEventElapsedTime(&ms[k], g->t_fork, ev[k]));
    }
    return AAI_OK;
}

int aai_peer_destroy(aai_peer *g) {
    if (!g) return AAI_OK;
    cudaSetDevice(g->device);
    cudaDeviceSynchronize();
    for (int p = 0; p < (int)g->remote.size(); ++p) {
        Remote &r = g->remote[(size_t)p];
        if (p == g->rank) continue;
        if (r.full) cudaIpcCloseMemHandle(r.full);
        if (r.shm) munmap(r.shm, 4096);
    }
    for (cudaEvent_t e : g->landed)
        if (e) cudaEventDestroy(e);
    if (g->pulled) cudaEventDestroy(g->pulled);
    for (cudaEvent_t e : g->op_ev) cudaEventDestroy(e);
    for (cudaEvent_t e : g->k_ev) cudaEventDestroy(e);
    for (cudaEvent_t e : {g->fork, g->join_up, g->join_pl, g->join_dn, g->k_last, g->t_fork, g->t_up, g->t_pl, g->t_k, g->t_dn})
        if (e) cudaEventDestroy(e);
    for (cudaStream_t q : {g->own, g->up, g->pl, g->dn})
        if (q) cudaStreamDestroy(q);
    if (g->full.data) cudaFree(g->full.data);
    if (g->band.data) cudaFree(g->band.data);
    if (g->shm) munmap(g->shm, 4096);
    if (g->shm_name[0]) shm_unlink(g->shm_name);
    cudaGetLastError();
    delete g;
    return AAI_OK;
}

}  // extern "C"
