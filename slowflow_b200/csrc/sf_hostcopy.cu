// sf_hostcopy.cu -- transfers between caller memory and the device for the host-buffer entry points.
//
// The reference allocates its images with plain malloc (image.c:17-33), so an unmodified call site hands the library
// pageable buffers.  cudaMemcpyAsync stages those through the driver's own bounce buffer on ONE host thread: ~11 GB/s
// measured, i.e. 10 ms for the 117 MB of a 2560x1440 pair against 2.5 ms of GPU work.  Here large pageable copies are
// cut into chunks that a few short-lived host threads copy into page-locked slots of the context and hand to the DMA
// engine on their own streams; page-locked or registered caller memory takes the direct path (host_copies).
//
// CopyPipeline moves the caller memory of the calls that stream many stages (sf_sequence.cu, sf_epicflow.cu): with
// page-locked memory, uploads run on an h2d stream and downloads on a d2h stream while the compute stream works.
#include <string.h>

#include <algorithm>
#include <thread>
#include <vector>

#include "sf_context.cuh"

namespace sf {

constexpr size_t HC_CHUNK = (size_t)1 << 20; // bytes per slot
constexpr int HC_MAX_WORKERS = 8, HC_SLOTS = 4;
// copy threads per call: SLOWFLOW_GPU_COPY_THREADS (1..8), default 4
static int hc_workers() {
    static const int n = [] {
        const char *e = getenv("SLOWFLOW_GPU_COPY_THREADS");
        const int v = e ? atoi(e) : 4;
        return v < 1 ? 1 : (v > HC_MAX_WORKERS ? HC_MAX_WORKERS : v);
    }();
    return n;
}

struct HostStager {
    unsigned char *slot[HC_MAX_WORKERS][HC_SLOTS] = {};
    cudaEvent_t done[HC_MAX_WORKERS][HC_SLOTS] = {};
    cudaStream_t stream[HC_MAX_WORKERS] = {};
    int workers = 0;
    cudaEvent_t gate = nullptr; // recorded on the context's stream: device data ready (D2H) / buffers free (H2D)
    bool ok = false;
    ~HostStager() {
        for (int w = 0; w < HC_MAX_WORKERS; w++) {
            for (int s = 0; s < HC_SLOTS; s++) {
                if (slot[w][s]) cudaFreeHost(slot[w][s]);
                if (done[w][s]) cudaEventDestroy(done[w][s]);
            }
            if (stream[w]) cudaStreamDestroy(stream[w]);
        }
        if (gate) cudaEventDestroy(gate);
    }
    bool init() {
        if (ok) return true;
        workers = hc_workers();
        for (int w = 0; w < workers; w++) {
            if (cudaStreamCreateWithFlags(&stream[w], cudaStreamNonBlocking) != cudaSuccess) return false;
            for (int s = 0; s < HC_SLOTS; s++) {
                if (cudaMallocHost(&slot[w][s], HC_CHUNK) != cudaSuccess) return false;
                if (cudaEventCreateWithFlags(&done[w][s], cudaEventDisableTiming) != cudaSuccess) return false;
            }
        }
        if (cudaEventCreateWithFlags(&gate, cudaEventDisableTiming) != cudaSuccess) return false;
        ok = true;
        return true;
    }
};

void host_stager_free(HostStager *h) { delete h; }

static bool is_pageable(const void *p) {
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
        cudaGetLastError();
        return true;
    }
    return at.type == cudaMemoryTypeUnregistered;
}

// One direction of a batch of copies.  H2D: returns once every byte has been handed to the DMA engine and makes the
// context's stream wait for the transfers.  D2H: waits for the context's stream first and returns when the data is in
// the caller's buffers.
static int staged_batch(sfgpu_ctx *c, const std::vector<HostCopy> &list, bool h2d) {
    if (!c->stager) c->stager = new HostStager();
    HostStager &hs = *c->stager;
    if (!hs.init()) {
        set_error("pinned staging buffers could not be allocated");
        return SFGPU_ERR_CUDA;
    }
    // everything already queued on the context's stream comes first (D2H: the results; H2D: earlier users of dst)
    const int HC_WORKERS = hs.workers;
    SF_CUDA(cudaEventRecord(hs.gate, c->stream));
    for (int w = 0; w < HC_WORKERS; w++) SF_CUDA(cudaStreamWaitEvent(hs.stream[w], hs.gate, 0));
    struct Piece { unsigned char *dev; unsigned char *host; size_t bytes; };
    std::vector<Piece> pieces;
    for (const HostCopy &hc : list)
        for (size_t off = 0; off < hc.bytes; off += HC_CHUNK)
            pieces.push_back(Piece{(unsigned char *)hc.dev + off, (unsigned char *)hc.host + off, std::min(HC_CHUNK, hc.bytes - off)});
    const int device = c->device;
    bool failed[HC_MAX_WORKERS] = {};
    auto work = [&](int w) {
        if (cudaSetDevice(device) != cudaSuccess) { failed[w] = true; return; }
        int used[HC_SLOTS] = {};
        std::vector<std::pair<int, const Piece *>> pending; // D2H: slot -> piece still to be copied out
        for (size_t k = w, n = 0; k < pieces.size(); k += HC_WORKERS, n++) {
            const Piece &p = pieces[k];
            const int s = (int)(n % HC_SLOTS);
            if (used[s]) { // the slot's previous transfer must have finished
                if (cudaEventSynchronize(hs.done[w][s]) != cudaSuccess) { failed[w] = true; return; }
                if (!h2d)
                    for (auto it = pending.begin(); it != pending.end(); ++it)
                        if (it->first == s) { memcpy(it->second->host, hs.slot[w][s], it->second->bytes); pending.erase(it); break; }
            }
            if (h2d) {
                memcpy(hs.slot[w][s], p.host, p.bytes);
                if (cudaMemcpyAsync(p.dev, hs.slot[w][s], p.bytes, cudaMemcpyHostToDevice, hs.stream[w]) != cudaSuccess) failed[w] = true;
            } else {
                if (cudaMemcpyAsync(hs.slot[w][s], p.dev, p.bytes, cudaMemcpyDeviceToHost, hs.stream[w]) != cudaSuccess) failed[w] = true;
                pending.push_back(std::make_pair(s, &p));
            }
            if (cudaEventRecord(hs.done[w][s], hs.stream[w]) != cudaSuccess) failed[w] = true;
            used[s] = 1;
            if (failed[w]) return;
        }
        // drain: H2D slots must not be reused by the next call before their DMA has read them; D2H data must land
        for (int s = 0; s < HC_SLOTS; s++)
            if (used[s] && cudaEventSynchronize(hs.done[w][s]) != cudaSuccess) failed[w] = true;
        for (auto &pr : pending) memcpy(pr.second->host, hs.slot[w][pr.first], pr.second->bytes);
    };
    std::vector<std::thread> pool;
    int inline_from = HC_WORKERS; // workers that could not get a thread run on the calling thread
    for (int w = 1; w < HC_WORKERS; w++) {
        try {
            pool.emplace_back(work, w);
        } catch (...) {
            inline_from = w;
            break;
        }
    }
    work(0);
    for (int w = inline_from; w < HC_WORKERS; w++) work(w);
    for (auto &t : pool) t.join();
    for (int w = 0; w < HC_WORKERS; w++)
        if (failed[w]) {
            set_error("staged host copy failed");
            return SFGPU_ERR_CUDA;
        }
    if (h2d) { // the context's stream continues after the uploads (they are complete: the workers drained their slots)
        for (int w = 0; w < HC_WORKERS; w++) {
            SF_CUDA(cudaEventRecord(hs.done[w][0], hs.stream[w]));
            SF_CUDA(cudaStreamWaitEvent(c->stream, hs.done[w][0], 0));
        }
    }
    return SFGPU_OK;
}

// Copies of one call in one direction.  Pageable buffers of at least 2 chunks go through the staged path (together, so
// that the worker threads are spawned once); everything else is a plain cudaMemcpyAsync on the context's stream.
int host_copies(sfgpu_ctx *c, const std::vector<HostCopy> &list, bool h2d) {
    std::vector<HostCopy> staged, direct;
    for (const HostCopy &hc : list)
        (c->staged_host_copies && hc.bytes >= 2 * HC_CHUNK && is_pageable(hc.host) ? staged : direct).push_back(hc);
    if (h2d)
        for (const HostCopy &hc : direct) SF_CUDA(cudaMemcpyAsync(hc.dev, hc.host, hc.bytes, cudaMemcpyHostToDevice, c->stream));
    if (!staged.empty()) {
        const int rc = staged_batch(c, staged, h2d);
        if (rc != SFGPU_OK) return rc;
    }
    if (!h2d)
        for (const HostCopy &hc : direct) SF_CUDA(cudaMemcpyAsync(hc.host, hc.dev, hc.bytes, cudaMemcpyDeviceToHost, c->stream));
    return SFGPU_OK;
}

enum { UPLOADED, PASSED, DRAINED }; // the event rings of sfgpu_ctx::copy_ev

// Pageable caller memory (the reference's image_new is malloc): cudaMemcpyAsync would stage it synchronously through the
// driver and no transfer would overlap anything, so such a call takes the staged copies above, stage by stage.
int CopyPipeline::start(const std::vector<const void *> &buffers) {
    pageable = std::any_of(buffers.begin(), buffers.end(), is_pageable);
    if (pageable) return SFGPU_OK;
    for (cudaStream_t *st : {&c->h2d, &c->d2h})
        if (!*st) SF_CUDA(cudaStreamCreateWithFlags(st, cudaStreamNonBlocking));
    for (auto &ring : c->copy_ev)
        for (cudaEvent_t &e : ring)
            if (!e) SF_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    // the previous call may still read the io area: compute has passed stage -1 (slot 3, free until pass(3))
    SF_CUDA(cudaEventRecord(c->copy_ev[PASSED][3], c->stream));
    SF_CUDA(cudaStreamWaitEvent(c->h2d, c->copy_ev[PASSED][3], 0));
    return SFGPU_OK;
}

int CopyPipeline::upload(int k, const std::vector<HostCopy> &list, int passed, int drained) {
    if (pageable) return host_copies(c, list, true);
    if (passed >= 0) SF_CUDA(cudaStreamWaitEvent(c->h2d, c->copy_ev[PASSED][passed & 3], 0));
    if (drained >= 0) SF_CUDA(cudaStreamWaitEvent(c->h2d, c->copy_ev[DRAINED][drained & 3], 0));
    for (const HostCopy &hc : list) SF_CUDA(cudaMemcpyAsync(hc.dev, hc.host, hc.bytes, cudaMemcpyHostToDevice, c->h2d));
    SF_CUDA(cudaEventRecord(c->copy_ev[UPLOADED][k & 3], c->h2d));
    return SFGPU_OK;
}

int CopyPipeline::wait(int uploaded, int drained) {
    if (pageable) return SFGPU_OK;
    if (uploaded >= 0) SF_CUDA(cudaStreamWaitEvent(c->stream, c->copy_ev[UPLOADED][uploaded & 3], 0));
    if (drained >= 0) SF_CUDA(cudaStreamWaitEvent(c->stream, c->copy_ev[DRAINED][drained & 3], 0));
    return SFGPU_OK;
}

int CopyPipeline::pass(int k) {
    if (!pageable) SF_CUDA(cudaEventRecord(c->copy_ev[PASSED][k & 3], c->stream));
    return SFGPU_OK;
}

int CopyPipeline::download(int k, const std::vector<HostCopy> &list) {
    if (pageable) return host_copies(c, list, false);
    SF_CUDA(cudaStreamWaitEvent(c->d2h, c->copy_ev[PASSED][k & 3], 0));
    for (const HostCopy &hc : list) SF_CUDA(cudaMemcpyAsync(hc.host, hc.dev, hc.bytes, cudaMemcpyDeviceToHost, c->d2h));
    SF_CUDA(cudaEventRecord(c->copy_ev[DRAINED][k & 3], c->d2h));
    return SFGPU_OK;
}

int CopyPipeline::finish(int status) {
    for (cudaStream_t st : {c->h2d, c->stream, c->d2h}) {
        const cudaError_t e = st ? cudaStreamSynchronize(st) : cudaSuccess;
        if (status == SFGPU_OK && !cuda_ok(e, "copy pipeline: cudaStreamSynchronize")) status = SFGPU_ERR_CUDA;
    }
    return status;
}

} // namespace sf
