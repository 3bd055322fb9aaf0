// ohp_multi.cuh -- include/ohp_multi.h: one process, several B200s; a contiguous block of streams, a context, a host
// thread and its own CUDA streams per device, no collective (SURVEY 8e).  Included at the end of ohp_capi.cu (it reads a
// context's output arena for the per-stream checksums).
#pragma once

#include "../../include/ohp_multi.h"

#include <condition_variable>
#include <memory>

namespace ohp {

struct MultiJob
{
    const ohp_stream_spec* streams = nullptr;
    size_t n_streams = 0;
    const ohp_ramp_event* events = nullptr;
    size_t n_events = 0;
    const uint8_t* h_in = nullptr;
    uint64_t in_bytes = 0;
    uint8_t* h_out = nullptr;
    uint64_t out_bytes = 0;
    uint64_t* out_bytes_per_stream = nullptr;
    uint64_t* sums = nullptr;
};

struct MultiWorker
{
    size_t index = 0;
    int device = -1;
    ohp_context* ctx = nullptr;
    std::thread thread;
    int rc = OHP_OK;
    std::string error;
    uint64_t chunks = 0;
    std::vector<ohp_stream_spec> specs;  // the block, re-based
    std::vector<uint64_t> outb;
    uint64_t* d_ranges = nullptr; uint64_t d_ranges_cap = 0; // (begin, end) of every stream's output in the device arena
    uint64_t* d_sums = nullptr;   uint64_t d_sums_cap = 0;
    uint64_t* h_ranges = nullptr; uint64_t h_ranges_cap = 0; // pinned
};

} // namespace ohp

struct ohp_multi
{
    std::vector<std::unique_ptr<ohp::MultiWorker>> workers;
    std::mutex lock;
    std::condition_variable go, done;
    uint64_t generation = 0; // bumped per job
    size_t pending = 0;
    bool quit = false;
    ohp::MultiJob job;
    std::string error;
};

namespace ohp {

static constexpr uint64_t kMultiArenaAlign = 256; // a block's arenas start on what the single-device layout's streams sit on

static int multi_fail(MultiWorker& w, int status, const std::string& what)
{
    w.rc = status;
    w.error = what;
    return status;
}

// One device's share of a job.  Runs on the device's own thread.
static int multi_run_block(MultiWorker& w, const MultiJob& j, size_t n_devices)
{
    w.rc = OHP_OK;
    w.error.clear();
    w.chunks = 0;
    size_t first = 0, count = 0;
    ohp_multi_shard(j.n_streams, n_devices, w.index, &first, &count);
    if (count == 0) return OHP_OK;
    const ohp_stream_spec* block = j.streams + first;
    // what of the arenas and of the events the block touches
    uint64_t in_lo = UINT64_MAX, in_hi = 0, out_lo = UINT64_MAX, ev_lo = UINT64_MAX, ev_hi = 0;
    for (size_t s = 0; s < count; s++) {
        const ohp_stream_spec& sp = block[s];
        const uint64_t frame_bytes = (uint64_t)sp.channels * (sp.bit_depth / 8u);
        if (frame_bytes != 0 && sp.total_frames > UINT64_MAX / frame_bytes) {
            return multi_fail(w, OHP_E_OUT_OF_RANGE, "stream " + std::to_string(first + s) + " reaches outside the arenas");
        }
        const uint64_t len = sp.total_frames * frame_bytes;
        if (sp.src_base > j.in_bytes || len > j.in_bytes - sp.src_base || sp.dst_base > j.out_bytes) {
            return multi_fail(w, OHP_E_OUT_OF_RANGE, "stream " + std::to_string(first + s) + " reaches outside the arenas");
        }
        if (len) {
            in_lo = std::min(in_lo, sp.src_base);
            in_hi = std::max(in_hi, sp.src_base + len);
        }
        out_lo = std::min(out_lo, sp.dst_base);
        if (sp.num_events) {
            if ((uint64_t)sp.first_event + sp.num_events > j.n_events) {
                return multi_fail(w, OHP_E_INVALID_ARG, "stream " + std::to_string(first + s) + ": events outside the array");
            }
            ev_lo = std::min<uint64_t>(ev_lo, sp.first_event);
            ev_hi = std::max<uint64_t>(ev_hi, (uint64_t)sp.first_event + sp.num_events);
        }
    }
    if (in_lo == UINT64_MAX) in_lo = in_hi = 0;
    if (ev_lo == UINT64_MAX) ev_lo = ev_hi = 0;
    in_lo -= in_lo % kMultiArenaAlign;
    out_lo -= out_lo % kMultiArenaAlign;
    w.specs.assign(block, block + count);
    for (auto& sp : w.specs) {
        sp.src_base = sp.src_base >= in_lo ? sp.src_base - in_lo : 0; // (a stream without PCM may sit below the block's first byte)
        sp.dst_base -= out_lo;
        sp.first_event = sp.num_events ? sp.first_event - (uint32_t)ev_lo : 0u; // (an empty slice may point anywhere up to the end)
    }
    // How far the block's output reaches is only known once its schedules have been walked, but streams do not write over
    // each other: it ends before the first stream of ANOTHER block that begins behind this block's last one (or with the
    // arena).  That is the room the device arena is sized for, and what the single-device call holds every stream against.
    uint64_t out_last = 0, out_hi = j.out_bytes;
    for (size_t s = 0; s < count; s++) out_last = std::max(out_last, block[s].dst_base);
    for (size_t s = 0; s < j.n_streams; s++) {
        if (s >= first && s < first + count) continue;
        const uint64_t at = j.streams[s].dst_base;
        if (at > out_last && at < out_hi) out_hi = at;
    }
    // The host call bridges small holes between the block's output ranges: it copies the device's bytes over them and
    // puts back, when it ends, what they held when it began.  Where another block's stream begins inside the block's
    // span, that stream may be written into such a hole in the meantime, and putting the hole back would undo it: such a
    // block copies its ranges back one by one.
    bool foreign_inside = false;
    for (size_t s = 0; s < j.n_streams && !foreign_inside; s++) {
        if (s >= first && s < first + count) continue;
        const uint64_t at = j.streams[s].dst_base;
        foreign_inside = at >= out_lo && at < out_hi;
    }
    w.outb.assign(count, 0);
    uint64_t chunks = 0;
    const int rc = run_streams_host(w.ctx, w.specs.data(), count, j.events ? j.events + ev_lo : nullptr, (size_t)(ev_hi - ev_lo),
                                    j.h_in + in_lo, in_hi - in_lo, j.h_out + out_lo, out_hi - out_lo,
                                    w.outb.data(), &chunks, foreign_inside ? 0 : RangeSet::kBridge);
    if (rc != OHP_OK) {
        // the call names streams by their place in the block
        return multi_fail(w, rc, std::string(ohp_last_error(w.ctx)) + " (streams counted from " + std::to_string(first) + ")");
    }
    w.chunks = chunks;
    if (j.out_bytes_per_stream) std::memcpy(j.out_bytes_per_stream + first, w.outb.data(), count * sizeof(uint64_t));
    if (j.sums) {
        // per-stream checksums of what sits in THIS device's output arena: 8 bytes per stream come back
        ohp_context* ctx = w.ctx;
        auto cuda = [&](cudaError_t e, const char* what) { return e == cudaSuccess ? OHP_OK : multi_fail(w, OHP_E_CUDA, std::string(what) + ": " + cudaGetErrorString(e)); };
        if (w.h_ranges_cap < 2 * count) {
            if (w.h_ranges) (void)cudaFreeHost(w.h_ranges);
            w.h_ranges = nullptr; w.h_ranges_cap = 0;
            if (cuda(cudaMallocHost(reinterpret_cast<void**>(&w.h_ranges), 2 * count * sizeof(uint64_t)), "cudaMallocHost") != OHP_OK) return w.rc;
            w.h_ranges_cap = 2 * count;
        }
        if (w.d_ranges_cap < 2 * count) {
            if (w.d_ranges) (void)cudaFree(w.d_ranges);
            w.d_ranges = nullptr; w.d_ranges_cap = 0;
            if (cuda(cudaMalloc(reinterpret_cast<void**>(&w.d_ranges), 2 * count * sizeof(uint64_t)), "cudaMalloc") != OHP_OK) return w.rc;
            w.d_ranges_cap = 2 * count;
        }
        if (w.d_sums_cap < count) {
            if (w.d_sums) (void)cudaFree(w.d_sums);
            w.d_sums = nullptr; w.d_sums_cap = 0;
            if (cuda(cudaMalloc(reinterpret_cast<void**>(&w.d_sums), count * sizeof(uint64_t)), "cudaMalloc") != OHP_OK) return w.rc;
            w.d_sums_cap = count;
        }
        for (size_t s = 0; s < count; s++) {
            w.h_ranges[2 * s] = w.specs[s].dst_base;
            w.h_ranges[2 * s + 1] = w.specs[s].dst_base + w.outb[s];
        }
        cudaStream_t st = ctx->stream;
        if (cuda(cudaMemcpyAsync(w.d_ranges, w.h_ranges, 2 * count * sizeof(uint64_t), cudaMemcpyHostToDevice, st), "cudaMemcpyAsync") != OHP_OK) return w.rc;
        uint64_t grid = (uint64_t)ctx->sm_count * 8u;
        if (grid > count) grid = count;
        checksum_kernel<<<(unsigned)grid, 256, 0, st>>>(ctx->d_out, w.d_ranges, count, w.d_sums, 2u);
        if (cuda(cudaGetLastError(), "checksum_kernel") != OHP_OK) return w.rc;
        ctx->launches++;
        // (the ranges' pinned buffer doubles as the landing place: the upload has been consumed by then, stream order)
        if (cuda(cudaMemcpyAsync(w.h_ranges, w.d_sums, count * sizeof(uint64_t), cudaMemcpyDeviceToHost, st), "cudaMemcpyAsync") != OHP_OK) return w.rc;
        if (cuda(cudaStreamSynchronize(st), "cudaStreamSynchronize") != OHP_OK) return w.rc;
        std::memcpy(j.sums + first, w.h_ranges, count * sizeof(uint64_t));
    }
    return OHP_OK;
}

static void multi_worker_main(ohp_multi* m, MultiWorker* w)
{
    // creation is the thread's first job: the context, its streams and its pinned buffers belong to this thread's device
    {
        ohp_context* ctx = nullptr;
        const int rc = ohp_create(w->device, &ctx);
        if (rc != OHP_OK) { w->rc = rc; w->error = ohp_last_error(nullptr); }
        else {
            w->ctx = ctx;
            if (ctx->have_local_cpus) (void)sched_setaffinity(0, sizeof ctx->local_cpus, &ctx->local_cpus);
        }
        std::lock_guard<std::mutex> g(m->lock);
        if (--m->pending == 0) m->done.notify_all();
    }
    uint64_t seen = 0;
    for (;;) {
        MultiJob job;
        {
            std::unique_lock<std::mutex> g(m->lock);
            m->go.wait(g, [&] { return m->quit || m->generation != seen; });
            if (m->quit) break;
            seen = m->generation;
            job = m->job;
        }
        if (w->ctx) {
            try {
                (void)multi_run_block(*w, job, m->workers.size());
            }
            catch (const std::exception& e) { // the block's re-based specs and staging vectors: out of host memory
                (void)multi_fail(*w, OHP_E_NO_MEMORY, e.what());
            }
        }
        std::lock_guard<std::mutex> g(m->lock);
        if (--m->pending == 0) m->done.notify_all();
    }
    if (w->ctx) {
        (void)cudaSetDevice(w->device);
        if (w->d_ranges) (void)cudaFree(w->d_ranges);
        if (w->d_sums) (void)cudaFree(w->d_sums);
        if (w->h_ranges) (void)cudaFreeHost(w->h_ranges);
        (void)ohp_destroy(w->ctx);
        w->ctx = nullptr;
    }
}

} // namespace ohp

extern "C" {

void ohp_multi_shard(size_t n_streams, size_t n_devices, size_t index, size_t* first, size_t* count)
{
    size_t lo = 0, hi = 0;
    if (n_devices != 0 && index < n_devices) {
        // S * g / G without overflow: S = q * G + r
        const size_t q = n_streams / n_devices, r = n_streams % n_devices;
        lo = q * index + r * index / n_devices;
        hi = q * (index + 1) + r * (index + 1) / n_devices;
    }
    if (first) *first = lo;
    if (count) *count = hi - lo;
}

int ohp_multi_create(const int* devices, size_t n_devices, ohp_multi** out)
{
    if (!out) return OHP_E_INVALID_ARG;
    *out = nullptr;
    if (!devices || n_devices == 0 || n_devices > 64) return ohp::fail(nullptr, OHP_E_INVALID_ARG, "ohp_multi_create: 1 to 64 devices");
    ohp_multi* m = new (std::nothrow) ohp_multi();
    if (!m) return ohp::fail(nullptr, OHP_E_NO_MEMORY, "out of host memory");
    m->pending = n_devices;
    for (size_t i = 0; i < n_devices; i++) {
        std::unique_ptr<ohp::MultiWorker> w(new ohp::MultiWorker());
        w->index = i;
        w->device = devices[i];
        m->workers.push_back(std::move(w));
    }
    for (auto& w : m->workers) w->thread = std::thread(ohp::multi_worker_main, m, w.get());
    {
        std::unique_lock<std::mutex> g(m->lock);
        m->done.wait(g, [&] { return m->pending == 0; });
    }
    for (auto& w : m->workers) {
        if (w->rc != OHP_OK) {
            const int rc = w->rc;
            const std::string msg = "device " + std::to_string(w->device) + ": " + w->error;
            (void)ohp_multi_destroy(m);
            return ohp::fail(nullptr, rc, msg.c_str());
        }
    }
    *out = m;
    return OHP_OK;
}

int ohp_multi_destroy(ohp_multi* m)
{
    if (!m) return OHP_E_INVALID_ARG;
    {
        std::lock_guard<std::mutex> g(m->lock);
        m->quit = true;
    }
    m->go.notify_all();
    for (auto& w : m->workers) {
        if (w->thread.joinable()) w->thread.join();
    }
    delete m;
    return OHP_OK;
}

size_t ohp_multi_num_devices(const ohp_multi* m) { return m ? m->workers.size() : 0; }
const char* ohp_multi_last_error(const ohp_multi* m) { return m ? m->error.c_str() : "null ohp_multi"; }
ohp_context* ohp_multi_context(ohp_multi* m, size_t index) { return (m && index < m->workers.size()) ? m->workers[index]->ctx : nullptr; }

int ohp_multi_run_streams_host(ohp_multi* m, const ohp_stream_spec* h_streams, size_t n_streams,
                               const ohp_ramp_event* h_events, size_t n_events,
                               const uint8_t* h_in, uint64_t in_bytes, uint8_t* h_out, uint64_t out_bytes,
                               uint64_t* h_stream_out_bytes, uint64_t* h_checksums, uint64_t* total_chunks)
{
    if (!m) return OHP_E_INVALID_ARG;
    m->error.clear();
    if (total_chunks) *total_chunks = 0;
    if (n_streams == 0) return OHP_OK;
    if (!h_streams || (!h_events && n_events) || (!h_in && in_bytes) || (!h_out && out_bytes)) {
        m->error = "null pointer";
        return OHP_E_INVALID_ARG;
    }
    {
        std::lock_guard<std::mutex> g(m->lock);
        m->job.streams = h_streams;   m->job.n_streams = n_streams;
        m->job.events = h_events;     m->job.n_events = n_events;
        m->job.h_in = h_in;           m->job.in_bytes = in_bytes;
        m->job.h_out = h_out;         m->job.out_bytes = out_bytes;
        m->job.out_bytes_per_stream = h_stream_out_bytes;
        m->job.sums = h_checksums;
        m->pending = m->workers.size();
        m->generation++;
    }
    m->go.notify_all();
    {
        // every device's share is synchronous: when the last thread reports, nothing is in flight anywhere
        std::unique_lock<std::mutex> g(m->lock);
        m->done.wait(g, [&] { return m->pending == 0; });
    }
    uint64_t chunks = 0;
    for (auto& w : m->workers) {
        if (w->rc != OHP_OK) {
            m->error = "device index " + std::to_string(w->index) + " (CUDA device " + std::to_string(w->device) + "): " + w->error;
            return w->rc;
        }
        chunks += w->chunks;
    }
    if (total_chunks) *total_chunks = chunks;
    return OHP_OK;
}

int ohp_multi_host_alloc(ohp_multi* m, uint64_t bytes, void** out_hptr)
{
    if (!m || m->workers.empty() || !out_hptr) return OHP_E_INVALID_ARG;
    const int rc = ohp_host_alloc(m->workers[0]->ctx, bytes, out_hptr);
    if (rc != OHP_OK) m->error = ohp_last_error(m->workers[0]->ctx);
    return rc;
}

int ohp_multi_host_free(ohp_multi* m, void* hptr)
{
    if (!m || m->workers.empty()) return OHP_E_INVALID_ARG;
    return ohp_host_free(m->workers[0]->ctx, hptr);
}

} // extern "C"
