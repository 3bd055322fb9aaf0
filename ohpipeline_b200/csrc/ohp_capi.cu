// ohp_capi.cu -- the C ABI declared in include/ohp_b200.h, ohp_schedule_device.h and ohp_flywheel.h: contexts, launches,
// in-flight tuning, host-buffer pipelines.  The kernels are in the .cuh files included below.
//
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -shared -Xcompiler -fPIC
// There is no CPU fallback anywhere in this file: without a usable sm_100 device every compute entry
// point returns OHP_E_NO_DEVICE / OHP_E_CUDA.
#include "ohp_kernels.cuh"
#include "ohp_ramp_convert_kernel.cuh"
#include "ohp_schedule_kernels.cuh"
#include "ohp_flywheel_kernels.cuh"
#include "../../include/ohp_schedule_device.h"
#include "../../include/ohp_starvation_device.h"
#include "../../include/ohp_starvation_recent.h"

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <algorithm>
#include <cctype>
#include <mutex>
#include <sched.h>
#include <new>
#include <string>
#include <thread>
#include <vector>

namespace ohp {

// ---------------------------------------------------------------------------------------------
// host side

static const uint16_t kRampTable[OHP_RAMP_TABLE_ENTRIES] = {
#include "ramp_table.inc"
};

static thread_local std::string g_create_error;

// In-flight tuning.  How many chunks a CTA should keep in flight is the one knob whose best value depends on the batch
// in a way the shape cannot settle: configs[1] (uniform 5760-byte chunks) peaks sharply at 12 (0.985 of the copy peak
// against 0.895 at 16 and above, 0.945 at 10), configs[2] and small chunks want everything the ring holds
// (profiles/README.md).  So a context learns it per batch signature: the first launches of a signature each run with a
// different candidate between CUDA events on the caller's stream, later launches read the finished timings and use the
// fastest.  Results never depend on the cap; only large batches are tuned.
constexpr int kTuneCandidates = 3;  // few, so that a benchmark's customary warm-up launches do (nearly) all the exploring
static const uint32_t kTuneCaps[kTuneCandidates] = {kRingSlots, 12u, 24u};
static const uint32_t kTuneSerial[kTuneCandidates] = {0u, 1u, 0u}; // the loader's placement mode that goes with each cap
constexpr uint64_t kTuneMinBytes = 256ull << 20; // batches below this are launch-latency territory: not worth tuning
constexpr uint64_t kTuneMinChunks = 65536;
// The first launch of a new shape runs cold (instruction cache, TLBs, the descriptors' first trip through L2), a few
// per cent slower than it will ever be again: its candidate gets a second, warm trial.
constexpr int kTuneTrials = kTuneCandidates + 1;
static const int kTrialCandidate[kTuneTrials] = {0, 1, 2, 0};
struct TuneEntry
{
    uint64_t n = 0, in_bytes = 0, out_bytes = 0;
    int launched = 0;                 // trials started so far
    bool done[kTuneTrials] = {};      // trial's time has been read
    bool have[kTuneCandidates] = {};
    float ms[kTuneCandidates] = {};   // latest trial of each candidate
    cudaEvent_t ev[kTuneTrials][2] = {};
    uint64_t last_use = 0;
};

} // namespace ohp

struct ohp_context
{
    int device = -1;
    int sm_count = 0;
    int ctas_per_sm = 0;
    cudaStream_t stream = nullptr;     // compute
    cudaStream_t copy_in = nullptr;    // H2D
    cudaStream_t copy_out = nullptr;   // D2H
    uint16_t* d_table2 = nullptr;
    uint32_t* d_status = nullptr;
    uint32_t* h_status = nullptr;      // pinned
    // ohp_process_host staging (grown on demand)
    uint8_t* d_in = nullptr;  uint64_t d_in_cap = 0;
    uint8_t* d_out = nullptr; uint64_t d_out_cap = 0;
    ohp_chunk_desc* d_descs = nullptr; uint64_t d_descs_cap = 0;
    // ohp_run_streams_host staging (grown on demand)
    ohp_stream_spec* d_specs = nullptr; uint64_t d_specs_cap = 0;
    ohp_ramp_event* d_events = nullptr; uint64_t d_events_cap = 0;
    uint64_t* d_begin = nullptr; uint64_t d_begin_cap = 0;
    uint64_t* d_outb = nullptr; uint64_t d_outb_cap = 0;
    uint64_t* d_counts = nullptr; uint64_t d_counts_cap = 0;  // ohp_run_streams_device: exact playables per stream
    cudaEvent_t sched_event = nullptr;                           // ... recorded behind a copy the host waits for
    cudaEvent_t fly_event = nullptr;                             // ohp_run_streams_device_flywheel: behind the planned jobs' count
    cudaEvent_t scratch_done = nullptr;                          // behind the last call that used the scratch (ScratchTurn)
    uint64_t* h_regions = nullptr;                               // ... the regions' total (pinned; [4..8): sched::FlySlots)
    // ohp_run_streams_device_flywheel (grown on demand)
    ohp_starvation* d_records = nullptr; uint64_t d_records_cap = 0; // when the caller passes no record array
    uint64_t* d_slot = nullptr; uint64_t d_slot_cap = 0;             // flywheel slots, scanned in place
    uint32_t* d_owner = nullptr; uint64_t d_owner_cap = 0;           // the stream that holds each event
    ohp::sched::FlySlots* d_fly_slots = nullptr;
    ohp_chunk_desc* d_fly_descs = nullptr; uint64_t d_fly_descs_cap = 0; // prep, then blocks, per starvation event
    ohp_flywheel_job* d_fly_jobs = nullptr; uint64_t d_fly_jobs_cap = 0;
    uint8_t* d_fly_train = nullptr; uint64_t d_fly_train_cap = 0;    // training blocks
    uint8_t* d_fly_gen = nullptr; uint64_t d_fly_gen_cap = 0;        // generated audio
    // ohp_run_streams_device_flywheel_recent, when the caller passes no arrays of its own (grown on demand)
    ohp_recent_audio* d_recent = nullptr; uint64_t d_recent_cap = 0;
    uint32_t* d_recent_count = nullptr; uint64_t d_recent_count_cap = 0;
    std::vector<uint64_t> h_begin, h_outb;
    cudaEvent_t ev_start = nullptr, ev_stop = nullptr;
    bool timing = false;
    bool timed = false;
    uint64_t launches = 0;
    std::vector<cudaEvent_t> slice_events; // ohp_process_host pipeline, reused across calls
    uint32_t cap_bytes = ohp::kRingBytes;   // in-flight limits per CTA (experiments: OHP_CAP_BYTES / OHP_CAP_CHUNKS)
    uint32_t cap_chunks = ohp::kRingSlots;
    uint32_t chunk_block = ohp::kChunkBlock;
    bool cap_pinned = false;               // OHP_CAP_CHUNKS / OHP_CAP_BYTES given: no tuning
    uint32_t serial_place = 0;             // loader placement mode when not tuned (experiments: OHP_SERIAL_PLACE=1)
    bool autotune = true;                  // OHP_AUTOTUNE=0 turns it off
    std::vector<ohp::TuneEntry> tune;      // one entry per batch signature seen (a few)
    uint64_t tune_clock = 0;               // least-recently-used eviction among them
    uint32_t last_cap_chunks = ohp::kRingSlots; // what the most recent launch used (ohp_inflight_cap)
    cpu_set_t local_cpus;                  // cores of the NUMA node this GPU hangs off (empty set: unknown)
    bool have_local_cpus = false;
    std::string error;
};

namespace ohp {

// A warp per stream while the warps still fit the GPU at once (148 SMs x 12 resident warps of schedule_kernel), a thread
// per stream beyond: with more warps than that the walks go in waves and the 32-fold redundant general path is paid in
// issue slots (round 2, configs[2]: 2.97 -> 2.80 ms specs-to-bytes, configs[3]: 5.96 -> 4.47 ms; profiles/README.md).
constexpr size_t kScheduleWarpTeamMaxStreams = 2048;

static int fail(ohp_context* ctx, int status, const char* what, cudaError_t e = cudaSuccess)
{
    std::string msg = what;
    if (e != cudaSuccess) {
        msg += ": ";
        msg += cudaGetErrorString(e);
    }
    if (ctx) ctx->error = msg; else g_create_error = msg;
    return status;
}

#define OHP_CUDA(ctx, call)                                                     \
    do {                                                                        \
        cudaError_t e_ = (call);                                                \
        if (e_ != cudaSuccess) return fail((ctx), OHP_E_CUDA, #call, e_);       \
    } while (0)

// Sliced host-buffer calls launch many small kernels: per-kernel timing and in-flight tuning are off for their duration
// and come back however the call ends.
struct SliceMode
{
    ohp_context* ctx;
    bool timing, autotune;
    explicit SliceMode(ohp_context* c) : ctx(c), timing(c->timing), autotune(c->autotune) { c->timing = false; c->autotune = false; }
    ~SliceMode() { ctx->timing = timing; ctx->autotune = autotune; }
    SliceMode(const SliceMode&) = delete;
    SliceMode& operator=(const SliceMode&) = delete;
};

// The synchronous host-buffer calls drive three streams.  However such a call ends -- a failed launch or copy in the
// middle of the slice loop included -- nothing of it may still be in flight when it returns: the caller is free to reuse
// or free h_in / h_out the moment it has the status.
struct DrainOnExit
{
    ohp_context* ctx;
    cudaStream_t compute;
    DrainOnExit(ohp_context* c, cudaStream_t st) : ctx(c), compute(st) {}
    ~DrainOnExit()
    {
        if (ctx->copy_in) (void)cudaStreamSynchronize(ctx->copy_in);
        if (compute) (void)cudaStreamSynchronize(compute);
        if (ctx->copy_out) (void)cudaStreamSynchronize(ctx->copy_out);
        (void)cudaGetLastError(); // the call's own status has been decided already
    }
    DrainOnExit(const DrainOnExit&) = delete;
    DrainOnExit& operator=(const DrainOnExit&) = delete;
};

// The context's scratch (the staging arenas, d_descs, d_begin, d_counts, the flywheel and recent-audio buffers) is shared
// by every call that stages through it -- ohp_process_host, ohp_run_streams_host, ohp_run_streams_device and its flywheel
// variants -- and the asynchronous ones return while their kernels still read it.  Each such call holds a ScratchTurn:
// on entry the caller's stream, the compute stream and the H2D stream wait (on the device, not the host) for the
// previous call's work, and however the call returns its own work is recorded behind it.  So calls may follow one another
// on any streams without an ohp_sync in between; a never-recorded event is no wait at all.
struct ScratchTurn
{
    ohp_context* ctx;
    cudaStream_t st;
    int rc = OHP_OK; // OHP_E_CUDA when a wait could not be enqueued: the call must not go on
    ScratchTurn(ohp_context* c, cudaStream_t s) : ctx(c), st(s)
    {
        for (cudaStream_t w : {s, c->stream, c->copy_in}) {
            const cudaError_t e = cudaStreamWaitEvent(w, c->scratch_done, 0);
            if (e != cudaSuccess) { rc = fail(c, OHP_E_CUDA, "cudaStreamWaitEvent (context scratch)", e); break; }
        }
    }
    ~ScratchTurn()
    {
        if (cudaEventRecord(ctx->scratch_done, st) != cudaSuccess) (void)cudaGetLastError();
    }
    ScratchTurn(const ScratchTurn&) = delete;
    ScratchTurn& operator=(const ScratchTurn&) = delete;
};

// What a host-buffer call copies back.  Only bytes some chunk writes belong to the call: everything else in h_out is
// the caller's and must read afterwards as it did before.  A slice's covered ranges are merged into few, large D2H
// copies; a small hole between two of them (alignment padding between streams, typically < 16 bytes) is bridged.  What
// a bridge drags along is either covered by another slice -- whose own copy, earlier or later on the in-order copy
// stream, leaves the final bytes -- or covered by nothing in the whole batch: those holes are found by one pass over the
// whole batch BEFORE anything is issued, their bytes saved, and put back once the copies have drained.
class RangeSet
{
public:
    static constexpr uint64_t kBridge = 4096;
    explicit RangeSet(uint64_t bridge = kBridge) : iBridge(bridge) {} // 0: no hole is bridged
    void Add(uint64_t off, uint64_t len)
    {
        if (len == 0) return;
        if (!iRanges.empty() && off == iRanges.back().hi) { iRanges.back().hi = off + len; return; }
        if (!iRanges.empty() && off < iRanges.back().hi) iSorted = false;
        iRanges.push_back(Range{off, off + len});
    }
    // Sort and merge what was added; f(lo, hi) for every maximal covered range, g(lo, hi) for every hole <= the bridge
    // limit between two of them (which is then bridged: the ranges either side reach f as one).
    template <class F, class G>
    void Merge(F f, G g)
    {
        if (iRanges.empty()) return;
        if (!iSorted) std::sort(iRanges.begin(), iRanges.end(), [](const Range& a, const Range& b) { return a.lo < b.lo; });
        uint64_t lo = iRanges[0].lo, hi = iRanges[0].hi;
        for (size_t i = 1; i < iRanges.size(); i++) {
            const Range& r = iRanges[i];
            if (r.lo <= hi) { hi = r.hi > hi ? r.hi : hi; continue; }
            if (r.lo - hi <= iBridge) { g(hi, r.lo); hi = r.hi; continue; }
            f(lo, hi);
            lo = r.lo; hi = r.hi;
        }
        f(lo, hi);
        iRanges.clear();
        iSorted = true;
    }
private:
    struct Range { uint64_t lo, hi; };
    std::vector<Range> iRanges;
    bool iSorted = true;
    uint64_t iBridge;
};

class CopyBackPlan
{
public:
    explicit CopyBackPlan(uint8_t* h_out, uint64_t bridge = RangeSet::kBridge) : iOut(h_out), iBatch(bridge), iSlice(bridge) {}
    ~CopyBackPlan() { Restore(); }
    RangeSet& Batch() { return iBatch; }   // every range the whole call covers ...
    void SaveHoles()                       // ... then, before the first copy is issued
    {
        iBatch.Merge([](uint64_t, uint64_t) {},
                     [this](uint64_t lo, uint64_t hi) {
                         iHoles.push_back(Hole{lo, (uint32_t)(hi - lo), iSaved.size()});
                         iSaved.insert(iSaved.end(), iOut + lo, iOut + hi);
                     });
    }
    RangeSet& Slice() { return iSlice; }   // the ranges of one slice ...
    const std::vector<std::pair<uint64_t, uint64_t>>& Copies() // ... and the [lo, hi) copies that bring them back
    {
        iCopies.clear();
        iSlice.Merge([this](uint64_t lo, uint64_t hi) { iCopies.emplace_back(lo, hi); }, [](uint64_t, uint64_t) {});
        return iCopies;
    }
    void Restore() // only after the copies have completed
    {
        for (const Hole& h : iHoles) std::memcpy(iOut + h.off, iSaved.data() + h.at, h.len);
        iHoles.clear();
        iSaved.clear();
    }
private:
    struct Hole { uint64_t off; uint32_t len; size_t at; };
    uint8_t* iOut;
    RangeSet iBatch, iSlice;
    std::vector<Hole> iHoles;
    std::vector<uint8_t> iSaved;
    std::vector<std::pair<uint64_t, uint64_t>> iCopies;
};

static int check_desc(const ohp_chunk_desc& d, uint64_t in_bytes, uint64_t out_bytes, DescDerived* derived = nullptr)
{
    DescFields f;
    f.src_off = d.src_off; f.dst_off = d.dst_off; f.bytes = d.bytes; f.ramp_start = d.ramp_start; f.ramp_end = d.ramp_end;
    f.attenuation = d.attenuation; f.bit_depth = d.bit_depth; f.channels = d.channels; f.flags = d.flags;
    f.out_fmt = d.out_fmt; f.aux = d.aux;
    DescDerived dv;
    const uint32_t err = check_desc_fields(f, in_bytes, out_bytes, dv);
    if (derived) *derived = dv;
    return err == 0 ? OHP_OK : (err == 1u ? OHP_E_INVALID_DESC : OHP_E_OUT_OF_RANGE);
}

static int launch(ohp_context* ctx, const ohp_chunk_desc* d_descs, size_t n, const uint8_t* d_in, uint64_t in_bytes,
                  uint8_t* d_out, uint64_t out_bytes, cudaStream_t st)
{
    if (n == 0) return OHP_OK;
    if ((reinterpret_cast<uint64_t>(d_in) & 15u) || (reinterpret_cast<uint64_t>(d_descs) & 15u)) {
        return fail(ctx, OHP_E_INVALID_ARG, "input arena and descriptor array must be 16-byte aligned");
    }
    KernelParams p;
    p.descs = d_descs;
    p.n = n;
    p.in = d_in;
    p.in_bytes = in_bytes;
    p.out = d_out;
    p.out_bytes = out_bytes;
    p.table2 = ctx->d_table2;
    p.status = ctx->d_status;
    p.cap_bytes = ctx->cap_bytes;
    p.cap_chunks = ctx->cap_chunks;
    p.serial_place = ctx->serial_place;
    uint64_t grid = (uint64_t)ctx->sm_count * (uint64_t)ctx->ctas_per_sm;
    // chunks are dealt in runs of chunk_block: long runs keep what a CTA has in flight inside one stretch of each arena,
    // short ones keep every CTA busy when the batch is small (at least ~8 runs per CTA)
    uint64_t chunk_block = ctx->chunk_block;
    while (chunk_block > kMinChunkBlock && n / chunk_block < grid * 8) chunk_block >>= 1;
    p.chunk_block = (uint32_t)chunk_block;
    const uint64_t blocks = (n + chunk_block - 1) / chunk_block;
    if (grid > blocks) grid = blocks;
    // in-flight tuning (see TuneEntry)
    TuneEntry* tune = nullptr;
    int trial = -1;
    if (ctx->autotune && !ctx->cap_pinned && in_bytes + out_bytes >= kTuneMinBytes && n >= kTuneMinChunks) {
        for (TuneEntry& t : ctx->tune) {
            if (t.n == n && t.in_bytes == in_bytes && t.out_bytes == out_bytes) tune = &t;
        }
        if (!tune) {
            if (ctx->tune.size() < 8) {
                ctx->tune.emplace_back();
                tune = &ctx->tune.back();
            } else {
                tune = &ctx->tune[0];
                for (TuneEntry& t : ctx->tune) if (t.last_use < tune->last_use) tune = &t;
                for (int c = 0; c < kTuneCandidates; c++) { tune->have[c] = false; }
                for (int t = 0; t < kTuneTrials; t++) { tune->done[t] = false; }
                tune->launched = 0;
            }
            tune->n = n; tune->in_bytes = in_bytes; tune->out_bytes = out_bytes;
        }
        tune->last_use = ++ctx->tune_clock;
        for (int t = 0; t < tune->launched; t++) {
            if (!tune->done[t] && cudaEventQuery(tune->ev[t][1]) == cudaSuccess) {
                float ms = 0.f;
                if (cudaEventElapsedTime(&ms, tune->ev[t][0], tune->ev[t][1]) == cudaSuccess) {
                    tune->ms[kTrialCandidate[t]] = ms;
                    tune->have[kTrialCandidate[t]] = true;
                    tune->done[t] = true;
                }
            }
        }
        (void)cudaGetLastError(); // cudaErrorNotReady from the query is not an error
        int best = -1;
        for (int c = 0; c < kTuneCandidates; c++) {
            if (tune->have[c] && (best < 0 || tune->ms[c] < tune->ms[best])) best = c;
        }
        if (tune->launched == kTuneCandidates && tune->have[0] && tune->have[1] && tune->have[2]) {
            // the warm re-trial of the first candidate is only worth a launch if it could still win
            const float other = tune->ms[1] < tune->ms[2] ? tune->ms[1] : tune->ms[2];
            if (tune->ms[0] > 1.06f * other) tune->launched = kTuneTrials;
        }
        if (tune->launched < kTuneTrials) {
            trial = tune->launched;
            for (int k = 0; k < 2; k++) {
                if (!tune->ev[trial][k]) OHP_CUDA(ctx, cudaEventCreate(&tune->ev[trial][k]));
            }
            p.cap_chunks = kTuneCaps[kTrialCandidate[trial]];
            p.serial_place = kTuneSerial[kTrialCandidate[trial]];
        } else if (best >= 0) {
            p.cap_chunks = kTuneCaps[best];
            p.serial_place = kTuneSerial[best];
        }
    }
    ctx->last_cap_chunks = p.cap_chunks;
    if (ctx->timing) OHP_CUDA(ctx, cudaEventRecord(ctx->ev_start, st));
    if (trial >= 0) OHP_CUDA(ctx, cudaEventRecord(tune->ev[trial][0], st));
    if (p.serial_place) ramp_convert_kernel<true><<<(unsigned)grid, kThreads, sizeof(SharedStorage), st>>>(p);
    else ramp_convert_kernel<false><<<(unsigned)grid, kThreads, sizeof(SharedStorage), st>>>(p);
    OHP_CUDA(ctx, cudaGetLastError());
    if (trial >= 0) {
        OHP_CUDA(ctx, cudaEventRecord(tune->ev[trial][1], st));
        tune->launched = trial + 1;
    }
    if (ctx->timing) {
        OHP_CUDA(ctx, cudaEventRecord(ctx->ev_stop, st));
        ctx->timed = true;
    }
    ctx->launches++;
    return OHP_OK;
}

// Cores of the NUMA node the device's PCIe root port belongs to (sysfs).  Pinned buffers are allocated from a thread
// bound to them, so that DMA between host memory and this GPU does not cross the socket interconnect: with one
// process per GPU on a two-socket box that is the difference between every rank hammering socket 0's memory and each
// rank using its own.
static bool device_local_cpus(int device, cpu_set_t* out)
{
    char bus[32] = {0};
    if (cudaDeviceGetPCIBusId(bus, (int)sizeof bus, device) != cudaSuccess) {
        (void)cudaGetLastError();
        return false;
    }
    for (char* c = bus; *c; c++) *c = (char)std::tolower((unsigned char)*c);
    char path[128];
    std::snprintf(path, sizeof path, "/sys/bus/pci/devices/%s/numa_node", bus);
    FILE* f = std::fopen(path, "r");
    if (!f) return false;
    int node = -1;
    const int got = std::fscanf(f, "%d", &node);
    std::fclose(f);
    if (got != 1 || node < 0) return false;
    std::snprintf(path, sizeof path, "/sys/devices/system/node/node%d/cpulist", node);
    f = std::fopen(path, "r");
    if (!f) return false;
    char list[1024] = {0};
    const bool ok = std::fgets(list, (int)sizeof list, f) != nullptr;
    std::fclose(f);
    if (!ok) return false;
    CPU_ZERO(out);
    int count = 0;
    for (const char* c = list; *c;) {
        if (!std::isdigit((unsigned char)*c)) { c++; continue; }
        char* end = nullptr;
        long lo = std::strtol(c, &end, 10), hi = lo;
        if (*end == '-') hi = std::strtol(end + 1, &end, 10);
        for (long k = lo; k <= hi && k < CPU_SETSIZE; k++) { CPU_SET((int)k, out); count++; }
        c = end;
    }
    return count > 0;
}

template <class T>
static int grow(ohp_context* ctx, T*& ptr, uint64_t& cap, uint64_t need)
{
    if (need <= cap) return OHP_OK;
    if (ptr) OHP_CUDA(ctx, cudaFree(ptr));
    ptr = nullptr;
    cap = 0;
    const uint64_t want = need + need / 8 + 256;
    OHP_CUDA(ctx, cudaMalloc(reinterpret_cast<void**>(&ptr), want));
    cap = want;
    return OHP_OK;
}

// Device buffers another stream may still be reading: grown only once the device is idle.
template <class T>
static int grow_idle(ohp_context* ctx, T*& ptr, uint64_t& cap, uint64_t need)
{
    if (need <= cap) return OHP_OK;
    OHP_CUDA(ctx, cudaDeviceSynchronize());
    return grow(ctx, ptr, cap, need);
}

// What words [2], [3] of the status block (the schedule kernels') say, bits != 0: the status, and the message in buf.
static int schedule_error(uint32_t bits, uint32_t stream_word, char* buf, size_t size)
{
    const uint32_t stream_index = 0xffffffffu - stream_word;
    if (bits & (1u << sched::kErrSpec)) {
        std::snprintf(buf, size, "stream %u: spec not representable (rate, frame size, chunk size, event slice or sink)", stream_index);
        return OHP_E_INVALID_ARG;
    }
    if (bits & (1u << sched::kErrAssert)) {
        std::snprintf(buf, size, "stream %u: the reference would ASSERT on this schedule", stream_index);
        return OHP_E_INVALID_DESC;
    }
    if (bits & (1u << sched::kErrBound)) {
        std::snprintf(buf, size, "stream %u: more playables than its descriptor region holds", stream_index);
        return OHP_E_NO_MEMORY;
    }
    std::snprintf(buf, size, "stream %u: more than %d pending message splits in one stage", stream_index, sched::kStackDepth);
    return OHP_E_NO_MEMORY;
}

// ohp_schedule_count_device: only the schedule kernels have run on the caller's buffers
static int schedule_status(ohp_context* ctx, cudaStream_t st)
{
    OHP_CUDA(ctx, cudaMemcpyAsync(ctx->h_status, ctx->d_status, 16 * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    OHP_CUDA(ctx, cudaStreamSynchronize(st));
    const uint32_t bits = ctx->h_status[2];
    if (bits == 0) return OHP_OK;
    const uint32_t stream_word = ctx->h_status[3];
    OHP_CUDA(ctx, cudaMemsetAsync(ctx->d_status + 2, 0, 2 * sizeof(uint32_t), st));
    OHP_CUDA(ctx, cudaStreamSynchronize(st));
    char buf[160];
    const int status = schedule_error(bits, stream_word, buf, sizeof buf);
    return fail(ctx, status, buf);
}

// Every error word of the status block -- [0], [1] the chunk kernels', [2], [3] the schedule kernels', [12], [13] the
// flywheel kernel's -- is read and cleared together, so that an error is reported once, by the first call or ohp_sync that
// reads it, and never again by a later one.  The status is the first of: a flywheel job, a stream the walk refused, a chunk
// descriptor (or the watchdog); ohp_last_error names every error found, in that order.
static int read_status(ohp_context* ctx, cudaStream_t st)
{
    OHP_CUDA(ctx, cudaMemcpyAsync(ctx->h_status, ctx->d_status, 16 * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    OHP_CUDA(ctx, cudaStreamSynchronize(st));
    const uint32_t fly_bits = ctx->h_status[12], job = ctx->h_status[13];
    const uint32_t sched_bits = ctx->h_status[2], stream_word = ctx->h_status[3];
    const uint32_t bits = ctx->h_status[0], first = ctx->h_status[1];
    if (fly_bits == 0 && sched_bits == 0 && bits == 0) return OHP_OK;
    OHP_CUDA(ctx, cudaMemsetAsync(ctx->d_status, 0, 4 * sizeof(uint32_t), st));
    OHP_CUDA(ctx, cudaMemsetAsync(ctx->d_status + 12, 0, 2 * sizeof(uint32_t), st));
    OHP_CUDA(ctx, cudaStreamSynchronize(st));
    int status = OHP_OK;
    std::string msg;
    auto note = [&](int s, const char* what) {
        if (status == OHP_OK) status = s;
        if (!msg.empty()) msg += "; ";
        msg += what;
    };
    char buf[160];
    if (fly_bits != 0) {
        std::snprintf(buf, sizeof buf, "device rejected flywheel job %u (%s)", job - 1, (fly_bits & 1u) ? "invalid" : "out of range");
        note((fly_bits & 1u) ? OHP_E_INVALID_DESC : OHP_E_OUT_OF_RANGE, buf);
    }
    if (sched_bits != 0) { // a walk enqueued by ohp_run_streams_device refused a stream
        const int s = schedule_error(sched_bits, stream_word, buf, sizeof buf);
        note(s, buf);
    }
    if (bits & kErrWatchdog) {
        note(OHP_E_CUDA, "kernel watchdog: a pipeline barrier never completed");
    } else if (bits != 0) {
        std::snprintf(buf, sizeof buf, "device rejected chunk descriptor %u (%s)", first - 1,
                      (bits & kErrInvalidDesc) ? "invalid" : "out of range");
        note((bits & kErrInvalidDesc) ? OHP_E_INVALID_DESC : OHP_E_OUT_OF_RANGE, buf);
    }
    return fail(ctx, status, msg.c_str());
}

} // namespace ohp

using namespace ohp;

extern "C" {

uint32_t ohp_abi_version(void) { return OHP_ABI_VERSION; }

int ohp_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        (void)cudaGetLastError();
        return 0;
    }
    return n;
}

const uint16_t* ohp_ramp_table(void) { return kRampTable; }

uint32_t ohp_median_multiplier(uint32_t ramp_start, uint32_t ramp_end, uint32_t direction, int enabled)
{
    if (!enabled) return 0x8000u;           // MsgAudio::MedianRampMultiplier, Msg.cpp:2065-2067
    if (direction == 3u) return 0;          // EMute, Msg.cpp:2068-2070 / 912-913
    uint32_t med;
    if (direction == 1u) med = ramp_start + ((ramp_end - ramp_start) / 2);       // EUp,   Msg.cpp:906-908
    else if (direction == 2u) med = ramp_start - ((ramp_start - ramp_end) / 2);  // EDown, Msg.cpp:909-911
    else med = ramp_start;
    const uint32_t idx = (OHP_RAMP_MAX - OHP_RAMP_MIN - med + (1u << 4)) >> 5;
    return idx < OHP_RAMP_TABLE_ENTRIES ? kRampTable[idx] : 0u;
}

uint32_t ohp_chunk_out_bytes(const ohp_chunk_desc* d)
{
    if (!d) return 0;
    DescDerived dv;
    (void)check_desc(*d, UINT64_MAX, UINT64_MAX, &dv);
    return dv.out_bytes;
}

int ohp_validate(const ohp_chunk_desc* descs, size_t n, uint64_t in_bytes, uint64_t out_bytes, size_t* bad_index)
{
    if (!descs && n) return OHP_E_INVALID_ARG;
    // the first offending descriptor in [lo, hi), or hi
    auto scan = [&](size_t lo, size_t hi, int* rc_out) -> size_t {
        for (size_t i = lo; i < hi; i++) {
            const int rc = check_desc(descs[i], in_bytes, out_bytes);
            if (rc != OHP_OK) { *rc_out = rc; return i; }
        }
        return hi;
    };
    // large batches (ohp_process_host checks millions of descriptors before the first byte moves): over a few threads
    unsigned workers = 1;
    if (n >= (1u << 18)) {
        workers = std::thread::hardware_concurrency();
        workers = workers == 0 ? 1u : (workers > 8u ? 8u : workers);
    }
    size_t first_bad = n;
    int first_rc = OHP_OK;
    if (workers <= 1) {
        first_bad = scan(0, n, &first_rc);
    }
    else {
        std::vector<size_t> bad(workers, n);
        std::vector<int> rcs(workers, OHP_OK);
        std::vector<std::thread> pool;
        const size_t per = (n + workers - 1) / workers;
        for (unsigned t = 0; t < workers; t++) {
            const size_t lo = (size_t)t * per < n ? (size_t)t * per : n;
            const size_t hi = lo + per < n ? lo + per : n;
            pool.emplace_back([&, t, lo, hi] { const size_t b = scan(lo, hi, &rcs[t]); bad[t] = b < hi ? b : n; });
        }
        for (std::thread& th : pool) th.join();
        for (unsigned t = 0; t < workers; t++) {
            if (bad[t] < first_bad) { first_bad = bad[t]; first_rc = rcs[t]; }
        }
    }
    if (first_bad < n) {
        if (bad_index) *bad_index = first_bad;
        return first_rc;
    }
    return OHP_OK;
}

int ohp_create(int device, ohp_context** out_ctx)
{
    if (!out_ctx) return OHP_E_INVALID_ARG;
    *out_ctx = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) {
        (void)cudaGetLastError();
        return fail(nullptr, OHP_E_NO_DEVICE, "no CUDA device available (this library has no CPU fallback)", e);
    }
    if (device < 0 || device >= n) return fail(nullptr, OHP_E_INVALID_ARG, "device index out of range");
    cudaDeviceProp prop;
    e = cudaGetDeviceProperties(&prop, device);
    if (e != cudaSuccess) return fail(nullptr, OHP_E_CUDA, "cudaGetDeviceProperties", e);
    if (prop.major != 10) {
        return fail(nullptr, OHP_E_NO_DEVICE, "device is not an sm_100 (Blackwell B200) part; kernels are built for sm_100a only");
    }
    ohp_context* ctx = new (std::nothrow) ohp_context();
    if (!ctx) return fail(nullptr, OHP_E_NO_MEMORY, "out of host memory");
    ctx->device = device;
    ctx->sm_count = prop.multiProcessorCount;
    ctx->have_local_cpus = device_local_cpus(device, &ctx->local_cpus);
    if (const char* e = std::getenv("OHP_CAP_BYTES")) {
        const long v = std::atol(e);
        if (v >= (long)(2 * (kSlotFront + kMaxChunk + 16 + kSlotBack)) && v <= (long)kRingBytes) { ctx->cap_bytes = (uint32_t)v; ctx->cap_pinned = true; }
    }
    if (const char* e = std::getenv("OHP_AUTOTUNE")) ctx->autotune = std::atoi(e) != 0;
    if (const char* e = std::getenv("OHP_CHUNK_BLOCK")) {
        const long v = std::atol(e);
        if (v >= 1 && v <= 65536) ctx->chunk_block = (uint32_t)v;
    }
    if (const char* e = std::getenv("OHP_CAP_CHUNKS")) {
        const long v = std::atol(e);
        if (v >= 1 && v <= (long)kRingSlots) { ctx->cap_chunks = (uint32_t)v; ctx->cap_pinned = true; }
    }
    if (const char* e = std::getenv("OHP_SERIAL_PLACE")) ctx->serial_place = std::atoi(e) != 0 ? 1u : 0u;
#define OHP_CREATE(call)                                                          \
    do {                                                                          \
        cudaError_t e_ = (call);                                                  \
        if (e_ != cudaSuccess) {                                                  \
            fail(nullptr, OHP_E_CUDA, #call, e_);                                 \
            ohp_destroy(ctx);                                                     \
            return OHP_E_CUDA;                                                    \
        }                                                                         \
    } while (0)
    OHP_CREATE(cudaSetDevice(device));
    {
        // the compute stream at the device's greatest priority: the walk and kernel times of DESIGN 4 were measured so
        int least = 0, greatest = 0;
        OHP_CREATE(cudaDeviceGetStreamPriorityRange(&least, &greatest));
        OHP_CREATE(cudaStreamCreateWithPriority(&ctx->stream, cudaStreamNonBlocking, greatest));
    }
    OHP_CREATE(cudaStreamCreateWithFlags(&ctx->copy_in, cudaStreamNonBlocking));
    OHP_CREATE(cudaStreamCreateWithFlags(&ctx->copy_out, cudaStreamNonBlocking));
    OHP_CREATE(cudaEventCreate(&ctx->ev_start));
    OHP_CREATE(cudaEventCreate(&ctx->ev_stop));
    OHP_CREATE(cudaEventCreateWithFlags(&ctx->scratch_done, cudaEventDisableTiming));
    OHP_CREATE(cudaMalloc(reinterpret_cast<void**>(&ctx->d_table2), sizeof(uint16_t) * OHP_RAMP_TABLE_ENTRIES));
    OHP_CREATE(cudaMalloc(reinterpret_cast<void**>(&ctx->d_status), 16 * sizeof(uint32_t)));
    OHP_CREATE(cudaMallocHost(reinterpret_cast<void**>(&ctx->h_status), 16 * sizeof(uint32_t)));
    OHP_CREATE(cudaMemset(ctx->d_status, 0, 16 * sizeof(uint32_t)));
    {
        uint16_t t2[OHP_RAMP_TABLE_ENTRIES];
        for (unsigned i = 0; i < OHP_RAMP_TABLE_ENTRIES; i++) t2[i] = (uint16_t)(2u * kRampTable[i]);
        OHP_CREATE(cudaMemcpy(ctx->d_table2, t2, sizeof t2, cudaMemcpyHostToDevice));
        uint32_t magic[33];
        magic[0] = magic[1] = 0;
        for (uint32_t ch = 2; ch <= 32; ch++) magic[ch] = (uint32_t)((((uint64_t)1 << 32) + ch - 1) / ch);
        OHP_CREATE(cudaMemcpyToSymbol(c_ch_magic, magic, sizeof magic));
    }
    {
        int per_sm = 0;
        OHP_CREATE(cudaFuncSetAttribute(ramp_convert_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(SharedStorage)));
        OHP_CREATE(cudaFuncSetAttribute(ramp_convert_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(SharedStorage)));
        // The schedule and scan kernels need (next to) no shared memory and would get the L1-heavy split of an SM's 256 KB;
        // they ask for ramp_convert_kernel's split instead (an SM cannot change its split while CTAs are resident).  The
        // walk times of DESIGN 4.2 were measured so.
        OHP_CREATE(cudaFuncSetAttribute(sched::schedule_kernel<false, 32>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
        OHP_CREATE(cudaFuncSetAttribute(sched::schedule_kernel<true, 32>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
        OHP_CREATE(cudaFuncSetAttribute(sched::schedule_kernel<false, 1>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
        OHP_CREATE(cudaFuncSetAttribute(sched::schedule_kernel<true, 1>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
        OHP_CREATE(cudaFuncSetAttribute(sched::schedule_record_kernel<32>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
        OHP_CREATE(cudaFuncSetAttribute(sched::schedule_record_kernel<1>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
        OHP_CREATE(cudaFuncSetAttribute(sched::schedule_recent_kernel<32>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
        OHP_CREATE(cudaFuncSetAttribute(sched::schedule_recent_kernel<1>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
        OHP_CREATE(cudaFuncSetAttribute(sched::scan_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
        OHP_CREATE(cudaFuncSetAttribute(ramp_convert_kernel<true>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
        OHP_CREATE(cudaFuncSetAttribute(ramp_convert_kernel<false>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
        OHP_CREATE(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, ramp_convert_kernel<false>, kThreads, sizeof(SharedStorage)));
        ctx->ctas_per_sm = per_sm > 0 ? per_sm : 1;
    }
#undef OHP_CREATE
    *out_ctx = ctx;
    return OHP_OK;
}

int ohp_destroy(ohp_context* ctx)
{
    if (!ctx) return OHP_E_INVALID_ARG;
    if (ctx->device >= 0) (void)cudaSetDevice(ctx->device);
    if (ctx->copy_in) (void)cudaStreamSynchronize(ctx->copy_in);
    if (ctx->stream) (void)cudaStreamSynchronize(ctx->stream);
    if (ctx->copy_out) (void)cudaStreamSynchronize(ctx->copy_out);
    if (ctx->scratch_done) (void)cudaEventSynchronize(ctx->scratch_done); // the last call may have been on the caller's stream
    (void)cudaGetLastError();
    if (ctx->d_in) (void)cudaFree(ctx->d_in);
    if (ctx->d_out) (void)cudaFree(ctx->d_out);
    if (ctx->d_descs) (void)cudaFree(ctx->d_descs);
    if (ctx->d_table2) (void)cudaFree(ctx->d_table2);
    if (ctx->d_status) (void)cudaFree(ctx->d_status);
    if (ctx->d_specs) (void)cudaFree(ctx->d_specs);
    if (ctx->d_events) (void)cudaFree(ctx->d_events);
    if (ctx->d_begin) (void)cudaFree(ctx->d_begin);
    if (ctx->d_outb) (void)cudaFree(ctx->d_outb);
    if (ctx->d_counts) (void)cudaFree(ctx->d_counts);
    if (ctx->h_regions) (void)cudaFreeHost(ctx->h_regions);
    for (void* p : {(void*)ctx->d_records, (void*)ctx->d_slot, (void*)ctx->d_owner, (void*)ctx->d_fly_slots, (void*)ctx->d_fly_descs,
                    (void*)ctx->d_fly_jobs, (void*)ctx->d_fly_train, (void*)ctx->d_fly_gen, (void*)ctx->d_recent, (void*)ctx->d_recent_count}) {
        if (p) (void)cudaFree(p);
    }
    if (ctx->sched_event) (void)cudaEventDestroy(ctx->sched_event);
    if (ctx->fly_event) (void)cudaEventDestroy(ctx->fly_event);
    if (ctx->scratch_done) (void)cudaEventDestroy(ctx->scratch_done);
    if (ctx->h_status) (void)cudaFreeHost(ctx->h_status);
    if (ctx->ev_start) (void)cudaEventDestroy(ctx->ev_start);
    if (ctx->ev_stop) (void)cudaEventDestroy(ctx->ev_stop);
    for (cudaEvent_t e : ctx->slice_events) (void)cudaEventDestroy(e);
    for (ohp::TuneEntry& t : ctx->tune) {
        for (int c = 0; c < ohp::kTuneTrials; c++) {
            if (t.ev[c][0]) (void)cudaEventDestroy(t.ev[c][0]);
            if (t.ev[c][1]) (void)cudaEventDestroy(t.ev[c][1]);
        }
    }
    if (ctx->stream) (void)cudaStreamDestroy(ctx->stream);
    if (ctx->copy_in) (void)cudaStreamDestroy(ctx->copy_in);
    if (ctx->copy_out) (void)cudaStreamDestroy(ctx->copy_out);
    delete ctx;
    return OHP_OK;
}

const char* ohp_last_error(const ohp_context* ctx)
{
    return ctx ? ctx->error.c_str() : g_create_error.c_str();
}

int ohp_process_device(ohp_context* ctx, const ohp_chunk_desc* d_descs, size_t n, const uint8_t* d_in, uint64_t in_bytes,
                       uint8_t* d_out, uint64_t out_bytes, void* stream)
{
    if (!ctx) return OHP_E_INVALID_ARG;
    if (n && (!d_descs || !d_out || (!d_in && in_bytes))) return fail(ctx, OHP_E_INVALID_ARG, "null device pointer");
    OHP_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = stream ? static_cast<cudaStream_t>(stream) : ctx->stream;
    return launch(ctx, d_descs, n, d_in, in_bytes, d_out, out_bytes, st);
}

int ohp_sync(ohp_context* ctx, void* stream)
{
    if (!ctx) return OHP_E_INVALID_ARG;
    OHP_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = stream ? static_cast<cudaStream_t>(stream) : ctx->stream;
    OHP_CUDA(ctx, cudaStreamSynchronize(st));
    return read_status(ctx, st);
}

int ohp_process_host(ohp_context* ctx, const ohp_chunk_desc* h_descs, size_t n, const uint8_t* h_in, uint64_t in_bytes,
                     uint8_t* h_out, uint64_t out_bytes)
{
    if (!ctx) return OHP_E_INVALID_ARG;
    if (n == 0) return OHP_OK;
    if (!h_descs || !h_out || (!h_in && in_bytes)) return fail(ctx, OHP_E_INVALID_ARG, "null host pointer");
    size_t bad = 0;
    const int vrc = ohp_validate(h_descs, n, in_bytes, out_bytes, &bad);
    if (vrc != OHP_OK) {
        char buf[96];
        std::snprintf(buf, sizeof buf, "chunk descriptor %zu rejected (%s)", bad,
                      vrc == OHP_E_INVALID_DESC ? "invalid" : "out of range");
        return fail(ctx, vrc, buf);
    }
    OHP_CUDA(ctx, cudaSetDevice(ctx->device));
    const ScratchTurn turn(ctx, ctx->stream);
    if (turn.rc != OHP_OK) return turn.rc;
    int rc;
    if ((rc = grow(ctx, ctx->d_in, ctx->d_in_cap, in_bytes + 16)) != OHP_OK) return rc;
    if ((rc = grow(ctx, ctx->d_out, ctx->d_out_cap, out_bytes + 16)) != OHP_OK) return rc;
    if ((rc = grow(ctx, ctx->d_descs, ctx->d_descs_cap, (uint64_t)n * sizeof(ohp_chunk_desc))) != OHP_OK) return rc;

    // Slices of consecutive descriptors, each moving about kSliceBytes over PCIe, pipelined over three streams:
    //   copy_in: H2D of the slice's descriptors and of the input span its chunks read
    //   stream : kernel over the slice
    //   copy_out: D2H of the output span its chunks write
    // The device arenas are full size, so slices never alias; the input span is [min offset, max end) over the slice,
    // the output goes back range by range (CopyBackPlan): h_out bytes no chunk covers are left as the caller had them.
    const uint64_t kSliceBytes = 48ull << 20;
    // declared in this order: on every exit the streams drain first, then the bridged holes are put back
    CopyBackPlan plan(h_out);
    const DrainOnExit drain(ctx, ctx->stream);
    auto add_ranges = [&](RangeSet& set, const ohp_chunk_desc& d) {
        if (d.out_fmt == OHP_OUT_PACKED_BE) { set.Add(d.dst_off, d.bytes); return; }
        DescDerived dv;
        (void)check_desc(d, in_bytes, out_bytes, &dv);
        if (d.out_fmt == OHP_OUT_PLANAR32_BE) {
            // one range per channel plane: the planes are aux frames apart and only dv.frames of each are written
            for (uint32_t c = 0; c < d.channels; c++) set.Add(d.dst_off + (uint64_t)c * d.aux * 4u, (uint64_t)dv.frames * 4u);
        } else {
            set.Add(d.dst_off, dv.out_bytes);
        }
    };
    for (size_t i = 0; i < n; i++) add_ranges(plan.Batch(), h_descs[i]);
    plan.SaveHoles();
    std::vector<cudaEvent_t>& evs = ctx->slice_events;
    size_t ev_used = 0;
    auto next_event = [&](cudaEvent_t* out_ev) -> cudaError_t {
        if (ev_used == evs.size()) {
            cudaEvent_t e;
            cudaError_t err = cudaEventCreateWithFlags(&e, cudaEventDisableTiming);
            if (err != cudaSuccess) return err;
            evs.push_back(e);
        }
        *out_ev = evs[ev_used++];
        return cudaSuccess;
    };
    const SliceMode slice_mode(ctx); // per-kernel events are only meaningful for a single launch; slices are PCIe-bound
    size_t lo = 0;
    while (lo < n) {
        uint64_t in_lo = UINT64_MAX, in_hi = 0, moved = 0;
        size_t hi = lo;
        while (hi < n && (moved < kSliceBytes || hi == lo)) {
            const ohp_chunk_desc& d = h_descs[hi];
            if (d.bytes) {
                if (!(d.flags & OHP_F_SILENCE)) {
                    in_lo = d.src_off < in_lo ? d.src_off : in_lo;
                    in_hi = d.src_off + d.bytes > in_hi ? d.src_off + d.bytes : in_hi;
                }
                add_ranges(plan.Slice(), d);
                moved += 2ull * d.bytes;
            }
            hi++;
        }
        cudaEvent_t ev_in, ev_k;
        OHP_CUDA(ctx, next_event(&ev_in));
        OHP_CUDA(ctx, next_event(&ev_k));
        OHP_CUDA(ctx, cudaMemcpyAsync(ctx->d_descs + lo, h_descs + lo, (hi - lo) * sizeof(ohp_chunk_desc),
                                      cudaMemcpyHostToDevice, ctx->copy_in));
        if (in_hi > in_lo) {
            OHP_CUDA(ctx, cudaMemcpyAsync(ctx->d_in + in_lo, h_in + in_lo, in_hi - in_lo, cudaMemcpyHostToDevice, ctx->copy_in));
        }
        OHP_CUDA(ctx, cudaEventRecord(ev_in, ctx->copy_in));
        OHP_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, ev_in, 0));
        if ((rc = launch(ctx, ctx->d_descs + lo, hi - lo, ctx->d_in, in_bytes, ctx->d_out, out_bytes, ctx->stream)) != OHP_OK) return rc;
        OHP_CUDA(ctx, cudaEventRecord(ev_k, ctx->stream));
        OHP_CUDA(ctx, cudaStreamWaitEvent(ctx->copy_out, ev_k, 0));
        for (const auto& c : plan.Copies()) {
            OHP_CUDA(ctx, cudaMemcpyAsync(h_out + c.first, ctx->d_out + c.first, c.second - c.first, cudaMemcpyDeviceToHost, ctx->copy_out));
        }
        lo = hi;
    }
    OHP_CUDA(ctx, cudaStreamSynchronize(ctx->copy_out));
    OHP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return read_status(ctx, ctx->stream);
}

int ohp_checksums_device(ohp_context* ctx, const uint8_t* d_out, const uint64_t* d_stream_off, size_t n_streams,
                         uint64_t* d_sums, void* stream)
{
    if (!ctx) return OHP_E_INVALID_ARG;
    if (n_streams == 0) return OHP_OK;
    if (!d_out || !d_stream_off || !d_sums) return fail(ctx, OHP_E_INVALID_ARG, "null device pointer");
    OHP_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = stream ? static_cast<cudaStream_t>(stream) : ctx->stream;
    uint64_t grid = (uint64_t)ctx->sm_count * 8u;
    if (grid > n_streams) grid = n_streams;
    checksum_kernel<<<(unsigned)grid, 256, 0, st>>>(d_out, d_stream_off, n_streams, d_sums, 1u);
    OHP_CUDA(ctx, cudaGetLastError());
    ctx->launches++;
    return OHP_OK;
}

int ohp_device_alloc(ohp_context* ctx, uint64_t bytes, void** out_dptr)
{
    if (!ctx || !out_dptr) return OHP_E_INVALID_ARG;
    OHP_CUDA(ctx, cudaSetDevice(ctx->device));
    OHP_CUDA(ctx, cudaMalloc(out_dptr, bytes ? bytes : 1));
    return OHP_OK;
}

int ohp_device_free(ohp_context* ctx, void* dptr)
{
    if (!ctx) return OHP_E_INVALID_ARG;
    OHP_CUDA(ctx, cudaSetDevice(ctx->device));
    OHP_CUDA(ctx, cudaFree(dptr));
    return OHP_OK;
}

int ohp_host_alloc(ohp_context* ctx, uint64_t bytes, void** out_hptr)
{
    if (!ctx || !out_hptr) return OHP_E_INVALID_ARG;
    OHP_CUDA(ctx, cudaSetDevice(ctx->device));
    // allocate (and thereby touch and pin) the pages from a thread bound to the GPU's NUMA node
    cpu_set_t saved;
    const bool rebind = ctx->have_local_cpus && sched_getaffinity(0, sizeof saved, &saved) == 0
                        && sched_setaffinity(0, sizeof ctx->local_cpus, &ctx->local_cpus) == 0;
    const cudaError_t e = cudaMallocHost(out_hptr, bytes ? bytes : 1);
    if (rebind) (void)sched_setaffinity(0, sizeof saved, &saved);
    if (e != cudaSuccess) return fail(ctx, OHP_E_CUDA, "cudaMallocHost", e);
    return OHP_OK;
}

int ohp_host_free(ohp_context* ctx, void* hptr)
{
    if (!ctx) return OHP_E_INVALID_ARG;
    OHP_CUDA(ctx, cudaFreeHost(hptr));
    return OHP_OK;
}

int ohp_memcpy_h2d(ohp_context* ctx, void* dptr, const void* hptr, uint64_t bytes, void* stream)
{
    if (!ctx) return OHP_E_INVALID_ARG;
    OHP_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = stream ? static_cast<cudaStream_t>(stream) : ctx->stream;
    OHP_CUDA(ctx, cudaMemcpyAsync(dptr, hptr, bytes, cudaMemcpyHostToDevice, st));
    return OHP_OK;
}

int ohp_memcpy_d2h(ohp_context* ctx, void* hptr, const void* dptr, uint64_t bytes, void* stream)
{
    if (!ctx) return OHP_E_INVALID_ARG;
    OHP_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = stream ? static_cast<cudaStream_t>(stream) : ctx->stream;
    OHP_CUDA(ctx, cudaMemcpyAsync(hptr, dptr, bytes, cudaMemcpyDeviceToHost, st));
    return OHP_OK;
}

// Device-side schedule builder (include/ohp_schedule_device.h) -------------------------------------------------


// Threads per stream in the schedule kernels: a warp while warps-per-stream still fit the GPU a few times over, else one
// thread.  OHP_SCHED_TEAM=1|32 pins it (experiments).
static int schedule_team(size_t n_streams)
{
    static const int pinned = [] {
        const char* e = std::getenv("OHP_SCHED_TEAM");
        const int v = e ? std::atoi(e) : 0;
        return (v == 1 || v == 32) ? v : 0;
    }();
    if (pinned) return pinned;
    return n_streams <= kScheduleWarpTeamMaxStreams ? 32 : 1;
}

// Streams per warp when a thread walks a stream (see schedule_kernel): as many as it takes to have about one warp per warp
// scheduler (4 per SM), no more.  Threads of a warp that walk different streams take turns wherever their paths differ, so
// fewer streams per warp are faster per warp -- until there are more warps than schedulers: the walk is 690 KB of code,
// and warps sharing a scheduler share an instruction cache they each drag a different part of it through.  Measured
// (profiles/README.md, GPU call 32): 4096 streams (configs[2]) 32 per warp 1.09 ms, 8 per warp 0.79, 2 per warp 1.37;
// 16384 streams (configs[3]) 32 per warp 1.95 ms, 16 per warp 2.15, 1 per warp 3.7.  OHP_SCHED_LANES=k pins it (experiments).
static uint32_t schedule_lanes(const ohp_context* ctx, size_t n_streams)
{
    static const int pinned = [] {
        const char* e = std::getenv("OHP_SCHED_LANES");
        const int v = e ? std::atoi(e) : 0;
        return (v >= 1 && v <= 32) ? v : 0;
    }();
    if (pinned) return (uint32_t)pinned;
    const size_t schedulers = (size_t)(ctx->sm_count > 0 ? ctx->sm_count : 148) * 4u;
    const size_t lanes = (n_streams + schedulers - 1) / schedulers;
    return lanes < 1 ? 1u : (lanes > 32 ? 32u : (uint32_t)lanes);
}

int ohp_schedule_count_device(ohp_context* ctx, const ohp_stream_spec* d_streams, size_t n_streams,
                              const ohp_ramp_event* d_events, size_t n_events, uint64_t* d_chunk_begin,
                              uint64_t* d_stream_out_bytes, uint64_t* total_chunks, void* stream)
{
    if (!ctx) return OHP_E_INVALID_ARG;
    if (!total_chunks) return fail(ctx, OHP_E_INVALID_ARG, "null total_chunks");
    *total_chunks = 0;
    if (!d_chunk_begin || (n_streams && !d_streams) || (n_events && !d_events)) return fail(ctx, OHP_E_INVALID_ARG, "null device pointer");
    OHP_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = stream ? static_cast<cudaStream_t>(stream) : ctx->stream;
    sched::ScheduleParams p{};
    p.streams = d_streams; p.n_streams = n_streams; p.events = d_events; p.n_events = n_events;
    p.chunk_count = d_chunk_begin; p.out_bytes = d_stream_out_bytes;
    p.status = ctx->d_status + 2;
    if (n_streams) {
        if (schedule_team(n_streams) == 32) {
            sched::schedule_kernel<false, 32><<<sched::schedule_grid(n_streams, 32), sched::kScheduleBlock, 0, st>>>(p);
        } else {
            p.lanes_per_warp = schedule_lanes(ctx, n_streams);
            sched::schedule_kernel<false, 1><<<sched::schedule_grid(n_streams, 1, p.lanes_per_warp), sched::kScheduleBlock, 0, st>>>(p);
        }
        OHP_CUDA(ctx, cudaGetLastError());
        ctx->launches++;
    }
    sched::scan_kernel<<<1, sched::kScanThreads, 0, st>>>(d_chunk_begin, n_streams);
    OHP_CUDA(ctx, cudaGetLastError());
    ctx->launches++;
    uint64_t* h_total = reinterpret_cast<uint64_t*>(ctx->h_status + 14); // 8-byte aligned tail of the pinned status block
    OHP_CUDA(ctx, cudaMemcpyAsync(h_total, d_chunk_begin + n_streams, sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    OHP_CUDA(ctx, cudaStreamSynchronize(st));
    const uint64_t total = *h_total;
    const int rc = schedule_status(ctx, st);
    if (rc != OHP_OK) return rc;
    *total_chunks = total;
    return OHP_OK;
}

int ohp_schedule_emit_device(ohp_context* ctx, const ohp_stream_spec* d_streams, size_t n_streams,
                             const ohp_ramp_event* d_events, size_t n_events, const uint64_t* d_chunk_begin,
                             ohp_chunk_desc* d_chunks, ohp_chunk_info* d_info, void* stream)
{
    if (!ctx) return OHP_E_INVALID_ARG;
    if (n_streams == 0) return OHP_OK;
    if (!d_streams || !d_chunk_begin || !d_chunks || (n_events && !d_events)) return fail(ctx, OHP_E_INVALID_ARG, "null device pointer");
    if (reinterpret_cast<uint64_t>(d_chunks) & 15u) return fail(ctx, OHP_E_INVALID_ARG, "descriptor array must be 16-byte aligned");
    OHP_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = stream ? static_cast<cudaStream_t>(stream) : ctx->stream;
    sched::ScheduleParams p{};
    p.streams = d_streams; p.n_streams = n_streams; p.events = d_events; p.n_events = n_events;
    p.chunk_begin = d_chunk_begin; p.descs = d_chunks; p.info = d_info;
    p.status = ctx->d_status + 2;
    if (schedule_team(n_streams) == 32) {
        sched::schedule_kernel<true, 32><<<sched::schedule_grid(n_streams, 32), sched::kScheduleBlock, 0, st>>>(p);
    } else {
        p.lanes_per_warp = schedule_lanes(ctx, n_streams);
        sched::schedule_kernel<true, 1><<<sched::schedule_grid(n_streams, 1, p.lanes_per_warp), sched::kScheduleBlock, 0, st>>>(p);
    }
    OHP_CUDA(ctx, cudaGetLastError());
    ctx->launches++;
    return OHP_OK;
}

} // extern "C"

namespace ohp {

// The whole stage for a batch of streams in HOST memory (include/ohp_schedule_device.h).  Holes of up to `bridge` bytes
// between the streams' output ranges go back with the ranges around them and get the caller's bytes back at the end
// (CopyBackPlan): that is only right where nothing else writes into h_out while the call runs.
static int run_streams_host(ohp_context* ctx, const ohp_stream_spec* h_streams, size_t n_streams,
                            const ohp_ramp_event* h_events, size_t n_events,
                            const uint8_t* h_in, uint64_t in_bytes, uint8_t* h_out, uint64_t out_bytes,
                            uint64_t* h_stream_out_bytes, uint64_t* total_chunks, uint64_t bridge)
{
    if (!ctx) return OHP_E_INVALID_ARG;
    if (total_chunks) *total_chunks = 0;
    if (n_streams == 0) return OHP_OK;
    if (!h_streams || !h_out || (!h_in && in_bytes) || (n_events && !h_events)) return fail(ctx, OHP_E_INVALID_ARG, "null host pointer");
    OHP_CUDA(ctx, cudaSetDevice(ctx->device));
    const ScratchTurn turn(ctx, ctx->stream);
    if (turn.rc != OHP_OK) return turn.rc;
    int rc;
    if ((rc = grow(ctx, ctx->d_specs, ctx->d_specs_cap, (uint64_t)n_streams * sizeof(ohp_stream_spec))) != OHP_OK) return rc;
    if ((rc = grow(ctx, ctx->d_events, ctx->d_events_cap, (uint64_t)(n_events ? n_events : 1) * sizeof(ohp_ramp_event))) != OHP_OK) return rc;
    if ((rc = grow(ctx, ctx->d_begin, ctx->d_begin_cap, (uint64_t)(n_streams + 1) * sizeof(uint64_t))) != OHP_OK) return rc;
    if ((rc = grow(ctx, ctx->d_outb, ctx->d_outb_cap, (uint64_t)n_streams * sizeof(uint64_t))) != OHP_OK) return rc;
    if ((rc = grow(ctx, ctx->d_in, ctx->d_in_cap, in_bytes + 16)) != OHP_OK) return rc;
    if ((rc = grow(ctx, ctx->d_out, ctx->d_out_cap, out_bytes + 16)) != OHP_OK) return rc;
    cudaStream_t st = ctx->stream;
    // 1. descriptors, born and kept in HBM: specs and events are all that crosses PCIe on their behalf
    OHP_CUDA(ctx, cudaMemcpyAsync(ctx->d_specs, h_streams, n_streams * sizeof(ohp_stream_spec), cudaMemcpyHostToDevice, st));
    if (n_events) OHP_CUDA(ctx, cudaMemcpyAsync(ctx->d_events, h_events, n_events * sizeof(ohp_ramp_event), cudaMemcpyHostToDevice, st));
    uint64_t total = 0;
    if ((rc = ohp_schedule_count_device(ctx, ctx->d_specs, n_streams, ctx->d_events, n_events, ctx->d_begin, ctx->d_outb, &total, st)) != OHP_OK) return rc;
    if (total_chunks) *total_chunks = total;
    if ((rc = grow(ctx, ctx->d_descs, ctx->d_descs_cap, (total ? total : 1) * sizeof(ohp_chunk_desc))) != OHP_OK) return rc;
    if ((rc = ohp_schedule_emit_device(ctx, ctx->d_specs, n_streams, ctx->d_events, n_events, ctx->d_begin, ctx->d_descs, nullptr, st)) != OHP_OK) return rc;
    ctx->h_begin.resize(n_streams + 1);
    ctx->h_outb.resize(n_streams);
    OHP_CUDA(ctx, cudaMemcpyAsync(ctx->h_begin.data(), ctx->d_begin, (n_streams + 1) * sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    OHP_CUDA(ctx, cudaMemcpyAsync(ctx->h_outb.data(), ctx->d_outb, n_streams * sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    OHP_CUDA(ctx, cudaStreamSynchronize(st));
    if (h_stream_out_bytes) std::memcpy(h_stream_out_bytes, ctx->h_outb.data(), n_streams * sizeof(uint64_t));
    // every stream's spans must lie inside the arenas (the kernel checks each chunk too; this names the stream)
    for (size_t s = 0; s < n_streams; s++) {
        const ohp_stream_spec& sp = h_streams[s];
        const uint64_t frame_bytes = (uint64_t)sp.channels * (sp.bit_depth / 8u);
        const bool wraps = frame_bytes != 0 && sp.total_frames > UINT64_MAX / frame_bytes;
        const uint64_t in_len = sp.total_frames * frame_bytes;
        if (wraps || sp.src_base > in_bytes || in_len > in_bytes - sp.src_base || sp.dst_base > out_bytes || ctx->h_outb[s] > out_bytes - sp.dst_base) {
            char buf[96];
            std::snprintf(buf, sizeof buf, "stream %zu reaches outside the arenas", s);
            return fail(ctx, OHP_E_OUT_OF_RANGE, buf);
        }
    }
    // 2. PCM in slices of whole streams, H2D / kernel / D2H pipelined over three streams (as ohp_process_host)
    const uint64_t kSliceBytes = 48ull << 20;
    std::vector<cudaEvent_t>& evs = ctx->slice_events;
    size_t ev_used = 0;
    auto next_event = [&](cudaEvent_t* out_ev) -> cudaError_t {
        if (ev_used == evs.size()) {
            cudaEvent_t e;
            cudaError_t err = cudaEventCreateWithFlags(&e, cudaEventDisableTiming);
            if (err != cudaSuccess) return err;
            evs.push_back(e);
        }
        *out_ev = evs[ev_used++];
        return cudaSuccess;
    };
    const SliceMode slice_mode(ctx);
    CopyBackPlan plan(h_out, bridge); // a stream's chunks tile [dst_base, dst_base + its output bytes): one range per stream
    const DrainOnExit drain(ctx, st);
    for (size_t s = 0; s < n_streams; s++) plan.Batch().Add(h_streams[s].dst_base, ctx->h_outb[s]);
    plan.SaveHoles();
    size_t lo = 0;
    rc = OHP_OK;
    while (lo < n_streams && rc == OHP_OK) {
        uint64_t in_lo = UINT64_MAX, in_hi = 0, moved = 0;
        size_t hi = lo;
        while (hi < n_streams && (moved < kSliceBytes || hi == lo)) {
            const ohp_stream_spec& sp = h_streams[hi];
            const uint64_t in_len = sp.total_frames * (uint64_t)(sp.channels * (sp.bit_depth / 8u));
            if (in_len) {
                in_lo = sp.src_base < in_lo ? sp.src_base : in_lo;
                in_hi = sp.src_base + in_len > in_hi ? sp.src_base + in_len : in_hi;
            }
            plan.Slice().Add(sp.dst_base, ctx->h_outb[hi]);
            moved += in_len + ctx->h_outb[hi];
            hi++;
        }
        const uint64_t c_lo = ctx->h_begin[lo], c_hi = ctx->h_begin[hi];
        cudaEvent_t ev_in, ev_k;
        OHP_CUDA(ctx, next_event(&ev_in));
        OHP_CUDA(ctx, next_event(&ev_k));
        if (in_hi > in_lo) {
            OHP_CUDA(ctx, cudaMemcpyAsync(ctx->d_in + in_lo, h_in + in_lo, in_hi - in_lo, cudaMemcpyHostToDevice, ctx->copy_in));
        }
        OHP_CUDA(ctx, cudaEventRecord(ev_in, ctx->copy_in));
        OHP_CUDA(ctx, cudaStreamWaitEvent(st, ev_in, 0));
        rc = launch(ctx, ctx->d_descs + c_lo, (size_t)(c_hi - c_lo), ctx->d_in, in_bytes, ctx->d_out, out_bytes, st);
        if (rc != OHP_OK) break;
        OHP_CUDA(ctx, cudaEventRecord(ev_k, st));
        OHP_CUDA(ctx, cudaStreamWaitEvent(ctx->copy_out, ev_k, 0));
        for (const auto& c : plan.Copies()) {
            OHP_CUDA(ctx, cudaMemcpyAsync(h_out + c.first, ctx->d_out + c.first, c.second - c.first, cudaMemcpyDeviceToHost, ctx->copy_out));
        }
        lo = hi;
    }
    OHP_CUDA(ctx, cudaStreamSynchronize(ctx->copy_out));
    OHP_CUDA(ctx, cudaStreamSynchronize(st));
    if (rc != OHP_OK) return rc;
    return read_status(ctx, st);
}

} // namespace ohp

extern "C" {

int ohp_run_streams_host(ohp_context* ctx, const ohp_stream_spec* h_streams, size_t n_streams,
                         const ohp_ramp_event* h_events, size_t n_events,
                         const uint8_t* h_in, uint64_t in_bytes, uint8_t* h_out, uint64_t out_bytes,
                         uint64_t* h_stream_out_bytes, uint64_t* total_chunks)
{
    return run_streams_host(ctx, h_streams, n_streams, h_events, n_events, h_in, in_bytes, h_out, out_bytes,
                            h_stream_out_bytes, total_chunks, RangeSet::kBridge);
}

// The whole stage for a batch resident in HBM (include/ohp_schedule_device.h).
//
// ONE walk per stream: a closed-form upper bound (sched::stream_chunk_bound) gives every stream a region of the context's
// descriptor buffer, the walk writes what the stream has and zero-fills the rest of its region (a zero-byte descriptor is
// a playable MsgPlayable::Read does nothing for, and costs ramp_convert_kernel a record and a ticket).  No count pass, and
// the only host round trip is for the regions' total (bound + scan are a few microseconds of GPU time).
// A stream that outgrows its region (none of the shapes this repo generates does, the bound is held against the exact
// counts in tests/test_schedule_walk.py and tests/test_chunk_bound.py) sends the whole call through the two-pass path;
// tests/test_gpu_region_overflow.py makes streams outgrow regions capped by OHP_REGION_CAP.
// records (ohp_run_streams_device_flywheel): the emitting walk also leaves the starvation records there; with recent
// (ohp_run_streams_device_flywheel_recent) their pieces of recent audio too.
static int run_streams_device_two_pass(ohp_context* ctx, const ohp_stream_spec* d_streams, size_t n_streams,
                                       const ohp_ramp_event* d_events, size_t n_events,
                                       const uint8_t* d_in, uint64_t in_bytes, uint8_t* d_out, uint64_t out_bytes,
                                       uint64_t* d_stream_out_bytes, uint64_t* total_chunks, ohp_starvation* records, cudaStream_t st,
                                       const sched::RecentOut* recent = nullptr)
{
    int rc;
    uint64_t total = 0;
    if ((rc = ohp_schedule_count_device(ctx, d_streams, n_streams, d_events, n_events, ctx->d_begin, d_stream_out_bytes, &total, st)) != OHP_OK) return rc;
    if (total_chunks) *total_chunks = total;
    if (total > ctx->d_descs_cap / sizeof(ohp_chunk_desc)) {
        // the buffer may still be read by a launch enqueued earlier on another stream
        OHP_CUDA(ctx, cudaDeviceSynchronize());
        if ((rc = grow(ctx, ctx->d_descs, ctx->d_descs_cap, total * sizeof(ohp_chunk_desc))) != OHP_OK) return rc;
    }
    if (!records) {
        if ((rc = ohp_schedule_emit_device(ctx, d_streams, n_streams, d_events, n_events, ctx->d_begin, ctx->d_descs, nullptr, st)) != OHP_OK) return rc;
    }
    else {
        sched::ScheduleParams p{};
        p.streams = d_streams; p.n_streams = n_streams; p.events = d_events; p.n_events = n_events;
        p.chunk_begin = ctx->d_begin; p.descs = ctx->d_descs; p.info = nullptr;
        p.status = ctx->d_status + 2;
        p.records = records;
        if (schedule_team(n_streams) == 32) {
            if (recent) sched::schedule_recent_kernel<32><<<sched::schedule_grid(n_streams, 32), sched::kScheduleBlock, 0, st>>>(p, *recent);
            else sched::schedule_record_kernel<32><<<sched::schedule_grid(n_streams, 32), sched::kScheduleBlock, 0, st>>>(p);
        } else {
            p.lanes_per_warp = schedule_lanes(ctx, n_streams);
            const unsigned grid = sched::schedule_grid(n_streams, 1, p.lanes_per_warp);
            if (recent) sched::schedule_recent_kernel<1><<<grid, sched::kScheduleBlock, 0, st>>>(p, *recent);
            else sched::schedule_record_kernel<1><<<grid, sched::kScheduleBlock, 0, st>>>(p);
        }
        OHP_CUDA(ctx, cudaGetLastError());
        ctx->launches++;
    }
    return launch(ctx, ctx->d_descs, (size_t)total, d_in, in_bytes, d_out, out_bytes, st);
}

// What ohp_run_streams_device_flywheel adds to the call (null: ohp_run_streams_device).
struct FlyArgs
{
    uint8_t* out;
    uint64_t out_bytes;
    ohp_starvation* records; // the caller's, or the context's
    uint64_t* off;
    uint64_t* len;
    // ohp_run_streams_device_flywheel_recent: planned from the recent audio (the caller's arrays, or the context's)
    bool with_recent;
    sched::RecentOut recent;
    uint64_t prep_per() const { return with_recent ? OHP_FLYWHEEL_MAX_PREP_RECENT : OHP_FLYWHEEL_MAX_PREP; }
};

// The slots' total is known (h_regions[4..8)): refuse what the call cannot lay out.
static int fly_check(ohp_context* ctx, const FlyArgs& fly)
{
    const sched::FlySlots& fs = *reinterpret_cast<const sched::FlySlots*>(ctx->h_regions + 4);
    char buf[160];
    if (fs.shared != 0) {
        std::snprintf(buf, sizeof buf, "%llu events lie in the slices of two streams: a starvation record needs one stream per event",
                      (unsigned long long)fs.shared);
        return fail(ctx, OHP_E_INVALID_ARG, buf);
    }
    if (fs.bytes > fly.out_bytes || fs.bytes > sched::kSlotBytesMask || (fs.bytes && !fly.out)) {
        std::snprintf(buf, sizeof buf, "flywheel output: the starvation events' slots need %llu bytes, d_fly_out holds %llu",
                      (unsigned long long)fs.bytes, (unsigned long long)(fly.out ? fly.out_bytes : 0));
        return fail(ctx, OHP_E_OUT_OF_RANGE, buf);
    }
    return OHP_OK;
}

// Plan every starvation event's flywheel ramp from its record (device: nothing but the planned jobs' count comes back,
// behind ctx->fly_event) ...
static int fly_plan(ohp_context* ctx, const ohp_stream_spec* d_streams, size_t n_streams, size_t n_events, const FlyArgs& fly,
                    cudaStream_t st)
{
    const sched::FlySlots fs = *reinterpret_cast<const sched::FlySlots*>(ctx->h_regions + 4);
    if (fs.count == 0) return OHP_OK; // not one starvation event: the call is ohp_run_streams_device's, launch for launch
    const uint64_t per = fly.prep_per() + flyplan::kMaxBlocks;
    int rc;
    if ((rc = grow_idle(ctx, ctx->d_fly_descs, ctx->d_fly_descs_cap, fs.count * per * sizeof(ohp_chunk_desc))) != OHP_OK) return rc;
    if ((rc = grow_idle(ctx, ctx->d_fly_jobs, ctx->d_fly_jobs_cap, fs.count * sizeof(ohp_flywheel_job))) != OHP_OK) return rc;
    if (!ctx->fly_event) OHP_CUDA(ctx, cudaEventCreateWithFlags(&ctx->fly_event, cudaEventDisableTiming));
    sched::scan_kernel<<<1, sched::kScanThreads, 0, st>>>(ctx->d_slot, n_events);
    OHP_CUDA(ctx, cudaGetLastError());
    sched::PlanParams pp;
    pp.streams = d_streams; pp.n_streams = n_streams; pp.n_events = n_events; pp.records = fly.records; pp.slot = ctx->d_slot;
    pp.prep = ctx->d_fly_descs; pp.jobs = ctx->d_fly_jobs; pp.blocks = ctx->d_fly_descs + fs.count * fly.prep_per();
    pp.fly_off = fly.off; pp.fly_len = fly.len; pp.slots = ctx->d_fly_slots;
    if (fly.with_recent) sched::plan_recent_kernel<<<(unsigned)((n_events + 127) / 128), 128, 0, st>>>(pp, fly.recent.recent, fly.recent.count);
    else sched::plan_kernel<<<(unsigned)((n_events + 127) / 128), 128, 0, st>>>(pp);
    OHP_CUDA(ctx, cudaGetLastError());
    ctx->launches += 2;
    OHP_CUDA(ctx, cudaMemcpyAsync(ctx->h_regions + 4, ctx->d_fly_slots, sizeof(sched::FlySlots), cudaMemcpyDeviceToHost, st));
    OHP_CUDA(ctx, cudaEventRecord(ctx->fly_event, st));
    return OHP_OK;
}

// ... and play it: FlywheelInput::Prepare (prep), FlywheelRamperManager::Ramp (the compacted jobs), RampGenerator's blocks.
static int fly_play(ohp_context* ctx, const uint8_t* d_in, uint64_t in_bytes, const FlyArgs& fly, cudaStream_t st)
{
    const sched::FlySlots& fs = *reinterpret_cast<const sched::FlySlots*>(ctx->h_regions + 4);
    if (fs.count == 0) return OHP_OK;
    OHP_CUDA(ctx, cudaEventSynchronize(ctx->fly_event));
    const uint64_t count = fs.count, bytes = fs.bytes, planned = fs.planned;
    int rc;
    if ((rc = grow_idle(ctx, ctx->d_fly_train, ctx->d_fly_train_cap, bytes)) != OHP_OK) return rc;
    if ((rc = grow_idle(ctx, ctx->d_fly_gen, ctx->d_fly_gen_cap, bytes)) != OHP_OK) return rc;
    const ohp_chunk_desc* prep = ctx->d_fly_descs;
    const ohp_chunk_desc* blocks = ctx->d_fly_descs + count * fly.prep_per();
    if ((rc = launch(ctx, prep, (size_t)(count * fly.prep_per()), d_in, in_bytes, ctx->d_fly_train, bytes, st)) != OHP_OK) return rc;
    if ((rc = ohp_flywheel_device(ctx, ctx->d_fly_jobs, (size_t)planned, ctx->d_fly_train, bytes, ctx->d_fly_gen, bytes, st)) != OHP_OK) return rc;
    return launch(ctx, blocks, (size_t)(count * flyplan::kMaxBlocks), ctx->d_fly_gen, bytes, fly.out, fly.out_bytes, st);
}

// The body of ohp_run_streams_device and, with fly, of ohp_run_streams_device_flywheel.
static int run_streams_device(ohp_context* ctx, const ohp_stream_spec* d_streams, size_t n_streams,
                              const ohp_ramp_event* d_events, size_t n_events,
                              const uint8_t* d_in, uint64_t in_bytes, uint8_t* d_out, uint64_t out_bytes,
                              uint64_t* d_stream_out_bytes, uint64_t* total_chunks, void* stream, const FlyArgs* fly)
{
    if (!ctx) return OHP_E_INVALID_ARG;
    if (total_chunks) *total_chunks = 0;
    if (n_streams == 0) return OHP_OK;
    if (!d_streams || !d_out || (!d_in && in_bytes) || (n_events && !d_events)) return fail(ctx, OHP_E_INVALID_ARG, "null device pointer");
    OHP_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = stream ? static_cast<cudaStream_t>(stream) : ctx->stream;
    const ScratchTurn turn(ctx, st);
    if (turn.rc != OHP_OK) return turn.rc;
    int rc;
    if ((rc = grow(ctx, ctx->d_begin, ctx->d_begin_cap, (uint64_t)(n_streams + 1) * sizeof(uint64_t))) != OHP_OK) return rc;
    if ((rc = grow(ctx, ctx->d_counts, ctx->d_counts_cap, (uint64_t)n_streams * sizeof(uint64_t))) != OHP_OK) return rc;
    if (!ctx->h_regions) OHP_CUDA(ctx, cudaHostAlloc(reinterpret_cast<void**>(&ctx->h_regions), 8 * sizeof(uint64_t), cudaHostAllocDefault));
    if (!ctx->sched_event) OHP_CUDA(ctx, cudaEventCreateWithFlags(&ctx->sched_event, cudaEventDisableTiming));
    ohp_starvation* records = nullptr;
    FlyArgs flyArgs{}; // *fly with the context's scratch in place of the arrays the caller left NULL
    if (fly) {
        // records (none yet: all ones), slots (none: zero), owners (none: all ones), the slots' totals, where the flywheel
        // audio goes (nowhere yet)
        records = fly->records;
        if (!records && (rc = grow_idle(ctx, ctx->d_records, ctx->d_records_cap, (uint64_t)(n_events ? n_events : 1) * sizeof(ohp_starvation))) != OHP_OK) return rc;
        if (!records) records = ctx->d_records;
        if ((rc = grow_idle(ctx, ctx->d_slot, ctx->d_slot_cap, (uint64_t)(n_events + 1) * sizeof(uint64_t))) != OHP_OK) return rc;
        if ((rc = grow_idle(ctx, ctx->d_owner, ctx->d_owner_cap, (uint64_t)(n_events ? n_events : 1) * sizeof(uint32_t))) != OHP_OK) return rc;
        if (!ctx->d_fly_slots) OHP_CUDA(ctx, cudaMalloc(reinterpret_cast<void**>(&ctx->d_fly_slots), sizeof(sched::FlySlots)));
        OHP_CUDA(ctx, cudaMemsetAsync(ctx->d_fly_slots, 0, sizeof(sched::FlySlots), st));
        OHP_CUDA(ctx, cudaMemsetAsync(ctx->d_slot, 0, (n_events + 1) * sizeof(uint64_t), st));
        if (n_events) {
            OHP_CUDA(ctx, cudaMemsetAsync(records, 0xff, n_events * sizeof(ohp_starvation), st));
            OHP_CUDA(ctx, cudaMemsetAsync(ctx->d_owner, 0xff, n_events * sizeof(uint32_t), st));
            OHP_CUDA(ctx, cudaMemsetAsync(fly->off, 0, n_events * sizeof(uint64_t), st));
            OHP_CUDA(ctx, cudaMemsetAsync(fly->len, 0, n_events * sizeof(uint64_t), st));
        }
        flyArgs = *fly;
        flyArgs.records = records;
        if (fly->with_recent) {
            // piece counts: 0 until a record is written
            const uint64_t n = n_events ? n_events : 1;
            if (!flyArgs.recent.recent && (rc = grow_idle(ctx, ctx->d_recent, ctx->d_recent_cap, n * sched::kRecentPieces * sizeof(ohp_recent_audio))) != OHP_OK) return rc;
            if (!flyArgs.recent.count && (rc = grow_idle(ctx, ctx->d_recent_count, ctx->d_recent_count_cap, n * sizeof(uint32_t))) != OHP_OK) return rc;
            if (!flyArgs.recent.recent) flyArgs.recent.recent = ctx->d_recent;
            if (!flyArgs.recent.count) flyArgs.recent.count = ctx->d_recent_count;
            if (n_events) OHP_CUDA(ctx, cudaMemsetAsync(flyArgs.recent.count, 0, n_events * sizeof(uint32_t), st));
        }
        fly = &flyArgs;
    }
    const sched::RecentOut* recent = fly && fly->with_recent ? &fly->recent : nullptr;
    const char* cap_env = std::getenv("OHP_REGION_CAP"); // OHP_REGION_CAP=n: regions of at most n descriptors (tests)
    const uint64_t region_cap = cap_env ? std::strtoull(cap_env, nullptr, 10) : ~0ull;
    auto bound = [&]() -> int { // regions: bound per stream (and, with fly, the flywheel slots)
        if (fly) {
            sched::bound_slots_kernel<<<(unsigned)((n_streams + 127) / 128), 128, 0, st>>>(d_streams, n_streams, d_events, n_events, ctx->d_begin,
                                                                                        ctx->d_slot, ctx->d_owner, ctx->d_fly_slots, region_cap);
        }
        else {
            sched::bound_kernel<<<(unsigned)((n_streams + 127) / 128), 128, 0, st>>>(d_streams, n_streams, d_events, n_events, ctx->d_begin,
                                                                                  region_cap);
        }
        OHP_CUDA(ctx, cudaGetLastError());
        return OHP_OK;
    };
    // with fly, the flywheel work follows whichever way the bytes were made (planned in front of ramp_convert_kernel where
    // the one walk made them, so that the host waits for the planned jobs' count while that kernel runs)
    bool planned = false;
    auto finish = [&](int aRc) -> int {
        if (aRc != OHP_OK || !fly) return aRc;
        if (!planned && (aRc = fly_plan(ctx, d_streams, n_streams, n_events, *fly, st)) != OHP_OK) return aRc;
        planned = true;
        return fly_play(ctx, d_in, in_bytes, *fly, st);
    };
    const char* one_walk_env = std::getenv("OHP_ONE_WALK"); // OHP_ONE_WALK=0: count + scan + emit as in round 1
    const bool one_walk = !one_walk_env || std::atoi(one_walk_env) != 0;
    if (!one_walk) {
        if (fly) {
            // the bounds land in d_begin, which the count overwrites
            if ((rc = bound()) != OHP_OK) return rc;
            ctx->launches++;
            OHP_CUDA(ctx, cudaMemcpyAsync(ctx->h_regions + 4, ctx->d_fly_slots, sizeof(sched::FlySlots), cudaMemcpyDeviceToHost, st));
            OHP_CUDA(ctx, cudaStreamSynchronize(st));
            if ((rc = fly_check(ctx, *fly)) != OHP_OK) return rc;
        }
        return finish(run_streams_device_two_pass(ctx, d_streams, n_streams, d_events, n_events, d_in, in_bytes, d_out, out_bytes,
                                                  d_stream_out_bytes, total_chunks, records, st, recent));
    }
    // 1. regions: bound per stream, exclusive scan
    if ((rc = bound()) != OHP_OK) return rc;
    sched::scan_kernel<<<1, sched::kScanThreads, 0, st>>>(ctx->d_begin, n_streams);
    OHP_CUDA(ctx, cudaGetLastError());
    ctx->launches += 2;
    // 2. everything on the caller's stream, and the walk is launched BEFORE the host knows how many descriptors the
    //    regions add up to -- the total (8 bytes, pinned) comes back while the walk runs, so the host's round trip costs
    //    the GPU nothing.  The walk writes nothing for a stream whose region would end beyond the buffer; if the total says
    //    the buffer was too small (first call of a shape), it grows and the walk runs again.
    OHP_CUDA(ctx, cudaMemcpyAsync(ctx->h_regions, ctx->d_begin + n_streams, sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    if (fly) OHP_CUDA(ctx, cudaMemcpyAsync(ctx->h_regions + 4, ctx->d_fly_slots, sizeof(sched::FlySlots), cudaMemcpyDeviceToHost, st));
    OHP_CUDA(ctx, cudaEventRecord(ctx->sched_event, st));
    const int team = schedule_team(n_streams);
    auto walk = [&]() -> int {
        sched::ScheduleParams p{};
        p.streams = d_streams; p.n_streams = n_streams; p.events = d_events; p.n_events = n_events;
        p.chunk_begin = ctx->d_begin; p.descs = ctx->d_descs; p.info = nullptr;
        p.descs_cap = ctx->d_descs_cap / sizeof(ohp_chunk_desc);
        p.status = ctx->d_status + 2;
        p.counts_out = ctx->d_counts; p.out_bytes = d_stream_out_bytes;
        p.lanes_per_warp = schedule_lanes(ctx, n_streams);
        p.records = records;
        const unsigned grid = team == 32 ? sched::schedule_grid(n_streams, 32) : sched::schedule_grid(n_streams, 1, p.lanes_per_warp);
        if (recent) {
            if (team == 32) sched::schedule_recent_kernel<32><<<grid, sched::kScheduleBlock, 0, st>>>(p, *recent);
            else sched::schedule_recent_kernel<1><<<grid, sched::kScheduleBlock, 0, st>>>(p, *recent);
        }
        else if (records) {
            if (team == 32) sched::schedule_record_kernel<32><<<grid, sched::kScheduleBlock, 0, st>>>(p);
            else sched::schedule_record_kernel<1><<<grid, sched::kScheduleBlock, 0, st>>>(p);
        }
        else if (team == 32) sched::schedule_kernel<true, 32><<<grid, sched::kScheduleBlock, 0, st>>>(p);
        else sched::schedule_kernel<true, 1><<<grid, sched::kScheduleBlock, 0, st>>>(p);
        OHP_CUDA(ctx, cudaGetLastError());
        ctx->launches++;
        return OHP_OK;
    };
    if (ctx->d_descs_cap >= sizeof(ohp_chunk_desc) && (rc = walk()) != OHP_OK) return rc; // (no buffer yet: after the total)
    OHP_CUDA(ctx, cudaEventSynchronize(ctx->sched_event));
    const uint64_t regions = *ctx->h_regions;
    if (fly && (rc = fly_check(ctx, *fly)) != OHP_OK) return rc;
    // (at least one descriptor: with none, regions that add up to 0 -- every stream refused, or outgrowing a region of 0 --
    //  would leave the walk unlaunched, and what it reports unreported)
    const uint64_t need = regions ? regions : 1;
    if (need > ctx->d_descs_cap / sizeof(ohp_chunk_desc)) {
        OHP_CUDA(ctx, cudaDeviceSynchronize()); // the buffer may still be read by a launch enqueued earlier on another stream
        if ((rc = grow(ctx, ctx->d_descs, ctx->d_descs_cap, need * sizeof(ohp_chunk_desc))) != OHP_OK) return rc;
        if ((rc = walk()) != OHP_OK) return rc;
    }
    if (fly) {
        if ((rc = fly_plan(ctx, d_streams, n_streams, n_events, *fly, st)) != OHP_OK) return rc;
        planned = true;
    }
    if (total_chunks) {
        // the exact number of playables, and what the walk refused: in front of ramp_convert_kernel in the stream, so the
        // host waits for the walk only
        ctx->h_outb.resize(n_streams);
        OHP_CUDA(ctx, cudaMemcpyAsync(ctx->h_outb.data(), ctx->d_counts, n_streams * sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
        OHP_CUDA(ctx, cudaMemcpyAsync(ctx->h_status, ctx->d_status, 16 * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
        OHP_CUDA(ctx, cudaEventRecord(ctx->sched_event, st));
    }
    if ((rc = launch(ctx, ctx->d_descs, (size_t)regions, d_in, in_bytes, d_out, out_bytes, st)) != OHP_OK) return rc;
    if (!total_chunks) return finish(OHP_OK);
    OHP_CUDA(ctx, cudaEventSynchronize(ctx->sched_event));
    const uint32_t bits = ctx->h_status[2];
    uint64_t total = 0;
    bool outgrown = false; // a stream of THIS call outgrew its region (the status bit may be an earlier call's)
    for (size_t s = 0; s < n_streams; s++) {
        outgrown |= ctx->h_outb[s] == sched::kOutgrown;
        total += ctx->h_outb[s];
    }
    int earlier = OHP_OK;
    if (bits != 0) {
        // waits for ramp_convert_kernel too (the call has failed anyway) and clears whatever that kernel reports beside the
        // walk's refusal: the error is this call's, no later ohp_sync reports it again
        const int src = read_status(ctx, st);
        // a stream outgrew its region and none was refused for what it is (read_status reports those first): nothing
        // wrong with the batch, take the exact two-pass path
        const uint32_t refused = (1u << sched::kErrSpec) | (1u << sched::kErrAssert);
        if (outgrown && !(bits & refused)) {
            return finish(run_streams_device_two_pass(ctx, d_streams, n_streams, d_events, n_events, d_in, in_bytes, d_out, out_bytes,
                                                      d_stream_out_bytes, total_chunks, records, st, recent));
        }
        // only an earlier call without the total outgrew a region: this call's work is whole, and reports that error
        // once it is done (as that call's ohp_sync would have)
        if (bits != (1u << sched::kErrBound)) return src;
        earlier = src;
    }
    *total_chunks = total;
    rc = finish(OHP_OK);
    return rc != OHP_OK ? rc : earlier;
}

int ohp_run_streams_device(ohp_context* ctx, const ohp_stream_spec* d_streams, size_t n_streams,
                           const ohp_ramp_event* d_events, size_t n_events,
                           const uint8_t* d_in, uint64_t in_bytes, uint8_t* d_out, uint64_t out_bytes,
                           uint64_t* d_stream_out_bytes, uint64_t* total_chunks, void* stream)
{
    return run_streams_device(ctx, d_streams, n_streams, d_events, n_events, d_in, in_bytes, d_out, out_bytes,
                              d_stream_out_bytes, total_chunks, stream, nullptr);
}

int ohp_run_streams_device_flywheel(ohp_context* ctx, const ohp_stream_spec* d_streams, size_t n_streams,
                                    const ohp_ramp_event* d_events, size_t n_events,
                                    const uint8_t* d_in, uint64_t in_bytes, uint8_t* d_out, uint64_t out_bytes,
                                    uint8_t* d_fly_out, uint64_t fly_out_bytes, ohp_starvation* d_starvations,
                                    uint64_t* d_fly_off, uint64_t* d_fly_len, uint64_t* d_stream_out_bytes,
                                    uint64_t* total_chunks, void* stream)
{
    if (!ctx) return OHP_E_INVALID_ARG;
    if (n_events && (!d_fly_off || !d_fly_len)) {
        if (total_chunks) *total_chunks = 0;
        return fail(ctx, OHP_E_INVALID_ARG, "null device pointer (d_fly_off / d_fly_len)");
    }
    const FlyArgs fly{d_fly_out, d_fly_out ? fly_out_bytes : 0, d_starvations, d_fly_off, d_fly_len};
    return run_streams_device(ctx, d_streams, n_streams, d_events, n_events, d_in, in_bytes, d_out, out_bytes,
                              d_stream_out_bytes, total_chunks, stream, &fly);
}

int ohp_run_streams_device_flywheel_recent(ohp_context* ctx, const ohp_stream_spec* d_streams, size_t n_streams,
                                           const ohp_ramp_event* d_events, size_t n_events,
                                           const uint8_t* d_in, uint64_t in_bytes, uint8_t* d_out, uint64_t out_bytes,
                                           uint8_t* d_fly_out, uint64_t fly_out_bytes, ohp_starvation* d_starvations,
                                           uint64_t* d_fly_off, uint64_t* d_fly_len, uint64_t* d_stream_out_bytes,
                                           ohp_recent_audio* d_recent, uint32_t* d_recent_count, uint64_t* total_chunks, void* stream)
{
    if (!ctx) return OHP_E_INVALID_ARG;
    if (n_events && (!d_fly_off || !d_fly_len)) {
        if (total_chunks) *total_chunks = 0;
        return fail(ctx, OHP_E_INVALID_ARG, "null device pointer (d_fly_off / d_fly_len)");
    }
    const FlyArgs fly{d_fly_out, d_fly_out ? fly_out_bytes : 0, d_starvations, d_fly_off, d_fly_len, true, {d_recent, d_recent_count}};
    return run_streams_device(ctx, d_streams, n_streams, d_events, n_events, d_in, in_bytes, d_out, out_bytes,
                              d_stream_out_bytes, total_chunks, stream, &fly);
}

int ohp_fill_streams_device(ohp_context* ctx, uint8_t* d_in, uint64_t in_bytes, const ohp_stream_spec* d_streams,
                            size_t n_streams, uint64_t seed_base, uint64_t first_stream_id, void* stream)
{
    if (!ctx) return OHP_E_INVALID_ARG;
    if (n_streams == 0) return OHP_OK;
    if (!d_in || !d_streams) return fail(ctx, OHP_E_INVALID_ARG, "null device pointer");
    (void)in_bytes; // the caller laid the streams out inside the arena (ohp_run_streams_* checks every stream's span)
    OHP_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = stream ? static_cast<cudaStream_t>(stream) : ctx->stream;
    uint64_t grid = (uint64_t)ctx->sm_count * 8u;
    if (grid > n_streams) grid = n_streams;
    fill_streams_kernel<<<(unsigned)grid, 256, 0, st>>>(d_in, d_streams, n_streams, seed_base, first_stream_id);
    OHP_CUDA(ctx, cudaGetLastError());
    ctx->launches++;
    return OHP_OK;
}

// Flywheel ramp generator (include/ohp_flywheel.h) ---------------------------------------------------------------

uint32_t ohp_flywheel_out_bytes(const ohp_flywheel_job* job)
{
    if (!job) return 0;
    return job->out_frames * job->channels * (job->bit_depth / 8u);
}

int ohp_flywheel_validate(const ohp_flywheel_job* jobs, size_t n, uint64_t in_bytes, uint64_t out_bytes, size_t* bad_index)
{
    if (!jobs && n) return OHP_E_INVALID_ARG;
    for (size_t i = 0; i < n; i++) {
        const uint32_t err = fly::check_job(jobs[i], in_bytes, out_bytes);
        if (err) {
            if (bad_index) *bad_index = i;
            return err == 1u ? OHP_E_INVALID_DESC : OHP_E_OUT_OF_RANGE;
        }
    }
    return OHP_OK;
}

int ohp_flywheel_device(ohp_context* ctx, const ohp_flywheel_job* d_jobs, size_t n, const uint8_t* d_in, uint64_t in_bytes,
                        uint8_t* d_out, uint64_t out_bytes, void* stream)
{
    if (!ctx) return OHP_E_INVALID_ARG;
    if (n == 0) return OHP_OK;
    if (!d_jobs || !d_in || !d_out) return fail(ctx, OHP_E_INVALID_ARG, "null device pointer");
    if (reinterpret_cast<uint64_t>(d_jobs) & 15u) return fail(ctx, OHP_E_INVALID_ARG, "job array must be 16-byte aligned");
    OHP_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = stream ? static_cast<cudaStream_t>(stream) : ctx->stream;
    fly::FlywheelParams p;
    p.jobs = d_jobs; p.n = n; p.in = d_in; p.in_bytes = in_bytes; p.out = d_out; p.out_bytes = out_bytes;
    p.status = ctx->d_status + 12;
    const uint64_t grid = (n + fly::kWarpsPerCta - 1) / fly::kWarpsPerCta;
    fly::flywheel_kernel<<<(unsigned)grid, fly::kWarpsPerCta * 32, 0, st>>>(p);
    OHP_CUDA(ctx, cudaGetLastError());
    ctx->launches++;
    return OHP_OK;
}

uint64_t ohp_launch_count(const ohp_context* ctx) { return ctx ? ctx->launches : 0; }

uint32_t ohp_inflight_cap(const ohp_context* ctx) { return ctx ? ctx->last_cap_chunks : 0; }

// Instrumentation builds only (-DOHP_PROFILE_WAITS): copy out and clear the 16 status words.
int ohp_debug_counters(ohp_context* ctx, uint32_t* out16)
{
    if (!ctx || !out16) return OHP_E_INVALID_ARG;
    OHP_CUDA(ctx, cudaSetDevice(ctx->device));
    OHP_CUDA(ctx, cudaDeviceSynchronize());
    OHP_CUDA(ctx, cudaMemcpy(out16, ctx->d_status, 16 * sizeof(uint32_t), cudaMemcpyDeviceToHost));
    OHP_CUDA(ctx, cudaMemset(ctx->d_status + 4, 0, 12 * sizeof(uint32_t)));
    return OHP_OK;
}

int ohp_set_timing(ohp_context* ctx, int enabled)
{
    if (!ctx) return OHP_E_INVALID_ARG;
    ctx->timing = enabled != 0;
    ctx->timed = false;
    return OHP_OK;
}

double ohp_last_kernel_ms(ohp_context* ctx)
{
    if (!ctx || !ctx->timing || !ctx->timed) return -1.0;
    if (cudaEventSynchronize(ctx->ev_stop) != cudaSuccess) return -1.0;
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, ctx->ev_start, ctx->ev_stop) != cudaSuccess) return -1.0;
    return (double)ms;
}

} // extern "C"

#include "ohp_multi.cuh"
