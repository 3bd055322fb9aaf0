// ohp_schedule_kernels.cuh -- device-side ramp-schedule builder (SURVEY 8f #1): per-stream ramp events -> chunk
// descriptors, on the GPU, so that the only host-serial step in front of ramp_convert_kernel disappears.
//
// A TEAM OF THREADS WALKS ONE STREAM (host/schedule_walk.h, which also compiles for the host so the CPU suite can test
// it).  Streams are independent (SURVEY 8e); inside a stream only the ramp recurrence is sequential (every message's
// ramp starts where the previous one ended), the rest of a steady stretch is done 32 messages at a time (bulk_step).  Two passes over the same walk: COUNT (chunks and
// output bytes per stream), an exclusive scan, then EMIT (descriptors written at each stream's offset).  All integer;
// the result is bit-identical to ohp_schedule_build (host) and to the reference's playables (tests/golden).
#pragma once

#include <cstdint>
#include <cuda_runtime.h>

#include "../host/schedule_walk.h"
#include "../host/flywheel_plan.h"

namespace ohp {
namespace sched {

struct ScheduleParams
{
    const ohp_stream_spec* streams;
    uint64_t n_streams;
    const ohp_ramp_event* events;
    uint64_t n_events;
    uint64_t* chunk_count;     // COUNT: [n_streams] chunks per stream (scanned in place into chunk_begin afterwards)
    uint64_t* out_bytes;       // COUNT: [n_streams] output bytes per stream (may be null)
    const uint64_t* chunk_begin; // EMIT: [n_streams + 1]
    ohp_chunk_desc* descs;     // EMIT
    ohp_chunk_info* info;      // EMIT, may be null
    uint32_t* status;          // [0] error bits (1 << code), [1] 0xffffffff - lowest failing stream (atomicMax; 0 = none)
    // ONE-WALK mode (regions from stream_chunk_bound): EMIT also reports what COUNT would have, and fills each region's tail
    uint64_t* counts_out;      // [n_streams] exact playables per stream (null: two-pass mode)
    uint64_t descs_cap;        // descriptors the buffer holds; a stream whose region would end beyond writes nothing (0: no check)
    uint32_t lanes_per_warp;   // TEAM = 1: streams a warp walks (its first lanes, one each; the others idle); 0 = 32
    ohp_starvation* records;   // schedule_record_kernel: [n_events], the record of event e at [e]
};

constexpr uint32_t kErrBound = 4u; // a stream has more playables than stream_chunk_bound allowed for: the caller takes two passes

// Regions for the one-walk mode: bound[s] playables at most for stream s (scanned into region offsets afterwards).
__global__ void __launch_bounds__(128) bound_kernel(const ohp_stream_spec* __restrict__ streams, uint64_t n_streams,
                                                    const ohp_ramp_event* __restrict__ events, uint64_t n_events, uint64_t* __restrict__ bound)
{
    const uint64_t s = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n_streams) return;
    bound[s] = stream_chunk_bound(streams[s], events, n_events);
}


// TEAM threads walk one stream: TEAM = 32 (a warp per stream: no divergence between streams, 32 descriptors per bulk
// step written side by side) when streams are few enough for that to fill the GPU, TEAM = 1 (a thread per stream) when
// there are so many streams that they alone do.  All lanes of a team hold the same state; see schedule_walk.h.
#ifndef OHP_SCHED_MIN_BLOCKS
#define OHP_SCHED_MIN_BLOCKS 3 /* <= 168 registers.  The walk times of DESIGN 4.2 were measured with this bound; 5 (96 registers) spills. */
#endif
// RECENT: the records' pieces of recent audio too, at recent[e * kRecentPieces ...] and recent_count[e] for event e.
template <bool EMIT, int TEAM, bool RECORD, bool RECENT = false>
__device__ __forceinline__ void schedule_body(const ScheduleParams p, ohp_recent_audio* recent = nullptr, uint32_t* recent_count = nullptr)
{
    const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    uint64_t s = t / TEAM;
    const uint32_t lane = (uint32_t)(t % TEAM);
    if (TEAM == 1 && p.lanes_per_warp != 0) {
        // a thread per stream, but fewer streams than lanes in a warp: threads of a warp walk different streams and
        // take turns wherever their paths differ, so a warp takes about as long as its streams take one after the other
        if ((t & 31u) >= p.lanes_per_warp) return;
        s = (t >> 5) * p.lanes_per_warp + (t & 31u);
    }
    if (s >= p.n_streams) return;
    const ohp_stream_spec sp = p.streams[s];
    uint64_t nChunks, outBytes;
    ohp_chunk_desc* descs = EMIT ? p.descs + p.chunk_begin[s] : nullptr;
    ohp_chunk_info* info = (EMIT && p.info) ? p.info + p.chunk_begin[s] : nullptr;
    const bool regions = EMIT && p.counts_out != nullptr;
    // (regions: launched before the host has sized the buffer -- a stream whose region would end beyond it is left for the
    //  second launch that follows when that turns out to be the case)
    if (regions && p.descs_cap != 0 && p.chunk_begin[s + 1] > p.descs_cap) return;
    const uint64_t limit = regions ? p.chunk_begin[s + 1] - p.chunk_begin[s] : ~0ull;
    uint32_t rc = run_stream<EMIT, TEAM, true, RECORD, RECENT>(sp, p.events, p.n_events, descs, info, nChunks, outBytes, lane, limit,
                                                               RECORD ? p.records + sp.first_event : nullptr, s, false, nullptr,
                                                               RECENT ? recent + (uint64_t)sp.first_event * kRecentPieces : nullptr,
                                                               RECENT ? recent_count + sp.first_event : nullptr);
    if (regions) {
        if (rc == kOk && nChunks > limit) rc = kErrBound;
        // the rest of the region: zero-byte descriptors (all lanes of the team, two 128-bit stores each)
        const uint64_t from = rc == kOk ? nChunks : 0;
        uint4* d4 = reinterpret_cast<uint4*>(descs);
        for (uint64_t i = 2 * from + lane; i < 2 * limit; i += TEAM) d4[i] = make_uint4(0, 0, 0, 0);
    }
    if (lane != 0) return;
    if (rc != kOk) {
        atomicOr(&p.status[0], 1u << rc);
        atomicMax(&p.status[1], 0xffffffffu - (uint32_t)(s > 0xfffffffeull ? 0xfffffffeull : s));
    }
    if (!EMIT) {
        p.chunk_count[s] = nChunks;
        if (p.out_bytes) p.out_bytes[s] = outBytes;
    }
    else if (regions) {
        p.counts_out[s] = rc == kOk ? nChunks : 0;
        if (p.out_bytes) p.out_bytes[s] = outBytes;
    }
}

template <bool EMIT, int TEAM>
__global__ void __launch_bounds__(128, OHP_SCHED_MIN_BLOCKS) schedule_kernel(const ScheduleParams p)
{
    schedule_body<EMIT, TEAM, false>(p);
}

// The emitting walk that also leaves a starvation record per OHP_EV_STARVATION it applies (ohp_run_streams_device_flywheel).
template <int TEAM>
__global__ void __launch_bounds__(128, OHP_SCHED_MIN_BLOCKS) schedule_record_kernel(const ScheduleParams p)
{
    schedule_body<true, TEAM, true>(p);
}

// ... that also leaves each record's pieces of recent audio (ohp_run_streams_device_flywheel_recent).
struct RecentOut
{
    ohp_recent_audio* recent;  // [n_events * kRecentPieces]
    uint32_t* count;           // [n_events]
};
template <int TEAM>
__global__ void __launch_bounds__(128, OHP_SCHED_MIN_BLOCKS) schedule_recent_kernel(const ScheduleParams p, const RecentOut r)
{
    schedule_body<true, TEAM, true, true>(p, r.recent, r.count);
}

// FLYWHEEL SLOTS.  Event e's flywheel audio goes to a slot of align16(ToSamples(20 ms) x frame bytes) of its stream; the
// slots lie back to back in event order.  slot[e] (n_events + 1 entries, zeroed by the caller) is scanned in place into
// offsets afterwards; it carries the slot's bytes in its low kSlotCountShift bits and a 1 above them for every starvation
// event, so that the scan also numbers the starvation events (their descriptor regions).
constexpr int kSlotCountShift = 40;
constexpr uint64_t kSlotBytesMask = (1ull << kSlotCountShift) - 1;

struct FlySlots
{
    uint64_t bytes;     // slots' total
    uint64_t count;     // starvation events in the streams' slices
    uint64_t shared;    // events that two streams' slices both hold
    uint64_t planned;   // plan_kernel: jobs in the compacted job list
};

OHP_HD uint64_t fly_slot_bytes(const ohp_stream_spec& sp)
{
    const uint32_t jps = core::jiffies_per_sample_or_zero(sp.sample_rate);
    if (jps == 0) return 0; // the walk refuses the stream
    const uint64_t bytes = (uint64_t)(OHP_FLYWHEEL_RAMP_JIFFIES / jps) * sp.channels * (sp.bit_depth / 8u);
    return (bytes + 15u) & ~15ull;
}

// bound_kernel and the slots in one pass over the streams.  owner[e] (all ones from the caller) takes the stream that holds
// event e: a second stream holding it is counted in slots->shared.
__global__ void __launch_bounds__(128) bound_slots_kernel(const ohp_stream_spec* __restrict__ streams, uint64_t n_streams,
                                                          const ohp_ramp_event* __restrict__ events, uint64_t n_events,
                                                          uint64_t* __restrict__ bound, uint64_t* __restrict__ slot,
                                                          uint32_t* __restrict__ owner, FlySlots* __restrict__ slots)
{
    const uint64_t s = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n_streams) return;
    const ohp_stream_spec sp = streams[s];
    bound[s] = stream_chunk_bound(sp, events, n_events);
    const uint64_t first = sp.first_event;
    const uint64_t end = first + sp.num_events < n_events ? first + sp.num_events : n_events;
    const uint64_t size = fly_slot_bytes(sp);
    uint64_t bytes = 0, count = 0, shared = 0;
    for (uint64_t e = first; e < end; e++) {
        if (atomicCAS(&owner[e], 0xffffffffu, (uint32_t)s) != 0xffffffffu) shared++;
        if (events[e].op != OHP_EV_STARVATION) continue;
        slot[e] = (1ull << kSlotCountShift) | size;
        bytes += size;
        count++;
    }
    if (bytes | count) {
        atomicAdd(reinterpret_cast<unsigned long long*>(&slots->bytes), (unsigned long long)bytes);
        atomicAdd(reinterpret_cast<unsigned long long*>(&slots->count), (unsigned long long)count);
    }
    if (shared) atomicAdd(reinterpret_cast<unsigned long long*>(&slots->shared), (unsigned long long)shared);
}

// One thread per event: where its flywheel audio goes (fly_off, fly_len) and, for the k-th starvation event, the
// descriptors of two of the three launches in fixed regions -- prep[k * OHP_FLYWHEEL_MAX_PREP ...], blocks[k *
// flyplan::kMaxBlocks ...] -- planned from its record (flyplan::plan); whatever a region does not use is zero (empty
// descriptors).  Jobs go to a compacted list (slots->planned of them, in no particular order: each writes its own slot),
// so that a starvation that is not played runs no flywheel job.  The training block and the generated audio take the same
// offsets in the two scratch arenas as the output in the caller's (a training block is at most a fifth of its slot).
struct PlanParams
{
    const ohp_stream_spec* streams;
    uint64_t n_streams;
    uint64_t n_events;
    const ohp_starvation* records;
    const uint64_t* slot;      // scanned: [n_events + 1]
    ohp_chunk_desc* prep;
    ohp_flywheel_job* jobs;
    ohp_chunk_desc* blocks;
    uint64_t* fly_off;
    uint64_t* fly_len;
    FlySlots* slots;
};

// RECENT: planned from the record's pieces of recent audio (flyplan::plan_recent), OHP_FLYWHEEL_MAX_PREP_RECENT prep
// descriptors per starvation event; a record whose pieces the walk could not keep all of (OHP_RECENT_INCOMPLETE) is not.
template <bool RECENT>
__device__ __forceinline__ void plan_body(const PlanParams p, const ohp_recent_audio* recent = nullptr, const uint32_t* recent_count = nullptr)
{
    constexpr uint32_t kPrep = RECENT ? OHP_FLYWHEEL_MAX_PREP_RECENT : OHP_FLYWHEEL_MAX_PREP;
    const uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= p.n_events) return;
    const uint64_t here = p.slot[e], next = p.slot[e + 1];
    const uint64_t off = here & kSlotBytesMask;
    p.fly_off[e] = off;
    p.fly_len[e] = 0;
    if ((next >> kSlotCountShift) == (here >> kSlotCountShift)) return; // not a starvation event of a stream
    const uint64_t k = here >> kSlotCountShift;
    ohp_chunk_desc* prep = p.prep + k * kPrep;
    ohp_chunk_desc* blocks = p.blocks + k * flyplan::kMaxBlocks;
    ohp_flywheel_job job;
    uint32_t nPrep = 0, nBlocks = 0;
    const ohp_starvation rec = p.records[e];
    if (rec.event == e && rec.stream < p.n_streams) {
        const ohp_stream_spec sp = p.streams[rec.stream];
        int status;
        if constexpr (RECENT) {
            const uint32_t n = recent_count[e];
            status = n <= kRecentPieces ? flyplan::plan_recent(sp, rec, recent + e * kRecentPieces, n, off, off, off, prep, nPrep, job, blocks, nBlocks)
                                        : OHP_E_INVALID_ARG;
        }
        else {
            status = flyplan::plan(sp, rec, off, off, off, prep, nPrep, job, blocks, nBlocks);
        }
        if (status == OHP_OK) {
            p.fly_len[e] = (uint64_t)job.out_frames * sp.channels * (sp.bit_depth / 8u);
            p.jobs[atomicAdd(reinterpret_cast<unsigned long long*>(&p.slots->planned), 1ull)] = job;
        }
        else {
            nPrep = nBlocks = 0;
        }
    }
    for (uint32_t i = nPrep; i < kPrep; i++) prep[i] = flyplan::zero_desc();
    for (uint32_t i = nBlocks; i < flyplan::kMaxBlocks; i++) blocks[i] = flyplan::zero_desc();
}

__global__ void __launch_bounds__(128) plan_kernel(const PlanParams p)
{
    plan_body<false>(p);
}

__global__ void __launch_bounds__(128) plan_recent_kernel(const PlanParams p, const ohp_recent_audio* __restrict__ recent,
                                                          const uint32_t* __restrict__ recent_count)
{
    plan_body<true>(p, recent, recent_count);
}

// threads per block; grid for n streams
constexpr unsigned kScheduleBlock = 128;
inline unsigned schedule_grid(uint64_t n_streams, int team, uint32_t lanes_per_warp = 0)
{
    if (team == 1 && lanes_per_warp != 0) {
        const uint64_t warps = (n_streams + lanes_per_warp - 1) / lanes_per_warp;
        return (unsigned)((warps * 32u + kScheduleBlock - 1) / kScheduleBlock);
    }
    return (unsigned)((n_streams * (uint64_t)team + kScheduleBlock - 1) / kScheduleBlock);
}

// In-place exclusive scan of counts[0..n) into begin[0..n] (begin has n+1 entries; begin[n] = total).  One CTA.
// 256 threads: the walk times of DESIGN 4.2 were measured with this scan.
constexpr unsigned kScanThreads = 256;
__global__ void __launch_bounds__(kScanThreads) scan_kernel(uint64_t* begin, uint64_t n)
{
    __shared__ uint64_t warp_sum[kScanThreads / 32];
    __shared__ uint64_t carry;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (uint64_t first = 0; first < n; first += kScanThreads) {
        const uint64_t i = first + threadIdx.x;
        const uint64_t v = i < n ? begin[i] : 0;
        uint64_t x = v;
        for (int o = 1; o < 32; o <<= 1) {
            const uint64_t y = __shfl_up_sync(0xffffffffu, x, o);
            if (lane >= (uint32_t)o) x += y;
        }
        if (lane == 31) warp_sum[warp] = x;
        __syncthreads();
        if (warp == 0) {
            uint64_t w = lane < kScanThreads / 32 ? warp_sum[lane] : 0;
            for (int o = 1; o < (int)(kScanThreads / 32); o <<= 1) {
                const uint64_t y = __shfl_up_sync(0xffffffffu, w, o);
                if (lane >= (uint32_t)o) w += y;
            }
            if (lane < kScanThreads / 32) warp_sum[lane] = w;
        }
        __syncthreads();
        const uint64_t before = carry + (warp ? warp_sum[warp - 1] : 0) + (x - v);
        if (i < n) begin[i] = before;
        __syncthreads();
        if (threadIdx.x == kScanThreads - 1) carry = before + v;
        __syncthreads();
    }
    if (threadIdx.x == 0) begin[n] = carry;
}

} // namespace sched
} // namespace ohp
