/*
 * ohp_schedule_device.h -- C ABI of the DEVICE-side ramp-schedule builder (exported by libohp_b200.so).
 *
 * Same job as ohp_schedule_build (include/ohp_schedule.h) -- per-stream ramp events in, one ohp_chunk_desc per
 * MsgPlayable out -- but the walk runs on the GPU, a warp (or, for very many streams, a thread) per stream, so descriptors are born in HBM next to
 * the kernel that consumes them (ohp_process_device).  It replaces, for a batch of independent streams,
 *     Ramper::ProcessAudio            (OpenHome/Media/Pipeline/Ramper.cpp:114-134)
 *     Muter::ProcessAudio             (Muter.cpp:210-262)
 *     StarvationRamper::ProcessMsgOut / ApplyRamp (StarvationRamper.cpp:791-832, 579-603)
 *     MsgAudio::Split / SetRamp / SetMuted        (Msg.cpp:1949-2046)      Ramp::Set / Split (Msg.cpp:590-807)
 *     MsgAudioPcm::CreatePlayable / MsgSilence::CreatePlayable (Msg.cpp:2234-2262, 2472-2492)
 *     MsgPlayable::Split              (Msg.cpp:2591-2624)
 * and produces bit-identical descriptors (tests/test_gpu_schedule.py: against ohp_schedule_build and against the
 * playables the reference itself produced, tests/golden).
 *
 * Two calls, because the caller owns the descriptor array and needs its size first:
 *   1. ohp_schedule_count_device  walks every stream, counts its playables and output bytes, scans the counts into
 *                                 d_chunk_begin[0..n_streams] and returns the total (synchronous: it reads the total
 *                                 and the error status back).  Where the reference would ASSERT on a stream the call
 *                                 fails with OHP_E_INVALID_DESC, for a spec the message model cannot represent with
 *                                 OHP_E_INVALID_ARG; ohp_last_error names the stream.
 *   2. ohp_schedule_emit_device   walks again and writes descriptor k of stream s to d_chunks[d_chunk_begin[s] + k]
 *                                 (asynchronous on `stream`).
 * All pointers are DEVICE pointers; d_streams / d_events / d_chunks must be 16-byte aligned.
 */
#ifndef OHP_SCHEDULE_DEVICE_H
#define OHP_SCHEDULE_DEVICE_H

#include "ohp_b200.h"
#include "ohp_schedule.h"

#ifdef __cplusplus
extern "C" {
#endif

int ohp_schedule_count_device(ohp_context* ctx, const ohp_stream_spec* d_streams, size_t n_streams,
                              const ohp_ramp_event* d_events, size_t n_events,
                              uint64_t* d_chunk_begin /* n_streams + 1 */, uint64_t* d_stream_out_bytes /* n_streams, may be NULL */,
                              uint64_t* total_chunks /* host, out */, void* stream);
int ohp_schedule_emit_device(ohp_context* ctx, const ohp_stream_spec* d_streams, size_t n_streams,
                             const ohp_ramp_event* d_events, size_t n_events, const uint64_t* d_chunk_begin,
                             ohp_chunk_desc* d_chunks, ohp_chunk_info* d_info /* may be NULL */, void* stream);

/*
 * The whole stage in one call, for a batch of streams whose PCM sits in HOST memory: stream specs and ramp events in,
 * the bytes every stream's driver would have read out.  It is MsgFactory::CreateMsgAudioPcm -> pipeline elements ->
 * CreatePlayable -> MsgPlayable::Read(IPcmProcessor&) for n_streams independent pipelines (Msg.cpp:2234-2262, 2646-2653
 * and the stage files above), with no per-message work on any host core: the descriptors are built on the GPU and stay
 * there (specs + events are all that crosses PCIe on their behalf), PCM moves in slices of whole streams, H2D / kernel /
 * D2H pipelined.  h_in / h_out should be pinned (ohp_host_alloc) for full PCIe speed.  Synchronous.
 *   h_stream_out_bytes (n_streams, may be NULL): bytes each stream produced at h_out + dst_base.
 *   total_chunks (may be NULL): playables read.
 * Only bytes some stream produces are written: gaps between streams in h_out read afterwards as the caller left them.
 * On any error nothing of the call is still in flight when it returns.
 * Errors: as ohp_schedule_count_device (the reference would ASSERT: OHP_E_INVALID_DESC; spec not representable:
 * OHP_E_INVALID_ARG), OHP_E_OUT_OF_RANGE when a stream reaches outside the arenas.
 */
int ohp_run_streams_host(ohp_context* ctx, const ohp_stream_spec* h_streams, size_t n_streams,
                         const ohp_ramp_event* h_events, size_t n_events,
                         const uint8_t* h_in, uint64_t in_bytes, uint8_t* h_out, uint64_t out_bytes,
                         uint64_t* h_stream_out_bytes, uint64_t* total_chunks);

/*
 * The same stage for a batch that is already RESIDENT IN HBM: stream specs, ramp events and PCM in device memory in,
 * every stream's output bytes in device memory out -- the schedule walk and the ramp + convert kernel, enqueued on
 * `stream` (NULL = the context's own).  The descriptors live in a buffer the context owns and reuses: one region per
 * stream, sized by a closed-form bound on its playables (ohp_schedule_chunk_bounds), filled by ONE walk per stream,
 * unused slots left empty.  The call returns once everything is enqueued; the host waits only for the regions' total
 * (8 bytes, while the walk is already running).  ohp_sync(ctx, stream) waits and reports device-side errors.
 *   d_stream_out_bytes (n_streams, device, may be NULL): bytes each stream produced at d_out + dst_base.
 *   total_chunks (host, may be NULL): playables read.  Asking for it makes the call wait for the walk (not for the
 *     ramp + convert kernel), report a stream the walk refuses here instead of at the next ohp_sync, and -- should a
 *     stream ever have more playables than its region holds (none of this repo's generators produces one; the bound is
 *     held against exact counts in the tests) -- redo the batch through count + emit.  Without it that case is an
 *     OHP_E_NO_MEMORY from the next ohp_sync.
 * Calls on one context may follow one another on any streams without an ohp_sync in between: a call that uses the
 * context's scratch (this one, its flywheel variants, ohp_process_host, ohp_run_streams_host) waits on the device for
 * the previous such call's work.  One host thread at a time per context.  The status block is the context's: when the
 * work of two calls on two streams fails at once, the first ohp_sync of either reports both.
 * Environment (tests): OHP_ONE_WALK=0 takes count + scan + emit.
 * Errors as ohp_run_streams_host.
 */
int ohp_run_streams_device(ohp_context* ctx, const ohp_stream_spec* d_streams, size_t n_streams,
                           const ohp_ramp_event* d_events, size_t n_events,
                           const uint8_t* d_in, uint64_t in_bytes, uint8_t* d_out, uint64_t out_bytes,
                           uint64_t* d_stream_out_bytes, uint64_t* total_chunks, void* stream);

/*
 * Synthetic PCM for benchmarks and tests, generated in place in HBM: stream s of the batch receives, at d_in +
 * src_base, total_frames * frame bytes of the splitmix64 sequence seeded with seed_base | (first_stream_id + s)
 * (8 bytes per step, little-endian).  A stream's bytes depend on its GLOBAL id only, so they are the same wherever the
 * stream is sharded to and the same the CPU reference arm generates (oracle/: ohpo_fill_pcm with that seed).
 * Asynchronous on `stream`.
 */
int ohp_fill_streams_device(ohp_context* ctx, uint8_t* d_in, uint64_t in_bytes, const ohp_stream_spec* d_streams,
                            size_t n_streams, uint64_t seed_base, uint64_t first_stream_id, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* OHP_SCHEDULE_DEVICE_H */
