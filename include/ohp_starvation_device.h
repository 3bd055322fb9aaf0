/*
 * ohp_starvation_device.h -- C ABI of the whole stage for a batch RESIDENT IN HBM, StarvationRamper's flywheel ramps included
 * (exported by libohp_b200.so).
 *
 * ohp_run_streams_device (ohp_schedule_device.h) produces every stream's bytes; a starving StarvationRamper also plays
 * 20 ms of generated audio -- the flywheel ramp (ohp_flywheel.h) -- that is not part of the stream's output.  This call
 * produces both, with nothing per message or per starvation on the host:
 *   1. the schedule walk, which also records every OHP_EV_STARVATION it applies (what ohp_schedule_build records:
 *      ohp_starvation, ohp_schedule.h);
 *   2. the ramp + convert kernel: the streams' bytes, exactly as ohp_run_streams_device writes them;
 *   3. a plan per record (ohp_flywheel_plan, on the device), then FlywheelInput::Prepare, FlywheelRamperManager::Ramp and
 *      RampGenerator's ramped 1 ms blocks (INTEGRATION.md 1b) as three launches.
 * Everything is enqueued on `stream` (NULL = the context's own); the host waits only for what ohp_run_streams_device waits
 * for, which now also carries the flywheel slots' total.  A batch without starvation events launches what
 * ohp_run_streams_device launches.  Calls may follow one another on any streams without an ohp_sync in between, one host
 * thread at a time per context (ohp_schedule_device.h).
 *
 * FLYWHEEL OUTPUT.  Event e of the events array gets a slot of d_fly_out at d_fly_off[e] = the sum, over the
 * OHP_EV_STARVATION events before it in the array, of align16(Jiffies::ToSamples(20 ms, rate) x frame bytes) of the stream
 * whose slice holds the event; every other event's slot is empty.  d_fly_len[e] = the bytes the starving element plays
 * there (Jiffies::ToSamples(20 ms, rate) x frame bytes) where the starvation was planned and plays, 0 otherwise -- it
 * plays nothing (halted, muted, not yet audible), the last millisecond was not PCM of one attenuation, or the shape does
 * not fit the reference's flywheel buffers (ohp_flywheel_plan's refusals).  Only the bytes of played slots are written.
 *   d_starvations ([n_events], may be NULL): the record of event e at [e]; where e left none, every byte of [e] is 0xff
 *     (event = 0xffffffff).  Records carry no recent audio: ohp_run_streams_device_flywheel_recent (ohp_starvation_recent.h)
 *     also keeps it and plays the starvations with silence or a change of attenuation in their last millisecond.
 *   d_fly_off, d_fly_len ([n_events] each): required when n_events > 0.
 * Errors: as ohp_run_streams_device; OHP_E_OUT_OF_RANGE when fly_out_bytes is below the slots' total (ohp_last_error names
 * the bytes needed; nothing is written to d_fly_out); OHP_E_INVALID_ARG when two streams' event slices share an event.
 */
#ifndef OHP_STARVATION_DEVICE_H
#define OHP_STARVATION_DEVICE_H

#include "ohp_b200.h"
#include "ohp_schedule.h"

#ifdef __cplusplus
extern "C" {
#endif

int ohp_run_streams_device_flywheel(ohp_context* ctx, const ohp_stream_spec* d_streams, size_t n_streams,
                                    const ohp_ramp_event* d_events, size_t n_events,
                                    const uint8_t* d_in, uint64_t in_bytes, uint8_t* d_out, uint64_t out_bytes,
                                    uint8_t* d_fly_out, uint64_t fly_out_bytes,
                                    ohp_starvation* d_starvations /* [n_events] or NULL; event = 0xffffffff where event e left no record */,
                                    uint64_t* d_fly_off, uint64_t* d_fly_len /* [n_events] each */,
                                    uint64_t* d_stream_out_bytes, uint64_t* total_chunks, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* OHP_STARVATION_DEVICE_H */
