/*
 * ohp_starvation_recent.h -- ohp_run_streams_device_flywheel (ohp_starvation_device.h) with StarvationRamper's recent audio
 * kept piece by piece on the device (exported by libohp_b200.so).
 *
 * ohp_run_streams_device_flywheel plans a starvation only where the element's last millisecond is PCM of one attenuation.
 * This call plays every starvation as ohp_flywheel_plan_batch_recent plans it from ohp_schedule_build's records and pieces:
 * silence in the last millisecond, a change of attenuation there, and PCM runs split by either all play as the element
 * plays them.  The schedule walk keeps, per StarvationRamper stage, the element's recent audio (ProcessAudioOut,
 * StarvationRamper.cpp:548-577) in a ring of OHP_DEVICE_RECENT_PIECES pieces and writes it beside every record; a planner
 * on the device restates ohp_flywheel_plan_recent on those pieces.
 *
 * Arguments: every argument of ohp_run_streams_device_flywheel, with the same meaning and the same slot layout, in the same
 * order up to d_stream_out_bytes; then
 *   d_recent       ([n_events * OHP_DEVICE_RECENT_PIECES] or NULL): event e's pieces at d_recent[e * OHP_DEVICE_RECENT_PIECES],
 *                  oldest first, as ohp_schedule_build keeps them (ohp_schedule_recent_audio) -- except that the oldest PCM
 *                  piece may begin earlier or later than the class model's: only the last OHP_FLYWHEEL_TRAINING_JIFFIES,
 *                  which is all StartFlywheelRamp reads, are the same;
 *   d_recent_count ([n_events] or NULL): the number of pieces there; 0 where e left no record; OHP_RECENT_INCOMPLETE where
 *                  the record needs more than OHP_DEVICE_RECENT_PIECES pieces (see below).
 * NULL: the context keeps them in scratch memory of its own (as it does the records when d_starvations is NULL).
 *
 * Results: the streams' bytes, sizes, chunk count, records and errors are those of ohp_run_streams_device_flywheel.
 * d_fly_len[e] != 0 exactly for the events of the records ohp_flywheel_plan_batch_recent plans, and each played slot holds
 * what that plan's three launches write.  Not played, as on the host: a starvation that plays nothing, less than 1 ms since
 * the element's recent audio was emptied, too few frames for FlywheelInput's planes, more than OHP_FLYWHEEL_MAX_PREP_RECENT
 * prep descriptors, shapes the flywheel does not take, and the cut that never ends (ohp_flywheel_plan_recent).
 *
 * ONE DEVIATION.  The ring holds OHP_DEVICE_RECENT_PIECES pieces.  A record for which the class model keeps more (its
 * pieces behind the oldest sum to less than 1 ms: a run of very short MsgSilences) cannot be represented: its count is
 * OHP_RECENT_INCOMPLETE and the starvation is not played.  No generator of this repository comes near (at most 3 pieces).
 */
#ifndef OHP_STARVATION_RECENT_H
#define OHP_STARVATION_RECENT_H

#include "ohp_starvation_device.h"

#define OHP_DEVICE_RECENT_PIECES 16u        /* pieces of recent audio the device walk keeps per StarvationRamper stage */
#define OHP_RECENT_INCOMPLETE    0xffffffffu

#ifdef __cplusplus
extern "C" {
#endif

int ohp_run_streams_device_flywheel_recent(ohp_context* ctx, const ohp_stream_spec* d_streams, size_t n_streams,
                                           const ohp_ramp_event* d_events, size_t n_events,
                                           const uint8_t* d_in, uint64_t in_bytes, uint8_t* d_out, uint64_t out_bytes,
                                           uint8_t* d_fly_out, uint64_t fly_out_bytes,
                                           ohp_starvation* d_starvations /* [n_events] or NULL */,
                                           uint64_t* d_fly_off, uint64_t* d_fly_len /* [n_events] each */,
                                           uint64_t* d_stream_out_bytes,
                                           ohp_recent_audio* d_recent /* [n_events * OHP_DEVICE_RECENT_PIECES] or NULL */,
                                           uint32_t* d_recent_count /* [n_events] or NULL */,
                                           uint64_t* total_chunks, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* OHP_STARVATION_RECENT_H */
