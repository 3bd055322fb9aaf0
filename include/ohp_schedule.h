/*
 * ohp_schedule.h -- C ABI of the host-side ramp-schedule runner: turns per-stream ramp events
 * into the chunk descriptors (ohp_chunk_desc) the GPU hot path consumes.
 *
 * It replaces, for a batch of independent streams, the control-plane idiom every ramp-setting
 * pipeline element uses
 *     if (msg->Jiffies() > remaining) split = msg->Split(remaining);
 *     current = msg->SetRamp(current, remaining, direction, split);
 * (Ramper.cpp:114-134, Muter.cpp:210-262, StarvationRamper.cpp:579-603,791-832) followed by
 * MsgAudioPcm::CreatePlayable (Msg.cpp:2234-2262), MsgSilence::CreatePlayable (Msg.cpp:2472-2492)
 * and, when a driver block size is given, MsgPlayable::Split (Msg.cpp:2591-2624).
 *
 * The message model underneath (Ramp::Set/Split, MsgAudio::SetRamp/Split, Jiffies rounding) is
 * the C++ mirror in ohpipeline_b200/host/; this header is its plain-C surface.
 */
#ifndef OHP_SCHEDULE_H
#define OHP_SCHEDULE_H

#include <stddef.h>
#include <stdint.h>
#include "ohp_b200.h"
#include "ohp_flywheel.h"

#ifdef __cplusplus
extern "C" {
#endif

/* Jiffies::kPerSecond (Msg.h:193) */
#define OHP_JIFFIES_PER_SECOND 56448000u
#define OHP_JIFFIES_PER_MS     56448u
#define OHP_MAX_STAGES 4u

/* Ramp::EDirection (Msg.h:259-265) */
#define OHP_DIR_NONE 0u
#define OHP_DIR_UP   1u
#define OHP_DIR_DOWN 2u
#define OHP_DIR_MUTE 3u

typedef enum ohp_event_op {
    OHP_EV_RAMP_DOWN = 1,       /* arg = duration in jiffies; stage ramps down from its current value,
                                   then mutes (Muter.cpp:210-262 / StarvationRamper.cpp:579-603)      */
    OHP_EV_RAMP_UP = 2,         /* arg = duration in jiffies; ramps up from the current value, then runs */
    OHP_EV_MUTE = 3,            /* stage calls SetMuted on every following message (Muter eMuted)     */
    OHP_EV_UNMUTE = 4,          /* stage returns to running at Ramp::kMax                            */
    OHP_EV_SET_ATTENUATION = 5, /* arg = MsgAudioPcm::SetAttenuation value for following PCM msgs (Attenuator.cpp:55-58) */
    OHP_EV_INSERT_SILENCE = 6,  /* arg = jiffies; a MsgSilence enters the chain ahead of the next PCM msg */
    OHP_EV_MAX_MSG_JIFFIES = 7, /* arg = jiffies; stage splits larger msgs first (StarvationRamper kMaxAudioOutJiffies,
                                   StarvationRamper.cpp:802-805); 0 disables                          */
    /* The calls and messages the reference's own elements react to.  A stage driven by these IS that element: its state
     * machine, including what a MsgSilence or a MsgHalt passing through does to a ramp in progress (ops 1-4 above are the
     * bare "ramp from the current value over arg jiffies" idiom every element shares, and ramp MsgSilence like audio).
     * tests/test_elements_vs_reference.py runs them beside the Ramper, Muter and StarvationRamper objects themselves.     */
    OHP_EV_RAMPER_STREAM = 8,   /* a MsgDecodedStream reaches a Ramper (Ramper.cpp:72-93): arg != 0 -- IsRampApplicable --
                                   starts its ramp up from Ramp::kMin over arg jiffies, arg = 0 leaves it at Ramp::kMax.
                                   A MsgSilence (Ramper.cpp:106-112) or MsgHalt (:65-70) ends the ramp there and then    */
    OHP_EV_MUTER_MUTE = 9,      /* Muter::Mute() with iRampDuration = arg (Muter.cpp:57-99): at once while halted, else a
                                   ramp down from Ramp::kMax; called during a ramp up it turns the ramp round where it is
                                   (remaining = arg - remaining).  Where the reference ASSERTS (already muting) so does this */
    OHP_EV_MUTER_UNMUTE = 10,   /* Muter::Unmute() (Muter.cpp:101-137), the mirror image; from muted: ramp up from Ramp::kMin,
                                   or straight to running while halted                                                    */
    OHP_EV_HALT = 11,           /* a MsgHalt passes the stage and the animator acknowledges it at once: a Ramper stops
                                   ramping; a Muter ramping down goes straight to muted and is halted until the next audio
                                   (Muter.cpp:159-167, 264-290)                                                           */
    OHP_EV_STARVATION = 12      /* the StarvationRamper's reservoir runs dry (StarvationRamper.cpp:622-673): if it is running,
                                   or ramping up and audible, the flywheel ramp plays (generated audio: ohp_flywheel.h; not part
                                   of this stream's output), a MsgHalt follows, and the audio after it ramps up from Ramp::kMin
                                   over arg jiffies (iRampUpJiffies).  The stage also holds messages to kMaxAudioOutJiffies = 5 ms */
} ohp_event_op;

typedef struct ohp_ramp_event {
    uint64_t at_jiffies; /* stream position (jiffies of audio that passed the stage) at which it fires;
                            a message straddling it is Split() there first                           */
    uint32_t stage;      /* 0..OHP_MAX_STAGES-1; stages run in index order like pipeline elements    */
    uint32_t op;         /* ohp_event_op                                                             */
    uint32_t arg;
    uint32_t reserved;
} ohp_ramp_event;

typedef struct ohp_stream_spec {
    uint32_t sample_rate;       /* one of the 18 PCM rates Jiffies::PerSample accepts (Msg.cpp:424-470) */
    uint32_t bit_depth;         /* 8/16/24/32                                                          */
    uint32_t channels;
    uint32_t in_little_endian;  /* wire format of the stream's PCM (AudioDataEndian)                   */
    uint32_t chunk_frames;      /* frames per MsgAudioPcm fed into the chain; chunk bytes <= 9216      */
    uint32_t out_fmt;           /* OHP_OUT_PACKED_BE or OHP_OUT_PACKED_LE                              */
    uint64_t total_frames;
    uint64_t src_base;          /* byte offset of the stream's PCM in the input arena                  */
    uint64_t dst_base;          /* byte offset of the stream's output in the output arena              */
    uint32_t first_event;       /* slice [first_event, first_event+num_events) of the events array,   */
    uint32_t num_events;        /*   sorted by at_jiffies                                              */
    uint32_t driver_block_frames; /* 0: one playable per message; else the driver pulls blocks of this
                                   many frames and MsgPlayable::Split()s playables to fit              */
    uint32_t codec_read_frames; /* 0: messages of chunk_frames (CodecWav, or no codec).  Else the codec reads this many
                                   frames at a time (CodecAiffBase: 9216 B rounded down to frames), CodecController cuts
                                   each read into chunk_frames pieces and DecodedAudioAggregator packs short pieces
                                   together again (ohpipeline_b200/host/codec_source.h)                 */
} ohp_stream_spec;

/* Per-chunk facts that are not needed on the device but pin descriptor parity. */
typedef struct ohp_chunk_info {
    uint32_t direction; /* Ramp::Direction() of the playable's ramp  */
    uint32_t jiffies;   /* MsgPlayable::Jiffies()                    */
} ohp_chunk_info;

typedef struct ohp_schedule ohp_schedule;

/* Run every stream's events through the stage chain (threaded over streams; threads<=0 = all cores). */
int    ohp_schedule_build(const ohp_stream_spec* streams, size_t n_streams,
                          const ohp_ramp_event* events, size_t n_events,
                          int threads, ohp_schedule** out);
/* Same result from the class-free walk the GPU schedule kernels compile (ohpipeline_b200/host/schedule_walk.h;
 * device entry points in ohp_schedule_device.h): no message objects, two passes (count, emit).  It records the same
 * starvations as ohp_schedule_build (ohp_schedule_starvations), without the recent audio's pieces. */
int    ohp_schedule_build_walk(const ohp_stream_spec* streams, size_t n_streams,
                               const ohp_ramp_event* events, size_t n_events,
                               int threads, ohp_schedule** out);
/* The closed-form upper bound on each stream's playables that ohp_run_streams_device sizes its descriptor regions with
 * (one walk per stream instead of count + emit); bounds[s] = 0 for a stream the walk refuses.  Exported so that the CPU
 * suite can hold it against the exact counts. */
int    ohp_schedule_chunk_bounds(const ohp_stream_spec* streams, size_t n_streams,
                                 const ohp_ramp_event* events, size_t n_events, uint64_t* bounds);
size_t ohp_schedule_num_chunks(const ohp_schedule* s);
const ohp_chunk_desc* ohp_schedule_chunks(const ohp_schedule* s);
const ohp_chunk_info* ohp_schedule_chunk_info(const ohp_schedule* s);
/* n_streams+1 prefix offsets into the chunk array */
const uint64_t* ohp_schedule_stream_chunk_begin(const ohp_schedule* s);
/* output bytes each stream produces (its chunks' dst ranges tile [dst_base, dst_base+out_bytes)) */
const uint64_t* ohp_schedule_stream_out_bytes(const ohp_schedule* s);
const char* ohp_schedule_last_error(void);
void   ohp_schedule_free(ohp_schedule* s);

/*
 * What a stream's StarvationRamper stage was doing when its reservoir ran dry (OHP_EV_STARVATION): everything the flywheel
 * ramp it then plays is made from.  ohp_schedule_build records one per starvation event it applies, streams in order, and
 * so does the class-free walk (ohp_schedule_build_walk; on the device: ohp_run_streams_device_flywheel,
 * ohp_starvation_device.h), which keeps no recent audio: its ohp_schedule_recent_begin is all zeros.
 * tests/test_elements_vs_reference.py holds the audio planned from these records against what the real StarvationRamper
 * object plays when it is starved at the same position.
 *
 * The element keeps a clone of every MsgAudioPcm and MsgSilence it hands on (ProcessAudioOut, StarvationRamper.cpp:548-577);
 * only a flywheel ramp and a new stream empty that store -- a MsgHalt does not.  StartFlywheelRamp (:491-536) cuts it to the
 * last kTrainingJiffies (1 ms) and reads it through FlywheelInput with the messages' ramps cleared, attenuation kept.
 * (Attenuation is applied ONCE here, as everywhere in this library.  The reference attenuates a cell in place whenever a
 * playable of it is read, Msg.cpp:2736-2756, and the element's clones share their cells with the messages it handed on:
 * had the driver already read a cell when the element starves, the flywheel would see it attenuated twice -- a matter of
 * thread timing there, not reproduced; the comparison with the real element is made before anything downstream reads.)
 */
typedef struct ohp_starvation {
    uint64_t stream;         /* index into the batch                                                                   */
    uint64_t pcm_jiffies;    /* PCM of the stream that had passed the element, in jiffies: not always a whole number of
                                samples (stages before it split messages wherever their events fall)                    */
    uint32_t event;          /* index of the event in the batch's events array                                          */
    uint32_t ramp;           /* iCurrentRampValue, what RampGenerator starts from: what the element's own SetRamp calls last
                                returned (Ramp::kMax before its first ramp; after a completed ramp up Ramp::kMax too, unless
                                the messages carried a lower ramp from a stage before it: then where that one stood)     */
    uint32_t plays;          /* 1: StartFlywheelRamp (running, or ramping up and audible, :640-650); 0: nothing to ramp
                                down from (halted, muted, starting): no flywheel audio                                  */
    uint32_t recent_jiffies; /* how much of the element's recent audio, counted back from its end, is PCM of one
                                attenuation and nothing else (no MsgSilence between), saturated at 2^32 - 1.  Below
                                OHP_FLYWHEEL_TRAINING_JIFFIES the training block holds silence (a MsgSilence that passed,
                                or the padding of :509-518) or a change of attenuation: ohp_flywheel_plan refuses it.
                                (With a MsgSilence there the reference itself may never return: its cut, :495-507, splits
                                the silence at a jiffy count that need not be a whole sample, MsgSilence::SplitCompleted
                                rounds the front part down, Msg.cpp:2530-2535, and the loop goes on splitting off messages
                                of zero jiffies -- at 44.1 kHz x 2^n whenever the silence lies under the cut.)             */
    uint32_t attenuation;    /* MsgAudioPcm attenuation of that PCM (OHP_UNITY_ATTENUATION: none)                        */
    uint32_t reserved;
} ohp_starvation;
size_t ohp_schedule_num_starvations(const ohp_schedule* s);
const ohp_starvation* ohp_schedule_starvations(const ohp_schedule* s);

/*
 * The three launches of one starvation (INTEGRATION.md 1b), as data:
 *   FlywheelInput::Prepare over the last kTrainingJiffies of PCM -> prep[0..*n_prep): descriptors with sink
 *     OHP_OUT_PLANAR32_BE, reading the stream's own bytes in the input arena, writing the training block at training_off;
 *   FlywheelRamperManager::Ramp -> *job (training block at training_off, generated audio at generated_off of the next
 *     launch's arenas);
 *   RampGenerator::Start / EndBlock -> blocks[0..*n_blocks): one ramped descriptor per 1 ms, reading at generated_off,
 *     writing what the driver reads at out_off.
 * prep must have room for OHP_FLYWHEEL_MAX_PREP descriptors.  It is one descriptor where the training block is a whole
 * number of frames T = Jiffies::ToSamples(1 ms).  At the 44.1 kHz family of rates 1 ms is T frames and k jiffies more
 * (k = 128 from 11.025 kHz up), so the reference's cut leaves T + 1 frames whenever pcm_jiffies falls less than k jiffies
 * after a sample boundary (always, when the messages are whole samples: MsgAudioPcm::CreatePlayable rounds both ends of
 * a message down to a sample, Msg.cpp:2234-2262); FlywheelInput sized its planes for T, so every channel's last subsample lands on the
 * first slot of the next channel's plane and the last channel's beyond the block (StarvationRamper.cpp:90-111, 158-186).
 * The plan reproduces exactly that block: frames 1 .. T-1 as one descriptor, the first slot of each plane as one
 * one-subsample descriptor each (mono: frames 0 .. T-1 in one descriptor).  No two descriptors write the same byte.
 * Returns OHP_OK; OHP_E_INVALID_ARG for a starvation that plays nothing (plays == 0) or whose training block is not PCM of
 * one attenuation throughout (see recent_jiffies), OHP_E_INVALID_DESC where the reference would ASSERT (rates / channel
 * counts FlywheelRamper cannot take: ohp_flywheel_validate), OHP_E_NO_MEMORY when cap is too small.
 */
#define OHP_FLYWHEEL_MAX_PREP 9u /* 1 + OHP_FLYWHEEL_MAX_CHANNELS */
int    ohp_flywheel_plan(const ohp_stream_spec* stream, const ohp_starvation* starvation,
                         uint64_t training_off, uint64_t generated_off, uint64_t out_off,
                         ohp_chunk_desc* prep, size_t* n_prep, ohp_flywheel_job* job,
                         ohp_chunk_desc* blocks, size_t cap, size_t* n_blocks);

/*
 * The same with silence in the last millisecond.  ohp_schedule_build also keeps, per starvation record, the element's recent
 * audio piece by piece -- every MsgSilence as it passed, PCM in runs of one attenuation -- oldest first, as far back as the
 * last millisecond needs: record k's pieces are [ohp_schedule_recent_begin(s)[k], ...[k + 1]) of ohp_schedule_recent_audio(s).
 * ohp_flywheel_plan_recent restates StartFlywheelRamp's cut and FlywheelInput::Prepare on those pieces: silence becomes
 * silent planar descriptors, every run of PCM its own descriptor with its own attenuation, a frame too many is laid out as
 * FlywheelInput lays it out.  Refused (OHP_E_INVALID_ARG): a starvation that plays nothing; less than 1 ms in all since
 * the recent audio was last emptied (the reference pads with silence and hands FlywheelRamper a block of another length);
 * pieces that give FlywheelInput fewer frames than its planes have (the rest of the plane is whatever the previous
 * starvation left there); more descriptors than prep_cap.  OHP_E_INVALID_DESC: shapes the flywheel does not take, and THE
 * CUT THAT NEVER ENDS -- a MsgSilence under the cut at a jiffy count that is not a whole sample: the reference does not
 * return from that one (recent_jiffies above).
 */
typedef struct ohp_recent_audio {
    uint64_t pcm_jiffies;   /* PCM: where in the stream's PCM the piece begins (jiffies); silence: 0        */
    uint32_t jiffies;
    uint32_t silence;       /* 1: a MsgSilence                                                              */
    uint32_t attenuation;   /* PCM: MsgAudioPcm attenuation of the piece                                    */
    uint32_t reserved;
} ohp_recent_audio;
const ohp_recent_audio* ohp_schedule_recent_audio(const ohp_schedule* s);
const uint64_t* ohp_schedule_recent_begin(const ohp_schedule* s); /* ohp_schedule_num_starvations(s) + 1 entries */
/* prep descriptors ohp_flywheel_plan_batch_recent (and the device's planner) allow one starvation: more are not planned */
#define OHP_FLYWHEEL_MAX_PREP_RECENT 64u
int    ohp_flywheel_plan_recent(const ohp_stream_spec* stream, const ohp_starvation* starvation,
                                const ohp_recent_audio* recent, size_t n_recent,
                                uint64_t training_off, uint64_t generated_off, uint64_t out_off,
                                ohp_chunk_desc* prep, size_t prep_cap, size_t* n_prep, ohp_flywheel_job* job,
                                ohp_chunk_desc* blocks, size_t cap, size_t* n_blocks);

/*
 * ohp_flywheel_plan for every starvation of a batch at once: the arrays the three launches take.  Starvations that play
 * nothing, whose training block is not PCM throughout, or whose shape FlywheelRamper does not take are left out (which of
 * them were planned: ohp_flywheel_batch_planned).  The k-th planned starvation's training block, generated audio and
 * output lie back to back with the others', each 16-byte aligned, from training_base / generated_base / out_base of the
 * respective arenas; ohp_flywheel_batch_out_off()[k] .. [k] + ohp_flywheel_batch_out_len()[k] is where the driver
 * reads what that starving element plays.  On the device (INTEGRATION.md 1b):
 *     ohp_process_device(ctx, prep,   n_prep,   d_pcm,       pcm_bytes,       d_training,  training_bytes,  s);
 *     ohp_flywheel_device(ctx, jobs,  n_jobs,   d_training,  training_bytes,  d_generated, generated_bytes, s);
 *     ohp_process_device(ctx, blocks, n_blocks, d_generated, generated_bytes, d_out,       out_bytes,       s);
 * OHP_E_INVALID_ARG for a record whose stream index is outside the batch.
 */
typedef struct ohp_flywheel_batch ohp_flywheel_batch;
int    ohp_flywheel_plan_batch(const ohp_stream_spec* streams, size_t n_streams,
                               const ohp_starvation* starvations, size_t n_starvations,
                               uint64_t training_base, uint64_t generated_base, uint64_t out_base, ohp_flywheel_batch** out);
/* ... planned from the recent audio (ohp_flywheel_plan_recent): recent / recent_begin as ohp_schedule_build left them */
int    ohp_flywheel_plan_batch_recent(const ohp_stream_spec* streams, size_t n_streams,
                                      const ohp_starvation* starvations, size_t n_starvations,
                                      const ohp_recent_audio* recent, const uint64_t* recent_begin,
                                      uint64_t training_base, uint64_t generated_base, uint64_t out_base, ohp_flywheel_batch** out);
size_t ohp_flywheel_batch_num_planned(const ohp_flywheel_batch* b);
const uint32_t* ohp_flywheel_batch_planned(const ohp_flywheel_batch* b);   /* indices into `starvations`, ascending      */
const uint64_t* ohp_flywheel_batch_out_off(const ohp_flywheel_batch* b);   /* per planned starvation                     */
const uint64_t* ohp_flywheel_batch_out_len(const ohp_flywheel_batch* b);
size_t ohp_flywheel_batch_num_prep(const ohp_flywheel_batch* b);
const ohp_chunk_desc* ohp_flywheel_batch_prep(const ohp_flywheel_batch* b);
const ohp_flywheel_job* ohp_flywheel_batch_jobs(const ohp_flywheel_batch* b); /* one per planned starvation              */
size_t ohp_flywheel_batch_num_blocks(const ohp_flywheel_batch* b);
const ohp_chunk_desc* ohp_flywheel_batch_blocks(const ohp_flywheel_batch* b);
/* how far the three arenas are used: sizes[0] training, [1] generated, [2] out (each including its base) */
void   ohp_flywheel_batch_arena_bytes(const ohp_flywheel_batch* b, uint64_t sizes[3]);
void   ohp_flywheel_batch_free(ohp_flywheel_batch* b);

/*
 * RampGenerator::Start + EndBlock (Media/Pipeline/StarvationRamper.cpp:235-247, 351-364): the generated flywheel audio
 * of `job` (ohp_flywheel.h), resident at [src_off, ...) of the ramp pass's input arena, leaves as one MsgAudioPcm per
 * 1 ms block, ramped down from current_ramp over the whole generated length (SetMuted once the ramp has reached
 * Ramp::kMin).  Writes one descriptor per block to out[0..cap) with dst_off advancing from `dst_off`; returns their
 * number, or a negative ohp_status (-OHP_E_INVALID_DESC where the reference would ASSERT, -OHP_E_NO_MEMORY when cap is
 * too small).  *final_ramp (may be NULL) = RampGenerator::iCurrentRampValue afterwards.
 */
int    ohp_flywheel_ramp_chunks(const ohp_flywheel_job* job, uint32_t current_ramp, uint64_t src_off, uint64_t dst_off,
                                ohp_chunk_desc* out, size_t cap, uint32_t* final_ramp);

/* Scalar helpers mirroring the reference (exported for binding-level tests) ------------------- */
/* Jiffies::PerSample (Msg.cpp:424-470); 0 for an unsupported rate (the reference throws SampleRateInvalid). */
uint32_t ohp_jiffies_per_sample(uint32_t sample_rate);
/* Ramp::Set (Msg.cpp:590-712) on {start,end,direction,enabled}; returns 1 iff a split ramp was produced,
 * 0 if not, <0 where the reference would ASSERT. */
typedef struct ohp_ramp { uint32_t start, end, direction, enabled; } ohp_ramp;
int      ohp_ramp_set(ohp_ramp* ramp, uint32_t start, uint32_t fragment_size, uint32_t remaining_duration,
                      uint32_t direction, ohp_ramp* split, uint32_t* split_pos);
/* Ramp::Split (Msg.cpp:784-807): *ramp becomes the first part, returns the remainder in *remaining. */
int      ohp_ramp_split(ohp_ramp* ramp, uint32_t new_size, uint32_t current_size, ohp_ramp* remaining);

#ifdef __cplusplus
}
#endif
#endif /* OHP_SCHEDULE_H */
