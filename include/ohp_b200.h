/*
 * ohp_b200.h -- C ABI of the B200-native batch implementation of ohPipeline's
 * decoded-PCM hot path: Ramp application (RampApplicator) fused with the
 * IPcmProcessor sample-format conversion that MsgPlayable::Read performs.
 *
 * This is the drop-in boundary.  Nothing like it exists in the reference (the
 * reference path is an in-process C++ virtual-call chain); each entry point
 * names the reference interface it replaces.  Citations are relative to the
 * ohPipeline source root.
 *
 *   reference                                                    this ABI
 *   ---------------------------------------------------------    -------------------------
 *   MsgPlayablePcm members iAudioData->Ptr(iOffset), iSize,      struct ohp_chunk_desc
 *     iBitDepth, iNumChannels, iAttenuation, iRamp
 *     (OpenHome/Media/Pipeline/Msg.h:1071-1078,1101-1102)
 *   MsgPlayable::Read(IPcmProcessor&)          (Msg.cpp:2646)    ohp_process_device / ohp_process_host
 *   MsgPlayablePcm::ReadBlock                  (Msg.cpp:2753)      (PCM chunks)
 *   MsgPlayableSilence::ReadBlock              (Msg.cpp:2874)      (OHP_F_SILENCE chunks)
 *   RampApplicator::Start/GetNextSample        (Msg.cpp:820-899)   (OHP_F_RAMP_ENABLED)
 *   MsgPlayablePcm::ApplyAttenuation           (Msg.cpp:2736)      (attenuation != 256)
 *   DecodedAudio::ConstructPcm/CopyToBigEndian (Msg.cpp:347-408)   (OHP_F_IN_LITTLE_ENDIAN, fused)
 *   IPcmProcessor::ProcessFragment sinks       (Msg.h:1204-1240)   ohp_out_fmt
 *   RampApplicator::MedianMultiplier           (Msg.cpp:901-920) ohp_median_multiplier
 *   kRampArray                                 (RampArray.h:7-75) ohp_ramp_table
 *
 * All functions return an ohp_status (0 = OK) and never throw across the ABI.
 * There is no CPU fallback: every compute entry point fails with
 * OHP_E_NO_DEVICE / OHP_E_CUDA when no sm_100 device is usable.
 */
#ifndef OHP_B200_H
#define OHP_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define OHP_ABI_VERSION 3u

/* Ramp::kMax / Ramp::kMin (Msg.h:257-258) */
#define OHP_RAMP_MAX 16384u
#define OHP_RAMP_MIN 0u
/* MsgAudioPcm::kUnityAttenuation (Msg.cpp:2219) */
#define OHP_UNITY_ATTENUATION 256u
/* AudioData::kMaxBytes (Msg.h:117): largest PCM playable the reference can hold */
#define OHP_MAX_PCM_CHUNK_BYTES 9216u
#define OHP_RAMP_TABLE_ENTRIES 512u

typedef enum ohp_status {
    OHP_OK = 0,
    OHP_E_INVALID_ARG = 1,   /* null pointer, bad handle, bad size                              */
    OHP_E_INVALID_DESC = 2,  /* a chunk descriptor the reference would ASSERT on                */
    OHP_E_NO_DEVICE = 3,     /* no CUDA device / not an sm_100 part                             */
    OHP_E_CUDA = 4,          /* a CUDA runtime call failed; see ohp_last_error                  */
    OHP_E_OUT_OF_RANGE = 5,  /* descriptor addresses bytes outside the in/out arena             */
    OHP_E_NO_MEMORY = 6
} ohp_status;

/* ohp_chunk_desc::aux for OHP_OUT_PACKED_LE */
#define OHP_LE_APPEND 1u

/* chunk flags */
#define OHP_F_RAMP_ENABLED     0x01u /* Ramp::IsEnabled() (selects the lossy 16-bit path, Msg.cpp:2761) */
#define OHP_F_SILENCE          0x02u /* MsgPlayableSilence: zeros, ramp ignored (Msg.cpp:2874-2893)      */
#define OHP_F_IN_LITTLE_ENDIAN 0x04u /* source bytes are little-endian subsamples (Msg.cpp:380-408)      */

/* Output formats = the IPcmProcessor implementations in the reference tree. */
typedef enum ohp_out_fmt {
    OHP_OUT_PACKED_BE = 0,   /* ProcessorPcmBufTest: verbatim packed big-endian (ProcessorAudioUtils.cpp:31-52)            */
    OHP_OUT_PACKED_LE = 1,   /* ProcessorPcmSwpEndianPacked: per-subsample byte swap, 8/16/24 only
                                (Tests/TestCodecInteractiveMain.cpp:546-590).  aux = 0: what that sink HOLDS after the read,
                                to the letter -- its SwapEndianness16/24 overwrite where ProcessorPcmBufTest appends, so of a
                                ramped 16/24-bit playable (read in fragments of <= 256 bytes, Msg.cpp:2761-2780) only the last
                                fragment is left, and that is all the chunk writes; aux = OHP_LE_APPEND: every fragment, in
                                order (what the stream-level calls and MsgPlayable::Descriptor use)                        */
    OHP_OUT_PLANAR32_BE = 2, /* FlywheelInput: planar, 4 bytes/subsample, left-justified BE (StarvationRamper.cpp:117-186);
                                aux = frames per channel plane                                                             */
    OHP_OUT_FROM32_BE = 3,   /* RampGenerator: 32-bit BE in -> packed aux-bit BE out (StarvationRamper.cpp:281-326)        */
    OHP_OUT_SONGCAST = 4     /* Sender: two channels from index aux, <=3 bytes/subsample (Av/Songcast/Sender.cpp:356-377)  */
} ohp_out_fmt;

/*
 * One MsgPlayable.  32 bytes, 16-byte aligned so a warp can fetch it as two 128-bit loads.
 * `bytes` is the playable's payload size in SOURCE bytes and must be a whole number of
 * frames (bytes % (channels*bit_depth/8) == 0), as MsgPlayable sizes are.
 * A descriptor whose fields from `bytes` on are all zero is an empty slot: it is skipped, never rejected.
 */
typedef struct ohp_chunk_desc {
    uint64_t src_off;     /* byte offset of the first payload byte in the input arena; ignored for silence */
    uint64_t dst_off;     /* byte offset of the first output byte in the output arena                      */
    uint32_t bytes;       /* MsgPlayable::iSize                                                            */
    uint16_t ramp_start;  /* Ramp::iStart, 0..16384                                                        */
    uint16_t ramp_end;    /* Ramp::iEnd,   0..16384                                                        */
    uint16_t attenuation; /* MsgPlayablePcm::iAttenuation; 256 = unity; !=256 requires bit_depth 16        */
    uint8_t  bit_depth;   /* 8, 16, 24, 32                                                                 */
    uint8_t  channels;    /* 1..32 (DecodedAudio::kMaxNumChannels is 8; every sink and mode is tested at 1..32) */
    uint8_t  flags;       /* OHP_F_*                                                                       */
    uint8_t  out_fmt;     /* ohp_out_fmt                                                                   */
    uint16_t aux;         /* per-format parameter, see ohp_out_fmt                                         */
} ohp_chunk_desc;

typedef struct ohp_context ohp_context; /* opaque; one per GPU, thread-compatible */

/* Library / device ---------------------------------------------------------------------------- */
uint32_t    ohp_abi_version(void);
/* Number of usable CUDA devices (0 when there is none; never fails). */
int         ohp_device_count(void);
/* Create a context on `device`.  Uploads the ramp table (kRampArray, RampArray.h:7-75). */
int         ohp_create(int device, ohp_context** out_ctx);
int         ohp_destroy(ohp_context* ctx);
/* Text of the most recent failure on this context (or of ohp_create when ctx is NULL). */
const char* ohp_last_error(const ohp_context* ctx);
/* The 512-entry Q15 ramp curve this library applies (host copy, for cross-checking). */
const uint16_t* ohp_ramp_table(void);
/* RampApplicator::MedianMultiplier (Msg.cpp:901-920) with MsgAudio::MedianRampMultiplier's
 * short-circuits (Msg.cpp:2063-2074): 0x8000 when !enabled, 0 when muted.  The reference reads
 * kRampArray[512] (out of bounds) when the median ramp is 0; this returns 0 there.              */
uint32_t    ohp_median_multiplier(uint32_t ramp_start, uint32_t ramp_end, uint32_t direction, int enabled);

/* Descriptor helpers -------------------------------------------------------------------------- */
/* Bytes chunk `d` writes at dst_off (differs from d->bytes for planar/from32/songcast). */
uint32_t    ohp_chunk_out_bytes(const ohp_chunk_desc* d);
/* Check `n` descriptors against the reference's ASSERTs and the arena sizes.
 * On failure *bad_index (may be NULL) receives the first offending descriptor. */
int         ohp_validate(const ohp_chunk_desc* descs, size_t n, uint64_t in_bytes, uint64_t out_bytes,
                         size_t* bad_index);

/* Hot path ------------------------------------------------------------------------------------ */
/*
 * Replaces MsgPlayable::Read for `n` playables at once.  All pointers are DEVICE pointers on the
 * context's device; `stream` is a cudaStream_t (NULL = the context's own stream).  Asynchronous:
 * returns after enqueueing.  Descriptors are checked on the device; a violation is reported by
 * the next ohp_sync as OHP_E_INVALID_DESC / OHP_E_OUT_OF_RANGE and that chunk is skipped.
 */
int         ohp_process_device(ohp_context* ctx, const ohp_chunk_desc* d_descs, size_t n,
                               const uint8_t* d_in, uint64_t in_bytes,
                               uint8_t* d_out, uint64_t out_bytes, void* stream);
/*
 * Same, with HOST buffers: validates, copies descriptors and input to the device, runs the
 * kernel and copies the output back, pipelined in slices over the context's copy streams.
 * Synchronous.  h_in / h_out may be pageable; pinned memory (ohp_host_alloc) is faster.
 * Only bytes some chunk covers are written to h_out: everything else reads afterwards as the caller left it (a hole of
 * up to 4 KiB between two covered ranges is overwritten and restored while the call runs).  However the call ends, no
 * copy or kernel of it is still in flight when it returns.
 */
int         ohp_process_host(ohp_context* ctx, const ohp_chunk_desc* h_descs, size_t n,
                             const uint8_t* h_in, uint64_t in_bytes,
                             uint8_t* h_out, uint64_t out_bytes);
/* Wait for everything enqueued on the context's stream (or `stream`) and report device-side
 * descriptor errors.  An error is reported once, by the first call or ohp_sync that reads it;
 * ohp_last_error names every error found. */
int         ohp_sync(ohp_context* ctx, void* stream);

/*
 * Per-stream 64-bit checksums of the output arena: stream s covers bytes
 * [stream_off[s], stream_off[s+1]) of d_out; sum_s = SUM_i (byte_i + 1) * (i + 1) mod 2^64 with i
 * the byte index inside the stream.  Device pointers; `d_stream_off` has n_streams+1 entries.
 */
int         ohp_checksums_device(ohp_context* ctx, const uint8_t* d_out, const uint64_t* d_stream_off,
                                 size_t n_streams, uint64_t* d_sums, void* stream);

/* Memory helpers (thin wrappers so a host language needs no CUDA binding of its own) ---------- */
int         ohp_device_alloc(ohp_context* ctx, uint64_t bytes, void** out_dptr);
int         ohp_device_free(ohp_context* ctx, void* dptr);
int         ohp_host_alloc(ohp_context* ctx, uint64_t bytes, void** out_hptr); /* pinned */
int         ohp_host_free(ohp_context* ctx, void* hptr);
int         ohp_memcpy_h2d(ohp_context* ctx, void* dptr, const void* hptr, uint64_t bytes, void* stream);
int         ohp_memcpy_d2h(ohp_context* ctx, void* hptr, const void* dptr, uint64_t bytes, void* stream);

/* Instrumentation ----------------------------------------------------------------------------- */
/* Kernel launches issued by this context since creation (bench.py's gpu_launches). */
uint64_t    ohp_launch_count(const ohp_context* ctx);
/* Chunks per thread block the most recent ohp_process_device launch kept in flight.  Large batches are tuned: the first
 * few launches of a batch shape (same n, in_bytes, out_bytes) each try a candidate between CUDA events on the caller's
 * stream, later ones use the fastest (OHP_AUTOTUNE=0 or OHP_CAP_CHUNKS=<k> in the environment switch that off).
 * The value never changes results. */
uint32_t    ohp_inflight_cap(const ohp_context* ctx);
/* Device time, in ms, of the most recent ohp_process_device kernel(s), measured with CUDA events
 * on the launching stream; blocks until they finish.  -1 when timing is disabled. */
int         ohp_set_timing(ohp_context* ctx, int enabled);
double      ohp_last_kernel_ms(ohp_context* ctx);

#ifdef __cplusplus
}
#endif
#endif /* OHP_B200_H */
