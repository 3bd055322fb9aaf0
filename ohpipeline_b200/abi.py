"""Plain-data mirror of include/ohp_b200.h and include/ohp_schedule.h (numpy dtypes + constants).

No library is loaded here; see capi.py for the ctypes binding.  Field order and sizes must match the C
headers exactly -- tests/test_abi.py checks sizeof/offsetof against the built library.
"""
import numpy as np

ABI_VERSION = 3

RAMP_MAX = 16384          # Ramp::kMax, OpenHome/Media/Pipeline/Msg.h:257
RAMP_MIN = 0
UNITY_ATTENUATION = 256   # MsgAudioPcm::kUnityAttenuation, Msg.cpp:2219
MAX_PCM_CHUNK_BYTES = 9216  # AudioData::kMaxBytes, Msg.h:117
JIFFIES_PER_SECOND = 56448000  # Jiffies::kPerSecond, Msg.h:193
JIFFIES_PER_MS = 56448
MAX_STAGES = 4

# ohp_status
OK, E_INVALID_ARG, E_INVALID_DESC, E_NO_DEVICE, E_CUDA, E_OUT_OF_RANGE, E_NO_MEMORY = range(7)

# chunk flags
F_RAMP_ENABLED = 0x01
F_SILENCE = 0x02
F_IN_LITTLE_ENDIAN = 0x04

# ohp_out_fmt
OUT_PACKED_BE = 0
OUT_PACKED_LE = 1
OUT_PLANAR32_BE = 2
OUT_FROM32_BE = 3
OUT_SONGCAST = 4
LE_APPEND = 1  # aux of OUT_PACKED_LE: every fragment (0: what the reference's sink holds after the read)

# Ramp::EDirection
DIR_NONE, DIR_UP, DIR_DOWN, DIR_MUTE = range(4)

# ohp_event_op
EV_RAMP_DOWN = 1
EV_RAMP_UP = 2
EV_MUTE = 3
EV_UNMUTE = 4
EV_SET_ATTENUATION = 5
EV_INSERT_SILENCE = 6
EV_MAX_MSG_JIFFIES = 7
EV_RAMPER_STREAM = 8
EV_MUTER_MUTE = 9
EV_MUTER_UNMUTE = 10
EV_HALT = 11
EV_STARVATION = 12

CHUNK_DESC = np.dtype([
    ("src_off", "<u8"), ("dst_off", "<u8"), ("bytes", "<u4"),
    ("ramp_start", "<u2"), ("ramp_end", "<u2"), ("attenuation", "<u2"),
    ("bit_depth", "u1"), ("channels", "u1"), ("flags", "u1"), ("out_fmt", "u1"),
    ("aux", "<u2"),
])
assert CHUNK_DESC.itemsize == 32

CHUNK_INFO = np.dtype([("direction", "<u4"), ("jiffies", "<u4")])

# include/ohp_container.h
CONTAINER_INFO = np.dtype([
    ("kind", "<u4"), ("sample_rate", "<u4"), ("bit_depth_src", "<u4"), ("bit_depth", "<u4"), ("channels", "<u4"),
    ("little_endian", "<u4"), ("bit_rate", "<u4"), ("streaming", "<u4"), ("data_offset", "<u8"), ("audio_bytes", "<u8"),
    ("total_frames", "<u8"), ("track_length_jiffies", "<u8"),
])
assert CONTAINER_INFO.itemsize == 64
CONTAINER_WAV, CONTAINER_AIFF, CONTAINER_AIFC = 1, 2, 3
CONTAINER_OK, CONTAINER_E_UNRECOGNISED, CONTAINER_E_ENDED, CONTAINER_E_CORRUPT, CONTAINER_E_UNSUPPORTED, CONTAINER_E_ARG = range(6)

# include/ohp_schedule.h: ohp_starvation
STARVATION = np.dtype([
    ("stream", "<u8"), ("pcm_jiffies", "<u8"), ("event", "<u4"), ("ramp", "<u4"), ("plays", "<u4"), ("recent_jiffies", "<u4"),
    ("attenuation", "<u4"), ("reserved", "<u4"),
])
assert STARVATION.itemsize == 40
FLYWHEEL_MAX_PREP = 9
# include/ohp_schedule.h: ohp_recent_audio
RECENT_AUDIO = np.dtype([("pcm_jiffies", "<u8"), ("jiffies", "<u4"), ("silence", "<u4"), ("attenuation", "<u4"), ("reserved", "<u4")])
assert RECENT_AUDIO.itemsize == 24
FLYWHEEL_MAX_PREP_RECENT = 64
# include/ohp_starvation_recent.h
DEVICE_RECENT_PIECES = 16              # pieces of recent audio the device walk keeps per StarvationRamper stage
RECENT_INCOMPLETE = 0xFFFFFFFF         # a record that needs more pieces than that: not played

# include/ohp_flywheel.h
FLYWHEEL_JOB = np.dtype([
    ("src_off", "<u8"), ("dst_off", "<u8"), ("sample_rate", "<u4"), ("out_frames", "<u4"),
    ("train_frames", "<u2"), ("channels", "u1"), ("bit_depth", "u1"), ("reserved", "<u4"),
])
assert FLYWHEEL_JOB.itemsize == 32
FLYWHEEL_DEGREE = 3
FLYWHEEL_TRAINING_JIFFIES = 56448      # StarvationRamper::kTrainingJiffies (StarvationRamper.cpp:374)
FLYWHEEL_RAMP_JIFFIES = 20 * 56448     # StarvationRamper::kRampDownJiffies (StarvationRamper.cpp:375)

RAMP_EVENT = np.dtype([
    ("at_jiffies", "<u8"), ("stage", "<u4"), ("op", "<u4"), ("arg", "<u4"), ("reserved", "<u4"),
])
assert RAMP_EVENT.itemsize == 24

STREAM_SPEC = np.dtype([
    ("sample_rate", "<u4"), ("bit_depth", "<u4"), ("channels", "<u4"), ("in_little_endian", "<u4"),
    ("chunk_frames", "<u4"), ("out_fmt", "<u4"),
    ("total_frames", "<u8"), ("src_base", "<u8"), ("dst_base", "<u8"),
    ("first_event", "<u4"), ("num_events", "<u4"), ("driver_block_frames", "<u4"), ("codec_read_frames", "<u4"),
])
assert STREAM_SPEC.itemsize == 64

RAMP = np.dtype([("start", "<u4"), ("end", "<u4"), ("direction", "<u4"), ("enabled", "<u4")])

PCM_SAMPLE_RATES = (7350, 8000, 11025, 12000, 14700, 16000, 22050, 24000, 29400, 32000,
                    44100, 48000, 88200, 96000, 176400, 192000, 352800, 384000)


def jiffies_per_sample(rate: int) -> int:
    """Jiffies::PerSample (Msg.cpp:424-470) for PCM rates; 0 if unsupported."""
    return JIFFIES_PER_SECOND // rate if rate in PCM_SAMPLE_RATES else 0


def chunk_out_bytes(descs: np.ndarray) -> np.ndarray:
    """Vectorised ohp_chunk_out_bytes."""
    b = (descs["bit_depth"] // 8).astype(np.uint64)
    ch = descs["channels"].astype(np.uint64)
    nbytes = descs["bytes"].astype(np.uint64)
    frames = nbytes // np.maximum(b * ch, 1)
    out = nbytes.copy()
    fmt = descs["out_fmt"]
    # ProcessorPcmSwpEndianPacked to the letter (aux 0): of a ramped 16/24-bit playable only the last <= 256-byte fragment
    fb = np.maximum(b * ch, 1)
    spf = np.maximum(256 // fb, 1)
    last = (frames - (np.maximum(frames, 1) - 1) // spf * spf) * fb
    ramped = (descs["flags"] & F_RAMP_ENABLED) != 0
    out = np.where((fmt == OUT_PACKED_LE) & (descs["aux"] == 0) & ramped & (b >= 2) & (frames > 0), last, out)
    out = np.where(fmt == OUT_PLANAR32_BE, frames * ch * 4, out)
    out = np.where(fmt == OUT_FROM32_BE, (nbytes // 4) * (descs["aux"].astype(np.uint64) // 8), out)
    out = np.where(fmt == OUT_SONGCAST, frames * np.minimum(ch, 2) * np.minimum(b, 3), out)
    return out
