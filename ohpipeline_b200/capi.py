"""ctypes binding of the C ABI (include/ohp_b200.h, include/ohp_schedule.h).

This is the Python stand-in for the cgo/JNI/ctypes stub a host application would write (see INTEGRATION.md).
The libraries are built in-tree by __graft_entry__.build():
    ohpipeline_b200/libohp_b200.so   CUDA kernels + C ABI (nvcc, sm_100a)
    ohpipeline_b200/libohp_host.so   host message model + schedule runner (g++)
There is NO fallback: a missing library raises ImportError-like OhpError at first use, and every compute
entry point fails with a non-zero status when no sm_100 GPU is present.
"""
import ctypes as C
import os

import numpy as np

from . import abi

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_CUDA = os.environ.get("OHP_LIB_CUDA") or os.path.join(_HERE, "libohp_b200.so")  # override: kernel-tuning experiments
LIB_HOST = os.path.join(_HERE, "libohp_host.so")


class OhpError(RuntimeError):
    def __init__(self, status, message):
        super().__init__("ohp status %d: %s" % (status, message))
        self.status = status


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


_cuda = None
_host = None


def cuda_lib():
    """Load libohp_b200.so (raises if it was not built -- there is nothing to fall back to)."""
    global _cuda
    if _cuda is None:
        if not os.path.exists(LIB_CUDA):
            raise OhpError(-1, "%s not built; run __graft_entry__.build()" % LIB_CUDA)
        L = C.CDLL(LIB_CUDA)
        L.ohp_abi_version.restype = C.c_uint32
        L.ohp_device_count.restype = C.c_int
        L.ohp_create.restype = C.c_int
        L.ohp_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
        L.ohp_destroy.restype = C.c_int
        L.ohp_destroy.argtypes = [C.c_void_p]
        L.ohp_last_error.restype = C.c_char_p
        L.ohp_last_error.argtypes = [C.c_void_p]
        L.ohp_ramp_table.restype = C.POINTER(C.c_uint16)
        L.ohp_median_multiplier.restype = C.c_uint32
        L.ohp_median_multiplier.argtypes = [C.c_uint32, C.c_uint32, C.c_uint32, C.c_int]
        if hasattr(L, "ohp_chunk_out_bytes"):  # absent only from older experiment builds loaded through OHP_LIB_CUDA
            L.ohp_chunk_out_bytes.restype = C.c_uint32
            L.ohp_chunk_out_bytes.argtypes = [C.c_void_p]
        L.ohp_validate.restype = C.c_int
        L.ohp_validate.argtypes = [C.c_void_p, C.c_size_t, C.c_uint64, C.c_uint64, C.POINTER(C.c_size_t)]
        L.ohp_process_device.restype = C.c_int
        L.ohp_process_device.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_uint64,
                                         C.c_void_p, C.c_uint64, C.c_void_p]
        L.ohp_process_host.restype = C.c_int
        L.ohp_process_host.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64]
        L.ohp_sync.restype = C.c_int
        L.ohp_sync.argtypes = [C.c_void_p, C.c_void_p]
        L.ohp_checksums_device.restype = C.c_int
        L.ohp_checksums_device.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p]
        for name in ("ohp_device_alloc", "ohp_host_alloc"):
            f = getattr(L, name); f.restype = C.c_int; f.argtypes = [C.c_void_p, C.c_uint64, C.POINTER(C.c_void_p)]
        for name in ("ohp_device_free", "ohp_host_free"):
            f = getattr(L, name); f.restype = C.c_int; f.argtypes = [C.c_void_p, C.c_void_p]
        for name in ("ohp_memcpy_h2d", "ohp_memcpy_d2h"):
            f = getattr(L, name); f.restype = C.c_int
            f.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p]
        L.ohp_launch_count.restype = C.c_uint64
        L.ohp_launch_count.argtypes = [C.c_void_p]
        if hasattr(L, "ohp_inflight_cap"):
            L.ohp_inflight_cap.restype = C.c_uint32
            L.ohp_inflight_cap.argtypes = [C.c_void_p]
        if hasattr(L, "ohp_flywheel_device"):  # include/ohp_flywheel.h
            L.ohp_flywheel_out_bytes.restype = C.c_uint32
            L.ohp_flywheel_out_bytes.argtypes = [C.c_void_p]
            L.ohp_flywheel_validate.restype = C.c_int
            L.ohp_flywheel_validate.argtypes = [C.c_void_p, C.c_size_t, C.c_uint64, C.c_uint64, C.POINTER(C.c_size_t)]
            L.ohp_flywheel_device.restype = C.c_int
            L.ohp_flywheel_device.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64,
                                              C.c_void_p]
        if hasattr(L, "ohp_schedule_count_device"):  # include/ohp_schedule_device.h
            L.ohp_schedule_count_device.restype = C.c_int
            L.ohp_schedule_count_device.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p,
                                                    C.c_void_p, C.POINTER(C.c_uint64), C.c_void_p]
            L.ohp_schedule_emit_device.restype = C.c_int
            L.ohp_schedule_emit_device.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p,
                                                   C.c_void_p, C.c_void_p, C.c_void_p]
        if hasattr(L, "ohp_run_streams_host"):
            L.ohp_run_streams_host.restype = C.c_int
            L.ohp_run_streams_host.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p, C.c_uint64,
                                               C.c_void_p, C.c_uint64, C.c_void_p, C.POINTER(C.c_uint64)]
        if hasattr(L, "ohp_run_streams_device_flywheel"):
            L.ohp_run_streams_device_flywheel.restype = C.c_int
            L.ohp_run_streams_device_flywheel.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p,
                                                          C.c_uint64, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_void_p,
                                                          C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_uint64), C.c_void_p]
        if hasattr(L, "ohp_run_streams_device_flywheel_recent"):  # include/ohp_starvation_recent.h
            L.ohp_run_streams_device_flywheel_recent.restype = C.c_int
            L.ohp_run_streams_device_flywheel_recent.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p,
                                                                 C.c_uint64, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_void_p,
                                                                 C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                                                 C.POINTER(C.c_uint64), C.c_void_p]
        if hasattr(L, "ohp_run_streams_device"):
            L.ohp_run_streams_device.restype = C.c_int
            L.ohp_run_streams_device.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p, C.c_uint64,
                                                 C.c_void_p, C.c_uint64, C.c_void_p, C.POINTER(C.c_uint64), C.c_void_p]
            L.ohp_fill_streams_device.restype = C.c_int
            L.ohp_fill_streams_device.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_size_t, C.c_uint64, C.c_uint64,
                                                  C.c_void_p]
        # include/ohp_multi.h
        L.ohp_multi_create.restype = C.c_int
        L.ohp_multi_create.argtypes = [C.POINTER(C.c_int), C.c_size_t, C.POINTER(C.c_void_p)]
        L.ohp_multi_destroy.restype = C.c_int
        L.ohp_multi_destroy.argtypes = [C.c_void_p]
        L.ohp_multi_num_devices.restype = C.c_size_t
        L.ohp_multi_num_devices.argtypes = [C.c_void_p]
        L.ohp_multi_last_error.restype = C.c_char_p
        L.ohp_multi_last_error.argtypes = [C.c_void_p]
        L.ohp_multi_shard.restype = None
        L.ohp_multi_shard.argtypes = [C.c_size_t, C.c_size_t, C.c_size_t, C.POINTER(C.c_size_t), C.POINTER(C.c_size_t)]
        L.ohp_multi_run_streams_host.restype = C.c_int
        L.ohp_multi_run_streams_host.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p, C.c_uint64,
                                                 C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.POINTER(C.c_uint64)]
        L.ohp_multi_host_alloc.restype = C.c_int
        L.ohp_multi_host_alloc.argtypes = [C.c_void_p, C.c_uint64, C.POINTER(C.c_void_p)]
        L.ohp_multi_host_free.restype = C.c_int
        L.ohp_multi_host_free.argtypes = [C.c_void_p, C.c_void_p]
        L.ohp_multi_context.restype = C.c_void_p
        L.ohp_multi_context.argtypes = [C.c_void_p, C.c_size_t]
        L.ohp_set_timing.restype = C.c_int
        L.ohp_set_timing.argtypes = [C.c_void_p, C.c_int]
        L.ohp_last_kernel_ms.restype = C.c_double
        L.ohp_last_kernel_ms.argtypes = [C.c_void_p]
        _cuda = L
    return _cuda


def host_lib():
    global _host
    if _host is None:
        if not os.path.exists(LIB_HOST):
            raise OhpError(-1, "%s not built; run __graft_entry__.build()" % LIB_HOST)
        L = C.CDLL(LIB_HOST)
        L.ohp_schedule_build.restype = C.c_int
        L.ohp_schedule_build.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_int, C.POINTER(C.c_void_p)]
        L.ohp_schedule_build_walk.restype = C.c_int
        L.ohp_schedule_build_walk.argtypes = L.ohp_schedule_build.argtypes
        L.ohp_schedule_num_starvations.restype = C.c_size_t
        L.ohp_schedule_num_starvations.argtypes = [C.c_void_p]
        L.ohp_schedule_starvations.restype = C.c_void_p
        L.ohp_schedule_starvations.argtypes = [C.c_void_p]
        L.ohp_flywheel_plan.restype = C.c_int
        L.ohp_flywheel_plan.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64, C.c_void_p, C.POINTER(C.c_size_t),
                                        C.c_void_p, C.c_void_p, C.c_size_t, C.POINTER(C.c_size_t)]
        L.ohp_schedule_recent_audio.restype = C.c_void_p
        L.ohp_schedule_recent_audio.argtypes = [C.c_void_p]
        L.ohp_schedule_recent_begin.restype = C.c_void_p
        L.ohp_schedule_recent_begin.argtypes = [C.c_void_p]
        L.ohp_flywheel_plan_recent.restype = C.c_int
        L.ohp_flywheel_plan_recent.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_uint64, C.c_uint64, C.c_uint64,
                                               C.c_void_p, C.c_size_t, C.POINTER(C.c_size_t), C.c_void_p, C.c_void_p, C.c_size_t,
                                               C.POINTER(C.c_size_t)]
        L.ohp_flywheel_plan_batch.restype = C.c_int
        L.ohp_flywheel_plan_batch.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_uint64, C.c_uint64, C.c_uint64,
                                              C.POINTER(C.c_void_p)]
        L.ohp_flywheel_plan_batch_recent.restype = C.c_int
        L.ohp_flywheel_plan_batch_recent.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_uint64,
                                                     C.c_uint64, C.c_uint64, C.POINTER(C.c_void_p)]
        for name in ("num_planned", "num_prep", "num_blocks"):
            f = getattr(L, "ohp_flywheel_batch_" + name); f.restype = C.c_size_t; f.argtypes = [C.c_void_p]
        for name in ("planned", "out_off", "out_len", "prep", "jobs", "blocks"):
            f = getattr(L, "ohp_flywheel_batch_" + name); f.restype = C.c_void_p; f.argtypes = [C.c_void_p]
        L.ohp_flywheel_batch_arena_bytes.restype = None
        L.ohp_flywheel_batch_arena_bytes.argtypes = [C.c_void_p, C.POINTER(C.c_uint64)]
        L.ohp_flywheel_batch_free.restype = None
        L.ohp_flywheel_batch_free.argtypes = [C.c_void_p]
        L.ohp_flywheel_ramp_chunks.restype = C.c_int
        L.ohp_flywheel_ramp_chunks.argtypes = [C.c_void_p, C.c_uint32, C.c_uint64, C.c_uint64, C.c_void_p, C.c_size_t,
                                               C.POINTER(C.c_uint32)]
        L.ohp_container_parse.restype = C.c_int
        L.ohp_container_parse.argtypes = [C.c_void_p, C.c_uint64, C.c_uint32, C.c_void_p]
        L.ohp_container_stream_spec.restype = C.c_int
        L.ohp_container_stream_spec.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64, C.c_void_p]
        L.ohp_codec_message_frames.restype = C.c_size_t
        L.ohp_codec_message_frames.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t]
        L.ohp_schedule_chunk_bounds.restype = C.c_int
        L.ohp_schedule_chunk_bounds.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p]
        L.ohp_schedule_num_chunks.restype = C.c_size_t
        L.ohp_schedule_num_chunks.argtypes = [C.c_void_p]
        for name in ("ohp_schedule_chunks", "ohp_schedule_chunk_info", "ohp_schedule_stream_chunk_begin",
                     "ohp_schedule_stream_out_bytes"):
            f = getattr(L, name); f.restype = C.c_void_p; f.argtypes = [C.c_void_p]
        L.ohp_schedule_last_error.restype = C.c_char_p
        L.ohp_schedule_free.argtypes = [C.c_void_p]
        L.ohp_jiffies_per_sample.restype = C.c_uint32
        L.ohp_jiffies_per_sample.argtypes = [C.c_uint32]
        L.ohp_ramp_set.restype = C.c_int
        L.ohp_ramp_set.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p,
                                   C.POINTER(C.c_uint32)]
        L.ohp_ramp_split.restype = C.c_int
        L.ohp_ramp_split.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p]
        _host = L
    return _host


def flywheel_plan_recent(stream, starvation, recent, training_off=0, generated_off=0, out_off=0, prep_cap=64):
    """ohp_flywheel_plan_recent: as flywheel_plan, from the element's recent audio piece by piece (silence included)."""
    stream = np.ascontiguousarray(stream, dtype=abi.STREAM_SPEC).reshape(1)
    starvation = np.ascontiguousarray(starvation, dtype=abi.STARVATION).reshape(1)
    recent = np.ascontiguousarray(recent, dtype=abi.RECENT_AUDIO)
    prep = np.zeros(max(prep_cap, 1), dtype=abi.CHUNK_DESC)
    job = np.zeros(1, dtype=abi.FLYWHEEL_JOB)
    blocks = np.zeros(64, dtype=abi.CHUNK_DESC)
    n, n_prep = C.c_size_t(0), C.c_size_t(0)
    L = host_lib()
    rc = L.ohp_flywheel_plan_recent(_ptr(stream), _ptr(starvation), _ptr(recent) if len(recent) else None, len(recent),
                                    C.c_uint64(training_off), C.c_uint64(generated_off), C.c_uint64(out_off),
                                    _ptr(prep), prep_cap, C.byref(n_prep), _ptr(job), _ptr(blocks), len(blocks), C.byref(n))
    if rc != 0:
        raise OhpError(rc, L.ohp_schedule_last_error().decode())
    return prep[:n_prep.value].copy(), job, blocks[:n.value].copy()


class FlywheelBatch:
    """ohp_flywheel_plan_batch: the arrays of the three launches for every starvation of a batch that plays and is planned."""

    def __init__(self, planned, out_off, out_len, prep, jobs, blocks, arena_bytes):
        self.planned, self.out_off, self.out_len = planned, out_off, out_len
        self.prep, self.jobs, self.blocks = prep, jobs, blocks
        self.training_bytes, self.generated_bytes, self.out_bytes = arena_bytes


def flywheel_plan_batch(streams, starvations, training_base=0, generated_base=0, out_base=0, recent=None, recent_begin=None):
    """ohp_flywheel_plan_batch; with recent / recent_begin (Schedule.recent, .recent_begin) ohp_flywheel_plan_batch_recent."""
    streams = np.ascontiguousarray(streams, dtype=abi.STREAM_SPEC)
    starvations = np.ascontiguousarray(starvations, dtype=abi.STARVATION)
    L = host_lib()
    h = C.c_void_p()
    if recent_begin is not None:
        recent = np.ascontiguousarray(recent, dtype=abi.RECENT_AUDIO)
        recent_begin = np.ascontiguousarray(recent_begin, dtype=np.uint64)
        assert len(recent_begin) == len(starvations) + 1 and int(recent_begin[-1]) <= len(recent)
        rc = L.ohp_flywheel_plan_batch_recent(_ptr(streams) if len(streams) else None, len(streams),
                                              _ptr(starvations) if len(starvations) else None, len(starvations),
                                              _ptr(recent) if len(recent) else None, _ptr(recent_begin),
                                              C.c_uint64(training_base), C.c_uint64(generated_base), C.c_uint64(out_base), C.byref(h))
    else:
        rc = L.ohp_flywheel_plan_batch(_ptr(streams) if len(streams) else None, len(streams),
                                       _ptr(starvations) if len(starvations) else None, len(starvations),
                                       C.c_uint64(training_base), C.c_uint64(generated_base), C.c_uint64(out_base), C.byref(h))
    if rc != 0:
        raise OhpError(rc, L.ohp_schedule_last_error().decode())
    try:
        def take(name, n, dtype):
            a = np.zeros(n, dtype=dtype)
            if n:
                C.memmove(_ptr(a), getattr(L, "ohp_flywheel_batch_" + name)(h), a.nbytes)
            return a
        n = L.ohp_flywheel_batch_num_planned(h)
        sizes = (C.c_uint64 * 3)()
        L.ohp_flywheel_batch_arena_bytes(h, sizes)
        return FlywheelBatch(take("planned", n, np.uint32), take("out_off", n, np.uint64), take("out_len", n, np.uint64),
                             take("prep", L.ohp_flywheel_batch_num_prep(h), abi.CHUNK_DESC), take("jobs", n, abi.FLYWHEEL_JOB),
                             take("blocks", L.ohp_flywheel_batch_num_blocks(h), abi.CHUNK_DESC), tuple(int(x) for x in sizes))
    finally:
        L.ohp_flywheel_batch_free(h)


# ---------------------------------------------------------------------------------------------------
# host message model / schedule runner

def jiffies_per_sample(rate):
    return int(host_lib().ohp_jiffies_per_sample(rate))


def ramp_set(ramp, start, fragment_size, remaining_duration, direction):
    """Ramp::Set.  ramp = (start, end, direction, enabled).  Returns (rc, ramp, split, split_pos)."""
    r = np.array([tuple(ramp)], dtype=abi.RAMP)
    s = np.zeros(1, dtype=abi.RAMP)
    pos = C.c_uint32(0)
    rc = host_lib().ohp_ramp_set(_ptr(r), start, fragment_size, remaining_duration, direction, _ptr(s), C.byref(pos))
    return rc, tuple(int(x) for x in r[0]), tuple(int(x) for x in s[0]), pos.value


def ramp_split(ramp, new_size, current_size):
    r = np.array([tuple(ramp)], dtype=abi.RAMP)
    rem = np.zeros(1, dtype=abi.RAMP)
    rc = host_lib().ohp_ramp_split(_ptr(r), new_size, current_size, _ptr(rem))
    return rc, tuple(int(x) for x in r[0]), tuple(int(x) for x in rem[0])


def container_parse(data, max_bit_depth=32):
    """ohp_container_parse on a bytes-like object: (status, info record)."""
    buf = np.frombuffer(bytes(data), dtype=np.uint8)
    info = np.zeros(1, dtype=abi.CONTAINER_INFO)
    rc = host_lib().ohp_container_parse(_ptr(buf) if buf.size else None, buf.size, max_bit_depth, _ptr(info))
    return int(rc), info[0]


def container_stream_spec(info, container_len, arena_offset=0, dst_base=0):
    """ohp_container_stream_spec: (status, STREAM_SPEC record)."""
    rec = np.array([info], dtype=abi.CONTAINER_INFO)
    spec = np.zeros(1, dtype=abi.STREAM_SPEC)
    rc = host_lib().ohp_container_stream_spec(_ptr(rec), container_len, arena_offset, dst_base, _ptr(spec))
    return int(rc), spec[0]


def codec_message_frames(spec):
    """Frames of every message the stream enters the pipeline with (ohp_codec_message_frames)."""
    rec = np.array([spec], dtype=abi.STREAM_SPEC)
    n = host_lib().ohp_codec_message_frames(_ptr(rec), None, 0)
    out = np.zeros(n, dtype=np.uint32)
    host_lib().ohp_codec_message_frames(_ptr(rec), _ptr(out), n)
    return out


def flywheel_ramp_chunks(job, current_ramp, src_off, dst_off):
    """RampGenerator::Start/EndBlock for one flywheel job: (descriptors, final ramp value).
    Raises OhpError where the reference would ASSERT."""
    job = np.ascontiguousarray(job, dtype=abi.FLYWHEEL_JOB).reshape(1)
    descs = np.zeros(64, dtype=abi.CHUNK_DESC)
    final = C.c_uint32(0)
    n = host_lib().ohp_flywheel_ramp_chunks(_ptr(job), current_ramp, src_off, dst_off, _ptr(descs), len(descs), C.byref(final))
    if n < 0:
        raise OhpError(-n, host_lib().ohp_schedule_last_error().decode())
    return descs[:n].copy(), int(final.value)


def flywheel_validate(jobs, in_bytes, out_bytes):
    """ohp_flywheel_validate; returns (status, bad_index)."""
    jobs = np.ascontiguousarray(jobs, dtype=abi.FLYWHEEL_JOB)
    bad = C.c_size_t(0)
    rc = cuda_lib().ohp_flywheel_validate(_ptr(jobs), len(jobs), in_bytes, out_bytes, C.byref(bad))
    return int(rc), int(bad.value)


def flywheel_job(rate, channels, bits, src_off=0, dst_off=0):
    """A job shaped like StarvationRamper's: 1 ms of training, 20 ms of generated audio."""
    jps = abi.jiffies_per_sample(rate)
    j = np.zeros(1, dtype=abi.FLYWHEEL_JOB)
    j[0] = (src_off, dst_off, rate, abi.FLYWHEEL_RAMP_JIFFIES // jps, abi.FLYWHEEL_TRAINING_JIFFIES // jps, channels, bits, 0)
    return j


def schedule_chunk_bounds(streams, events):
    """ohp_schedule_chunk_bounds: the per-stream upper bound on playables ohp_run_streams_device sizes its regions with."""
    streams = np.ascontiguousarray(streams, dtype=abi.STREAM_SPEC)
    events = np.ascontiguousarray(events, dtype=abi.RAMP_EVENT)
    out = np.zeros(len(streams), dtype=np.uint64)
    rc = host_lib().ohp_schedule_chunk_bounds(_ptr(streams), len(streams), _ptr(events) if len(events) else None, len(events), _ptr(out))
    if rc != 0:
        raise OhpError(rc, "ohp_schedule_chunk_bounds")
    return out


class Schedule:
    """Result of ohp_schedule_build: chunk descriptors for a batch of streams."""

    def __init__(self, chunks, info, chunk_begin, out_bytes, starvations=None):
        self.chunks = chunks
        self.info = info
        self.stream_chunk_begin = chunk_begin
        self.stream_out_bytes = out_bytes
        self.starvations = starvations if starvations is not None else np.zeros(0, dtype=abi.STARVATION)  # ohp_schedule_build only
        self.recent = np.zeros(0, dtype=abi.RECENT_AUDIO)       # ... the elements' recent audio, piece by piece
        self.recent_begin = np.zeros(len(self.starvations) + 1, dtype=np.uint64)  # ... record k's pieces: [begin[k], begin[k + 1])

    def recent_of(self, k):
        return self.recent[int(self.recent_begin[k]):int(self.recent_begin[k + 1])]


def schedule_build(streams, events, threads=0, walk=False):
    """Run the ramp events of every stream through the stage chain; returns a Schedule.
    Raises OhpError(E_INVALID_DESC) where the reference would ASSERT.
    walk=True: the class-free walk (ohp_schedule_build_walk), the source the GPU schedule kernels compile."""
    L = host_lib()
    streams = np.ascontiguousarray(streams, dtype=abi.STREAM_SPEC)
    events = np.ascontiguousarray(events, dtype=abi.RAMP_EVENT)
    h = C.c_void_p()
    build = L.ohp_schedule_build_walk if walk else L.ohp_schedule_build
    rc = build(_ptr(streams), len(streams), _ptr(events), len(events), threads, C.byref(h))
    if rc != 0:
        raise OhpError(rc, L.ohp_schedule_last_error().decode())
    try:
        n = L.ohp_schedule_num_chunks(h)
        chunks = np.zeros(n, dtype=abi.CHUNK_DESC)
        info = np.zeros(n, dtype=abi.CHUNK_INFO)
        if n:
            C.memmove(_ptr(chunks), L.ohp_schedule_chunks(h), n * abi.CHUNK_DESC.itemsize)
            C.memmove(_ptr(info), L.ohp_schedule_chunk_info(h), n * abi.CHUNK_INFO.itemsize)
        ns = len(streams)
        begin = np.zeros(ns + 1, dtype=np.uint64)
        outb = np.zeros(ns, dtype=np.uint64)
        C.memmove(_ptr(begin), L.ohp_schedule_stream_chunk_begin(h), (ns + 1) * 8)
        if ns:
            C.memmove(_ptr(outb), L.ohp_schedule_stream_out_bytes(h), ns * 8)
        nst = L.ohp_schedule_num_starvations(h)
        starved = np.zeros(nst, dtype=abi.STARVATION)
        if nst:
            C.memmove(_ptr(starved), L.ohp_schedule_starvations(h), nst * abi.STARVATION.itemsize)
        rbegin = np.zeros(nst + 1, dtype=np.uint64)
        if not walk:
            C.memmove(_ptr(rbegin), L.ohp_schedule_recent_begin(h), rbegin.nbytes)
        recent = np.zeros(int(rbegin[-1]), dtype=abi.RECENT_AUDIO)
        if len(recent):
            C.memmove(_ptr(recent), L.ohp_schedule_recent_audio(h), recent.nbytes)
    finally:
        L.ohp_schedule_free(h)
    sched = Schedule(chunks, info, begin, outb, starved)
    sched.recent, sched.recent_begin = recent, rbegin
    return sched


def flywheel_plan(stream, starvation, training_off=0, generated_off=0, out_off=0):
    """ohp_flywheel_plan: the three launches of one starvation as data -> (prep descriptors, job, block descriptors).
    Raises OhpError where the starvation plays nothing, its training block is not PCM throughout, or the reference would ASSERT."""
    stream = np.ascontiguousarray(stream, dtype=abi.STREAM_SPEC).reshape(1)
    starvation = np.ascontiguousarray(starvation, dtype=abi.STARVATION).reshape(1)
    prep = np.zeros(abi.FLYWHEEL_MAX_PREP, dtype=abi.CHUNK_DESC)
    job = np.zeros(1, dtype=abi.FLYWHEEL_JOB)
    blocks = np.zeros(64, dtype=abi.CHUNK_DESC)
    n = C.c_size_t(0)
    n_prep = C.c_size_t(0)
    L = host_lib()
    rc = L.ohp_flywheel_plan(_ptr(stream), _ptr(starvation), C.c_uint64(training_off), C.c_uint64(generated_off), C.c_uint64(out_off),
                             _ptr(prep), C.byref(n_prep), _ptr(job), _ptr(blocks), len(blocks), C.byref(n))
    if rc != 0:
        raise OhpError(rc, L.ohp_schedule_last_error().decode())
    return prep[:n_prep.value].copy(), job, blocks[:n.value].copy()


# ---------------------------------------------------------------------------------------------------
# GPU context

def device_count():
    return int(cuda_lib().ohp_device_count())


def ramp_table():
    p = cuda_lib().ohp_ramp_table()
    return np.array([p[i] for i in range(512)], dtype=np.uint16)


def median_multiplier(start, end, direction, enabled):
    return int(cuda_lib().ohp_median_multiplier(start, end, direction, int(bool(enabled))))


def validate(descs, in_bytes, out_bytes):
    """ohp_validate; returns (status, bad_index)."""
    descs = np.ascontiguousarray(descs, dtype=abi.CHUNK_DESC)
    bad = C.c_size_t(0)
    rc = cuda_lib().ohp_validate(_ptr(descs), len(descs), in_bytes, out_bytes, C.byref(bad))
    return int(rc), int(bad.value)


class Context:
    """One ohp_context (one GPU).  All pointer arguments are raw addresses (int) or numpy arrays."""

    def __init__(self, device=0):
        self._L = cuda_lib()
        h = C.c_void_p()
        rc = self._L.ohp_create(device, C.byref(h))
        if rc != 0:
            raise OhpError(rc, self._L.ohp_last_error(None).decode())
        self._h = h
        self.device = device

    def close(self):
        if self._h:
            self._L.ohp_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != 0:
            raise OhpError(rc, self._L.ohp_last_error(self._h).decode())

    def process_device(self, d_descs, n, d_in, in_bytes, d_out, out_bytes, stream=None):
        """Asynchronous: device pointers (ints).  stream = raw cudaStream_t or None."""
        self._check(self._L.ohp_process_device(self._h, C.c_void_p(d_descs), n, C.c_void_p(d_in), in_bytes,
                                               C.c_void_p(d_out), out_bytes, C.c_void_p(stream or 0)))

    def process_host(self, descs, inp, out):
        """Synchronous, host numpy buffers: H2D + kernel + D2H inside the call."""
        descs = np.ascontiguousarray(descs, dtype=abi.CHUNK_DESC)
        assert inp.dtype == np.uint8 and out.dtype == np.uint8 and inp.flags.c_contiguous and out.flags.c_contiguous
        self._check(self._L.ohp_process_host(self._h, _ptr(descs), len(descs), _ptr(inp), inp.size, _ptr(out), out.size))

    def process_host_ptr(self, descs_ptr, n, in_ptr, in_bytes, out_ptr, out_bytes):
        self._check(self._L.ohp_process_host(self._h, C.c_void_p(descs_ptr), n, C.c_void_p(in_ptr), in_bytes,
                                             C.c_void_p(out_ptr), out_bytes))

    def sync(self, stream=None):
        self._check(self._L.ohp_sync(self._h, C.c_void_p(stream or 0)))

    def checksums_device(self, d_out, d_stream_off, n_streams, d_sums, stream=None):
        self._check(self._L.ohp_checksums_device(self._h, C.c_void_p(d_out), C.c_void_p(d_stream_off), n_streams,
                                                 C.c_void_p(d_sums), C.c_void_p(stream or 0)))

    def device_alloc(self, nbytes):
        p = C.c_void_p()
        self._check(self._L.ohp_device_alloc(self._h, nbytes, C.byref(p)))
        return p.value

    def device_free(self, ptr):
        self._check(self._L.ohp_device_free(self._h, C.c_void_p(ptr)))

    def host_alloc(self, nbytes):
        """Pinned host memory as a numpy uint8 array (freed with host_free(arr))."""
        p = C.c_void_p()
        self._check(self._L.ohp_host_alloc(self._h, nbytes, C.byref(p)))
        buf = (C.c_uint8 * nbytes).from_address(p.value)
        arr = np.frombuffer(buf, dtype=np.uint8)
        return arr, p.value

    def host_free(self, ptr):
        self._check(self._L.ohp_host_free(self._h, C.c_void_p(ptr)))

    def memcpy_h2d(self, dptr, harr, stream=None):
        self._check(self._L.ohp_memcpy_h2d(self._h, C.c_void_p(dptr), _ptr(harr), harr.nbytes, C.c_void_p(stream or 0)))

    def memcpy_d2h(self, harr, dptr, stream=None):
        self._check(self._L.ohp_memcpy_d2h(self._h, _ptr(harr), C.c_void_p(dptr), harr.nbytes, C.c_void_p(stream or 0)))

    def launch_count(self):
        return int(self._L.ohp_launch_count(self._h))

    def inflight_cap(self):
        return int(self._L.ohp_inflight_cap(self._h))

    def flywheel_device(self, d_jobs, n, d_in, in_bytes, d_out, out_bytes, stream=None):
        """Asynchronous: FlywheelRamperManager::Ramp + RampGenerator::ProcessFragment for n jobs (device pointers)."""
        self._check(self._L.ohp_flywheel_device(self._h, C.c_void_p(d_jobs), n, C.c_void_p(d_in), in_bytes,
                                                C.c_void_p(d_out), out_bytes, C.c_void_p(stream or 0)))

    # device-side schedule builder (include/ohp_schedule_device.h); all pointers are raw device addresses
    def schedule_count_device(self, d_streams, n_streams, d_events, n_events, d_chunk_begin, d_out_bytes=0, stream=None):
        total = C.c_uint64(0)
        self._check(self._L.ohp_schedule_count_device(self._h, C.c_void_p(d_streams), n_streams, C.c_void_p(d_events),
                                                      n_events, C.c_void_p(d_chunk_begin), C.c_void_p(d_out_bytes),
                                                      C.byref(total), C.c_void_p(stream or 0)))
        return int(total.value)

    def schedule_emit_device(self, d_streams, n_streams, d_events, n_events, d_chunk_begin, d_chunks, d_info=0, stream=None):
        self._check(self._L.ohp_schedule_emit_device(self._h, C.c_void_p(d_streams), n_streams, C.c_void_p(d_events),
                                                     n_events, C.c_void_p(d_chunk_begin), C.c_void_p(d_chunks),
                                                     C.c_void_p(d_info), C.c_void_p(stream or 0)))

    def schedule_build_device(self, streams, events):
        """Host-array convenience around the two calls: uploads specs and events, builds the descriptors ON THE GPU
        and returns a Schedule of host copies (tests); production callers keep everything in HBM."""
        streams = np.ascontiguousarray(streams, dtype=abi.STREAM_SPEC)
        events = np.ascontiguousarray(events, dtype=abi.RAMP_EVENT)
        ns, ne = len(streams), len(events)
        ptrs = []

        def dalloc(nbytes):
            ptrs.append(self.device_alloc(max(int(nbytes), 16)))
            return ptrs[-1]

        try:
            d_streams = dalloc(streams.nbytes)
            d_events = dalloc(events.nbytes)
            d_begin = dalloc((ns + 1) * 8)
            d_outb = dalloc(ns * 8)
            if ns:
                self.memcpy_h2d(d_streams, streams.view(np.uint8).reshape(-1))
            if ne:
                self.memcpy_h2d(d_events, events.view(np.uint8).reshape(-1))
            total = self.schedule_count_device(d_streams, ns, d_events, ne, d_begin, d_outb)
            chunks = np.zeros(total, dtype=abi.CHUNK_DESC)
            info = np.zeros(total, dtype=abi.CHUNK_INFO)
            begin = np.zeros(ns + 1, dtype=np.uint64)
            outb = np.zeros(ns, dtype=np.uint64)
            d_chunks = dalloc(chunks.nbytes)
            d_info = dalloc(info.nbytes)
            self.schedule_emit_device(d_streams, ns, d_events, ne, d_begin, d_chunks, d_info)
            if total:
                self.memcpy_d2h(chunks.view(np.uint8).reshape(-1), d_chunks)
                self.memcpy_d2h(info.view(np.uint8).reshape(-1), d_info)
            self.memcpy_d2h(begin.view(np.uint8), d_begin)
            if ns:
                self.memcpy_d2h(outb.view(np.uint8), d_outb)
            self.sync()
        finally:
            for q in ptrs:
                self.device_free(q)
        return Schedule(chunks, info, begin, outb)

    def run_streams_host(self, streams, events, inp, out):
        """ohp_run_streams_host: specs + events + host PCM in, bytes out; returns (per-stream output bytes, chunks)."""
        streams = np.ascontiguousarray(streams, dtype=abi.STREAM_SPEC)
        events = np.ascontiguousarray(events, dtype=abi.RAMP_EVENT)
        assert inp.dtype == np.uint8 and out.dtype == np.uint8 and inp.flags.c_contiguous and out.flags.c_contiguous
        outb = np.zeros(len(streams), dtype=np.uint64)
        total = C.c_uint64(0)
        self._check(self._L.ohp_run_streams_host(self._h, _ptr(streams) if len(streams) else None, len(streams),
                                                 _ptr(events) if len(events) else None, len(events),
                                                 _ptr(inp) if inp.size else None, inp.size, _ptr(out), out.size,
                                                 _ptr(outb) if len(streams) else None, C.byref(total)))
        return outb, int(total.value)

    def run_streams_device(self, d_streams, n_streams, d_events, n_events, d_in, in_bytes, d_out, out_bytes,
                           d_stream_out_bytes=0, stream=None, want_total=True):
        """ohp_run_streams_device: the whole stage for a batch resident in HBM (raw device addresses), enqueued on `stream`.
        want_total: also wait for the schedule walks and return the number of playables (else None: nothing but the
        regions' size is waited for)."""
        total = C.c_uint64(0)
        self._check(self._L.ohp_run_streams_device(self._h, C.c_void_p(d_streams), n_streams, C.c_void_p(d_events), n_events,
                                                   C.c_void_p(d_in), in_bytes, C.c_void_p(d_out), out_bytes,
                                                   C.c_void_p(d_stream_out_bytes), C.byref(total) if want_total else None,
                                                   C.c_void_p(stream or 0)))
        return int(total.value) if want_total else None

    def run_streams_device_flywheel(self, d_streams, n_streams, d_events, n_events, d_in, in_bytes, d_out, out_bytes,
                                    d_fly_out, fly_out_bytes, d_fly_off, d_fly_len, d_starvations=0, d_stream_out_bytes=0,
                                    stream=None, want_total=True):
        """ohp_run_streams_device_flywheel: run_streams_device, plus the flywheel audio every starving StarvationRamper plays
        (event e's at d_fly_out + d_fly_off[e], d_fly_len[e] bytes) and, where d_starvations is given, the starvation
        records (abi.STARVATION, one per event).  Raw device addresses; returns the playables read (None without want_total)."""
        total = C.c_uint64(0)
        self._check(self._L.ohp_run_streams_device_flywheel(self._h, C.c_void_p(d_streams), n_streams, C.c_void_p(d_events), n_events,
                                                            C.c_void_p(d_in), in_bytes, C.c_void_p(d_out), out_bytes,
                                                            C.c_void_p(d_fly_out), fly_out_bytes, C.c_void_p(d_starvations),
                                                            C.c_void_p(d_fly_off), C.c_void_p(d_fly_len),
                                                            C.c_void_p(d_stream_out_bytes), C.byref(total) if want_total else None,
                                                            C.c_void_p(stream or 0)))
        return int(total.value) if want_total else None

    def run_streams_device_flywheel_recent(self, d_streams, n_streams, d_events, n_events, d_in, in_bytes, d_out, out_bytes,
                                           d_fly_out, fly_out_bytes, d_fly_off, d_fly_len, d_starvations=0, d_stream_out_bytes=0,
                                           stream=None, want_total=True, d_recent=0, d_recent_count=0):
        """ohp_run_streams_device_flywheel_recent: run_streams_device_flywheel with every starvation planned from the element's
        recent audio, silence included; where given, event e's pieces (abi.RECENT_AUDIO) at d_recent + e *
        abi.DEVICE_RECENT_PIECES and their number (uint32, abi.RECENT_INCOMPLETE: more than the walk keeps) at d_recent_count[e]."""
        total = C.c_uint64(0)
        self._check(self._L.ohp_run_streams_device_flywheel_recent(
            self._h, C.c_void_p(d_streams), n_streams, C.c_void_p(d_events), n_events, C.c_void_p(d_in), in_bytes, C.c_void_p(d_out),
            out_bytes, C.c_void_p(d_fly_out), fly_out_bytes, C.c_void_p(d_starvations), C.c_void_p(d_fly_off), C.c_void_p(d_fly_len),
            C.c_void_p(d_stream_out_bytes), C.c_void_p(d_recent), C.c_void_p(d_recent_count),
            C.byref(total) if want_total else None, C.c_void_p(stream or 0)))
        return int(total.value) if want_total else None

    def fill_streams_device(self, d_in, in_bytes, d_streams, n_streams, seed_base, first_stream_id=0, stream=None):
        """ohp_fill_streams_device: seeded synthetic PCM per stream, generated in HBM."""
        self._check(self._L.ohp_fill_streams_device(self._h, C.c_void_p(d_in), in_bytes, C.c_void_p(d_streams), n_streams,
                                                    C.c_uint64(seed_base), C.c_uint64(first_stream_id), C.c_void_p(stream or 0)))

    def set_timing(self, enabled):
        self._check(self._L.ohp_set_timing(self._h, int(bool(enabled))))

    def last_kernel_ms(self):
        return float(self._L.ohp_last_kernel_ms(self._h))


def multi_shard(n_streams, n_devices, index):
    """ohp_multi_shard: (first, count) of the block of streams device `index` of n_devices takes."""
    first, count = C.c_size_t(0), C.c_size_t(0)
    cuda_lib().ohp_multi_shard(n_streams, n_devices, index, C.byref(first), C.byref(count))
    return int(first.value), int(count.value)


class MultiContext:
    """One ohp_multi (include/ohp_multi.h): a context, a host thread and its own CUDA streams per device, streams dealt in
    contiguous blocks, no collective."""

    def __init__(self, devices):
        self._L = cuda_lib()
        devs = (C.c_int * len(devices))(*devices)
        h = C.c_void_p()
        rc = self._L.ohp_multi_create(devs, len(devices), C.byref(h))
        if rc != 0:
            raise OhpError(rc, self._L.ohp_last_error(None).decode())
        self._h = h
        self.devices = list(devices)

    def close(self):
        if self._h:
            self._L.ohp_multi_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != 0:
            raise OhpError(rc, self._L.ohp_multi_last_error(self._h).decode())

    def host_alloc(self, nbytes):
        p = C.c_void_p()
        self._check(self._L.ohp_multi_host_alloc(self._h, nbytes, C.byref(p)))
        return np.frombuffer((C.c_uint8 * nbytes).from_address(p.value), dtype=np.uint8), p.value

    def host_free(self, ptr):
        self._check(self._L.ohp_multi_host_free(self._h, C.c_void_p(ptr)))

    def inflight_cap(self, index):
        return int(self._L.ohp_inflight_cap(C.c_void_p(self._L.ohp_multi_context(self._h, index))))

    def run_streams_host(self, streams, events, inp, out, checksums=True):
        """ohp_multi_run_streams_host -> (per-stream output bytes, per-stream checksums or None, playables read)."""
        streams = np.ascontiguousarray(streams, dtype=abi.STREAM_SPEC)
        events = np.ascontiguousarray(events, dtype=abi.RAMP_EVENT)
        assert inp.dtype == np.uint8 and out.dtype == np.uint8 and inp.flags.c_contiguous and out.flags.c_contiguous
        outb = np.zeros(len(streams), dtype=np.uint64)
        sums = np.zeros(len(streams), dtype=np.uint64) if checksums else None
        total = C.c_uint64(0)
        self._check(self._L.ohp_multi_run_streams_host(self._h, _ptr(streams) if len(streams) else None, len(streams),
                                                       _ptr(events) if len(events) else None, len(events),
                                                       _ptr(inp) if inp.size else None, inp.size, _ptr(out) if out.size else None, out.size,
                                                       _ptr(outb) if len(streams) else None,
                                                       _ptr(sums) if checksums and len(streams) else None, C.byref(total)))
        return outb, sums, int(total.value)
