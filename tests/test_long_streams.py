"""The stage past 32 bits, on the host: streams longer than 2^32 jiffies (76.1 s) with events at and beside 2^32 and
2^33, ramps of 2^32 - 1 jiffies, starvations whose StarvationRamper saw more than 2^32 jiffies of unbroken PCM
(tests/long_util.py).  A wrapped position still produces plausible playables, so every check is a comparison with an
independent computation at these magnitudes: the class-free walk against the class model, its recent audio against the
class model's, the class model against the C oracle's own message model and against the reference's own element objects,
the oracle's bytes against the reference's, and the device walk's FP64 ramp recurrence restated against integer division.

The comparisons with the reference run where its build (oracle/_ref/libohref.so) is present, and skip elsewhere."""
import os
import subprocess

import numpy as np
import pytest

from ohpipeline_b200 import abi, capi
from long_util import T32, fp64_edge_streams, long_streams, split

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def long_w():
    return long_streams()


@pytest.fixture(scope="module")
def model(long_w):
    return capi.schedule_build(long_w.streams, long_w.events)


@pytest.mark.parametrize("threads", [1, 0], ids=["one_thread", "all_threads"])
def test_walk_equals_the_class_model_past_2_32(long_w, model, threads):
    walk = capi.schedule_build(long_w.streams, long_w.events, threads=threads, walk=True)
    assert np.array_equal(walk.stream_chunk_begin, model.stream_chunk_begin)
    assert np.array_equal(walk.stream_out_bytes, model.stream_out_bytes)
    assert np.array_equal(walk.chunks, model.chunks)
    assert np.array_equal(walk.info, model.info)
    assert len(walk.starvations) == len(model.starvations)
    for f in abi.STARVATION.names:
        assert np.array_equal(walk.starvations[f], model.starvations[f]), f
    # what the streams reach: records past 2^32 and 2^33, saturated runs of PCM, every stream's bytes
    sv = model.starvations
    assert (sv["pcm_jiffies"] > T32).sum() >= 30 and (sv["pcm_jiffies"] > 2 * T32).sum() >= 10
    assert (sv["recent_jiffies"] == 0xFFFFFFFF).sum() >= 8
    assert (sv["plays"] == 1).sum() >= 20


def test_walk_equals_the_class_model_on_fp64_edge_streams():
    w, _ = fp64_edge_streams()
    want = capi.schedule_build(w.streams, w.events)
    for threads in (1, 0):
        got = capi.schedule_build(w.streams, w.events, threads=threads, walk=True)
        assert np.array_equal(got.chunks, want.chunks) and np.array_equal(got.info, want.info)
        assert np.array_equal(got.stream_chunk_begin, want.stream_chunk_begin)
        assert np.array_equal(got.stream_out_bytes, want.stream_out_bytes)


def test_the_oracle_message_model_equals_the_class_model(port, long_w, model):
    """ohp_oracle.c's own stage model (the oracle the GPU tests compare bytes with) against the class model, descriptor
    for descriptor, and its end-to-end bytes against the class model's descriptors processed by the oracle."""
    rc, chunks, info, begin, outb = port.schedule_run(long_w.streams, long_w.events)
    assert rc == 0
    assert np.array_equal(begin, model.stream_chunk_begin) and np.array_equal(outb, model.stream_out_bytes)
    assert np.array_equal(chunks, model.chunks)
    assert np.array_equal(info, model.info)
    inp = port.fill_pcm(long_w.in_bytes, long_w.seed)
    rc, out, _, _ = port.run(long_w.streams, long_w.events, inp, long_w.out_bytes)
    assert rc == 0
    rc, want = port.process_chunks(model.chunks, inp, long_w.out_bytes)
    assert rc == 0 and np.array_equal(out, want)


def test_chunk_bounds_cover_every_long_stream(long_w, model):
    bounds = capi.schedule_chunk_bounds(long_w.streams, long_w.events)
    exact = np.diff(model.stream_chunk_begin.astype(np.int64))
    assert (exact <= bounds.astype(np.int64)).all(), np.nonzero(exact > bounds.astype(np.int64))[0]
    w, _ = fp64_edge_streams()
    bounds = capi.schedule_chunk_bounds(w.streams, w.events)
    exact = np.diff(capi.schedule_build(w.streams, w.events, walk=True).stream_chunk_begin.astype(np.int64))
    assert (exact <= bounds.astype(np.int64)).all()


def test_fp64_recurrence_restated_equals_integer_division(tmp_path):
    """The device walk's FP64 ramp step (schedule_walk.h, bulk_step with a warp's team) RESTATED on the host with
    std::fma (IEEE-identical to the GPU's DFMA) and 1.0 / x, not the device code itself -- tests/test_gpu_long_streams.py
    runs the real branch.  Held against core::mul_add_div on every edge case fp64_edge_streams() produces and on 10^7
    seeded adversarial cases (exact multiples of the divisor and their neighbours, remaining within 2^10 of 2^32 - 1,
    size 2^21 - 1)."""
    _, cases = fp64_edge_streams()
    path = tmp_path / "cases.bin"
    arr = np.array([c[:3] for c in cases], dtype=np.uint32)
    with open(path, "wb") as f:
        f.write(np.uint64(len(arr)).tobytes())
        f.write(arr.tobytes())
    exe = str(tmp_path / "fp64_recurrence")
    subprocess.run(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-Wall", "-Wextra", "-o", exe,
                    os.path.join(ROOT, "tests", "cpp", "fp64_recurrence.cpp")], check=True)
    sweep = 4_000_000                                    # three neighbouring divisors each: > 10^7 cases
    r = subprocess.run([exe, str(path), str(sweep)], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-4000:]
    last = r.stdout.strip().splitlines()[-1].split()
    assert last[0] == "checked" and int(last[1]) >= len(cases) + 10_000_000 and int(last[3]) >= 500_000, r.stdout


def starving(w):
    """The indices of w's streams with a StarvationRamper stage."""
    first = w.streams["first_event"].astype(np.int64)
    at = np.nonzero(w.events["op"] == abi.EV_STARVATION)[0]
    return {int(s) for s in np.unique(np.searchsorted(first, at, side="right") - 1)}


def test_walk_keeps_the_recent_audio_of_the_class_model_past_2_32(tmp_path):
    """The walk with the recent audio kept (schedule_walk.h, RECENT, through tests/cpp/recent_harness.cpp, with and
    without the bulk step) against the class model's records and pieces, on the long streams that starve."""
    from recent_util import build
    from test_starvation_walk_recent import check_walk
    w = long_streams()
    keep = starving(w)
    sched, _ = check_walk(build(tmp_path, "recent_harness"), tmp_path, split(w, lambda k: k in keep))
    sv = sched.starvations
    assert (sv["pcm_jiffies"] > T32).sum() >= 20 and len(sched.recent) >= len(sv)


def element_streams(w):
    """The streams of w whose stages are all element objects (no bare ramp op, no message cap), without the ones whose
    StarvationRamper would cut silence for ever (test_elements_vs_reference.without_endless_cuts)."""
    from test_elements_vs_reference import without_endless_cuts
    bare = (abi.EV_RAMP_DOWN, abi.EV_RAMP_UP, abi.EV_MUTE, abi.EV_UNMUTE, abi.EV_MAX_MSG_JIFFIES)
    first = w.streams["first_event"].astype(np.int64)
    ops = [set(int(o) for o in w.events["op"][f:f + int(n)]) for f, n in zip(first, w.streams["num_events"])]
    sub = split(w, lambda k: not (ops[k] & set(bare)))
    return without_endless_cuts(sub)


def test_class_model_is_the_reference_element_objects_past_2_32(ref, port):
    """The reference's own Ramper, Muter and StarvationRamper objects (ref.elements_run) against the class model on the
    long element streams: playables, bytes, sizes.  Then every starvation past 2^32 that plays: the flywheel audio planned
    from the class model's record (ohp_flywheel_plan, played by the C port) against what the real StarvationRamper plays
    (ref.elements_generated_audio).  A disagreement here is a finding about one side at these magnitudes, to be recorded,
    not smoothed over."""
    from test_elements_vs_reference import _flywheel_on_cpu, one_stream
    w = element_streams(long_streams())
    assert len(w.streams) >= 6
    inp = port.fill_pcm(w.in_bytes, w.seed)
    rc, out, chunks, info, begin, outb, generated = ref.elements_run(w.streams, w.events, inp, w.out_bytes)
    assert rc == 0
    model = capi.schedule_build(w.streams, w.events)
    assert np.array_equal(model.chunks, chunks) and np.array_equal(model.info, info)
    assert np.array_equal(model.stream_chunk_begin, begin) and np.array_equal(model.stream_out_bytes, outb)
    rc, want = port.process_chunks(model.chunks, inp, w.out_bytes)
    assert rc == 0 and np.array_equal(out, want)
    compared = 0
    for s in range(len(w.streams)):
        st, ev = one_stream(w, s)
        playing = capi.schedule_build(st, ev).starvations
        playing = playing[playing["plays"] == 1]
        if not len(playing):
            continue
        rc, audio, ramps = ref.elements_generated_audio(st, ev, inp)
        assert rc == 0, s
        assert [int(r) for r in playing["ramp"]] == [int(r) for r in ramps], s
        jps = abi.jiffies_per_sample(int(st[0]["sample_rate"]))
        per = abi.FLYWHEEL_RAMP_JIFFIES // jps * int(st[0]["channels"]) * int(st[0]["bit_depth"]) // 8
        assert audio.size == per * len(playing), s
        for k in range(len(playing)):
            if int(playing["pcm_jiffies"][k]) <= T32:
                continue
            played = _flywheel_on_cpu(port, st, playing[k:k + 1], inp)
            assert np.array_equal(played, audio[k * per:(k + 1) * per]), (s, k, playing[k])
            compared += 1
    assert compared >= 10


def test_oracle_bytes_are_the_reference_bytes_past_2_32(ref, port, long_w):
    """port.run (the oracle the GPU tests compare with) against ref.run (the stage model on the reference's own message
    classes) on every long stream: playables and bytes."""
    inp = port.fill_pcm(long_w.in_bytes, long_w.seed)
    rc, want, want_chunks, want_info = ref.run(long_w.streams, long_w.events, inp, long_w.out_bytes, threads=2)
    assert rc == 0
    rc, got, chunks, info = port.run(long_w.streams, long_w.events, inp, long_w.out_bytes)
    assert rc == 0
    assert np.array_equal(chunks, want_chunks) and np.array_equal(info, want_info)
    assert np.array_equal(got, want)
