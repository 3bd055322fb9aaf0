"""The class-free schedule walk (ohpipeline_b200/host/schedule_walk.h -- the source the GPU schedule kernels compile,
run here on host threads through ohp_schedule_build_walk) against the reference's playables (tests/golden) and
against the class-based host model.  CPU only; tests/test_gpu_schedule.py repeats this on the device."""
import glob
import os

import numpy as np
import pytest

from ohpipeline_b200 import abi, capi, workloads

GOLDEN = sorted(g for g in glob.glob(os.path.join(os.path.dirname(__file__), "golden", "*.npz"))
                if not g.endswith(("ramp_algebra.npz", "flywheel.npz")))


def check(w_streams, w_events):
    try:
        host = capi.schedule_build(w_streams, w_events)
    except capi.OhpError as eh:
        with pytest.raises(capi.OhpError) as ew:
            capi.schedule_build(w_streams, w_events, walk=True)
        assert ew.value.status == eh.status
        return None
    walk = capi.schedule_build(w_streams, w_events, walk=True)
    assert np.array_equal(walk.stream_chunk_begin, host.stream_chunk_begin)
    assert np.array_equal(walk.stream_out_bytes, host.stream_out_bytes)
    assert np.array_equal(walk.chunks, host.chunks)
    assert np.array_equal(walk.info, host.info)
    return host


@pytest.mark.parametrize("path", GOLDEN, ids=[os.path.basename(p)[:-4] for p in GOLDEN])
def test_walk_reproduces_reference_playables(path):
    g = np.load(path)
    walk = capi.schedule_build(g["streams"], g["events"], threads=2, walk=True)
    assert np.array_equal(walk.chunks, g["chunks"])
    assert np.array_equal(walk.info, g["info"])


@pytest.mark.parametrize("seed", range(40, 52))
def test_walk_matches_class_model_on_mixed_workloads(seed):
    w = workloads.mixed(n_streams=80, seed=seed, max_frames=4000)
    check(w.streams, w.events)


def test_walk_matches_class_model_on_baseline_configs():
    for w in (workloads.config1(6.2), workloads.config2(n_streams=8, seconds=0.5),
              workloads.config3(n_streams=40, seconds=1.0), workloads.config5(n_streams=16, seconds=0.25)):
        assert check(w.streams, w.events) is not None


def test_walk_refuses_what_the_class_model_refuses():
    w = workloads.config5(n_streams=4, seconds=0.02)
    for field, index, value, status in (("sample_rate", 2, 12345, abi.E_INVALID_ARG), ("bit_depth", 1, 20, abi.E_INVALID_DESC),
                                        ("out_fmt", 0, abi.OUT_PLANAR32_BE, abi.E_INVALID_ARG),
                                        ("chunk_frames", 3, 0, abi.E_INVALID_ARG), ("channels", 1, 33, abi.E_INVALID_ARG),
                                        ("channels", 2, 257, abi.E_INVALID_ARG), ("chunk_frames", 0, 0x80000001, abi.E_INVALID_ARG)):
        bad = w.streams.copy()
        bad[field][index] = value
        with pytest.raises(capi.OhpError) as e:
            capi.schedule_build(bad, w.events, walk=True)
        assert e.value.status == status, field
        assert check(bad, w.events) is None
    # seed 21 of the 3001-stream mix holds a MsgSilence split below one sample: the reference ASSERTs
    w = workloads.mixed(n_streams=3001, seed=21, max_frames=700)
    assert check(w.streams, w.events) is None


@pytest.mark.parametrize("seed", range(8))
def test_bulk_step_edges_match_class_model(seed):
    w = workloads.steady_edges(seed)
    # stream by stream, so that one the reference ASSERTs on does not hide its neighbours
    asserted = 0
    for k in range(len(w.streams)):
        s = w.streams[k:k + 1].copy()
        ev = w.events[int(s[0]["first_event"]):int(s[0]["first_event"]) + int(s[0]["num_events"])].copy()
        s[0]["first_event"] = 0
        if check(s, ev) is None:
            asserted += 1
    assert asserted < len(w.streams) // 4


@pytest.mark.parametrize("seed", [4, 21, 22, 23])
def test_walk_matches_class_model_on_pipeline_shaped_mix(seed):
    w = workloads.config4(n_streams=300, seconds=0.3, seed=seed)
    assert check(w.streams, w.events) is not None


def test_starvation_ramps_at_every_rate_take_exactly_their_duration():
    """SuiteStarvationRamper's properties (TestStarvationRamper.cpp:324-346, 634-692, 861-915) on the host model and the
    walk, for all 18 rates x 4 depths: the ramp down takes exactly 20 ms of audio, the ramp up exactly 50 ms, every
    playable's ramp starts where the previous one ended, what lies between is muted, the rest untouched."""
    w = workloads.all_rates()
    host = check(w.streams, w.events)
    assert host is not None and len(w.streams) == 18 * 4
    ms = abi.JIFFIES_PER_MS
    for s in range(len(w.streams)):
        a, b = int(host.stream_chunk_begin[s]), int(host.stream_chunk_begin[s + 1])
        c, info = host.chunks[a:b], host.info[a:b]
        down = info["direction"] == abi.DIR_DOWN
        up = info["direction"] == abi.DIR_UP
        assert int(info["jiffies"][down].sum()) == 20 * ms and int(info["jiffies"][up].sum()) == 50 * ms
        for sel, first, last in ((down, abi.RAMP_MAX, 0), (up, 0, abi.RAMP_MAX)):
            starts, ends = c["ramp_start"][sel], c["ramp_end"][sel]
            assert starts[0] == first and ends[-1] == last
            assert np.array_equal(starts[1:], ends[:-1])
        i_down, i_up = np.nonzero(down)[0], np.nonzero(up)[0]
        between = c[i_down[-1] + 1:i_up[0]]
        assert len(between) and (between["flags"] & abi.F_SILENCE).all()          # Halt: muted audio plays as silence
        outside = np.concatenate([c[:i_down[0]], c[i_up[-1] + 1:]])
        assert not (outside["flags"] & (abi.F_RAMP_ENABLED | abi.F_SILENCE)).any()


@pytest.mark.parametrize("rate,bits", [(44100, 16), (192000, 24), (48000, 32)])
def test_ramp_lengths_of_the_pipeline_elements(rate, bits):
    """SuiteRamper / SuiteMuter (TestRamper.cpp:399-437, TestMuter.cpp:306-338): a ramp takes exactly the jiffies it was
    configured with -- Ramper's long and short ramps (500 / 50 ms, Pipeline.h:102-104), Muter's 500 ms, StarvationRamper's
    20 ms down / 50 ms up -- wherever in a message it starts; audio outside it is untouched (up) or muted (after down)."""
    ms = abi.JIFFIES_PER_MS
    jps = abi.jiffies_per_sample(rate)
    chunk = workloads.max_chunk_frames(rate, bits, 2)
    total = rate * 2
    for dur_ms in (20, 50, 500):
        for op, mute_first in ((abi.EV_RAMP_DOWN, False), (abi.EV_RAMP_UP, True)):
            start = 300 * ms + 12345            # mid-message, mid-sample
            ev = ([(0, 0, abi.EV_MUTE, 0)] if mute_first else []) + [(start, 0, op, dur_ms * ms)]
            w = workloads._finish("ramp length", [workloads._spec(rate, bits, 2, False, chunk, total)], [ev], seed=1)
            host = check(w.streams, w.events)
            assert host is not None
            d = host.info["direction"]
            sel = d == (abi.DIR_DOWN if op == abi.EV_RAMP_DOWN else abi.DIR_UP)
            assert int(host.info["jiffies"][sel].sum()) == dur_ms * ms
            c = host.chunks[sel]
            assert c["ramp_start"][0] == (abi.RAMP_MAX if op == abi.EV_RAMP_DOWN else 0)
            assert c["ramp_end"][-1] == (0 if op == abi.EV_RAMP_DOWN else abi.RAMP_MAX)
            assert np.array_equal(c["ramp_start"][1:], c["ramp_end"][:-1])
            first, last = np.nonzero(sel)[0][[0, -1]]
            before, after = host.chunks[:first], host.chunks[last + 1:]
            quiet = abi.F_SILENCE
            if op == abi.EV_RAMP_DOWN:
                assert not (before["flags"] & (abi.F_RAMP_ENABLED | quiet)).any() and (after["flags"] & quiet).all() and len(after)
            else:
                assert (before["flags"] & quiet).all() and not (after["flags"] & (abi.F_RAMP_ENABLED | quiet)).any() and len(after)
            # the bytes in front of the ramp are whole samples: the split at a mid-sample jiffy rounds down (Msg.cpp:2236-2240)
            assert int(before["bytes"].sum()) == (start // jps) * 2 * bits // 8


def test_closed_form_bound_covers_every_stream():
    """ohp_run_streams_device builds the descriptors in ONE walk per stream into regions sized by a closed-form upper bound
    (sched::stream_chunk_bound): the bound must hold for every stream of every generator, and stay close where streams are
    long (padding descriptors cost the hot path a record and a ticket each)."""
    from ohpipeline_b200 import workloads as W
    cases = [W.config1(6.2), W.config2(8, 1.0), W.config3(48, 1.0), W.config4(200, 0.25), W.config5(32, 1.0), W.all_rates()]
    cases += [W.mixed(64, s, 4000) for s in range(6)] + [W.steady_edges(s, 64) for s in range(4)]
    cases += [W.elements(s, 32, illegal=(s % 2 == 0)) for s in range(4)] + [W.config4(64, 0.1, seed=s) for s in range(4)]
    streams = 0
    for w in cases:
        bounds = capi.schedule_chunk_bounds(w.streams, w.events)
        exact = 0
        for k in range(len(w.streams)):
            st = w.streams[k:k + 1].copy()
            ev = w.events[int(st[0]["first_event"]):int(st[0]["first_event"]) + int(st[0]["num_events"])]
            st[0]["first_event"] = 0
            try:
                n = len(capi.schedule_build(st, ev, walk=True).chunks)
            except capi.OhpError:
                continue                      # the reference ASSERTs: no descriptors either way
            assert n <= int(bounds[k]), (w.name, k, n, int(bounds[k]))
            exact += n
            streams += 1
        if w.name.startswith(("config2", "config3", "config5")):
            assert int(bounds.sum()) <= 1.06 * exact, (w.name, int(bounds.sum()), exact)
    assert streams > 900
    # a spec the walk refuses has no region
    bad = W.config5(2, 0.05)
    bad.streams["sample_rate"][1] = 12345
    assert int(capi.schedule_chunk_bounds(bad.streams, bad.events)[1]) == 0
