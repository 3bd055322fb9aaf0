"""Starvation records from the class-free walk (ohp_schedule_build_walk, the source the device walk compiles) against the
class-based model's (ohp_schedule_build), field by field; and the flywheel planner the device compiles
(ohpipeline_b200/host/flywheel_plan.h) against the class-based ohp_flywheel_plan + ohp_flywheel_ramp_chunks,
descriptor for descriptor, through a small C++ harness."""
import os
import subprocess

import numpy as np
import pytest

from ohpipeline_b200 import abi, capi
from ohpipeline_b200 import workloads as W
from flywheel_util import RATES, every_shape_streams, starved_streams

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MS = abi.JIFFIES_PER_MS


def records(w):
    """(class-based records, walk records) of a workload; the walk keeps no recent audio."""
    want = capi.schedule_build(w.streams, w.events).starvations
    walk = capi.schedule_build(w.streams, w.events, walk=True)
    assert np.array_equal(walk.recent_begin, np.zeros(len(walk.starvations) + 1, dtype=np.uint64))
    return want, walk.starvations


def assert_same_records(w):
    want, got = records(w)
    assert len(got) == len(want), w.name
    for f in abi.STARVATION.names:
        assert np.array_equal(got[f], want[f]), (w.name, f)
    return want


def edge_cases():
    """Hand-built streams at the edges of what a StarvationRamper records."""
    out = []
    spec = lambda rate=48000, bits=16, ch=2, frames=48000 // 5, chunk=None, block=0: W._spec(  # noqa: E731
        rate, bits, ch, False, chunk or W.max_chunk_frames(rate, bits, ch), frames, abi.OUT_PACKED_BE, block)
    end = (48000 // 5) * abi.jiffies_per_sample(48000)
    # the reservoir runs dry exactly where the stream ends (once, then twice)
    out.append(W._finish("at_end", [spec(), spec()], [[(end, 1, abi.EV_STARVATION, 50 * MS)],
                                                      [(end, 1, abi.EV_STARVATION, 50 * MS), (end, 1, abi.EV_STARVATION, 50 * MS)]], seed=1))
    # before any audio, halted, a Muter muted in front of it, a second starvation inside the ramp up before it is audible
    out.append(W._finish("plays_nothing", [spec()] * 4, [
        [(0, 1, abi.EV_STARVATION, 50 * MS), (20 * MS, 1, abi.EV_STARVATION, 50 * MS)],
        [(30 * MS, 1, abi.EV_HALT, 0), (30 * MS, 1, abi.EV_STARVATION, 50 * MS), (90 * MS, 1, abi.EV_STARVATION, 50 * MS)],
        [(5 * MS, 0, abi.EV_MUTER_MUTE, 10 * MS), (60 * MS + 777, 1, abi.EV_STARVATION, 50 * MS)],
        [(40 * MS + 123, 1, abi.EV_STARVATION, 50 * MS), (40 * MS + 123, 1, abi.EV_STARVATION, 50 * MS),
         (41 * MS, 1, abi.EV_STARVATION, 50 * MS), (70 * MS + 9, 1, abi.EV_STARVATION, 50 * MS)],
    ], seed=2))
    # a StarvationRamper on stage 0 and on stage 3, two of them in one stream, behind attenuations and a Ramper's ramp
    out.append(W._finish("stages", [spec(44100, 24, 6), spec(96000, 32, 2), spec(44100, 16, 2, chunk=441, block=300)], [
        [(25 * MS + 4321, 0, abi.EV_STARVATION, 50 * MS), (130 * MS, 0, abi.EV_STARVATION, 30 * MS)],
        [(0, 1, abi.EV_RAMPER_STREAM, 40 * MS), (33 * MS + 1, 3, abi.EV_STARVATION, 50 * MS), (61 * MS + 17, 3, abi.EV_STARVATION, 50 * MS)],
        [(0, 0, abi.EV_RAMPER_STREAM, 40 * MS), (10 * MS, 0, abi.EV_SET_ATTENUATION, 100), (22 * MS + 999, 1, abi.EV_STARVATION, 50 * MS),
         (30 * MS, 2, abi.EV_SET_ATTENUATION, 64), (47 * MS + 5, 3, abi.EV_STARVATION, 20 * MS), (80 * MS, 1, abi.EV_STARVATION, 50 * MS),
         (95 * MS, 2, abi.EV_SET_ATTENUATION, 256), (120 * MS + 3, 3, abi.EV_STARVATION, 50 * MS)],
    ], seed=3))
    return out


@pytest.mark.parametrize("attenuation", [False, True], ids=["plain", "attenuation"])
def test_walk_records_what_the_class_model_records_on_elements(attenuation):
    n = 0
    for seed in range(50):
        n += len(assert_same_records(W.elements(seed, n_streams=24, attenuation=attenuation)))
    assert n > 500


def test_walk_records_what_the_class_model_records_on_starved_streams():
    for name, w, _ in starved_streams():
        assert len(assert_same_records(w)) >= 1, name


@pytest.mark.parametrize("w", edge_cases(), ids=lambda w: w.name)
def test_walk_records_at_the_edges(w):
    want = assert_same_records(w)
    assert len(want) >= 2
    if w.name == "at_end":
        assert len(want) == 3
    if w.name == "plays_nothing":
        assert (want["plays"] == 0).sum() >= 3


def harness(tmp_path):
    exe = str(tmp_path / "flywheel_plan_harness")
    pkg = os.path.join(ROOT, "ohpipeline_b200")
    subprocess.run(["g++", "-std=c++17", "-O1", "-Wall", "-Wextra", "-o", exe, os.path.join(ROOT, "tests", "cpp", "flywheel_plan_harness.cpp"),
                    "-L" + pkg, "-lohp_host", "-Wl,-rpath," + pkg], check=True)
    return exe


def shape_records():
    """Every rate x depth x 1-8 channels (and 9, 10: refused), at pcm positions on, just after and well after a sample
    boundary; plus records every refusal applies to."""
    specs, recs = [], []
    for rate in RATES:
        jps = abi.jiffies_per_sample(rate)
        for bits in (8, 16, 24, 32):
            for ch in range(1, 11):
                sp = np.zeros(1, dtype=abi.STREAM_SPEC)[0]
                sp["sample_rate"], sp["bit_depth"], sp["channels"], sp["in_little_endian"] = rate, bits, ch, ch % 2
                sp["chunk_frames"], sp["out_fmt"], sp["total_frames"], sp["src_base"] = 1, abi.OUT_PACKED_BE, rate, 4096 * ch
                for k, pcm in enumerate((37 * MS // jps * jps, 37 * MS // jps * jps + 100, 37 * MS + 12345, MS, MS - 1, rate * jps,
                                         rate * jps + jps)):
                    r = np.zeros(1, dtype=abi.STARVATION)[0]
                    r["pcm_jiffies"], r["ramp"], r["plays"] = pcm, (16384, 9000, 1, 0, 16383)[k % 5], int(k != 3 or ch != 2)
                    r["recent_jiffies"] = (MS, 5 * MS, MS - 1, 2**32 - 1)[k % 4]
                    r["attenuation"] = 100 if bits == 16 and k % 2 else 256
                    specs.append(sp)
                    recs.append(r)
    return specs, recs


def test_device_planner_equals_the_class_based_plan(tmp_path):
    specs, recs = shape_records()
    for name, w, _ in starved_streams() + [(w.name, w, 0) for w in edge_cases() + [every_shape_streams()]] + \
            [("elements", W.elements(s, n_streams=24, attenuation=bool(s % 2)), 0) for s in range(8)]:
        sv = capi.schedule_build(w.streams, w.events).starvations
        for r in sv:
            specs.append(w.streams[int(r["stream"])])
            recs.append(r)
    path = tmp_path / "records.bin"
    with open(path, "wb") as f:
        f.write(np.uint64(len(recs)).tobytes())
        for sp, r in zip(specs, recs):
            f.write(np.array([sp], dtype=abi.STREAM_SPEC).tobytes())
            f.write(np.array([r], dtype=abi.STARVATION).tobytes())
    r = subprocess.run([harness(tmp_path), str(path)], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-4000:]
    lines = r.stdout.strip().splitlines()
    assert lines[-1].startswith("checked %d " % len(recs)), lines[-1]
    assert len(lines) == 1, "\n".join(lines[:20])
    planned = int(lines[-1].split()[-1])
    assert 1000 < planned < len(recs)
