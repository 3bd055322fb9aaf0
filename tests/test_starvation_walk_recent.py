"""The recent audio the device walk keeps (ohpipeline_b200/host/schedule_walk.h with RECENT, built on the host by
tests/cpp/recent_harness.cpp) against the class model's (ohp_schedule_build): the records field by field, the pieces after
StartFlywheelRamp's cut, OHP_RECENT_INCOMPLETE exactly where the class model keeps more than the ring holds; and the
device planner flyplan::plan_recent against ohp_flywheel_plan_recent, status and descriptors."""
import subprocess

import numpy as np
import pytest

from ohpipeline_b200 import abi, capi
from ohpipeline_b200 import workloads as W
from flywheel_util import DEPTHS, RATES, every_shape_streams, starved_streams
from recent_util import K, MS, T, build, cut, host_walk, refusal_streams, silence_heavy_streams
from test_starvation_walk import edge_cases


def workloads():
    out = [W.elements(s, n_streams=24, attenuation=a) for s in range(50) for a in (False, True)]
    out += [w for _, w, _ in starved_streams()] + [every_shape_streams()] + edge_cases()
    return out + [silence_heavy_streams(), refusal_streams()]


@pytest.fixture(scope="module")
def walk_exe(tmp_path_factory):
    return build(tmp_path_factory.mktemp("recent"), "recent_harness")


def check_walk(exe, tmp_path, w):
    """-> (class-model schedule, records the walk's pieces are incomplete for)."""
    sched = capi.schedule_build(w.streams, w.events)
    sv = sched.starvations
    ev = sv["event"].astype(np.int64)
    incomplete = 0
    for bulk, (rcs, rec, cnt, pcs) in zip((True, False), host_walk(exe, tmp_path, w)):
        assert np.all(rcs == 0), w.name
        have = np.nonzero(rec["event"] != 0xFFFFFFFF)[0]
        assert np.array_equal(have, np.sort(ev)), w.name
        for f in abi.STARVATION.names:
            assert np.array_equal(rec[ev][f], sv[f]), (w.name, f)
        assert np.all(cnt[np.setdiff1d(np.arange(len(w.events)), ev)] == 0), w.name
        for k, e in enumerate(ev):
            want = sched.recent_of(k)
            if cnt[e] == abi.RECENT_INCOMPLETE:
                assert len(want) > K, (w.name, bulk, k)
                incomplete += 1
                continue
            assert len(want) <= K and cnt[e] >= 1 or len(want) == 0, (w.name, bulk, k, len(want), cnt[e])
            got = pcs[e][:cnt[e]]
            assert cut(got) == cut(want), (w.name, bulk, k)
            if not bulk:   # message by message the pieces are the class model's, the front one included
                assert cut(got) == cut(want) and len(got) == len(want), (w.name, k)
    return sched, incomplete


def test_walk_keeps_the_recent_audio_of_the_class_model(walk_exe, tmp_path):
    most, incomplete = 0, 0
    for w in workloads():
        sched, inc = check_walk(walk_exe, tmp_path, w)
        incomplete += inc
        if len(sched.starvations):
            most = max(most, int(np.diff(sched.recent_begin).max()))
    assert incomplete >= 2   # the overflowing stream, with and without the bulk step
    assert most > K


def test_the_ring_holds_what_every_other_generator_needs():
    most = 0
    for w in workloads()[:-2]:
        rb = capi.schedule_build(w.streams, w.events).recent_begin
        if len(rb) > 1:
            most = max(most, int(np.diff(rb).max()))
    assert 2 <= most <= K, most


def test_silence_heavy_streams_play_what_the_pcm_only_plan_refuses():
    w = silence_heavy_streams()
    sched = capi.schedule_build(w.streams, w.events)
    sv = sched.starvations
    recent = set(capi.flywheel_plan_batch(w.streams, sv, recent=sched.recent, recent_begin=sched.recent_begin).planned.tolist())
    plain = set(capi.flywheel_plan_batch(w.streams, sv).planned.tolist())
    assert plain <= recent
    assert len(recent - plain) >= 300, len(recent - plain)
    silent = [k for k in recent - plain if any(int(p["silence"]) for p in sched.recent_of(k))]
    assert len(silent) >= 200, len(silent)


def synthetic_records():
    """(spec, record, pieces) at every rate x depth x 1-10 channels: silence on, just after and well after a sample
    boundary, the 44.1 kHz cut that never ends, under 1 ms in all, fewer frames than the planes, more than 64
    descriptors, a piece outside the stream, attenuation changing between PCM runs."""
    out = []
    for rate in RATES:
        jps = abi.jiffies_per_sample(rate)
        for bits in DEPTHS:
            for ch in range(1, 11):
                sp = np.zeros(1, dtype=abi.STREAM_SPEC)[0]
                sp["sample_rate"], sp["bit_depth"], sp["channels"], sp["in_little_endian"] = rate, bits, ch, ch % 2
                sp["chunk_frames"], sp["out_fmt"], sp["total_frames"], sp["src_base"] = 1, abi.OUT_PACKED_BE, rate, 4096 * ch
                r = np.zeros(1, dtype=abi.STARVATION)[0]
                r["plays"], r["ramp"], r["attenuation"] = 1, 9000, 256
                att = 100 if bits == 16 else 256

                def pcm(at, n, a=256):
                    return (at, n, 0, a, 0)

                def sil(n):
                    return (0, n, 1, 256, 0)

                base = 37 * MS // jps * jps
                cases = [
                    [pcm(base - 3 * MS, 3 * MS), sil(5 * jps)],                                   # silence on a sample boundary
                    [pcm(base - 2 * MS + 100, 2 * MS), sil(3 * jps), pcm(base + 100, MS // 3)],   # just after
                    [pcm(base - MS, MS // 2 + 12345), sil(jps), pcm(base, MS // 2)],              # well after
                    [pcm(base - 2 * MS, 2 * MS), sil(2 * T // jps * jps)],                        # all silence (44.1 kHz: never ends)
                    [pcm(base, MS // 2), sil(jps)],                                               # under 1 ms
                    [pcm(base, T - 3 * jps), sil(jps // 2 + 1)],                                  # fewer frames than the planes
                    [p for i in range(T // jps) for p in (pcm(base + i * jps, jps), sil(jps))],  # 1-sample pieces: > 64 from 66 kHz up
                    [pcm(rate * jps - MS // 2, MS), sil(jps)],                                    # outside the stream
                    [pcm(base - MS, MS // 2, att), pcm(base - MS // 2, MS // 2, 256), pcm(base, MS // 3, att)],  # attenuation changes
                    [sil(jps), pcm(base - MS, MS + 7, att), sil(2 * jps), pcm(base + 7, 100)],
                ]
                for c in cases:
                    out.append((sp, r, np.array(c, dtype=abi.RECENT_AUDIO)))
    return out


def test_device_planner_equals_the_class_based_plan_recent(tmp_path):
    items = synthetic_records()
    for w in [W.elements(s, n_streams=24, attenuation=bool(s % 2)) for s in range(12)] + [w for _, w, _ in starved_streams()] + \
            [every_shape_streams(), silence_heavy_streams(), refusal_streams()] + edge_cases():
        sched = capi.schedule_build(w.streams, w.events)
        for k, r in enumerate(sched.starvations):
            items.append((w.streams[int(r["stream"])], r, sched.recent_of(k)))
    path = tmp_path / "records.bin"
    with open(path, "wb") as f:
        f.write(np.uint64(len(items)).tobytes())
        for sp, r, p in items:
            f.write(np.array([sp], dtype=abi.STREAM_SPEC).tobytes())
            f.write(np.array([r], dtype=abi.STARVATION).tobytes())
            f.write(np.uint32(len(p)).tobytes())
            f.write(np.ascontiguousarray(p, dtype=abi.RECENT_AUDIO).tobytes())
    exe = build(tmp_path, "recent_harness")
    r = subprocess.run([exe, "plan", str(path)], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-4000:]
    lines = r.stdout.strip().splitlines()
    assert lines[-1].startswith("checked %d " % len(items)), lines[-1]
    assert len(lines) == 1, "\n".join(lines[:20])
    planned = int(lines[-1].split()[-1])
    assert 3000 < planned < len(items)
    # every refusal the planner has is met: status by status, from the class-based planner
    seen = set()
    for sp, rec, p in items[:len(synthetic_records())]:
        try:
            capi.flywheel_plan_recent(sp, np.array([rec], dtype=abi.STARVATION), p)
            seen.add("ok")
        except capi.OhpError as e:
            seen.add(str(e).split(": ", 1)[-1].split(" (")[0][:40])
    assert len(seen) >= 7, seen


def test_header_exports_the_call_and_compiles_as_strict_c99(tmp_path):
    from test_abi import ROOT, declared_functions
    assert declared_functions("ohp_starvation_recent.h") == ["ohp_run_streams_device_flywheel_recent"]
    assert hasattr(capi.cuda_lib(), "ohp_run_streams_device_flywheel_recent")
    hdr = open(f"{ROOT}/include/ohp_starvation_recent.h").read()
    assert "#define OHP_DEVICE_RECENT_PIECES %du" % abi.DEVICE_RECENT_PIECES in hdr
    assert "#define OHP_RECENT_INCOMPLETE    0x%xu" % abi.RECENT_INCOMPLETE in hdr
    assert "#define OHP_FLYWHEEL_MAX_PREP_RECENT %du" % abi.FLYWHEEL_MAX_PREP_RECENT in open(f"{ROOT}/include/ohp_schedule.h").read()
    src = tmp_path / "one.c"
    src.write_text('#include "ohp_starvation_recent.h"\nint main(void) { return (int)sizeof(&ohp_run_streams_device_flywheel_recent) == 0; }\n')
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror", "-I" + f"{ROOT}/include", "-c", str(src), "-o",
                    str(tmp_path / "one.o")], check=True)
