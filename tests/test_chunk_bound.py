"""sched::stream_chunk_bound, the closed-form bound ohp_run_streams_device sizes each stream's descriptor region with,
against the exact playables of the walk the device compiles (run_stream<false>), through tests/cpp/chunk_bound_fuzz.cpp.
A stream with more playables than its bound takes the two-pass fallback at best (tests/test_gpu_region_overflow.py) and
fails at worst, so a change to the walk that adds playables must fail here, on the CPU, first:
  * a seeded fuzz of random streams: every op, four stages, caps from one sample up, codec reads, driver blocks, silence;
  * one stream per term of the bound, built to reach that term, with its slack (bound - exact) pinned: a slack below
    the term's share of the bound means the term is nearly reached, and any playable the walk gains shows up here.
CPU only."""
import os
import shutil
import struct
import subprocess

import numpy as np
import pytest

from ohpipeline_b200 import abi
from ohpipeline_b200 import workloads as W

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MS = abi.JIFFIES_PER_MS
RATE = 48000
JPS = abi.jiffies_per_sample(RATE)


@pytest.fixture(scope="module")
def harness(tmp_path_factory):
    if shutil.which("g++") is None:
        pytest.skip("no g++")
    exe = str(tmp_path_factory.mktemp("bound") / "chunk_bound_fuzz")
    r = subprocess.run(["g++", "-std=c++17", "-O2", "-Wall", "-Wextra", "-I" + os.path.join(ROOT, "include"), "-o", exe,
                        os.path.join(ROOT, "tests", "cpp", "chunk_bound_fuzz.cpp")], stdout=subprocess.PIPE,
                       stderr=subprocess.STDOUT, text=True)
    assert r.returncode == 0, r.stdout[-3000:]
    return exe


def test_bound_covers_random_streams(harness):
    """150 000 random streams (seed fixed): not one has more playables than its bound."""
    out = subprocess.run([harness, "fuzz", "20261022", "150000"], stdout=subprocess.PIPE, text=True, check=True,
                         timeout=600).stdout
    lines = out.strip().splitlines()
    summary = dict(zip(lines[-2].split()[::2], (int(x) for x in lines[-2].split()[1::2])))
    covered = dict(zip(lines[-1].split()[1::2], (int(x) for x in lines[-1].split()[2::2])))
    assert summary["violations"] == 0, out[-3000:]
    assert summary["accepted"] >= 100000, summary
    # every op, one-sample caps, codec reads, driver blocks and 9-32 channels, in thousands of accepted streams each
    for k in ["op%d" % i for i in range(1, 13)] + ["one_sample_cap", "codec", "driver", "wide"]:
        assert covered[k] >= 2000, (k, covered)


def spec(chunk, frames, bits=16, ch=2, driver=0, codec=0):
    s = W._spec(RATE, bits, ch, False, chunk, frames, driver_block_frames=driver)
    s["codec_read_frames"] = codec
    return s


def mid(frame, extra=11):
    """A position inside a sample, inside a message."""
    return frame * JPS + extra


def term_streams():
    """-> [(term, spec, events, the term's share of the bound, pinned slack)]"""
    out = []
    # messages the codec delivers: 3000 one-frame messages
    out.append(("messages", spec(1, 3000), [], 3000, 4))
    # behind a block-reading codec: 235-frame reads of 8-bit mono (each a whole message: 235 frames is at least
    # DecodedAudioAggregator's 5 ms - 7680 jiffies), cut from nothing (9216-frame chunks)
    out.append(("codec_reads", spec(9216, 235 * 100, bits=8, ch=1, codec=235), [], 101, 8))
    # one MsgSilence per event (one sample each, between messages)
    out.append(("silence", spec(480, 4800), [(k * 40 * JPS, 0, abi.EV_INSERT_SILENCE, JPS) for k in range(100)], 100, 4))
    # a stage holding messages to one sample: every frame a playable
    out.append(("stage_cap", spec(480, 4800), [(0, 1, abi.EV_MAX_MSG_JIFFIES, JPS)], 4801, 17))
    # per event, a split and a ramp that ends inside a message
    ev = [(mid(k * 600 + 37), 0, abi.EV_RAMP_DOWN if k % 2 == 0 else abi.EV_RAMP_UP, 150 * JPS + 13) for k in range(60)]
    out.append(("events", spec(100, 36000), ev, 120, 4))
    # ... where the call turns a ramp round (Muter::Mute during its ramp up, Unmute during its ramp down)
    ev = [(mid(k * 500 + 37, 11), 2, abi.EV_MUTER_MUTE if k % 2 == 0 else abi.EV_MUTER_UNMUTE, 300 * JPS + 5) for k in range(40)]
    out.append(("events_turned", spec(100, 20000), ev, 80, 4))
    # ... and starvations (a MsgHalt, the ramp up; the stage's 5 ms hold takes nothing from 100-frame messages)
    ev = [(mid(k * 1000 + 300, 7), 1, abi.EV_STARVATION, 150 * JPS + 3) for k in range(30)]
    out.append(("events_starvation", spec(100, 30000), ev, 60, 4))
    # two stages' ramps crossing: stage 1 ramps down and back up 20 times across stage 0's one long ramp down
    ev = [(0, 0, abi.EV_RAMP_DOWN, 48000 * JPS)]
    for k in range(20):
        ev += [((k * 2000 + 500) * JPS, 1, abi.EV_RAMP_DOWN, 100 * JPS), ((k * 2000 + 1000) * JPS, 1, abi.EV_RAMP_UP, 100 * JPS)]
    out.append(("stage_pairs", spec(480, 48000), ev, 40, 7))
    # a driver pulling 7-frame blocks
    out.append(("driver_blocks", spec(100, 3000, driver=7), [], 429, 9))
    return out


def test_bound_is_nearly_reached_term_by_term(harness, tmp_path):
    cases = term_streams()
    path = str(tmp_path / "terms.bin")
    with open(path, "wb") as f:
        for _, s, ev, _, _ in cases:
            w = W._finish("term", [s], [ev], seed=1)
            f.write(struct.pack("<II", 1, len(w.events)) + w.streams.tobytes() + w.events.tobytes())
    lines = subprocess.run([harness, "file", path], stdout=subprocess.PIPE, text=True, check=True).stdout.split()
    got = np.array(lines, dtype=np.int64).reshape(-1, 3)
    assert len(got) == len(cases)
    for (term, _, _, share, slack), (rc, exact, bound) in zip(cases, got):
        assert rc == 0, term
        assert exact <= bound, (term, exact, bound)
        assert bound - exact == slack, (term, exact, bound)
        assert slack * 4 < share, (term, slack, share)
