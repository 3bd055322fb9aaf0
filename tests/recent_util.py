"""Shared inputs and helpers for the recent-audio tests (the device walk's pieces of recent audio and
ohp_run_streams_device_flywheel_recent): streams that starve with silence, a halt or a change of attenuation in their
last millisecond, and StartFlywheelRamp's cut."""
import os
import subprocess

import numpy as np

from ohpipeline_b200 import abi
from ohpipeline_b200 import workloads as W
from flywheel_util import DEPTHS, RATES

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MS = abi.JIFFIES_PER_MS
T = abi.FLYWHEEL_TRAINING_JIFFIES
K = abi.DEVICE_RECENT_PIECES


def silence_heavy_streams():
    """One 200 ms stream per rate x bit depth (1-8 channels in turn), each starving up to twelve times, 16 ms apart, with something
    at varying distances before each starvation: a MsgSilence of 1 sample to 2 ms (OHP_EV_INSERT_SILENCE), two of them
    with a message of PCM between, a MsgHalt, or (16-bit) a change of attenuation.  Every sixth stream has a second
    StarvationRamper (stage 3), every fifth starves once more where it ends.  One more stream inserts a 1-sample MsgSilence
    after every 2-frame message for 7 ms: its element's recent audio holds more pieces than the device walk keeps."""
    specs, events, slack = [], [], []
    k = 0
    for rate in RATES:
        jps = abi.jiffies_per_sample(rate)
        train = T // jps
        for bits in DEPTHS:
            ch = 1 + k % 8
            fb = ch * bits // 8
            chunk = W.max_chunk_frames(rate, bits, ch)
            total = rate * 2 // 10
            grid = chunk * jps
            ev, sil = [], 0   # sil: silence jiffies inserted so far (a stage's position counts them)
            stages = (1, 3) if k % 6 == 0 else (1,)

            def starve(at):
                for i, st in enumerate(stages):
                    ev.append((at + 7 * jps * i, st, abi.EV_STARVATION, 5 * MS))

            def silence(src, n):
                nonlocal sil
                ev.append((src, 0, abi.EV_INSERT_SILENCE, n * jps))
                sil += n * jps

            for j in range(12):
                b = -(-(12 + 16 * j) * MS // grid) * grid   # a message boundary of the source
                if b + 3 * grid >= total * jps:
                    break
                n = (1, 2, 5, train // 2, train - 1, train + 3, 2 * train)[(k * 7 + j) % 7]
                d = (0, 1, jps // 2, 100, MS // 3, MS - 1, MS + 3 * jps)[(k * 3 + j) % 7]
                kind = (k + j) % 5
                if kind == 3 and bits != 16:
                    kind = 0
                if kind in (0, 1):
                    silence(b, n)
                    starve(b + sil + d)
                elif kind == 2:
                    ev.append((b + sil + d // 2, 1, abi.EV_HALT, 0))
                    starve(b + sil + d)
                elif kind == 3:
                    ev.append((b + sil, 0, abi.EV_SET_ATTENUATION, (64, 100, 256, 1)[j % 4]))
                    starve(b + sil + d)
                else:
                    silence(b, n)
                    silence(b + grid, 1 + n // 3)
                    starve(b + grid + sil + d)
            if k % 5 == 0:
                starve(total * jps + sil)
            specs.append(W._spec(rate, bits, ch, bool(k % 2), chunk, total))
            events.append(ev)
            slack.append(sil // jps * fb)
            k += 1
    # the ring overflows: 2-frame messages, a 1-sample MsgSilence after each from 5 ms to 12 ms
    rate, jps = 48000, abi.jiffies_per_sample(48000)
    ev, sil = [], 0
    for f in range(240, 576, 2):
        ev.append((f * jps, 0, abi.EV_INSERT_SILENCE, jps))
        if f == 400:
            ev.append((f * jps + sil, 1, abi.EV_STARVATION, MS // 2))
        sil += jps
    ev.append((600 * jps + sil, 1, abi.EV_STARVATION, MS // 2))
    ev.append((700 * jps + sil, 1, abi.EV_STARVATION, MS // 2))
    specs.append(W._spec(rate, 16, 2, False, 2, rate * 2 // 100))
    events.append(ev)
    slack.append(sil // jps * 4)
    return W._finish("silence heavy", specs, events, seed=21, slack=slack)


def refusal_streams():
    """Starvations the recent-audio plan refuses, each in a stream beside starvations that play: the cut that never ends
    (44.1 kHz, 2 ms of silence right under it) and less than 1 ms since the last flywheel ramp emptied the recent audio.
    (The ring overflow is in silence_heavy_streams.)"""
    specs, events = [], []
    j44 = abi.jiffies_per_sample(44100)
    specs.append(W._spec(44100, 16, 2, False, 220, 44100 // 10))
    events.append([(20 * 220 * j44, 0, abi.EV_INSERT_SILENCE, 88 * j44), (20 * 220 * j44 + 88 * j44, 1, abi.EV_STARVATION, 5 * MS),
                   (60 * MS, 1, abi.EV_STARVATION, 5 * MS)])
    j48 = abi.jiffies_per_sample(48000)
    specs.append(W._spec(48000, 24, 2, True, 240, 48000 // 10))
    events.append([(30 * MS + 5 * j48, 1, abi.EV_STARVATION, 5 * MS), (30 * MS + 5 * j48 + MS // 2, 1, abi.EV_STARVATION, 5 * MS),
                   (70 * MS, 1, abi.EV_STARVATION, 5 * MS)])
    slack = [88 * 4, 0]
    return W._finish("refusals", specs, events, seed=22, slack=slack)


def cut(pieces):
    """StartFlywheelRamp's cut (ohp_flywheel_plan_recent): what is left of the pieces for the last T jiffies, as tuples;
    all of them where they add up to less."""
    p = [(int(x["pcm_jiffies"]), int(x["jiffies"]), int(x["silence"]), int(x["attenuation"])) for x in pieces]
    excess = sum(x[1] for x in p) - T
    while p and excess > 0:
        pcm, j, s, a = p[0]
        if j > excess:
            p[0] = (pcm if s else pcm + excess, j - excess, s, a)
            break
        excess -= j
        p.pop(0)
    return p


def build(tmp_path, name):
    exe = str(tmp_path / name)
    pkg = os.path.join(ROOT, "ohpipeline_b200")
    subprocess.run(["g++", "-std=c++17", "-O1", "-Wall", "-Wextra", "-o", exe, os.path.join(ROOT, "tests", "cpp", "recent_harness.cpp"),
                    "-L" + pkg, "-lohp_host", "-Wl,-rpath," + pkg], check=True)
    return exe


def host_walk(exe, tmp_path, w):
    """The walk with the recent audio kept, on the host -> [(status, records, counts, pieces)] with and without the bulk step."""
    src, dst = tmp_path / "walk_in.bin", tmp_path / "walk_out.bin"
    with open(src, "wb") as f:
        f.write(np.array([len(w.streams), len(w.events)], dtype=np.uint64).tobytes())
        f.write(np.ascontiguousarray(w.streams).tobytes())
        f.write(np.ascontiguousarray(w.events).tobytes())
    subprocess.run([exe, "walk", str(src), str(dst)], check=True, timeout=600)
    raw = np.fromfile(dst, dtype=np.uint8)
    ns, ne = len(w.streams), len(w.events)
    out, at = [], 0
    for _ in range(2):
        def take(dt, n):
            nonlocal at
            a = raw[at:at + n * dt.itemsize].view(dt)
            at += n * dt.itemsize
            return a
        rcs = take(np.dtype(np.uint32), ns)
        rec = take(abi.STARVATION, ne)
        cnt = take(np.dtype(np.uint32), ne)
        pcs = take(abi.RECENT_AUDIO, ne * K).reshape(ne, K)
        out.append((rcs, rec, cnt, pcs))
    assert at == raw.size
    return out
