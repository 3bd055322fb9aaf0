"""Shared inputs for the flywheel tests: training blocks in FlywheelInput's layout (planar, 32-bit big-endian)."""
import numpy as np

from ohpipeline_b200 import abi

# (rate, channels, bit depth) accepted by RampGenerator's fixed buffers (ohp_flywheel_validate)
SHAPES = [(44100, 2, 16), (48000, 2, 24), (192000, 2, 24), (96000, 6, 32), (384000, 2, 8), (176400, 1, 16),
          (88200, 8, 24), (352800, 2, 32), (32000, 3, 16), (8000, 2, 8)]

RATES = list(abi.PCM_SAMPLE_RATES)  # the 18 PCM rates Jiffies::PerSample takes
DEPTHS = (8, 16, 24, 32)


def train_frames(rate):
    return abi.FLYWHEEL_TRAINING_JIFFIES // abi.jiffies_per_sample(rate)


def block_frames(rate):
    """Frames in one of RampGenerator's 1 ms blocks (OHP_FLYWHEEL_BLOCK_JIFFIES)."""
    return abi.JIFFIES_PER_MS // abi.jiffies_per_sample(rate)


def shape_split():
    """(accepted, refused): every (rate, channels 1-8, bit depth) StarvationRamper can meet, split by
    ohp_flywheel_validate.  Only 352.8 and 384 kHz are refused: there a training block of many channels overruns
    FlywheelInput's fixed buffer, or a 1 ms block RampGenerator's."""
    from ohpipeline_b200 import capi
    accepted, refused = [], []
    for rate in RATES:
        for bits in DEPTHS:
            for ch in range(1, 9):
                ok = capi.flywheel_validate(capi.flywheel_job(rate, ch, bits), 1 << 30, 1 << 30)[0] == abi.OK
                (accepted if ok else refused).append((rate, ch, bits))
    assert len(accepted) == 550 and len(refused) == 26
    assert all(rate in (352800, 384000) for rate, _, _ in refused)
    return accepted, refused


def accepted_shapes():
    """Every (rate, channels, bit depth) the flywheel plays: 550 of the 576 with 1-8 channels."""
    return shape_split()[0]


def training_block(rate, channels, kind, seed):
    """kind: 'tone' (what the predictor is for), 'noise' (full-range: every accumulator wraps), 'dc', 'zero',
    'step', 'max'."""
    rng = np.random.default_rng(seed)
    t = np.arange(train_frames(rate))
    planes = []
    for c in range(channels):
        if kind == "tone":
            x = 0.4 * np.sin(2 * np.pi * (220.0 * (c + 1)) * t / rate + 0.3 * c) * 2**31 + rng.normal(0, 2**18, t.size)
        elif kind == "noise":
            x = rng.integers(-2**31, 2**31, t.size).astype(np.float64)
        elif kind == "dc":
            x = np.full(t.size, (c + 1) * 1.1e8)
        elif kind == "zero":
            x = np.zeros(t.size)
        elif kind == "step":
            x = np.where(t < t.size // 2, -1.5e9, 1.5e9)
        else:
            x = np.where(t % 2 == 0, 2.0**31 - 1, -2.0**31)
        planes.append(np.clip(x, -2**31, 2**31 - 1).astype(np.int64).astype(np.int32).astype(">i4").view(np.uint8))
    return np.concatenate(planes)


def starved_streams():
    """Streams whose StarvationRamper stage (stage 1) starves at positions aligned to nothing: twice (the second time 17 ms
    into the 50 ms ramp up from the first), behind a Ramper's ramp, an attenuation, a MsgHalt.  -> [(name, Workload, pcm seed)]
    tests/golden/starvation_flywheel.npz holds what the reference's own element object plays for each."""
    from ohpipeline_b200 import workloads
    MS = abi.JIFFIES_PER_MS
    out = []
    # at 37 ms + 400 jiffies the 44.1 and 88.2 kHz streams are less than 128 jiffies past a sample boundary, at 37 ms + 12345
    # the 176.4 and 352.8 kHz ones: the reference's training block is a frame too long there (ohp_flywheel_plan)
    for rate, ch, bits, le, off in [(44100, 2, 16, True, 400), (48000, 2, 24, False, 12345), (192000, 2, 24, True, 12345),
                                    (96000, 6, 32, False, 12345), (176400, 1, 16, False, 12345), (88200, 8, 24, True, 400),
                                    (352800, 2, 8, False, 12345)]:
        first = 37 * MS + off
        second = first + 17 * MS + 777
        spec = workloads._spec(rate, bits, ch, le, workloads.max_chunk_frames(rate, bits, ch), rate * 3 // 10)
        events = [(0, 0, abi.EV_RAMPER_STREAM, 40 * MS), (first, 1, abi.EV_STARVATION, 50 * MS), (second, 1, abi.EV_STARVATION, 50 * MS)]
        out.append(("%d_%d_%d" % (rate, ch, bits), workloads._finish("starved", [spec], [events], seed=77), 1000 + rate + ch))
    spec = workloads._spec(44100, 16, 2, False, workloads.max_chunk_frames(44100, 16, 2), 44100 * 2 // 10)
    events = [(10 * MS, 0, abi.EV_SET_ATTENUATION, 100), (60 * MS + 4321, 1, abi.EV_STARVATION, 50 * MS)]
    out.append(("attenuated", workloads._finish("starved", [spec], [events], seed=78), 555))
    spec = workloads._spec(96000, 24, 2, False, 480, 96000 * 2 // 10)
    events = [(12 * MS + MS // 2, 1, abi.EV_HALT, 0), (13 * MS, 1, abi.EV_STARVATION, 50 * MS)]
    out.append(("after_halt", workloads._finish("starved", [spec], [events], seed=79), 3))
    return out


def every_shape_streams():
    """One 120 ms stream per rate x bit depth x 1-8 channels (576), each starved twice behind a Ramper's ramp: first at
    37 ms on a sample boundary, 100 jiffies after one or at 37 ms + 12345 jiffies (in turn, so every rate x depth meets all
    three, and the 44.1 kHz family a training block a frame too long), then again 17 ms + 777 jiffies later, inside the
    50 ms ramp up.  Wire endianness alternates; every fourth 16-bit stream is attenuated.  Two records per stream, 1152 in
    all, every one of which plays; the 52 at the 26 refused shapes plan nothing."""
    from ohpipeline_b200 import workloads
    MS = abi.JIFFIES_PER_MS
    specs, events = [], []
    k = 0
    for rate in RATES:
        jps = abi.jiffies_per_sample(rate)
        on_sample = 37 * MS // jps * jps
        for bits in DEPTHS:
            for ch in range(1, 9):
                first = (on_sample, on_sample + 100, 37 * MS + 12345)[k % 3]
                second = first + 17 * MS + 777
                specs.append(workloads._spec(rate, bits, ch, bool(k % 2), workloads.max_chunk_frames(rate, bits, ch),
                                             rate * 12 // 100))
                ev = [(0, 0, abi.EV_RAMPER_STREAM, 40 * MS), (first, 1, abi.EV_STARVATION, 50 * MS),
                      (second, 1, abi.EV_STARVATION, 50 * MS)]
                if bits == 16 and k % 4 == 1:
                    ev.append((10 * MS, 0, abi.EV_SET_ATTENUATION, 100))
                events.append(ev)
                k += 1
    return workloads._finish("every shape", specs, events, seed=11)
