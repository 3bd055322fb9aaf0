"""Flywheel ramp generator, CPU side: the C oracle (oracle/ohp_oracle.c) and the host RampGenerator mirror
(ohp_flywheel_ramp_chunks) against
  * the known answers of the reference's own tests (Media/Tests/TestFlywheelRamper.cpp Test1-Test6),
  * the reference itself: FlywheelRamper.cpp + StarvationRamper.cpp linked into oracle/_ref (where it was built),
  * tests/golden/flywheel.npz, recorded from oracle/_ref by tests/golden/make_golden_flywheel.py."""
import os

import numpy as np
import pytest

from ohpipeline_b200 import abi, capi
from flywheel_util import (DEPTHS, RATES, SHAPES, accepted_shapes, every_shape_streams, shape_split, training_block,
                           train_frames)
from util import make_desc

GOLDEN = os.path.join(os.path.dirname(__file__), "golden", "flywheel.npz")

# TestFlywheelRamper.cpp:492-518
BURG_IN_1 = [111411200, 110362624, 108855296, 107937792, 108265472, 108462080, 108199936, 108527616, 107479040, 105578496,
             102170624, 97845248, 93257728, 88342528, 83034112, 77004800, 70844416, 63963136, 56885248, 51183616, 46399488,
             41418752, 36306944, 31457280, 27000832, 21430272, 15597568, 10027008, 4521984, 196608, -5439488, -10420224,
             -15335424, -20905984, -26083328, -32112640, -37552128, -42270720, -47251456, -52232192, -55836672, -59834368,
             -63700992, -67960832]
BURG_IN_2 = [80150528, 78249984, 75628544, 74055680, 73924608, 73924608, 73400320, 72744960, 72351744, 70189056, 67174400,
             64225280, 60948480, 57999360, 53673984, 49676288, 46596096, 42598400, 38731776, 36044800, 34144256, 31588352,
             28966912, 26673152, 24838144, 21889024, 18087936, 14548992, 9961472, 7208960, 3735552, 131072, -3342336,
             -7602176, -10616832, -14417920, -18546688, -21626880, -25296896, -28901376, -32505856, -35913728, -38731776,
             -42401792]


def libs(port):
    from oracle import pyoracle
    out = [port]
    if pyoracle.Ref.available():
        out.append(pyoracle.Ref())
    return out


def test_burg_known_answers(port):
    """SuiteFlywheelRamper::Test6 (TestFlywheelRamper.cpp:568-608)."""
    for lib in libs(port):
        for data, want in ((BURG_IN_1, [-16619, 8835, -374]), (BURG_IN_2, [-14748, 5235, 1360])):
            s = (np.array(data, dtype=np.int64) >> 16).astype(np.int16)
            assert list(lib.burgs_method(s, 3)) == want


def test_feedback_model_known_answers(port):
    """SuiteFlywheelRamper::Test1, Test2, Test5 (TestFlywheelRamper.cpp:111-262, 395-556)."""
    for lib in libs(port):
        v = [0x01000000, 0x02000000, 0x04000000, 0x08000000]
        got = lib.feedback_model(8, 1, 1, 1, v, v, 4)
        assert [int(x) for x in got] == [0x00aa0000, 0x00555400, 0x002b5200, 0x0016fa00]
        # Test2: scaling by coefficient / data / output format, two states
        table = {(1, 1, 1): (0x20000, 0x400), (2, 1, 1): (0x40000, 0x1000), (3, 1, 1): (0x80000, 0x4000),
                 (4, 1, 1): (0x100000, 0x10000), (1, 2, 1): (0x40000, 0x800), (1, 3, 1): (0x80000, 0x1000),
                 (1, 4, 1): (0x100000, 0x2000), (1, 1, 2): (0x10000, 0x200), (1, 1, 3): (0x8000, 0x100),
                 (1, 1, 4): (0x4000, 0x80), (2, 2, 2): (0x40000, 0x1000)}
        fixtures = _test2_inputs()
        for fmt, want in table.items():
            got = lib.feedback_model(fixtures["descale"], fmt[0], fmt[1], fmt[2], fixtures["coeffs"], fixtures["samples"], 2)
            assert tuple(int(x) for x in got) == want, fmt
        # Test5: an oscillator -- one coefficient of -1 (2.30) at position k gives period 2(k+1)
        for k, want in ((0, [0xc0000000, 0x40000000] * 3),
                        (1, [0, 0xc0000000, 0, 0x40000000, 0, 0xc0000000]),
                        (2, [0, 0, 0xc0000000, 0, 0, 0x40000000, 0, 0, 0xc0000000, 0, 0, 0x40000000])):
            coeffs = [0] * 6
            coeffs[k] = 0xc0000000
            got = lib.feedback_model(8, 2, 2, 2, coeffs, [0x40000000, 0, 0, 0, 0, 0], len(want))
            assert [int(x) & 0xffffffff for x in got] == want, k


def _test2_inputs():
    # TestFlywheelRamper.cpp:159-174: kDataInDescaleBits = 8, coeffs {0x01000000, 0}, samples {0x01000000, 0}
    return {"descale": 8, "coeffs": [0x01000000, 0], "samples": [0x01000000, 0]}


@pytest.mark.parametrize("kind", ["tone", "noise", "dc", "zero", "step", "max"])
def test_oracle_matches_linked_reference(port, ref, kind):
    """The real RampGenerator (FlywheelRamperManager::Ramp on its own thread, ProcessFragment, EndBlock) vs the port:
    generated audio, per-block ramp descriptors, final ramp value, and the ramped bytes a driver would read."""
    for n, (rate, ch, bits) in enumerate(SHAPES):
        for start in (abi.RAMP_MAX, 9000, 1, 0):
            training = training_block(rate, ch, kind, seed=100 + n)
            rc, raw, ramped, descs, info, final = ref.flywheel(rate, ch, bits, start, training)
            assert rc == 0
            job = capi.flywheel_job(rate, ch, bits)
            rc2, out = port.flywheel(job, training, raw.size)
            assert rc2 == 0
            assert np.array_equal(out, raw), (rate, ch, bits, kind)
            pd, pfinal = port.flywheel_ramp_chunks(job, start, 0, 0)
            assert np.array_equal(pd, descs), (rate, ch, bits, start)
            assert pfinal == final
            rc3, pr = port.process_chunks(pd, out, out.size)
            assert rc3 == 0 and np.array_equal(pr, ramped)


def test_host_ramp_chunks_match_oracle(port):
    """ohp_flywheel_ramp_chunks (product, host message model) vs the oracle's RampGenerator::EndBlock restatement."""
    for rate, ch, bits in SHAPES:
        job = capi.flywheel_job(rate, ch, bits, src_off=4096, dst_off=123)
        for start in (abi.RAMP_MAX, 16383, 12345, 4097, 100, 1, 0):
            want, wfinal = port.flywheel_ramp_chunks(job, start, 4096, 123)
            got, gfinal = capi.flywheel_ramp_chunks(job, start, 4096, 123)
            assert np.array_equal(got, want), (rate, ch, bits, start)
            assert gfinal == wfinal
            assert int(abi.chunk_out_bytes(got).sum()) == int(job["out_frames"][0]) * ch * bits // 8


def test_validate_accepts_exactly_what_the_oracle_plays(port):
    """ohp_flywheel_validate (and the kernel, which shares check_job) against the oracle's own refusals: every rate x depth
    x 0-10 channels, a training block a frame short or long, and 0 or 1 frames of output."""
    n = accepted = 0
    for rate in RATES:
        for bits in DEPTHS:
            for ch in range(0, 11):
                base = capi.flywheel_job(rate, ch, bits)
                variants = [base]
                for field, value in (("train_frames", train_frames(rate) - 1), ("train_frames", train_frames(rate) + 1),
                                     ("out_frames", 0), ("out_frames", 1)):
                    v = base.copy()
                    v[field] = value
                    variants.append(v)
                for job in variants:
                    in_bytes = int(job["train_frames"][0]) * 4 * ch
                    out_bytes = int(job["out_frames"][0]) * ch * bits // 8
                    ok = capi.flywheel_validate(job, in_bytes, out_bytes)[0] == abi.OK
                    rc, _ = port.flywheel(job, np.zeros(max(in_bytes, 1), np.uint8)[:in_bytes], out_bytes)
                    assert ok == (rc == 0), (rate, ch, bits, job)
                    n += 1
                    accepted += ok
    assert n == 18 * 4 * 11 * 5
    # 550 shapes as StarvationRamper asks for them, and the same shapes with 0 or 1 frames of output
    assert accepted == 3 * 550


def test_host_ramp_chunks_match_oracle_at_every_shape(port):
    """test_host_ramp_chunks_match_oracle at every shape the flywheel plays: 550 shapes x 7 start values."""
    for rate, ch, bits in accepted_shapes():
        job = capi.flywheel_job(rate, ch, bits, src_off=4096, dst_off=123)
        for start in (abi.RAMP_MAX, 16383, 12345, 4097, 100, 1, 0):
            want, wfinal = port.flywheel_ramp_chunks(job, start, 4096, 123)
            assert want is not None, (rate, ch, bits, start)
            got, gfinal = capi.flywheel_ramp_chunks(job, start, 4096, 123)
            assert np.array_equal(got, want), (rate, ch, bits, start)
            assert gfinal == wfinal, (rate, ch, bits, start)
            assert int(abi.chunk_out_bytes(got).sum()) == int(job["out_frames"][0]) * ch * bits // 8


def test_every_shape_streams_records_and_plan(port):
    """flywheel_util.every_shape_streams(): the class-free walk records what the class model records, field by field; every
    record plays; the host planner plans exactly the records at accepted shapes, two per shape, splits training blocks
    across messages, and plans the oracle's ramped blocks."""
    w = every_shape_streams()
    assert len(w.streams) == 576
    want = capi.schedule_build(w.streams, w.events).starvations
    got = capi.schedule_build(w.streams, w.events, walk=True).starvations
    assert len(got) == len(want) == 1152
    for f in abi.STARVATION.names:
        assert np.array_equal(got[f], want[f]), f
    assert np.all(want["plays"] == 1)
    b = capi.flywheel_plan_batch(w.streams, want)
    assert len(b.planned) == len(b.jobs) == 1100
    shape = lambda k: tuple(int(w.streams[int(want["stream"][k])][f]) for f in ("sample_rate", "channels", "bit_depth"))  # noqa: E731
    accepted, refused = shape_split()
    planned = [shape(int(k)) for k in b.planned]
    assert sorted(planned) == sorted(accepted * 2)
    unplanned = sorted(set(range(len(want))) - set(int(k) for k in b.planned))
    assert sorted(shape(k) for k in unplanned) == sorted(refused * 2)
    assert len(b.prep) == 2464
    # the blocks the host planner plans are the oracle's RampGenerator blocks, job by job
    blocks = []
    for i, k in enumerate(b.planned):
        d, _ = port.flywheel_ramp_chunks(b.jobs[i], int(want["ramp"][k]), int(b.jobs[i]["dst_off"]), int(b.out_off[i]))
        assert d is not None, shape(int(k))
        blocks.append(d)
    assert np.array_equal(np.concatenate(blocks), b.blocks)


def test_golden_flywheel_vectors(port):
    g = np.load(GOLDEN)
    jobs, starts = g["jobs"], g["starts"]
    for k in range(len(jobs)):
        job = jobs[k:k + 1].copy()
        training = g["training_%d" % k]
        rc, out = port.flywheel(job, training, int(g["raw_%d" % k].size))
        assert rc == 0
        assert np.array_equal(out, g["raw_%d" % k]), k
        descs, final = capi.flywheel_ramp_chunks(job, int(starts[k]), 0, 0)
        assert np.array_equal(descs, g["descs_%d" % k]), k
        assert final == int(g["finals"][k])
        rc, ramped = port.process_chunks(descs, out, out.size)
        assert rc == 0 and np.array_equal(ramped, g["ramped_%d" % k]), k


def test_validate_refuses_what_the_reference_cannot_hold():
    ok = capi.flywheel_job(48000, 2, 24)
    assert capi.flywheel_validate(ok, 1 << 20, 1 << 20) == (abi.OK, 0)
    for field, value in (("sample_rate", 12345), ("bit_depth", 20), ("channels", 0), ("channels", 9), ("train_frames", 47)):
        bad = ok.copy()
        bad[field] = value
        assert capi.flywheel_validate(bad, 1 << 20, 1 << 20)[0] == abi.E_INVALID_DESC, field
    # 384 kHz x 8 channels x 32 bit: one 1 ms block (12288 B) overruns RampGenerator's 6144-byte buffer
    assert capi.flywheel_validate(capi.flywheel_job(384000, 8, 32), 1 << 20, 1 << 20)[0] == abi.E_INVALID_DESC
    # 384 kHz x 6 channels: the training block (9216 B) overruns FlywheelInput's 7680-byte buffer
    assert capi.flywheel_validate(capi.flywheel_job(384000, 6, 8), 1 << 20, 1 << 20)[0] == abi.E_INVALID_DESC
    assert capi.flywheel_validate(ok, 100, 1 << 20)[0] == abi.E_OUT_OF_RANGE
    assert capi.flywheel_validate(ok, 1 << 20, 100)[0] == abi.E_OUT_OF_RANGE
    both = np.concatenate([ok, capi.flywheel_job(48000, 2, 20)])
    assert capi.flywheel_validate(both, 1 << 20, 1 << 20) == (abi.E_INVALID_DESC, 1)


def test_planar_sink_matches_the_real_flywheel_input(port, ref):
    """FlywheelInput::Prepare (StarvationRamper.cpp:90-186) over real messages vs the oracle's OHP_OUT_PLANAR32_BE sink:
    the last millisecond of a stream as 1-3 messages of any depth / endianness, plus leading silence."""
    rng = np.random.default_rng(5)
    for rate, ch, bits in [(44100, 2, 16), (48000, 2, 24), (96000, 6, 32), (192000, 8, 24), (48000, 1, 8), (88200, 3, 32)]:
        for le in (False, True):
            for with_silence in (False, True):
                T = train_frames(rate)
                fb = ch * bits // 8
                pieces = sorted(set(int(x) for x in rng.integers(1, T, 2))) + [T]
                wire = rng.integers(0, 256, T * fb, dtype=np.uint8)
                descs = []
                first = 0
                for k, upto in enumerate(pieces):
                    silence = with_silence and k == 0
                    d = make_desc(src_off=0 if silence else first * fb, dst_off=first * 4, bytes=(upto - first) * fb,
                                  bit_depth=bits, channels=ch, out_fmt=abi.OUT_PLANAR32_BE, aux=T,
                                  flags=(abi.F_SILENCE if silence else (abi.F_IN_LITTLE_ENDIAN if le and bits > 8 else 0)))
                    descs.append(d)
                    first = upto
                descs = np.concatenate(descs)
                rc, want = ref.flywheel_input(descs, wire, rate, T * abi.jiffies_per_sample(rate))
                assert rc == 0 and want.size == T * 4 * ch
                rc, got = port.process_chunks(descs, wire, want.size)
                assert rc == 0
                assert np.array_equal(got, want), (rate, ch, bits, le, with_silence)


def test_burg_denominator_that_wraps_to_zero(port, ref, tmp_path):
    """FlywheelRamper::BurgsMethod divides by a 32-bit sum of squares that is left to wrap (FlywheelRamper.cpp:252-282).
    Wrapped to exactly zero under a numerator that is not, the reference takes an integer division by zero and dies (SIGFPE);
    with 8-bit audio, whose squares are multiples of 2^16, that is about one sum in 2^16 -- a random schedule found one
    (profiles/starvation_fuzz.py, seed 100226, stream 21, its second starvation).  The port, and the kernel after it, leave
    that coefficient at 0 (oracle/ohp_oracle.c, csrc/ohp_flywheel_kernels.cuh): a documented deviation, since there is no
    output of the reference to be equal to.  Here: the reference dies on that training block in a process of its own, the
    port generates audio, and the same stream's first starvation plays the same in both."""
    import subprocess
    import sys
    from ohpipeline_b200 import workloads
    w = workloads.elements(100226, n_streams=24)
    inp = port.fill_pcm(w.in_bytes, w.seed)
    st = w.streams[21:22].copy()
    ev = w.events[int(st[0]["first_event"]):int(st[0]["first_event"]) + int(st[0]["num_events"])].copy()
    st[0]["first_event"] = 0
    assert (int(st[0]["sample_rate"]), int(st[0]["bit_depth"]), int(st[0]["channels"])) == (48000, 8, 2)
    sv = capi.schedule_build(st, ev).starvations
    assert len(sv) == 2 and list(sv["plays"]) == [1, 1]
    blocks = []
    for k in range(2):
        prep, job, _ = capi.flywheel_plan(st, sv[k:k + 1])
        rc, training = port.process_chunks(prep, inp, int(job["train_frames"][0]) * 4 * 2)
        assert rc == 0
        rc, out = port.flywheel(job, training, int(job["out_frames"][0]) * 2)
        assert rc == 0 and out.any()
        blocks.append((training, out, int(sv["ramp"][k])))
    # the first starvation: reference and port agree
    rc, raw, *_ = ref.flywheel(48000, 2, 8, blocks[0][2], blocks[0][0])
    assert rc == 0 and np.array_equal(raw, blocks[0][1])
    # the second: the reference does not survive its own arithmetic
    path = tmp_path / "training.npy"
    np.save(path, blocks[1][0])
    code = ("import sys, numpy as np; sys.path.insert(0, %r); from oracle import pyoracle;"
            "print(pyoracle.Ref().flywheel(48000, 2, 8, %d, np.load(%r))[0])"
            % (os.path.dirname(os.path.dirname(os.path.abspath(__file__))), blocks[1][2], str(path)))
    r = subprocess.run([sys.executable, "-c", code], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=120)
    assert r.returncode == -8, (r.returncode, r.stdout, r.stderr[-500:])   # SIGFPE
