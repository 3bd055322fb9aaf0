"""Flywheel ramp generator on the GPU (ohp_flywheel_device) against the C oracle, the reference's golden vectors
(tests/golden/flywheel.npz, recorded from the real RampGenerator) and, end to end, the whole starvation sequence
FlywheelInput (planar sink) -> flywheel kernel -> RampGenerator's ramped blocks -> ramp + convert kernel."""
import os

import numpy as np
import pytest

from ohpipeline_b200 import abi, capi
from flywheel_util import RATES, SHAPES, accepted_shapes, block_frames, shape_split, training_block, train_frames
from util import make_desc

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(__file__), "golden", "flywheel.npz")
KINDS = ["tone", "noise", "dc", "zero", "step", "max"]


def run_jobs(ctx, jobs, inp, out_bytes, fill=0x5A):
    out, err = launch(ctx, jobs, inp, out_bytes, fill)
    if err is not None:
        raise err
    return out


def launch(ctx, jobs, inp, out_bytes, fill):
    """One flywheel launch -> (output, the OhpError it raised or None); the output is read back either way."""
    import torch
    d_jobs = torch.from_numpy(jobs.view(np.uint8).copy()).cuda()
    d_in = torch.from_numpy(np.ascontiguousarray(inp)).cuda()
    d_out = torch.full((max(out_bytes, 1),), fill, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    err = None
    try:
        ctx.flywheel_device(d_jobs.data_ptr(), len(jobs), d_in.data_ptr(), int(inp.size), d_out.data_ptr(), out_bytes)
        ctx.sync()
    except capi.OhpError as e:
        err = e
    return d_out.cpu().numpy()[:out_bytes], err


def out_len(job):
    return int(job["out_frames"]) * int(job["channels"]) * (int(job["bit_depth"]) // 8)


def covered(jobs, out_bytes):
    """The output bytes some job writes."""
    mask = np.zeros(out_bytes, dtype=bool)
    for j in jobs:
        mask[int(j["dst_off"]):int(j["dst_off"]) + out_len(j)] = True
    return mask


def assert_jobs_match(got, want, jobs, mask, what):
    """Every byte a job writes is the oracle's; naming the job of the first one that is not."""
    bad = np.nonzero((got != want) & mask)[0]
    if bad.size:
        i = int(bad[0])
        k = next(k for k, j in enumerate(jobs) if int(j["dst_off"]) <= i < int(j["dst_off"]) + out_len(j))
        raise AssertionError("%s: byte %d differs (got %#x want %#x) in job %d: %s, %d bytes differ in all"
                             % (what, i, got[i], want[i], k, jobs[k], bad.size))


def batch(kinds, shapes, seed, dst_align=1):
    """One job per (kind, shape): training blocks and outputs laid out back to back (dst optionally misaligned)."""
    jobs, blocks = [], []
    src = dst = 0
    for n, (kind, (rate, ch, bits)) in enumerate((k, s) for k in kinds for s in shapes):
        j = capi.flywheel_job(rate, ch, bits, src_off=src, dst_off=dst)
        t = training_block(rate, ch, kind, seed + n)
        jobs.append(j)
        blocks.append(t)
        src += t.size
        dst += int(j["out_frames"][0]) * ch * bits // 8
        if dst_align > 1:
            dst = (dst + dst_align - 1) // dst_align * dst_align
        else:
            dst += n % 3  # ragged: exercises the byte-store path
    return np.concatenate(jobs), np.concatenate(blocks), dst + 16


@pytest.mark.parametrize("kind", ["tone", "noise", "dc", "zero", "step", "max"])
def test_flywheel_kernel_matches_oracle(ctx, port, kind):
    jobs, inp, out_bytes = batch([kind], SHAPES, seed=300)
    assert capi.flywheel_validate(jobs, inp.size, out_bytes)[0] == abi.OK
    rc, want = port.flywheel(jobs, inp, out_bytes)
    assert rc == 0
    got = run_jobs(ctx, jobs, inp, out_bytes, fill=0)
    if not np.array_equal(got, want):
        i = int(np.nonzero(got != want)[0][0])
        k = int(np.searchsorted(jobs["dst_off"], i, side="right") - 1)
        raise AssertionError("byte %d differs (got %#x want %#x) in job %d: %s" % (i, got[i], want[i], k, jobs[k]))


def test_flywheel_kernel_aligned_destinations_and_many_jobs(ctx, port):
    """Word-store path (4-byte aligned destinations), more jobs than one wave of warps."""
    jobs, inp, out_bytes = batch(["tone", "noise", "step"] * 40, SHAPES, seed=500, dst_align=16)
    assert len(jobs) == 1200
    rc, want = port.flywheel(jobs, inp, out_bytes)
    assert rc == 0
    got = run_jobs(ctx, jobs, inp, out_bytes, fill=0)
    assert np.array_equal(got, want)


def every_shape_batch(seed):
    """Every accepted shape x every training-block kind, in an order shuffled with `seed` (so the warps of one CTA hold
    different shapes).  Destinations alternate between 16-byte aligned (the word stores, the tail loop after them, and
    the switch to byte stores inside a job whose tiles are not whole words) and ragged (the byte stores), with a gap of
    1-16 bytes before each; some training blocks start at offsets that are not a multiple of 4."""
    rng = np.random.default_rng(seed)
    work = [(kind, shape) for kind in KINDS for shape in accepted_shapes()]
    jobs, blocks = [], []
    src = dst = 0
    for n, i in enumerate(rng.permutation(len(work))):
        kind, (rate, ch, bits) = work[int(i)]
        if n % 5 == 2:
            pad = 1 + n % 3
            blocks.append(np.full(pad, 0xC3, dtype=np.uint8))
            src += pad
        if n % 2 == 0:
            dst = (dst + 16) // 16 * 16
        else:
            dst += 1 + n % 3
            dst += dst % 4 == 0
        j = capi.flywheel_job(rate, ch, bits, src_off=src, dst_off=dst)
        t = training_block(rate, ch, kind, seed + int(i))
        jobs.append(j)
        blocks.append(t)
        src += t.size
        dst += out_len(j[0])
    return np.concatenate(jobs), np.concatenate(blocks), dst + 16


def test_flywheel_kernel_at_every_accepted_shape(ctx, port):
    """550 shapes x 6 kinds of training block in one launch: the eight rates whose 1 ms block is shorter than a 32-frame
    tile, and the 80 shapes (odd channel counts at 8 or 24 bits) whose tiles end inside a 4-byte word."""
    fill = 0x5A
    jobs, inp, out_bytes = every_shape_batch(seed=900)
    assert len(jobs) == 550 * len(KINDS)
    assert np.any(jobs["src_off"] % 4 != 0)
    assert np.sum(jobs["dst_off"] % 16 == 0) >= len(jobs) // 2 and np.sum(jobs["dst_off"] % 4 != 0) == len(jobs) // 2
    assert capi.flywheel_validate(jobs, inp.size, out_bytes)[0] == abi.OK
    rc, want = port.flywheel(jobs, inp, out_bytes)
    assert rc == 0
    got, err = launch(ctx, jobs, inp, out_bytes, fill)
    assert err is None, err
    mask = covered(jobs, out_bytes)
    assert_jobs_match(got, want, jobs, mask, "every shape")
    assert np.all(got[~mask] == fill)


def test_flywheel_kernel_output_lengths_at_tile_and_block_edges(ctx, port):
    """Any out_frames (StarvationRamper always asks for 20 ms, the API takes any length): 1, 2, a tile -1 / 0 / +1, a
    1 ms block -1 / 0 / +1, two blocks + 1 and 20 ms, at every rate, 1 and 3 channels x 8 and 24 bits, destinations
    4-byte aligned."""
    fill = 0x5A
    jobs, blocks = [], []
    src = dst = 0
    for rate in RATES:
        b = block_frames(rate)
        lengths = sorted({1, 2, 31, 32, 33, b - 1, b, b + 1, 2 * b + 1, abi.FLYWHEEL_RAMP_JIFFIES // abi.jiffies_per_sample(rate)})
        for ch in (1, 3):
            for bits in (8, 24):
                for frames in lengths:
                    j = capi.flywheel_job(rate, ch, bits, src_off=src, dst_off=dst)
                    j["out_frames"] = frames
                    t = training_block(rate, ch, "tone", len(jobs))
                    jobs.append(j)
                    blocks.append(t)
                    src += t.size
                    dst = (dst + out_len(j[0]) + 4) // 4 * 4
    jobs, inp, out_bytes = np.concatenate(jobs), np.concatenate(blocks), dst
    assert capi.flywheel_validate(jobs, inp.size, out_bytes)[0] == abi.OK
    rc, want = port.flywheel(jobs, inp, out_bytes)
    assert rc == 0
    got, err = launch(ctx, jobs, inp, out_bytes, fill)
    assert err is None, err
    mask = covered(jobs, out_bytes)
    assert_jobs_match(got, want, jobs, mask, "output lengths")
    assert np.all(got[~mask] == fill)


@pytest.mark.parametrize("index", range(26))
def test_refused_shape_among_valid_jobs(ctx, port, index):
    """Each of the 26 shapes ohp_flywheel_validate refuses, as one job among seven valid ones: the launch fails with
    E_INVALID_DESC naming that job, its destination keeps the fill, every other job writes the oracle's bytes, and the
    context runs the valid jobs cleanly afterwards.  (With several refused jobs the message names whichever warp got
    there first, so there is one per launch.)"""
    fill = 0x5A
    accepted, refused = shape_split()
    pos = index % 8
    shapes = [accepted[(37 * index + 79 * i) % len(accepted)] for i in range(7)]
    shapes.insert(pos, refused[index])
    jobs, blocks = [], []
    src = dst = 0
    for n, (rate, ch, bits) in enumerate(shapes):
        j = capi.flywheel_job(rate, ch, bits, src_off=src, dst_off=dst)
        t = training_block(rate, ch, KINDS[n % len(KINDS)], 40 * index + n)
        jobs.append(j)
        blocks.append(t)
        src += t.size
        dst = (dst + out_len(j[0]) + 16) // 16 * 16
    jobs, inp, out_bytes = np.concatenate(jobs), np.concatenate(blocks), dst
    assert capi.flywheel_validate(jobs, inp.size, out_bytes) == (abi.E_INVALID_DESC, pos)
    valid = np.delete(jobs, pos)
    rc, want = port.flywheel(valid, inp, out_bytes)
    assert rc == 0
    got, err = launch(ctx, jobs, inp, out_bytes, fill)
    assert err is not None and err.status == abi.E_INVALID_DESC, err
    assert "flywheel job %d (invalid)" % pos in str(err), str(err)
    mask = covered(valid, out_bytes)
    assert_jobs_match(got, want, valid, mask, "refused %s" % (refused[index],))
    assert np.all(got[~mask] == fill)  # the refused job's destination and the gaps
    again, err = launch(ctx, valid, inp, out_bytes, fill)
    assert err is None, err
    assert np.array_equal(again, got)


def test_flywheel_kernel_reproduces_reference_golden_vectors(ctx):
    g = np.load(GOLDEN)
    for k in range(len(g["jobs"])):
        job = g["jobs"][k:k + 1].copy()
        raw = g["raw_%d" % k]
        got = run_jobs(ctx, job, g["training_%d" % k], raw.size)
        assert np.array_equal(got, raw), "case %d: generated audio differs from the reference's RampGenerator" % k


def test_whole_starvation_sequence_on_the_gpu(ctx, port):
    """recent audio (wire format) --PLANAR32 sink--> training block --flywheel--> generated audio --ramped blocks-->
    what the driver reads; every stage on the device, every stage checked against the oracle chain."""
    import torch
    rng = np.random.default_rng(77)
    cases = [(48000, 2, 24, True, abi.RAMP_MAX), (44100, 2, 16, False, 7000), (192000, 2, 24, False, abi.RAMP_MAX),
             (96000, 6, 32, True, abi.RAMP_MAX), (88200, 4, 8, False, 300)]
    for rate, ch, bits, le, start in cases:
        T = train_frames(rate)
        B = bits // 8
        # 1. the last 1 ms of audio as two messages (a split lands mid-block), unramped (FlywheelPlayableCreator clears ramps)
        t = np.arange(T)
        pcm = np.zeros((T, ch), dtype=np.int64)
        for c in range(ch):
            pcm[:, c] = (0.5 * np.sin(2 * np.pi * 300.0 * (c + 1) * t / rate) * 2 ** (bits - 1)).astype(np.int64)
        pcm += rng.integers(-3, 4, pcm.shape)
        pcm = np.clip(pcm, -2 ** (bits - 1), 2 ** (bits - 1) - 1)
        be = np.zeros((T, ch, B), dtype=np.uint8)
        for b in range(B):
            be[:, :, b] = (pcm >> (8 * (B - 1 - b))) & 0xff
        wire = (be[:, :, ::-1] if le else be).reshape(-1).copy()
        cut = (T // 3) * ch * B
        flags = abi.F_IN_LITTLE_ENDIAN if (le and B > 1) else 0
        d1 = make_desc(src_off=0, dst_off=0, bytes=cut, bit_depth=bits, channels=ch, flags=flags,
                       out_fmt=abi.OUT_PLANAR32_BE, aux=T)
        d2 = make_desc(src_off=cut, dst_off=(T // 3) * 4, bytes=wire.size - cut, bit_depth=bits, channels=ch, flags=flags,
                       out_fmt=abi.OUT_PLANAR32_BE, aux=T)
        prep = np.concatenate([d1, d2])
        train_bytes = T * 4 * ch
        rc, want_train = port.process_chunks(prep, wire, train_bytes)
        assert rc == 0
        # 2. the flywheel job and RampGenerator's ramped blocks
        job = capi.flywheel_job(rate, ch, bits)
        gen_bytes = int(job["out_frames"][0]) * ch * B
        rc, want_gen = port.flywheel(job, want_train, gen_bytes)
        assert rc == 0
        blocks, final = capi.flywheel_ramp_chunks(job, start, 0, 0)
        rc, want_out = port.process_chunks(blocks, want_gen, gen_bytes)
        assert rc == 0
        assert final == 0  # a flywheel ramp always ends in silence
        # the same three steps on the device, buffers chained in HBM
        d_wire = torch.from_numpy(wire).cuda()
        d_train = torch.zeros(train_bytes, dtype=torch.uint8, device="cuda")
        d_gen = torch.zeros(gen_bytes, dtype=torch.uint8, device="cuda")
        d_out = torch.zeros(gen_bytes, dtype=torch.uint8, device="cuda")
        d_prep = torch.from_numpy(prep.view(np.uint8).copy()).cuda()
        d_job = torch.from_numpy(job.view(np.uint8).copy()).cuda()
        d_blocks = torch.from_numpy(blocks.view(np.uint8).copy()).cuda()
        torch.cuda.synchronize()
        ctx.process_device(d_prep.data_ptr(), len(prep), d_wire.data_ptr(), wire.size, d_train.data_ptr(), train_bytes)
        ctx.flywheel_device(d_job.data_ptr(), 1, d_train.data_ptr(), train_bytes, d_gen.data_ptr(), gen_bytes)
        ctx.process_device(d_blocks.data_ptr(), len(blocks), d_gen.data_ptr(), gen_bytes, d_out.data_ptr(), gen_bytes)
        ctx.sync()
        assert np.array_equal(d_train.cpu().numpy(), want_train), (rate, ch, bits)
        assert np.array_equal(d_gen.cpu().numpy(), want_gen), (rate, ch, bits)
        assert np.array_equal(d_out.cpu().numpy(), want_out), (rate, ch, bits)


def test_device_rejects_bad_flywheel_jobs_loudly(ctx):
    ok = capi.flywheel_job(48000, 2, 24)
    bad = ok.copy()
    bad["bit_depth"] = 20
    jobs = np.concatenate([ok, bad])
    jobs["dst_off"][1] = 8192
    inp = training_block(48000, 2, "tone", 1)
    with pytest.raises(capi.OhpError) as e:
        run_jobs(ctx, jobs, np.concatenate([inp, inp]), 16384)
    assert e.value.status == abi.E_INVALID_DESC and "flywheel job 1" in str(e.value)
    far = ok.copy()
    far["dst_off"] = 1 << 40
    with pytest.raises(capi.OhpError) as e:
        run_jobs(ctx, far, inp, 16384)
    assert e.value.status == abi.E_OUT_OF_RANGE
    # and the context keeps working
    got = run_jobs(ctx, ok, inp, 5760)
    assert got.any()


def test_planned_starvations_on_the_gpu_play_what_the_reference_element_plays(ctx, port):
    """ohp_schedule_build's starvation records -> ohp_flywheel_plan -> the three launches on the device, against
    tests/golden/starvation_flywheel.npz: what the reference's own StarvationRamper object played when it was starved at the
    same positions (recorded by tests/golden/make_golden_starvation.py).  Some of these training blocks are a frame too long
    in the reference (44.1 kHz family): one-subsample planar descriptors at odd offsets."""
    import torch
    from flywheel_util import starved_streams
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "starvation_flywheel.npz"))
    many = 0
    for name, w, seed in starved_streams():
        inp = port.fill_pcm(w.in_bytes, seed)
        d_in = torch.from_numpy(inp).cuda()
        sv = capi.schedule_build(w.streams, w.events).starvations
        played = []
        for k in range(len(sv)):
            if not sv["plays"][k]:
                continue
            prep, job, blocks = capi.flywheel_plan(w.streams, sv[k:k + 1])
            many += len(prep) > 1
            ch, B = int(job["channels"][0]), int(job["bit_depth"][0]) // 8
            train_bytes = int(job["train_frames"][0]) * 4 * ch
            gen_bytes = int(job["out_frames"][0]) * ch * B
            d_train = torch.full((train_bytes,), 0xEE, dtype=torch.uint8, device="cuda")
            d_gen = torch.zeros(gen_bytes, dtype=torch.uint8, device="cuda")
            d_out = torch.zeros(gen_bytes, dtype=torch.uint8, device="cuda")
            d_prep = torch.from_numpy(prep.view(np.uint8).copy()).cuda()
            d_job = torch.from_numpy(job.view(np.uint8).copy()).cuda()
            d_blocks = torch.from_numpy(blocks.view(np.uint8).copy()).cuda()
            torch.cuda.synchronize()
            ctx.process_device(d_prep.data_ptr(), len(prep), d_in.data_ptr(), inp.size, d_train.data_ptr(), train_bytes)
            ctx.flywheel_device(d_job.data_ptr(), 1, d_train.data_ptr(), train_bytes, d_gen.data_ptr(), gen_bytes)
            ctx.process_device(d_blocks.data_ptr(), len(blocks), d_gen.data_ptr(), gen_bytes, d_out.data_ptr(), gen_bytes)
            ctx.sync()
            rc, want_train = port.process_chunks(prep, inp, train_bytes)
            assert rc == 0 and np.array_equal(d_train.cpu().numpy(), want_train), (name, k)
            played.append(d_out.cpu().numpy())
        assert np.array_equal(np.concatenate(played), g["audio_" + name]), name
    assert many >= 3
