"""Parity tests proper: the CUDA path, called through the C ABI, against the C oracle on identical seeded inputs.

Bar: bit-exact (the path is integer/byte work).  Run with `-m gpu` on a B200.
"""
import numpy as np
import pytest

from ohpipeline_b200 import abi, capi, workloads as W
from util import alignment_specs, covered_mask, describe_first_diff, make_desc, pack_chunks

pytestmark = pytest.mark.gpu


def run_host(ctx, chunks, inp, out_bytes, fill=0xA5):
    out = np.full(out_bytes, fill, dtype=np.uint8)
    ctx.process_host(chunks, inp, out)
    return out


def run_device(ctx, chunks, inp, out_bytes, fill=0xA5):
    """Device-resident call (what bench.py's `value` times): torch only provides the memory and the stream."""
    import torch
    d_desc = torch.from_numpy(chunks.view(np.uint8).copy()).cuda()
    d_in = torch.from_numpy(np.ascontiguousarray(inp)).cuda() if inp.size else torch.zeros(16, dtype=torch.uint8, device="cuda")
    d_out = torch.full((max(out_bytes, 1),), fill, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    stream = torch.cuda.Stream()  # the caller's stream (NULL would mean the context's own)
    st = stream.cuda_stream
    ctx.process_device(d_desc.data_ptr(), len(chunks), d_in.data_ptr(), int(inp.size), d_out.data_ptr(), out_bytes, st)
    ctx.sync(st)
    return d_out.cpu().numpy()[:out_bytes]


def oracle_out(port, chunks, inp, out_bytes, fill=0xA5):
    """Oracle output with untouched bytes (gaps between streams) left at `fill` like the GPU buffers."""
    rc, want = port.process_chunks(chunks, inp, out_bytes)
    assert rc == 0, "oracle rejected chunk %d" % (-rc - 1)
    mask = np.zeros(out_bytes, dtype=bool)
    ob = abi.chunk_out_bytes(chunks)
    for d, n in zip(chunks, ob):
        mask[int(d["dst_off"]):int(d["dst_off"]) + int(n)] = True
    want[~mask] = fill
    return want


def check_workload(ctx, port, w, device=True, host=True):
    inp = port.fill_pcm(w.in_bytes, w.seed)
    sched = capi.schedule_build(w.streams, w.events)
    want = oracle_out(port, sched.chunks, inp, w.out_bytes)
    if device:
        got = run_device(ctx, sched.chunks, inp, w.out_bytes)
        assert np.array_equal(got, want), "device path: " + describe_first_diff(got, want, sched.chunks)
    if host:
        got = run_host(ctx, sched.chunks, inp, w.out_bytes)
        # every byte: what no chunk covers (gaps between streams) must still hold the caller's fill
        assert np.array_equal(got, want), "host path: " + describe_first_diff(got, want, sched.chunks)
    return sched


def test_config1_single_stream_ramp_down_mute_up(ctx, port):
    """BASELINE configs[0]: stereo 16-bit 44.1 kHz, 20 ms ramp down, muted, 20 ms ramp up."""
    sched = check_workload(ctx, port, W.config1(6.5))
    flags = sched.chunks["flags"]
    assert (flags & abi.F_RAMP_ENABLED).any() and (flags & abi.F_SILENCE).any()


def test_config2_stereo24_full_length_ramps(ctx, port):
    check_workload(ctx, port, W.config2(n_streams=8, seconds=0.5))


def test_config3_8ch_32bit_le_starvation_ramps(ctx, port):
    sched = check_workload(ctx, port, W.config3(n_streams=12, seconds=1.0))
    # the pattern must actually have produced ramps that start and stop mid-buffer
    assert (sched.chunks["bytes"] % 7680 != 0).any()
    check_workload(ctx, port, W.config3(n_streams=4, seconds=0.25, rate=192000), host=False)


def test_every_rate_and_depth(ctx, port):
    """7350 Hz ... 384 kHz x 8/16/24/32 bits (SuiteStarvationRamper's sweep), stereo and 6-channel."""
    check_workload(ctx, port, W.all_rates())
    check_workload(ctx, port, W.all_rates(channels=6, seconds=0.2), host=False)


def test_config5_stereo24_96k(ctx, port):
    check_workload(ctx, port, W.config5(n_streams=16, seconds=0.25))


@pytest.mark.parametrize("seed", [4, 5, 6])
def test_config4_pipeline_shaped_mixed_formats(ctx, port, seed):
    """BASELINE configs[3] as the bench runs it (SURVEY 8d config 4): codec-sized messages, Ramper / StarvationRamper /
    Muter ramps stacked on three stages, driver blocks, MsgSilence, attenuation windows, P1 and P2 sinks."""
    sched = check_workload(ctx, port, W.config4(n_streams=96, seconds=0.12, seed=seed))
    f = sched.chunks["flags"]
    assert (f & abi.F_RAMP_ENABLED).any() and (f & abi.F_SILENCE).any() and (f & abi.F_IN_LITTLE_ENDIAN).any()
    assert (sched.chunks["out_fmt"] == abi.OUT_PACKED_LE).any() and (sched.chunks["attenuation"] != 256).any()


@pytest.mark.parametrize("seed", range(12))
def test_config4_mixed_formats(ctx, port, seed):
    """BASELINE configs[3] in miniature: every bit depth, 1-8 channels, both endians, P1/P2, partial and split
    ramps, muted stretches, MsgSilence, attenuation, MsgPlayable::Split at driver block boundaries."""
    check_workload(ctx, port, W.mixed(n_streams=48, seed=seed))


def test_mixed_covers_the_interesting_chunk_kinds(port):
    """Guard the generator: the mixed workloads must keep exercising each path (runs on the GPU box only because
    it shares the marker; it needs no GPU)."""
    seen = {"silence": 0, "ramped": 0, "flat_enabled": 0, "le": 0, "p2": 0, "atten": 0, "tag6": 0, "tiny": 0, "unaligned": 0}
    for seed in range(12):
        w = W.mixed(n_streams=48, seed=seed)
        c = capi.schedule_build(w.streams, w.events).chunks
        ramped = (c["flags"] & abi.F_RAMP_ENABLED) != 0
        seen["silence"] += int(((c["flags"] & abi.F_SILENCE) != 0).sum())
        seen["ramped"] += int(ramped.sum())
        seen["flat_enabled"] += int((ramped & (c["ramp_start"] == c["ramp_end"])).sum())
        seen["le"] += int(((c["flags"] & abi.F_IN_LITTLE_ENDIAN) != 0).sum())
        seen["p2"] += int((c["out_fmt"] == abi.OUT_PACKED_LE).sum())
        seen["atten"] += int((c["attenuation"] != 256).sum())
        seen["tag6"] += int((ramped & (c["channels"] == 6) & (c["bit_depth"] == 32)).sum())
        seen["tiny"] += int(((c["bytes"] > 0) & (c["bytes"] < 64)).sum())
        seen["unaligned"] += int(((c["src_off"] % 4 != 0) | (c["dst_off"] % 4 != 0)).sum())
    for k, v in seen.items():
        assert v > 0, (k, seen)


# ----------------------------------------------------------------------------------------------------------------
# hand-built descriptors: edge cases the reference's tests exercise

@pytest.mark.parametrize("bits", [8, 16, 24, 32])
@pytest.mark.parametrize("le", [False, True])
def test_every_alignment_of_source_and_destination(ctx, port, bits, le):
    """Chunks at every src/dst byte offset mod 16 (a split playable starts wherever the ramp ended)."""
    descs, in_bytes, out_bytes = pack_chunks(alignment_specs(bits, le))
    inp = port.fill_pcm(in_bytes, 99 + bits)
    want = oracle_out(port, descs, inp, out_bytes)
    got = run_device(ctx, descs, inp, out_bytes)
    assert np.array_equal(got, want), describe_first_diff(got, want, descs)


def test_host_paths_leave_uncovered_output_bytes_alone(ctx, port):
    """ohp_process_host / ohp_run_streams_host copy back what chunks cover and nothing else: holes of every size between
    chunks and between streams -- inside a slice, across slices, with descriptors in any order -- read afterwards as
    the caller left them (never as stale device memory)."""
    rng = np.random.default_rng(5)
    specs = []
    for k in range(200):
        ch = int(rng.integers(1, 5))
        frames = int(rng.integers(1, 200))
        specs.append(dict(bytes=frames * ch * 3, bit_depth=24, channels=ch, flags=abi.F_RAMP_ENABLED if k % 2 else 0,
                          ramp_start=int(rng.integers(0, 16385)), ramp_end=int(rng.integers(0, 16385)),
                          src_pad=int(rng.integers(0, 3)), dst_pad=int(rng.choice((0, 0, 1, 3, 17, 4095, 4097, 70000)))))
    descs, in_bytes, out_bytes = pack_chunks(specs)
    inp = port.fill_pcm(in_bytes, 11)
    want = oracle_out(port, descs, inp, out_bytes, fill=0x5A)
    for order in (np.arange(len(descs)), np.arange(len(descs))[::-1], rng.permutation(len(descs))):
        d = np.ascontiguousarray(descs[order])
        got = run_host(ctx, d, inp, out_bytes, fill=0x5A)
        assert np.array_equal(got, want), describe_first_diff(got, want, descs)
    # several slices (a slice closes after 48 MB moved), streams 100 bytes apart in the output, descriptors backwards
    w = W.config2(n_streams=8, seconds=6.5)
    w.streams["dst_base"] += np.arange(8, dtype=np.uint64) * 100
    out_bytes = w.out_bytes + 800
    inp = port.fill_pcm(w.in_bytes, w.seed)
    sched = capi.schedule_build(w.streams, w.events)
    want = oracle_out(port, sched.chunks, inp, out_bytes, fill=0x5A)
    got = run_host(ctx, np.ascontiguousarray(sched.chunks[::-1]), inp, out_bytes, fill=0x5A)
    assert np.array_equal(got, want), describe_first_diff(got, want, sched.chunks)
    # the whole-stage call, streams up to 15 bytes apart and two of them far away
    w = W.mixed(n_streams=40, seed=21, max_frames=3000)
    w.streams["dst_base"][20:] += 100000
    w.streams["dst_base"][30:] += 5000
    out_bytes = w.out_bytes + 105000
    inp = port.fill_pcm(w.in_bytes, w.seed)
    sched = capi.schedule_build(w.streams, w.events)
    want = oracle_out(port, sched.chunks, inp, out_bytes, fill=0x5A)
    got = np.full(out_bytes, 0x5A, dtype=np.uint8)
    ctx.run_streams_host(w.streams, w.events, inp, got)
    assert np.array_equal(got, want), describe_first_diff(got, want, sched.chunks)


def test_known_answers_from_the_reference_tests(ctx, port):
    """0x7f7f7f at full ramp -> 0x7f7e00 (TestMuter.cpp:332, TestPipeline.cpp:564); end of a full ramp down is 0."""
    frames = 64
    inp = np.full(frames * 6, 0x7F, dtype=np.uint8)
    d = make_desc(bytes=frames * 6, bit_depth=24, channels=2, flags=abi.F_RAMP_ENABLED, ramp_start=16384, ramp_end=16384)
    out = run_device(ctx, d, inp, frames * 6)
    assert bytes(out[:6]) == bytes([0x7F, 0x7E, 0x00, 0x7F, 0x7E, 0x00])
    assert np.array_equal(out, np.tile(np.array([0x7F, 0x7E, 0x00], dtype=np.uint8), frames * 2))
    d = make_desc(bytes=frames * 6, bit_depth=24, channels=2, flags=abi.F_RAMP_ENABLED, ramp_start=16384, ramp_end=0)
    out = run_device(ctx, d, inp, frames * 6)
    assert bytes(out[-6:]) == bytes(6)
    first = (int(out[0]) << 8) | int(out[1])
    assert first == 0x7F7E
    vals = (out.reshape(-1, 3)[:, 0].astype(int) << 8) | out.reshape(-1, 3)[:, 1]
    assert (np.diff(vals[::2]) <= 0).all() and np.array_equal(vals[::2], vals[1::2])  # monotone, channels equal


def test_attenuation_is_unsigned_arithmetic(ctx, port):
    """0x7f7f at 64/256 -> 0x7f7f/4 (TestMsg.cpp:982-996); negatives floor because iAttenuation is unsigned."""
    samples = np.array([0x7F7F, 0x8000, 0xFFFF, 0x0001, 0x8001, 0x1234], dtype=">u2")
    inp = samples.view(np.uint8).copy()
    for att in (0, 1, 64, 255, 257, 511):
        d = make_desc(bytes=inp.size, bit_depth=16, channels=1, attenuation=att)
        want = oracle_out(port, d, inp, inp.size)
        got = run_device(ctx, d, inp, inp.size)
        assert np.array_equal(got, want), (att, got, want)
    d = make_desc(bytes=inp.size, bit_depth=16, channels=1, attenuation=64)
    got = run_device(ctx, d, inp, inp.size)
    assert ((int(got[0]) << 8) | int(got[1])) == 0x7F7F // 4


def test_silence_and_six_channel_pattern(ctx, port):
    """MsgPlayableSilence: zeros, ramp ignored; 6 channels carry the 00 00 00 c0 tag in the first 32 bytes of each
    9216-rounded block whatever the bit depth (Msg.cpp:2874-2893); 10 channels (TestMsg.cpp:1293)."""
    specs = []
    for bits in (8, 16, 24, 32):
        for ch in (1, 2, 6, 10):
            fb = ch * bits // 8
            for frames in (1, 3, 500, 9216 // fb, 9216 // fb + 7, 3 * (9216 // fb) + 11):
                specs.append(dict(bytes=frames * fb, bit_depth=bits, channels=ch, flags=abi.F_SILENCE | abi.F_RAMP_ENABLED,
                                  ramp_start=12000, ramp_end=3000, dst_pad=frames % 5))
    descs, in_bytes, out_bytes = pack_chunks(specs)
    inp = np.zeros(16, dtype=np.uint8)
    want = oracle_out(port, descs, inp, out_bytes)
    got = run_device(ctx, descs, inp, out_bytes)
    assert np.array_equal(got, want), describe_first_diff(got, want, descs)
    six = descs[(descs["channels"] == 6) & (descs["bytes"] >= 32)][0]
    o = int(six["dst_off"])
    assert list(got[o + 3:o + 32:4]) == [0x00, 0x10, 0x20, 0x30, 0x40, 0x50, 0x60, 0x70]


def test_single_frame_and_maximum_chunks(ctx, port):
    """N == 1 uses Start() alone (Msg.cpp:835); a full 9216-byte cell for every format that divides it."""
    specs = []
    for bits in (8, 16, 24, 32):
        b = bits // 8
        for ch in (1, 2, 3, 5, 6, 7, 8):
            fb = ch * b
            for frames in (1, 2, 9216 // fb):
                for (s, e) in ((16384, 0), (0, 16384), (5000, 5000), (123, 16000)):
                    specs.append(dict(bytes=frames * fb, bit_depth=bits, channels=ch, flags=abi.F_RAMP_ENABLED,
                                      ramp_start=s, ramp_end=e))
    descs, in_bytes, out_bytes = pack_chunks(specs, align=16)
    inp = port.fill_pcm(in_bytes, 4242)
    want = oracle_out(port, descs, inp, out_bytes)
    got = run_device(ctx, descs, inp, out_bytes)
    assert np.array_equal(got, want), describe_first_diff(got, want, descs)


def test_edge_sample_values(ctx, port):
    """0x7f.., 0xff.., 0x80 00.., zeros and +/-1 through every multiplier of the table (sign paths, Q15 0x7fff)."""
    for bits in (8, 16, 24, 32):
        b = bits // 8
        pats = [bytes([0x7F] * b), bytes([0xFF] * b), bytes([0x80] + [0] * (b - 1)), bytes(b), bytes([0] * (b - 1) + [1]),
                bytes([0x80] + [0] * (b - 2) + [1]) if b > 1 else bytes([0x81])]
        frames = 2048
        inp = np.frombuffer(b"".join(pats[i % len(pats)] for i in range(frames)), dtype=np.uint8).copy()
        specs = [dict(bytes=inp.size, bit_depth=bits, channels=1, flags=abi.F_RAMP_ENABLED, ramp_start=16384, ramp_end=0)]
        descs, _, out_bytes = pack_chunks(specs)
        want = oracle_out(port, descs, inp, out_bytes)
        got = run_device(ctx, descs, inp, out_bytes)
        assert np.array_equal(got, want), (bits, describe_first_diff(got, want, descs))


def test_empty_batch_and_zero_byte_chunks(ctx, port):
    """A 1-jiffy split yields a 0-byte playable (TestMsg.cpp:1106-1359): Read() does nothing."""
    out = np.full(64, 0xA5, dtype=np.uint8)
    ctx.process_host(np.zeros(0, dtype=abi.CHUNK_DESC), np.zeros(16, dtype=np.uint8), out)
    assert (out == 0xA5).all()
    specs = [dict(bytes=0, bit_depth=24, channels=2, flags=abi.F_RAMP_ENABLED), dict(bytes=12, bit_depth=24, channels=2),
             dict(bytes=0, bit_depth=16, channels=2, flags=abi.F_SILENCE)]
    descs, in_bytes, out_bytes = pack_chunks(specs)
    inp = port.fill_pcm(in_bytes, 5)
    want = oracle_out(port, descs, inp, out_bytes)
    got = run_device(ctx, descs, inp, out_bytes)
    assert np.array_equal(got, want)


def test_packed_le_output_is_byte_swapped_be_output(ctx, port):
    """P2 (ProcessorPcmSwpEndianPacked) with every fragment kept (aux = OHP_LE_APPEND) == per-subsample byte reversal of P1,
    for 8/16/24-bit."""
    for bits in (8, 16, 24):
        b = bits // 8
        frames, ch = 777, 3
        n = frames * ch * b
        inp = port.fill_pcm(n + 16, bits)
        outs = {}
        for fmt in (abi.OUT_PACKED_BE, abi.OUT_PACKED_LE):
            d = make_desc(bytes=n, bit_depth=bits, channels=ch, flags=abi.F_RAMP_ENABLED, ramp_start=9000, ramp_end=100, out_fmt=fmt,
                          aux=abi.LE_APPEND if fmt == abi.OUT_PACKED_LE else 0)
            outs[fmt] = run_device(ctx, d, inp, n)
            assert np.array_equal(outs[fmt], oracle_out(port, d, inp, n))
        assert np.array_equal(outs[abi.OUT_PACKED_LE].reshape(-1, b)[:, ::-1], outs[abi.OUT_PACKED_BE].reshape(-1, b))


def test_packed_le_sink_to_the_letter(ctx, port):
    """aux = 0: the chunk writes what the reference's ProcessorPcmSwpEndianPacked is left holding after the read -- all of an
    8-bit or unramped playable, the last <= 256-byte fragment of a ramped 16/24-bit one (its SwapEndianness16/24 overwrite,
    TestCodecInteractiveMain.cpp:570-590).  The port this compares with is pinned against the class itself
    (tests/test_reference_sinks_codecs.py)."""
    rng = np.random.default_rng(40)
    specs = []
    for k in range(300):
        bits = int(rng.choice((8, 16, 24)))
        ch = int(rng.integers(1, 9))
        fb = ch * bits // 8
        frames = int(rng.choice((1, 2, 256 // fb, 256 // fb + 1, 2 * (256 // fb), int(rng.integers(1, 9216 // fb + 1)))))
        specs.append(dict(bytes=frames * fb, bit_depth=bits, channels=ch,
                          flags=(abi.F_RAMP_ENABLED if k % 3 else 0) | (abi.F_IN_LITTLE_ENDIAN if k % 5 == 0 else 0),
                          ramp_start=int(rng.integers(0, 16385)), ramp_end=int(rng.integers(0, 16385)),
                          out_fmt=abi.OUT_PACKED_LE, aux=int(k % 7 == 0), src_pad=int(rng.integers(0, 5)), dst_pad=int(rng.integers(0, 5))))
    descs, in_bytes, out_bytes = pack_chunks(specs)
    inp = port.fill_pcm(in_bytes, 41)
    assert (abi.chunk_out_bytes(descs) < descs["bytes"]).any()
    want = oracle_out(port, descs, inp, out_bytes)
    got = run_device(ctx, descs, inp, out_bytes)
    assert np.array_equal(got, want), describe_first_diff(got, want, descs)
    got = run_host(ctx, descs, inp, out_bytes)
    assert np.array_equal(got, want), describe_first_diff(got, want, descs)


def test_device_rejects_bad_descriptors_loudly(ctx):
    import torch
    bad = make_desc(bytes=25, bit_depth=24, channels=2)
    d_desc = torch.from_numpy(bad.view(np.uint8).copy()).cuda()
    d_in = torch.zeros(64, dtype=torch.uint8, device="cuda")
    d_out = torch.zeros(64, dtype=torch.uint8, device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    ctx.process_device(d_desc.data_ptr(), 1, d_in.data_ptr(), 64, d_out.data_ptr(), 64, st)
    with pytest.raises(capi.OhpError) as e:
        ctx.sync(st)
    assert e.value.status == abi.E_INVALID_DESC
    ctx.sync(st)  # the error is reported once
    with pytest.raises(capi.OhpError) as e:
        ctx.process_host(make_desc(bytes=24, bit_depth=24, channels=2, src_off=1 << 30), np.zeros(64, np.uint8), np.zeros(64, np.uint8))
    assert e.value.status == abi.E_OUT_OF_RANGE


# ----------------------------------------------------------------------------------------------------------------
# full-size properties (sizes the scalar oracle cannot finish in seconds)

def test_full_size_config5_slice_properties(ctx, port):
    """4096 streams x 0.5 s of config 5 (1.2 GB in): (1) per-stream checksums equal across streams that share a seed,
    (2) linearity of the ramp in the sample value's sign (x -> ~x maps r -> ~r for the 16-bit ramp path is NOT a
    property of floor), so instead: idempotence of the unramped path and a checksum-of-checksums against a sampled
    oracle run."""
    import torch
    n_streams, seconds = 4096, 0.5
    w = W.config5(n_streams=n_streams, seconds=seconds)
    sched = capi.schedule_build(w.streams, w.events)
    per_stream = int(w.streams["total_frames"][0]) * 6
    # every stream gets the SAME pcm (seeded once), so every stream must produce the same bytes
    one = port.fill_pcm(per_stream, 55)
    d_in = torch.from_numpy(one).cuda().repeat(n_streams)
    assert d_in.numel() == w.in_bytes
    d_out = torch.zeros(w.out_bytes, dtype=torch.uint8, device="cuda")
    d_desc = torch.from_numpy(sched.chunks.view(np.uint8).copy()).cuda()
    st = torch.cuda.current_stream().cuda_stream
    ctx.process_device(d_desc.data_ptr(), len(sched.chunks), d_in.data_ptr(), w.in_bytes, d_out.data_ptr(), w.out_bytes, st)
    ctx.sync(st)
    offs = np.concatenate([w.streams["dst_base"], [w.streams["dst_base"][-1] + per_stream]]).astype(np.uint64)
    d_off = torch.from_numpy(offs.view(np.int64).copy()).cuda()
    d_sums = torch.zeros(n_streams, dtype=torch.int64, device="cuda")
    ctx.checksums_device(d_out.data_ptr(), d_off.data_ptr(), n_streams, d_sums.data_ptr(), st)
    ctx.sync(st)
    sums = d_sums.cpu().numpy().view(np.uint64)
    # oracle for ONE stream
    w1 = W.config5(n_streams=1, seconds=seconds)
    rc, want, _, _ = port.run(w1.streams, w1.events, one, w1.out_bytes)
    assert rc == 0
    assert int(sums[0]) == port.checksum(want[:per_stream])
    assert (sums == sums[0]).all()
    # and the bytes of a few streams outright
    for s in (0, 1, n_streams // 2, n_streams - 1):
        got = d_out[int(offs[s]):int(offs[s]) + per_stream].cpu().numpy()
        assert np.array_equal(got, want[:per_stream])


# ----------------------------------------------------------------------------------------------------------------
# golden vectors recorded from the reference itself (tests/golden/, see make_golden.py)

import glob as _glob
import hashlib as _hashlib
import os as _os
import zlib as _zlib

_GOLDEN = sorted(p for p in _glob.glob(_os.path.join(_os.path.dirname(__file__), "golden", "*.npz"))
                 if not p.endswith(("ramp_algebra.npz", "flywheel.npz")))


@pytest.mark.parametrize("path", _GOLDEN, ids=[_os.path.basename(p)[:-4] for p in _GOLDEN])
def test_cuda_path_reproduces_reference_golden_vectors(ctx, port, path):
    """Descriptors from the product's host message model + bytes from the CUDA kernel == what the reference's
    MsgFactory -> SetRamp -> CreatePlayable -> Read(ProcessorPcmBufTest) produced."""
    g = np.load(path)
    inp = port.fill_pcm(int(g["in_bytes"]), int(g["seed"]))
    sched = capi.schedule_build(g["streams"], g["events"])
    assert np.array_equal(sched.chunks, g["chunks"])
    out_bytes = int(g["out_bytes"])
    for runner in (run_device, run_host):
        out = runner(ctx, sched.chunks, inp, out_bytes)
        ob = abi.chunk_out_bytes(sched.chunks)
        crc = np.array([_zlib.crc32(out[int(d["dst_off"]):int(d["dst_off"]) + int(n)].tobytes())
                        for d, n in zip(sched.chunks, ob)], dtype=np.uint32)
        bad = np.nonzero(crc != g["chunk_crc"])[0]
        assert bad.size == 0, "chunk %d differs from the reference: %s" % (bad[0], sched.chunks[bad[0]])
    # bytes no chunk covers were pre-filled with 0xA5 by run_device; the reference buffer has zeros there
    mask = np.zeros(out_bytes, dtype=bool)
    for d, n in zip(sched.chunks, ob):
        mask[int(d["dst_off"]):int(d["dst_off"]) + int(n)] = True
    out = run_device(ctx, sched.chunks, inp, out_bytes, fill=0)
    assert _hashlib.sha256(out.tobytes()).digest() == g["out_sha256"].tobytes()


# ----------------------------------------------------------------------------------------------------------------
# the other IPcmProcessor sinks of the reference tree (SURVEY 8f #2): FlywheelInput, RampGenerator, Songcast Sender

def _compare_whole(ctx, port, descs, inp, out_bytes):
    rc, want = port.process_chunks(descs, inp, out_bytes)
    assert rc == 0, "oracle rejected chunk %d" % (-rc - 1)
    got = run_device(ctx, descs, inp, out_bytes, fill=0)
    assert np.array_equal(got, want), describe_first_diff(got, want, descs)
    got = np.full(out_bytes, 0x5A, dtype=np.uint8)
    ctx.process_host(descs, inp, got)
    m = covered_mask(descs, out_bytes)
    assert np.array_equal(got[m], want[m]), "host path differs from the oracle"
    assert (got[~m] == 0x5A).all(), "ohp_process_host wrote bytes no chunk covers (planar output is strided)"


def test_planar32_sink_flywheel_input(ctx, port):
    """FlywheelInput (StarvationRamper.cpp:117-186): interleaved -> planar 4-byte BE left-justified, several playables
    appended into the same planes the way Prepare() reads a queue of messages."""
    rng = np.random.default_rng(31)
    descs = []
    src = dst = 0
    for bits in (8, 16, 24, 32):
        b = bits // 8
        for ch in (1, 2, 3, 6, 8):
            parts = [int(x) for x in rng.integers(1, 120, 3)]
            total = sum(parts) + int(rng.integers(0, 5))
            done = 0
            for i, frames in enumerate(parts):
                silence = (i == 1 and ch in (2, 6))
                d = make_desc(bytes=frames * ch * b, bit_depth=bits, channels=ch, out_fmt=abi.OUT_PLANAR32_BE, aux=total,
                              flags=(abi.F_SILENCE if silence else (abi.F_IN_LITTLE_ENDIAN if (bits + ch) % 3 == 0 else 0))
                              | (abi.F_RAMP_ENABLED if i == 2 else 0),
                              ramp_start=int(rng.integers(0, 16385)), ramp_end=int(rng.integers(0, 16385)),
                              src_off=src, dst_off=dst + done * 4)
                descs.append(d[0])
                if not silence:
                    src += frames * ch * b + int(rng.integers(0, 3))
                done += frames
            dst += ch * total * 4 + 4 * int(rng.integers(0, 3))
    descs = np.array(descs, dtype=abi.CHUNK_DESC)
    inp = port.fill_pcm(src + 64, 3131)
    _compare_whole(ctx, port, descs, inp, dst + 64)


def test_from32_sink_ramp_generator(ctx, port):
    """RampGenerator::ProcessFragment (StarvationRamper.cpp:281-326): 32-bit BE in, packed 8/16/24/32-bit BE out."""
    rng = np.random.default_rng(32)
    specs = []
    for ob in (8, 16, 24, 32):
        for ch in (1, 2, 5, 6, 8):
            for frames in (1, 7, 48, 192, 9216 // (4 * ch)):
                specs.append(dict(bytes=frames * ch * 4, bit_depth=32, channels=ch, out_fmt=abi.OUT_FROM32_BE, aux=ob,
                                  flags=(abi.F_RAMP_ENABLED if frames % 2 else 0), ramp_start=int(rng.integers(0, 16385)),
                                  ramp_end=int(rng.integers(0, 16385)), src_pad=int(rng.integers(0, 4)), dst_pad=int(rng.integers(0, 4))))
    descs, in_bytes, out_bytes = pack_chunks(specs)
    inp = port.fill_pcm(in_bytes, 3232)
    _compare_whole(ctx, port, descs, inp, out_bytes)


def test_songcast_sink(ctx, port):
    """Sender::DoProcessFragment (Av/Songcast/Sender.cpp:356-377): two channels from FirstChannelToSend, at most
    three bytes per subsample; mono sends one; silence goes through the same path."""
    rng = np.random.default_rng(33)
    specs = []
    for bits in (8, 16, 24, 32):
        b = bits // 8
        for ch in (1, 2, 3, 6, 8, 10, 12):
            first = 0 if ch < 10 else 8  # Sender::FirstChannelToSend, Sender.cpp:351-354
            for frames in (1, 5, 64, 9216 // (ch * b)):
                kind = int(rng.integers(0, 4))
                flags = [0, abi.F_RAMP_ENABLED, abi.F_RAMP_ENABLED | abi.F_IN_LITTLE_ENDIAN, abi.F_SILENCE][kind]
                specs.append(dict(bytes=frames * ch * b, bit_depth=bits, channels=ch, out_fmt=abi.OUT_SONGCAST, aux=first, flags=flags,
                                  ramp_start=int(rng.integers(0, 16385)), ramp_end=int(rng.integers(0, 16385)),
                                  src_pad=int(rng.integers(0, 4)), dst_pad=int(rng.integers(0, 4))))
    descs, in_bytes, out_bytes = pack_chunks(specs)
    inp = port.fill_pcm(in_bytes, 3333)
    _compare_whole(ctx, port, descs, inp, out_bytes)


def test_converting_sinks_reject_what_the_reference_asserts_on(ctx):
    bad = [make_desc(bytes=32, bit_depth=16, channels=2, out_fmt=abi.OUT_FROM32_BE, aux=16),       # RampGenerator is fed 32-bit only
           make_desc(bytes=32, bit_depth=32, channels=2, out_fmt=abi.OUT_FROM32_BE, aux=12),
           make_desc(bytes=32, bit_depth=32, channels=2, out_fmt=abi.OUT_FROM32_BE, aux=16, flags=abi.F_SILENCE),  # ProcessSilence ASSERTS
           make_desc(bytes=32, bit_depth=16, channels=2, out_fmt=abi.OUT_PLANAR32_BE, aux=7),      # plane shorter than the playable
           make_desc(bytes=32, bit_depth=16, channels=2, out_fmt=abi.OUT_SONGCAST, aux=1)]         # first channel + 2 > channels
    for d in bad:
        assert capi.validate(d, 1 << 20, 1 << 20)[0] == abi.E_INVALID_DESC, d
        with pytest.raises(capi.OhpError):
            ctx.process_host(d, np.zeros(64, np.uint8), np.zeros(4096, np.uint8))


def test_inflight_tuning_never_changes_results(ctx, port):
    """Large batches are tuned: the first launches of a batch shape each keep a different number of chunks in flight
    (ohp_inflight_cap).  Every launch must produce the same bytes, and those are the oracle's.  Two batch shapes: uniform
    stereo 24-bit, and mixed formats shaped like a pipeline's output."""
    for w in (W.config5(n_streams=1024, seconds=0.4), W.config4(n_streams=760, seconds=0.25, seed=7)):
        check_tuned_launches(ctx, port, w)


def check_tuned_launches(ctx, port, w):
    import torch
    sched = capi.schedule_build(w.streams, w.events)
    assert len(sched.chunks) >= 65536 and w.in_bytes + w.out_bytes >= (256 << 20), w.name
    inp = port.fill_pcm(w.in_bytes, w.seed)
    d_desc = torch.from_numpy(sched.chunks.view(np.uint8).copy()).cuda()
    d_in = torch.from_numpy(inp).cuda()
    stream = torch.cuda.Stream()
    st = stream.cuda_stream
    caps, first = [], None
    for launch in range(7):
        d_out = torch.zeros(w.out_bytes, dtype=torch.uint8, device="cuda")
        torch.cuda.synchronize()
        ctx.process_device(d_desc.data_ptr(), len(sched.chunks), d_in.data_ptr(), w.in_bytes, d_out.data_ptr(), w.out_bytes, st)
        ctx.sync(st)
        caps.append(ctx.inflight_cap())
        if first is None:
            first = d_out
        else:
            assert torch.equal(d_out, first), (w.name, launch, caps)
    assert len(set(caps[:3])) == 3, (w.name, caps)           # three candidates explored ...
    assert caps[4] == caps[5] == caps[6], (w.name, caps)     # ... (the first one again, warm, if it was close) then the fastest is kept
    # the first 24 streams against the oracle
    k = int(sched.stream_chunk_begin[24])
    sub = sched.chunks[:k]
    hi = int(w.streams["dst_base"][24])
    rc, want = port.process_chunks(sub, inp, hi)
    assert rc == 0
    mask = covered_mask(sub, hi)
    assert np.array_equal(first[:hi].cpu().numpy()[mask], want[mask]), w.name
