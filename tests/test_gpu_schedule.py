"""Device-side schedule builder (include/ohp_schedule_device.h, SURVEY 8f #1) against
  * the playables the REFERENCE produced (tests/golden/*.npz, recorded from oracle/_ref), and
  * the host message model (ohp_schedule_build), on the BASELINE configs and on randomized mixed workloads:
descriptors, chunk info (direction, jiffies), per-stream chunk ranges and output sizes must be identical.
Then the descriptors built on the GPU drive the hot path and the bytes are checked against the oracle."""
import glob
import os

import numpy as np
import pytest

from ohpipeline_b200 import abi, capi, workloads
from util import covered_mask

pytestmark = pytest.mark.gpu

GOLDEN = sorted(g for g in glob.glob(os.path.join(os.path.dirname(__file__), "golden", "*.npz"))
                if not g.endswith(("ramp_algebra.npz", "flywheel.npz")))


def same_schedule(dev, host):
    assert len(dev.chunks) == len(host.chunks)
    assert np.array_equal(dev.stream_chunk_begin, host.stream_chunk_begin)
    assert np.array_equal(dev.stream_out_bytes, host.stream_out_bytes)
    if not np.array_equal(dev.chunks, host.chunks):
        i = int(np.nonzero(dev.chunks != host.chunks)[0][0])
        raise AssertionError("descriptor %d differs: device %s host %s" % (i, dev.chunks[i], host.chunks[i]))
    assert np.array_equal(dev.info, host.info)


def check_both(ctx, w):
    """Device walk vs host model: identical schedules, or the same refusal where the reference would ASSERT."""
    try:
        host = capi.schedule_build(w.streams, w.events)
    except capi.OhpError as eh:
        with pytest.raises(capi.OhpError) as ed:
            ctx.schedule_build_device(w.streams, w.events)
        assert ed.value.status == eh.status
        return None
    same_schedule(ctx.schedule_build_device(w.streams, w.events), host)
    return host


@pytest.mark.parametrize("path", GOLDEN, ids=[os.path.basename(p)[:-4] for p in GOLDEN])
def test_device_schedule_reproduces_reference_playables(ctx, path):
    g = np.load(path)
    dev = ctx.schedule_build_device(g["streams"], g["events"])
    assert np.array_equal(dev.chunks, g["chunks"]), "descriptors differ from the reference's playables"
    assert np.array_equal(dev.info, g["info"])


@pytest.mark.parametrize("make", [
    lambda: workloads.config1(6.2),
    lambda: workloads.config2(n_streams=40, seconds=0.5),
    lambda: workloads.config3(n_streams=70, seconds=1.0),
    lambda: workloads.config5(n_streams=100, seconds=0.25),
], ids=["config1", "config2", "config3", "config5"])
def test_device_schedule_matches_host_on_baseline_configs(ctx, make):
    assert check_both(ctx, make()) is not None


@pytest.mark.parametrize("seed", [4, 11, 12, 13, 14, 15, 16, 17])
def test_device_schedule_matches_host_on_mixed_workloads(ctx, seed):
    assert check_both(ctx, workloads.mixed(n_streams=96, seed=seed, max_frames=5000)) is not None


@pytest.mark.parametrize("seed", [1, 5, 6])
def test_device_walk_is_the_element_model(ctx, seed):
    """Stages that ARE the reference's elements (Ramper, StarvationRamper, Muter: ops 8-12 of include/ohp_schedule.h): the walk
    the GPU runs against the host model, which tests/test_elements_vs_reference.py holds against the element objects
    themselves (and tests/golden/elements_11.npz, recorded from those objects, is among the golden files above)."""
    assert check_both(ctx, workloads.elements(seed, n_streams=64)) is not None
    # Mute() twice in a row: the reference ASSERTS, host and device refuse alike
    assert check_both(ctx, workloads.elements(seed, n_streams=64, illegal=True)) is None


def test_device_schedule_many_streams(ctx):
    """More streams than one wave of threads; ragged event slices; one partial warp."""
    assert check_both(ctx, workloads.mixed(n_streams=3001, seed=22, max_frames=700)) is not None
    # seed 21 holds a stream on which the reference ASSERTs (a MsgSilence split below one sample): same refusal
    assert check_both(ctx, workloads.mixed(n_streams=3001, seed=21, max_frames=700)) is None


def test_device_schedule_empty_and_degenerate(ctx):
    none = ctx.schedule_build_device(np.zeros(0, dtype=abi.STREAM_SPEC), np.zeros(0, dtype=abi.RAMP_EVENT))
    assert len(none.chunks) == 0 and list(none.stream_chunk_begin) == [0]
    # a stream without audio produces nothing; its neighbours are unaffected
    w = workloads.config5(n_streams=3, seconds=0.02)
    w.streams["total_frames"][1] = 0
    same_schedule(ctx.schedule_build_device(w.streams, w.events), capi.schedule_build(w.streams, w.events))


def test_device_schedule_fails_where_the_host_model_fails(ctx):
    w = workloads.config5(n_streams=4, seconds=0.02)
    # unsupported sample rate: Jiffies::PerSample throws SampleRateInvalid (Msg.cpp:424-470) -> not representable
    bad = w.streams.copy()
    bad["sample_rate"][2] = 12345
    with pytest.raises(capi.OhpError) as e:
        ctx.schedule_build_device(bad, w.events)
    assert e.value.status == abi.E_INVALID_ARG and "stream 2" in str(e.value)
    with pytest.raises(capi.OhpError) as eh:
        capi.schedule_build(bad, w.events)
    assert eh.value.status == abi.E_INVALID_ARG
    # bit depth the reference ASSERTs on (DecodedAudio::ConstructPcm, Msg.cpp:349-366)
    bad = w.streams.copy()
    bad["bit_depth"][1] = 20
    with pytest.raises(capi.OhpError) as e:
        ctx.schedule_build_device(bad, w.events)
    with pytest.raises(capi.OhpError) as eh:
        capi.schedule_build(bad, w.events)
    assert e.value.status == eh.value.status
    # a converting sink is not a schedule output
    bad = w.streams.copy()
    bad["out_fmt"][0] = abi.OUT_PLANAR32_BE
    with pytest.raises(capi.OhpError) as e:
        ctx.schedule_build_device(bad, w.events)
    assert e.value.status == abi.E_INVALID_ARG
    # event slice outside the events array
    bad = w.streams.copy()
    bad["first_event"][3] = len(w.events)
    bad["num_events"][3] = 1
    with pytest.raises(capi.OhpError) as e:
        ctx.schedule_build_device(bad, w.events)
    assert e.value.status == abi.E_INVALID_ARG
    # the context is still usable afterwards
    same_schedule(ctx.schedule_build_device(w.streams, w.events), capi.schedule_build(w.streams, w.events))


def test_silence_split_below_one_sample_asserts_on_both(ctx):
    """A MsgSilence split below one sample leaves a zero-length first part on which Ramp::Set ASSERTs (DESIGN.md
    'reference behaviours' #5): host model and device walk must both report it."""
    rate = 44100
    jps = abi.jiffies_per_sample(rate)
    s = np.zeros(1, dtype=abi.STREAM_SPEC)
    s[0]["sample_rate"] = rate; s[0]["bit_depth"] = 16; s[0]["channels"] = 2; s[0]["chunk_frames"] = 100
    s[0]["total_frames"] = 400; s[0]["num_events"] = 2
    ev = np.zeros(2, dtype=abi.RAMP_EVENT)
    ev[0] = (0, 0, abi.EV_INSERT_SILENCE, 10 * jps, 0)
    ev[1] = (0, 0, abi.EV_RAMP_DOWN, jps // 2, 0)     # remaining < one sample: Split(remaining) on silence
    with pytest.raises(capi.OhpError) as eh:
        capi.schedule_build(s, ev)
    with pytest.raises(capi.OhpError) as ed:
        ctx.schedule_build_device(s, ev)
    assert ed.value.status == eh.value.status == abi.E_INVALID_DESC


def test_descriptors_built_on_the_gpu_drive_the_hot_path(ctx, port):
    """events -> (GPU) descriptors -> (GPU) ramp + convert, nothing but specs and PCM crossing PCIe; bytes vs oracle."""
    import torch
    w = workloads.mixed(n_streams=64, seed=31, max_frames=4000)
    inp = port.fill_pcm(w.in_bytes, w.seed)
    rc, want, chunks, _ = port.run(w.streams, w.events, inp, w.out_bytes)
    assert rc == 0
    d_streams = torch.from_numpy(w.streams.view(np.uint8).copy()).cuda()
    d_events = torch.from_numpy(w.events.view(np.uint8).copy()).cuda()
    d_begin = torch.zeros(len(w.streams) + 1, dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()  # the context's stream does not order against torch's
    total = ctx.schedule_count_device(d_streams.data_ptr(), len(w.streams), d_events.data_ptr(), len(w.events),
                                      d_begin.data_ptr())
    assert total == len(chunks)
    d_desc = torch.zeros(total * abi.CHUNK_DESC.itemsize, dtype=torch.uint8, device="cuda")
    ctx.schedule_emit_device(d_streams.data_ptr(), len(w.streams), d_events.data_ptr(), len(w.events),
                             d_begin.data_ptr(), d_desc.data_ptr())
    d_in = torch.from_numpy(inp).cuda()
    d_out = torch.zeros(w.out_bytes, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    ctx.process_device(d_desc.data_ptr(), total, d_in.data_ptr(), w.in_bytes, d_out.data_ptr(), w.out_bytes)
    ctx.sync()
    got = d_out.cpu().numpy()
    mask = covered_mask(chunks, w.out_bytes)
    assert np.array_equal(got[mask], want[mask])


@pytest.mark.parametrize("make", [
    lambda: workloads.config1(6.2),
    lambda: workloads.config4(n_streams=80, seconds=0.12, seed=9),
    lambda: workloads.mixed(n_streams=64, seed=33, max_frames=4000),
    lambda: workloads.config5(n_streams=700, seconds=0.25),     # > 48 MB each way: several slices in flight
], ids=["config1", "config4", "mixed", "config5_sliced"])
def test_whole_stage_in_one_call_from_host_buffers(ctx, port, make):
    """ohp_run_streams_host: specs + events + host PCM in, bytes out -- descriptors never exist on the host.
    Bytes, per-stream output sizes and chunk count against the oracle."""
    w = make()
    inp = port.fill_pcm(w.in_bytes, w.seed)
    rc, want, chunks, _ = port.run(w.streams, w.events, inp, w.out_bytes)
    assert rc == 0
    host = capi.schedule_build(w.streams, w.events)
    got = np.zeros(w.out_bytes, dtype=np.uint8)
    outb, total = ctx.run_streams_host(w.streams, w.events, inp, got)
    assert total == len(chunks)
    assert np.array_equal(outb, host.stream_out_bytes)
    mask = covered_mask(chunks, w.out_bytes)
    assert np.array_equal(got[mask], want[mask])


def test_whole_stage_call_reports_what_the_parts_report(ctx):
    w = workloads.config5(n_streams=4, seconds=0.02)
    inp = np.zeros(w.in_bytes, dtype=np.uint8)
    out = np.zeros(w.out_bytes, dtype=np.uint8)
    # nothing to do
    outb, total = ctx.run_streams_host(w.streams[:0], w.events[:0], inp, out)
    assert total == 0 and len(outb) == 0
    # a spec the message model cannot represent
    bad = w.streams.copy()
    bad["sample_rate"][2] = 12345
    with pytest.raises(capi.OhpError) as e:
        ctx.run_streams_host(bad, w.events, inp, out)
    assert e.value.status == abi.E_INVALID_ARG and "stream 2" in str(e.value)
    # a stream that reaches outside the output arena
    with pytest.raises(capi.OhpError) as e:
        ctx.run_streams_host(w.streams, w.events, inp, out[:w.out_bytes // 2])
    assert e.value.status == abi.E_OUT_OF_RANGE
    # ... and outside the input arena
    with pytest.raises(capi.OhpError) as e:
        ctx.run_streams_host(w.streams, w.events, inp[:w.in_bytes // 2], out)
    assert e.value.status == abi.E_OUT_OF_RANGE
    # the context is still usable
    outb, total = ctx.run_streams_host(w.streams, w.events, inp, out)
    assert total == len(capi.schedule_build(w.streams, w.events).chunks)


@pytest.mark.parametrize("make", [
    lambda: workloads.config4(n_streams=80, seconds=0.12, seed=9),
    lambda: workloads.mixed(n_streams=64, seed=35, max_frames=4000),
    lambda: workloads.config2(n_streams=24, seconds=0.4),
], ids=["config4", "mixed", "config2"])
def test_whole_stage_for_a_batch_resident_in_hbm(ctx, port, make):
    """ohp_fill_streams_device + ohp_run_streams_device: the per-stream seeded bytes are the ones the oracle's generator
    gives, and specs + events + PCM in HBM come back as the bytes the oracle computes, every stream's size included.
    Twice, with a second batch in between: the context reuses its descriptor buffer."""
    import torch
    w = make()
    seed_base, first_id = 9 << 32, 12345
    d_streams = torch.from_numpy(w.streams.view(np.uint8).copy()).cuda()
    d_events = (torch.from_numpy(w.events.view(np.uint8).copy()).cuda() if len(w.events)
                else torch.zeros(32, dtype=torch.uint8, device="cuda"))
    d_in = torch.zeros(w.in_bytes + 16, dtype=torch.uint8, device="cuda")
    d_out = torch.full((w.out_bytes + 16,), 0x5A, dtype=torch.uint8, device="cuda")
    d_outb = torch.zeros(len(w.streams), dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    ctx.fill_streams_device(d_in.data_ptr(), w.in_bytes, d_streams.data_ptr(), len(w.streams), seed_base, first_id)
    ctx.sync()
    inp = port.fill_streams(w.streams, w.in_bytes, seed_base, first_id)
    assert np.array_equal(d_in.cpu().numpy()[:w.in_bytes], inp), "the GPU and the CPU arm would not see the same PCM"
    rc, want, chunks, _ = port.run(w.streams, w.events, inp, w.out_bytes)
    assert rc == 0
    host = capi.schedule_build(w.streams, w.events)
    mask = covered_mask(chunks, w.out_bytes)
    for round_ in range(2):
        total = ctx.run_streams_device(d_streams.data_ptr(), len(w.streams), d_events.data_ptr(), len(w.events),
                                       d_in.data_ptr(), w.in_bytes, d_out.data_ptr(), w.out_bytes, d_outb.data_ptr())
        ctx.sync()
        assert total == len(chunks)
        assert np.array_equal(d_outb.cpu().numpy().view(np.uint64), host.stream_out_bytes)
        got = d_out.cpu().numpy()[:w.out_bytes]
        assert np.array_equal(got[mask], want[mask])
        assert (got[~mask] == 0x5A).all(), "bytes no chunk covers were written"
        if round_ == 0:
            # more chunks: the walk into the existing buffer stops short, the buffer grows and the walk runs again
            other = workloads.config5(n_streams=300, seconds=0.05)
            o_inp = port.fill_pcm(other.in_bytes, other.seed)
            rc, o_want, o_chunks, _ = port.run(other.streams, other.events, o_inp, other.out_bytes)
            assert rc == 0
            o_in = torch.from_numpy(np.concatenate([o_inp, np.zeros(16, np.uint8)])).cuda()
            o_out = torch.full((other.out_bytes + 16,), 0x5A, dtype=torch.uint8, device="cuda")
            o_s = torch.from_numpy(other.streams.view(np.uint8).copy()).cuda()
            o_e = torch.from_numpy(other.events.view(np.uint8).copy()).cuda()
            torch.cuda.synchronize()
            n_other = ctx.run_streams_device(o_s.data_ptr(), len(other.streams), o_e.data_ptr(), len(other.events),
                                             o_in.data_ptr(), other.in_bytes, o_out.data_ptr(), other.out_bytes)
            ctx.sync()
            assert n_other == len(o_chunks)
            o_got = o_out.cpu().numpy()[:other.out_bytes]
            o_mask = covered_mask(o_chunks, other.out_bytes)
            assert np.array_equal(o_got[o_mask], o_want[o_mask]), "bytes of the batch that regrew the descriptor buffer"
            assert (o_got[~o_mask] == 0x5A).all()
            d_out.fill_(0x5A)
            torch.cuda.synchronize()


@pytest.mark.parametrize("mode", ["one_walk", "two_pass"])
def test_whole_stage_device_call_in_every_mode(ctx, port, mode, monkeypatch):
    """ohp_run_streams_device's default, one walk per stream into bounded regions, and its fallback, the round-1 count +
    scan + emit path (OHP_ONE_WALK=0): same bytes, same sizes, same count, with and without the chunk total."""
    import torch
    monkeypatch.setenv("OHP_ONE_WALK", "1" if mode == "one_walk" else "0")
    for w in (workloads.config4(n_streams=120, seconds=0.12, seed=3), workloads.elements(4, n_streams=60), workloads.config5(n_streams=90, seconds=0.1)):
        inp = port.fill_pcm(w.in_bytes, w.seed)
        rc, want, chunks, _ = port.run(w.streams, w.events, inp, w.out_bytes)
        assert rc == 0
        host = capi.schedule_build(w.streams, w.events)
        d_streams = torch.from_numpy(w.streams.view(np.uint8).copy()).cuda()
        d_events = torch.from_numpy(w.events.view(np.uint8).copy()).cuda()
        d_in = torch.from_numpy(inp).cuda()
        d_out = torch.full((w.out_bytes + 16,), 0x5A, dtype=torch.uint8, device="cuda")
        d_outb = torch.zeros(len(w.streams), dtype=torch.int64, device="cuda")
        torch.cuda.synchronize()
        total = ctx.run_streams_device(d_streams.data_ptr(), len(w.streams), d_events.data_ptr(), len(w.events),
                                       d_in.data_ptr(), w.in_bytes, d_out.data_ptr(), w.out_bytes, d_outb.data_ptr())
        ctx.sync()
        assert total == len(chunks)
        assert np.array_equal(d_outb.cpu().numpy().view(np.uint64), host.stream_out_bytes)
        got = d_out.cpu().numpy()[:w.out_bytes]
        mask = covered_mask(chunks, w.out_bytes)
        assert np.array_equal(got[mask], want[mask]) and (got[~mask] == 0x5A).all()
        # fully asynchronous (no chunk total asked for): same bytes
        d_out.fill_(0x5A)
        torch.cuda.synchronize()
        assert ctx.run_streams_device(d_streams.data_ptr(), len(w.streams), d_events.data_ptr(), len(w.events), d_in.data_ptr(), w.in_bytes,
                                      d_out.data_ptr(), w.out_bytes, 0, None, want_total=False) is None
        ctx.sync()
        got = d_out.cpu().numpy()[:w.out_bytes]
        assert np.array_equal(got[mask], want[mask]) and (got[~mask] == 0x5A).all()


def test_whole_stage_device_call_reports_errors(ctx):
    import torch
    w = workloads.config5(n_streams=4, seconds=0.02)
    bad = w.streams.copy()
    bad["sample_rate"][1] = 12345
    d_in = torch.zeros(w.in_bytes + 16, dtype=torch.uint8, device="cuda")
    d_out = torch.zeros(w.out_bytes + 16, dtype=torch.uint8, device="cuda")
    d_e = torch.from_numpy(w.events.view(np.uint8).copy()).cuda()
    d_bad = torch.from_numpy(bad.view(np.uint8).copy()).cuda()
    d_ok = torch.from_numpy(w.streams.view(np.uint8).copy()).cuda()
    torch.cuda.synchronize()
    with pytest.raises(capi.OhpError) as e:
        ctx.run_streams_device(d_bad.data_ptr(), 4, d_e.data_ptr(), len(w.events), d_in.data_ptr(), w.in_bytes, d_out.data_ptr(), w.out_bytes)
    assert e.value.status == abi.E_INVALID_ARG and "stream 1" in str(e.value)
    # a stream reaching outside the output arena is caught chunk by chunk on the device and reported by the sync
    ctx.run_streams_device(d_ok.data_ptr(), 4, d_e.data_ptr(), len(w.events), d_in.data_ptr(), w.in_bytes, d_out.data_ptr(), w.out_bytes // 2)
    with pytest.raises(capi.OhpError) as e:
        ctx.sync()
    assert e.value.status == abi.E_OUT_OF_RANGE
    assert ctx.run_streams_device(d_ok.data_ptr(), 4, d_e.data_ptr(), len(w.events), d_in.data_ptr(), w.in_bytes, d_out.data_ptr(), w.out_bytes) > 0
    ctx.sync()


def test_whole_stage_device_call_is_the_first_thing_a_context_does(port):
    """A fresh context has no descriptor buffer: the walk that is normally launched before the host knows the regions'
    total has nowhere to write yet, and must wait for it."""
    import torch
    ctx = capi.Context(0)
    try:
        w = workloads.config5(n_streams=40, seconds=0.05)
        inp = port.fill_pcm(w.in_bytes, w.seed)
        rc, want, chunks, _ = port.run(w.streams, w.events, inp, w.out_bytes)
        assert rc == 0
        d_streams = torch.from_numpy(w.streams.view(np.uint8).copy()).cuda()
        d_events = torch.from_numpy(w.events.view(np.uint8).copy()).cuda()
        d_in = torch.from_numpy(inp).cuda()
        d_out = torch.zeros(w.out_bytes + 16, dtype=torch.uint8, device="cuda")
        torch.cuda.synchronize()
        assert ctx.run_streams_device(d_streams.data_ptr(), len(w.streams), d_events.data_ptr(), len(w.events), d_in.data_ptr(), w.in_bytes,
                                      d_out.data_ptr(), w.out_bytes, 0, None, want_total=False) is None
        ctx.sync()
        mask = covered_mask(chunks, w.out_bytes)
        assert np.array_equal(d_out.cpu().numpy()[:w.out_bytes][mask], want[mask])
        assert ctx.run_streams_device(d_streams.data_ptr(), len(w.streams), d_events.data_ptr(), len(w.events), d_in.data_ptr(), w.in_bytes,
                                      d_out.data_ptr(), w.out_bytes) == len(chunks)
        ctx.sync()
    finally:
        ctx.close()
