"""The stage past 32 bits on the GPU: the device walk on streams longer than 2^32 jiffies and on the FP64 recurrence's
edge cases in every walk configuration, the whole stage against the C oracle on those streams, arenas past 4 GiB
(descriptors, streams and checksum ranges above and across 2^32, sentinels where a truncated address would land) and
one MsgSilence of 2^32 - 1 bytes.  Device memory peaks near 9 GiB; every test frees what it allocated."""
import os
import subprocess
import sys

import numpy as np
import pytest

from ohpipeline_b200 import abi, capi
from long_util import T32, far_arena_layout, fp64_edge_streams, long_streams, split
from util import covered_mask, make_desc

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
FILL = 0x5A


def dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).reshape(-1).copy()).cuda()


def same_schedule(got, want, name):
    assert np.array_equal(got.stream_chunk_begin, want.stream_chunk_begin), name
    assert np.array_equal(got.stream_out_bytes, want.stream_out_bytes), name
    assert np.array_equal(got.chunks, want.chunks), name
    assert np.array_equal(got.info, want.info), name


def child():
    """Runs in a child process with the walk configuration in its environment: the device walk against the host walk
    (ohp_schedule_count_device + ohp_schedule_emit_device), and ohp_run_streams_device -- where OHP_ONE_WALK and
    OHP_SCHED_TEAM choose the walk -- against the host model's sizes and the oracle's bytes, on both generators."""
    import torch
    from oracle import pyoracle
    port = pyoracle.Port()
    ctx = capi.Context(0)
    try:
        for name, w in (("long", long_streams()), ("fp64", fp64_edge_streams()[0])):
            host = capi.schedule_build(w.streams, w.events, walk=True)
            same_schedule(ctx.schedule_build_device(w.streams, w.events), host, name)
            inp = port.fill_pcm(w.in_bytes, w.seed)
            rc, want, chunks, _ = port.run(w.streams, w.events, inp, w.out_bytes)
            assert rc == 0, name
            d_streams, d_events, d_in = dev(w.streams), dev(w.events), dev(inp)
            d_out = torch.full((w.out_bytes,), FILL, dtype=torch.uint8, device="cuda")
            d_outb = torch.zeros(len(w.streams), dtype=torch.int64, device="cuda")
            torch.cuda.synchronize()
            total = ctx.run_streams_device(d_streams.data_ptr(), len(w.streams), d_events.data_ptr(), len(w.events),
                                           d_in.data_ptr(), inp.size, d_out.data_ptr(), w.out_bytes, d_outb.data_ptr())
            ctx.sync()
            assert total == len(host.chunks), name
            assert np.array_equal(d_outb.cpu().numpy().view(np.uint64), host.stream_out_bytes), name
            got = d_out.cpu().numpy()
            mask = covered_mask(chunks, w.out_bytes)
            assert np.array_equal(got[mask], want[mask]) and np.all(got[~mask] == FILL), name
            del d_streams, d_events, d_in, d_out, d_outb
            torch.cuda.empty_cache()
    finally:
        ctx.close()


@pytest.mark.parametrize("env", [{}, {"OHP_ONE_WALK": "0"}, {"OHP_SCHED_TEAM": "1"}, {"OHP_SCHED_TEAM": "32"}],
                         ids=["default", "two_pass", "team1", "team32"])
def test_device_walk_equals_the_host_walk(env):
    """default: one walk per stream inside ohp_run_streams_device; OHP_ONE_WALK=0: count and emit in two passes.  With
    OHP_SCHED_TEAM=32 a warp walks each stream, so every fp64_edge_streams() message k >= 1 of a ramp goes through the
    FP64 branch: the streams are uniform (no codec block reads), their messages are below 2^21 jiffies, one
    stage ramps and no other event, silence or size cap cuts the run (the generator's docstring)."""
    e = {k: v for k, v in os.environ.items() if not k.startswith("OHP_")}
    e.update(env)
    e["PYTHONPATH"] = os.pathsep.join([ROOT, HERE] + ([e["PYTHONPATH"]] if e.get("PYTHONPATH") else []))
    r = subprocess.run([sys.executable, "-c", "import test_gpu_long_streams as t; t.child()"], cwd=ROOT, env=e,
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-4000:] + r.stderr[-4000:]


def test_whole_stage_on_long_streams_equals_the_oracle(ctx, port):
    import torch
    w = long_streams()
    inp = port.fill_pcm(w.in_bytes, w.seed)
    rc, want, chunks, _ = port.run(w.streams, w.events, inp, w.out_bytes)
    assert rc == 0
    model = capi.schedule_build(w.streams, w.events)
    d_streams, d_events, d_in = dev(w.streams), dev(w.events), dev(inp)
    d_out = torch.full((w.out_bytes,), FILL, dtype=torch.uint8, device="cuda")
    d_outb = torch.zeros(len(w.streams), dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    total = ctx.run_streams_device(d_streams.data_ptr(), len(w.streams), d_events.data_ptr(), len(w.events), d_in.data_ptr(),
                                   inp.size, d_out.data_ptr(), w.out_bytes, d_outb.data_ptr())
    ctx.sync()
    assert total == len(model.chunks)
    assert np.array_equal(d_outb.cpu().numpy().view(np.uint64), model.stream_out_bytes)
    got = d_out.cpu().numpy()
    mask = np.zeros(w.out_bytes, dtype=bool)
    for d, n in zip(chunks, abi.chunk_out_bytes(chunks)):
        mask[int(d["dst_off"]):int(d["dst_off"]) + int(n)] = True
    assert np.array_equal(got[mask], want[mask]) and np.all(got[~mask] == FILL)
    del d_streams, d_events, d_in, d_out, d_outb
    torch.cuda.empty_cache()


def test_flywheel_on_long_streams_equals_the_oracle_route(ctx, port):
    """The streams with a StarvationRamper, through ohp_run_streams_device_flywheel and _flywheel_recent
    (test_gpu_starvations_recent.check): the device walk's records past 2^32 (recent_jiffies saturated) and its pieces of
    recent audio as the class model keeps them, every played slot as the oracle route and the host route play it."""
    from test_gpu_starvations_recent import check
    w = long_streams()
    starving = {int(s) for s in np.unique(np.searchsorted(w.streams["first_event"].astype(np.int64),
                                                          np.nonzero(w.events["op"] == abi.EV_STARVATION)[0], side="right") - 1)}
    sub = split(w, lambda k: k in starving)
    sched, r, old, _ = check(ctx, sub, port)
    sv = sched.starvations
    assert (sv["pcm_jiffies"] > T32).sum() >= 20 and (sv["recent_jiffies"] == 0xFFFFFFFF).any()
    assert int((old["len"] != 0).sum()) >= 10 and int((r["len"] != 0).sum()) >= int((old["len"] != 0).sum())


def test_flywheel_jobs_past_4_gib_equal_the_oracle(ctx, port):
    """ohp_flywheel_device with training blocks and outputs at and across 2^32, against the oracle on the same jobs
    rebased to 0 (offsets mod 16 kept); what no job covers keeps its fill, below the batch and at offset mod 2^32 too."""
    import torch
    import test_gpu_flywheel as fw
    jobs, inp, out_len = fw.batch(["tone", "noise", "step"], fw.SHAPES, seed=900)
    rc, want = port.flywheel(jobs, inp, out_len)
    assert rc == 0
    mask = fw.covered(jobs, out_len)
    arena = T32 + (8 << 20)
    for shift_in, shift_out in ((T32 - 4096, T32 - 1024), (T32 + 4096, T32 + 32)):
        far = jobs.copy()
        far["src_off"] += np.uint64(shift_in)
        far["dst_off"] += np.uint64(shift_out)
        assert capi.flywheel_validate(far, arena, arena)[0] == abi.OK
        d_in = torch.zeros(arena, dtype=torch.uint8, device="cuda")
        d_out = torch.full((arena,), FILL, dtype=torch.uint8, device="cuda")
        d_in[shift_in:shift_in + inp.size] = torch.from_numpy(inp).cuda()
        d_jobs = dev(far)
        torch.cuda.synchronize()
        ctx.flywheel_device(d_jobs.data_ptr(), len(far), d_in.data_ptr(), arena, d_out.data_ptr(), arena)
        ctx.sync()
        got = d_out[shift_out:shift_out + out_len].cpu().numpy()
        fw.assert_jobs_match(got, want, jobs, mask, "far jobs")
        assert np.all(got[~mask] == FILL)
        for s in {0, 1, shift_out - 1, shift_out % T32, (shift_out + out_len) % T32, 4095}:
            if not shift_out <= s < shift_out + out_len:
                assert int(d_out[s].item()) == FILL, s
        del d_in, d_out, d_jobs
        torch.cuda.empty_cache()


def every_sink_descs():
    """Four descriptors per sink (P1, P2, planar, from-32, Songcast; silence into P1), at every offset mod 16, laid out
    from 0 in both arenas -> (descs, in_len, out_len)."""
    specs = []
    rng = np.random.default_rng(77)
    for fmt, bits, ch, aux in ((abi.OUT_PACKED_BE, 16, 2, 0), (abi.OUT_PACKED_LE, 24, 2, abi.LE_APPEND), (abi.OUT_PLANAR32_BE, 16, 3, 0),
                               (abi.OUT_FROM32_BE, 32, 2, 24), (abi.OUT_SONGCAST, 24, 6, 0), (abi.OUT_PACKED_BE, 8, 6, 0)):
        for k in range(4):
            frames = int(rng.integers(40, 9216 // (ch * bits // 8)))
            flags = (abi.F_RAMP_ENABLED if k % 2 else 0) | (abi.F_IN_LITTLE_ENDIAN if k == 2 else 0)
            if fmt == abi.OUT_PACKED_BE and bits == 8 and k == 3:
                flags = abi.F_SILENCE
            specs.append(dict(bytes=frames * ch * bits // 8, bit_depth=bits, channels=ch, out_fmt=fmt, flags=flags,
                              aux=frames if fmt == abi.OUT_PLANAR32_BE else aux,
                              ramp_start=int(rng.integers(0, 16385)), ramp_end=int(rng.integers(0, 16385))))
    descs = np.zeros(len(specs), dtype=abi.CHUNK_DESC)
    src = dst = 0
    for i, c in enumerate(specs):
        d = make_desc(**c)
        src += int(rng.integers(0, 16))
        dst += int(rng.integers(0, 16))
        d["src_off"], d["dst_off"] = src, dst
        descs[i] = d[0]
        if not (c["flags"] & abi.F_SILENCE):
            src += c["bytes"]
        dst += int(abi.chunk_out_bytes(d)[0])
    return descs, src + 64, dst + 64


def test_descriptors_past_4_gib_equal_the_oracle(ctx, port):
    """ohp_process_device with src_off / dst_off at and across 2^32 over every sink, against the oracle on the same
    descriptors rebased to 0 (offsets mod 16 kept); sentinels below the batch and at offset mod 2^32 stay untouched."""
    import torch
    descs, in_len, out_len = every_sink_descs()
    inp = port.fill_pcm(in_len, 4242)
    rc, want = port.process_chunks(descs, inp, out_len)
    assert rc == 0
    mask = covered_mask(descs, out_len)
    arena = T32 + (8 << 20)
    for shift_in, shift_out in ((T32 - 4096, T32 - 2048), (T32 + 4096 + 32, T32 + 16)):
        far = descs.copy()
        far["src_off"] += np.uint64(shift_in)
        far["dst_off"] += np.uint64(shift_out)
        assert capi.validate(far, arena, arena)[0] == abi.OK
        d_in = torch.zeros(arena, dtype=torch.uint8, device="cuda")
        d_out = torch.full((arena,), FILL, dtype=torch.uint8, device="cuda")
        d_in[shift_in:shift_in + in_len] = torch.from_numpy(inp).cuda()
        d_desc = dev(far)
        torch.cuda.synchronize()
        ctx.process_device(d_desc.data_ptr(), len(far), d_in.data_ptr(), arena, d_out.data_ptr(), arena)
        ctx.sync()
        got = d_out[shift_out:shift_out + out_len].cpu().numpy()
        assert np.array_equal(got[mask], want[mask]) and np.all(got[~mask] == FILL), (shift_in, shift_out)
        for s in {0, 1, shift_out - 1, shift_out % T32, (shift_out + out_len) % T32, 4095, 16}:
            if not shift_out <= s < shift_out + out_len:
                assert int(d_out[s].item()) == FILL, s
        del d_in, d_out, d_desc
        torch.cuda.empty_cache()


def test_streams_past_4_gib_equal_the_oracle(ctx, port):
    """ohp_fill_streams_device and ohp_run_streams_device on far_arena_layout (one stream across 2^32 in each arena,
    the rest above it), ohp_checksums_device over ranges above 2^32, and ohp_run_streams_host with a pageable host
    output of the same size: the bytes of each stream are the oracle's on the layout rebased to 0; sentinels stay."""
    import torch
    from ohpipeline_b200 import workloads as W
    w = W.config4(n_streams=48, seconds=0.1, seed=11)
    st, in_bytes, out_bytes, s_in, s_out = far_arena_layout(w)
    seed = 0x1234 << 32
    inp0 = port.fill_streams(w.streams, w.in_bytes, seed)
    rc, want, _, _ = port.run(w.streams, w.events, inp0, w.out_bytes)
    assert rc == 0
    model = capi.schedule_build(w.streams, w.events)
    outb = model.stream_out_bytes
    d_in = torch.full((in_bytes,), FILL, dtype=torch.uint8, device="cuda")
    d_out = torch.full((out_bytes,), FILL, dtype=torch.uint8, device="cuda")
    d_streams, d_events = dev(st), dev(w.events)
    torch.cuda.synchronize()
    ctx.fill_streams_device(d_in.data_ptr(), in_bytes, d_streams.data_ptr(), len(st), seed)
    ctx.run_streams_device(d_streams.data_ptr(), len(st), d_events.data_ptr(), len(w.events), d_in.data_ptr(), in_bytes,
                           d_out.data_ptr(), out_bytes)
    ctx.sync()
    fb = st["channels"].astype(np.int64) * (st["bit_depth"].astype(np.int64) // 8)
    for k in range(len(st)):
        a, n = int(st["src_base"][k]), int(st["total_frames"][k]) * int(fb[k])
        o = int(w.streams["src_base"][k])
        assert np.array_equal(d_in[a:a + n].cpu().numpy(), inp0[o:o + n]), ("input", k)
        a, n, o = int(st["dst_base"][k]), int(outb[k]), int(w.streams["dst_base"][k])
        assert np.array_equal(d_out[a:a + n].cpu().numpy(), want[o:o + n]), ("output", k)
    assert all(int(d_in[int(s)].item()) == FILL for s in s_in)
    assert all(int(d_out[int(s)].item()) == FILL for s in s_out)
    # checksums over the far ranges: streams 2.. lie above 2^32 (stream 1 straddles it in the output arena)
    d_sums = torch.zeros(len(st), dtype=torch.int64, device="cuda")
    tiling = np.concatenate([st["dst_base"][2:].astype(np.uint64), [np.uint64(int(st["dst_base"][-1]) + int(outb[-1]))]])
    assert int(tiling[0]) > T32
    d_tile = dev(tiling)
    torch.cuda.synchronize()
    ctx.checksums_device(d_out.data_ptr(), d_tile.data_ptr(), len(st) - 2, d_sums.data_ptr())
    ctx.sync()
    sums = d_sums.cpu().numpy().view(np.uint64)
    for k in range(len(st) - 2):
        a, b = int(tiling[k]), int(tiling[k + 1])
        assert int(sums[k]) == port.checksum(d_out[a:b].cpu().numpy()), k
    del d_in, d_out, d_streams, d_events, d_sums, d_tile
    torch.cuda.empty_cache()
    # the host route: pageable numpy buffers of the same size, only covered bytes change
    h_in = np.zeros(in_bytes, dtype=np.uint8)
    for k in range(len(st)):
        a, n, o = int(st["src_base"][k]), int(st["total_frames"][k]) * int(fb[k]), int(w.streams["src_base"][k])
        h_in[a:a + n] = inp0[o:o + n]
    h_out = np.full(out_bytes, FILL, dtype=np.uint8)
    got_outb, _ = ctx.run_streams_host(st, w.events, h_in, h_out)
    assert np.array_equal(got_outb, outb)
    changed = 0
    for k in range(len(st)):
        a, n, o = int(st["dst_base"][k]), int(outb[k]), int(w.streams["dst_base"][k])
        assert np.array_equal(h_out[a:a + n], want[o:o + n]), ("host", k)
        changed += int(np.count_nonzero(h_out[a:a + n] != FILL))
    assert int(np.count_nonzero(h_out != FILL)) == changed       # nothing outside the streams, zeros included
    del h_in, h_out


def test_one_huge_silence_descriptor(ctx):
    """MsgSilence of 2^32 - 1 bytes, 8-bit mono, into the packed big-endian sink (check_desc_fields bounds silence only
    for converting sinks), with a 6-channel silence of about 2^31 bytes beside it: write_silence walks each with one warp
    and 32-bit counters that stay below 2^32 (words < 2^28, i0 + 15 < bytes).  Checked on the device: all zeros, and
    the 6-channel tag 00 00 00 c0 at the start of every 9216-byte block (MsgPlayableSilence::ReadBlock)."""
    import torch
    big = T32 - 1
    six_bytes = ((1 << 31) + 12345) // (6 * 2) * (6 * 2)          # whole 16-bit 6-channel frames
    six_off = big + 16 + 3                                          # unaligned start
    out_bytes = six_off + six_bytes + 64
    descs = np.concatenate([make_desc(bytes=big, bit_depth=8, channels=1, flags=abi.F_SILENCE, dst_off=0),
                            make_desc(bytes=six_bytes, bit_depth=16, channels=6, flags=abi.F_SILENCE, dst_off=six_off)])
    assert capi.validate(descs, 16, out_bytes)[0] == abi.OK
    d_out = torch.full((out_bytes,), FILL, dtype=torch.uint8, device="cuda")
    d_in = torch.zeros(16, dtype=torch.uint8, device="cuda")
    d_desc = dev(descs)
    torch.cuda.synchronize()
    ctx.process_device(d_desc.data_ptr(), 2, d_in.data_ptr(), 16, d_out.data_ptr(), out_bytes)
    ctx.sync()
    assert int(torch.count_nonzero(d_out[:big]).item()) == 0
    assert int(d_out[big].item()) == FILL and int(d_out[big + 1:six_off].ne(FILL).sum().item()) == 0
    six = d_out[six_off:six_off + six_bytes]
    block = 9216 - 9216 % 12
    r = torch.arange(block, device="cuda")
    pattern = torch.where((r < 32) & (r % 4 == 3), (r // 4) * 16, torch.zeros_like(r)).to(torch.uint8)
    whole = six_bytes // block * block
    assert bool(torch.equal(six[:whole].view(-1, block), pattern.expand(whole // block, block)))
    assert bool(torch.equal(six[whole:], pattern[:six_bytes - whole]))
    for b in ((1 << 31) // block * block, (1 << 31) // block * block + block, six_bytes // block * block):
        if b + 32 <= six_bytes:
            assert six[b:b + 32].cpu().numpy().tolist() == [0, 0, 0, 0, 0, 0, 0, 0x10, 0, 0, 0, 0x20, 0, 0, 0, 0x30,
                                                            0, 0, 0, 0x40, 0, 0, 0, 0x50, 0, 0, 0, 0x60, 0, 0, 0, 0x70][:32], b
    assert int(d_out[six_off + six_bytes:].ne(FILL).sum().item()) == 0
    del d_out, d_in, d_desc, six, r, pattern
    torch.cuda.empty_cache()


def test_offsets_near_2_64_are_refused(ctx, port):
    """src_off / dst_off within a chunk of 2^64: ohp_validate and the device check refuse them with OHP_E_OUT_OF_RANGE
    (the bounds are compared without an addition that could wrap), and the context then runs a valid batch cleanly."""
    import torch
    top = (1 << 64) - 1
    for field, off in (("src_off", top - 15), ("dst_off", top - 15), ("src_off", top - 9215), ("dst_off", top)):
        d = make_desc(bytes=64, bit_depth=16, channels=2)
        d[field] = off
        assert capi.validate(d, 1 << 20, 1 << 20) == (abi.E_OUT_OF_RANGE, 0), (field, off)
        d_desc, d_in = dev(d), torch.zeros(1 << 20, dtype=torch.uint8, device="cuda")
        d_out = torch.zeros(1 << 20, dtype=torch.uint8, device="cuda")
        torch.cuda.synchronize()
        with pytest.raises(capi.OhpError) as e:
            ctx.process_device(d_desc.data_ptr(), 1, d_in.data_ptr(), 1 << 20, d_out.data_ptr(), 1 << 20)
            ctx.sync()
        assert e.value.status == abi.E_OUT_OF_RANGE
    job = capi.flywheel_job(48000, 2, 16, src_off=top - 15, dst_off=0)
    assert capi.flywheel_validate(job, 1 << 20, 1 << 20)[0] == abi.E_OUT_OF_RANGE
    job = capi.flywheel_job(48000, 2, 16, src_off=0, dst_off=top - 15)
    assert capi.flywheel_validate(job, 1 << 20, 1 << 20)[0] == abi.E_OUT_OF_RANGE
    torch.cuda.synchronize()
    descs, in_len, out_len = every_sink_descs()
    inp = port.fill_pcm(in_len, 99)
    rc, want = port.process_chunks(descs, inp, out_len)
    got = np.zeros(out_len, dtype=np.uint8)
    ctx.process_host(descs, inp, got)
    assert rc == 0 and np.array_equal(got, want)
