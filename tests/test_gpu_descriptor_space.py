"""The hot path over its whole descriptor space on the GPU: every batch of descriptor_space.py (every depth x 1-32
channels x every packed-sink mode at every (head, destination phase) pair, the converting sinks at 1-32 channels, silence
around write_silence's blocks, every ramp length of 16-bit mono up to 4608 frames and of 8-bit mono up to 9216) through
ohp_process_device with both compiled loaders and once through ohp_process_host, against the C oracle; then streams at
9-32 channels through the whole stage, and their starvations, which the flywheel (at most 8 channels) does not play.

Every call: the status is clean, every byte a chunk covers is the oracle's, every other byte of the arena still holds
the fill, and 4 KiB guard bands either side of the arena are untouched.  A mismatch names the chunk and its cell."""
import os
import subprocess
import sys

import numpy as np
import pytest

from ohpipeline_b200 import capi
import descriptor_space as D

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
GUARD = 4096
FILL = 0xA5
KEYS = ("OHP_SERIAL_PLACE", "OHP_CAP_CHUNKS", "OHP_CAP_BYTES", "OHP_CHUNK_BLOCK", "OHP_AUTOTUNE")


@pytest.fixture
def configured(monkeypatch):
    """configured(cfg) -> a fresh context created under exactly these settings (the previous one is closed)."""
    opened = []

    def make(cfg):
        while opened:
            opened.pop().close()
        for k in KEYS:
            monkeypatch.delenv(k, raising=False)
        monkeypatch.setenv("OHP_AUTOTUNE", "0")
        for k, v in cfg.items():
            monkeypatch.setenv(k, str(v))
        opened.append(capi.Context(0))
        return opened[-1]

    yield make
    while opened:
        opened.pop().close()


@pytest.fixture(scope="module")
def matrix(port):
    """The batches with the oracle's output of each (uncovered bytes: the fill)."""
    out = []
    for b in D.batches(port):
        assert capi.validate(b.descs, b.in_bytes, b.out_bytes) == (0, 0), b.name   # nothing invalid goes to the GPU
        rc, want = port.process_chunks(b.descs, b.inp[:b.in_bytes], b.out_bytes)
        assert rc == 0, (b.name, -rc - 1)
        want[~D.covered(b.descs, b.out_bytes)] = FILL
        b.want = want
        out.append(b)
    return out


def check_arena(buf, want, descs, what):
    assert (buf[:GUARD] == FILL).all(), "%s: wrote below the arena" % what
    assert (buf[GUARD + len(want):] == FILL).all(), "%s: wrote past the arena" % what
    got = buf[GUARD:GUARD + len(want)]
    if np.array_equal(got, want):
        return
    bad = np.nonzero(got != want)[0]
    i = int(bad[0])
    k = D.owner(descs, i)
    if k < 0:
        raise AssertionError("%s: byte %d outside every chunk changed (%#x), %d bytes differ" % (what, i, got[i], len(bad)))
    cls = D.classify(descs)
    wrong = sorted({D.owner(descs, int(j)) for j in bad[:4096:64]})
    raise AssertionError("%s: %d bytes differ; first at output byte %d (got %#x want %#x), %d bytes into chunk %d: %s -- %s; "
                         "chunks with differences include %s" % (
                             what, len(bad), i, got[i], want[i], i - int(descs[k]["dst_off"]), k, descs[k],
                             D.describe(cls[k]), [(j, D.describe(cls[j])) for j in wrong[:6]]))


@pytest.mark.parametrize("serial", [0, 1], ids=["scan_place", "serial_place"])
def test_matrix_through_ohp_process_device(configured, matrix, serial):
    import torch
    ctx = configured(dict(OHP_SERIAL_PLACE=serial))
    for b in matrix:
        d_desc = torch.from_numpy(b.descs.view(np.uint8).copy()).cuda()
        d_in = torch.from_numpy(b.inp).cuda()
        assert d_in.data_ptr() % 16 == 0          # so that every chunk's head is the one classify() saw
        d_out = torch.full((b.out_bytes + 2 * GUARD,), FILL, dtype=torch.uint8, device="cuda")
        assert (d_out.data_ptr() + GUARD) % 16 == 0   # ... and its destination phase
        torch.cuda.synchronize()
        st = torch.cuda.current_stream().cuda_stream
        ctx.process_device(d_desc.data_ptr(), len(b.descs), d_in.data_ptr(), b.in_bytes, d_out.data_ptr() + GUARD, b.out_bytes, st)
        ctx.sync(st)
        check_arena(d_out.cpu().numpy(), b.want, b.descs, "%s, OHP_SERIAL_PLACE=%d" % (b.name, serial))
        del d_desc, d_in, d_out


def test_matrix_through_ohp_process_host(ctx, matrix):
    for b in matrix:
        buf = np.full(b.out_bytes + 2 * GUARD, FILL, dtype=np.uint8)
        ctx.process_host(b.descs, b.inp[:b.in_bytes], buf[GUARD:GUARD + b.out_bytes])
        check_arena(buf, b.want, b.descs, "%s, ohp_process_host" % b.name)


# ------------------------------------------------------------------------------------------------------------------
# the stage at 9-32 channels

@pytest.fixture(scope="module")
def wide(port):
    """(workload, input, the oracle's end-to-end output with the fill where no chunk writes, the oracle's descriptors)."""
    out = []
    for w in D.wide_streams():
        inp = port.fill_pcm(w.in_bytes, w.seed)
        rc, want, chunks, _ = port.run(w.streams, w.events, inp, w.out_bytes)
        assert rc == 0, w.name
        want[~D.covered(chunks, w.out_bytes)] = FILL
        out.append((w, inp, want, chunks))
    return out


def same_schedule(dev, host, what):
    assert np.array_equal(dev.stream_chunk_begin, host.stream_chunk_begin), what
    assert np.array_equal(dev.stream_out_bytes, host.stream_out_bytes), what
    if not np.array_equal(dev.chunks, host.chunks):
        i = int(np.nonzero(dev.chunks != host.chunks)[0][0])
        raise AssertionError("%s: descriptor %d differs: device %s host %s" % (what, i, dev.chunks[i], host.chunks[i]))
    assert np.array_equal(dev.info, host.info), what


def stage(ctx, w, inp, want, chunks):
    """The device walk against the host model, then both whole-stage calls against the oracle."""
    import torch
    same_schedule(ctx.schedule_build_device(w.streams, w.events), capi.schedule_build(w.streams, w.events), w.name)
    d_streams = torch.from_numpy(w.streams.view(np.uint8).copy()).cuda()
    d_events = torch.from_numpy(w.events.view(np.uint8).copy()).cuda()
    d_in = torch.from_numpy(inp).cuda()
    d_out = torch.full((w.out_bytes + 2 * GUARD,), FILL, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    total = ctx.run_streams_device(d_streams.data_ptr(), len(w.streams), d_events.data_ptr(), len(w.events), d_in.data_ptr(),
                                   w.in_bytes, d_out.data_ptr() + GUARD, w.out_bytes)
    ctx.sync()
    assert total == len(chunks), w.name
    check_arena(d_out.cpu().numpy(), want, chunks, "run_streams_device " + w.name)
    buf = np.full(w.out_bytes + 2 * GUARD, FILL, dtype=np.uint8)
    _, total = ctx.run_streams_host(w.streams, w.events, inp, buf[GUARD:GUARD + w.out_bytes])
    assert total == len(chunks), w.name
    check_arena(buf, want, chunks, "run_streams_host " + w.name)


def test_wide_streams_through_the_whole_stage(ctx, wide):
    for w, inp, want, chunks in wide:
        stage(ctx, w, inp, want, chunks)


def walk_child():
    """Runs in the child: stage() on every batch of wide streams."""
    from oracle import pyoracle
    port = pyoracle.Port()
    ctx = capi.Context(0)
    try:
        for w in D.wide_streams():
            inp = port.fill_pcm(w.in_bytes, w.seed)
            rc, want, chunks, _ = port.run(w.streams, w.events, inp, w.out_bytes)
            assert rc == 0, w.name
            want[~D.covered(chunks, w.out_bytes)] = FILL
            stage(ctx, w, inp, want, chunks)
    finally:
        ctx.close()


@pytest.mark.parametrize("team", [1, 32], ids=["team1", "team32"])
def test_wide_streams_in_every_walk_team_setting(team):
    """OHP_SCHED_TEAM is read once per process: a thread per stream, or a warp per stream, each in a child process."""
    env = {k: v for k, v in os.environ.items() if not k.startswith("OHP_")}
    env["OHP_SCHED_TEAM"] = str(team)
    env["PYTHONPATH"] = os.pathsep.join([ROOT, HERE] + ([env["PYTHONPATH"]] if env.get("PYTHONPATH") else []))
    r = subprocess.run([sys.executable, "-c", "import test_gpu_descriptor_space as t; t.walk_child()"], cwd=ROOT, env=env,
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-4000:] + r.stderr[-4000:]


def test_starvations_above_the_flywheel_channels_play_nothing(ctx, port):
    """RampGenerator::kMaxChannels is 8: a StarvationRamper on a 9-32 channel stream records its starvations and plays no
    flywheel audio.  Both flywheel calls write the host route's records, plan nothing, leave the flywheel arena's fill and
    write the stream bytes ohp_run_streams_device writes."""
    import test_gpu_starvations as base
    import test_gpu_starvations_recent as recent
    starved = 0
    for w in D.wide_streams():
        sv = capi.schedule_build(w.streams, w.events).starvations
        if not len(sv):
            continue
        assert len(capi.flywheel_plan_batch(w.streams, sv).planned) == 0, w.name
        starved += len(sv)
        _, r = base.check(ctx, w, port)
        assert np.all(r["len"] == 0) and np.all(r["fly"] == base.FLY_FILL), w.name
        _, r, _, _ = recent.check(ctx, w, port)
        assert np.all(r["len"] == 0) and np.all(r["fly"] == base.FLY_FILL), w.name
    assert starved >= 20, starved
