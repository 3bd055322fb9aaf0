"""The hot path in every launch configuration a context can pick at run time, against the C oracle.

A context decides per batch how ramp_convert_kernel is launched: which placement loop its loader warp runs
(ramp_convert_kernel<true> places chunks in the ring one at a time, <false> a warp-wide scan at a time), how many chunks a
CTA keeps in flight, how many ring bytes they may take, and in runs of how many consecutive chunks the batch is dealt to
the CTAs.  The tuner picks the first two by timing three candidates on large batches, and the run length is halved on
small ones, so the same batch runs differently from box to box and from size to size; the bytes must never depend on it.
ohp_create reads the same settings from OHP_SERIAL_PLACE, OHP_CAP_CHUNKS, OHP_CAP_BYTES and OHP_CHUNK_BLOCK (OHP_AUTOTUNE=0
keeps the tuner out), and every test here creates a fresh context for each setting.  ohp_inflight_cap reads the
in-flight cap back, and the profiler names the kernel that ran; the byte cap and the run length cannot be read back.

The schedule walk's team and lane settings (OHP_SCHED_TEAM, OHP_SCHED_LANES) are read once per process, so each of them
runs in a child process of its own; they cannot be read back either.

Every call: the status is clean, every byte a chunk covers is the oracle's, every other byte of the arena still holds
the fill, and 4 KiB guard bands either side of the arena are untouched."""
import itertools
import os
import subprocess
import sys

import numpy as np
import pytest

from ohpipeline_b200 import abi, capi, workloads as W
from util import alignment_specs, covered_mask, describe_first_diff, make_desc, pack_chunks

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
GUARD = 4096
FILL = 0xA5
POISON = 0xEE
KEYS = ("OHP_SERIAL_PLACE", "OHP_CAP_CHUNKS", "OHP_CAP_BYTES", "OHP_CHUNK_BLOCK", "OHP_AUTOTUNE")
RING_SLOTS, RING_BYTES = 32, 105472
MIN_CAP_BYTES = 2 * (9216 + 16 + 80)    # two slots of the largest chunk: the least OHP_CAP_BYTES accepts

# the tuner's three candidates (kTuneCaps / kTuneSerial in ohp_capi.cu)
TUNER = [dict(OHP_SERIAL_PLACE=0, OHP_CAP_CHUNKS=32), dict(OHP_SERIAL_PLACE=1, OHP_CAP_CHUNKS=12),
         dict(OHP_SERIAL_PLACE=0, OHP_CAP_CHUNKS=24)]
# the edges of every setting, every combination
SWEEP = [dict(OHP_SERIAL_PLACE=s, OHP_CAP_CHUNKS=c, OHP_CAP_BYTES=b, OHP_CHUNK_BLOCK=k)
         for s, c, b, k in itertools.product((0, 1), (1, 2, 8, 31), (MIN_CAP_BYTES, 40000, RING_BYTES), (1, 3, 4, 16))]


def cfg_id(cfg):
    short = dict(OHP_SERIAL_PLACE="serial", OHP_CAP_CHUNKS="chunks", OHP_CAP_BYTES="bytes", OHP_CHUNK_BLOCK="block")
    return "-".join("%s%d" % (short[k], v) for k, v in cfg.items())


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


# ------------------------------------------------------------------------------------------------------------------
# batches of descriptors, each with its oracle output (computed once)

class Batch:
    def __init__(self, name, descs, inp, in_bytes, out_bytes, port):
        """inp may run past in_bytes (a poisoned tail the kernel must not use); in_bytes is what the kernel is told."""
        self.name, self.descs, self.in_bytes, self.out_bytes = name, np.ascontiguousarray(descs), int(in_bytes), int(out_bytes)
        self.inp = np.ascontiguousarray(inp)
        real = self.descs[abi.chunk_out_bytes(self.descs) > 0]  # (the oracle has no all-zero padding descriptor)
        rc, want = port.process_chunks(real, self.inp[:self.in_bytes], self.out_bytes)
        assert rc == 0, "%s: oracle rejected chunk %d" % (name, -rc - 1)
        mask = covered_mask(real, self.out_bytes)
        want[~mask] = FILL
        self.want = want
        self._dev = None

    def device(self):
        import torch
        if self._dev is None:
            self._dev = (torch.from_numpy(self.descs.view(np.uint8).copy()).cuda(), torch.from_numpy(self.inp).cuda())
        return self._dev


def from_workload(w, port, name):
    sched = capi.schedule_build(w.streams, w.events)
    return Batch(name, sched.chunks, port.fill_pcm(w.in_bytes, w.seed), w.in_bytes, w.out_bytes, port)


def max_size_chunks(rng):
    """9216-byte chunks of every format that divides it, at every source head offset mod 16, with 1-3 frame chunks
    between them."""
    formats = [(8, 1), (8, 3), (16, 2), (16, 6), (24, 2), (24, 4), (32, 2), (32, 8)]
    descs, src, dst = [], 0, 0
    for bits, ch in formats:
        fb = ch * bits // 8
        for head in range(16):
            flags = (abi.F_RAMP_ENABLED if head % 3 else 0) | (abi.F_IN_LITTLE_ENDIAN if head % 2 else 0)
            src += (head - src) % 16
            dst += int(rng.integers(0, 16))
            descs.append(make_desc(bytes=9216, bit_depth=bits, channels=ch, flags=flags, src_off=src, dst_off=dst,
                                   ramp_start=int(rng.integers(0, 16385)), ramp_end=int(rng.integers(0, 16385)),
                                   out_fmt=abi.OUT_PACKED_LE if (bits < 32 and head % 4 == 1) else abi.OUT_PACKED_BE,
                                   aux=abi.LE_APPEND if head % 8 == 1 else 0)[0])
            src += 9216
            dst += int(abi.chunk_out_bytes(np.array(descs[-1:], dtype=abi.CHUNK_DESC))[0])
            n = int(rng.integers(1, 4)) * fb
            descs.append(make_desc(bytes=n, bit_depth=bits, channels=ch, flags=flags ^ abi.F_RAMP_ENABLED, src_off=src,
                                   dst_off=dst, ramp_start=int(rng.integers(0, 16385)), ramp_end=int(rng.integers(0, 16385)))[0])
            src += n + int(rng.integers(0, 3))
            dst += n
    return np.array(descs, dtype=abi.CHUNK_DESC), src + 64, dst + 64


def sinks_and_silence(rng):
    """Silence two chunks in three, and every converting sink: planar 32-bit, 32-bit to packed, Songcast, packed LE in
    both modes."""
    specs = []
    for k in range(600):
        bits = int(rng.choice((8, 16, 24, 32)))
        ch = int(rng.integers(1, 9))
        fb = ch * bits // 8
        frames = int(rng.choice((1, 2, 17, int(rng.integers(1, 9216 // fb + 1)), 9216 // fb)))
        silence = rng.random() < 0.66
        sink = int(rng.integers(0, 5))
        flags = (abi.F_SILENCE if silence else 0) | (abi.F_RAMP_ENABLED if rng.random() < 0.6 else 0) \
            | (abi.F_IN_LITTLE_ENDIAN if rng.random() < 0.4 else 0)
        spec = dict(bytes=frames * fb, bit_depth=bits, channels=ch, flags=flags, ramp_start=int(rng.integers(0, 16385)),
                    ramp_end=int(rng.integers(0, 16385)), src_pad=int(rng.integers(0, 5)), dst_pad=int(rng.integers(0, 5)))
        if sink == 1:
            spec.update(out_fmt=abi.OUT_PLANAR32_BE, aux=frames + int(rng.integers(0, 3)))
        elif sink == 2 and not silence:
            frames = min(frames, 9216 // (4 * ch))
            spec.update(bit_depth=32, bytes=frames * ch * 4, out_fmt=abi.OUT_FROM32_BE, aux=int(rng.choice((8, 16, 24, 32))))
        elif sink == 3:
            spec.update(out_fmt=abi.OUT_SONGCAST, aux=int(rng.integers(0, ch - 1)) if ch > 2 else 0)
        elif sink == 4 and not silence and bits < 32:
            spec.update(out_fmt=abi.OUT_PACKED_LE, aux=int(rng.integers(0, 2)))
        specs.append(spec)
    return pack_chunks(specs)


def with_padding(descs, rng):
    """Zero-byte descriptors and all-zero padding descriptors (what ohp_run_streams_device fills a stream's region with)
    between the real ones."""
    out = []
    for d in descs:
        for _ in range(int(rng.integers(0, 3))):
            if rng.random() < 0.5:
                out.append(np.zeros(1, dtype=abi.CHUNK_DESC)[0])
            else:
                out.append(make_desc(bytes=0, bit_depth=int(rng.choice((8, 16, 24, 32))), channels=int(rng.integers(1, 9)),
                                     flags=int(rng.integers(0, 8)), dst_off=int(d["dst_off"]), src_off=int(d["src_off"]))[0])
        out.append(d)
    return np.array(out, dtype=abi.CHUNK_DESC)


def arena_tail(bits, port, rng):
    """in_bytes ends inside a 16-byte word, exactly where the last chunk ends; a few more chunks end in that word too.
    The bytes behind in_bytes are poison."""
    b = bits // 8
    specs = []
    for k in range(40):
        ch = int(rng.integers(1, 9))
        specs.append(dict(bytes=int(rng.integers(1, 200)) * ch * b, bit_depth=bits, channels=ch,
                          flags=(abi.F_RAMP_ENABLED if k % 2 else 0) | (abi.F_IN_LITTLE_ENDIAN if k % 3 == 0 else 0),
                          ramp_start=int(rng.integers(0, 16385)), ramp_end=int(rng.integers(0, 16385)),
                          src_pad=int(rng.integers(0, 7)), dst_pad=int(rng.integers(0, 7))))
    descs, _, out_bytes = pack_chunks(specs)
    last = descs[-1]
    in_bytes = int(last["src_off"]) + int(last["bytes"])
    if in_bytes % 16 == 0:                                   # move everything by one frame: mid-word
        descs["src_off"] += b
        in_bytes += b
    assert in_bytes % 16 != 0
    tail = []
    dst = out_bytes
    for fb in (b, 2 * b, 3 * b, 5 * b):                      # chunks that end in the last word, at and before in_bytes
        for cut in (0, b):
            n = min(fb * 7, in_bytes - cut)
            n -= n % fb
            ch = fb // b
            tail.append(make_desc(bytes=n, bit_depth=bits, channels=ch, src_off=in_bytes - cut - n, dst_off=dst,
                                  flags=abi.F_RAMP_ENABLED, ramp_start=16384, ramp_end=int(rng.integers(0, 16385)))[0])
            dst += n
    descs = np.concatenate([descs, np.array(tail, dtype=abi.CHUNK_DESC)])
    inp = np.full((in_bytes + 15) // 16 * 16 + 64, POISON, dtype=np.uint8)
    inp[:in_bytes] = port.fill_pcm(in_bytes, 500 + bits)
    return Batch("arena_tail_%d" % bits, descs, inp, in_bytes, dst + 16, port)


@pytest.fixture(scope="module")
def batches(port):
    rng = np.random.default_rng(2024)
    out = [from_workload(W.mixed(n_streams=48, seed=s), port, "mixed_%d" % s) for s in (1, 2, 3)]
    out.append(from_workload(W.config4(n_streams=96, seconds=0.12, seed=4), port, "config4"))
    specs = [s for bits in (8, 16, 24, 32) for le in (False, True) for s in alignment_specs(bits, le)]
    descs, in_bytes, out_bytes = pack_chunks(specs)
    out.append(Batch("every_alignment", descs, port.fill_pcm(in_bytes, 99), in_bytes, out_bytes, port))
    descs, in_bytes, out_bytes = max_size_chunks(rng)
    out.append(Batch("max_size_chunks", descs, port.fill_pcm(in_bytes, 98), in_bytes, out_bytes, port))
    descs, in_bytes, out_bytes = sinks_and_silence(rng)
    out.append(Batch("sinks_and_silence", descs, port.fill_pcm(in_bytes, 97), in_bytes, out_bytes, port))
    w = W.mixed(n_streams=64, seed=9)
    sched = capi.schedule_build(w.streams, w.events)
    out.append(Batch("padding", with_padding(sched.chunks, rng), port.fill_pcm(w.in_bytes, w.seed), w.in_bytes, w.out_bytes, port))
    out += [arena_tail(bits, port, rng) for bits in (8, 16, 24, 32)]
    big = from_workload(W.mixed(n_streams=2000, seed=7), port, "large")
    # enough chunks that runs of 16 survive the halving (at least 8 runs per CTA at up to 4 CTAs on each of 148 SMs)
    assert len(big.descs) >= 80000, len(big.descs)
    out.append(big)
    return out


def run_batch(ctx, b, cfg):
    import torch
    d_desc, d_in = b.device()
    d_out = torch.full((b.out_bytes + 2 * GUARD,), FILL, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    st = torch.cuda.current_stream().cuda_stream
    ctx.process_device(d_desc.data_ptr(), len(b.descs), d_in.data_ptr(), b.in_bytes, d_out.data_ptr() + GUARD, b.out_bytes, st)
    ctx.sync(st)                                             # raises on a rejected chunk or the watchdog
    assert ctx.inflight_cap() == cfg.get("OHP_CAP_CHUNKS", RING_SLOTS)
    check_arena(d_out.cpu().numpy(), b.want, b.descs, "%s, %s" % (b.name, cfg_id(cfg)))


def check_arena(buf, want, descs, what):
    assert (buf[:GUARD] == FILL).all(), "%s: wrote below the arena" % what
    assert (buf[GUARD + len(want):] == FILL).all(), "%s: wrote past the arena" % what
    got = buf[GUARD:GUARD + len(want)]
    if not np.array_equal(got, want):
        raise AssertionError("%s: %s" % (what, describe_first_diff(got, want, descs)))


@pytest.mark.parametrize("cfg", TUNER, ids=cfg_id)
def test_tuner_candidates_on_every_batch(configured, batches, cfg):
    ctx = configured(cfg)
    for b in batches:
        run_batch(ctx, b, cfg)


@pytest.mark.parametrize("cfg", SWEEP, ids=cfg_id)
def test_launch_settings_at_their_edges(configured, batches, cfg):
    """Caps of 1 and 2 chunks in flight and two maximum-size slots of ring bytes keep the ring full: the loader wraps,
    wastes the end of the ring and blocks on the oldest slot all the time.  Runs of 1 and 3 chunks deal the batch
    unevenly; runs of 16 survive only on the large batch."""
    ctx = configured(cfg)
    for b in batches:
        run_batch(ctx, b, cfg)


def test_placement_setting_picks_the_kernel(configured, batches):
    import torch
    from torch.profiler import ProfilerActivity, profile
    b = batches[0]
    for serial in (0, 1):
        cfg = dict(OHP_SERIAL_PLACE=serial, OHP_CAP_CHUNKS=12)
        ctx = configured(cfg)
        run_batch(ctx, b, cfg)                               # (module load outside the trace)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            run_batch(ctx, b, cfg)
            torch.cuda.synchronize()
        names = [e.key for e in prof.key_averages() if "ramp_convert_kernel" in e.key]
        want = "ramp_convert_kernel<%s>" % ("true" if serial else "false")
        assert names and all(want in n for n in names), (serial, names)


# ------------------------------------------------------------------------------------------------------------------
# whole-stage calls: region padding interleaved with the real descriptors, and the host pipeline's slices

@pytest.fixture(scope="module")
def stage_workloads(port):
    out = []
    for w in (W.config4(n_streams=96, seconds=0.12, seed=6), W.mixed(n_streams=64, seed=12, max_frames=5000)):
        inp = port.fill_pcm(w.in_bytes, w.seed)
        rc, want, chunks, _ = port.run(w.streams, w.events, inp, w.out_bytes)
        assert rc == 0
        want[~covered_mask(chunks, w.out_bytes)] = FILL
        out.append((w, inp, want, chunks))
    return out


@pytest.mark.parametrize("cfg", TUNER, ids=cfg_id)
def test_tuner_candidates_through_the_whole_stage(configured, stage_workloads, cfg):
    import torch
    ctx = configured(cfg)
    for w, inp, want, chunks in stage_workloads:
        what = "%s, %s" % (w.name, cfg_id(cfg))
        d_streams = torch.from_numpy(w.streams.view(np.uint8).copy()).cuda()
        d_events = torch.from_numpy(w.events.view(np.uint8).copy()).cuda()
        d_in = torch.from_numpy(inp).cuda()
        for want_total in (True, False):
            d_out = torch.full((w.out_bytes + 2 * GUARD,), FILL, dtype=torch.uint8, device="cuda")
            torch.cuda.synchronize()
            total = ctx.run_streams_device(d_streams.data_ptr(), len(w.streams), d_events.data_ptr(), len(w.events), d_in.data_ptr(),
                                           w.in_bytes, d_out.data_ptr() + GUARD, w.out_bytes, 0, None, want_total=want_total)
            ctx.sync()
            assert total == (len(chunks) if want_total else None)
            assert ctx.inflight_cap() == cfg["OHP_CAP_CHUNKS"]
            check_arena(d_out.cpu().numpy(), want, chunks, "run_streams_device " + what)
        buf = np.full(w.out_bytes + 2 * GUARD, FILL, dtype=np.uint8)
        _, total = ctx.run_streams_host(w.streams, w.events, inp, buf[GUARD:GUARD + w.out_bytes])
        assert total == len(chunks)
        assert ctx.inflight_cap() == cfg["OHP_CAP_CHUNKS"]
        check_arena(buf, want, chunks, "run_streams_host " + what)


# ------------------------------------------------------------------------------------------------------------------
# the schedule walk at every team and lane setting, one child process each

def walk_child():
    """Runs in the child: the device walk against the host model, then one whole-stage call against the oracle."""
    from oracle import pyoracle
    from test_gpu_schedule import check_both
    port = pyoracle.Port()
    ctx = capi.Context(0)
    try:
        stage = [W.mixed(n_streams=301, seed=23, max_frames=3000), W.config4(n_streams=97, seconds=0.12, seed=9)]
        for w in stage + [W.mixed(n_streams=2100, seed=22, max_frames=700), W.elements(5, n_streams=64)]:
            assert check_both(ctx, w) is not None, w.name
        # where the reference would ASSERT (Mute() twice; a MsgSilence split below one sample): the same refusal
        assert check_both(ctx, W.elements(5, n_streams=64, illegal=True)) is None
        assert check_both(ctx, W.mixed(n_streams=2100, seed=23, max_frames=700)) is None
        for w in stage:
            inp = port.fill_pcm(w.in_bytes, w.seed)
            rc, want, chunks, _ = port.run(w.streams, w.events, inp, w.out_bytes)
            assert rc == 0
            want[~covered_mask(chunks, w.out_bytes)] = FILL
            out = np.full(w.out_bytes + 2 * GUARD, FILL, dtype=np.uint8)
            ptrs = [ctx.device_alloc(max(a.nbytes, 16)) for a in (w.streams, w.events, inp, out)]
            try:
                d_streams, d_events, d_in, d_out = ptrs
                ctx.memcpy_h2d(d_streams, w.streams.view(np.uint8))
                ctx.memcpy_h2d(d_events, w.events.view(np.uint8))
                ctx.memcpy_h2d(d_in, inp)
                ctx.memcpy_h2d(d_out, out)
                total = ctx.run_streams_device(d_streams, len(w.streams), d_events, len(w.events), d_in, w.in_bytes,
                                               d_out + GUARD, w.out_bytes)
                ctx.memcpy_d2h(out, d_out)
                ctx.sync()
            finally:
                for p in ptrs:
                    ctx.device_free(p)
            assert total == len(chunks), w.name
            check_arena(out, want, chunks, w.name)
    finally:
        ctx.close()


@pytest.mark.parametrize("team,lanes", [(32, None), (1, 1), (1, 7), (1, 28), (1, 32)],
                         ids=["team32", "team1-lanes1", "team1-lanes7", "team1-lanes28", "team1-lanes32"])
def test_schedule_walk_at_every_team_and_lane_setting(team, lanes):
    """A warp per stream, or a thread per stream with 1, 7, 28 or 32 streams to a warp, on batches below and above the
    2048 streams where the context changes from one to the other by itself."""
    env = {k: v for k, v in os.environ.items() if not k.startswith("OHP_")}
    env["OHP_SCHED_TEAM"] = str(team)
    if lanes is not None:
        env["OHP_SCHED_LANES"] = str(lanes)
    env["PYTHONPATH"] = os.pathsep.join([ROOT, HERE] + ([env["PYTHONPATH"]] if env.get("PYTHONPATH") else []))
    r = subprocess.run([sys.executable, "-c", "import test_gpu_launch_configs as t; t.walk_child()"], cwd=ROOT, env=env,
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-4000:] + r.stderr[-4000:]
