"""A context from one call to the next.  Every other GPU test syncs after each asynchronous call; here calls follow one
another with no sync between them -- on one stream, and on two streams issued back to back -- while the context's scratch
(staging arenas, descriptor and region buffers, flywheel and recent-audio buffers) is grown, regrown and reused by
smaller batches, and errors are provoked to see that each is reported once and leaves nothing behind.  Every result is
the C oracle's; a call issued next to another must also give the bytes the same call gives alone on a synced context.
Each test has a context of its own, so the state it starts from is known."""
import functools
import types

import numpy as np
import pytest

from ohpipeline_b200 import abi, capi
from ohpipeline_b200 import workloads as W
from recent_util import K, cut
from util import covered_mask
import test_gpu_starvations as base
import test_gpu_starvations_recent as rbase

pytestmark = pytest.mark.gpu

FILL, FLY_FILL = base.FILL, base.FLY_FILL
SEED_BASE, FIRST_ID = 7 << 32, 1000


@pytest.fixture
def fresh():
    import torch
    ctx = capi.Context(0)
    try:
        yield ctx
    finally:
        torch.cuda.synchronize()
        ctx.close()


def first_diff(got, want):
    bad = np.nonzero(got != want)[0]
    return "equal" if bad.size == 0 else "%d bytes differ, first at %d: %d, want %d" % (bad.size, bad[0], got[bad[0]], want[bad[0]])


def dev(a):
    import torch
    a = np.ascontiguousarray(a).view(np.uint8).reshape(-1)
    return torch.from_numpy(a.copy() if a.size else np.zeros(16, np.uint8)).cuda()


class Expect:
    """What every call on workload w with input inp must leave, from the oracle: the output arena (fill where no chunk
    writes), sizes, count, records, flywheel slots of both flywheel calls, and the flywheel host route's output."""

    def __init__(self, port, w, inp, flywheel=True):
        self.w, self.inp = w, inp
        rc, want, chunks, _ = port.run(w.streams, w.events, inp, w.out_bytes)
        assert rc == 0
        self.chunks = chunks
        self.out = np.where(covered_mask(chunks, w.out_bytes), want, np.uint8(FILL))
        self.sched = capi.schedule_build(w.streams, w.events)
        self.outb, self.total = self.sched.stream_out_bytes, len(chunks)
        if not flywheel:
            return
        sv, ne = self.sched.starvations, len(w.events)
        self.ev = sv["event"].astype(np.int64)
        self.off, self.size, self.fly_bytes = base.slots(w)
        self.rec = np.full(ne * abi.STARVATION.itemsize, 0xFF, np.uint8).view(abi.STARVATION)
        self.rec[self.ev] = sv
        self.incomplete = {k for k in range(len(sv)) if len(self.sched.recent_of(k)) > K}

        def slots_of(route, skip=()):
            fly, ln = np.full(self.fly_bytes, FLY_FILL, np.uint8), np.zeros(ne, np.uint64)
            for k, v in route.items():
                if k not in skip:
                    e = int(sv["event"][k])
                    fly[int(self.off[e]):int(self.off[e]) + len(v)] = v
                    ln[e] = len(v)
            return fly, ln
        oracle = base.oracle_route(port, w, inp, sv)
        self.fly, self.len = slots_of(oracle)
        self.fly_recent, self.len_recent = slots_of(rbase.oracle_route(port, inp, sv, rbase.plan_recent(w, self.sched)),
                                                    self.incomplete)
        # ohp_flywheel_plan_batch's three launches (process_device, flywheel_device, process_device): the oracle's bytes
        self.plan = capi.flywheel_plan_batch(w.streams, sv)
        self.route = np.full(max(self.plan.out_bytes, 1), FILL, np.uint8)
        for i, k in enumerate(self.plan.planned):
            o = int(self.plan.out_off[i])
            self.route[o:o + int(self.plan.out_len[i])] = oracle[int(k)]


_EXPECT = {}


def expect(port, key, make, device_fill=False, flywheel=True):
    """Expect of a workload, computed once per session.  device_fill: the input ohp_fill_streams_device generates."""
    if key not in _EXPECT:
        w = make()
        inp = port.fill_streams(w.streams, w.in_bytes, SEED_BASE, FIRST_ID) if device_fill else port.fill_pcm(w.in_bytes, w.seed)
        _EXPECT[key] = Expect(port, w, inp, flywheel)
    return _EXPECT[key]


def small(port):
    return expect(port, "small", lambda: W.elements(1, n_streams=48), device_fill=True)


def large(port):
    return expect(port, "large", lambda: W.elements(7, n_streams=2500, seconds=0.25), device_fill=True)


def host_batch(port):
    """A few thousand descriptors for ohp_process_host."""
    return expect(port, "host", lambda: W.mixed(n_streams=128, seed=31, max_frames=4000), flywheel=False)


class Batch:
    """A workload in HBM: specs, events and input arena (uploaded, or left for ohp_fill_streams_device)."""

    def __init__(self, e, upload=True):
        import torch
        self.e, self.w, self.ne = e, e.w, len(e.w.events)
        self.streams, self.events = dev(e.w.streams), dev(e.w.events)
        self.inp = dev(e.inp) if upload else torch.zeros(e.w.in_bytes + 16, dtype=torch.uint8, device="cuda")

    def outputs(self, fly=True):
        import torch
        n = max(self.ne, 1)
        o = dict(out=torch.full((self.w.out_bytes,), FILL, dtype=torch.uint8, device="cuda"),
                 outb=torch.zeros(len(self.w.streams), dtype=torch.int64, device="cuda"))
        if fly:
            o.update(fly_arrays(n), fly=torch.full((max(self.e.fly_bytes, 1),), FLY_FILL, dtype=torch.uint8, device="cuda"))
        return o


def fly_arrays(n):
    import torch
    return dict(off=torch.full((n,), -1, dtype=torch.int64, device="cuda"), len=torch.full((n,), -1, dtype=torch.int64, device="cuda"),
                rec=torch.zeros(n * abi.STARVATION.itemsize, dtype=torch.uint8, device="cuda"),
                recent=torch.zeros(n * K * abi.RECENT_AUDIO.itemsize, dtype=torch.uint8, device="cuda"),
                count=torch.full((n,), -1, dtype=torch.int32, device="cuda"))


def issue(ctx, b, o, kind, stream=None, total=True, arrays=True, fly_bytes=None):
    """Enqueue one stage call -- kind "plain" (ohp_run_streams_device), "fly" (_flywheel) or "recent" (_flywheel_recent) --
    from b into the outputs o.  arrays=False: the records and recent audio stay in the context's scratch."""
    w = b.w
    args = (b.streams.data_ptr(), len(w.streams), b.events.data_ptr(), b.ne, b.inp.data_ptr(), w.in_bytes, o["out"].data_ptr(), w.out_bytes)
    if kind == "plain":
        return ctx.run_streams_device(*args, o["outb"].data_ptr(), stream, want_total=total)
    fly = (o["fly"].data_ptr(), b.e.fly_bytes if fly_bytes is None else fly_bytes, o["off"].data_ptr(), o["len"].data_ptr(),
           o["rec"].data_ptr() if arrays else 0, o["outb"].data_ptr(), stream, total)
    if kind == "fly":
        return ctx.run_streams_device_flywheel(*args, *fly)
    return ctx.run_streams_device_flywheel_recent(*args, *fly, d_recent=o["recent"].data_ptr() if arrays else 0,
                                                  d_recent_count=o["count"].data_ptr() if arrays else 0)


def verify(e, o, kind, got_total=None, arrays=True, what=""):
    """The outputs of one stage call (after a sync) against the oracle."""
    w, ne = e.w, len(e.w.events)
    out = o["out"].cpu().numpy()
    assert np.array_equal(out, e.out), (what, first_diff(out, e.out))
    assert np.array_equal(o["outb"].cpu().numpy().view(np.uint64), e.outb), what
    if got_total is not None:
        assert got_total == e.total, what
    if kind == "plain":
        return
    assert np.array_equal(o["off"].cpu().numpy()[:ne].view(np.uint64), e.off), what
    want_fly, want_len = (e.fly, e.len) if kind == "fly" else (e.fly_recent, e.len_recent)
    assert np.array_equal(o["len"].cpu().numpy()[:ne].view(np.uint64), want_len), what
    fly = o["fly"].cpu().numpy()[:e.fly_bytes]
    assert np.array_equal(fly, want_fly), (what, first_diff(fly, want_fly))
    if not arrays:
        return
    rec = o["rec"].cpu().numpy()[:ne * abi.STARVATION.itemsize]
    assert np.array_equal(rec, e.rec.view(np.uint8)), (what, "records (all ones where an event left none)")
    if kind == "recent":
        count = o["count"].cpu().numpy()[:ne].view(np.uint32)
        assert np.all(np.delete(count, e.ev) == 0), what
        recent = o["recent"].cpu().numpy()[:ne * K * abi.RECENT_AUDIO.itemsize].view(abi.RECENT_AUDIO).reshape(ne, K)
        for k, ev in enumerate(e.ev):
            if k in e.incomplete:
                assert count[ev] == abi.RECENT_INCOMPLETE, (what, k)
            else:
                assert count[ev] <= K and cut(recent[ev][:count[ev]]) == cut(e.sched.recent_of(k)), (what, k)


def stream_offsets(w):
    return np.append(w.streams["dst_base"].astype(np.uint64), np.uint64(w.out_bytes))


def sums_of(port, e):
    off = stream_offsets(e.w)
    return np.array([port.checksum(e.out[int(off[s]):int(off[s + 1])]) for s in range(len(e.w.streams))], dtype=np.uint64)


# ---------------------------------------------------------------------------------------------------------------------
# A. Ordered scripts on one stream: no sync between the device calls, one at the end


@pytest.mark.parametrize("sizes", [("small", "large", "small"), ("large", "small")], ids=["small_large_small", "large_small"])
def test_every_call_in_one_unsynced_script(fresh, port, sizes):
    """Every entry point that touches the context's scratch, on one stream, with the device-only calls between them: each
    batch's input generated on the device, the stage call with and without the chunk total, ohp_run_streams_host and
    ohp_process_host taking turns with it on the descriptor and region buffers, checksums of an output still being
    written, both flywheel calls with the caller's arrays and with none, and the flywheel host route.  Small -> large makes
    the first stage call of the large batch walk into a buffer that is too small, grow it and walk again; large -> small
    reuses every buffer for a smaller batch, the flywheel calls' arrays still holding a batch with more events."""
    import torch
    ctx = fresh
    A = torch.cuda.Stream()
    a = A.cuda_stream
    ph = host_batch(port)
    exps = {"small": small(port), "large": large(port)}
    n_max = max(len(e.w.events) for e in exps.values())
    shared = fly_arrays(n_max)  # the caller's flywheel arrays, reused by every step
    checks = []
    for step, size in enumerate(sizes):
        e = exps[size]
        w, ns = e.w, len(e.w.streams)
        b = Batch(e, upload=False)
        o = {k: b.outputs() for k in ("plain_total", "plain", "fly", "fly_null", "recent", "recent_null")}
        for k in ("fly", "recent"):
            o[k].update(shared)
        d_off = dev(stream_offsets(w))
        d_sums = torch.zeros(ns, dtype=torch.int64, device="cuda")
        plan = e.plan
        d_prep, d_jobs, d_blocks = dev(plan.prep), dev(plan.jobs), dev(plan.blocks)
        d_train = torch.zeros(max(plan.training_bytes, 1), dtype=torch.uint8, device="cuda")
        d_gen = torch.zeros(max(plan.generated_bytes, 1), dtype=torch.uint8, device="cuda")
        d_route = torch.full((max(plan.out_bytes, 1),), FILL, dtype=torch.uint8, device="cuda")
        A.wait_stream(torch.cuda.current_stream())  # the tensors above are initialised on torch's stream
        what = "step %d (%s)" % (step, size)
        ctx.fill_streams_device(b.inp.data_ptr(), w.in_bytes, b.streams.data_ptr(), ns, SEED_BASE, FIRST_ID, stream=a)
        t = issue(ctx, b, o["plain_total"], "plain", a)
        checks.append((e, o["plain_total"], "plain", t, True, what + " run_streams_device, total"))
        h_out = np.full(w.out_bytes, FILL, np.uint8)
        outb, t_host = ctx.run_streams_host(w.streams, w.events, e.inp, h_out)
        assert np.array_equal(h_out, e.out) and np.array_equal(outb, e.outb) and t_host == e.total, (what, first_diff(h_out, e.out))
        assert issue(ctx, b, o["plain"], "plain", a, total=False) is None
        checks.append((e, o["plain"], "plain", None, True, what + " run_streams_device, no total"))
        p_out = np.full(ph.w.out_bytes, FILL, np.uint8)
        ctx.process_host(ph.chunks, ph.inp, p_out)
        assert np.array_equal(p_out, ph.out), (what, "process_host", first_diff(p_out, ph.out))
        ctx.checksums_device(o["plain"]["out"].data_ptr(), d_off.data_ptr(), ns, d_sums.data_ptr(), stream=a)
        t = issue(ctx, b, o["fly"], "fly", a)
        with torch.cuda.stream(A):  # the shared arrays as this call leaves them, before the next call overwrites them
            o["fly"] = dict(o["fly"], **{k: v.clone() for k, v in shared.items()})
        checks.append((e, o["fly"], "fly", t, True, what + " flywheel, total"))
        assert issue(ctx, b, o["fly_null"], "fly", a, total=False, arrays=False) is None
        checks.append((e, o["fly_null"], "fly", None, False, what + " flywheel, no arrays"))
        ctx.process_device(d_prep.data_ptr(), len(plan.prep), b.inp.data_ptr(), w.in_bytes, d_train.data_ptr(), plan.training_bytes, stream=a)
        ctx.flywheel_device(d_jobs.data_ptr(), len(plan.jobs), d_train.data_ptr(), plan.training_bytes, d_gen.data_ptr(),
                            plan.generated_bytes, stream=a)
        ctx.process_device(d_blocks.data_ptr(), len(plan.blocks), d_gen.data_ptr(), plan.generated_bytes, d_route.data_ptr(),
                           plan.out_bytes, stream=a)
        t = issue(ctx, b, o["recent"], "recent", a)
        with torch.cuda.stream(A):
            o["recent"] = dict(o["recent"], **{k: v.clone() for k, v in shared.items()})
        checks.append((e, o["recent"], "recent", t, True, what + " flywheel recent, total"))
        assert issue(ctx, b, o["recent_null"], "recent", a, total=False, arrays=False) is None
        checks.append((e, o["recent_null"], "recent", None, False, what + " flywheel recent, no arrays"))
        checks.append((e, (d_sums, d_route, b.inp), "device", None, None, what))
    ctx.sync(a)
    torch.cuda.synchronize()
    for e, o, kind, t, arrays, what in checks:
        if kind == "device":
            d_sums, d_route, d_in = o
            assert np.array_equal(d_in.cpu().numpy()[:e.w.in_bytes], e.inp), (what, "fill_streams_device")
            assert np.array_equal(d_sums.cpu().numpy().view(np.uint64), sums_of(port, e)), (what, "checksums_device")
            route = d_route.cpu().numpy()
            assert np.array_equal(route, e.route), (what, "flywheel host route", first_diff(route, e.route))
        else:
            verify(e, o, kind, t, arrays, what)


def test_tuner_evictions_leave_the_bytes_alone(fresh, port):
    """One >= 65536-chunk, >= 256 MB descriptor batch through ohp_process_device under ten out_bytes values: ten batch
    signatures for an eight-entry tuning table, so entries are evicted and signatures come back untuned.  Three launches of
    each signature in a row (three candidate caps), then every signature once more; one stream, one sync.  Every launch
    writes the bytes of the first, which are the oracle's."""
    import torch
    ctx = fresh
    w = W.config5(n_streams=700, seconds=0.5)
    inp = port.fill_pcm(w.in_bytes, w.seed)
    rc, want, chunks, _ = port.run(w.streams, w.events, inp, w.out_bytes)
    assert rc == 0 and len(chunks) >= 65536 and w.in_bytes + w.out_bytes >= 256 << 20
    want = np.where(covered_mask(chunks, w.out_bytes), want, np.uint8(FILL))
    d_desc, d_in = dev(chunks), dev(inp)
    sigs = [w.out_bytes + 16 * k for k in range(10)]
    order = [s for s in sigs for _ in range(3)] + sigs
    outs = [torch.full((sigs[-1],), FILL, dtype=torch.uint8, device="cuda") for _ in order]
    A = torch.cuda.Stream()
    A.wait_stream(torch.cuda.current_stream())
    caps = []
    for o, out_bytes in zip(outs, order):
        ctx.process_device(d_desc.data_ptr(), len(chunks), d_in.data_ptr(), w.in_bytes, o.data_ptr(), out_bytes, stream=A.cuda_stream)
        caps.append(ctx.inflight_cap())
    ctx.sync(A.cuda_stream)
    assert len(set(caps)) > 1, caps
    first = outs[0].cpu().numpy()
    assert np.array_equal(first[:w.out_bytes], want), first_diff(first[:w.out_bytes], want)
    assert np.all(first[w.out_bytes:] == FILL)
    for i, o in enumerate(outs[1:], 1):
        assert torch.equal(o, outs[0]), (i, order[i], caps[i])


# ---------------------------------------------------------------------------------------------------------------------
# B. Unordered pairs: call 2 issued right after call 1 returns, no sync between them.  A call 1 without the chunk total
# still has its walk reading the region buffer when it returns: only pair 1 has one, and its call 2 writes no region.


@functools.lru_cache(maxsize=None)
def big():
    """configs[3] at its 16384 streams (7.9 GB each way): a walk of a couple of milliseconds.  Input generated on the
    device; the oracle only for a sample of streams."""
    return W.config4()


def mid(port):
    return expect(port, "mid", lambda: W.config4(n_streams=80, seconds=0.12, seed=9), flywheel=False)


class Big:
    """The big batch in HBM and one output per run."""

    def __init__(self, ctx, w):
        import torch
        self.w, self.ns = w, len(w.streams)
        self.streams, self.events = dev(w.streams), dev(w.events)
        self.inp = torch.zeros(w.in_bytes + 16, dtype=torch.uint8, device="cuda")
        torch.cuda.synchronize()
        ctx.fill_streams_device(self.inp.data_ptr(), w.in_bytes, self.streams.data_ptr(), self.ns, SEED_BASE, FIRST_ID)
        ctx.sync()

    def issue(self, ctx, o, stream, total):
        w = self.w
        return ctx.run_streams_device(self.streams.data_ptr(), self.ns, self.events.data_ptr(), len(w.events), self.inp.data_ptr(),
                                      w.in_bytes, o["out"].data_ptr(), w.out_bytes, o["outb"].data_ptr(), stream, want_total=total)

    def outputs(self):
        import torch
        return dict(out=torch.full((self.w.out_bytes,), FILL, dtype=torch.uint8, device="cuda"),
                    outb=torch.zeros(self.ns, dtype=torch.int64, device="cuda"))


def sample_matches_oracle(port, w, o, what):
    """Streams 0-31 (the first descriptor regions) and eight spread over the batch, through the oracle as a batch of their
    own laid out with the same gaps; their bytes in o["out"] are the oracle's, the gaps keep the fill."""
    n = len(w.streams)
    idx = sorted(set(range(32)) | set(np.linspace(32, n - 1, 8).astype(int).tolist()))
    dst = np.append(w.streams["dst_base"].astype(np.int64), w.out_bytes)
    streams = w.streams[idx].copy()
    events, slack, first = [], [], 0
    for k, i in enumerate(idx):
        lo, ne = int(w.streams[i]["first_event"]), int(w.streams[i]["num_events"])
        events.append(w.events[lo:lo + ne])
        streams[k]["first_event"] = first
        first += ne
        nbytes = int(w.streams[i]["total_frames"]) * int(w.streams[i]["channels"]) * (int(w.streams[i]["bit_depth"]) // 8)
        slack.append(int(dst[i + 1] - dst[i]) - nbytes)
    events = np.concatenate(events)
    in_bytes, out_bytes = W.layout(streams, slack_bytes=slack)
    inp = np.zeros(in_bytes, np.uint8)
    for k, i in enumerate(idx):
        sp = streams[k]
        nb = int(sp["total_frames"]) * int(sp["channels"]) * (int(sp["bit_depth"]) // 8)
        inp[int(sp["src_base"]):int(sp["src_base"]) + nb] = port.fill_pcm(nb, (SEED_BASE | (FIRST_ID + i)) & 0xFFFFFFFFFFFFFFFF)
    rc, want, chunks, _ = port.run(streams, events, inp, out_bytes)
    assert rc == 0
    got = np.concatenate([o["out"][int(dst[i]):int(dst[i + 1])].cpu().numpy() for i in idx])
    mask = covered_mask(chunks, out_bytes)[:got.size]
    assert np.array_equal(got[mask], want[:got.size][mask]), (what, first_diff(got[mask], want[:got.size][mask]))
    assert np.all(got[~mask] == FILL), what


def same(o, ref, what):
    import torch
    for k in ref:
        assert torch.equal(o[k], ref[k]), (what, k)


@pytest.mark.parametrize("own_stream", [False, True], ids=["caller_stream", "context_stream"])
def test_pair_device_stage_without_total_then_process_host(fresh, port, own_stream):
    """ohp_run_streams_device without the chunk total returns with its walk still running; ohp_process_host's descriptors
    must not land in the descriptor buffer before that walk and its kernel are done with it."""
    import torch
    ctx, w, ph = fresh, big(), host_batch(port)
    b = Big(ctx, w)
    A = None if own_stream else torch.cuda.Stream().cuda_stream
    ref = b.outputs()
    torch.cuda.synchronize()
    assert b.issue(ctx, ref, A, total=False) is None
    ctx.sync(A)
    p_ref = np.full(ph.w.out_bytes, FILL, np.uint8)
    ctx.process_host(ph.chunks, ph.inp, p_ref)
    assert np.array_equal(p_ref, ph.out)
    sample_matches_oracle(port, w, ref, "alone")
    o = b.outputs()
    torch.cuda.synchronize()
    assert b.issue(ctx, o, A, total=False) is None
    p_out = np.full(ph.w.out_bytes, FILL, np.uint8)
    ctx.process_host(ph.chunks, ph.inp, p_out)
    ctx.sync(A)
    assert np.array_equal(p_out, ph.out), ("process_host next to the stage call", first_diff(p_out, ph.out))
    same(o, ref, "stage call next to process_host")
    sample_matches_oracle(port, w, o, "paired")


@pytest.mark.parametrize("second", ["run_streams_host", "run_streams_device"])
def test_pair_device_stage_then_another_stage_call(fresh, port, second):
    """ohp_run_streams_device with the chunk total returns with its kernel still reading the descriptor buffer; the next
    call -- ohp_run_streams_host, or ohp_run_streams_device on another stream -- walks into that buffer."""
    import torch
    ctx, w, m = fresh, big(), mid(port)
    b = Big(ctx, w)
    A, B = torch.cuda.Stream().cuda_stream, torch.cuda.Stream().cuda_stream
    mb = Batch(m)
    ref, m_ref = b.outputs(), mb.outputs(fly=False)
    torch.cuda.synchronize()
    total = b.issue(ctx, ref, A, total=True)
    ctx.sync(A)
    sample_matches_oracle(port, w, ref, "alone")

    def call2(mo):
        if second == "run_streams_host":
            out = np.full(m.w.out_bytes, FILL, np.uint8)
            outb, t = ctx.run_streams_host(m.w.streams, m.w.events, m.inp, out)
            mo["out"].copy_(torch.from_numpy(out))
            mo["outb"].copy_(torch.from_numpy(outb.view(np.int64)))
            return t
        return issue(ctx, mb, mo, "plain", B, total=True)
    t2 = call2(m_ref)
    ctx.sync(B)
    torch.cuda.synchronize()
    verify(m, m_ref, "plain", t2, what="call 2 alone")
    o, mo = b.outputs(), mb.outputs(fly=False)
    torch.cuda.synchronize()
    assert b.issue(ctx, o, A, total=True) == total
    t2 = call2(mo)
    ctx.sync(A)
    ctx.sync(B)
    torch.cuda.synchronize()
    same(o, ref, "call 1 next to " + second)
    sample_matches_oracle(port, w, o, "paired")
    verify(m, mo, "plain", t2, what=second + " next to call 1")


@pytest.mark.parametrize("kind", ["fly", "recent"])
def test_pair_flywheel_calls_on_two_streams(fresh, port, kind):
    """ohp_run_streams_device_flywheel(_recent) with the chunk total returns with its flywheel launches still reading the
    plan's descriptors, jobs, training and generated audio; a second such call on another stream plans into the same
    buffers."""
    import torch
    ctx = fresh
    e1, e2 = large(port), small(port)
    b1, b2 = Batch(e1, upload=True), Batch(e2, upload=True)
    A, B = torch.cuda.Stream().cuda_stream, torch.cuda.Stream().cuda_stream
    r1, r2 = b1.outputs(), b2.outputs()
    torch.cuda.synchronize()
    t1 = issue(ctx, b1, r1, kind, A, total=True)
    ctx.sync(A)
    assert issue(ctx, b2, r2, kind, B, total=False) is None
    ctx.sync(B)
    verify(e1, r1, kind, t1, what="call 1 alone")
    verify(e2, r2, kind, what="call 2 alone")
    o1, o2 = b1.outputs(), b2.outputs()
    torch.cuda.synchronize()
    assert issue(ctx, b1, o1, kind, A, total=True) == t1
    assert issue(ctx, b2, o2, kind, B, total=False) is None
    ctx.sync(A)
    ctx.sync(B)
    torch.cuda.synchronize()
    same(o1, r1, "call 1 next to call 2")
    same(o2, r2, "call 2 next to call 1")


# ---------------------------------------------------------------------------------------------------------------------
# C. Status words: an error is reported by the first call or ohp_sync that covers its work, and then it is gone


@pytest.mark.parametrize("total", [True, False], ids=["total", "no_total"])
def test_two_errors_in_one_batch_are_reported_once(fresh, port, total):
    """One stream the walk refuses (stream 1) and two that reach outside d_out, in one ohp_run_streams_device batch: the
    call (or its first sync) reports E_INVALID_ARG naming stream 1 and names the descriptor too; the next sync is clean,
    and so is a clean batch on the same context, with the oracle's bytes."""
    import torch
    ctx = fresh
    w = W.config5(n_streams=4, seconds=0.02)
    bad = w.streams.copy()
    bad["sample_rate"][1] = 12345
    d_bad, d_ev = dev(bad), dev(w.events)
    d_in = torch.zeros(w.in_bytes + 16, dtype=torch.uint8, device="cuda")
    d_out = torch.zeros(w.out_bytes + 16, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    with pytest.raises(capi.OhpError) as err:
        ctx.run_streams_device(d_bad.data_ptr(), 4, d_ev.data_ptr(), len(w.events), d_in.data_ptr(), w.in_bytes, d_out.data_ptr(),
                               w.out_bytes // 2, 0, None, want_total=total)
        ctx.sync()
    assert err.value.status == abi.E_INVALID_ARG and "stream 1" in str(err.value), str(err.value)
    assert "out of range" in str(err.value), str(err.value)
    ctx.sync()
    e = small(port)
    b = Batch(e)
    o = b.outputs(fly=False)
    torch.cuda.synchronize()
    t = issue(ctx, b, o, "plain", None, total=total)
    ctx.sync()
    verify(e, o, "plain", t, what="clean batch after the two errors")


def test_flywheel_and_descriptor_errors_on_one_stream(fresh, port):
    """An invalid flywheel job, then an out-of-range chunk descriptor, on one stream: one sync reports the flywheel error
    (it comes first) and names both; the next sync is clean."""
    import torch
    ctx = fresh
    ok = capi.flywheel_job(48000, 2, 24)
    bad = ok.copy()
    bad["bit_depth"] = 20
    jobs = np.concatenate([ok, bad])
    jobs["dst_off"][1] = 8192
    d_jobs = dev(jobs)
    d_train = torch.zeros(1 << 16, dtype=torch.uint8, device="cuda")
    d_gen = torch.zeros(16384, dtype=torch.uint8, device="cuda")
    e = host_batch(port)
    descs = e.chunks.copy()
    bad_at = int(np.nonzero(descs["bytes"][3:])[0][0]) + 3
    descs["dst_off"][bad_at] = e.w.out_bytes  # out of range
    d_desc, d_in = dev(descs), dev(e.inp)
    d_out = torch.full((e.w.out_bytes,), FILL, dtype=torch.uint8, device="cuda")
    A = torch.cuda.Stream()
    A.wait_stream(torch.cuda.current_stream())
    ctx.flywheel_device(d_jobs.data_ptr(), 2, d_train.data_ptr(), d_train.numel(), d_gen.data_ptr(), d_gen.numel(), stream=A.cuda_stream)
    ctx.process_device(d_desc.data_ptr(), len(descs), d_in.data_ptr(), e.w.in_bytes, d_out.data_ptr(), e.w.out_bytes, stream=A.cuda_stream)
    with pytest.raises(capi.OhpError) as err:
        ctx.sync(A.cuda_stream)
    assert err.value.status == abi.E_INVALID_DESC and "flywheel job 1" in str(err.value), str(err.value)
    assert "chunk descriptor %d (out of range)" % bad_at in str(err.value), str(err.value)
    ctx.sync(A.cuda_stream)
    # every other descriptor wrote the oracle's bytes
    got = d_out.cpu().numpy()
    skip = covered_mask(e.chunks[bad_at:bad_at + 1], e.w.out_bytes)
    assert np.array_equal(got[~skip], e.out[~skip]) and np.all(got[skip] == FILL)


def clean_round(ctx, port, what):
    """One call of every kind on one stream, each against the oracle: none may report an earlier error."""
    import torch
    e, ph = small(port), host_batch(port)
    p_out = np.full(ph.w.out_bytes, FILL, np.uint8)
    ctx.process_host(ph.chunks, ph.inp, p_out)
    assert np.array_equal(p_out, ph.out), (what, "process_host")
    h_out = np.full(e.w.out_bytes, FILL, np.uint8)
    outb, t = ctx.run_streams_host(e.w.streams, e.w.events, e.inp, h_out)
    assert np.array_equal(h_out, e.out) and np.array_equal(outb, e.outb) and t == e.total, (what, "run_streams_host")
    b = Batch(e)
    plan = e.plan
    d_prep, d_jobs, d_blocks = dev(plan.prep), dev(plan.jobs), dev(plan.blocks)
    d_train = torch.zeros(max(plan.training_bytes, 1), dtype=torch.uint8, device="cuda")
    d_gen = torch.zeros(max(plan.generated_bytes, 1), dtype=torch.uint8, device="cuda")
    d_route = torch.full((max(plan.out_bytes, 1),), FILL, dtype=torch.uint8, device="cuda")
    runs = [(kind, total, b.outputs()) for kind in ("plain", "fly", "recent") for total in (True, False)]
    torch.cuda.synchronize()
    results = [(kind, o, issue(ctx, b, o, kind, None, total)) for kind, total, o in runs]
    ctx.process_device(d_prep.data_ptr(), len(plan.prep), b.inp.data_ptr(), e.w.in_bytes, d_train.data_ptr(), plan.training_bytes)
    ctx.flywheel_device(d_jobs.data_ptr(), len(plan.jobs), d_train.data_ptr(), plan.training_bytes, d_gen.data_ptr(), plan.generated_bytes)
    ctx.process_device(d_blocks.data_ptr(), len(plan.blocks), d_gen.data_ptr(), plan.generated_bytes, d_route.data_ptr(), plan.out_bytes)
    ctx.sync()
    for kind, o, t in results:
        verify(e, o, kind, t, what="%s: %s" % (what, kind))
    assert np.array_equal(d_route.cpu().numpy(), e.route), (what, "flywheel host route")


def test_every_call_after_every_error(fresh, port):
    """After each error the suite provokes -- a bad chunk descriptor, a bad flywheel job, a spec the walk refuses, a batch
    the reference would ASSERT on, a stream outside the arenas, a flywheel arena too small -- the next call of every kind
    gives the oracle's bytes and no error."""
    import torch
    ctx = fresh
    ph = host_batch(port)
    d_in, d_desc = dev(ph.inp), dev(ph.chunks)
    d_out = torch.zeros(ph.w.out_bytes, dtype=torch.uint8, device="cuda")
    e = small(port)
    b = Batch(e)
    torch.cuda.synchronize()

    def bad_descriptor():
        descs = ph.chunks.copy()
        descs["bit_depth"][int(np.nonzero(descs["bytes"])[0][5])] = 20
        d = dev(descs)
        torch.cuda.synchronize()
        ctx.process_device(d.data_ptr(), len(descs), d_in.data_ptr(), ph.w.in_bytes, d_out.data_ptr(), ph.w.out_bytes)
        ctx.sync()

    def bad_job():
        job = capi.flywheel_job(48000, 2, 24)
        job["bit_depth"] = 20
        d_job, d_gen = dev(job), torch.zeros(8192, dtype=torch.uint8, device="cuda")
        torch.cuda.synchronize()
        ctx.flywheel_device(d_job.data_ptr(), 1, d_in.data_ptr(), ph.w.in_bytes, d_gen.data_ptr(), d_gen.numel())
        ctx.sync()

    def refused_spec():
        s = e.w.streams.copy()
        s["sample_rate"][2] = 12345
        bb = Batch(e)
        bb.streams = dev(s)
        torch.cuda.synchronize()
        issue(ctx, bb, bb.outputs(fly=False), "plain")

    def walk_assert():
        w = W.elements(5, n_streams=64, illegal=True)
        bb = Batch(types.SimpleNamespace(w=w, inp=np.zeros(w.in_bytes, np.uint8)))
        torch.cuda.synchronize()
        issue(ctx, bb, bb.outputs(fly=False), "plain")

    def outside_arenas():
        o = b.outputs(fly=False)
        torch.cuda.synchronize()
        ctx.run_streams_device(b.streams.data_ptr(), len(e.w.streams), b.events.data_ptr(), b.ne, b.inp.data_ptr(), e.w.in_bytes,
                               o["out"].data_ptr(), e.w.out_bytes // 2, 0, None, want_total=False)
        ctx.sync()

    def small_fly_arena():
        o = b.outputs()
        torch.cuda.synchronize()
        issue(ctx, b, o, "fly", fly_bytes=e.fly_bytes - 16)

    for provoke, status in [(bad_descriptor, abi.E_INVALID_DESC), (bad_job, abi.E_INVALID_DESC), (refused_spec, abi.E_INVALID_ARG),
                            (walk_assert, abi.E_INVALID_DESC), (outside_arenas, abi.E_OUT_OF_RANGE),
                            (small_fly_arena, abi.E_OUT_OF_RANGE)]:
        with pytest.raises(capi.OhpError) as err:
            provoke()
        assert err.value.status == status, (provoke.__name__, str(err.value))
        clean_round(ctx, port, "after " + provoke.__name__)
