"""The one-walk stage when streams outgrow their descriptor regions.  ohp_run_streams_device and its two flywheel variants
give every stream a region of sched::stream_chunk_bound descriptors; a stream with more playables than its region holds
writes none of them and makes the call take count + emit instead (with the chunk total) or fail with OHP_E_NO_MEMORY at
the next ohp_sync (without it).  No stream of this repo's generators outgrows its bound (tests/test_chunk_bound.py), so
OHP_REGION_CAP=n caps every region at n descriptors here, and n picks the streams that outgrow theirs: all, none, the
first, the last, or those with more than n playables.

Every result is the C oracle's: the output arena is filled first and bytes no chunk covers keep the fill; stream sizes,
the chunk total, starvation records, recent audio and flywheel slots are those of ohp_schedule_build and of the oracle and
host routes of the flywheel."""
import contextlib
import os
import subprocess
import sys
import types

import numpy as np
import pytest

from ohpipeline_b200 import abi, capi
from ohpipeline_b200 import workloads as W
from flywheel_util import every_shape_streams
from recent_util import silence_heavy_streams
from test_gpu_context_sequences import FILL, Batch, expect, first_diff, fresh, issue, verify  # noqa: F401 (fresh: fixture)
import test_gpu_starvations as base
import test_gpu_starvations_recent as rbase

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CAP = "OHP_REGION_CAP"
REDO = 4  # the two-pass redo's launches: count walk, scan, emitting walk, ramp_convert_kernel


@contextlib.contextmanager
def region_cap(n):
    """Regions of at most n descriptors for the calls issued inside (the library reads the setting on every call)."""
    old = os.environ.get(CAP)
    os.environ[CAP] = str(n)
    try:
        yield
    finally:
        if old is None:
            del os.environ[CAP]
        else:
            os.environ[CAP] = old


@pytest.fixture(autouse=True)
def _no_walk_settings(monkeypatch):
    for k in (CAP, "OHP_ONE_WALK"):
        monkeypatch.delenv(k, raising=False)


def counts_of(e):
    return np.diff(e.sched.stream_chunk_begin.astype(np.int64))


def arranged(w, last):
    """w with its stream of most playables moved to the end (last) or the front of the streams array (the streams keep
    their events and arena ranges)."""
    c = np.diff(capi.schedule_build(w.streams, w.events).stream_chunk_begin.astype(np.int64))
    top = int(np.argmax(c))
    rest = [i for i in range(len(c)) if i != top]
    idx = rest + [top] if last else [top] + rest
    return W.Workload("%s, top stream %s" % (w.name, "last" if last else "first"), w.streams[idx].copy(), w.events,
                      w.in_bytes, w.out_bytes, w.seed)


def plain(port, last=False):
    """64 streams with silence, stage caps and ramps on every stage; one of them has the most playables by far."""
    return expect(port, ("overflow_plain", last), lambda: arranged(W.mixed(n_streams=64, seed=12, max_frames=5000), last),
                  flywheel=False)


def starving(port, which):
    """flywheel_util.every_shape_streams() (576 streams starved twice each) or recent_util.silence_heavy_streams()."""
    make = every_shape_streams if which == "every_shape" else silence_heavy_streams
    return expect(port, ("overflow_" + which,), make)


def cap_for(which, c):
    """-> (cap, which streams outgrow their regions)."""
    top = int(c.max())
    # (all: regions of one descriptor fewer than the smallest stream's playables -- a region total of 0 would take
    #  ramp_convert_kernel's launch out of the count; test_first_call_of_a_shape has it)
    cap = {"all": int(c.min()) - 1, "none": top, "first": top - 1, "last": top - 1, "some": int(np.median(c))}[which]
    over = c > cap
    want = {"all": np.ones_like(over), "none": np.zeros_like(over)}
    if which in ("first", "last"):
        want[which] = np.arange(len(c)) == (0 if which == "first" else len(c) - 1)
    if which in want:
        assert np.array_equal(over, want[which]), (which, c)
    else:
        assert 0 < over.sum() < len(c), c
    return cap, over


def call(ctx, b, o, kind, total=True, arrays=True, stream=None):
    """One call -> (its result, the launches it made)."""
    import torch
    torch.cuda.synchronize()
    n0 = ctx.launch_count()
    t = issue(ctx, b, o, kind, stream, total=total, arrays=arrays)
    return t, ctx.launch_count() - n0


def with_total(ctx, e, kind, which, arrays=True, what=""):
    """Clean calls (the context's buffers at this batch's size; their launches), then the same call with the regions
    capped: the oracle's results, no error at the next ohp_sync, and the two-pass redo's launches exactly when a stream
    outgrew its region."""
    cap, over = cap_for(which, counts_of(e))
    what = "%s %s %s, cap %d (%d streams outgrow their regions)" % (what, e.w.name, kind, cap, int(over.sum()))
    b = Batch(e)
    for _ in range(2):  # (the first call of a shape may walk twice: the second's launches are the count to compare with)
        o = b.outputs(fly=kind != "plain")
        t, clean = call(ctx, b, o, kind, arrays=arrays)
        ctx.sync()
        verify(e, o, kind, t, arrays, what + ": uncapped")
    o = b.outputs(fly=kind != "plain")
    with region_cap(cap):
        t, launches = call(ctx, b, o, kind, arrays=arrays)
    ctx.sync()
    verify(e, o, kind, t, arrays, what)
    assert launches == clean + (REDO if over.any() else 0), (what, launches, clean)
    return over


# ---------------------------------------------------------------------------------------------------------------------
# with the chunk total: the two-pass redo


@pytest.mark.parametrize("which", ["all", "none", "first", "last", "some"])
def test_with_total_at_every_cap(fresh, port, which):
    with_total(fresh, plain(port, last=which == "last"), "plain", which)


@pytest.mark.parametrize("arrays", [True, False], ids=["caller_arrays", "context_scratch"])
@pytest.mark.parametrize("kind", ["fly", "recent"])
@pytest.mark.parametrize("batch", ["every_shape", "silence_heavy"])
def test_flywheel_calls_redo_with_their_plan(fresh, port, batch, kind, arrays):
    """The flywheel plan is made from the first walk's records before the call knows a stream outgrew its region; the redo
    walks again and the plan plays after it.  Records, recent audio, slots and every played slot are those of the oracle
    route and of the host route (plan_batch / plan_batch_recent, then process / flywheel / process)."""
    import torch
    e = starving(port, batch)
    w = e.w
    sv = e.sched.starvations
    # the host route's slots are the oracle route's, so the device's (checked against the latter) are both
    if kind == "fly":
        route, want, skip = base.host_route(fresh, w, e.inp, sv), e.fly, set()
    else:
        route, want, skip = rbase.host_route(fresh, w, e.inp, rbase.plan_recent(w, e.sched)), e.fly_recent, e.incomplete
    torch.cuda.synchronize()
    assert len(route) > 50
    for k, v in route.items():
        if k not in skip:
            o = int(e.off[int(sv["event"][k])])
            assert np.array_equal(want[o:o + len(v)], v), (batch, kind, k)
    for which in ("all", "some"):
        over = with_total(fresh, e, kind, which, arrays)
        # starvations in the streams that outgrew their regions
        starved = {int(s) for s in sv["stream"]}
        assert len(starved & set(np.nonzero(over)[0].tolist())) >= 10, (batch, which)


# ---------------------------------------------------------------------------------------------------------------------
# without the chunk total: OHP_E_NO_MEMORY, once


def without_total(ctx, e, which):
    """The call fails at the next ohp_sync naming the lowest stream that outgrew its region, and only there; the streams
    that fit have the oracle's bytes and sizes, the others wrote nothing and report 0 bytes.  A clean call follows."""
    import torch
    cap, over = cap_for(which, counts_of(e))
    what = "%s, cap %d" % (e.w.name, cap)
    b = Batch(e)
    o = b.outputs(fly=False)
    with region_cap(cap):
        assert call(ctx, b, o, "plain", total=False)[0] is None
    with pytest.raises(capi.OhpError) as err:
        ctx.sync()
    lowest = int(np.nonzero(over)[0][0])
    assert err.value.status == abi.E_NO_MEMORY, (what, str(err.value))
    assert "stream %d: more playables than its descriptor region holds" % lowest in str(err.value), (what, str(err.value))
    ctx.sync()
    torch.cuda.synchronize()
    want, outb = e.out.copy(), e.outb.copy()
    for s in np.nonzero(over)[0]:
        dst = int(e.w.streams["dst_base"][s])
        want[dst:dst + int(e.outb[s])] = FILL
        outb[s] = 0
    got = o["out"].cpu().numpy()
    assert np.array_equal(got, want), (what, first_diff(got, want))
    assert np.array_equal(o["outb"].cpu().numpy().view(np.uint64), outb), what
    o = b.outputs(fly=False)
    t, _ = call(ctx, b, o, "plain")
    ctx.sync()
    verify(e, o, "plain", t, what=what + ": the clean call after")


@pytest.mark.parametrize("which", ["all", "first", "last", "some"])
def test_without_total_the_next_sync_reports_it(fresh, port, which):
    without_total(fresh, plain(port, last=which == "last"), which)


# ---------------------------------------------------------------------------------------------------------------------
# the first call of a shape, and calls next to one another


def test_first_call_of_a_shape(fresh, port):
    """A first call whose buffer turns out too small (the walk runs, the buffer grows, the walk runs again) with a stream
    that outgrows its region; and on a context that has no descriptor buffer yet, regions of 0 descriptors."""
    ctx = fresh
    small = expect(port, ("overflow_tiny",), lambda: W.config5(n_streams=2, seconds=0.02), flywheel=False)
    e = plain(port)
    b = Batch(small)
    o = b.outputs(fly=False)
    t, _ = call(ctx, b, o, "plain")
    ctx.sync()
    verify(small, o, "plain", t, what="small batch first")
    cap, over = cap_for("some", counts_of(e))
    assert over[0]  # stream 0's region lies inside the small buffer: the first walk finds it too small as well
    # the capped regions outgrow the buffer the small batch left (grow(): 1/8 and 256 bytes more than asked for)
    held = int(capi.schedule_chunk_bounds(small.w.streams, small.w.events).sum()) * 9 // 8 + 9
    assert int(np.minimum(capi.schedule_chunk_bounds(e.w.streams, e.w.events).astype(np.int64), cap).sum()) > held
    b = Batch(e)
    o = b.outputs(fly=False)
    with region_cap(cap):
        t, launches = call(ctx, b, o, "plain")
    ctx.sync()
    verify(e, o, "plain", t, what="first call of the shape, cap %d" % cap)
    assert launches == 2 + 2 + 1 + REDO, launches   # bound + scan, two walks, ramp_convert_kernel, the redo
    import torch
    for ek, kind in ((e, "plain"), (starving(port, "silence_heavy"), "recent")):
        c = capi.Context(0)
        try:
            b = Batch(ek)
            o = b.outputs(fly=kind != "plain")
            with region_cap(0):
                t, _ = call(c, b, o, kind)
            c.sync()
            verify(ek, o, kind, t, what="regions of 0 descriptors on a new context, " + kind)
        finally:
            torch.cuda.synchronize()
            c.close()


def test_a_batch_without_regions_still_reports_its_streams(port):
    """Every stream refused: regions add up to 0, and on a new context (no descriptor buffer yet) the walk must still
    run and report the lowest stream."""
    import torch
    w = W.config5(n_streams=3, seconds=0.02)
    w.streams["sample_rate"] = 12345
    e = types.SimpleNamespace(w=w, inp=np.zeros(w.in_bytes, np.uint8))
    for total in (True, False):
        c = capi.Context(0)
        try:
            b = Batch(e)
            o = b.outputs(fly=False)
            with pytest.raises(capi.OhpError) as err:
                call(c, b, o, "plain", total=total)
                c.sync()
            assert err.value.status == abi.E_INVALID_ARG and "stream 0" in str(err.value), (total, str(err.value))
            c.sync()
        finally:
            torch.cuda.synchronize()
            c.close()


@pytest.mark.parametrize("first_total", [True, False], ids=["total_then_total", "no_total_then_total"])
def test_overflow_on_one_stream_then_a_call_on_another(fresh, port, first_total):
    """Call 1 outgrows regions on stream A; call 2, with regions uncapped, follows on stream B without a sync between.
    With the total call 1 redoes its batch; without it, its OHP_E_NO_MEMORY is reported exactly once -- by call 2, which
    reads the context's status block, or by a sync -- and call 2 does not take it for its own.  Both calls' bytes are
    the oracle's."""
    import torch
    ctx = fresh
    e1, e2 = plain(port), starving(port, "silence_heavy")
    b1, b2 = Batch(e1), Batch(e2)
    cap, over = cap_for("some", counts_of(e1))
    A, B = torch.cuda.Stream(), torch.cuda.Stream()
    for b, kind in ((b1, "plain"), (b2, "fly")):  # the buffers at their size: no walk is launched twice below
        call(ctx, b, b.outputs(fly=kind != "plain"), kind)
    ctx.sync()
    o1, o2 = b1.outputs(fly=False), b2.outputs()
    torch.cuda.synchronize()
    errors = []
    with region_cap(cap):
        t1 = issue(ctx, b1, o1, "plain", A.cuda_stream, total=first_total)
    n0 = ctx.launch_count()
    try:
        t2 = issue(ctx, b2, o2, "fly", B.cuda_stream)
    except capi.OhpError as err:
        errors.append(err)
        t2 = e2.total  # (the call reported an error that is not its own: its work is whole, the total is not returned)
    launches2 = ctx.launch_count() - n0
    for st in (A, B, A):
        try:
            ctx.sync(st.cuda_stream)
        except capi.OhpError as err:
            errors.append(err)
    torch.cuda.synchronize()
    verify(e2, o2, "fly", t2, what="call 2")
    assert launches2 == 9, launches2  # bound + scan, walk, plan (2), ramp_convert_kernel, flywheel (3): no redo
    if first_total:
        assert not errors, [str(x) for x in errors]
        verify(e1, o1, "plain", t1, what="call 1")
        return
    lowest = int(np.nonzero(over)[0][0])
    assert len(errors) == 1, [str(x) for x in errors]
    assert errors[0].status == abi.E_NO_MEMORY and "stream %d: more playables" % lowest in str(errors[0]), str(errors[0])
    got = o1["out"].cpu().numpy()
    fit = np.ones(len(e1.w.streams), bool)
    fit[over] = False
    for s in range(len(e1.w.streams)):
        lo, n = int(e1.w.streams["dst_base"][s]), int(e1.outb[s])
        want = e1.out[lo:lo + n] if fit[s] else np.full(n, FILL, np.uint8)
        assert np.array_equal(got[lo:lo + n], want), ("call 1 stream", s, bool(fit[s]))


# ---------------------------------------------------------------------------------------------------------------------
# both walk teams, one child process each (the team is read once per process)


def team_child():
    from oracle import pyoracle
    port = pyoracle.Port()
    ctx = capi.Context(0)
    try:
        for which in ("all", "first", "last", "some"):
            with_total(ctx, plain(port, last=which == "last"), "plain", which)
        for batch, kind in (("every_shape", "fly"), ("silence_heavy", "recent")):
            for arrays in (True, False):
                with_total(ctx, starving(port, batch), kind, "some", arrays)
        without_total(ctx, plain(port), "some")
    finally:
        ctx.close()
    ctx = capi.Context(0)
    try:
        test_first_call_of_a_shape(ctx, port)
    finally:
        ctx.close()


@pytest.mark.parametrize("team", [1, 32])
def test_both_walk_teams(team):
    env = {k: v for k, v in os.environ.items() if not k.startswith("OHP_")}
    env["OHP_SCHED_TEAM"] = str(team)
    env["PYTHONPATH"] = os.pathsep.join([ROOT, HERE] + ([env["PYTHONPATH"]] if env.get("PYTHONPATH") else []))
    r = subprocess.run([sys.executable, "-c", "import test_gpu_region_overflow as t; t.team_child()"], cwd=ROOT, env=env,
                       capture_output=True, text=True, timeout=1500)
    assert r.returncode == 0, r.stdout[-4000:] + r.stderr[-4000:]
