"""ohp_run_streams_device_flywheel_recent on the GPU: the streams' bytes as ohp_run_streams_device writes them, the walk's
records as the class model records them, its pieces of recent audio as the class model keeps them (after
StartFlywheelRamp's cut), and the flywheel audio of every starvation ohp_flywheel_plan_batch_recent plans as the host route
plays it (plan_batch_recent -> process / flywheel / process on the device) and as the C oracle plays it.  Every starvation
ohp_run_streams_device_flywheel plays, this call plays with the same bytes."""
import os
import subprocess
import sys

import numpy as np
import pytest

from ohpipeline_b200 import abi, capi
from ohpipeline_b200 import workloads as W
from flywheel_util import every_shape_streams, starved_streams
from recent_util import K, cut, refusal_streams, silence_heavy_streams
import test_gpu_starvations as base

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
FILL, FLY_FILL = base.FILL, base.FLY_FILL


def run_recent(ctx, w, inp, fly_bytes=None, outputs=True):
    """The new call -> dict of host copies (outputs=False: the records and pieces stay in the context's scratch)."""
    import torch
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).reshape(-1).copy()).cuda()  # noqa: E731
    d_streams, d_events, d_in = dev(w.streams), dev(w.events if len(w.events) else np.zeros(16, np.uint8)), dev(inp)
    ne = len(w.events)
    fly_bytes = base.slots(w)[2] if fly_bytes is None else fly_bytes
    d_fly = torch.full((max(fly_bytes, 1),), FLY_FILL, dtype=torch.uint8, device="cuda")
    d_out = torch.full((w.out_bytes,), FILL, dtype=torch.uint8, device="cuda")
    d_outb = torch.zeros(len(w.streams), dtype=torch.int64, device="cuda")
    d_off = torch.full((max(ne, 1),), -1, dtype=torch.int64, device="cuda")
    d_len = torch.full((max(ne, 1),), -1, dtype=torch.int64, device="cuda")
    d_rec = torch.zeros((max(ne, 1) * abi.STARVATION.itemsize,), dtype=torch.uint8, device="cuda")
    d_recent = torch.zeros((max(ne, 1) * K * abi.RECENT_AUDIO.itemsize,), dtype=torch.uint8, device="cuda")
    d_count = torch.full((max(ne, 1),), -1, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    r = {}
    launches = ctx.launch_count()
    r["total"] = ctx.run_streams_device_flywheel_recent(
        d_streams.data_ptr(), len(w.streams), d_events.data_ptr(), ne, d_in.data_ptr(), inp.size, d_out.data_ptr(), w.out_bytes,
        d_fly.data_ptr(), fly_bytes, d_off.data_ptr(), d_len.data_ptr(), d_rec.data_ptr() if outputs else 0, d_outb.data_ptr(),
        d_recent=d_recent.data_ptr() if outputs else 0, d_recent_count=d_count.data_ptr() if outputs else 0)
    ctx.sync()
    r["launches"] = ctx.launch_count() - launches
    r["out"], r["fly"] = d_out.cpu().numpy(), d_fly.cpu().numpy()[:fly_bytes]
    r["outb"], r["off"], r["len"] = d_outb.cpu().numpy().view(np.uint64), d_off.cpu().numpy()[:ne].view(np.uint64), d_len.cpu().numpy()[:ne].view(np.uint64)
    r["rec"] = d_rec.cpu().numpy()[:ne * abi.STARVATION.itemsize].view(abi.STARVATION)
    r["recent"] = d_recent.cpu().numpy()[:ne * K * abi.RECENT_AUDIO.itemsize].view(abi.RECENT_AUDIO).reshape(ne, K)
    r["count"] = d_count.cpu().numpy()[:ne].view(np.uint32)
    return r


def plan_recent(w, sched):
    return capi.flywheel_plan_batch(w.streams, sched.starvations, recent=sched.recent, recent_begin=sched.recent_begin)


def host_route(ctx, w, inp, b):
    """What the plan's three launches play for each planned record -> {record index: bytes}."""
    import torch
    if len(b.planned) == 0:
        return {}
    d_in = torch.from_numpy(inp).cuda()
    d_train = torch.zeros(max(b.training_bytes, 1), dtype=torch.uint8, device="cuda")
    d_gen = torch.zeros(max(b.generated_bytes, 1), dtype=torch.uint8, device="cuda")
    d_out = torch.zeros(max(b.out_bytes, 1), dtype=torch.uint8, device="cuda")
    dev = lambda a: torch.from_numpy(a.view(np.uint8).reshape(-1).copy()).cuda()  # noqa: E731
    d_prep, d_jobs, d_blocks = dev(b.prep), dev(b.jobs), dev(b.blocks)
    torch.cuda.synchronize()
    ctx.process_device(d_prep.data_ptr(), len(b.prep), d_in.data_ptr(), inp.size, d_train.data_ptr(), b.training_bytes)
    ctx.flywheel_device(d_jobs.data_ptr(), len(b.jobs), d_train.data_ptr(), b.training_bytes, d_gen.data_ptr(), b.generated_bytes)
    ctx.process_device(d_blocks.data_ptr(), len(b.blocks), d_gen.data_ptr(), b.generated_bytes, d_out.data_ptr(), b.out_bytes)
    ctx.sync()
    out = d_out.cpu().numpy()
    return {int(k): out[int(o):int(o) + int(n)] for k, o, n in zip(b.planned, b.out_off, b.out_len)}


def oracle_route(port, inp, sv, b):
    """What the C oracle plays from the plan's prep descriptors and job layout -> {record index: bytes}."""
    if len(b.planned) == 0:
        return {}
    rc, train = port.process_chunks(b.prep, inp, b.training_bytes)
    assert rc == 0
    rc, gen = port.flywheel(b.jobs, train, b.generated_bytes)
    assert rc == 0
    blocks = []
    for i, k in enumerate(b.planned):
        d, _ = port.flywheel_ramp_chunks(b.jobs[i], int(sv["ramp"][k]), int(b.jobs[i]["dst_off"]), int(b.out_off[i]))
        assert d is not None, int(k)
        blocks.append(d)
    rc, out = port.process_chunks(np.concatenate(blocks), gen, b.out_bytes)
    assert rc == 0
    return {int(k): out[int(o):int(o) + int(n)] for k, o, n in zip(b.planned, b.out_off, b.out_len)}


def check(ctx, w, port, seed=None, outputs=True):
    """The whole comparison for one batch -> (class-model schedule, new call's result, existing call's result, incomplete
    record indices)."""
    inp = port.fill_pcm(w.in_bytes, w.seed if seed is None else seed)
    old = base.run(ctx, w, inp)
    r = run_recent(ctx, w, inp, outputs=outputs)
    # the streams' bytes, sizes and count: ohp_run_streams_device's
    assert np.array_equal(r["out"], old["out2"]) and np.array_equal(r["outb"], old["outb2"]) and r["total"] == old["total2"], w.name
    sched = capi.schedule_build(w.streams, w.events)
    sv = sched.starvations
    ev = sv["event"].astype(np.int64)
    incomplete = set()
    if outputs:
        # the records: the class model's, at their events
        have = np.nonzero(r["rec"]["event"] != 0xFFFFFFFF)[0]
        assert np.array_equal(have, np.sort(ev)), w.name
        for f in abi.STARVATION.names:
            assert np.array_equal(r["rec"][ev][f], sv[f]), (w.name, f)
        # the pieces: the class model's after the cut; incomplete exactly where it keeps more than the ring holds
        assert np.all(r["count"][np.setdiff1d(np.arange(len(w.events)), ev)] == 0), w.name
        for k, e in enumerate(ev):
            want = sched.recent_of(k)
            if len(want) > K:
                assert r["count"][e] == abi.RECENT_INCOMPLETE, (w.name, k)
                incomplete.add(k)
                continue
            assert cut(r["recent"][e][:r["count"][e]]) == cut(want), (w.name, k)
    else:
        incomplete = {k for k in range(len(sv)) if len(sched.recent_of(k)) > K}
    # which slots play and what they hold: the host route's and the oracle route's bytes
    off, size, total = base.slots(w)
    assert np.array_equal(r["off"], off), w.name
    b = plan_recent(w, sched)
    want = host_route(ctx, w, inp, b)
    oracle = oracle_route(port, inp, sv, b)
    assert sorted(oracle) == sorted(want), w.name
    played = {int(ev[k]): (v, oracle[k]) for k, v in want.items() if k not in incomplete}
    assert sorted(np.nonzero(r["len"])[0].tolist()) == sorted(played), w.name
    covered = np.zeros(total, dtype=bool)
    for e, (v, o_bytes) in played.items():
        o, n = int(off[e]), int(r["len"][e])
        assert n == len(v) == len(o_bytes) and n <= int(size[e])
        assert np.array_equal(r["fly"][o:o + n], o_bytes), (w.name, e, "differs from the oracle route")
        assert np.array_equal(r["fly"][o:o + n], v), (w.name, e, "differs from the host route")
        covered[o:o + n] = True
    assert np.all(r["fly"][~covered] == FLY_FILL), w.name
    # a superset of what ohp_run_streams_device_flywheel plays, with the same bytes
    for e in np.nonzero(old["len"])[0]:
        o, n = int(off[e]), int(old["len"][e])
        assert int(r["len"][e]) == n and np.array_equal(r["fly"][o:o + n], old["fly"][o:o + n]), (w.name, int(e))
    return sched, r, old, incomplete


def test_batches_against_the_host_and_oracle_routes(ctx, port):
    plays = 0
    for w in base.batches() + [every_shape_streams()]:
        _, r, _, _ = check(ctx, w, port)
        plays += int((r["len"] != 0).sum())
    for _, w, seed in starved_streams():
        check(ctx, w, port, seed)
    assert plays > 1000


def test_silence_heavy_streams_play_more(ctx, port):
    w = silence_heavy_streams()
    sched, r, old, incomplete = check(ctx, w, port)
    more = int((r["len"] != 0).sum()) - int((old["len"] != 0).sum())
    assert more >= 300, more
    # the overflowing stream: its records the host plans, the device walk could not keep, and plays nothing for
    assert len(incomplete) >= 1
    off, size, _ = base.slots(w)
    for k in incomplete:
        e = int(sched.starvations["event"][k])
        assert r["count"][e] == abi.RECENT_INCOMPLETE and r["len"][e] == 0
        assert np.all(r["fly"][int(off[e]):int(off[e]) + int(size[e])] == FLY_FILL)


def test_refusals_keep_the_fill_and_leave_the_others_alone(ctx, port):
    """The cut that never ends and under 1 ms since the recent audio was emptied: not played, slot kept, the stream's other
    starvations played.  (More than OHP_FLYWHEEL_MAX_PREP_RECENT prep descriptors needs more pieces than the ring keeps:
    on the device such a record is incomplete, covered above; the planner's own refusal is held against the host's in
    test_starvation_walk_recent.)"""
    w = refusal_streams()
    sched, r, _, _ = check(ctx, w, port)
    sv = sched.starvations
    off, size, _ = base.slots(w)
    refused = []
    for k in range(len(sv)):
        try:
            capi.flywheel_plan_recent(w.streams[int(sv["stream"][k])], sv[k:k + 1], sched.recent_of(k))
        except capi.OhpError as e:
            refused.append((k, e.status))
    assert sorted(s for _, s in refused) == [abi.E_INVALID_ARG, abi.E_INVALID_DESC]
    for k, _ in refused:
        e = int(sv["event"][k])
        assert r["len"][e] == 0 and np.all(r["fly"][int(off[e]):int(off[e]) + int(size[e])] == FLY_FILL)
    assert int((r["len"] != 0).sum()) == len(sv) - 2


def child():
    """Runs in a child process with the environment of the parametrization below."""
    from oracle import pyoracle
    port = pyoracle.Port()
    ctx = capi.Context(0)
    try:
        for w in [silence_heavy_streams(), base.batches()[-1], refusal_streams()]:
            check(ctx, w, port)
    finally:
        ctx.close()


@pytest.mark.parametrize("env", [{"OHP_ONE_WALK": "0"}, {"OHP_SCHED_TEAM": "1"}, {"OHP_SCHED_TEAM": "32"}],
                         ids=["two_pass", "team1", "team32"])
def test_every_walk_configuration(env):
    e = {k: v for k, v in os.environ.items() if not k.startswith("OHP_")}
    e.update(env)
    e["PYTHONPATH"] = os.pathsep.join([ROOT, HERE] + ([e["PYTHONPATH"]] if e.get("PYTHONPATH") else []))
    r = subprocess.run([sys.executable, "-c", "import test_gpu_starvations_recent as t; t.child()"], cwd=ROOT, env=e,
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-4000:] + r.stderr[-4000:]


def test_without_starvations_it_is_run_streams_device(ctx, port):
    w = W.mixed(n_streams=200, seed=5, max_frames=3000)
    assert not np.any(w.events["op"] == abi.EV_STARVATION)
    inp = port.fill_pcm(w.in_bytes, w.seed)
    old = base.run(ctx, w, inp)
    r = run_recent(ctx, w, inp)
    assert np.array_equal(r["out"], old["out2"]) and np.array_equal(r["outb"], old["outb2"]) and r["total"] == old["total2"]
    assert r["launches"] == old["launches2"]
    assert np.all(r["len"] == 0) and np.all(r["off"] == 0) and np.all(r["rec"]["event"] == 0xFFFFFFFF) and np.all(r["count"] == 0)


def test_context_scratch_when_the_caller_passes_no_arrays(ctx, port):
    _, r, _, _ = check(ctx, silence_heavy_streams(), port, outputs=False)
    assert int((r["len"] != 0).sum()) > 500


def test_errors_and_recovery(ctx, port):
    import torch
    w = silence_heavy_streams()
    inp = port.fill_pcm(w.in_bytes, w.seed)
    # a flywheel arena too small
    need = base.slots(w)[2]
    with pytest.raises(capi.OhpError) as e:
        run_recent(ctx, w, inp, fly_bytes=need - 16)
    assert e.value.status == base.OUT_OF_RANGE and str(need) in str(e.value)
    torch.cuda.synchronize()
    check(ctx, w, port)
    # two streams' slices share an event
    s = refusal_streams()
    shared = W.Workload("shared", np.concatenate([s.streams[:1], s.streams[:1]]), s.events, s.in_bytes, s.out_bytes, s.seed)
    with pytest.raises(capi.OhpError) as e:
        run_recent(ctx, shared, port.fill_pcm(s.in_bytes, s.seed))
    assert e.value.status == abi.E_INVALID_ARG and "two streams" in str(e.value)
    torch.cuda.synchronize()
    check(ctx, s, port)
    # a batch the reference ASSERTs on: refused as ohp_run_streams_device_flywheel refuses it
    bad = W.elements(5, n_streams=64, illegal=True)
    inp = port.fill_pcm(bad.in_bytes, bad.seed)
    with pytest.raises(capi.OhpError) as new:
        run_recent(ctx, bad, inp)
    torch.cuda.synchronize()
    with pytest.raises(capi.OhpError) as old:
        base.run(ctx, bad, inp, plain=False)
    torch.cuda.synchronize()
    assert new.value.status == old.value.status == base.INVALID_DESC and str(new.value) == str(old.value)
    check(ctx, W.elements(1, n_streams=48), port)
