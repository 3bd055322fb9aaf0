"""ohp_run_streams_device_flywheel on the GPU: every stream's bytes as ohp_run_streams_device writes them, the walk's
starvation records as the class model records them, and the flywheel audio of every starvation that plays as the host
route plays it (ohp_schedule_build -> ohp_flywheel_plan_batch -> process / flywheel / process on the device) and as the C
oracle plays it (the same prep descriptors and job layout through oracle/ohp_oracle.c, with the oracle's own RampGenerator
blocks) -- and, for flywheel_util.starved_streams(), as the reference's own StarvationRamper object plays it (tests/golden)."""
import os
import subprocess
import sys

import numpy as np
import pytest

from ohpipeline_b200 import abi, capi
from ohpipeline_b200 import workloads as W
from flywheel_util import every_shape_streams, shape_split

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
FILL, FLY_FILL = 0x5A, 0xA5
INVALID_DESC, OUT_OF_RANGE = 2, 5  # ohp_status


def slots(w):
    """The documented layout: (offset per event, slot bytes per event, total)."""
    size = np.zeros(len(w.events), dtype=np.uint64)
    for sp in w.streams:
        fb = int(sp["channels"]) * (int(sp["bit_depth"]) // 8)
        frames = abi.FLYWHEEL_RAMP_JIFFIES // abi.jiffies_per_sample(int(sp["sample_rate"]))
        lo, hi = int(sp["first_event"]), int(sp["first_event"]) + int(sp["num_events"])
        starving = w.events["op"][lo:hi] == abi.EV_STARVATION
        size[lo:hi][starving] = (frames * fb + 15) // 16 * 16
    off = np.concatenate([[0], np.cumsum(size)[:-1]]).astype(np.uint64) if len(size) else size
    return off, size, int(size.sum())


def run(ctx, w, inp, fly_bytes=None, records=True, plain=True):
    """Both calls on the same batch -> dict of host copies."""
    import torch
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).reshape(-1).copy()).cuda()  # noqa: E731
    d_streams, d_events, d_in = dev(w.streams), dev(w.events if len(w.events) else np.zeros(16, np.uint8)), dev(inp)
    ne = len(w.events)
    total_slots = slots(w)[2]
    fly_bytes = total_slots if fly_bytes is None else fly_bytes
    d_fly = torch.full((max(fly_bytes, 1),), FLY_FILL, dtype=torch.uint8, device="cuda")
    d_out = torch.full((w.out_bytes,), FILL, dtype=torch.uint8, device="cuda")
    d_outb = torch.zeros(len(w.streams), dtype=torch.int64, device="cuda")
    d_off = torch.full((max(ne, 1),), -1, dtype=torch.int64, device="cuda")
    d_len = torch.full((max(ne, 1),), -1, dtype=torch.int64, device="cuda")
    d_rec = torch.zeros((max(ne, 1) * abi.STARVATION.itemsize,), dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    r = {}
    launches = ctx.launch_count()
    r["total"] = ctx.run_streams_device_flywheel(d_streams.data_ptr(), len(w.streams), d_events.data_ptr(), ne, d_in.data_ptr(),
                                                 inp.size, d_out.data_ptr(), w.out_bytes, d_fly.data_ptr(), fly_bytes,
                                                 d_off.data_ptr(), d_len.data_ptr(), d_rec.data_ptr() if records else 0,
                                                 d_outb.data_ptr())
    ctx.sync()
    r["launches"] = ctx.launch_count() - launches
    r["out"], r["fly"] = d_out.cpu().numpy(), d_fly.cpu().numpy()[:fly_bytes]
    r["outb"], r["off"], r["len"] = d_outb.cpu().numpy().view(np.uint64), d_off.cpu().numpy()[:ne].view(np.uint64), d_len.cpu().numpy()[:ne].view(np.uint64)
    r["rec"] = d_rec.cpu().numpy()[:ne * abi.STARVATION.itemsize].view(abi.STARVATION)
    if plain:
        d_out2 = torch.full((w.out_bytes,), FILL, dtype=torch.uint8, device="cuda")
        d_outb2 = torch.zeros(len(w.streams), dtype=torch.int64, device="cuda")
        torch.cuda.synchronize()
        launches = ctx.launch_count()
        r["total2"] = ctx.run_streams_device(d_streams.data_ptr(), len(w.streams), d_events.data_ptr(), ne, d_in.data_ptr(), inp.size,
                                             d_out2.data_ptr(), w.out_bytes, d_outb2.data_ptr())
        ctx.sync()
        r["launches2"] = ctx.launch_count() - launches
        r["out2"], r["outb2"] = d_out2.cpu().numpy(), d_outb2.cpu().numpy().view(np.uint64)
    return r


def host_route(ctx, w, inp, sv):
    """What ohp_flywheel_plan_batch's three launches play for each planned record -> {record index: bytes}."""
    import torch
    b = capi.flywheel_plan_batch(w.streams, sv)
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


def oracle_route(port, w, inp, sv):
    """What the C oracle plays for each planned record -> {record index: bytes}.  Only the prep descriptors and the job
    layout come from ohp_flywheel_plan_batch; then ohpo_process_chunks (the training blocks), ohpo_flywheel, the oracle's
    RampGenerator::EndBlock restatement (ohpo_flywheel_ramp_chunks, not the product's ohp_flywheel_ramp_chunks) and
    ohpo_process_chunks again."""
    b = capi.flywheel_plan_batch(w.streams, sv)
    if len(b.planned) == 0:
        return {}
    rc, train = port.process_chunks(b.prep, inp, b.training_bytes)
    assert rc == 0
    rc, gen = port.flywheel(b.jobs, train, b.generated_bytes)
    assert rc == 0
    blocks = []
    for i, k in enumerate(b.planned):
        d, _ = port.flywheel_ramp_chunks(b.jobs[i], int(sv["ramp"][k]), int(b.jobs[i]["dst_off"]), int(b.out_off[i]))
        assert d is not None, (w.name, int(k))
        blocks.append(d)
    rc, out = port.process_chunks(np.concatenate(blocks), gen, b.out_bytes)
    assert rc == 0
    return {int(k): out[int(o):int(o) + int(n)] for k, o, n in zip(b.planned, b.out_off, b.out_len)}


def check(ctx, w, port, seed=None):
    """The whole comparison for one batch; returns (records, flywheel result)."""
    inp = port.fill_pcm(w.in_bytes, w.seed if seed is None else seed)
    r = run(ctx, w, inp)
    # the streams' bytes, sizes and count: ohp_run_streams_device's
    assert np.array_equal(r["out"], r["out2"]) and np.array_equal(r["outb"], r["outb2"]) and r["total"] == r["total2"], w.name
    # the records: the class model's, at their events; no record elsewhere
    sv = capi.schedule_build(w.streams, w.events).starvations
    ev = r["rec"]["event"]
    have = np.nonzero(ev != 0xffffffff)[0]
    assert np.array_equal(have, np.sort(sv["event"].astype(np.int64))), w.name
    assert np.array_equal(ev[have], have)
    by_event = r["rec"][sv["event"].astype(np.int64)]
    for f in abi.STARVATION.names:
        assert np.array_equal(by_event[f], sv[f]), (w.name, f)
    assert np.all(r["rec"].view(np.uint8).reshape(len(w.events), -1)[ev == 0xffffffff] == 0xff)
    # the layout, which slots play, and what they hold: the host route's bytes
    off, size, total = slots(w)
    assert np.array_equal(r["off"], off), w.name
    want = host_route(ctx, w, inp, sv)
    oracle = oracle_route(port, w, inp, sv)
    assert sorted(oracle) == sorted(want), w.name
    played = {int(sv["event"][k]): (v, oracle[k]) for k, v in want.items()}
    assert sorted(np.nonzero(r["len"])[0].tolist()) == sorted(played), w.name
    covered = np.zeros(total, dtype=bool)
    for e, (v, o_bytes) in played.items():
        o, n = int(off[e]), int(r["len"][e])
        assert n == len(v) == len(o_bytes) and n <= int(size[e])
        assert np.array_equal(r["fly"][o:o + n], o_bytes), (w.name, e, "differs from the oracle route")
        assert np.array_equal(r["fly"][o:o + n], v), (w.name, e, "differs from the host route")
        covered[o:o + n] = True
    assert np.all(r["fly"][~covered] == FLY_FILL), w.name
    return sv, r


def batches():
    return [W.elements(s, n_streams=48) for s in (1, 2)] + [W.elements(s, n_streams=48, attenuation=True) for s in (3, 4)] + \
        [W.elements(7, n_streams=2500, seconds=0.25)]


def test_starved_streams_play_what_the_reference_element_plays(ctx, port):
    from flywheel_util import starved_streams
    g = np.load(os.path.join(HERE, "golden", "starvation_flywheel.npz"))
    for name, w, seed in starved_streams():
        sv, r = check(ctx, w, port, seed)
        order = np.argsort(sv["event"])
        played = [r["fly"][int(r["off"][e]):int(r["off"][e]) + int(r["len"][e])] for e in sv["event"][order].astype(np.int64) if r["len"][e]]
        assert np.array_equal(np.concatenate(played), g["audio_" + name]), name


def test_random_batches_against_the_host_route(ctx, port):
    plays = 0
    for w in batches():
        sv, r = check(ctx, w, port)
        plays += int((r["len"] != 0).sum())
    assert plays > 50


def test_every_shape_streams(ctx, port):
    """flywheel_util.every_shape_streams(): 576 shapes starved twice.  The 1100 records at the 550 accepted shapes play
    what the oracle route and the host route play; the 52 at the 26 refused shapes play nothing and keep their slots'
    fill; the streams' bytes are the oracle's end-to-end output."""
    w = every_shape_streams()
    sv, r = check(ctx, w, port)
    accepted, refused = shape_split()
    shape = lambda s: (int(s["sample_rate"]), int(s["channels"]), int(s["bit_depth"]))  # noqa: E731
    ev = sv["event"].astype(np.int64)
    shapes = [shape(w.streams[int(s)]) for s in sv["stream"]]
    played = {sh for sh, e in zip(shapes, ev) if r["len"][e]}
    assert played == set(accepted)
    silent = [e for sh, e in zip(shapes, ev) if sh in set(refused)]
    assert len(silent) == 52 and int((r["len"][ev] != 0).sum()) == 1100
    off, size, _ = slots(w)
    for e in silent:
        assert r["len"][e] == 0 and np.all(r["fly"][int(off[e]):int(off[e]) + int(size[e])] == FLY_FILL), e
    inp = port.fill_pcm(w.in_bytes, w.seed)
    rc, want, chunks, _ = port.run(w.streams, w.events, inp, w.out_bytes)
    assert rc == 0
    mask = np.zeros(w.out_bytes, dtype=bool)
    for d, n in zip(chunks, abi.chunk_out_bytes(chunks)):
        mask[int(d["dst_off"]):int(d["dst_off"]) + int(n)] = True
    assert np.array_equal(r["out"][mask], want[mask])
    assert np.all(r["out"][~mask] == FILL)


def child():
    """Runs in a child process with the environment of the parametrization below."""
    from oracle import pyoracle
    port = pyoracle.Port()
    ctx = capi.Context(0)
    try:
        for w in batches()[:1] + batches()[-1:] + [every_shape_streams()]:
            check(ctx, w, port)
    finally:
        ctx.close()


@pytest.mark.parametrize("env", [{"OHP_ONE_WALK": "0"}, {"OHP_SCHED_TEAM": "1"}, {"OHP_SCHED_TEAM": "32"}],
                         ids=["two_pass", "team1", "team32"])
def test_every_walk_configuration(env):
    e = {k: v for k, v in os.environ.items() if not k.startswith("OHP_")}
    e.update(env)
    e["PYTHONPATH"] = os.pathsep.join([ROOT, HERE] + ([e["PYTHONPATH"]] if e.get("PYTHONPATH") else []))
    r = subprocess.run([sys.executable, "-c", "import test_gpu_starvations as t; t.child()"], cwd=ROOT, env=e,
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-4000:] + r.stderr[-4000:]


def test_without_starvations_it_is_run_streams_device(ctx, port):
    w = W.mixed(n_streams=200, seed=5, max_frames=3000)
    assert not np.any(w.events["op"] == abi.EV_STARVATION)
    inp = port.fill_pcm(w.in_bytes, w.seed)
    r = run(ctx, w, inp)
    assert np.array_equal(r["out"], r["out2"]) and np.array_equal(r["outb"], r["outb2"]) and r["total"] == r["total2"]
    assert r["launches"] == r["launches2"]
    assert np.all(r["len"] == 0) and np.all(r["off"] == 0) and np.all(r["rec"]["event"] == 0xffffffff)


def test_too_small_a_flywheel_arena_is_refused_and_the_context_goes_on(ctx, port):
    w = W.elements(2, n_streams=48)
    inp = port.fill_pcm(w.in_bytes, w.seed)
    need = slots(w)[2]
    with pytest.raises(capi.OhpError) as e:
        run(ctx, w, inp, fly_bytes=need - 16, plain=False)
    assert e.value.status == OUT_OF_RANGE and str(need) in str(e.value)
    import torch
    torch.cuda.synchronize()
    check(ctx, w, port)


def test_what_the_walk_refuses_is_refused_the_same_way(ctx, port):
    """Mute() twice in a row: the reference ASSERTS; both calls refuse the batch with the same status, naming the same stream."""
    import torch
    w = W.elements(5, n_streams=64, illegal=True)
    inp = port.fill_pcm(w.in_bytes, w.seed)
    with pytest.raises(capi.OhpError) as fly:
        run(ctx, w, inp, plain=False)
    torch.cuda.synchronize()
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).reshape(-1).copy()).cuda()  # noqa: E731
    d_streams, d_events, d_in = dev(w.streams), dev(w.events), dev(inp)
    d_out = torch.zeros(w.out_bytes, dtype=torch.uint8, device="cuda")
    with pytest.raises(capi.OhpError) as plain:
        ctx.run_streams_device(d_streams.data_ptr(), len(w.streams), d_events.data_ptr(), len(w.events), d_in.data_ptr(), inp.size,
                               d_out.data_ptr(), w.out_bytes)
    torch.cuda.synchronize()
    assert fly.value.status == plain.value.status == INVALID_DESC
    assert str(fly.value) == str(plain.value)
    check(ctx, W.elements(1, n_streams=48), port)


def test_a_shape_the_flywheel_does_not_take_plays_nothing(ctx, port):
    MS = abi.JIFFIES_PER_MS
    spec = W._spec(48000, 16, 10, False, 240, 48000 // 4)
    w = W._finish("ten_channels", [spec], [[(40 * MS + 7, 1, abi.EV_STARVATION, 50 * MS)]], seed=12)
    sv, r = check(ctx, w, port)
    assert len(sv) == 1 and sv["plays"][0] == 1 and r["len"][0] == 0 and np.all(r["fly"] == FLY_FILL)


def test_exports_of_the_header():
    from test_abi import declared_functions
    names = declared_functions("ohp_starvation_device.h")
    assert names == ["ohp_run_streams_device_flywheel"]
    for n in names:
        assert hasattr(capi.cuda_lib(), n), n
