#!/usr/bin/env python
"""ohp_run_streams_device_flywheel and ohp_run_streams_device_flywheel_recent on a scaled `elements` batch (default 4096 streams x 1 s, every stream with a
StarvationRamper stage): what recording, planning and the three flywheel launches cost on top of ohp_run_streams_device
on the same batch (the recent-audio call alternating with the other two: it also keeps the recent audio in the walk and
plays the starvations with silence in their last millisecond), and the same work through the host route (ohp_schedule_build on every host core ->
ohp_flywheel_plan_batch -> upload -> process / flywheel / process) in wall clock.  Both device calls are timed as host
wall clock around call + stream synchronise, alternating, after warm-up; the card's name and power limit are read in
the same run.  With --out DIR the result is also written to DIR/starvation_bench.json.

    python profiles/starvation_bench.py [--streams 4096] [--seconds 1.0] [--reps 20] [--out DIR]"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                              text=True, timeout=60).stdout.strip()
    except OSError as e:
        return "unknown (%s)" % e


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--streams", type=int, default=4096)
    ap.add_argument("--seconds", type=float, default=1.0)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    from ohpipeline_b200 import abi, capi, workloads as W
    from test_gpu_starvations import slots

    w = W.elements(11, n_streams=a.streams, seconds=a.seconds)
    ctx = capi.Context(0)
    rng = np.random.default_rng(5)
    inp = rng.integers(0, 256, w.in_bytes, dtype=np.uint8)
    dev = lambda x: torch.from_numpy(np.ascontiguousarray(x).view(np.uint8).reshape(-1).copy()).cuda()  # noqa: E731
    d_streams, d_events, d_in = dev(w.streams), dev(w.events), dev(inp)
    ne = len(w.events)
    off, size, fly_bytes = slots(w)
    d_out = torch.zeros(w.out_bytes, dtype=torch.uint8, device="cuda")
    d_fly = torch.zeros(max(fly_bytes, 1), dtype=torch.uint8, device="cuda")
    d_off = torch.zeros(ne, dtype=torch.int64, device="cuda")
    d_len = torch.zeros(ne, dtype=torch.int64, device="cuda")
    d_rec = torch.zeros(ne * abi.STARVATION.itemsize, dtype=torch.uint8, device="cuda")
    d_len_r = torch.zeros(ne, dtype=torch.int64, device="cuda")
    d_recent = torch.zeros(ne * abi.DEVICE_RECENT_PIECES * abi.RECENT_AUDIO.itemsize, dtype=torch.uint8, device="cuda")
    d_count = torch.zeros(ne, dtype=torch.int32, device="cuda")
    args = (d_streams.data_ptr(), len(w.streams), d_events.data_ptr(), ne, d_in.data_ptr(), w.in_bytes, d_out.data_ptr(), w.out_bytes)

    def plain():
        ctx.run_streams_device(*args, want_total=False)
        ctx.sync()

    def fly():
        ctx.run_streams_device_flywheel(*args, d_fly.data_ptr(), fly_bytes, d_off.data_ptr(), d_len.data_ptr(), d_rec.data_ptr(),
                                        want_total=False)
        ctx.sync()

    def fly_recent():
        ctx.run_streams_device_flywheel_recent(*args, d_fly.data_ptr(), fly_bytes, d_off.data_ptr(), d_len_r.data_ptr(), d_rec.data_ptr(),
                                               want_total=False, d_recent=d_recent.data_ptr(), d_recent_count=d_count.data_ptr())
        ctx.sync()

    def host_route():
        sv = capi.schedule_build(w.streams, w.events).starvations
        b = capi.flywheel_plan_batch(w.streams, sv)
        d_prep, d_jobs, d_blocks = dev(b.prep), dev(b.jobs), dev(b.blocks)
        d_train = torch.empty(max(b.training_bytes, 1), dtype=torch.uint8, device="cuda")
        d_gen = torch.empty(max(b.generated_bytes, 1), dtype=torch.uint8, device="cuda")
        d_hout = torch.empty(max(b.out_bytes, 1), dtype=torch.uint8, device="cuda")
        ctx.process_device(d_prep.data_ptr(), len(b.prep), d_in.data_ptr(), w.in_bytes, d_train.data_ptr(), b.training_bytes)
        ctx.flywheel_device(d_jobs.data_ptr(), len(b.jobs), d_train.data_ptr(), b.training_bytes, d_gen.data_ptr(), b.generated_bytes)
        ctx.process_device(d_blocks.data_ptr(), len(b.blocks), d_gen.data_ptr(), b.generated_bytes, d_hout.data_ptr(), b.out_bytes)
        ctx.sync()
        return len(sv), len(b.planned)

    def timed(f):
        t = time.perf_counter()
        r = f()
        return (time.perf_counter() - t) * 1e3, r

    for _ in range(3):
        plain(); fly(); fly_recent()  # noqa: E702
    tp, tf, tr = [], [], []
    for _ in range(a.reps):
        tp.append(timed(plain)[0])
        tf.append(timed(fly)[0])
        tr.append(timed(fly_recent)[0])
    th = []
    for _ in range(3):
        ms, (n_records, n_planned) = timed(host_route)
        th.append(ms)
    played = int((d_len.cpu().numpy() != 0).sum())
    played_recent = int((d_len_r.cpu().numpy() != 0).sum())
    sched = capi.schedule_build(w.streams, w.events)
    n_planned_recent = len(capi.flywheel_plan_batch(w.streams, sched.starvations, recent=sched.recent,
                                                    recent_begin=sched.recent_begin).planned)
    res = {
        "card": card(), "streams": len(w.streams), "seconds": a.seconds, "events": ne,
        "starvation_events": int((w.events["op"] == abi.EV_STARVATION).sum()), "records": n_records,
        "planned_host": n_planned, "played_device": played, "planned_host_recent": n_planned_recent,
        "played_device_recent": played_recent, "fly_bytes": fly_bytes, "in_bytes": w.in_bytes, "out_bytes": w.out_bytes,
        "run_streams_device_ms": {"median": float(np.median(tp)), "min": float(np.min(tp)), "max": float(np.max(tp))},
        "run_streams_device_flywheel_ms": {"median": float(np.median(tf)), "min": float(np.min(tf)), "max": float(np.max(tf))},
        "run_streams_device_flywheel_recent_ms": {"median": float(np.median(tr)), "min": float(np.min(tr)), "max": float(np.max(tr))},
        "host_route_ms": {"median": float(np.median(th)), "min": float(np.min(th)), "max": float(np.max(th))},
        "host_cores": os.cpu_count(),
    }
    ctx.close()
    print(json.dumps(res, indent=1))
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "starvation_bench.json"), "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
