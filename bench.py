#!/usr/bin/env python
"""bench.py -- throughput of the fused ramp + format-convert path on N B200s (one process per GPU).

    python bench.py [--gpus N] [--steps K] [--warmup W]            # this repo's CUDA path
    python bench.py ... --dump-outputs DIR                         # + what the last timed step computed, as DIR/*.npy
    python bench.py --impl reference [--gpus N] --steps K --warmup W  # the reference's own CPU code (oracle/_ref)

A "step" is one pass of the hot path over one batch: BASELINE.json configs[1] by default (1024 streams, stereo,
24-bit, 192 kHz, 10 s each, every chunk ramped, packed 24-bit BE out).  At N > 1 every rank processes its own
batch of that size (streams shard with no data-path collective: weak scaling).

Both arms see the SAME bytes: a stream's PCM is the splitmix64 sequence seeded (config_id << 32) | global stream id
(ohp_fill_streams_device on the GPU, ohpo_fill_pcm on the CPU), and after every timed loop each rank checks what it
computed: per-stream 64-bit checksums of its output arena (ohp_checksums_device), gathered over the ranks on the host,
against the reference's own code run on a sample of its streams.

Printed on rank 0 as ONE JSON line:
  value      whole-job frames/s ("samples" in the reference's vocabulary = frames) with inputs resident in HBM
  e2e        the same metric through ohp_run_streams_host: pinned HOST buffers, H2D + kernels + D2H inside the timed region
  roofline   algorithmic bytes per launch / average launch duration (CUDA events on the launching stream) vs the
             measured HBM copy peak in MEASURED_PEAKS.json
  configs    every BASELINE.json config (configs[4] sharded 65536 / N streams per rank): ms per launch, fraction of the
             peak, and whether every rank's output matched the reference on the streams it checked
  cpu_baseline  the reference's CPU path (or the C oracle port) on this box's host cores, bounded sample
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from ohpipeline_b200 import abi, sharding, workloads  # noqa: E402

METRIC = "PCM samples/sec (fused ramp + format convert)"
UNIT = "samples/s"
DTYPE = "int32 Q15 fixed-point on 16-bit samples (u8 PCM bytes in/out)"
CONFIG_IDS = {"config1": 1, "config2": 2, "config3": 3, "config4": 4, "config5": 5, "mixed": 6}
BASELINE_INDEX = {"config1": 0, "config2": 1, "config3": 2, "config4": 3, "config5": 4}


def build_workload(name, streams, seconds):
    if name == "config2":
        return workloads.config2(n_streams=streams or 1024, seconds=seconds or 10.0)
    if name == "config5":
        return workloads.config5(n_streams=streams or 65536, seconds=seconds or 1.0)
    if name == "config3":
        return workloads.config3(n_streams=streams or 4096, seconds=seconds or 1.0,
                                 n_events=int(os.environ.get("OHP_C3_EVENTS", "8")))  # experiment knob: 0 = no ramps, uniform chunks
    if name == "config4":
        return workloads.config4(n_streams=streams or 16384, seconds=seconds or 0.25)
    if name == "mixed":  # the stress version of config4: tiny messages, one-sample caps, one-frame driver blocks
        return workloads.mixed(n_streams=streams or 16384, seed=4, max_frames=int((seconds or 1.0) * 48000))
    if name == "config1":
        return workloads.config1(seconds or 10.0)
    raise SystemExit("unknown workload %r" % name)


def seed_base(name):
    return CONFIG_IDS[name] << 32


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def recorded_traffic(workload_name, algo_bytes):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch, from the committed `ncu --set full` capture of a slice of
    the same workload (profiles/traffic.json), scaled to this launch by algorithmic bytes.  None when no capture exists."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(p):
        try:
            rec = json.load(open(p)).get(workload_name)
            if rec:
                return rec["capture_dram_bytes"] / rec["capture_algorithmic_bytes"] * algo_bytes
        except Exception:
            return None
    return None


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons through NVML while the timed regions run."""

    REASONS = {0x1: "gpu_idle", 0x2: "applications_clocks_setting", 0x4: "sw_power_cap", 0x8: "hw_slowdown",
               0x10: "sync_boost", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake_slowdown", 0x100: "display_clock_setting"}

    def __init__(self, device_index):
        super().__init__(daemon=True)
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self.power = []
        self._halt = threading.Event()
        self._active = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(device_index)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.ok = True
        except Exception:
            self.ok = False

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        while not self._halt.is_set():
            if self._active.is_set():
                try:
                    self.samples.append(int(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                    mask = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                    for bit, name in self.REASONS.items():
                        if mask & bit and name != "gpu_idle":
                            self.reasons.add(name)
                    self.power.append(nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0)
                except Exception:
                    pass
            time.sleep(0.02)

    def active(self, on):
        (self._active.set if on else self._active.clear)()

    def finish(self):
        self._halt.set()
        if self.ok:
            self.join(timeout=2)
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(s),
                "power_w_max": (round(max(self.power), 1) if self.power else None)}


# ----------------------------------------------------------------------------------------------------------------------
# the reference's CPU path (the checker of the GPU arm's results, and the thing the reference arm times)

def compact_streams(streams):
    """A copy of the given streams laid out back to back (16-byte aligned) in arenas of their own.  Returns
    (streams, in_bytes, out_room) -- out_room leaves space for inserted silence, which callers size from the GPU's
    per-stream output bytes or take generously."""
    sub = streams.copy()
    src = 0
    for i in range(len(sub)):
        n = int(sub["total_frames"][i]) * int(sub["channels"][i]) * (int(sub["bit_depth"][i]) // 8)
        sub["src_base"][i] = src
        src = (src + n + 15) // 16 * 16
    return sub, src


def reference_stream_checksums(w, picks, first_stream_id, out_bytes_of, range_len_of, threads):
    """Run the reference's own code (oracle/_ref; the C port where it did not travel) on streams `picks` of workload w,
    fed with the bytes ohp_fill_streams_device gives those streams, and return the per-stream checksum of each one's
    output range (its output bytes followed by the zero padding up to the next stream, as the GPU arena has it)."""
    from oracle import pyoracle
    port = pyoracle.Port()
    sub, in_bytes = compact_streams(w.streams[picks])
    dst = 0
    for i, s in enumerate(picks):
        sub["dst_base"][i] = dst
        dst = (dst + int(range_len_of[s]) + 15) // 16 * 16
    out_room = dst + 64
    inp = np.zeros(in_bytes, dtype=np.uint8)
    base = inp.ctypes.data
    import ctypes as C
    for i, s in enumerate(picks):
        n = int(sub["total_frames"][i]) * int(sub["channels"][i]) * (int(sub["bit_depth"][i]) // 8)
        port.lib.ohpo_fill_pcm(C.c_void_p(base + int(sub["src_base"][i])), C.c_uint64(n),
                               C.c_uint64((seed_base(w.key) | (first_stream_id + int(s))) & 0xFFFFFFFFFFFFFFFF))
    if pyoracle.Ref.available():
        kind = "reference"
        rc, out, _, _, outb = pyoracle.Ref().run(sub, w.events, inp, out_room, threads=max(1, min(threads, len(sub))),
                                                 want_descs=True, want_audio=True, want_sizes=True)
    else:
        kind = "port"
        rc, chunks, _, _, outb = port.schedule_run(sub, w.events)
        if rc == 0:
            rc, out = port.process_chunks(chunks, inp, out_room)
    assert rc == 0, rc
    sums = np.zeros(len(picks), dtype=np.uint64)
    ok_sizes = True
    for i, s in enumerate(picks):
        lo = int(sub["dst_base"][i])
        n = int(range_len_of[s])
        if int(outb[i]) != int(out_bytes_of[s]):
            ok_sizes = False
        seg = np.zeros(n, dtype=np.uint8)
        m = min(n, int(outb[i]))
        seg[:m] = out[lo:lo + m]
        b = int(sub["bit_depth"][i]) // 8
        if kind == "reference" and int(sub["out_fmt"][i]) == abi.OUT_PACKED_LE and b > 1:
            # the linked reference reads through ProcessorPcmBufTest (packed big-endian); the packed little-endian sink
            # (ProcessorPcmSwpEndianPacked) hands on the same subsamples byte-reversed
            seg[:m] = seg[:m].reshape(-1, b)[:, ::-1].reshape(-1)
        sums[i] = port.checksum(seg)
    return sums, kind, ok_sizes


def cpu_reference_run(w, n_streams, threads, steps, warmup):
    """Time the reference's own CPU path (oracle/_ref when present, else the C oracle port) on the first
    n_streams streams of workload w.  Returns (frames/s, ms per step, kind, cores, sample text)."""
    from oracle import pyoracle
    sub, in_bytes = compact_streams(w.streams[:n_streams])
    dst = 0
    for i in range(len(sub)):
        n = int(sub["total_frames"][i]) * int(sub["channels"][i]) * (int(sub["bit_depth"][i]) // 8)
        sub["dst_base"][i] = dst
        dst = (dst + n + 4096 + 15) // 16 * 16
    out_bytes = dst + 64
    inp = pyoracle.Port().fill_streams(sub, in_bytes, seed_base(w.key), 0)  # the bytes the GPU arm gives these streams
    frames = int(sub["total_frames"].sum())
    times = []
    if pyoracle.Ref.available():
        ref = pyoracle.Ref()
        kind = "reference"
        cores = min(threads, n_streams)
        for i in range(warmup + steps):
            t0 = time.perf_counter()
            rc, out, _, _ = ref.run(sub, w.events, inp, out_bytes, threads=cores, want_descs=False, want_audio=True)
            dt = time.perf_counter() - t0
            assert rc == 0, rc
            if i >= warmup:
                times.append(dt)
    else:
        port = pyoracle.Port()
        kind = "port"
        cores = 1
        for i in range(warmup + steps):
            t0 = time.perf_counter()
            rc, out, _, _ = port.run(sub, w.events, inp, out_bytes)
            dt = time.perf_counter() - t0
            assert rc == 0, rc
            if i >= warmup:
                times.append(dt)
    total = sum(times)
    sample = "first %d of %d streams of the workload, full length (%d frames/step), same seeded PCM as the GPU arm, %s" % (
        n_streams, len(w.streams), frames,
        "MsgFactory->SetRamp->CreatePlayable->Read(ProcessorPcmBufTest), one MsgFactory per thread" if kind == "reference"
        else "C oracle port, scalar")
    return frames * len(times) / total, 1e3 * total / len(times), kind, cores, sample


def pick_cpu_sample(w, threads, target_s=6.0):
    """Calibrate on one stream-slice, then size the sample so a step costs about target_s seconds of wall time."""
    from oracle import pyoracle
    per_stream_frames = int(w.streams["total_frames"][0])
    if not pyoracle.Ref.available():
        threads = 1
    probe = min(len(w.streams), max(1, threads))
    fps, _, _, _, _ = cpu_reference_run(w, probe, threads, steps=1, warmup=0)
    want_frames = fps * target_s
    n = int(max(probe, min(len(w.streams), want_frames // max(per_stream_frames, 1))))
    return max(1, n)


_REAL_STDOUT = None


def claim_stdout():
    """stdout carries ONE JSON line and nothing else: libraries that print there (NCCL's version banner comes from C
    code, at the first collective) are pointed at stderr, the line is written to the saved descriptor."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    sys.stdout.flush()
    os.write(_REAL_STDOUT if _REAL_STDOUT is not None else 1, (json.dumps(line) + "\n").encode())


# ----------------------------------------------------------------------------------------------------------------------
# one workload on this rank's GPU

class DeviceRun:
    """A workload resident in HBM on this rank: seeded input, descriptors built on the GPU, and the measurements."""

    def __init__(self, ctx, torch, w, first_stream_id, stream):
        self.ctx, self.torch, self.w, self.first_id, self.stream = ctx, torch, w, first_stream_id, stream
        self.st = stream.cuda_stream
        ns = len(w.streams)
        self.ns = ns
        self.d_specs = torch.from_numpy(w.streams.view(np.uint8).copy()).cuda()
        self.d_events = (torch.from_numpy(w.events.view(np.uint8).copy()).cuda() if len(w.events)
                         else torch.zeros(32, dtype=torch.uint8, device="cuda"))
        self.d_in = torch.empty(w.in_bytes + 16, dtype=torch.uint8, device="cuda")
        self.d_out = torch.zeros(w.out_bytes + 16, dtype=torch.uint8, device="cuda")
        self.d_begin = torch.zeros(ns + 1, dtype=torch.int64, device="cuda")
        self.d_outb = torch.zeros(max(ns, 1), dtype=torch.int64, device="cuda")
        torch.cuda.synchronize()
        # the same bytes the CPU arm generates for these streams
        ctx.fill_streams_device(self.d_in.data_ptr(), w.in_bytes, self.d_specs.data_ptr(), ns, seed_base(w.key), first_stream_id, self.st)
        ctx.sync(self.st)
        # descriptors, born in HBM
        t_dev = []
        for i in range(3):
            t0 = time.perf_counter()
            total = ctx.schedule_count_device(self.d_specs.data_ptr(), ns, self.d_events.data_ptr(), len(w.events),
                                              self.d_begin.data_ptr(), self.d_outb.data_ptr(), self.st)
            if i == 0:
                self.d_desc = torch.empty(max(total, 1) * abi.CHUNK_DESC.itemsize, dtype=torch.uint8, device="cuda")
                torch.cuda.synchronize()
            ctx.schedule_emit_device(self.d_specs.data_ptr(), ns, self.d_events.data_ptr(), len(w.events),
                                     self.d_begin.data_ptr(), self.d_desc.data_ptr(), 0, self.st)
            ctx.sync(self.st)
            t_dev.append(time.perf_counter() - t0)
        self.schedule_s = min(t_dev)
        self.n_chunks = total
        chunks = self.d_desc.cpu().numpy()[: total * abi.CHUNK_DESC.itemsize].view(abi.CHUNK_DESC)
        self.chunks = chunks
        self.out_bytes_of = self.d_outb.cpu().numpy().view(np.uint64)[:ns].copy()
        silence = (chunks["flags"] & abi.F_SILENCE) != 0
        nb = chunks["bytes"].astype(np.uint64)
        self.payload_out = int(abi.chunk_out_bytes(chunks).sum()) if total else 0
        self.payload_in = int(nb[~silence].sum())
        self.algo_bytes = self.payload_in + self.payload_out + total * abi.CHUNK_DESC.itemsize
        # a stream's checksum range: from its dst_base to the next stream's (zero padding included; d_out starts zeroed
        # and the path never writes what no chunk covers)
        offs = np.concatenate([w.streams["dst_base"], [w.out_bytes]]).astype(np.uint64)
        self.contiguous = bool((offs[1:] >= offs[:-1]).all())
        self.range_len_of = (offs[1:] - offs[:-1]) if self.contiguous else self.out_bytes_of
        self.d_off = torch.from_numpy(offs.view(np.int64).copy()).cuda()

    def step(self):
        w = self.w
        self.ctx.process_device(self.d_desc.data_ptr(), self.n_chunks, self.d_in.data_ptr(), w.in_bytes,
                                self.d_out.data_ptr(), w.out_bytes, self.st)

    def step_from_specs(self):
        w = self.w
        return self.ctx.run_streams_device(self.d_specs.data_ptr(), self.ns, self.d_events.data_ptr(), len(w.events),
                                           self.d_in.data_ptr(), w.in_bytes, self.d_out.data_ptr(), w.out_bytes, 0, self.st,
                                           want_total=False)

    def timed(self, fn, steps, warmup, barrier, dist):
        """warmup untimed calls, then `steps` calls between CUDA events on the launching stream, bracketed by a barrier +
        synchronize on both sides; max over ranks.  Returns ms per call."""
        torch = self.torch
        for _ in range(warmup):
            fn()
        self.ctx.sync(self.st)
        ev0 = torch.cuda.Event(enable_timing=True)
        ev1 = torch.cuda.Event(enable_timing=True)
        barrier()
        ev0.record(self.stream)
        for _ in range(steps):
            fn()
        ev1.record(self.stream)
        barrier()
        self.ctx.sync(self.st)
        ms = ev0.elapsed_time(ev1)
        if dist is not None:
            t = torch.tensor([ms], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms / steps

    def checksums(self):
        torch = self.torch
        sums = torch.zeros(max(self.ns, 1), dtype=torch.int64, device="cuda")
        self.ctx.checksums_device(self.d_out.data_ptr(), self.d_off.data_ptr(), self.ns, sums.data_ptr(), self.st)
        self.ctx.sync(self.st)
        return sums.cpu().numpy().view(np.uint64)[: self.ns].copy()

    def check_against_reference(self, n_check, threads):
        """Per-stream checksums of what sits in d_out, and the verdict of the reference's own code on a sample."""
        sums = self.checksums()
        if not self.contiguous:
            return sums, None, 0, "streams not laid out in order"
        n_check = min(n_check, self.ns)
        picks = np.unique(np.linspace(0, self.ns - 1, n_check).astype(np.int64))
        want, kind, ok_sizes = reference_stream_checksums(self.w, picks, self.first_id, self.out_bytes_of, self.range_len_of, threads)
        ok = bool(ok_sizes and np.array_equal(sums[picks], want))
        return sums, ok, len(picks), kind

    def dump_outputs(self, out_dir, sums, n_windows=256, window=4096):
        """Write what the last step left in the output arena, so that two builds can be compared output for output:
        output_sample.npy          n_windows x window output bytes (float32) at offsets drawn with a fixed seed,
        output_sample_offsets.npy  those offsets (float64),
        stream_checksums.npy       every stream's checksum of its whole output range, as (high, low) 32-bit halves
                                   (float64 holds both exactly).
        A few MB in all, whatever the workload's size."""
        os.makedirs(out_dir, exist_ok=True)
        n = self.w.out_bytes
        window = min(window, n)
        offs = np.sort(np.random.default_rng(0).integers(0, n - window + 1, size=n_windows))
        sample = self.torch.stack([self.d_out[o:o + window] for o in offs.tolist()]).cpu().numpy()
        np.save(os.path.join(out_dir, "output_sample.npy"), sample.astype(np.float32))
        np.save(os.path.join(out_dir, "output_sample_offsets.npy"), offs.astype(np.float64))
        halves = np.stack([sums >> np.uint64(32), sums & np.uint64(0xFFFFFFFF)], axis=1)
        np.save(os.path.join(out_dir, "stream_checksums.npy"), halves.astype(np.float64))

    def free(self):
        for name in ("d_specs", "d_events", "d_in", "d_out", "d_begin", "d_outb", "d_desc", "d_off"):
            if hasattr(self, name):
                delattr(self, name)
        self.torch.cuda.empty_cache()


def main():
    claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10, help="timed steps of the headline measurement (at least 1)")
    ap.add_argument("--warmup", type=int, default=4)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="", help="experiments: run this workload alone as the timed one (default: config2 + the configs array)")
    ap.add_argument("--streams", type=int, default=0)
    ap.add_argument("--seconds", type=float, default=0.0)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the per-config array (config1/3/4/5)")
    ap.add_argument("--no-check", action="store_true", help="experiments: skip the comparison with the reference")
    ap.add_argument("--check-streams", type=int, default=64, help="streams per rank and config compared with the reference")
    ap.add_argument("--e2e-steps", type=int, default=0, help="default: min(steps, 5)")
    ap.add_argument("--e2e-api", default="run_streams_host", choices=["run_streams_host", "process_host"])
    ap.add_argument("--chunk-frames", type=int, default=0, help="experiment: override the workload's frames per message")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="after the timed steps, write a seeded sample of the last step's output and every stream's "
                         "checksum to DIR/*.npy (rank 0's batch)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what the CUDA path computed; the reference arm has nothing of it to write")

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.warmup < 4:
        args.warmup = 4  # the first launches of a batch shape are the context's in-flight trials (ohp_inflight_cap)

    main_name = args.workload or "config2"
    w = build_workload(main_name, args.streams, args.seconds)
    w.key = main_name
    if args.chunk_frames:
        w.streams["chunk_frames"] = args.chunk_frames
    frames_per_step = w.total_frames
    subsamples_per_step = w.total_subsamples
    cfg = {"workload": w.name, "streams_per_gpu": int(len(w.streams)), "frames_per_step_per_gpu": frames_per_step,
           "l2": "inputs (%.2f GB per step per GPU) are larger than the 126 MB L2" % (w.in_bytes / 1e9),
           "sharding": "independent streams per rank, no data-path collective",
           "input": "splitmix64 per stream, seed (config_id << 32) | global stream id: the same bytes in both arms"}

    import multiprocessing
    host_threads = multiprocessing.cpu_count()

    # ------------------------------------------------------------------------------------------------------
    if args.impl == "reference":
        # the reference's own CPU implementation; rank 0 alone runs it
        if rank != 0:
            return 0
        n = pick_cpu_sample(w, host_threads)
        fps, ms, kind, cores, sample = cpu_reference_run(w, n, host_threads, args.steps, args.warmup)
        line = {"impl": "reference", "metric": METRIC, "value": fps, "unit": UNIT, "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": DTYPE, "data": "synthetic", "config": cfg,
                "cpu_baseline": {"value": fps, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
                "e2e": {"value": fps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        emit(line)
        return 0

    # ------------------------------------------------------------------------------------------------------
    import torch
    from ohpipeline_b200 import capi

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; this path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        os.environ["NCCL_DEBUG"] = "WARN"  # the image's default prints a version banner on stdout, next to the JSON line
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    ctx = capi.Context(local_rank)
    sampler = ClockSampler(local_rank)
    sampler.start()
    peak, peak_src = measured_peak()
    check_threads = max(1, host_threads // world)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def all_ranks(flag):
        """True only if `flag` holds on every rank (None counts as not checked -> False)."""
        v = 1 if flag else 0
        if dist is not None:
            t = torch.tensor([v], dtype=torch.int64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MIN)
            v = int(t.item())
        return bool(v)

    def total_over_ranks(x):
        if dist is None:
            return int(x)
        t = torch.tensor([int(x)], dtype=torch.int64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return int(t.item())

    # an explicit (non-default) stream: a NULL stream argument would select the context's own stream, and the
    # CUDA events must sit on the stream the kernels are launched on
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    assert stream.cuda_stream != 0

    # the timed workload: every rank its own batch (weak scaling), streams numbered rank * n ... so ranks differ
    first_id = rank * len(w.streams)
    run = DeviceRun(ctx, torch, w, first_id, stream)
    schedule_s_main = run.schedule_s
    t0 = time.perf_counter()
    host_sched_s = None
    if main_name == "config2" or args.workload:
        # the host model's descriptors (product code, threaded over streams) must be what the GPU built
        sched = capi.schedule_build(w.streams, w.events)
        host_sched_s = time.perf_counter() - t0
        if not np.array_equal(run.chunks, sched.chunks):
            raise SystemExit("bench.py: descriptors built on the GPU differ from the host model's")
        del sched
    n_chunks = run.n_chunks

    sampler.active(True)
    launches0 = ctx.launch_count()
    ms_per_step = run.timed(run.step, args.steps, args.warmup, barrier, dist)
    launches = ctx.launch_count() - launches0 - args.warmup
    inflight_cap = ctx.inflight_cap()
    value = frames_per_step * world / (ms_per_step * 1e-3)

    # what was just computed, on every rank, against the reference's own code on the same bytes
    sums, ok, n_checked, check_kind = (run.checksums(), None, 0, "skipped") if args.no_check else run.check_against_reference(args.check_streams, check_threads)
    if args.dump_outputs and rank == 0:
        run.dump_outputs(args.dump_outputs, sums)  # before the from-specs leg below writes the arena again
    all_sums = sharding.gather_checksums(sums, len(sums) * world, world, rank, dist)
    checksum_of_checksums = int(np.bitwise_xor.reduce(all_sums)) if len(all_sums) else 0
    main_bit_exact = None if args.no_check else all_ranks(ok)
    main_checked = total_over_ranks(n_checked)

    # the same stage from specs + events (both schedule passes inside the timed region)
    ms_from_specs = run.timed(run.step_from_specs, max(3, args.steps // 2), 5, barrier, dist)
    sums2 = run.checksums()
    from_specs_same = all_ranks(bool(np.array_equal(sums2, sums)))

    algo_bytes = run.algo_bytes
    in_payload, payload = run.payload_in, run.payload_out
    achieved = algo_bytes / (ms_per_step * 1e-3) / 1e9
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": recorded_traffic(main_name, algo_bytes), "peak_source": peak_src,
                "kernel": "ohp::ramp_convert_kernel", "algorithmic_bytes_per_launch": algo_bytes,
                "launch_ms": ms_per_step}
    from_specs = {"api": "ohp_run_streams_device (specs + events + PCM in HBM -> bytes in HBM: one schedule walk per stream into regions sized by a closed-form bound, then ramp_convert_kernel)",
                  "ms_per_step": ms_from_specs, "value": frames_per_step * world / (ms_from_specs * 1e-3), "unit": UNIT,
                  "frac": algo_bytes / (ms_from_specs * 1e-3) / 1e9 / peak, "same_checksums": from_specs_same}

    # ------------------------------------------------------------------------------------------------------
    # every other BASELINE config, to the same bar: timed on this rank's GPU, checked against the reference
    configs = []
    entry = {"workload": w.name, "baseline_config": BASELINE_INDEX.get(main_name), "streams_per_gpu": int(len(w.streams)),
             "chunks_per_launch": int(n_chunks), "ms_per_launch": ms_per_step, "frac": achieved / peak, "gbs_per_gpu": achieved,
             "bit_exact": main_bit_exact, "streams_checked": main_checked, "checked_against": check_kind,
             "scaling": "weak (every rank its own batch)", "inflight_chunks_per_cta": inflight_cap}
    configs.append(entry)
    keep_for_e2e = run
    if not args.workload and not args.no_configs:
        for name in ("config1", "config3", "config4", "config5"):
            wc = build_workload(name, 0, 0.0)
            wc.key = name
            n_total = len(wc.streams)
            if name == "config5" and world > 1:
                # BASELINE configs[4]: 65536 streams sharded over the ranks (contiguous blocks, re-based arenas)
                sub, _, lo, hi = sharding.shard_workload(wc.streams, wc.events, world, rank)
                last = wc.streams[hi - 1]
                in_b = int(last["src_base"]) + int(last["total_frames"]) * int(last["channels"]) * int(last["bit_depth"]) // 8 - int(wc.streams["src_base"][lo])
                out_b = (int(wc.streams["dst_base"][hi]) if hi < n_total else wc.out_bytes) - int(wc.streams["dst_base"][lo])
                ws = workloads.Workload(wc.name, sub, wc.events, (in_b + 15) // 16 * 16, (out_b + 15) // 16 * 16, wc.seed)
                ws.key = name
                wc_rank, fid, scaling = ws, lo, "strong (65536 streams sharded, %d per rank)" % (hi - lo)
            else:
                wc_rank, fid = wc, (rank * n_total if world > 1 else 0)
                scaling = "weak (every rank its own batch)" if world > 1 else "1 GPU"
            # make room: the timed workload's arenas are rebuilt for the e2e leg
            if keep_for_e2e is not None:
                keep_for_e2e.free()
                keep_for_e2e = None
            r = DeviceRun(ctx, torch, wc_rank, fid, stream)
            # configs[4] is the ">= 1 M stream-seconds" case of SURVEY 8d: >= 16 launches of 65536 one-second streams
            launches_c = max(16 if name == "config5" else 5, args.steps // 2)
            ms = r.timed(r.step, launches_c, args.warmup, barrier, dist)
            cap = ctx.inflight_cap()
            s_c, ok_c, n_c, kind_c = (r.checksums(), None, 0, "skipped") if args.no_check else r.check_against_reference(args.check_streams, check_threads)
            gathered = sharding.gather_checksums(s_c, total_over_ranks(len(s_c)), world, rank, dist)
            ms_fs = r.timed(r.step_from_specs, 5, 5, barrier, dist)
            ach = r.algo_bytes / (ms * 1e-3) / 1e9
            configs.append({"workload": wc.name, "baseline_config": BASELINE_INDEX[name], "streams_per_gpu": int(r.ns),
                            "chunks_per_launch": int(r.n_chunks), "ms_per_launch": ms, "frac": ach / peak, "gbs_per_gpu": ach,
                            "launches_timed": launches_c,
                            "stream_seconds_timed": launches_c * float(total_over_ranks(
                                int((wc_rank.streams["total_frames"] / wc_rank.streams["sample_rate"]).sum() + 0.5))),
                            "frames_per_s": total_over_ranks(wc_rank.total_frames) / (ms * 1e-3),
                            "bit_exact": None if args.no_check else all_ranks(ok_c), "streams_checked": total_over_ranks(n_c),
                            "checked_against": kind_c, "scaling": scaling, "inflight_chunks_per_cta": cap,
                            "from_specs_ms": ms_fs, "from_specs_frac": r.algo_bytes / (ms_fs * 1e-3) / 1e9 / peak,
                            "checksum_of_checksums": int(np.bitwise_xor.reduce(gathered)) if len(gathered) else 0,
                            "traffic": recorded_traffic(name, r.algo_bytes),
                            "l2": ("input %.1f MB: fits the 126 MB L2 (a latency case, not a bandwidth one)" % (wc_rank.in_bytes / 1e6)) if wc_rank.in_bytes < (126 << 20)
                                  else "input larger than L2"})
            r.free()
            del r
        configs.sort(key=lambda c: (c["baseline_config"] is None, c["baseline_config"]))

    # ------------------------------------------------------------------------------------------------------
    # end to end through the C ABI with HOST buffers: H2D + kernels + D2H inside the timed region
    e2e = None
    if not args.no_e2e:
        e2e_steps = args.e2e_steps or min(args.steps, 5)
        if keep_for_e2e is None:
            keep_for_e2e = DeviceRun(ctx, torch, w, first_id, stream)
        run = keep_for_e2e
        # every rank pins its batch (in + out) in host memory.  Where the box cannot hold all ranks' whole batches the e2e
        # leg runs on the first k streams of each rank's batch (same call, same per-stream work) and says so.
        ns = len(w.streams)
        k = ns
        frac = float(os.environ.get("OHP_E2E_MEM_FRACTION", "0.7"))
        avail = 0
        try:
            import psutil
            avail = psutil.virtual_memory().available
            need = (w.in_bytes + w.out_bytes) * world
            if need > frac * avail:
                k = max(1, min(ns, int(frac * avail / need * ns)))
        except ImportError:
            pass
        if dist is not None:
            kt = torch.tensor([k], dtype=torch.int64, device="cuda")
            dist.all_reduce(kt, op=dist.ReduceOp.MIN)
            k = int(kt.item())
        e_streams = w.streams[:k]
        e_in = int(w.streams["src_base"][k]) if k < ns else w.in_bytes
        e_out = int(w.streams["dst_base"][k]) if k < ns else w.out_bytes
        e_chunks = np.ascontiguousarray(run.chunks[: int(run.d_begin.cpu().numpy()[k])])
        e_frames = int(e_streams["total_frames"].sum())
        e_payload = int(run.out_bytes_of[:k].sum())
        want_sums = sums[:k]
        range_len = run.range_len_of
        h_in, h_in_ptr = ctx.host_alloc(e_in)
        h_out, h_out_ptr = ctx.host_alloc(e_out)
        ctx.memcpy_d2h(h_in, run.d_in.data_ptr(), run.st)
        ctx.sync(run.st)
        h_out[:] = 0
        run.free()
        del run, keep_for_e2e
        torch.cuda.empty_cache()
        # the call a user makes: stream specs + ramp events + host PCM in, bytes out (descriptors are built on the GPU
        # inside the call, every step); --e2e-api process_host times the descriptor-level entry point instead
        if args.e2e_api == "run_streams_host":
            def e2e_step():
                return ctx.run_streams_host(e_streams, w.events, h_in, h_out)
        else:
            def e2e_step():
                return ctx.process_host(e_chunks, h_in, h_out)
        for _ in range(2):
            e2e_step()
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            e2e_step()
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        if dist is not None:
            t = torch.tensor([dt], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t.item())
        e2e = {"value": e_frames * world * e2e_steps / dt, "unit": UNIT,
               "h2d_bytes_per_step": int(e_in + (e_streams.nbytes + w.events.nbytes if args.e2e_api == "run_streams_host"
                                                 else len(e_chunks) * abi.CHUNK_DESC.itemsize)),
               "d2h_bytes_per_step": int(e_payload + (k * 16 + 8 if args.e2e_api == "run_streams_host" else 0)),
               "ms_per_step": 1e3 * dt / e2e_steps, "steps": e2e_steps,
               "api": ("ohp_run_streams_host (pinned host buffers; specs + events + PCM H2D, descriptors built on the GPU, kernel, "
                       "PCM D2H, sliced by stream and pipelined)" if args.e2e_api == "run_streams_host" else
                       "ohp_process_host (pinned host buffers; descriptors + PCM H2D, kernel, PCM D2H, sliced and pipelined)"),
               "timer": "host wall clock around the synchronous calls, max over ranks"}
        if k < ns:
            e2e["sample"] = "first %d of %d streams per rank (host memory: %.0f GB available for %d ranks)" % (k, ns, avail / 1e9, world)
        # the bytes that came back over PCIe are the bytes the device-resident run produced (checked against the reference above)
        if not args.no_check:
            from oracle import pyoracle
            port = pyoracle.Port()
            picks = np.unique(np.linspace(0, k - 1, min(k, 16)).astype(np.int64))
            same = True
            for s in picks:
                lo = int(w.streams["dst_base"][s])
                same = same and port.checksum(h_out[lo:lo + int(range_len[s])]) == int(want_sums[s])
            e2e["bit_exact"] = all_ranks(same)
            e2e["streams_checked"] = total_over_ranks(len(picks))
        # the ceiling of this box for the same buffers: bare cudaMemcpyAsync, H2D and D2H at once, all ranks together
        try:
            d_a = torch.empty(e_in, dtype=torch.uint8, device="cuda")
            d_b = torch.empty(e_out, dtype=torch.uint8, device="cuda")
            s_in, s_out = torch.cuda.Stream(), torch.cuda.Stream()
            reps = 2
            barrier()
            t0 = time.perf_counter()
            for _ in range(reps):
                ctx.memcpy_h2d(d_a.data_ptr(), h_in, s_in.cuda_stream)
                ctx.memcpy_d2h(h_out, d_b.data_ptr(), s_out.cuda_stream)
            torch.cuda.synchronize()
            dtc = time.perf_counter() - t0
            if dist is not None:
                t = torch.tensor([dtc], dtype=torch.float64, device="cuda")
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                dtc = float(t.item())
            ceiling = (e_in + e_out) * world * reps / dtc / 1e9
            moved = (e2e["h2d_bytes_per_step"] + e2e["d2h_bytes_per_step"]) * world * e2e_steps / dt / 1e9
            e2e["pcie_gbs"] = moved
            e2e["ceiling_gbs"] = ceiling
            e2e["frac_of_ceiling"] = moved / ceiling
            e2e["ceiling"] = "bare cudaMemcpyAsync of the same pinned buffers, H2D and D2H concurrently, all %d ranks at once, both directions summed" % world
            del d_a, d_b
        except Exception as ex:  # the ceiling is an explanation, never a reason to lose the line
            e2e["ceiling_error"] = str(ex)[:200]
        ctx.host_free(h_in_ptr)
        ctx.host_free(h_out_ptr)
    sampler.active(False)
    clocks = sampler.finish()

    # ------------------------------------------------------------------------------------------------------
    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        n = pick_cpu_sample(w, host_threads, target_s=5.0)
        fps, ms, kind, cores, sample = cpu_reference_run(w, n, host_threads, steps=3, warmup=1)
        cpu_baseline = {"value": fps, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample, "ms_per_step": ms}

    if rank == 0:
        cfg.update({"chunks_per_step_per_gpu": n_chunks,
                    "host_schedule_build_s": (round(host_sched_s, 3) if host_sched_s is not None else None),
                    "device_schedule_build_s": round(schedule_s_main, 4),
                    "inflight_chunks_per_cta": inflight_cap,
                    "descriptors": "value: built on the GPU before the timed region (ohp_schedule_count_device + ohp_schedule_emit_device), identical to the host model's; value_from_specs: built inside it"})
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": DTYPE, "data": "synthetic", "config": cfg, "clocks": clocks,
                "e2e": e2e, "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu_baseline,
                "bit_exact": main_bit_exact, "streams_checked": main_checked, "checked_against": check_kind,
                "value_from_specs": from_specs, "configs": configs,
                "subsamples_per_s": subsamples_per_step * world / (ms_per_step * 1e-3),
                "payload_gb_per_s_per_gpu": (in_payload + payload) / (ms_per_step * 1e-3) / 1e9,
                "checksum_of_checksums": checksum_of_checksums}
        emit(line)
    ctx.close()
    if dist is not None:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
