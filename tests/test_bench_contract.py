"""bench.py's contract, as far as it can be checked without a GPU: the reference arm prints exactly ONE JSON line with
the agreed keys (it times the reference's CPU path, so it runs anywhere), and our arm refuses to run without a B200
instead of falling back to anything."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_bench(*args):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], cwd=ROOT, stdout=subprocess.PIPE,
                          stderr=subprocess.PIPE, text=True, timeout=600)


def test_reference_arm_prints_one_json_line_with_the_contract_keys():
    r = run_bench("--impl", "reference", "--steps", "1", "--warmup", "3", "--streams", "8", "--seconds", "0.25")
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["higher_is_better"] is True and d["unit"] == "samples/s"
    assert d["n_gpus"] == 1 and d["steps"] == 1 and d["warmup"] >= 3 and d["vs_baseline"] is None
    assert d["value"] > 0 and d["ms_per_step"] > 0
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1
    assert d["cpu_baseline"]["value"] == d["value"] and d["cpu_baseline"]["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"]


def test_our_arm_refuses_to_run_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    r = run_bench("--steps", "1", "--warmup", "3", "--streams", "2", "--seconds", "0.1")
    assert r.returncode != 0
    assert r.stdout.strip() == ""          # no number without the CUDA path
    assert "no CUDA device" in r.stderr or "no CPU fallback" in r.stderr


@pytest.mark.gpu
def test_dump_outputs_holds_what_the_timed_step_computed(tmp_path):
    """--steps sets the number of timed launches, and --dump-outputs writes float arrays that a second run with the same
    arguments reproduces exactly: a sample of the output arena that is the C port's output at the same offsets, and
    every stream's checksum."""
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    from oracle import pyoracle
    dumps = []
    for i in range(2):
        d = tmp_path / str(i)
        r = run_bench("--steps", "3", "--warmup", "4", "--streams", "8", "--seconds", "0.1", "--no-configs", "--no-e2e",
                      "--no-cpu-baseline", "--dump-outputs", str(d))
        assert r.returncode == 0, r.stderr[-2000:]
        line = json.loads(r.stdout)
        assert line["steps"] == 3 and line["gpu_launches"] == 3 and line["bit_exact"] is True
        files = sorted(d.glob("*.npy"))
        assert sum(f.stat().st_size for f in files) <= 64 << 20
        dumps.append({f.name: np.load(f) for f in files})
    assert sorted(dumps[0]) == ["output_sample.npy", "output_sample_offsets.npy", "stream_checksums.npy"]
    for name, a in dumps[0].items():
        assert a.dtype in (np.float32, np.float64) and np.array_equal(a, dumps[1][name]), name
    w = bench.build_workload("config2", 8, 0.1)
    port = pyoracle.Port()
    inp = port.fill_streams(w.streams, w.in_bytes, bench.seed_base("config2"), 0)
    rc, want = port.run(w.streams, w.events, inp, w.out_bytes)[:2]
    assert rc == 0
    # a stream's checksum covers its range of the arena: from its dst_base to the next stream's
    edges = np.concatenate([w.streams["dst_base"], [w.out_bytes]]).astype(np.int64)
    halves = dumps[0]["stream_checksums.npy"].astype(np.uint64)
    assert halves.shape == (len(w.streams), 2)
    got = (halves[:, 0] << np.uint64(32)) | halves[:, 1]
    assert [int(x) for x in got] == [port.checksum(want[edges[s]:edges[s + 1]]) for s in range(len(w.streams))]
    sample, offs = dumps[0]["output_sample.npy"], dumps[0]["output_sample_offsets.npy"].astype(np.int64)
    for row, o in zip(sample, offs):
        assert np.array_equal(row, want[o:o + len(row)]), o


def test_the_bench_check_agrees_with_the_port_on_a_mixed_batch():
    """bench.py compares each rank's per-stream checksums with the reference's own code run on a sample of streams fed the
    per-stream seeded bytes.  Here the C port stands in for the GPU (same arena layout, same fill, same checksum ranges):
    the sample's checksums must come out the same -- packed little-endian streams included, which the linked reference
    reads through its big-endian sink."""
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    from ohpipeline_b200 import workloads
    from oracle import pyoracle
    port = pyoracle.Port()
    w = workloads.config4(n_streams=48, seconds=0.05, seed=9)
    w.key = "config4"
    first_id = 1000
    inp = port.fill_streams(w.streams, w.in_bytes, bench.seed_base("config4"), first_id)
    rc, chunks, _, _, outb = port.schedule_run(w.streams, w.events)
    assert rc == 0
    rc, out = port.process_chunks(chunks, inp, w.out_bytes)
    assert rc == 0
    offs = np.concatenate([w.streams["dst_base"], [w.out_bytes]]).astype(np.uint64)
    range_len = offs[1:] - offs[:-1]
    # what ohp_checksums_device would return for an arena that started zeroed
    arena = np.zeros(w.out_bytes, dtype=np.uint8)
    for s in range(len(w.streams)):
        lo = int(w.streams["dst_base"][s])
        arena[lo:lo + int(outb[s])] = out[lo:lo + int(outb[s])]
    gpu_like = np.array([port.checksum(arena[int(offs[s]):int(offs[s + 1])]) for s in range(len(w.streams))], dtype=np.uint64)
    picks = np.unique(np.linspace(0, len(w.streams) - 1, 20).astype(np.int64))
    assert (w.streams["out_fmt"][picks] == 1).any(), "sample holds no packed little-endian stream"
    want, kind, ok_sizes = bench.reference_stream_checksums(w, picks, first_id, outb, range_len, threads=2)
    assert ok_sizes and np.array_equal(gpu_like[picks], want), kind
    # a different global stream id is a different stream
    other, _, _ = bench.reference_stream_checksums(w, picks, first_id + 1, outb, range_len, threads=2)
    assert not np.array_equal(other, want)
