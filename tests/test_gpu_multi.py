"""ohp_multi (include/ohp_multi.h): the whole stage over several devices from one process -- a contiguous block of streams, a
context, a host thread and its own CUDA streams per device, no collective; per-stream checksums gathered on the host
(SURVEY 8e).  On a box with one GPU the "devices" are several contexts on that GPU: the sharding, the re-basing of every
block's arenas and events, the gather and the error paths are the same code."""
import numpy as np
import pytest

from ohpipeline_b200 import abi, capi, workloads

pytestmark = pytest.mark.gpu


def device_lists():
    n = capi.device_count()
    lists = [[0], [0, 0], [0, 0, 0]]
    if n > 1:
        lists += [list(range(n)), list(range(n)) * 2]
    return lists


def stream_checksums(port, out, streams, outb):
    return np.array([port.checksum(out[int(s["dst_base"]):int(s["dst_base"]) + int(n)]) for s, n in zip(streams, outb)], dtype=np.uint64)


@pytest.mark.parametrize("make", [
    lambda: workloads.config4(n_streams=90, seconds=0.12, seed=19),
    lambda: workloads.mixed(n_streams=67, seed=41, max_frames=4000),
    lambda: workloads.elements(5, n_streams=24),
    lambda: workloads.config5(n_streams=701, seconds=0.25),      # every block several slices
    lambda: workloads.config1(seconds=0.5),                       # one stream: all blocks but one are empty
], ids=["config4", "mixed", "elements", "config5_sliced", "one_stream"])
def test_blocks_of_streams_over_devices_give_the_bytes_one_device_gives(ctx, port, make):
    w = make()
    inp = port.fill_pcm(w.in_bytes, w.seed)
    want = np.full(w.out_bytes, 0xA5, dtype=np.uint8)             # gaps between streams stay as the caller left them
    want_outb, want_total = ctx.run_streams_host(w.streams, w.events, inp, want)
    want_sums = stream_checksums(port, want, w.streams, want_outb)
    for devices in device_lists():
        m = capi.MultiContext(devices)
        try:
            for _ in range(2):                                     # the second call reuses every device's buffers
                got = np.full(w.out_bytes, 0xA5, dtype=np.uint8)
                outb, sums, total = m.run_streams_host(w.streams, w.events, inp, got)
                assert total == want_total and np.array_equal(outb, want_outb), devices
                assert np.array_equal(got, want), devices
                assert np.array_equal(sums, want_sums), devices
        finally:
            m.close()


def test_streams_may_lie_anywhere_in_the_arenas(ctx, port):
    """Blocks are blocks of the specs ARRAY; where their streams sit in the arenas is the caller's business (here: reversed,
    so that block 0's bytes are the arenas' last)."""
    w = workloads.mixed(n_streams=48, seed=43, max_frames=3000)
    inp = port.fill_pcm(w.in_bytes, w.seed)
    streams = w.streams[::-1].copy()
    want = np.zeros(w.out_bytes, dtype=np.uint8)
    want_outb, _ = ctx.run_streams_host(streams, w.events, inp, want)
    m = capi.MultiContext([0, 0, 0])
    try:
        got = np.zeros(w.out_bytes, dtype=np.uint8)
        outb, sums, _ = m.run_streams_host(streams, w.events, inp, got)
        assert np.array_equal(got, want) and np.array_equal(outb, want_outb)
        assert np.array_equal(sums, stream_checksums(port, want, streams, want_outb))
    finally:
        m.close()


def interleaved_blocks(k=32):
    """2k streams for two blocks whose outputs interleave.  Block 0 (specs 0..k-1) is slow: k streams of 4 MiB in 9216-byte
    messages, 3500-byte holes between them.  Block 1 (specs k..2k-1) is quick: 3000-byte streams of one-frame messages
    ramped down and up, one in each of block 0's holes but the third, which nothing covers, and the rest far behind block
    0's last stream.  Block 1's walk is the longer one, so its bytes arrive after block 0 has walked its streams and saved
    its holes, and long before block 0's 128 MiB have crossed the bus twice."""
    rate0, rate1 = 384000, 44100
    big = workloads._spec(rate0, 32, 8, False, 288, (4 << 20) // 32)
    small = workloads._spec(rate1, 8, 1, False, 1, 3000)
    streams = np.array([big] * k + [small] * k, dtype=abi.STREAM_SPEC)
    jps = abi.jiffies_per_sample(rate1)
    events = np.zeros(2 * k, dtype=abi.RAMP_EVENT)
    for i in range(k):
        events[2 * i] = (0, 0, abi.EV_RAMP_DOWN, 1500 * jps, 0)
        events[2 * i + 1] = (1500 * jps, 0, abi.EV_RAMP_UP, 1500 * jps, 0)
        streams[k + i]["first_event"], streams[k + i]["num_events"] = 2 * i, 2
    hole, big_bytes, small_bytes = 3500, 4 << 20, 3000
    src = dst = 0
    holes = []
    for s in range(k):
        streams[s]["src_base"], streams[s]["dst_base"] = src, dst
        src += big_bytes
        dst += big_bytes
        if s + 1 < k:
            holes.append(dst)
            dst += hole
    empty = holes.pop(2)
    tail = dst + 8192
    for i, s in enumerate(range(k, 2 * k)):
        streams[s]["src_base"] = src
        src += small_bytes
        if holes:
            streams[s]["dst_base"] = holes.pop(0) + 1 + i % 7
        else:
            streams[s]["dst_base"] = tail
            tail += small_bytes + 8192
    return streams, events, src, tail, (empty, empty + hole)


def test_blocks_that_interleave_in_the_output_arena(ctx, port):
    """A block's host call bridges holes of up to 4 KiB between its output ranges with the device's bytes and puts the
    caller's bytes back when it ends.  Here the holes of slow block 0 hold quick block 1's streams, which are written while
    block 0's call is still running: every byte must still be what one context writes, a hole nobody covers keeps the
    caller's bytes, and each stream's checksum is that of its bytes."""
    streams, events, in_bytes, out_bytes, (e_lo, e_hi) = interleaved_blocks()
    assert capi.multi_shard(len(streams), 2, 1) == (len(streams) // 2, len(streams) // 2)
    inp = port.fill_pcm(in_bytes, 77)
    want = np.full(out_bytes, 0xA5, dtype=np.uint8)
    want_outb, want_total = ctx.run_streams_host(streams, events, inp, want)
    assert (want[e_lo:e_hi] == 0xA5).all()
    want_sums = stream_checksums(port, want, streams, want_outb)
    m = capi.MultiContext([0, 0])
    try:
        for _ in range(2):                                         # the second call runs on grown buffers: no allocation
            got = np.full(out_bytes, 0xA5, dtype=np.uint8)
            outb, sums, total = m.run_streams_host(streams, events, inp, got)
            assert total == want_total and np.array_equal(outb, want_outb)
            bad = np.nonzero(got != want)[0]
            assert bad.size == 0, "%d bytes differ from one context's, the first at %d (streams at %s)" % (
                bad.size, bad[0], [int(s) for s in np.nonzero((streams["dst_base"] <= bad[0]) &
                                                              (bad[0] < streams["dst_base"] + want_outb))[0]])
            assert np.array_equal(sums, want_sums)
    finally:
        m.close()


def test_pinned_buffers_and_errors(ctx, port):
    w = workloads.config5(n_streams=12, seconds=0.05)
    m = capi.MultiContext([0, 0])
    try:
        h_in, p_in = m.host_alloc(w.in_bytes)
        h_out, p_out = m.host_alloc(w.out_bytes)
        h_in[:] = port.fill_pcm(w.in_bytes, w.seed)
        h_out[:] = 0
        outb, sums, total = m.run_streams_host(w.streams, w.events, h_in, h_out)
        rc, want, chunks, _ = port.run(w.streams, w.events, h_in, w.out_bytes)
        assert rc == 0 and total == len(chunks) and np.array_equal(h_out, want)
        # nothing to do
        outb, sums, total = m.run_streams_host(w.streams[:0], w.events[:0], h_in, h_out)
        assert total == 0 and len(outb) == 0
        # a spec the message model cannot represent, in the second device's block: its status, its index, the stream's number
        bad = w.streams.copy()
        bad["sample_rate"][9] = 12345
        with pytest.raises(capi.OhpError) as e:
            m.run_streams_host(bad, w.events, h_in, h_out)
        assert e.value.status == abi.E_INVALID_ARG and "device index 1" in str(e.value) and "stream 3" in str(e.value) \
            and "counted from 6" in str(e.value)
        # a stream outside the arenas
        with pytest.raises(capi.OhpError) as e:
            m.run_streams_host(w.streams, w.events, h_in[:w.in_bytes // 2], h_out)
        assert e.value.status == abi.E_OUT_OF_RANGE and "device index 1" in str(e.value)
        # ... and everything still works
        h_out[:] = 0
        m.run_streams_host(w.streams, w.events, h_in, h_out)
        assert np.array_equal(h_out, want)
        m.host_free(p_in)
        m.host_free(p_out)
    finally:
        m.close()
