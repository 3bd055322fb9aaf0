"""Generators for the stage past 32 bits: streams longer than 2^32 jiffies (76.1 s), ramps of up to 2^32 - 1 jiffies,
the device walk's FP64 ramp recurrence at its edge cases, and arenas past 4 GiB.

Every position in the ABI is 64-bit, and the code narrows to 32 bits in many places behind a guard next to each
narrowing.  These inputs reach the values those guards exist for; each generator asserts that it does."""
import math

import numpy as np

from ohpipeline_b200 import abi
from ohpipeline_b200 import workloads as W

MS = abi.JIFFIES_PER_MS
SEC = abi.JIFFIES_PER_SECOND
T32, T33 = 1 << 32, 1 << 33
RATES = (7350, 8000, 11025, 44100)


def edges(jps, t):
    """t - 1, t, t + 1 and the sample boundaries on either side of t."""
    return [t - 1, t, t + 1, t // jps * jps, (t // jps + 1) * jps]


def _shape(rate, i):
    """(bits, channels, little endian, chunk_frames, codec_read_frames, driver_block_frames) of variant i at `rate`:
    uniform 5 ms messages, the largest messages a cell holds, AIFF-style block reads, a driver pulling blocks."""
    bits = (8, 16)[i % 2]
    ch = 1 + (i // 2) % 2 if rate != 44100 else 1
    fb = ch * bits // 8
    chunk = W.max_chunk_frames(rate, bits, ch)
    read = block = 0
    kind = (i // 4) % 4
    if kind == 1:
        chunk = abi.MAX_PCM_CHUNK_BYTES // fb // 4               # ~0.1-0.6 s messages
    elif kind == 2:
        read = abi.MAX_PCM_CHUNK_BYTES // fb                      # CodecAiffBase reads blocks
    elif kind == 3:
        block = rate // 100 + i                                   # a driver pulling ~10 ms blocks
    return bits, ch, bool((i // 3) % 2), chunk, read, block


def _stream(rate, i, seconds, events, out_fmt=abi.OUT_PACKED_BE):
    bits, ch, le, chunk, read, block = _shape(rate, i)
    sp = W._spec(rate, bits, ch, le, chunk, int(rate * seconds), out_fmt, block)
    sp["codec_read_frames"] = read
    return sp, events


def _ramps(rate, i):
    """Stage 0 ramps down across 2^32 and up across 2^33; stage 2 caps messages from 2^32 - 1 on; on 16-bit streams
    stage 3 attenuates from 2^32 + 1 to 2^33 + 1."""
    jps = abi.jiffies_per_sample(rate)
    d = (20 * MS, SEC + 7)[i % 2]
    ev = [(T32 - d, 0, abi.EV_RAMP_DOWN, 2 * d), (T33 - d, 0, abi.EV_RAMP_UP, 2 * d + 1),
          (edges(jps, T32)[i % 5], 2, abi.EV_MAX_MSG_JIFFIES, 3 * MS + jps)]
    if _shape(rate, i)[0] == 16:
        ev += [(T32 + 1, 3, abi.EV_SET_ATTENUATION, 100 + i), (T33 + 1, 3, abi.EV_SET_ATTENUATION, abi.UNITY_ATTENUATION)]
    return _stream(rate, i, 165 + 13 * i % 40, ev)


def _mutes(rate, i):
    """Mute / unmute at and beside 2^32 and 2^33 on stage 1; a ramp up after each unmute on stage 0."""
    jps = abi.jiffies_per_sample(rate)
    e32, e33 = edges(jps, T32), edges(jps, T33)
    ev = [(e32[i % 5], 1, abi.EV_MUTE, 0), (e32[(i + 2) % 5] + 1, 1, abi.EV_UNMUTE, 0),
          (e32[(i + 2) % 5] + 1, 0, abi.EV_MUTE, 0), (e32[(i + 2) % 5] + 1, 0, abi.EV_RAMP_UP, 50 * MS),
          (e33[(i + 1) % 5], 1, abi.EV_MUTE, 0), (e33[(i + 4) % 5] + 9 * MS, 1, abi.EV_UNMUTE, 0)]
    return _stream(rate, i, 160 + 11 * i % 50, ev)


def _long_arg(rate, i, p2):
    """Ramps whose arg is 2^32 - 1 (down, straddling 2^32) and 2^32 - jps (up).  Messages share a ramp rounded up
    (Ramp::Set), so a 2^32-jiffy ramp still moves; it stays audible, so a packed little-endian sink can take it."""
    jps = abi.jiffies_per_sample(rate)
    down = T32 - 3 * SEC - i * 1013
    ev = [(down, 0, abi.EV_RAMP_DOWN, T32 - 1), (T32 + SEC + 3, 0, abi.EV_RAMP_UP, T32 - jps),
          (T32 + 1, 1, abi.EV_RAMP_DOWN, T32 - 1), (T32 + 2 * SEC, 1, abi.EV_RAMP_UP, T32 - 1)]
    return _stream(rate, i, 90 + 7 * i % 40, ev, abi.OUT_PACKED_LE if p2 else abi.OUT_PACKED_BE)


def _silence(rate, i):
    """MsgSilence inserted at the first sample boundary past 2^32 and past 2^33, events on the sample grid elsewhere."""
    jps = abi.jiffies_per_sample(rate)
    s32, s33 = -(-T32 // jps) * jps, -(-T33 // jps) * jps
    sil = [(7 + i) * (rate // 1000) * jps, (30 + i) * (rate // 1000) * jps]
    ev = [(s32, 0, abi.EV_INSERT_SILENCE, sil[0]), (s33, 0, abi.EV_INSERT_SILENCE, sil[1]),
          (s32 - SEC // jps * jps, 1, abi.EV_RAMP_DOWN, 20 * MS // jps * jps),
          (s32 + 2 * SEC // jps * jps, 1, abi.EV_RAMP_UP, 50 * MS // jps * jps),
          (s33 + 3 * SEC // jps * jps, 2, abi.EV_MUTE, 0), (s33 + 4 * SEC // jps * jps, 2, abi.EV_UNMUTE, 0)]
    sp, ev = _stream(rate, i, 170 + 9 * i % 60, ev)
    fb = int(sp["channels"]) * int(sp["bit_depth"]) // 8
    return sp, ev, sum(s // jps for s in sil) * fb


def _elements(rate, i):
    """Ramper (stage 0), StarvationRamper (stage 1), Muter (stage 2) acting at and beside 2^32 and 2^33.  Nothing but
    PCM reaches the StarvationRamper before its first starvation past 2^32: recent_jiffies saturates there."""
    jps = abi.jiffies_per_sample(rate)
    e32, e33 = edges(jps, T32), edges(jps, T33)
    ev = [(0, 0, abi.EV_RAMPER_STREAM, 50 * MS), (e32[(i + 1) % 5], 0, abi.EV_RAMPER_STREAM, 50 * MS),
          (e32[i % 5], 1, abi.EV_STARVATION, 50 * MS), (e32[i % 5] + 200 * MS + i, 1, abi.EV_STARVATION, 50 * MS),
          (e33[(i + 3) % 5], 1, abi.EV_STARVATION, 50 * MS), (e33[(i + 3) % 5] + 30 * MS, 1, abi.EV_STARVATION, 50 * MS),
          (e32[(i + 2) % 5], 2, abi.EV_MUTER_MUTE, 30 * MS), (e32[(i + 2) % 5] + 100 * MS, 2, abi.EV_MUTER_UNMUTE, 30 * MS),
          (e33[(i + 4) % 5], 2, abi.EV_MUTER_MUTE, 30 * MS), (e33[(i + 4) % 5] + 10 * MS, 2, abi.EV_HALT, 0),
          (e33[(i + 4) % 5] + 500 * MS, 2, abi.EV_MUTER_UNMUTE, 30 * MS), (e33[i % 5] + SEC, 0, abi.EV_HALT, 0)]
    if _shape(rate, i)[0] == 16:
        ev.append((T33 + 2 * SEC, 3, abi.EV_SET_ATTENUATION, 200))
    return _stream(rate, i, 160 + 17 * i % 60, ev)


def long_streams():
    """40 streams of 90-225 s at 7350, 8000, 11025 and 44100 Hz (8/16-bit, 1-2 channels, both wire endians, P1 and P2
    out, uniform messages, AIFF block reads, driver blocks) with events at and beside 2^32 and 2^33 jiffies."""
    specs, evs, slack = [], [], []
    for r, rate in enumerate(RATES):
        for k in range(10):
            i = 10 * r + k
            kind = k % 5
            extra = 0
            if kind == 0:
                sp, ev = _ramps(rate, i)
            elif kind == 1:
                sp, ev = _mutes(rate, i)
            elif kind == 2:
                sp, ev = _long_arg(rate, i, p2=k >= 5)
            elif kind == 3:
                sp, ev, extra = _silence(rate, i)
            else:
                sp, ev = _elements(rate, i)
            specs.append(sp)
            evs.append(ev)
            slack.append(extra)
    w = W._finish("long streams", specs, evs, seed=(9 << 32) + 1, slack=slack)
    # coverage: the generator reaches what it is for
    ends = w.streams["total_frames"].astype(np.uint64) * np.array([abi.jiffies_per_sample(int(r)) for r in w.streams["sample_rate"]], np.uint64)
    assert (ends > T33).sum() >= 30 and ends.min() > T32
    at, arg, op = w.events["at_jiffies"], w.events["arg"], w.events["op"]
    assert ((at > T32) & (at < T33)).sum() >= 80 and (at > T33).sum() >= 80
    ramp = (op == abi.EV_RAMP_DOWN) | (op == abi.EV_RAMP_UP)
    assert (ramp & (arg == T32 - 1)).any() and (ramp & (arg >= T32 - (1 << 16)) & (arg < T32 - 1)).any()
    assert ((op == abi.EV_STARVATION) & (at > T32)).sum() >= 30
    assert ((op == abi.EV_INSERT_SILENCE) & (at > T32)).sum() >= 8
    assert (w.streams["out_fmt"] == abi.OUT_PACKED_LE).sum() >= 4
    return w


def split(w, keep):
    """The streams of w with keep(k) true, as a workload of their own (same layout rules, same seed)."""
    idx = [k for k in range(len(w.streams)) if keep(k)]
    specs, evs = [], []
    for k in idx:
        s = w.streams[k]
        lo = int(s["first_event"])
        evs.append([tuple(int(x) for x in e)[:4] for e in w.events[lo:lo + int(s["num_events"])]])
        specs.append(s.copy())
    slack = [0] * len(idx)
    out = W._finish(w.name, specs, evs, seed=w.seed)
    # keep each stream's room for inserted silence: the output layout is the sum of what every stream writes
    for j, k in enumerate(idx):
        slack[j] = int(w.streams["dst_base"][k + 1] if k + 1 < len(w.streams) else w.out_bytes) - int(w.streams["dst_base"][k])
    dst = 0
    for j in range(len(idx)):
        out.streams["dst_base"][j] = dst
        dst += slack[j]
    out.out_bytes = dst
    return out


# ------------------------------------------------------------------------------------------------------------------
# the FP64 ramp recurrence

FP64_KINDS = ("minus1", "exact", "plus1")   # numerator = q * divisor - 1, q * divisor, q * divisor + 1


def recurrence(distance, size, remaining, n):
    """The bulk step's ramp recurrence in Python integers: per message (distance, remaining, numerator, delta), until
    delta is 0 or reaches distance (the walk's general path takes over there) or the ramp ends."""
    out = []
    for _ in range(n):
        if remaining < size or distance == 0:
            break
        num = distance * size + remaining - 1
        delta = num // remaining
        out.append((distance, remaining, num, delta))
        if delta == 0 or delta >= distance:
            break
        distance -= delta
        remaining -= size
    return out


def kind_of(num, rem):
    r = num % rem
    return "exact" if r == 0 else "minus1" if r == rem - 1 else "plus1" if r == 1 else None


def _solve(size, k, c, m, dist0=abi.RAMP_MAX):
    """A ramp length whose message k has numerator distance * size + remaining - 1 = m' * remaining + (c - 1), i.e.
    distance * size - c = m * remaining.  The length is k * size + (d * size - c) / m for the distance d message k
    starts with, which itself depends on the length: try the distances near the first guess, None where none fits."""
    if math.gcd(size, m) != 1:
        return None
    f = lambda d: recurrence(dist0, size, k * size + max(size, (d * size - c) // m), k + 1)  # noqa: E731
    d = dist0
    while d > 1:                                   # where the distance message k starts with meets the one asked for
        rec = f(d)
        if len(rec) <= k:
            return None
        if rec[k][0] >= d:
            break
        d = rec[k][0]
    r0 = c * pow(size, -1, m) % m                  # d * size = c (mod m)
    for d in range(d + 2 * m, max(d - 2 * m, 0), -1):
        if d % m != r0:
            continue
        rem = (d * size - c) // m
        if rem <= size or rem + k * size >= T32:
            continue
        rec = recurrence(dist0, size, rem + k * size, k + 1)
        if len(rec) > k and rec[k][0] == d:
            return rem + k * size
    return None


def fp64_edge_streams():
    """Streams whose ramps steer the device walk's FP64 recurrence (schedule_walk.h, bulk_step: a warp's team, uniform
    messages below 2^21 jiffies, one stage ramping) onto its edge cases: for some message k >= 1 of the ramp the
    numerator distance * size + remaining - 1 is q * remaining - 1, q * remaining or q * remaining + 1, with remaining
    up to 2^32 - 1 and distance from 1 to 16384; also ramps that end exactly on a message boundary and ramps that
    arrive early (delta >= distance).  Each stream is one uniform codec, no driver blocks, one stage-0 ramp from the
    first message boundary on and no other event: message 0 takes the general path (its event applies), every later
    message of the ramp lies in a bulk run, so with a team of 32 the FP64 branch evaluates it.
    Returns (workload, cases): cases = [(distance, size, remaining, kind)] the streams produce, checked here."""
    rng = np.random.default_rng(64)
    specs, evs, cases = [], [], []
    kinds = {k: 0 for k in FP64_KINDS}
    small_dist = big_rem = early = exact_end = 0
    rates = (48000, 44100, 7350, 384000, 192000, 8000)
    t = 0
    while len(specs) < 96:
        t += 1
        rate = rates[t % len(rates)]
        jps = abi.jiffies_per_sample(rate)
        cmax = min(W.max_chunk_frames(rate, 8, 1, ms=40), ((1 << 21) - 1) // jps, abi.MAX_PCM_CHUNK_BYTES)
        chunk = int(rng.integers(1, cmax + 1)) if t % 3 else cmax
        size = chunk * jps
        assert size < (1 << 21)
        mode = len(specs) % 8                  # a case that does not solve is drawn again with other parameters
        up = len(specs) % 2 == 1
        if mode < 6:
            k = int(rng.integers(1, 40)) if mode < 3 else int(rng.integers(40, 600))
            c = mode % 3
            # the smallest m keeps remaining just below 2^32
            m = abi.RAMP_MAX * size // T32 + 1 + (int(rng.choice((0, 0, 0, 1, 2, 4))) if mode < 3 else 0)
            while math.gcd(size, m) != 1:
                m += 1
            arg = _solve(size, k, c, m)
            if arg is None:
                continue
        elif mode == 6:
            arg = int(rng.integers(2, min(600, T32 // size))) * size                      # the ramp ends on a message boundary
        else:
            arg = int(rng.integers(size + 1, 60 * size))                  # ... and arrives early
        rec = recurrence(abi.RAMP_MAX, size, arg, 1 << 20)
        n_msgs = min(len(rec) + 2, k + 40 if mode < 6 else 1 << 12)
        ev = [(0, 0, abi.EV_MUTE, 0), (0, 0, abi.EV_RAMP_UP, arg)] if up else [(0, 0, abi.EV_RAMP_DOWN, arg)]
        sp = W._spec(rate, 8, 1, False, chunk, n_msgs * chunk)
        specs.append(sp)
        evs.append(ev)
        for j, (dist, rem, num, delta) in enumerate(rec[:n_msgs]):
            kd = kind_of(num, rem)
            if j >= 1 and kd is not None:
                cases.append((dist, size, rem, kd))
                kinds[kd] += 1
                small_dist += dist < 64
                big_rem += rem >= T32 - (1 << 28)
        last = rec[-1] if rec else None
        early += bool(last and last[3] >= last[0] and len(rec) > 1)
        exact_end += arg % size == 0 and len(rec) * size == arg
    assert min(kinds.values()) >= 20, kinds
    assert small_dist >= 1 and big_rem >= 3 and early >= 5 and exact_end >= 1, (small_dist, big_rem, early, exact_end)
    w = W._finish("fp64 edges", specs, evs, seed=(10 << 32) + 1)
    return w, cases


# ------------------------------------------------------------------------------------------------------------------
# arenas past 4 GiB

def far_arena_layout(w, base=T32):
    """w's streams moved up in both arenas by multiples of 16 (offsets mod 16 kept), 64 bytes apart: stream 0 straddles
    `base` in the input arena and stream 1 in the output arena, every later stream lies above `base`.  Returns
    (streams, in_bytes, out_bytes, in_sentinels, out_sentinels): sentinel offsets just below every stream and where
    an address truncated to 32 bits would land (offset mod 2^32), none inside a stream."""
    st = w.streams.copy()
    n = len(st)
    assert n >= 2
    fb = st["channels"].astype(np.int64) * (st["bit_depth"].astype(np.int64) // 8)
    in_len = st["total_frames"].astype(np.int64) * fb
    out_len = [int(st["dst_base"][k + 1] if k + 1 < n else w.out_bytes) - int(st["dst_base"][k]) for k in range(n)]

    def place(lens, orig, straddler):
        pos = np.zeros(n, dtype=np.int64)
        # the straddler's middle on `base`; the streams before it below, the rest after it
        at = (base - lens[straddler] // 2) // 16 * 16
        start = at - sum(-(-int(lens[k]) // 16) * 16 + 64 for k in range(straddler))
        cur = start
        for k in range(n):
            pos[k] = cur + int(orig[k]) % 16
            cur += -(-(int(lens[k]) + int(orig[k]) % 16) // 16) * 16 + 64
        assert pos[straddler] < base < pos[straddler] + lens[straddler]
        return pos, cur + 64

    src, in_bytes = place(in_len, st["src_base"], 0)
    dst, out_bytes = place(np.array(out_len), st["dst_base"], 1)
    st["src_base"], st["dst_base"] = src.astype(np.uint64), dst.astype(np.uint64)

    def sentinels(pos, lens):
        cand = set()
        for p, ln in zip(pos, lens):
            p, ln = int(p), int(ln)
            cand.update({p - 1, p % T32, (p + ln - 1) % T32, (p + ln) % T32})
            if p < T32 <= p + ln:
                cand.update({0, 1, (p + ln - 1) % T32})
        inside = lambda x: any(int(p) <= x < int(p) + int(ln) for p, ln in zip(pos, lens))  # noqa: E731
        return np.array(sorted(x for x in cand if not inside(x)), dtype=np.int64)

    s_in, s_out = sentinels(src, in_len), sentinels(dst, out_len)
    assert len(s_in) >= 2 * n and len(s_out) >= 2 * n
    assert min(int(p) for p in src) < T32 and all(int(p) >= base - (1 << 26) for p in src)
    return st, int(in_bytes), int(out_bytes), s_in, s_out
