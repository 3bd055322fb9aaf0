"""The hot path's descriptor space on the CPU: classify() against hand-worked chunks, the matrix batches of
descriptor_space.py against every cell of that classification (the coverage guard), the validator and the C oracle
against every batch, and streams at 9-32 channels through the schedule: the class model, the class-free walk, the
oracle's own schedule and the closed-form bound agree.  tests/test_gpu_descriptor_space.py runs the same batches and
streams on the GPU."""
import numpy as np
import pytest

from ohpipeline_b200 import abi, capi
import descriptor_space as D
from util import make_desc

R, IL, S = abi.F_RAMP_ENABLED, abi.F_IN_LITTLE_ENDIAN, abi.F_SILENCE


@pytest.fixture(scope="module")
def matrix(port):
    return D.batches(port)


def one(**kw):
    return D.classify(make_desc(**kw))[0]


def test_classify_restates_the_loader():
    c = one(bytes=64, bit_depth=16, channels=2, flags=R, src_off=32, dst_off=5)
    assert (c["kind"], c["path"], c["chm"], c["aligned"], c["img_phase"], c["dst_phase"]) == (D.K_PCM, D.P_WIDE_STEREO, D.CHM_STEREO, True, 0, 5)
    assert c["mode"] == D.M_RAMPED | D.M_TRANSFORM and c["length"] == D.L_ANY          # 32 subsamples
    # a head off the 16-byte boundary: the general path, whatever the channel layout
    assert one(bytes=64, bit_depth=16, channels=2, flags=R, src_off=33)["path"] == D.P_ANY
    assert one(bytes=96, bit_depth=8, channels=12, flags=R)["path"] == D.P_WIDE_MUL4
    assert one(bytes=90, bit_depth=8, channels=9, flags=R)["path"] == D.P_ANY
    # verbatim: the image leaves from where it landed; little-endian in and out is verbatim too
    c = one(bytes=30, bit_depth=24, channels=10, src_off=7, dst_off=3)
    assert (c["path"], c["img_phase"], c["head"], c["length"]) == (D.P_VERBATIM, 7, 7, D.L_GROUP)
    assert one(bytes=60, bit_depth=24, channels=10, flags=IL, out_fmt=abi.OUT_PACKED_LE, aux=1)["path"] == D.P_VERBATIM
    # little-endian in, 8-bit: nothing to swap
    assert one(bytes=60, bit_depth=8, channels=10, flags=IL)["path"] == D.P_VERBATIM
    # attenuation alone transforms; the tag on 6 channels
    c = one(bytes=12, bit_depth=16, channels=6, attenuation=255)
    assert c["path"] == D.P_ANY and c["mode"] == D.M_TAG6 | D.M_TRANSFORM and c["length"] == D.L_GROUP  # 6 subsamples
    assert one(bytes=8, bit_depth=16, channels=4, flags=R)["length"] == D.L_UNIT
    # the packed-LE sink to the letter: the image's last fragment (256 // 27 = 9 frames a fragment: frame 9 of 10)
    c = one(bytes=10 * 27, bit_depth=24, channels=9, flags=R, out_fmt=abi.OUT_PACKED_LE, aux=0, src_off=16)
    assert c["path"] == D.P_ANY and c["img_phase"] == (9 * 27) % 16
    # silence: packed -> written straight out, any length; converting -> through the slot, head 0
    c = one(bytes=3 * 9216, bit_depth=8, channels=7, flags=S | R, src_off=3)
    assert (c["kind"], c["path"], c["head"], c["length"], c["mode"]) == (D.K_SILENCE, D.P_SILENCE, 0, D.L_OVER, 0)
    c = one(bytes=9216, bit_depth=32, channels=32, flags=S, out_fmt=abi.OUT_SONGCAST, aux=30)
    assert (c["kind"], c["path"], c["length"]) == (D.K_SILENCE_CONV, D.P_SONGCAST, D.L_MAX)
    assert one(bytes=9212, bit_depth=32, channels=1, out_fmt=abi.OUT_FROM32_BE, aux=8)["length"] == D.L_LONG
    assert one(bytes=64, bit_depth=32, channels=1, out_fmt=abi.OUT_PLANAR32_BE, aux=16)["img_phase"] == -1
    assert one(bytes=0, bit_depth=32, channels=1)["path"] == D.P_SKIP


def mode_name(d):
    """The packed-sink modes of the matrix, as a descriptor spells them."""
    parts = []
    if d["flags"] & R:
        parts.append({(9000, 9000): "flat", (16384, 0): "down", (0, 16384): "up"}.get(
            (int(d["ramp_start"]), int(d["ramp_end"])), "ramped"))
    if d["flags"] & IL and d["bit_depth"] > 8:
        parts.append("le_in")
    if d["out_fmt"] == abi.OUT_PACKED_LE and d["bit_depth"] > 8:
        parts.append("le_out_letter" if (d["flags"] & R and d["aux"] == 0) else "le_out")
    if d["attenuation"] != abi.UNITY_ATTENUATION:
        parts.append("att%d" % d["attenuation"])
    return "+".join(parts) or "verbatim"


def required_modes(B):
    m = ["verbatim", "ramped", "flat", "down", "up"]
    if B >= 2:
        m += ["le_in", "ramped+le_in"]
    if B in (2, 3):
        m += ["le_out", "le_in+le_out", "ramped+le_out_letter", "ramped+le_in+le_out_letter", "ramped+le_in+le_out"]
    if B == 2:
        for a in (0, 1, 255, 257, 65535):
            m += ["att%d" % a, "ramped+att%d" % a, "le_in+le_out+att%d" % a]
    return m


def pow2_lengths(B, ch):
    return {n for k in range(1, 14) for n in (2 ** k - 1, 2 ** k, 2 ** k + 1) if n * B * ch <= D.MAX}


def required_cells():
    """family -> set of cells the matrix must hit."""
    req = {}
    req["mode"] = {(B, ch, m, h0) for B in D.DEPTHS for ch in D.CHANNELS for m in required_modes(B) for h0 in (True, False)}
    req["pair"] = {(B, chm, t, h, p) for B in D.DEPTHS for chm in range(4) for t in (True, False) for h in range(16)
                   for p in range(16)}
    req["length"] = {(path, B, ln) for path in (D.P_WIDE_STEREO, D.P_WIDE_MUL4, D.P_ANY, D.P_VERBATIM, D.P_PLANAR, D.P_SONGCAST)
                     for B in D.DEPTHS for ln in range(D.L_OVER)}
    req["length"] |= {(D.P_FROM32, 4, ln) for ln in range(D.L_OVER)} | {(D.P_SILENCE, B, ln) for B in D.DEPTHS for ln in range(7)}
    req["sink"] = {(path, B, ch, kind) for path, kinds in ((D.P_PLANAR, (D.K_PCM, D.K_SILENCE_CONV)),
                                                           (D.P_SONGCAST, (D.K_PCM, D.K_SILENCE_CONV)))
                   for B in D.DEPTHS for ch in D.CHANNELS for kind in kinds}
    req["sink"] |= {(D.P_FROM32, 4, ch, D.K_PCM) for ch in D.CHANNELS}
    req["planar"] = {(B, extra, p) for B in D.DEPTHS for extra in (0, 1, 3) for p in range(4)}
    req["from32"] = {(ob, h) for ob in (8, 16, 24, 32) for h in range(16)} | {(ob, ch) for ob in (8, 16, 24, 32) for ch in D.CHANNELS}
    req["songcast"] = {(B, h, first) for B in D.DEPTHS for h in range(16) for first in ("0", "1", "ch-2")}
    req["silence_block"] = {(B, ch, k, e) for B in D.DEPTHS for ch in D.CHANNELS for k in (1, 2, 3) for e in (-1, 0, 1)}
    req["ramp_16bit"] = {(n, r, v) for n in range(1, 4609) for r in D.RAMP_PAIRS_16 for v in (0x7FFF, 0x8000)}
    req["ramp_8bit"] = {(n, r, v) for n in range(4609, 9217) for r in ((16384, 0), (0, 16384)) for v in (0x7F, 0x80)}
    req["ramp_pow2"] = {(B, chm, n) for B in D.DEPTHS for chm, ch in ((D.CHM_MONO, 1), (D.CHM_STEREO, 2), (D.CHM_OTHER, 3),
                                                                        (D.CHM_MUL4, 4)) for n in pow2_lengths(B, ch)}
    return req


def hit_cells(batches):
    hit = {k: set() for k in required_cells()}
    for b in batches:
        d = {f: b.descs[f].tolist() for f in abi.CHUNK_DESC.names}
        c = {f: b.cls[f].tolist() for f in D.CLASS.names}
        for i in range(len(b.descs)):
            di = {f: v[i] for f, v in d.items()}
            path, B, ch, head = c["path"][i], c["B"][i], di["channels"], c["head"][i]
            frames = di["bytes"] // (B * ch)
            if path in (D.P_WIDE_STEREO, D.P_WIDE_MUL4, D.P_ANY, D.P_VERBATIM):
                hit["mode"].add((B, ch, mode_name(di), head == 0))
                hit["pair"].add((B, c["chm"][i], bool(c["mode"][i] & D.M_TRANSFORM), head, c["dst_phase"][i]))
            if path != D.P_SKIP:
                hit["length"].add((path, B, c["length"][i]))
            if path in (D.P_PLANAR, D.P_SONGCAST, D.P_FROM32):
                hit["sink"].add((path, B, ch, c["kind"][i]))
            if path == D.P_PLANAR:
                hit["planar"].add((B, di["aux"] - frames, c["dst_phase"][i] % 4))
            if path == D.P_FROM32:
                hit["from32"] |= {(di["aux"], head), (di["aux"], ch)}
            if path == D.P_SONGCAST and ch >= 4:
                a = di["aux"]
                hit["songcast"].add((B, head, "0" if a == 0 else "1" if a == 1 else "ch-2" if a == ch - 2 else "other"))
            if path == D.P_SILENCE:
                fb = B * ch
                block = D.MAX - D.MAX % fb
                q, r = divmod(di["bytes"], block)
                if r in (0, fb, block - fb):
                    hit["silence_block"].add((B, ch, q + (r == block - fb), {0: 0, fb: 1}.get(r, -1)))
            if di["flags"] & R and not di["flags"] & S and path != D.P_SKIP:
                ramp = (di["ramp_start"], di["ramp_end"])
                if ch == 1 and B in (1, 2):   # the ramp-length batches: a constant sample, its value where the chunk starts
                    o = di["src_off"]
                    hit["ramp_16bit" if B == 2 else "ramp_8bit"].add((frames, ramp, int.from_bytes(b.inp[o:o + B].tobytes(), "big")))
                hit["ramp_pow2"].add((B, c["chm"][i], frames))
    return hit


def test_coverage_guard(matrix):
    """Every required cell is hit by some chunk of the matrix; the failure names the missing cells."""
    req, hit = required_cells(), hit_cells(matrix)
    missing = {k: sorted(req[k] - hit[k], key=str) for k in req}
    total = sum(len(v) for v in req.values())
    report = "; ".join("%s: %d of %d missing, e.g. %s" % (k, len(v), len(req[k]), v[:8]) for k, v in missing.items() if v)
    assert not report, report
    print("\ncoverage guard: %d cells required (%s), every one hit by the %d chunks of %d batches" % (
        total, ", ".join("%s %d" % (k, len(v)) for k, v in req.items()), sum(len(b.descs) for b in matrix), len(matrix)))


def test_the_validator_and_the_oracle_take_every_batch(matrix, port):
    for b in matrix:
        assert capi.validate(b.descs, b.in_bytes, b.out_bytes) == (0, 0), b.name
        rc, _ = port.process_chunks(b.descs, b.inp[:b.in_bytes], b.out_bytes)
        assert rc == 0, (b.name, -rc - 1)
        # the input arena ends where a chunk ends (the tail past it is poison the kernel must not read)
        d = b.descs[(b.descs["flags"] & S) == 0]
        if len(d):
            assert int((d["src_off"] + d["bytes"]).max()) == b.in_bytes, b.name
        assert D.covered(b.descs, b.out_bytes).any()


# ------------------------------------------------------------------------------------------------------------------
# the stage at 9-32 channels

@pytest.fixture(scope="module")
def wide():
    return D.wide_streams()


def test_wide_streams_span_the_channel_counts(wide):
    chans = set(np.concatenate([w.streams["channels"] for w in wide]).tolist())
    assert chans == set(range(9, 33))
    st = np.concatenate([w.streams for w in wide])
    assert set(st["bit_depth"].tolist()) == {8, 16, 24, 32} and set(st["in_little_endian"].tolist()) == {0, 1}
    assert set(st["out_fmt"].tolist()) == {abi.OUT_PACKED_BE, abi.OUT_PACKED_LE}
    assert (st["driver_block_frames"] > 0).any() and (st["codec_read_frames"] > 0).any()
    ops = set(np.concatenate([w.events["op"] for w in wide]).tolist())
    assert ops == set(range(1, 13))


@pytest.mark.parametrize("k", range(7))
def test_wide_streams_walk_model_oracle_and_bound(wide, port, k):
    w = wide[k]
    host = capi.schedule_build(w.streams, w.events)
    walk = capi.schedule_build(w.streams, w.events, walk=True)
    for f in ("chunks", "info", "stream_chunk_begin", "stream_out_bytes"):
        assert np.array_equal(getattr(walk, f), getattr(host, f)), (w.name, f)
    assert (host.chunks["channels"] >= 9).all()
    inp = port.fill_pcm(w.in_bytes, w.seed)
    rc, want, chunks, _ = port.run(w.streams, w.events, inp, w.out_bytes)
    assert rc == 0, w.name
    assert np.array_equal(chunks, host.chunks), w.name
    rc, got = port.process_chunks(host.chunks, inp, w.out_bytes)
    assert rc == 0 and np.array_equal(got, want), w.name
    bounds = capi.schedule_chunk_bounds(w.streams, w.events)
    exact = np.diff(host.stream_chunk_begin.astype(np.int64))
    assert (exact <= bounds.astype(np.int64)).all(), (w.name, np.nonzero(exact > bounds.astype(np.int64))[0])
