"""The hot path's descriptor space, enumerated: classify() restates how ramp_convert_kernel's loader classifies a chunk
(decode_chunk in csrc/ohp_ramp_convert_kernel.cuh) and which consumer path it then takes (transform_dispatch and the sink
switch), and the generators below lay out deterministic batches that reach every cell of that classification at 1-32
channels.  tests/test_descriptor_space.py proves the coverage on the CPU; tests/test_gpu_descriptor_space.py runs the
batches on the GPU against the C oracle.  Also here: streams at 9-32 channels for the whole stage."""
import numpy as np

from ohpipeline_b200 import abi
from ohpipeline_b200 import workloads as W

MAX = abi.MAX_PCM_CHUNK_BYTES
POISON = 0xEE
CHANNELS = range(1, 33)
DEPTHS = (1, 2, 3, 4)

# kChm* of ohp_kernels.cuh
CHM_OTHER, CHM_MONO, CHM_STEREO, CHM_MUL4 = 0, 1, 2, 3
CHM_NAMES = ("other", "mono", "stereo", "mul4")
# kMode* of ohp_kernels.cuh
M_RAMPED, M_IN_LE, M_OUT_LE, M_TAG6, M_TRANSFORM = 1, 2, 4, 8, 16
# ChunkKind of ohp_kernels.cuh
K_SKIP, K_PCM, K_SILENCE, K_SILENCE_CONV = 0, 1, 2, 3
KIND_NAMES = ("skip", "pcm", "silence", "silence_conv")
PATHS = ("skip", "wide_stereo", "wide_mul4", "any", "verbatim", "planar", "from32", "songcast", "write_silence")
P_SKIP, P_WIDE_STEREO, P_WIDE_MUL4, P_ANY, P_VERBATIM, P_PLANAR, P_FROM32, P_SONGCAST, P_SILENCE = range(9)
# length classes by subsample count: a unit (4), a group (16), a lane step of transform_any (32 units = 128) and of
# transform_wide (32 groups = 512), longer, the largest whole-frame chunk <= 9216 bytes, and silence beyond that
LENGTHS = ("unit", "group", "any_step", "wide_step", "long", "max", "over")
L_UNIT, L_GROUP, L_ANY, L_WIDE, L_LONG, L_MAX, L_OVER = range(7)

CLASS = np.dtype([("kind", "u1"), ("B", "u1"), ("chm", "u1"), ("aligned", "?"), ("mode", "u1"), ("path", "u1"),
                  ("head", "u1"), ("img_phase", "i1"), ("dst_phase", "u1"), ("length", "u1")])


def chm_of(ch):
    ch = np.asarray(ch)
    return np.where(ch == 2, CHM_STEREO, np.where(ch % 4 == 0, CHM_MUL4, np.where(ch == 1, CHM_MONO, CHM_OTHER)))


def classify(descs, in_base=0, out_base=0):
    """Per chunk, what the loader decides (in_base / out_base: the arenas' device addresses, or just their phase mod 16).
    img_phase: where the finished image starts mod 16 when it is stored (-1: the sink writes global memory itself, or
    nothing is stored)."""
    d = np.asarray(descs)
    n = len(d)
    c = np.zeros(n, dtype=CLASS)
    B = (d["bit_depth"] // 8).astype(np.int64)
    ch = d["channels"].astype(np.int64)
    nbytes = d["bytes"].astype(np.int64)
    flags = d["flags"].astype(np.int64)
    fmt = d["out_fmt"].astype(np.int64)
    silence = (flags & abi.F_SILENCE) != 0
    packed = fmt <= abi.OUT_PACKED_LE
    kind = np.where(nbytes == 0, K_SKIP, np.where(silence, np.where(packed, K_SILENCE, K_SILENCE_CONV), K_PCM))
    head = np.where(silence, 0, (int(in_base) + d["src_off"].astype(np.int64)) & 15)
    ramped = ((flags & abi.F_RAMP_ENABLED) != 0) & ~silence
    in_le = ((flags & abi.F_IN_LITTLE_ENDIAN) != 0) & (B > 1) & ~silence
    out_le = (fmt == abi.OUT_PACKED_LE) & (B > 1)
    att = np.where(silence, abi.UNITY_ATTENUATION, d["attenuation"].astype(np.int64))
    transform = ramped | (in_le != out_le) | (att != abi.UNITY_ATTENUATION)
    mode = (ramped * M_RAMPED) | (in_le * M_IN_LE) | (out_le * M_OUT_LE) | ((ch == 6) * M_TAG6) | (transform * M_TRANSFORM)
    chm = chm_of(ch)
    aligned = head == 0
    path = np.full(n, P_SKIP)
    conv = (kind == K_PCM) | (kind == K_SILENCE_CONV)
    path[conv & packed & transform] = P_ANY
    path[conv & packed & transform & aligned & (chm == CHM_STEREO)] = P_WIDE_STEREO
    path[conv & packed & transform & aligned & (chm == CHM_MUL4)] = P_WIDE_MUL4
    path[conv & packed & ~transform] = P_VERBATIM
    path[conv & (fmt == abi.OUT_PLANAR32_BE)] = P_PLANAR
    path[conv & (fmt == abi.OUT_FROM32_BE)] = P_FROM32
    path[conv & (fmt == abi.OUT_SONGCAST)] = P_SONGCAST
    path[kind == K_SILENCE] = P_SILENCE
    out = abi.chunk_out_bytes(d).astype(np.int64)
    img = np.full(n, -1)
    img[(path == P_ANY) | (path == P_WIDE_STEREO) | (path == P_WIDE_MUL4) | (path == P_FROM32) | (path == P_SONGCAST)] = 0
    img[path == P_VERBATIM] = head[path == P_VERBATIM]
    # the packed little-endian sink keeps only the tail of a ramped image ("to the letter", aux 0)
    le = packed & (fmt == abi.OUT_PACKED_LE) & (path != P_SKIP) & (path != P_SILENCE)
    img[le] = (img[le] + nbytes[le] - out[le]) & 15
    img[out == 0] = -1
    sub = nbytes // np.maximum(B, 1)
    fb = np.maximum(B * ch, 1)
    length = np.select([sub <= 4, sub <= 16, sub <= 128, sub <= 512, nbytes > MAX, nbytes + fb > MAX],
                       [L_UNIT, L_GROUP, L_ANY, L_WIDE, L_OVER, L_MAX], L_LONG)
    c["kind"], c["B"], c["chm"], c["aligned"], c["mode"], c["path"] = kind, B, chm, aligned, mode, path
    c["head"], c["img_phase"], c["dst_phase"], c["length"] = head, img, (int(out_base) + d["dst_off"].astype(np.int64)) & 15, length
    return c


def describe(cell):
    return "%s B=%d %s%s mode=%s path=%s head=%d image@%d dst@%d length=%s" % (
        KIND_NAMES[cell["kind"]], cell["B"], CHM_NAMES[cell["chm"]], " aligned" if cell["aligned"] else "",
        "|".join(n for b, n in ((M_RAMPED, "ramped"), (M_IN_LE, "in_le"), (M_OUT_LE, "out_le"), (M_TAG6, "tag6"),
                                (M_TRANSFORM, "transform")) if cell["mode"] & b) or "0",
        PATHS[cell["path"]], cell["head"], cell["img_phase"], cell["dst_phase"], LENGTHS[cell["length"]])


# ------------------------------------------------------------------------------------------------------------------
# layout

def frame_counts(B, ch):
    """Whole-frame chunk sizes through every length class: 1-3 frames, the frame counts whose subsample count lands on or
    next to 4k for k in (1, 4, 32, 128, 512), and the largest whole-frame size <= 9216 bytes."""
    fb = B * ch
    top = MAX // fb
    out = {1, 2, 3, top}
    for t in (4, 16, 128, 512, 2048):
        out |= {(t - 1) // ch, t // ch, t // ch + 1, (t + ch - 1) // ch}
    return sorted(f for f in out if 1 <= f <= top)


class Specs:
    """Columns of a batch under construction: one chunk per add(), the layout is done at once by lay_out()."""

    def __init__(self):
        self.cols = {k: [] for k in ("bytes", "bit_depth", "channels", "flags", "ramp_start", "ramp_end", "attenuation",
                                     "out_fmt", "aux", "head", "dst_phase", "src")}

    def add(self, B, ch, frames, flags=0, out_fmt=abi.OUT_PACKED_BE, aux=0, ramp=(abi.RAMP_MAX, abi.RAMP_MAX),
            att=abi.UNITY_ATTENUATION, head=0, dst_phase=0, bytes_=None, src=-1):
        """src: -1 = a fresh stretch of input; k >= 0 = the shared source region k (see lay_out)."""
        c = self.cols
        c["bytes"].append(frames * B * ch if bytes_ is None else bytes_)
        c["bit_depth"].append(8 * B)
        c["channels"].append(ch)
        c["flags"].append(flags)
        c["ramp_start"].append(ramp[0])
        c["ramp_end"].append(ramp[1])
        c["attenuation"].append(att)
        c["out_fmt"].append(out_fmt)
        c["aux"].append(aux)
        c["head"].append(head)
        c["dst_phase"].append(dst_phase)
        c["src"].append(src)

    def __len__(self):
        return len(self.cols["bytes"])

    def lay_out(self, shared=()):
        """-> (descs, src_region_of_each_shared_source, in_bytes, out_bytes).  Every chunk starts at its head mod 16 in
        the input and at its dst_phase mod 16 in the output, 16 bytes or more from its neighbours (bytes between chunks
        keep the fill).  Chunks with src = k read the shared region k: len(shared[k]) bytes placed once at a 16-byte
        boundary, read from offset head.  The input arena ends exactly where the last fresh chunk ends."""
        c = {k: np.asarray(v, dtype=np.int64) for k, v in self.cols.items()}
        n = len(c["bytes"])
        d = np.zeros(n, dtype=abi.CHUNK_DESC)
        for k in ("bytes", "bit_depth", "channels", "flags", "ramp_start", "ramp_end", "attenuation", "out_fmt", "aux"):
            d[k] = c[k]
        silence = (c["flags"] & abi.F_SILENCE) != 0
        fresh = (c["src"] < 0) & ~silence
        # shared regions first, then one 16-byte aligned stretch per fresh chunk
        sh_len = np.array([len(s) + 16 for s in shared], dtype=np.int64)
        sh_base = np.concatenate([[0], np.cumsum((sh_len + 15) // 16 * 16)]).astype(np.int64)
        region = np.where(fresh, (c["head"] + c["bytes"] + 15) // 16 * 16 + 16, 0)
        start = sh_base[-1] + np.concatenate([[0], np.cumsum(region)[:-1]])
        src = np.where(fresh, start + c["head"], 0)
        use = (c["src"] >= 0) & ~silence
        src[use] = sh_base[c["src"][use]] + c["head"][use]
        d["src_off"] = src
        ends = np.where(fresh | use, src + c["bytes"], 0)
        in_bytes = int(ends.max()) if n else 0
        # output: the extent the sink writes, dst_phase bytes in, 16 bytes of fill between neighbours
        ob = abi.chunk_out_bytes(d).astype(np.int64)
        planar = c["out_fmt"] == abi.OUT_PLANAR32_BE
        frames = c["bytes"] // (c["bit_depth"] // 8 * c["channels"])
        extent = np.where(planar, np.where(frames > 0, (c["channels"] - 1) * c["aux"] * 4 + frames * 4, 0), ob)
        oreg = (c["dst_phase"] + extent + 15) // 16 * 16 + 16
        d["dst_off"] = 16 + np.concatenate([[0], np.cumsum(oreg)[:-1]]) + c["dst_phase"]
        out_bytes = int(16 + oreg.sum())
        return d, sh_base[:-1], in_bytes, out_bytes


class PairCycle:
    """Deals (head, destination phase) pairs per key so that every 256 consecutive chunks of a key see all 256 pairs, and
    every 16 consecutive ones all 16 heads."""

    def __init__(self):
        self.n = {}

    def next(self, key):
        p = self.n.get(key, 0)
        self.n[key] = p + 1
        p %= 256
        return p % 16, (p // 16 + p) % 16

    def count(self, key):
        return self.n.get(key, 0)


def packed_modes(B):
    """(name, flags, out_fmt, aux, attenuation, ramp) of every packed-sink mode a depth allows.  ramp None: the chunk's
    ramp is drawn from PARTIAL."""
    R, IL = abi.F_RAMP_ENABLED, abi.F_IN_LITTLE_ENDIAN
    BE, LE = abi.OUT_PACKED_BE, abi.OUT_PACKED_LE
    m = [("verbatim", 0, BE, 0, 256, None), ("ramped", R, BE, 0, 256, None),
         ("flat", R, BE, 0, 256, (9000, 9000)), ("down", R, BE, 0, 256, (16384, 0)), ("up", R, BE, 0, 256, (0, 16384))]
    if B <= 3:
        m += [("le_out_append", 0, LE, abi.LE_APPEND, 256, None)]
    if B >= 2:
        m += [("le_in", IL, BE, 0, 256, None), ("ramped_le_in", R | IL, BE, 0, 256, None)]
    if B in (2, 3):
        m += [("le_both", IL, LE, abi.LE_APPEND, 256, None), ("le_out_letter", R, LE, 0, 256, None),
              ("le_in_out_letter", R | IL, LE, 0, 256, None), ("le_in_out_append", R | IL, LE, abi.LE_APPEND, 256, None)]
    if B == 2:
        for a in (0, 1, 255, 257, 65535):
            m += [("att%d" % a, 0, BE, 0, a, None), ("att%d_ramped" % a, R, BE, 0, a, None),
                  ("att%d_le" % a, IL, LE, abi.LE_APPEND, a, None)]
    return m


RAMPS = ((16384, 0), (0, 16384), (12345, 6789), (1, 16384), (16383, 0), (700, 15000), (16384, 16383), (5000, 5000))
PARTIAL = tuple(r for r in RAMPS if r[0] != r[1] and sorted(r) != [0, 16384])   # neither flat nor full


def matrix_packed(chunks_per_mode=16):
    """A. Packed sinks: every depth x 1-32 channels x every mode, heads and destination phases dealt so that every
    (head, destination phase) pair occurs for every (depth, channel class, transform or verbatim), lengths cycled through
    frame_counts()."""
    s = Specs()
    pairs = PairCycle()
    reps = {}
    for B in DEPTHS:
        for ch in CHANNELS:
            fc = frame_counts(B, ch)
            for mi, (name, flags, fmt, aux, att, ramp) in enumerate(packed_modes(B)):
                transform = name != "verbatim" and name != "le_both" and not (name == "le_out_append" and B == 1)
                key = (B, int(chm_of(ch)), transform)
                reps.setdefault(key, (ch, flags, fmt, aux, att, ramp))
                for k in range(chunks_per_mode):
                    head, dph = pairs.next(key)
                    r = ramp or PARTIAL[(k + mi) % len(PARTIAL)]
                    s.add(B, ch, fc[(k + 3 * mi + ch) % len(fc)], flags, fmt, aux, r, att, head, dph)
    # top up the classes with few channel counts (mono, stereo) to all 256 pairs
    for key, (ch, flags, fmt, aux, att, ramp) in sorted(reps.items()):
        B = key[0]
        fc = frame_counts(B, ch)
        k = 0
        while pairs.count(key) < 256:
            head, dph = pairs.next(key)
            s.add(B, ch, fc[k % len(fc)], flags, fmt, aux, ramp or PARTIAL[k % len(PARTIAL)], att, head, dph)
            k += 1
    # every length through the group-wide instantiations (image on a 16-byte boundary: head 0)
    for B in DEPTHS:
        for ch in (2, 4, 12, 32):
            for i, f in enumerate(frame_counts(B, ch)):
                s.add(B, ch, f, abi.F_RAMP_ENABLED, ramp=RAMPS[i % len(RAMPS)], head=0, dst_phase=(7 * i) % 16)
    return s


def matrix_sinks():
    """B. The converting sinks at 1-32 channels: planar 32-bit with aux = frames, frames + 1, frames + 3 and the destination
    at phases 0-3; 32-bit to packed 8/16/24/32-bit at every head; Songcast from channel 0, 1 and ch - 2 at every depth and
    head.  Silence and little-endian input wherever the sink takes them."""
    R, IL, S = abi.F_RAMP_ENABLED, abi.F_IN_LITTLE_ENDIAN, abi.F_SILENCE
    flag_cycle = (0, R, R | IL, IL, S, R)
    s = Specs()
    for B in DEPTHS:
        for ch in CHANNELS:
            fc = frame_counts(B, ch)
            for k in range(24):
                f = fc[k % len(fc)]
                fl = flag_cycle[k % len(flag_cycle)]
                s.add(B, ch, f, fl, abi.OUT_PLANAR32_BE, f + (0, 1, 3)[k % 3], RAMPS[k % len(RAMPS)], head=(5 * k + ch) % 16,
                      dst_phase=k % 4 if k < 12 else (k * 7) % 16)
            first = sorted({0, 1, ch - 2} & set(range(0, max(ch - 1, 1))))
            for a in first:
                for head in range(16):
                    k = head + 16 * a
                    s.add(B, ch, fc[(k + B) % len(fc)], (0, R, R | IL, IL)[k % 4], abi.OUT_SONGCAST, a,
                          RAMPS[k % len(RAMPS)], head=head, dst_phase=(3 * head + a) % 16)
    fc_cycle = (0, R, R | IL, IL)
    for ch in CHANNELS:
        fc = frame_counts(4, ch)
        for ob in (8, 16, 24, 32):
            for head in range(16):
                k = head + ob
                s.add(4, ch, fc[k % len(fc)], fc_cycle[k % 4], abi.OUT_FROM32_BE, ob, RAMPS[k % len(RAMPS)], head=head,
                      dst_phase=(5 * head + ob // 8) % 16)
    return s


def matrix_silence():
    """C. Silence at 1-32 channels x every depth into the packed sink (ending one frame before, at and after each block
    write_silence cuts it into: 9216 - 9216 % frame bytes) and into the planar and Songcast sinks (<= 9216 bytes)."""
    S = abi.F_SILENCE
    s = Specs()
    for B in DEPTHS:
        for ch in CHANNELS:
            fb = B * ch
            block = MAX - MAX % fb
            sizes = sorted({k * block + e for k in (1, 2, 3) for e in (-fb, 0, fb)} | {fb, 2 * fb, 3 * fb, 5 * fb, 17 * fb})
            for i, n in enumerate(sizes):
                s.add(B, ch, 0, S, bytes_=n, dst_phase=(i * 5 + ch) % 16)
            for i, n in enumerate(x for x in (fb, 2 * fb, 5 * fb, block - fb, block) if 0 < x <= MAX):
                f = n // fb
                s.add(B, ch, f, S, abi.OUT_PLANAR32_BE, f + i % 3, dst_phase=i % 4)
                s.add(B, ch, f, S, abi.OUT_SONGCAST, (0, 1, ch - 2)[i % 3] if ch > 2 else 0, dst_phase=(i * 3) % 16)
    return s


def matrix_pow2():
    """D3. Ramps over 2^k - 1, 2^k and 2^k + 1 frames at every depth and channel class."""
    s = Specs()
    for B in DEPTHS:
        for ch in (1, 2, 3, 4, 9, 12, 31, 32):
            for k in range(1, 14):
                for i, f in enumerate((2 ** k - 1, 2 ** k, 2 ** k + 1)):
                    if f * B * ch > MAX:
                        continue
                    r = RAMPS[(k + i) % 5]
                    s.add(B, ch, f, abi.F_RAMP_ENABLED | (abi.F_IN_LITTLE_ENDIAN if k % 2 else 0), ramp=r,
                          head=(k + 3 * i) % 16, dst_phase=(k * 5 + i) % 16)
    return s


RAMP_PAIRS_16 = ((16384, 0), (0, 16384), (16383, 0), (1, 16384), (12345, 6789))


def ramp_lengths(B, lengths, ramp, samples):
    """D1/D2. Mono chunks of every length in `lengths` with a constant sample (one chunk per length and sample value),
    all reading one shared source region per value.  -> (Specs, shared regions)."""
    s = Specs()
    top = max(lengths)
    shared = []
    for v in samples:
        run = np.frombuffer(int(v).to_bytes(B, "big") * top, dtype=np.uint8)
        shared += [np.concatenate([np.zeros(h, np.uint8), run]) for h in range(16)]   # region 16 j + h: the run at head h
    for j in range(len(samples)):
        for i, n in enumerate(lengths):
            h = (i + j) % 16
            s.add(B, 1, n, abi.F_RAMP_ENABLED, ramp=ramp, head=h, dst_phase=(3 * i) % 16, src=16 * j + h)
    return s, shared


class Batch:
    """One batch of descriptors with its input (the arena, then a poisoned tail the kernel must not read)."""

    def __init__(self, name, specs, port, seed, shared=()):
        self.name = name
        self.descs, sh_off, in_bytes, self.out_bytes = specs.lay_out(shared)
        self.in_bytes = max(in_bytes, 16)   # (a batch of silence reads nothing, but an arena is never empty)
        inp = np.full(self.in_bytes + 64, POISON, dtype=np.uint8)
        inp[:self.in_bytes] = port.fill_pcm(self.in_bytes, seed)
        for off, v in zip(sh_off, shared):
            inp[int(off):int(off) + len(v)] = v
        self.inp = inp
        self.cls = classify(self.descs)


def batches(port):
    """Every batch of the matrix (A, B, C, D) in a deterministic order."""
    out = [Batch("A_packed", matrix_packed(), port, 1), Batch("B_sinks", matrix_sinks(), port, 2),
           Batch("C_silence", matrix_silence(), port, 3), Batch("D3_pow2", matrix_pow2(), port, 4)]
    for i, r in enumerate(RAMP_PAIRS_16):
        s, sh = ramp_lengths(2, range(1, 4609), r, (0x7FFF, 0x8000))
        out.append(Batch("D1_16bit_%d_%d" % r, s, port, 10 + i, sh))
    for i, r in enumerate(((16384, 0), (0, 16384))):
        s, sh = ramp_lengths(1, range(4609, 9217), r, (0x7F, 0x80))
        out.append(Batch("D2_8bit_%d_%d" % r, s, port, 20 + i, sh))
    return out


def _intervals(descs):
    """(start, length, chunk) of every byte range the chunks write (planar output: one range per channel plane)."""
    d = np.asarray(descs)
    ob = abi.chunk_out_bytes(d).astype(np.int64)
    lo = d["dst_off"].astype(np.int64)
    planar = d["out_fmt"] == abi.OUT_PLANAR32_BE
    idx = np.arange(len(d))
    pch = d["channels"][planar].astype(np.int64)
    pi = np.repeat(idx[planar], pch)
    pc = np.concatenate([np.arange(c) for c in pch]) if len(pch) else np.zeros(0, np.int64)
    frames = d["bytes"].astype(np.int64) // (d["bit_depth"].astype(np.int64) // 8 * d["channels"].astype(np.int64))
    starts = np.concatenate([lo[~planar], lo[pi] + pc * d["aux"][pi].astype(np.int64) * 4])
    lens = np.concatenate([ob[~planar], frames[pi] * 4])
    who = np.concatenate([idx[~planar], pi])
    keep = lens > 0
    return starts[keep], lens[keep], who[keep]


def covered(descs, out_bytes):
    """Mask of the output bytes some chunk writes (vectorised; the chunks of a batch never overlap)."""
    starts, lens, _ = _intervals(descs)
    edge = np.zeros(int(out_bytes) + 1, dtype=np.int8)
    np.add.at(edge, starts, 1)
    np.add.at(edge, starts + lens, -1)
    depth = np.cumsum(edge[:-1], dtype=np.int8)
    assert depth.max(initial=0) <= 1, "chunks overlap"
    return depth.astype(bool)


def owner(descs, i):
    """Index of the chunk that writes output byte i, or -1."""
    starts, lens, who = _intervals(descs)
    hit = np.nonzero((starts <= i) & (i < starts + lens))[0]
    return int(who[hit[0]]) if len(hit) else -1


# ------------------------------------------------------------------------------------------------------------------
# streams at 9-32 channels for the whole stage

def widen(w, seed, name):
    """The streams of workload `w` at 9-32 channels (dealt in turn), every other field as `w` made it: message sizes cut
    to what 9216 bytes hold at the new frame size (or set to it), codec reads of whole 9216-byte blocks (AIFF-style) on
    every fifth stream, the arenas laid out again."""
    rng = np.random.default_rng(seed)
    st = w.streams.copy()
    slack = []
    for i in range(len(st)):
        ch = 9 + (i + seed) % 24
        bits, rate = int(st[i]["bit_depth"]), int(st[i]["sample_rate"])
        fb = ch * bits // 8
        cmax = W.max_chunk_frames(rate, bits, ch)
        st[i]["channels"] = ch
        st[i]["chunk_frames"] = min(int(st[i]["chunk_frames"]), cmax) if rng.random() < 0.5 else cmax
        if int(st[i]["codec_read_frames"]) or i % 5 == 0:
            st[i]["chunk_frames"] = cmax
            st[i]["codec_read_frames"] = MAX // fb
        lo, hi = int(st[i]["first_event"]), int(st[i]["first_event"]) + int(st[i]["num_events"])
        ev = w.events[lo:hi]
        sil = ev["arg"][ev["op"] == abi.EV_INSERT_SILENCE].astype(np.int64)
        slack.append(int((sil // abi.jiffies_per_sample(rate)).sum()) * fb)
    in_bytes, out_bytes = W.layout(st, slack_bytes=slack)
    return W.Workload(name, st, w.events.copy(), in_bytes, out_bytes, w.seed)


def wide_streams():
    """Streams at 9-32 channels: the mixed generator's (every depth, eight rates, LE/BE input, P1/P2 sinks, ramps on three
    stages, mutes, MsgSilence, attenuation windows, driver blocks, message caps) and the element generator's (Ramper,
    StarvationRamper, Muter, MsgHalt: ops 8-12), re-channelled."""
    out = [widen(W.mixed(n_streams=72, seed=s, max_frames=4000), s, "wide_mixed_%d" % s) for s in (31, 32, 33)]
    out += [widen(W.elements(s, n_streams=48, attenuation=(s % 2 == 1)), s, "wide_elements_%d" % s) for s in (1, 2, 3)]
    out.append(widen(W.config4(n_streams=96, seconds=0.1, seed=8), 8, "wide_config4"))
    return out
