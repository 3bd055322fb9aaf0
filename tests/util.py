"""Shared helpers for the parity tests."""
import numpy as np

from ohpipeline_b200 import abi


def force_fmt(w, fmt):
    w.streams["out_fmt"] = fmt
    return w


def describe_first_diff(got, want, chunks):
    i = int(np.nonzero(got != want)[0][0])
    k = int(np.searchsorted(chunks["dst_off"], i, side="right") - 1)
    return "first difference at output byte %d (got %#x want %#x) in chunk %d: %s" % (
        i, got[i], want[i], k, chunks[k])


def make_desc(**kw):
    d = np.zeros(1, dtype=abi.CHUNK_DESC)
    d["attenuation"] = abi.UNITY_ATTENUATION
    d["ramp_start"] = abi.RAMP_MAX
    d["ramp_end"] = abi.RAMP_MAX
    for k, v in kw.items():
        d[k] = v
    return d


def pack_chunks(chunk_specs, align=1, rng=None):
    """chunk_specs: list of dicts (bytes, bit_depth, channels, flags, ramp_start, ramp_end, attenuation, out_fmt, aux,
    optional src_pad/dst_pad = bytes of padding placed before the chunk).  Lays chunks out back to back and returns
    (descs, in_bytes, out_bytes)."""
    descs = np.zeros(len(chunk_specs), dtype=abi.CHUNK_DESC)
    src = dst = 0
    for i, c in enumerate(chunk_specs):
        c = dict(c)
        src += c.pop("src_pad", 0)
        dst += c.pop("dst_pad", 0)
        d = make_desc(**c)
        d["src_off"] = src
        d["dst_off"] = dst
        descs[i] = d[0]
        if not (int(d["flags"][0]) & abi.F_SILENCE):
            src += int(d["bytes"][0])
        if int(d["out_fmt"][0]) == abi.OUT_PLANAR32_BE:
            dst += int(d["channels"][0]) * int(d["aux"][0]) * 4
        else:
            dst += int(abi.chunk_out_bytes(d)[0])
        if align > 1:
            src = (src + align - 1) // align * align
            dst = (dst + align - 1) // align * align
    return descs, src + 64, dst + 64


def alignment_specs(bits, le):
    """64 chunks of `bits`-bit audio, 1-8 channels, 1-39 frames, ramped or not, at every src/dst byte offset mod 16
    (pack_chunks specs: a split playable starts wherever the ramp ended)."""
    b = bits // 8
    specs = []
    rng = np.random.default_rng(bits + le)
    for k in range(64):
        ch = int(rng.integers(1, 9))
        frames = int(rng.integers(1, 40))
        specs.append(dict(bytes=frames * ch * b, bit_depth=bits, channels=ch,
                          flags=(abi.F_RAMP_ENABLED if k % 3 else 0) | (abi.F_IN_LITTLE_ENDIAN if le else 0),
                          ramp_start=int(rng.integers(0, 16385)), ramp_end=int(rng.integers(0, 16385)),
                          src_pad=int(rng.integers(0, 5)), dst_pad=int(rng.integers(0, 5))))
    return specs


def covered_mask(descs, out_bytes):
    """Boolean mask of the output bytes some chunk writes (planar output is strided per channel)."""
    mask = np.zeros(out_bytes, dtype=bool)
    ob = abi.chunk_out_bytes(descs)
    for d, n in zip(descs, ob):
        lo = int(d["dst_off"])
        if int(d["out_fmt"]) == abi.OUT_PLANAR32_BE:
            frames = int(d["bytes"]) // (int(d["channels"]) * int(d["bit_depth"]) // 8)
            for c in range(int(d["channels"])):
                a = lo + c * int(d["aux"]) * 4
                mask[a:a + frames * 4] = True
        else:
            mask[lo:lo + int(n)] = True
    return mask
