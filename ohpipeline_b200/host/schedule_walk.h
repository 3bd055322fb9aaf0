// schedule_walk.h -- one stream's walk through the ramp-setting stages on plain data, compiled for BOTH the device
// (csrc/ohp_schedule_kernels.cuh: one thread per stream) and the host (schedule.cpp: ohp_schedule_walk_host, the
// CPU-testable twin the "-m 'not gpu'" suite compares with the class-based host model).
//
// It restates stage_chain.h + msg_model.cpp without classes, allocation, recursion or exceptions.  The ramp algebra
// (Ramp::Set / Ramp::Split, Msg.cpp:590-807) is ramp_core.h, the source the host mirror compiles too; the
// message-level steps follow
//     MsgAudio::Split             Msg.cpp:1949-1969     msg_split
//     MsgSilence::SplitCompleted  Msg.cpp:2522-2545     msg_split (silence branch)
//     MsgAudio::SetRamp           Msg.cpp:1989-2046     msg_set_ramp
//     MsgAudioPcm::CreatePlayable Msg.cpp:2234-2262     create_playable
//     MsgSilence::CreatePlayable  Msg.cpp:2472-2492     create_playable (silence branch)
//     MsgPlayable::Split          Msg.cpp:2591-2624     playable_split
// and the stage idiom of Ramper.cpp:114-134, Muter.cpp:210-262, StarvationRamper.cpp:579-603, 791-832.
#pragma once

#include <cstdint>

#include "../../include/ohp_schedule.h"
#include "../../include/ohp_starvation_recent.h"
#include "ramp_core.h"
#include "codec_source.h"

namespace ohp {
namespace sched {

constexpr int kStages = (int)OHP_MAX_STAGES;
constexpr int kStackDepth = 16; // pending split remainders per stage (each Process pushes at most four)

// per-stream result codes
constexpr uint32_t kOk = 0u;
constexpr uint32_t kErrAssert = 1u;   // the reference would ASSERT                 -> OHP_E_INVALID_DESC
constexpr uint32_t kErrSpec = 2u;     // a spec the message model cannot represent  -> OHP_E_INVALID_ARG
constexpr uint32_t kErrDepth = 3u;    // more pending splits than kStackDepth       -> OHP_E_NO_MEMORY

struct Msg
{
    uint64_t cell;     // arena offset of the audio this message (and every split of it) refers to
    uint32_t size;     // jiffies (MsgAudio::iSize)
    uint32_t offset;   // jiffies into the cell (MsgAudio::iOffset)
    uint32_t total;    // MsgSilence::iSizeJiffiesTotal
    uint32_t atten;    // MsgAudioPcm::iAttenuation
    core::RampPod ramp;
    uint32_t silence;  // 1: MsgSilence
};

// 32-byte stack entry
struct Packed
{
    uint64_t cell;
    uint32_t size, offset, total;
    uint32_t ramp_se;  // start | end << 16
    uint32_t misc;     // atten | direction << 16 | enabled << 24 | silence << 25
    uint32_t pad;
};

OHP_HD Packed pack(const Msg& m)
{
    Packed p;
    p.cell = m.cell; p.size = m.size; p.offset = m.offset; p.total = m.total;
    p.ramp_se = m.ramp.start | (m.ramp.end << 16);
    p.misc = (m.atten & 0xffffu) | (m.ramp.direction << 16) | (m.ramp.enabled << 24) | (m.silence << 25);
    p.pad = 0;
    return p;
}
OHP_HD Msg unpack(const Packed& p)
{
    Msg m;
    m.cell = p.cell; m.size = p.size; m.offset = p.offset; m.total = p.total;
    m.ramp.start = p.ramp_se & 0xffffu; m.ramp.end = p.ramp_se >> 16;
    m.atten = p.misc & 0xffffu; m.ramp.direction = (p.misc >> 16) & 0xffu; m.ramp.enabled = (p.misc >> 24) & 1u;
    m.silence = (p.misc >> 25) & 1u;
    return m;
}

struct Playable
{
    uint64_t arena;
    uint32_t size;     // bytes
    uint32_t jiffies;
    uint32_t atten;
    core::RampPod ramp;
    uint32_t silence;
};

enum Mode : uint32_t { Running = 0, RampingDown = 1, RampingUp = 2, Muted = 3 };
// which of the reference's elements a stage is (stage_chain.h: decided by the ops of its events)
enum Element : uint32_t { Generic = 0, ElemRamper = 1, ElemMuter = 2, ElemStarvation = 3, ElemBad = 4 };

constexpr uint64_t kNever = ~0ull;

// One stage's state.  Indexed with compile-time constants only (the stage loop is unrolled), so on the device it lives
// in registers; the stacks of pending split remainders are the only thing in local memory, and only splits touch them.
struct Stage
{
    uint64_t pos;
    uint64_t nextAt;   // at_jiffies of this stage's next event (index nextEv), kNever when there is none left
    uint32_t mode, current, remaining, maxMsg, attenuation, nextEv, depth;
    uint32_t elem;     // Element
    uint32_t halted;   // Muter::iHalted / StarvationRamper Halted-or-Starting: no PCM has passed since the start or the last halt
};

// What stage_chain.h keeps per stage for a StarvationRamper's records (RECORD walks only; see note_starvation).
struct Starve
{
    uint64_t pcmJiffies; // PCM that has passed the stage
    uint64_t pcmRun;     // ... its latest unbroken run: nothing but PCM of one attenuation (pcmRunAtt) since the stream began,
    uint32_t pcmRunAtt;  // a MsgSilence passed or a flywheel ramp used the recent audio up
    uint32_t elemRamp;   // what the element's own SetRamp calls last returned (StarvationRamper::iCurrentRampValue)
};

// RECENT walks: the recent audio a StarvationRamper keeps (stage_chain.h NoteRecent / TrimRecent) in a ring of
// kRecentPieces per stage.  A piece is 16 bytes: where its PCM begins (kSilencePiece: a MsgSilence), jiffies, attenuation.
constexpr uint32_t kRecentPieces = OHP_DEVICE_RECENT_PIECES;
static_assert((kRecentPieces & (kRecentPieces - 1)) == 0, "the ring wraps with a mask");
constexpr uint64_t kSilencePiece = ~0ull;

struct RecentPiece
{
    uint64_t pcm;
    uint32_t jiffies;
    uint32_t attenuation;
};

struct RecentRing
{
    RecentPiece p[kRecentPieces];
    uint64_t total;      // jiffies of the pieces held
    uint32_t head, count;
    uint32_t dropped;    // a push found the ring full since it was last emptied
};

// What a walk keeps for the recent audio: nothing, or the rings and where the records' pieces go (record of the stream's
// k-th event: count[k], pieces out[k * kRecentPieces ...]).
template <bool RECENT> struct RecentCtx {};
template <> struct RecentCtx<true>
{
    ohp_recent_audio* out;
    uint32_t* count;
    uint32_t stride;     // team size: lane i writes pieces i, i + stride, ...
    RecentRing ring[kStages];
};

OHP_HD void recent_clear(RecentRing& r)
{
    r.total = 0; r.head = 0; r.count = 0; r.dropped = 0;
}

// TrimRecent: pieces the last millisecond no longer needs go; a lone run of PCM keeps its last 2 ms
OHP_HD void recent_trim(RecentRing& r)
{
    while (r.count > 1 && r.total - r.p[r.head].jiffies >= OHP_FLYWHEEL_TRAINING_JIFFIES) {
        r.total -= r.p[r.head].jiffies;
        r.head = (r.head + 1) & (kRecentPieces - 1);
        r.count--;
    }
    RecentPiece& front = r.p[r.head];
    if (r.count == 1 && front.pcm != kSilencePiece && front.jiffies > 4u * OHP_FLYWHEEL_TRAINING_JIFFIES) {
        const uint32_t drop = front.jiffies - 2u * OHP_FLYWHEEL_TRAINING_JIFFIES;
        front.pcm += drop;
        front.jiffies -= drop;
        r.total -= drop;
    }
}

// NoteRecent: a piece joins the last one where it continues it, else the ring.  A push into a full ring drops the oldest
// piece.  That loses something only where the class model would keep it -- where the pieces behind it add up to less
// than 1 ms -- and then the ring holds less than 1 ms until it is emptied: see note_starvation.
OHP_HD void recent_note(RecentRing& r, uint64_t aPcm, uint32_t aJiffies, uint32_t aAttenuation)
{
    if (aJiffies == 0) return;
    if (aPcm != kSilencePiece && r.count != 0) {
        RecentPiece& last = r.p[(r.head + r.count - 1) & (kRecentPieces - 1)];
        if (last.pcm != kSilencePiece && last.attenuation == aAttenuation && last.pcm + last.jiffies == aPcm
            && (uint64_t)last.jiffies + aJiffies <= 0x7fffffffu) {
            last.jiffies += aJiffies;
            r.total += aJiffies;
            recent_trim(r);
            return;
        }
    }
    if (r.count == kRecentPieces) {
        r.total -= r.p[r.head].jiffies;
        r.head = (r.head + 1) & (kRecentPieces - 1);
        r.count--;
        r.dropped = 1;
    }
    RecentPiece& p = r.p[(r.head + r.count) & (kRecentPieces - 1)];
    p.pcm = aPcm; p.jiffies = aJiffies; p.attenuation = aAttenuation;
    r.count++;
    r.total += aJiffies;
    recent_trim(r);
}

struct StreamCtx
{
    const ohp_ramp_event* ev;
    uint32_t nEv;
    uint32_t jps, frameBytes, channels, bits;
    uint32_t in_le, out_fmt;
    uint32_t blockBytes, blockFill;
    uint64_t dst_base;
    uint32_t lane;         // this thread's index in the team walking the stream (host: 0); lane 0 writes in the general path
    // sink
    uint64_t nChunks, outBytes;
    ohp_chunk_desc* descs; // EMIT: this stream's first descriptor
    ohp_chunk_info* info;  // EMIT, may be null
    uint64_t limit;        // EMIT: descriptors this stream may write (its region when regions come from stream_chunk_bound)
    // RECORD: one ohp_starvation per OHP_EV_STARVATION applied -- at rec[event] (event: index in this stream's slice), or
    // appended at rec[nRec++] where recAppend is set (the host twin keeps them in the order ohp_schedule_build does)
    ohp_starvation* rec;
    uint32_t recAppend, nRec;
    uint64_t stream, firstEvent;
    Starve sv[kStages];
};

// MsgAudio::Split (+ SplitCompleted): m keeps the first aJiffies, rest gets what follows.
OHP_HD uint32_t msg_split(Msg& m, uint32_t aJiffies, Msg& rest, uint32_t jps)
{
    if (!(aJiffies > 0)) return kErrAssert;
    if (!(aJiffies < m.size)) return kErrAssert;
    rest.cell = m.cell;
    rest.atten = m.atten;
    rest.silence = m.silence;
    rest.total = 0;
    rest.offset = m.offset + aJiffies;
    rest.size = m.size - aJiffies;
    if (m.ramp.enabled) {
        if (core::ramp_split(m.ramp, aJiffies, m.size, rest.ramp) != 0) return kErrAssert;
    }
    else {
        core::ramp_reset(rest.ramp);
    }
    m.size = aJiffies;
    if (m.silence) {
        // silence only exists in whole samples: the first part gives its sub-sample remainder to the second
        const uint32_t spare = m.size % jps;
        m.size -= spare;
        m.total = m.size;
        rest.size += spare;
        rest.total = rest.size - rest.size % jps;
    }
    return kOk;
}

// MsgAudio::SetRamp.  Returns the new "current" ramp value in aCurrent; aHaveSplit says whether aSplit was produced.
OHP_HD uint32_t msg_set_ramp(Msg& m, uint32_t aStart, uint32_t& aRemaining, uint32_t aDirection,
                                                 Msg& aSplit, bool& aHaveSplit, uint32_t& aCurrent, uint32_t jps)
{
    const uint32_t duration = aRemaining;
    aHaveSplit = false;
    if (m.ramp.enabled && m.ramp.direction == core::kDirMute) {
        if (aDirection == core::kDirDown) aRemaining = 0;
        aCurrent = m.ramp.end;
        return kOk;
    }
    core::RampPod second;
    uint32_t splitPos;
    const int rc = core::ramp_set(m.ramp, aStart, m.size, duration, aDirection, second, splitPos);
    if (rc == core::kRampAssert) return kErrAssert;
    if (rc == 1) {
        if (splitPos == 0) {
            m.ramp = second;
        }
        else if (splitPos != m.size) {
            const core::RampPod first = m.ramp; // Split() rescales the ramp; the values Set() chose are the ones to keep
            const uint32_t e = msg_split(m, splitPos, aSplit, jps);
            if (e != kOk) return e;
            m.ramp = first;
            aSplit.ramp = second;
            aHaveSplit = true;
        }
    }
    aRemaining -= m.size;
    if (aHaveSplit && aSplit.ramp.direction != aDirection && aDirection == core::kDirUp) {
        aRemaining += aSplit.size; // the split part runs against the requested ramp (Msg.cpp:2031-2034)
    }
    if ((aDirection == core::kDirDown && m.ramp.end == core::kRampMin) || (aDirection == core::kDirUp && m.ramp.end == core::kRampMax)) {
        aRemaining = 0; // finished early (Msg.cpp:2037-2043)
    }
    aCurrent = m.ramp.end;
    return kOk;
}

OHP_HD Playable create_playable(const Msg& m, const StreamCtx& cx)
{
    Playable p;
    p.jiffies = m.size;
    if (!m.silence) {
        // offset and size are each rounded DOWN to a sample boundary, the size first being extended by whatever the
        // offset lost, so no audio is dropped between adjacent splits
        uint32_t offsetJiffies = m.offset;
        const uint32_t offsetBytes = core::jiffies_to_bytes(offsetJiffies, cx.jps, cx.channels, cx.bits);
        uint32_t sizeJiffies = m.size + (m.offset - offsetJiffies);
        p.size = core::jiffies_to_bytes(sizeJiffies, cx.jps, cx.channels, cx.bits);
        if (m.ramp.direction != core::kDirMute) {
            p.silence = 0;
            p.arena = m.cell + offsetBytes;
            p.ramp = m.ramp;
            p.atten = m.atten;
        }
        else {
            // muted audio is replaced by silence and its ramp dropped (Msg.cpp:2252-2257)
            p.silence = 1;
            p.arena = 0;
            core::ramp_reset(p.ramp);
            p.atten = OHP_UNITY_ATTENUATION;
        }
    }
    else {
        uint32_t total = m.total;
        p.size = core::jiffies_to_bytes(total, cx.jps, cx.channels, cx.bits);
        p.silence = 1;
        p.arena = 0;
        p.ramp = m.ramp; // travels with the playable but is never applied to silence
        p.atten = OHP_UNITY_ATTENUATION;
    }
    return p;
}

// MsgPlayable::Split: p keeps the first aBytes (< p.size), rest gets what follows.
OHP_HD uint32_t playable_split(Playable& p, uint32_t aBytes, Playable& rest, const StreamCtx& cx)
{
    if (!(aBytes <= p.size) || aBytes == 0) return kErrAssert;
    const uint32_t frames = aBytes / cx.frameBytes;
    const uint32_t splitJiffies = frames * cx.jps;
    rest.silence = p.silence;
    rest.arena = p.silence ? 0 : p.arena + aBytes;
    rest.size = p.size - aBytes;
    rest.jiffies = p.jiffies - splitJiffies;
    rest.atten = OHP_UNITY_ATTENUATION; // reference quirk: SplitCompleted does not pass iAttenuation on (Msg.cpp:2803-2807)
    if (p.ramp.enabled) {
        if (core::ramp_split(p.ramp, aBytes, p.size, rest.ramp) != 0) return kErrAssert;
    }
    else {
        core::ramp_reset(rest.ramp);
    }
    p.size = aBytes;
    p.jiffies = splitJiffies;
    return kOk;
}

// One 32-byte descriptor (layout: include/ohp_b200.h) for playable p as this stream's aIndex-th chunk, writing at
// aOutOffset of the stream's output; two 128-bit stores on the device.
OHP_HD void emit_desc(const StreamCtx& cx, const Playable& p, uint64_t aIndex, uint64_t aOutOffset)
{
    const uint32_t flags = (p.ramp.enabled ? OHP_F_RAMP_ENABLED : 0u) | (p.silence ? OHP_F_SILENCE : 0u)
                         | ((!p.silence && cx.in_le) ? OHP_F_IN_LITTLE_ENDIAN : 0u);
    const uint64_t src = p.silence ? 0 : p.arena;
    const uint64_t dst = cx.dst_base + aOutOffset;
    const uint32_t w4 = p.size;
    const uint32_t w5 = (p.ramp.start & 0xffffu) | (p.ramp.end << 16);
    const uint32_t w6 = (p.atten & 0xffffu) | (cx.bits << 16) | (cx.channels << 24);
    const uint32_t w7 = flags | (cx.out_fmt << 8) | (cx.out_fmt == OHP_OUT_PACKED_LE ? OHP_LE_APPEND << 16 : 0u); // aux: as MsgPlayable::Descriptor
    if (aIndex >= cx.limit) return; // never outside the stream's region; the caller compares the count with the limit afterwards
#if defined(__CUDA_ARCH__)
    uint4* out = reinterpret_cast<uint4*>(cx.descs + aIndex);
    out[0] = make_uint4((uint32_t)src, (uint32_t)(src >> 32), (uint32_t)dst, (uint32_t)(dst >> 32));
    out[1] = make_uint4(w4, w5, w6, w7);
    if (cx.info) {
        *reinterpret_cast<uint2*>(cx.info + aIndex) = make_uint2(p.ramp.direction, p.jiffies);
    }
#else
    uint32_t* out = reinterpret_cast<uint32_t*>(cx.descs + aIndex);
    out[0] = (uint32_t)src; out[1] = (uint32_t)(src >> 32); out[2] = (uint32_t)dst; out[3] = (uint32_t)(dst >> 32);
    out[4] = w4; out[5] = w5; out[6] = w6; out[7] = w7;
    if (cx.info) {
        cx.info[aIndex].direction = p.ramp.direction;
        cx.info[aIndex].jiffies = p.jiffies;
    }
#endif
}

template <bool EMIT>
OHP_HD void on_playable(StreamCtx& cx, const Playable& p)
{
    if (EMIT && cx.lane == 0) emit_desc(cx, p, cx.nChunks, cx.outBytes);
    cx.nChunks++;
    cx.outBytes += p.size;
}

// PreDriver -> CreatePlayable, then a driver that pulls fixed blocks (stage_chain.h Drive()).
template <bool EMIT>
OHP_HD uint32_t drive(StreamCtx& cx, const Msg& m)
{
    Playable p = create_playable(m, cx);
    const uint32_t block = cx.blockBytes;
    if (block == 0 || p.size == 0) {
        on_playable<EMIT>(cx, p);
        return kOk;
    }
    for (;;) {
        const uint32_t room = block - cx.blockFill;
        if (p.size > room) {
            Playable rest;
            const uint32_t e = playable_split(p, room, rest, cx);
            if (e != kOk) return e;
            on_playable<EMIT>(cx, p);
            cx.blockFill = 0;
            p = rest;
        }
        else {
            on_playable<EMIT>(cx, p);
            cx.blockFill += p.size;
            if (cx.blockFill == block) cx.blockFill = 0;
            return kOk;
        }
    }
}

// Point s.nextEv / s.nextAt at this stage's first event at or after index aFrom (MsgSilence insertions are fed by Run()).
OHP_HD void stage_seek(const StreamCtx& cx, Stage& s, uint32_t stage, uint32_t aFrom)
{
    uint32_t i = aFrom;
    for (; i < cx.nEv; i++) {
        const ohp_ramp_event& e = cx.ev[i];
        if (e.stage == stage && e.op != OHP_EV_INSERT_SILENCE) break;
    }
    s.nextEv = i;
    s.nextAt = i < cx.nEv ? cx.ev[i].at_jiffies : kNever;
}

// stage_chain.h StageElement()
OHP_HD uint32_t stage_element(const StreamCtx& cx, uint32_t stage)
{
    uint32_t elem = Generic;
    bool bare = false;
    for (uint32_t i = 0; i < cx.nEv; i++) {
        const ohp_ramp_event& e = cx.ev[i];
        if (e.stage != stage) continue;
        uint32_t of = Generic;
        switch (e.op) {
        case OHP_EV_RAMPER_STREAM: of = ElemRamper; break;
        case OHP_EV_MUTER_MUTE: case OHP_EV_MUTER_UNMUTE: of = ElemMuter; break;
        case OHP_EV_STARVATION: of = ElemStarvation; break;
        case OHP_EV_RAMP_DOWN: case OHP_EV_RAMP_UP: case OHP_EV_MUTE: case OHP_EV_UNMUTE: bare = true; break;
        default: break;
        }
        if (of != Generic) {
            if (elem != Generic && elem != of) return ElemBad;
            elem = of;
        }
    }
    if (elem != Generic && bare) return ElemBad;
    return elem;
}

// stage_chain.h ApplyElementEvent(): false where the reference ASSERTS
OHP_HD bool apply_element_event(Stage& s, uint32_t op, uint32_t arg)
{
    switch (op) {
    case OHP_EV_RAMPER_STREAM: // Ramper.cpp:72-93
        if (arg != 0) { s.mode = RampingUp; s.current = core::kRampMin; s.remaining = arg; }
        else { s.mode = Running; s.current = core::kRampMax; s.remaining = 0; }
        break;
    case OHP_EV_MUTER_MUTE: // Muter.cpp:57-99
        if (s.mode == Running) {
            if (s.halted) { s.mode = Muted; }
            else { s.mode = RampingDown; s.remaining = arg; s.current = core::kRampMax; }
        }
        else if (s.mode == RampingUp) {
            if (s.remaining == arg) { s.mode = Muted; }
            else { s.mode = RampingDown; s.remaining = arg - s.remaining; }
        }
        else return false;
        break;
    case OHP_EV_MUTER_UNMUTE: // Muter.cpp:101-137
        if (s.mode == RampingDown) {
            if (s.remaining == arg) { s.mode = Running; }
            else { s.mode = RampingUp; s.remaining = arg - s.remaining; }
        }
        else if (s.mode == Muted) {
            if (s.halted) { s.mode = Running; }
            else { s.mode = RampingUp; s.remaining = arg; s.current = core::kRampMin; }
        }
        else return false;
        break;
    case OHP_EV_HALT:
        if (s.elem == ElemRamper) { // Ramper.cpp:65-70
            if (s.mode == RampingUp) s.mode = Running;
        }
        else if (s.elem == ElemMuter) { // Muter.cpp:159-167, 264-280
            if (s.mode == RampingDown) { s.mode = Muted; s.remaining = 0; s.current = core::kRampMin; }
            s.halted = 1;
        }
        else if (s.elem == ElemStarvation) { // StarvationRamper.cpp:728-736
            s.mode = Running;
            s.halted = 1;
        }
        break;
    case OHP_EV_STARVATION: // StarvationRamper.cpp:622-673
        if ((s.mode == Running && !s.halted) || (s.mode == RampingUp && s.current != core::kRampMin)) {
            s.mode = RampingUp; s.current = core::kRampMin; s.remaining = arg;
        }
        break;
    default: break;
    }
    return true;
}

// stage_chain.h ElementSeesSilence()
OHP_HD void element_sees_silence(Stage& s)
{
    if (s.elem == ElemRamper) { // Ramper.cpp:106-112
        s.mode = Running; s.current = core::kRampMax; s.remaining = 0;
    }
    else if (s.elem == ElemMuter) { // Muter.cpp:188-208
        if (s.mode == RampingDown) { s.mode = Muted; s.remaining = 0; s.current = core::kRampMin; }
        else if (s.mode == RampingUp) { s.mode = Running; s.remaining = 0; s.current = core::kRampMax; }
    }
}

OHP_HD bool apply_event(Stage& s, uint32_t op, uint32_t arg)
{
    switch (op) {
    case OHP_EV_RAMP_DOWN:
        if (s.mode == Muted || s.current == core::kRampMin) { s.mode = Muted; s.current = core::kRampMin; s.remaining = 0; }
        else { s.mode = RampingDown; s.remaining = arg; }
        break;
    case OHP_EV_RAMP_UP:
        if (s.mode == Running && s.current == core::kRampMax) { /* already at full level */ }
        else { s.mode = RampingUp; s.remaining = arg; }
        break;
    case OHP_EV_MUTE: s.mode = Muted; s.current = core::kRampMin; s.remaining = 0; break;
    case OHP_EV_UNMUTE: s.mode = Running; s.current = core::kRampMax; s.remaining = 0; break;
    case OHP_EV_SET_ATTENUATION: s.attenuation = arg; break;
    case OHP_EV_MAX_MSG_JIFFIES: s.maxMsg = arg; break;
    default: return apply_element_event(s, op, arg);
    }
    return true;
}

// stage_chain.h NoteStarvation(): called in front of every event a stage applies.  RECENT: the record's pieces too.
template <bool RECENT>
OHP_HD void note_starvation(StreamCtx& cx, RecentCtx<RECENT>& rs, const Stage& s, uint32_t stage, uint32_t aEvent)
{
    if (s.elem != ElemStarvation || cx.ev[aEvent].op != OHP_EV_STARVATION) return;
    const bool plays = (s.mode == Running && !s.halted) || (s.mode == RampingUp && s.current != core::kRampMin); // as apply_element_event
    Starve& r = cx.sv[stage];
    if (cx.lane == 0 && cx.rec) {
        ohp_starvation o;
        o.stream = cx.stream;
        o.pcm_jiffies = r.pcmJiffies;
        o.event = (uint32_t)(cx.firstEvent + aEvent);
        o.ramp = r.elemRamp;
        o.plays = plays ? 1u : 0u;
        o.recent_jiffies = r.pcmRun > 0xffffffffull ? 0xffffffffu : (uint32_t)r.pcmRun;
        o.attenuation = r.pcmRunAtt;
        o.reserved = 0;
        cx.rec[cx.recAppend ? cx.nRec++ : aEvent] = o;
    }
    if constexpr (RECENT) {
        // the class model's record holds more than kRecentPieces pieces exactly where the ring dropped one and holds less
        // than 1 ms (recent_note): such a record is incomplete, and the planner refuses it
        RecentRing& g = rs.ring[stage];
        const bool incomplete = g.dropped && g.total < OHP_FLYWHEEL_TRAINING_JIFFIES;
        if (cx.lane == 0) rs.count[aEvent] = incomplete ? OHP_RECENT_INCOMPLETE : g.count;
        for (uint32_t i = cx.lane; !incomplete && i < g.count; i += rs.stride) {
            const RecentPiece& q = g.p[(g.head + i) & (kRecentPieces - 1)];
            ohp_recent_audio a;
            a.pcm_jiffies = q.pcm == kSilencePiece ? 0 : q.pcm;
            a.jiffies = q.jiffies;
            a.silence = q.pcm == kSilencePiece ? 1u : 0u;
            a.attenuation = q.attenuation;
            a.reserved = 0;
            rs.out[(uint64_t)aEvent * kRecentPieces + i] = a;
        }
        if (plays) recent_clear(g);
    }
    if (plays) { r.pcmRun = 0; r.elemRamp = core::kRampMin; } // Pull(): FlywheelRamping -> RampingUp from kMin
}

OHP_HD bool push_msg(Stage& s, Packed* aRow, const Msg& m)
{
    if (s.depth == (uint32_t)kStackDepth) return false;
    aRow[s.depth++] = pack(m);
    return true;
}

// stage_chain.h Process(): one message through one stage; split remainders go onto the stage's stack (aRow).
// RECORD: aAttUp is the attenuation the stages in front of this one leave PCM with (their last that is not unity).
template <bool RECORD, bool RECENT>
OHP_HD uint32_t stage_process(StreamCtx& cx, RecentCtx<RECENT>& rs, Stage& s, uint32_t stage, Packed* aRow, Msg& msg, uint32_t aAttUp)
{
    while (s.nextAt <= s.pos) {
        if (RECORD) note_starvation<RECENT>(cx, rs, s, stage, s.nextEv);
        const ohp_ramp_event& e = cx.ev[s.nextEv];
        if (!apply_event(s, e.op, e.arg)) return kErrAssert;
        stage_seek(cx, s, stage, s.nextEv + 1);
    }
    Msg rest;
    if (s.nextAt < s.pos + msg.size) {
        uint32_t at = (uint32_t)(s.nextAt - s.pos);
        if (msg.silence) at -= at % cx.jps; // silence only splits on sample blocks
        if (at == 0) {
            if (RECORD) note_starvation<RECENT>(cx, rs, s, stage, s.nextEv);
            const ohp_ramp_event& e = cx.ev[s.nextEv];
            if (!apply_event(s, e.op, e.arg)) return kErrAssert;
            stage_seek(cx, s, stage, s.nextEv + 1);
        }
        else {
            const uint32_t e = msg_split(msg, at, rest, cx.jps);
            if (e != kOk) return e;
            if (!push_msg(s, aRow, rest)) return kErrDepth;
        }
    }
    if (s.maxMsg != 0 && msg.size > s.maxMsg) {
        if (s.maxMsg < cx.jps) return kErrSpec;
        const uint32_t e = msg_split(msg, s.maxMsg, rest, cx.jps);
        if (e != kOk) return e;
        if (!push_msg(s, aRow, rest)) return kErrDepth;
    }
    if (!msg.silence && s.attenuation != OHP_UNITY_ATTENUATION) {
        msg.atten = s.attenuation;
    }
    if (s.elem != Generic) {
        if (msg.silence) { // the element reacts, the message is handed on untouched
            element_sees_silence(s);
            if (RECORD) cx.sv[stage].pcmRun = 0;
            if constexpr (RECENT) {
                if (s.elem == ElemStarvation) recent_note(rs.ring[stage], kSilencePiece, msg.size, OHP_UNITY_ATTENUATION);
            }
            s.pos += msg.size;
            return kOk;
        }
        s.halted = 0;
    }
    if (s.mode == RampingDown || s.mode == RampingUp) {
        if (s.remaining > 0) {
            if (msg.size > s.remaining) {
                const uint32_t e = msg_split(msg, s.remaining, rest, cx.jps);
                if (e != kOk) return e;
                if (!push_msg(s, aRow, rest)) return kErrDepth;
                if (msg.size == 0) return kErrAssert; // a MsgSilence split below one sample (see stage_chain.h)
            }
            bool haveSplit;
            const uint32_t e = msg_set_ramp(msg, s.current, s.remaining, s.mode == RampingDown ? core::kDirDown : core::kDirUp,
                                            rest, haveSplit, s.current, cx.jps);
            if (e != kOk) return e;
            if (RECORD) cx.sv[stage].elemRamp = s.current;
            if (haveSplit && !push_msg(s, aRow, rest)) return kErrDepth;
        }
        if (s.remaining == 0) {
            if (s.mode == RampingUp) { s.mode = Running; s.current = core::kRampMax; }
            else { s.mode = Muted; s.current = core::kRampMin; }
        }
    }
    else if (s.mode == Muted) {
        core::ramp_set_muted(msg.ramp);
    }
    s.pos += msg.size;
    if (RECORD && !msg.silence && s.elem == ElemStarvation) {
        // the attenuation the message carries (stage_chain.h Process(): the stages up to this one are as it left them)
        Starve& r = cx.sv[stage];
        const uint32_t att = s.attenuation != OHP_UNITY_ATTENUATION ? s.attenuation : aAttUp;
        if (att != r.pcmRunAtt) { r.pcmRun = 0; r.pcmRunAtt = att; }
        if constexpr (RECENT) recent_note(rs.ring[stage], r.pcmJiffies, msg.size, att);
        r.pcmJiffies += msg.size;
        r.pcmRun += msg.size;
    }
    return kOk;
}

constexpr uint32_t kBulk = 32; // messages per bulk step

// Team-wide operations: a warp's shuffles on the device when a warp walks the stream, nothing for a team of one.
template <int STRIDE>
OHP_HD uint32_t team_scan_exclusive(uint32_t v, uint32_t aLane, uint32_t& aTotal)
{
#if defined(__CUDA_ARCH__)
    if (STRIDE == 32) {
        uint32_t x = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t y = __shfl_up_sync(0xffffffffu, x, o);
            if (aLane >= (uint32_t)o) x += y;
        }
        aTotal = __shfl_sync(0xffffffffu, x, 31);
        return x - v;
    }
#endif
    static_assert(STRIDE == 1 || STRIDE == 32, "a team is one thread or one warp");
    (void)aLane;
    aTotal = v;
    return 0;
}

template <int STRIDE>
OHP_HD bool team_any(bool aPred)
{
#if defined(__CUDA_ARCH__)
    if (STRIDE == 32) return __any_sync(0xffffffffu, aPred) != 0;
#endif
    return aPred;
}

// The walk's position in the source: what Run() of stage_chain.h keeps between messages.
struct Cursor
{
    uint64_t frame;       // frames of PCM fed so far
    uint64_t srcJiffies;  // the same in jiffies
    uint64_t silAt;       // at_jiffies of the next OHP_EV_INSERT_SILENCE event (index silEv), kNever when none is left
    uint32_t silEv;
};

OHP_HD void seek_silence(const StreamCtx& cx, Cursor& c, uint32_t aFrom)
{
    uint32_t i = aFrom;
    while (i < cx.nEv && cx.ev[i].op != OHP_EV_INSERT_SILENCE) i++;
    c.silEv = i;
    c.silAt = i < cx.nEv ? cx.ev[i].at_jiffies : kNever;
}

// Messages taken from the codec source but not yet fed (only behind a block-reading codec, CodecSource::read != 0,
// where message sizes are not uniform: the bulk step needs to see the sizes of the next ones).
struct Lookahead
{
    uint32_t frames[kBulk];
    uint32_t head, count;
};

OHP_HD void lookahead_fill(core::CodecSource& src, Lookahead& la)
{
    if (la.head != la.count) return;
    la.head = 0;
    la.count = 0;
    while (la.count < kBulk) {
        const uint32_t f = core::codec_source_next(src);
        if (f == 0) break;
        la.frames[la.count++] = f;
    }
}

// Frames of the next message to enter the stage chain (0: the stream is over).
OHP_HD uint32_t next_message(core::CodecSource& src, Lookahead& la)
{
    if (src.read == 0) return core::codec_source_next(src);
    lookahead_fill(src, la);
    return la.head != la.count ? la.frames[la.head++] : 0u;
}

// BULK STEP: up to kBulk consecutive messages at once, where nothing can happen to them but what is known up front.
//
// Between two events a stream is in a steady state: every stage is Running or Muted, or exactly one is ramping and
// the others are Running; no message is split, no stack is touched.  Then the only thing that is sequential is the
// ramping stage's recurrence (each message's ramp starts where the previous one ended, MsgAudio::SetRamp rounding up
// every time, Msg.cpp:603-605) -- one division per message.  Everything else (CreatePlayable's jiffy -> byte
// conversions, the descriptor) depends on the message's index and position alone.  So:
//   1. find the run: n messages that no event, ramp end, silence insertion, message-size cap or end of stream touches.
//      Uniform messages (CodecWav, or no codec): closed forms, a division only where something cuts the run short.
//      Behind a block-reading codec (CodecAiffBase + DecodedAudioAggregator: runs of 5 ms messages with a longer one
//      where two reads meet) the sizes come from a lookahead buffer and the same tests are made message by message;
//   2. run the recurrence over the run with the very code the general path uses (msg_set_ramp on a fresh message),
//      every lane of the team redundantly, lane (k % STRIDE) keeping message k's ramp, size and position; an early
//      finish (ramp reached kMin/kMax) or anything unusual ends the run there;
//   3. lane i builds and emits messages i, i + STRIDE, ...: STRIDE descriptors per step, written side by side;
//   3b. with a driver that pulls fixed blocks (MsgPlayable::Split, Msg.cpp:2591-2624) a message becomes several
//      playables; where the cuts fall follows from the message's position, so lanes agree on their output slots
//      through one prefix sum and each cuts its own message;
//   4. advance all state by n messages.
// Returns n; 0 means "take the general path for the next message".  What the reference would ASSERT on in the stages
// is left for the general path to find, at the same message; aErr only reports an ASSERT inside MsgPlayable::Split.
// UNIFORM: src.read == 0 (compiled separately so that the uniform case pays nothing for the ragged one's tests).
// RECORD: the StarvationRamper stages' PCM counters advance by the run (no event falls inside it, no MsgSilence either);
// the element's ramp value follows the recurrence where it is the stage that ramps.
// RECENT: the run joins the recent audio as one piece.
template <bool EMIT, int STRIDE, bool UNIFORM, bool RECORD, bool RECENT>
OHP_HD uint32_t bulk_step(const ohp_stream_spec& sp, StreamCtx& cx, RecentCtx<RECENT>& rs, Stage (&st)[kStages], core::CodecSource& src,
                          Lookahead& la, Cursor& cur, uint32_t& aErr)
{
    (void)rs;
    aErr = kOk;
    if (!(cx.bits == 8 || cx.bits == 16 || cx.bits == 24 || cx.bits == 32)) return 0;
    constexpr bool uniform = UNIFORM;
    uint32_t n, chunk = 0, size = 0;
    if (uniform) {
        chunk = src.chunk;
        size = chunk * cx.jps;
        if (size > 0xffffffffu / kBulk) return 0; // keep n * size in 32 bits (9216 one-byte frames at 7350 Hz: general path)
        n = kBulk;
        if (src.total_left < (uint64_t)n * chunk) n = (uint32_t)src.total_left / chunk;
    }
    else {
        lookahead_fill(src, la);
        n = la.count - la.head;
    }
    if (n == 0) return 0;
    if (cur.silAt <= cur.srcJiffies) return 0; // a MsgSilence is due first
    const uint64_t silRoom = cur.silAt - cur.srcJiffies; // message k goes ahead of it iff its position is below this
    if (uniform && silRoom <= (uint64_t)(n - 1) * size) n = (uint32_t)(silRoom - 1) / size + 1;
    // stages: what mode, which one ramps, what attenuation the messages leave with, how far the next event is
    uint32_t ramping = 0, muted = 0, atten = OHP_UNITY_ATTENUATION;
    uint32_t rMode = Running, rCurrent = 0, rRemaining = 0;
    uint32_t rLast = 0; // RECORD: what the last message's SetRamp returned (rCurrent before a completed ramp flips it)
    uint64_t eventRoom = kNever;     // jiffies that can pass every stage before its next event
    uint32_t sizeCap = 0xffffffffu;  // the tightest OHP_EV_MAX_MSG_JIFFIES in force
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int i = 0; i < kStages; i++) {
        const Stage& s = st[i];
        if (s.nextAt <= s.pos) return 0; // an event to apply first
        if (s.nextAt - s.pos < eventRoom) eventRoom = s.nextAt - s.pos;
        if (s.maxMsg != 0 && s.maxMsg < sizeCap) sizeCap = s.maxMsg;
        if (s.attenuation != OHP_UNITY_ATTENUATION) atten = s.attenuation;
        if (s.mode == Muted) muted++;
        else if (s.mode != Running) {
            ramping++;
            rMode = s.mode; rCurrent = s.current; rRemaining = s.remaining;
        }
    }
    if (ramping > 1 || (ramping == 1 && muted != 0)) return 0;
    if (ramping && rRemaining == 0) return 0; // a zero-length ramp: the general path flips the mode
    if (uniform) {
        if (size > sizeCap) return 0;
        if (eventRoom < (uint64_t)n * size) n = (uint32_t)eventRoom / size; // whole messages in front of the event
        if (ramping && rRemaining < n * size) n = rRemaining / size;        // ... and of the end of the ramp
        if (n == 0) return 0;
    }
    // the run, message by message: ragged sizes are tested as they come; the ramp recurrence advances
    core::RampPod mine[kBulk / STRIDE];
    uint32_t mineFrames[kBulk / STRIDE];
    uint32_t minePos[kBulk / STRIDE];   // frames of the run in front of the message
    uint32_t posFrames = 0;
    uint64_t posJiffies = 0;
    if (uniform && ramping) {
        // THE RAMP RECURRENCE, LEAN.  Every message of the run is fresh (no ramp of its own), whole, and lies inside
        // the ramp, so MsgAudio::SetRamp / Ramp::Set (msg_set_ramp / core::ramp_set) come down to
        //     delta = ceil(distance * size / remaining);  distance -= delta;  remaining -= size
        // with distance = how far the ramp still has to go (current for a ramp down, kRampMax - current for a ramp up).
        // This chain -- message k + 1 starts where k ended -- is what a stream's walk waits on (one warp per stream:
        // nothing else to issue meanwhile, so EVERY instruction in the loop costs its latency, on the chain or not), so
        // nothing but the chain is left in the loop.  Anything else -- a step of 0 (the reference ASSERTs:
        // Ramp::DoValidate), the ramp arriving (delta == distance: "finished early", Msg.cpp:2037-2043) or overshooting
        // -- ends the run in front of that message; the general path decides it.
        const bool down = rMode == RampingDown;
        const uint32_t dir = down ? core::kDirDown : core::kDirUp;
        uint32_t done = 0;
#if defined(__CUDA_ARCH__)
        if (STRIDE == kBulk && size < (1u << 21)) {
            // A warp, on the device: the chain runs through the FP64 pipe, on doubles that hold integers.  The divisors
            // are known up front (what is left of the ramp shrinks by one message each time), so the warp takes their 32
            // reciprocals side by side first and a step is fma, multiply, truncate, fma, compare.  EXACT: the numerator
            // distance * size + remaining - 1 is an integer below 2^31 * 2^21 + 2^32 < 2^53, so the first fma is exact;
            // the product with the reciprocal is off by less than 2^-19 (quotient <= 2^31 + 1, two roundings of 2^-53
            // each), so its truncation is the quotient or one beside it; the second fma gives that candidate's remainder
            // exactly (an integer of magnitude below 2^33), and its sign / size says which.  (4 M random and 12 M
            // adversarial numerators -- exact multiples of the divisor and their neighbours -- checked on the host
            // against integer division; every GPU schedule test compares the result with the host's integer walk.)
            // 38 instructions per message where the integer version had 57 (+ a call for the 64-bit division).
            // Measured and dropped: settling message k one iteration later, beside message k + 1's chain (a chain of
            // four operations, but 55 instructions: slower -- it is the instruction count that this loop pays for).
            const double sizeD = (double)size;
            double myInv = 0.0;
            if (rRemaining > cx.lane * size) myInv = 1.0 / (double)(rRemaining - cx.lane * size);
            double remD = (double)rRemaining;
            double distD = (double)(down ? rCurrent : core::kRampMax - rCurrent);
            double myFrom = 0.0; // distance in front of this lane's message (behind it: what the next lane has in front)
            uint32_t lane = cx.lane;
            asm volatile("" : "+r"(lane)); // held in a register: the compiler would otherwise recompute it from %tid in every iteration
            uint32_t k = 0;
            for (; k < n; k++) {
                const double inv = __shfl_sync(0xffffffffu, myInv, (int)k);
                const double numd = fma(distD, sizeD, remD - 1.0);
                double qd = trunc(numd * inv);
                const double r = fma(-qd, remD, numd);
                if (r < 0.0) qd -= 1.0;
                else if (r >= remD) qd += 1.0;
                if (qd == 0.0 || qd >= distD) break;
                if (k == lane) myFrom = distD;
                distD -= qd;
                remD -= sizeD;
            }
            done = k;
            double myTo = __shfl_down_sync(0xffffffffu, myFrom, 1);
            if (cx.lane + 1 >= done) myTo = distD;
            const uint32_t dist = __double2uint_rz(distD);
            rCurrent = down ? dist : core::kRampMax - dist;
            rRemaining -= done * size;
            if (cx.lane < done) {
                const uint32_t from = __double2uint_rz(myFrom), to = __double2uint_rz(myTo);
                core::RampPod& r = mine[0];
                r.start = down ? from : core::kRampMax - from;
                r.end = down ? to : core::kRampMax - to;
                r.direction = dir; r.enabled = 1;
            }
        }
        else
#endif
        {
            for (uint32_t k = 0; k < n; k++) {
                const uint32_t distance = down ? rCurrent : core::kRampMax - rCurrent;
                const uint32_t delta = core::mul_add_div(distance, size, rRemaining - 1, rRemaining);
                if (delta == 0 || delta >= distance) break;
                const uint32_t end = down ? rCurrent - delta : rCurrent + delta;
                if (k % STRIDE == cx.lane) {
                    core::RampPod& r = mine[k / STRIDE];
                    r.start = rCurrent; r.end = end; r.direction = dir; r.enabled = 1;
                }
                rCurrent = end;
                rRemaining -= size;
                done = k + 1;
            }
        }
        n = done;
        if (n == 0) return 0;
        rLast = rCurrent;
    }
    else if (!uniform) {
        const uint32_t dir = rMode == RampingDown ? core::kDirDown : core::kDirUp;
        uint32_t done = 0;
        for (uint32_t k = 0; k < n; k++) {
            const uint32_t f = uniform ? chunk : la.frames[la.head + k];
            const uint32_t sz = uniform ? size : f * cx.jps;
            if (!uniform) {
                if (sz > sizeCap || posJiffies + sz > eventRoom || posJiffies >= silRoom) break;
            }
            core::RampPod ramp;
            if (ramping) {
                if (!uniform && rRemaining < sz) break; // the ramp ends inside this message: it will be split
                Msg t, rest;
                t.cell = 0; t.size = sz; t.offset = 0; t.total = 0; t.atten = OHP_UNITY_ATTENUATION; t.silence = 0;
                core::ramp_reset(t.ramp);
                bool haveSplit;
                uint32_t remaining = rRemaining, current = rCurrent;
                const uint32_t e = msg_set_ramp(t, rCurrent, remaining, dir, rest, haveSplit, current, cx.jps);
                if (e != kOk || haveSplit) break;
                rRemaining = remaining; rCurrent = current;
                rLast = current;
                ramp = t.ramp;
            }
            else {
                core::ramp_reset(ramp);
            }
            if (k % STRIDE == cx.lane) {
                mine[k / STRIDE] = ramp;
                if (!uniform) { mineFrames[k / STRIDE] = f; minePos[k / STRIDE] = posFrames; }
            }
            if (!uniform) { posFrames += f; posJiffies += sz; }
            done = k + 1;
            if (ramping && rRemaining == 0) { // as stage_process: the ramp is over, this message was its last
                if (rMode == RampingUp) { rMode = Running; rCurrent = core::kRampMax; }
                else { rMode = Muted; rCurrent = core::kRampMin; }
                break;
            }
        }
        n = done;
        if (n == 0) return 0;
    }
    if (uniform) { // positions follow from the index
        posFrames = n * chunk;
        posJiffies = (uint64_t)n * size;
    }
    // every message of the run sits at offset 0 of its own cell; frames * frameBytes bytes each (CreatePlayable)
    Msg m;
    m.cell = 0; m.size = 0; m.offset = 0; m.total = 0; m.atten = atten; m.silence = 0;
    core::ramp_reset(m.ramp);
    if (muted) core::ramp_set_muted(m.ramp);
    const uint32_t block = cx.blockBytes;
    uint32_t pieces = 0; // playables emitted by the messages in front of this iteration's
    uint32_t err = kOk;
    if (EMIT || block != 0) {
        for (uint32_t i0 = 0; i0 < n; i0 += STRIDE) {
            const uint32_t i = i0 + cx.lane;
            const bool active = i < n;
            const uint32_t frames = !active ? 0u : (uniform ? chunk : mineFrames[i / STRIDE]);
            const uint32_t before_frames = !active ? 0u : (uniform ? i * chunk : minePos[i / STRIDE]);
            const uint32_t before_bytes = before_frames * cx.frameBytes;
            const uint32_t bytes = frames * cx.frameBytes;
            // a driver pulling fixed blocks (stage_chain.h Drive()): the message starts (fill + bytes before it) % block
            // into a block and is cut at every block boundary strictly inside it
            uint32_t fill = 0, count = active ? 1u : 0u;
            if (block != 0 && active) {
                fill = (cx.blockFill + before_bytes) % block;
                count += (fill + bytes - 1) / block;
            }
            uint32_t total;
            const uint32_t before = team_scan_exclusive<STRIDE>(count, cx.lane, total);
            if (active && (EMIT || ramping)) { // counting needs the cuts themselves only for what Ramp::Split may ASSERT on
                m.cell = sp.src_base + (cur.frame + before_frames) * cx.frameBytes;
                m.size = frames * cx.jps;
                if (ramping) m.ramp = mine[i / STRIDE];
                Playable p = create_playable(m, cx);
                uint64_t index = cx.nChunks + pieces + before;
                uint64_t off = cx.outBytes + before_bytes;
                while (block != 0 && p.size > block - fill) {
                    Playable rest;
                    const uint32_t e = playable_split(p, block - fill, rest, cx);
                    if (e != kOk) { err = e; break; }
                    if (EMIT) emit_desc(cx, p, index, off);
                    index++;
                    off += p.size;
                    fill = 0;
                    p = rest;
                }
                if (EMIT && err == kOk) emit_desc(cx, p, index, off);
            }
            pieces += total;
        }
        aErr = team_any<STRIDE>(err != kOk) ? kErrAssert : kOk; // playable_split's only failure is an ASSERT
    }
    else {
        pieces = n;
    }
    const uint64_t run_bytes = (uint64_t)posFrames * cx.frameBytes;
    if (block != 0) cx.blockFill = (uint32_t)((cx.blockFill + run_bytes) % block);
    // advance
    cx.nChunks += pieces;
    cx.outBytes += run_bytes;
    cur.frame += posFrames;
    cur.srcJiffies += posJiffies;
    if (uniform) src.total_left -= posFrames;
    else la.head += n;
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int i = 0; i < kStages; i++) {
        Stage& s = st[i];
        s.pos += posJiffies;
        if (RECORD && s.elem == ElemStarvation) {
            Starve& r = cx.sv[i];
            if ((s.mode == RampingDown || s.mode == RampingUp)) r.elemRamp = rLast;
            uint32_t att = OHP_UNITY_ATTENUATION;
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
            for (int j = 0; j <= i; j++) {
                if (st[j].attenuation != OHP_UNITY_ATTENUATION) att = st[j].attenuation;
            }
            if (att != r.pcmRunAtt) { r.pcmRun = 0; r.pcmRunAtt = att; }
            if constexpr (RECENT) recent_note(rs.ring[i], r.pcmJiffies, (uint32_t)posJiffies, att);
            r.pcmJiffies += posJiffies;
            r.pcmRun += posJiffies;
        }
        if (s.mode == RampingDown || s.mode == RampingUp) { s.mode = rMode; s.current = rCurrent; s.remaining = rRemaining; }
        if (s.elem != Generic) s.halted = 0; // PCM has passed
    }
    return n;
}

// One stream's walk.  The per-stage queues of stage_chain.h only ever grow at the front while a stage is being served
// and are drained before the stage returns, so each is a stack; Feed()'s recursion becomes: carry the message down
// the remaining stages (in registers), hand it to the driver, then resume with the top of the deepest non-empty stack.
// A team of STRIDE threads (device: a warp, or 1; host: 1) walks the stream holding identical state; they differ only
// in cx.lane, i.e. in which messages of a bulk step they emit.  BULK = false is the message-at-a-time walk alone.
template <bool EMIT, int STRIDE, bool BULK, bool RECORD, bool RECENT>
OHP_HD uint32_t walk_stream(const ohp_stream_spec& sp, StreamCtx& cx, RecentCtx<RECENT>& rs)
{
    static_assert(RECORD || !RECENT, "the recent audio goes with the records");
    Packed stack[kStages][kStackDepth];
    Stage st[kStages];
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int i = 0; i < kStages; i++) {
        st[i].pos = 0; st[i].mode = Running; st[i].current = core::kRampMax; st[i].remaining = 0; st[i].maxMsg = 0;
        st[i].attenuation = OHP_UNITY_ATTENUATION; st[i].depth = 0;
        st[i].elem = stage_element(cx, (uint32_t)i);
        st[i].halted = 1;
        if (RECORD) { cx.sv[i].pcmJiffies = 0; cx.sv[i].pcmRun = 0; cx.sv[i].pcmRunAtt = OHP_UNITY_ATTENUATION; cx.sv[i].elemRamp = core::kRampMax; }
        if constexpr (RECENT) recent_clear(rs.ring[i]);
        if (st[i].elem == ElemStarvation) st[i].maxMsg = 5u * OHP_JIFFIES_PER_MS; // kMaxAudioOutJiffies, StarvationRamper.cpp:376
        stage_seek(cx, st[i], (uint32_t)i, 0);
    }
    if (cx.jps == 0 || cx.frameBytes == 0) return kErrSpec;
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int i = 0; i < kStages; i++) {
        if (st[i].elem == ElemBad) return kErrSpec;
    }
    if (sp.chunk_frames == 0 || (uint64_t)sp.chunk_frames * cx.frameBytes > OHP_MAX_PCM_CHUNK_BYTES) return kErrSpec;

    // stage_chain.h Feed(0, item)
    auto feed = [&](const Msg& first) -> uint32_t {
        Msg m = first;
        int from = 0;
        for (;;) {
            uint32_t attUp = OHP_UNITY_ATTENUATION;
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
            for (int i = 0; i < kStages; i++) {
                if (i >= from) {
                    const uint32_t e = stage_process<RECORD, RECENT>(cx, rs, st[i], (uint32_t)i, stack[i], m, attUp);
                    if (e != kOk) return e;
                }
                if (RECORD && st[i].attenuation != OHP_UNITY_ATTENUATION) attUp = st[i].attenuation;
            }
            const uint32_t e2 = drive<EMIT>(cx, m);
            if (e2 != kOk) return e2;
            from = -1;
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
            for (int i = kStages - 1; i >= 0; i--) {
                if (from < 0 && st[i].depth != 0) {
                    from = i;
                    m = unpack(stack[i][--st[i].depth]);
                }
            }
            if (from < 0) return kOk;
        }
    };

    // stage_chain.h Run()
    Cursor cur;
    cur.frame = 0;
    cur.srcJiffies = 0;
    seek_silence(cx, cur, 0);
    core::CodecSource source;
    core::codec_source_init(source, sp.chunk_frames, sp.codec_read_frames, cx.frameBytes, cx.jps, sp.total_frames);
    Lookahead la;
    la.head = la.count = 0;
    for (;;) {
        if (BULK) {
            uint32_t e;
            const uint32_t n = source.read == 0 ? bulk_step<EMIT, STRIDE, true, RECORD, RECENT>(sp, cx, rs, st, source, la, cur, e)
                                                : bulk_step<EMIT, STRIDE, false, RECORD, RECENT>(sp, cx, rs, st, source, la, cur, e);
            if (e != kOk) return e;
#ifdef OHP_WALK_STATS
            if (n != 0) { g_bulk_calls++; g_bulk_msgs += n; }
#endif
            if (n != 0) continue;
        }
        const uint32_t frames = next_message(source, la);
#ifdef OHP_WALK_STATS
        if (frames != 0) g_general++;
#endif
        if (frames == 0) break;
        Msg m;
        while (cur.silAt <= cur.srcJiffies) {
            // MsgFactory::CreateMsgSilence / MsgSilence::Initialise (Msg.cpp:2547-2560)
            uint32_t jiffies = cx.ev[cur.silEv].arg;
            core::round_down_non_zero_sample_block(jiffies, cx.jps);
            m.cell = 0; m.size = jiffies; m.total = jiffies; m.offset = 0; m.atten = OHP_UNITY_ATTENUATION; m.silence = 1;
            core::ramp_reset(m.ramp);
            const uint32_t rc = feed(m);
            if (rc != kOk) return rc;
            seek_silence(cx, cur, cur.silEv + 1);
        }
        // DecodedAudio::ConstructPcm ASSERTs on the bit depth (Msg.cpp:349-366)
        if (!(cx.bits == 8 || cx.bits == 16 || cx.bits == 24 || cx.bits == 32)) return kErrAssert;
        m.cell = sp.src_base + cur.frame * cx.frameBytes;
        m.size = frames * cx.jps;
        m.total = 0; m.offset = 0; m.atten = OHP_UNITY_ATTENUATION; m.silence = 0;
        core::ramp_reset(m.ramp);
        const uint32_t rc = feed(m);
        if (rc != kOk) return rc;
        cur.frame += frames;
        cur.srcJiffies += (uint64_t)frames * cx.jps;
    }
    if (RECORD) {
        // stage_chain.h Run(): a reservoir that runs dry exactly where the stream ends still starves its StarvationRamper
        // (no message is left for the event to be applied in front of)
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
        for (int i = 0; i < kStages; i++) {
            Stage& s = st[i];
            while (s.elem == ElemStarvation && s.nextAt <= s.pos) {
                note_starvation<RECENT>(cx, rs, s, (uint32_t)i, s.nextEv);
                const ohp_ramp_event& e = cx.ev[s.nextEv];
                (void)apply_element_event(s, e.op, e.arg); // OHP_EV_HALT / OHP_EV_STARVATION: state only
                stage_seek(cx, s, (uint32_t)i, s.nextEv + 1);
            }
        }
    }
    return kOk;
}

// Fill the per-stream context from a spec and walk it.  aEvents is the WHOLE events array (aNumEvents entries).
// aLane: this thread's index in its team of STRIDE (0 on the host).
// RECORD: starvation records go to aRec -- the record of the stream's k-th event at aRec[k] (aRec: the stream's first
// event's place in an array over the whole events array), or, with aAppend, one after the other; aNumRecords counts them.
// RECENT (not with aAppend): the k-th event's record also leaves its pieces of recent audio at aRecent[k * kRecentPieces ...]
// and their number at aRecentCount[k] (both at the stream's first event's place, as aRec).
template <bool EMIT, int STRIDE = 1, bool BULK = true, bool RECORD = false, bool RECENT = false>
OHP_HD uint32_t run_stream(const ohp_stream_spec& sp, const ohp_ramp_event* aEvents, uint64_t aNumEvents,
                           ohp_chunk_desc* aDescs, ohp_chunk_info* aInfo, uint64_t& aNumChunks, uint64_t& aOutBytes,
                           uint32_t aLane = 0, uint64_t aLimit = ~0ull,
                           ohp_starvation* aRec = nullptr, uint64_t aStream = 0, bool aAppend = false, uint32_t* aNumRecords = nullptr,
                           ohp_recent_audio* aRecent = nullptr, uint32_t* aRecentCount = nullptr)
{
    aNumChunks = 0;
    aOutBytes = 0;
    if ((uint64_t)sp.first_event + sp.num_events > aNumEvents) return kErrSpec;
    if (!(sp.out_fmt == OHP_OUT_PACKED_BE || sp.out_fmt == OHP_OUT_PACKED_LE)) return kErrSpec;
    StreamCtx cx;
    cx.ev = aEvents + sp.first_event;
    cx.nEv = sp.num_events;
    cx.jps = core::jiffies_per_sample_or_zero(sp.sample_rate);
    cx.channels = sp.channels;
    cx.bits = sp.bit_depth;
    cx.frameBytes = sp.channels * (sp.bit_depth / 8u);
    cx.in_le = sp.in_little_endian ? 1u : 0u;
    cx.out_fmt = sp.out_fmt;
    cx.blockBytes = sp.driver_block_frames * cx.frameBytes;
    cx.blockFill = 0;
    cx.dst_base = sp.dst_base;
    cx.lane = aLane;
    cx.nChunks = 0;
    cx.outBytes = 0;
    cx.descs = EMIT ? aDescs : nullptr;
    cx.info = EMIT ? aInfo : nullptr;
    cx.limit = aLimit;
    if (RECORD) {
        cx.rec = aRec;
        cx.recAppend = aAppend ? 1u : 0u;
        cx.nRec = 0;
        cx.stream = aStream;
        cx.firstEvent = sp.first_event;
    }
    RecentCtx<RECENT> rs;
    if constexpr (RECENT) { rs.out = aRecent; rs.count = aRecentCount; rs.stride = (uint32_t)STRIDE; }
    else { (void)aRecent; (void)aRecentCount; }
    const uint32_t rc = walk_stream<EMIT, STRIDE, BULK, RECORD, RECENT>(sp, cx, rs);
    if (RECORD && aNumRecords) *aNumRecords = cx.nRec;
    if (rc != kOk) return rc;
    aNumChunks = cx.nChunks;
    aOutBytes = cx.outBytes;
    return kOk;
}

// An UPPER BOUND on the playables of a stream, in closed form from its spec and events -- what lets the descriptors be
// built in ONE walk: every stream gets a region of this many descriptors, writes what it has and zero-fills the rest
// (a zero-byte descriptor is a playable MsgPlayable::Read does nothing for, Msg.cpp:2649).  Counted:
//   * the messages the codec delivers (behind a block-reading codec: the pieces CodecController cuts, which
//     DecodedAudioAggregator only ever merges), one per MsgSilence;
//   * a stage that holds messages to a size smaller than the largest message there is: at most total / cap more;
//   * per event: the message it falls inside is split (1) and the ramp it starts ends inside a message (1); a MsgHalt, a
//     MsgDecodedStream or a call that turns a ramp round costs no more than that;
//   * two ramps running against each other cross in at most one message (Ramp::Set's split fragment, Msg.cpp:637-699),
//     and a message takes one ramp from each stage it passes: one per pair of events on DIFFERENT stages;
//   * a driver pulling fixed blocks cuts at every block boundary of the stream's output.
// 0 for a stream the walk will refuse anyway.  tests/test_schedule_walk.py holds it against the exact counts.
OHP_HD uint64_t stream_chunk_bound(const ohp_stream_spec& sp, const ohp_ramp_event* aEvents, uint64_t aNumEvents)
{
    if ((uint64_t)sp.first_event + sp.num_events > aNumEvents) return 0;
    const uint32_t jps = core::jiffies_per_sample_or_zero(sp.sample_rate);
    const uint64_t frameBytes = (uint64_t)sp.channels * (sp.bit_depth / 8u);
    if (jps == 0 || frameBytes == 0 || sp.chunk_frames == 0 || (uint64_t)sp.chunk_frames * frameBytes > OHP_MAX_PCM_CHUNK_BYTES) return 0;
    const ohp_ramp_event* ev = aEvents + sp.first_event;
    uint64_t msgs = (sp.total_frames + sp.chunk_frames - 1) / sp.chunk_frames;
    uint64_t largest = (uint64_t)sp.chunk_frames * jps;           // jiffies of the largest message that can enter a stage
    if (sp.codec_read_frames != 0) {
        msgs += (sp.total_frames + sp.codec_read_frames - 1) / sp.codec_read_frames + 1;
        const uint64_t cell = (OHP_MAX_PCM_CHUNK_BYTES / frameBytes) * jps;
        if (cell > largest) largest = cell;
    }
    uint64_t frames = sp.total_frames, nEv = 0;
    uint32_t cap[kStages];
    uint64_t perStage[kStages];
    for (int i = 0; i < kStages; i++) { cap[i] = 0; perStage[i] = 0; }
    for (uint32_t i = 0; i < sp.num_events; i++) {
        const ohp_ramp_event& e = ev[i];
        if (e.op == OHP_EV_INSERT_SILENCE) {
            msgs++;
            frames += e.arg / jps + 1;
            if (e.arg > largest) largest = e.arg;
            continue;
        }
        nEv++;
        if (e.stage >= (uint32_t)kStages) continue;
        perStage[e.stage]++;
        uint32_t c = 0;
        if (e.op == OHP_EV_MAX_MSG_JIFFIES) c = e.arg;
        else if (e.op == OHP_EV_STARVATION) c = 5u * OHP_JIFFIES_PER_MS;
        if (c != 0 && (cap[e.stage] == 0 || c < cap[e.stage])) cap[e.stage] = c;
    }
    const uint64_t total = frames * jps;
    uint64_t bound = msgs;
    for (int i = 0; i < kStages; i++) {
        if (cap[i] != 0 && largest > cap[i]) bound += total / (cap[i] < jps ? jps : cap[i]) + 1;
    }
    bound += 2u * nEv;
    for (int i = 0; i < kStages; i++) {
        for (int j = i + 1; j < kStages; j++) bound += perStage[i] * perStage[j];
    }
    if (sp.driver_block_frames != 0) bound += frames / sp.driver_block_frames + 1;
    return bound + 4;
}

} // namespace sched
} // namespace ohp
