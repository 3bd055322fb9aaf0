// flywheel_plan.h -- ohp_flywheel_plan (PCM training blocks only) and ohp_flywheel_ramp_chunks restated on plain data,
// compiled for BOTH the device (csrc/ohp_schedule_kernels.cuh: plan_kernel, one thread per starvation record) and the
// host (tests/test_starvation_walk.py builds a small harness on it and holds it against the class-based functions of
// schedule.cpp, descriptor for descriptor).  The message steps are those of the schedule walk: msg_set_ramp (MsgAudio::
// SetRamp) and create_playable (MsgAudioPcm::CreatePlayable) on the RampGenerator's 1 ms messages.
#pragma once

#include <cstdint>

#include "../../include/ohp_schedule.h"
#include "ramp_core.h"
#include "schedule_walk.h"

namespace ohp {
namespace flyplan {

// RampGenerator's messages for one 20 ms flywheel ramp: 1 ms each, the last one shorter (44.1 kHz family: 21)
constexpr uint32_t kMaxBlocks = OHP_FLYWHEEL_RAMP_JIFFIES / OHP_FLYWHEEL_BLOCK_JIFFIES + 1;

OHP_HD ohp_chunk_desc zero_desc()
{
    ohp_chunk_desc d;
    d.src_off = 0; d.dst_off = 0; d.bytes = 0; d.ramp_start = 0; d.ramp_end = 0; d.attenuation = 0;
    d.bit_depth = 0; d.channels = 0; d.flags = 0; d.out_fmt = 0; d.aux = 0;
    return d;
}

// ohp_flywheel_ramp_chunks: RampGenerator::Start + EndBlock (StarvationRamper.cpp:235-247, 351-364), one descriptor per
// 1 ms block into out[0..kMaxBlocks).  Returns OHP_OK with aN set, or OHP_E_INVALID_DESC where the reference ASSERTs.
OHP_HD int ramp_chunks(const ohp_flywheel_job& job, uint32_t aRamp, uint64_t aSrc, uint64_t aDst, ohp_chunk_desc* out, uint32_t& aN)
{
    aN = 0;
    sched::StreamCtx cx;
    cx.jps = core::jiffies_per_sample_or_zero(job.sample_rate);
    if (cx.jps == 0) return OHP_E_INVALID_DESC; // Jiffies::PerSample throws
    cx.channels = job.channels;
    cx.bits = job.bit_depth;
    const uint32_t blockFrames = OHP_FLYWHEEL_BLOCK_JIFFIES / cx.jps;
    uint32_t remainingRamp = cx.jps * job.out_frames;
    uint32_t remaining = job.out_frames;
    while (remaining > 0) {
        const uint32_t frames = remaining > blockFrames ? blockFrames : remaining;
        remaining -= frames;
        if (aN == kMaxBlocks) return OHP_E_NO_MEMORY;
        sched::Msg m;
        m.cell = aSrc; m.size = frames * cx.jps; m.offset = 0; m.total = 0; m.atten = OHP_UNITY_ATTENUATION; m.silence = 0;
        core::ramp_reset(m.ramp);
        if (aRamp == core::kRampMin) {
            core::ramp_set_muted(m.ramp);
        }
        else {
            sched::Msg split;
            bool haveSplit;
            if (sched::msg_set_ramp(m, aRamp, remainingRamp, core::kDirDown, split, haveSplit, aRamp, cx.jps) != sched::kOk || haveSplit) {
                return OHP_E_INVALID_DESC; // ASSERT(split == nullptr), StarvationRamper.cpp:359
            }
        }
        const sched::Playable p = sched::create_playable(m, cx);
        ohp_chunk_desc d = zero_desc(); // MsgPlayable::Descriptor, big-endian messages
        d.src_off = p.silence ? 0 : p.arena;
        d.dst_off = aDst;
        d.bytes = p.size;
        d.ramp_start = (uint16_t)p.ramp.start;
        d.ramp_end = (uint16_t)p.ramp.end;
        d.attenuation = (uint16_t)p.atten;
        d.bit_depth = (uint8_t)cx.bits;
        d.channels = (uint8_t)cx.channels;
        d.flags = (uint8_t)((p.ramp.enabled ? OHP_F_RAMP_ENABLED : 0u) | (p.silence ? OHP_F_SILENCE : 0u));
        d.out_fmt = OHP_OUT_PACKED_BE;
        out[aN++] = d;
        aSrc += p.size;
        aDst += p.size;
    }
    return OHP_OK;
}

// ohp_flywheel_plan: prep[0..aNumPrep) (room for OHP_FLYWHEEL_MAX_PREP), the job, blocks[0..aNumBlocks) (room for
// kMaxBlocks).  Refuses what it refuses, with the same status: plays nothing, not PCM of one attenuation for the last
// 1 ms, a record that does not fit the stream (OHP_E_INVALID_ARG); shapes the reference's flywheel buffers do not hold
// (OHP_E_INVALID_DESC).
OHP_HD int plan(const ohp_stream_spec& sp, const ohp_starvation& sv, uint64_t aTrainingOff, uint64_t aGeneratedOff, uint64_t aOutOff,
                ohp_chunk_desc* prep, uint32_t& aNumPrep, ohp_flywheel_job& job, ohp_chunk_desc* blocks, uint32_t& aNumBlocks)
{
    aNumPrep = 0;
    aNumBlocks = 0;
    const uint32_t jps = core::jiffies_per_sample_or_zero(sp.sample_rate);
    const uint32_t B = sp.bit_depth / 8u;
    const uint32_t C = sp.channels;
    const uint32_t frameBytes = C * B;
    if (jps == 0 || frameBytes == 0 || !(sp.bit_depth == 8 || sp.bit_depth == 16 || sp.bit_depth == 24 || sp.bit_depth == 32)) return OHP_E_INVALID_ARG;
    if (C > OHP_FLYWHEEL_MAX_CHANNELS) return OHP_E_INVALID_DESC;
    if (!sv.plays) return OHP_E_INVALID_ARG;
    if (sv.recent_jiffies < OHP_FLYWHEEL_TRAINING_JIFFIES || sv.pcm_jiffies < OHP_FLYWHEEL_TRAINING_JIFFIES) return OHP_E_INVALID_ARG;
    // StartFlywheelRamp's cut to the last kTrainingJiffies, every message rounded down to a sample at both ends
    const uint64_t lastFrame = sv.pcm_jiffies / jps;
    const uint64_t firstFrame = (sv.pcm_jiffies - OHP_FLYWHEEL_TRAINING_JIFFIES) / jps;
    const uint32_t got = (uint32_t)(lastFrame - firstFrame);
    const uint32_t train = OHP_FLYWHEEL_TRAINING_JIFFIES / jps; // FlywheelInput's planes
    if (lastFrame > sp.total_frames || (got != train && got != train + 1) || train < 2) return OHP_E_INVALID_ARG;
    {
        const uint32_t decimation = (sp.sample_rate == 192000u || sp.sample_rate == 176400u) ? 4u
                                  : (sp.sample_rate == 88200u || sp.sample_rate == 96000u) ? 2u : 1u;
        const uint32_t blockFrames = OHP_FLYWHEEL_BLOCK_JIFFIES / jps;
        if (train / decimation < OHP_FLYWHEEL_DEGREE + 1u || train * 4u * C > OHP_FLYWHEEL_MAX_INPUT_BYTES
            || blockFrames * frameBytes > OHP_FLYWHEEL_MAX_BLOCK_BYTES) {
            return OHP_E_INVALID_DESC;
        }
    }
    const uint8_t flags = (uint8_t)((sp.in_little_endian && B > 1) ? OHP_F_IN_LITTLE_ENDIAN : 0);
    // FlywheelPlayableCreator clears the messages' ramps, not their attenuation
    auto planar = [&](uint64_t aSrc, uint64_t aDstSlot, uint32_t aBytes, uint32_t aChannels) {
        ohp_chunk_desc d = zero_desc();
        d.src_off = aSrc;
        d.dst_off = aTrainingOff + aDstSlot * 4u;
        d.bytes = aBytes;
        d.ramp_start = (uint16_t)core::kRampMax;
        d.ramp_end = (uint16_t)core::kRampMax;
        d.attenuation = (uint16_t)sv.attenuation;
        d.bit_depth = (uint8_t)sp.bit_depth;
        d.channels = (uint8_t)aChannels;
        d.flags = flags;
        d.out_fmt = OHP_OUT_PLANAR32_BE;
        d.aux = (uint16_t)train;
        prep[aNumPrep++] = d;
    };
    const uint64_t src = sp.src_base + firstFrame * frameBytes;
    if (got == train || C == 1) {
        planar(src, 0, train * frameBytes, C); // mono with a frame too many: the last subsample falls beyond the block
    }
    else {
        // a frame too many: channel c's last subsample lands on channel c + 1's first slot, the last channel's beyond
        planar(src + frameBytes, 1, (train - 1) * frameBytes, C);
        planar(src, 0, B, 1);
        for (uint32_t c = 1; c < C; c++) planar(src + (uint64_t)train * frameBytes + (c - 1) * B, (uint64_t)c * train, B, 1);
    }
    // FlywheelRamperManager::Ramp: 20 ms from the 1 ms block
    job.src_off = aTrainingOff;
    job.dst_off = aGeneratedOff;
    job.sample_rate = sp.sample_rate;
    job.out_frames = OHP_FLYWHEEL_RAMP_JIFFIES / jps;
    job.train_frames = (uint16_t)train;
    job.channels = (uint8_t)C;
    job.bit_depth = (uint8_t)sp.bit_depth;
    job.reserved = 0;
    // RampGenerator plays it from the element's ramp value down
    const int rc = ramp_chunks(job, sv.ramp, aGeneratedOff, aOutOff, blocks, aNumBlocks);
    if (rc != OHP_OK) aNumPrep = 0;
    return rc;
}

// ohp_flywheel_plan_recent on the record's pieces of recent audio (pieces[0..aNumPieces), oldest first), with room for
// OHP_FLYWHEEL_MAX_PREP_RECENT prep descriptors: the same status, and on OHP_OK the same descriptors.  The pieces are walked
// three times (the cut, the frames FlywheelInput reads, the descriptors) instead of being collected.
OHP_HD int plan_recent(const ohp_stream_spec& sp, const ohp_starvation& sv, const ohp_recent_audio* pieces, uint32_t aNumPieces,
                       uint64_t aTrainingOff, uint64_t aGeneratedOff, uint64_t aOutOff,
                       ohp_chunk_desc* prep, uint32_t& aNumPrep, ohp_flywheel_job& job, ohp_chunk_desc* blocks, uint32_t& aNumBlocks)
{
    aNumPrep = 0;
    aNumBlocks = 0;
    const uint32_t jps = core::jiffies_per_sample_or_zero(sp.sample_rate);
    const uint32_t B = sp.bit_depth / 8u;
    const uint32_t C = sp.channels;
    const uint32_t frameBytes = C * B;
    if (jps == 0 || frameBytes == 0 || !(sp.bit_depth == 8 || sp.bit_depth == 16 || sp.bit_depth == 24 || sp.bit_depth == 32)) return OHP_E_INVALID_ARG;
    if (C > OHP_FLYWHEEL_MAX_CHANNELS) return OHP_E_INVALID_DESC;
    if (!sv.plays) return OHP_E_INVALID_ARG;
    const uint32_t train = OHP_FLYWHEEL_TRAINING_JIFFIES / jps;
    {
        const uint32_t decimation = (sp.sample_rate == 192000u || sp.sample_rate == 176400u) ? 4u
                                  : (sp.sample_rate == 88200u || sp.sample_rate == 96000u) ? 2u : 1u;
        const uint32_t blockFrames = OHP_FLYWHEEL_BLOCK_JIFFIES / jps;
        if (train < 2 || train / decimation < OHP_FLYWHEEL_DEGREE + 1u || train * 4u * C > OHP_FLYWHEEL_MAX_INPUT_BYTES
            || blockFrames * frameBytes > OHP_FLYWHEEL_MAX_BLOCK_BYTES) {
            return OHP_E_INVALID_DESC;
        }
    }
    // StartFlywheelRamp's cut: whole pieces go from the front while more than kTrainingJiffies is left, the piece under the
    // cut is split (head: that piece after the cut)
    uint64_t total = 0;
    for (uint32_t i = 0; i < aNumPieces; i++) total += pieces[i].jiffies;
    if (total < OHP_FLYWHEEL_TRAINING_JIFFIES) return OHP_E_INVALID_ARG;
    uint64_t excess = total - OHP_FLYWHEEL_TRAINING_JIFFIES;
    uint32_t first = 0;
    ohp_recent_audio head = {0, 0, 0, 0, 0};
    while (first < aNumPieces) {
        head = pieces[first];
        if (excess == 0) break;
        if (head.jiffies > excess) {
            if (head.silence && excess % jps != 0) return OHP_E_INVALID_DESC; // the cut that never ends
            head.jiffies -= (uint32_t)excess;
            if (!head.silence) head.pcm_jiffies += excess;
            excess = 0;
            break;
        }
        excess -= head.jiffies;
        first++;
    }
    // piece i (from `first`) through CreatePlayable: silence, first frame, frames, attenuation
    auto run = [&](uint32_t i, bool& aSilence, uint64_t& aFirstFrame, uint32_t& aFrames, uint32_t& aAtt) {
        const ohp_recent_audio& p = i == first ? head : pieces[i];
        aSilence = p.silence != 0;
        aAtt = p.silence ? OHP_UNITY_ATTENUATION : p.attenuation;
        if (p.silence) {
            aFirstFrame = 0;
            aFrames = p.jiffies / jps;
        }
        else {
            aFirstFrame = p.pcm_jiffies / jps;
            aFrames = (uint32_t)((p.pcm_jiffies + p.jiffies) / jps - aFirstFrame);
        }
        return p.silence || (p.pcm_jiffies + p.jiffies) / jps <= sp.total_frames;
    };
    uint64_t got = 0;
    uint32_t firstRun = aNumPieces, lastRun = aNumPieces; // the first and last pieces that give frames
    for (uint32_t i = first; i < aNumPieces; i++) {
        bool silence; uint64_t firstFrame; uint32_t frames, att;
        if (!run(i, silence, firstFrame, frames, att)) return OHP_E_INVALID_ARG; // a piece outside the stream
        if (frames == 0) continue;
        if (firstRun == aNumPieces) firstRun = i;
        lastRun = i;
        got += frames;
    }
    if (got < train || got > (uint64_t)train + 1u) return OHP_E_INVALID_ARG;
    const uint8_t le = (uint8_t)((sp.in_little_endian && B > 1) ? OHP_F_IN_LITTLE_ENDIAN : 0);
    bool full = false;
    // frames [aFrom, aFrom + aCount) of piece i, channels [aCh, aCh + aChannels), to slot aSlot of plane aCh and on
    auto emit = [&](uint32_t i, uint32_t aFrom, uint32_t aCount, uint32_t aCh, uint32_t aChannels, uint64_t aSlot) {
        if (aNumPrep == OHP_FLYWHEEL_MAX_PREP_RECENT) { full = true; return; }
        bool silence; uint64_t firstFrame; uint32_t frames, att;
        (void)run(i, silence, firstFrame, frames, att);
        ohp_chunk_desc d = zero_desc();
        d.src_off = silence ? 0 : sp.src_base + (firstFrame + aFrom) * frameBytes + (uint64_t)aCh * B;
        d.dst_off = aTrainingOff + aSlot * 4u;
        d.bytes = aCount * aChannels * B;
        d.ramp_start = (uint16_t)core::kRampMax;
        d.ramp_end = (uint16_t)core::kRampMax;
        d.attenuation = (uint16_t)att;
        d.bit_depth = (uint8_t)sp.bit_depth;
        d.channels = (uint8_t)aChannels;
        d.flags = (uint8_t)(silence ? OHP_F_SILENCE : le);
        d.out_fmt = OHP_OUT_PLANAR32_BE;
        d.aux = (uint16_t)train;
        prep[aNumPrep++] = d;
    };
    // frames [lo, hi) of those read go out whole; with a frame too many and more than one channel, every plane's first slot
    // is written last by another frame (as ohp_flywheel_plan_recent)
    const bool over = got == (uint64_t)train + 1u;
    const uint64_t lo = (over && C > 1) ? 1 : 0, hi = train;
    uint64_t at = 0;
    for (uint32_t i = first; i < aNumPieces; i++) {
        bool silence; uint64_t firstFrame; uint32_t frames, att;
        (void)run(i, silence, firstFrame, frames, att);
        if (frames == 0) continue;
        const uint64_t a = at > lo ? at : lo, b = (at + frames) < hi ? (at + frames) : hi;
        if (b > a) emit(i, (uint32_t)(a - at), (uint32_t)(b - a), 0, C, a);
        at += frames;
    }
    if (over && C > 1) {
        bool silence; uint64_t firstFrame; uint32_t frames, att;
        (void)run(lastRun, silence, firstFrame, frames, att);
        emit(firstRun, 0, 1, 0, 1, 0);
        for (uint32_t c = 1; c < C; c++) emit(lastRun, frames - 1, 1, c - 1, 1, (uint64_t)c * train);
    }
    if (full) {
        aNumPrep = 0;
        return OHP_E_INVALID_ARG;
    }
    job.src_off = aTrainingOff;
    job.dst_off = aGeneratedOff;
    job.sample_rate = sp.sample_rate;
    job.out_frames = OHP_FLYWHEEL_RAMP_JIFFIES / jps;
    job.train_frames = (uint16_t)train;
    job.channels = (uint8_t)C;
    job.bit_depth = (uint8_t)sp.bit_depth;
    job.reserved = 0;
    const int rc = ramp_chunks(job, sv.ramp, aGeneratedOff, aOutOff, blocks, aNumBlocks);
    if (rc != OHP_OK) aNumPrep = 0;
    return rc;
}

} // namespace flyplan
} // namespace ohp
