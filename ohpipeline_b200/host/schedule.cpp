// schedule.cpp -- the C ABI of include/ohp_schedule.h on top of the host message model.
//
// Runs every stream's ramp events through the stage chain (stage_chain.h) on the mirror classes
// (msg_model.h) and records one ohp_chunk_desc per MsgPlayable.  Threaded over streams; streams are
// independent (SURVEY 8e), so no synchronisation beyond the final gather.
#include "msg_model.h"
#include "stage_chain.h"
#include "schedule_walk.h"

#include <string>
#include <thread>
#include <memory>
#include <new>
#include <vector>

using namespace ohp;
using namespace ohp::media;

namespace {

struct MirrorApi
{
    using MsgAudio = media::MsgAudio;
    using MsgAudioPcm = media::MsgAudioPcm;
    using MsgSilence = media::MsgSilence;
    using MsgPlayable = media::MsgPlayable;
    using Factory = media::MsgFactory;
    static const uint32_t kRampMax = Ramp::kMax;
    static const uint32_t kRampMin = Ramp::kMin;
    static const Ramp::EDirection kDirUp = Ramp::EUp;
    static const Ramp::EDirection kDirDown = Ramp::EDown;
    static MsgAudioPcm* CreatePcm(Factory& f, const ohp_stream_spec& sp, uint64_t firstFrame, uint32_t frames)
    {
        const uint32_t frameBytes = sp.channels * (sp.bit_depth / 8u);
        return f.CreateMsgAudioPcm(sp.src_base + firstFrame * frameBytes, frames * frameBytes, sp.channels, sp.sample_rate,
                                   sp.bit_depth, sp.in_little_endian ? AudioDataEndian::Little : AudioDataEndian::Big,
                                   firstFrame * (uint64_t)Jiffies::PerSampleOrZero(sp.sample_rate));
    }
    static MsgSilence* CreateSilence(Factory& f, const ohp_stream_spec& sp, uint32_t& jiffies)
    {
        return f.CreateMsgSilence(jiffies, sp.sample_rate, sp.bit_depth, sp.channels);
    }
    static uint32_t JiffiesPerSample(uint32_t rate) { return Jiffies::PerSampleOrZero(rate); }
    static void Assert(bool ok) { OHP_ASSERT(ok); }
};

struct StreamRecord
{
    std::vector<ohp_chunk_desc> chunks;
    std::vector<ohp_chunk_info> info;
    uint64_t outBytes = 0;
    std::vector<ohp_starvation> starvations;
    std::vector<ohp_recent_audio> recent;   // ... their recent audio, piece by piece
    std::vector<uint64_t> recentCount;      // ... pieces per starvation
};

class DescSink
{
public:
    DescSink(const ohp_stream_spec& sp, StreamRecord& rec) : iSpec(sp), iRec(rec) {}
    void OnPlayable(MsgPlayable* p)
    {
        iRec.chunks.push_back(p->Descriptor(iSpec.dst_base + iRec.outBytes, iSpec.out_fmt));
        iRec.info.push_back(ohp_chunk_info{(uint32_t)p->Ramp().Direction(), p->Jiffies()});
        iRec.outBytes += p->Bytes();
        p->RemoveRef();
    }
private:
    const ohp_stream_spec& iSpec;
    StreamRecord& iRec;
};

thread_local std::string g_error;

} // namespace

struct ohp_schedule
{
    std::vector<ohp_chunk_desc> chunks;
    std::vector<ohp_chunk_info> info;
    std::vector<uint64_t> chunkBegin;
    std::vector<uint64_t> outBytes;
    std::vector<ohp_starvation> starvations;
    std::vector<ohp_recent_audio> recent;
    std::vector<uint64_t> recentBegin = std::vector<uint64_t>(1, 0); // starvations.size() + 1
};

struct ohp_flywheel_batch
{
    std::vector<uint32_t> planned;
    std::vector<uint64_t> outOff, outLen;
    std::vector<ohp_chunk_desc> prep, blocks;
    std::vector<ohp_flywheel_job> jobs;
    uint64_t arena[3] = {0, 0, 0};
};

extern "C" {

int ohp_schedule_build(const ohp_stream_spec* streams, size_t n_streams, const ohp_ramp_event* events, size_t n_events,
                       int threads, ohp_schedule** out)
{
    if (!out || (!streams && n_streams) || (!events && n_events)) {
        g_error = "null argument";
        return OHP_E_INVALID_ARG;
    }
    *out = nullptr;
    for (size_t s = 0; s < n_streams; s++) {
        if ((uint64_t)streams[s].first_event + streams[s].num_events > n_events) {
            g_error = "stream " + std::to_string(s) + ": event slice out of range";
            return OHP_E_INVALID_ARG;
        }
        if (!(streams[s].out_fmt == OHP_OUT_PACKED_BE || streams[s].out_fmt == OHP_OUT_PACKED_LE)) {
            g_error = "stream " + std::to_string(s) + ": schedule runs produce packed BE or LE output";
            return OHP_E_INVALID_ARG;
        }
    }
    if (threads <= 0) threads = (int)std::thread::hardware_concurrency();
    if (threads <= 0) threads = 1;
    if ((size_t)threads > n_streams) threads = (int)(n_streams ? n_streams : 1);

    std::vector<StreamRecord> recs(n_streams);
    std::vector<int> rcs((size_t)threads, 0);
    std::vector<std::string> errs((size_t)threads);
    auto worker = [&](int t) {
        MsgFactory factory;
        const size_t lo = n_streams * (size_t)t / (size_t)threads;
        const size_t hi = n_streams * (size_t)(t + 1) / (size_t)threads;
        for (size_t s = lo; s < hi; s++) {
            DescSink sink(streams[s], recs[s]);
            try {
                StageChain<MirrorApi, DescSink> chain(factory, streams[s], events + streams[s].first_event, sink);
                std::vector<StageChain<MirrorApi, DescSink>::Starvation> starved;
                chain.SetStarvationLog(&starved);
                const int rc = chain.Run();
                const uint32_t jps = Jiffies::PerSampleOrZero(streams[s].sample_rate);
                for (const auto& st : starved) {
                    ohp_starvation o;
                    o.stream = s;
                    o.pcm_jiffies = st.pcmJiffies;
                    o.event = streams[s].first_event + st.event;
                    o.ramp = st.ramp;
                    o.plays = st.plays;
                    o.recent_jiffies = st.recentJiffies;
                    o.attenuation = st.attenuation;
                    o.reserved = 0;
                    recs[s].starvations.push_back(o);
                    for (const auto& piece : st.recent) {
                        ohp_recent_audio a;
                        a.pcm_jiffies = piece.pcmJiffies;
                        a.jiffies = piece.jiffies;
                        a.silence = piece.silence;
                        a.attenuation = piece.attenuation;
                        a.reserved = 0;
                        recs[s].recent.push_back(a);
                    }
                    recs[s].recentCount.push_back(st.recent.size());
                }
                if (rc != 0) {
                    rcs[(size_t)t] = OHP_E_INVALID_ARG;
                    errs[(size_t)t] = "stream " + std::to_string(s) + ": spec not representable";
                    return;
                }
            }
            catch (const std::exception& e) {
                // the reference would ASSERT here
                rcs[(size_t)t] = OHP_E_INVALID_DESC;
                errs[(size_t)t] = "stream " + std::to_string(s) + ": " + e.what();
                return;
            }
        }
    };
    if (threads == 1) {
        worker(0);
    }
    else {
        std::vector<std::thread> pool;
        for (int t = 0; t < threads; t++) pool.emplace_back(worker, t);
        for (auto& th : pool) th.join();
    }
    for (size_t t = 0; t < (size_t)threads; t++) {
        if (rcs[t] != 0) {
            g_error = errs[t];
            return rcs[t];
        }
    }
    ohp_schedule* sch = new ohp_schedule();
    size_t total = 0;
    for (auto& r : recs) total += r.chunks.size();
    sch->chunks.reserve(total);
    sch->info.reserve(total);
    sch->chunkBegin.resize(n_streams + 1);
    sch->outBytes.resize(n_streams);
    for (size_t s = 0; s < n_streams; s++) {
        sch->chunkBegin[s] = sch->chunks.size();
        sch->outBytes[s] = recs[s].outBytes;
        sch->chunks.insert(sch->chunks.end(), recs[s].chunks.begin(), recs[s].chunks.end());
        sch->info.insert(sch->info.end(), recs[s].info.begin(), recs[s].info.end());
        sch->starvations.insert(sch->starvations.end(), recs[s].starvations.begin(), recs[s].starvations.end());
        for (const uint64_t n : recs[s].recentCount) sch->recentBegin.push_back(sch->recentBegin.back() + n);
        sch->recent.insert(sch->recent.end(), recs[s].recent.begin(), recs[s].recent.end());
        std::vector<ohp_chunk_desc>().swap(recs[s].chunks);
        std::vector<ohp_chunk_info>().swap(recs[s].info);
    }
    sch->chunkBegin[n_streams] = sch->chunks.size();
    *out = sch;
    return OHP_OK;
}

// The class-free walk (schedule_walk.h) on host threads: the same source the GPU schedule kernels compile, so the CPU
// suite can pin it against the class-based model above (and against the reference's playables) without a GPU.
int ohp_schedule_build_walk(const ohp_stream_spec* streams, size_t n_streams, const ohp_ramp_event* events, size_t n_events,
                            int threads, ohp_schedule** out)
{
    if (!out || (!streams && n_streams) || (!events && n_events)) {
        g_error = "null argument";
        return OHP_E_INVALID_ARG;
    }
    *out = nullptr;
    if (threads <= 0) threads = (int)std::thread::hardware_concurrency();
    if (threads <= 0) threads = 1;
    if ((size_t)threads > n_streams) threads = (int)(n_streams ? n_streams : 1);
    ohp_schedule* sch = new ohp_schedule();
    sch->chunkBegin.assign(n_streams + 1, 0);
    sch->outBytes.assign(n_streams, 0);
    std::vector<uint32_t> rcs(n_streams, 0);
    std::vector<std::vector<ohp_starvation>> starved(n_streams); // the emitting walk's records, stream by stream
    auto run = [&](bool emit) {
        auto worker = [&](int t) {
            const size_t lo = n_streams * (size_t)t / (size_t)threads;
            const size_t hi = n_streams * (size_t)(t + 1) / (size_t)threads;
            for (size_t s = lo; s < hi; s++) {
                uint64_t n = 0, bytes = 0;
                if (emit) {
                    starved[s].resize(streams[s].num_events);
                    uint32_t nRec = 0;
                    rcs[s] = sched::run_stream<true, 1, true, true>(streams[s], events, n_events, sch->chunks.data() + sch->chunkBegin[s],
                                                                    sch->info.data() + sch->chunkBegin[s], n, bytes, 0, ~0ull,
                                                                    starved[s].data(), s, true, &nRec);
                    starved[s].resize(nRec);
                }
                else {
                    rcs[s] = sched::run_stream<false>(streams[s], events, n_events, nullptr, nullptr, n, bytes);
                    sch->chunkBegin[s + 1] = n; // scanned below
                    sch->outBytes[s] = bytes;
                }
            }
        };
        if (threads == 1) {
            worker(0);
        }
        else {
            std::vector<std::thread> pool;
            for (int t = 0; t < threads; t++) pool.emplace_back(worker, t);
            for (auto& th : pool) th.join();
        }
    };
    run(false);
    for (size_t s = 0; s < n_streams; s++) {
        if (rcs[s] != sched::kOk) {
            g_error = "stream " + std::to_string(s) + (rcs[s] == sched::kErrAssert ? ": the reference would ASSERT on this schedule"
                                                        : rcs[s] == sched::kErrSpec ? ": spec not representable"
                                                                                    : ": too many pending message splits");
            const int rc = rcs[s] == sched::kErrAssert ? OHP_E_INVALID_DESC : (rcs[s] == sched::kErrSpec ? OHP_E_INVALID_ARG : OHP_E_NO_MEMORY);
            delete sch;
            return rc;
        }
    }
    for (size_t s = 0; s < n_streams; s++) sch->chunkBegin[s + 1] += sch->chunkBegin[s];
    sch->chunks.resize(sch->chunkBegin[n_streams]);
    sch->info.resize(sch->chunkBegin[n_streams]);
    run(true);
    for (size_t s = 0; s < n_streams; s++) {
        sch->starvations.insert(sch->starvations.end(), starved[s].begin(), starved[s].end());
    }
    sch->recentBegin.assign(sch->starvations.size() + 1, 0); // records without the recent audio's pieces
    *out = sch;
    return OHP_OK;
}

int ohp_schedule_chunk_bounds(const ohp_stream_spec* streams, size_t n_streams,
                              const ohp_ramp_event* events, size_t n_events, uint64_t* bounds)
{
    if ((n_streams && (!streams || !bounds)) || (n_events && !events)) return OHP_E_INVALID_ARG;
    for (size_t s = 0; s < n_streams; s++) bounds[s] = ohp::sched::stream_chunk_bound(streams[s], events, n_events);
    return OHP_OK;
}

size_t ohp_schedule_num_chunks(const ohp_schedule* s) { return s ? s->chunks.size() : 0; }
const ohp_chunk_desc* ohp_schedule_chunks(const ohp_schedule* s) { return s ? s->chunks.data() : nullptr; }
const ohp_chunk_info* ohp_schedule_chunk_info(const ohp_schedule* s) { return s ? s->info.data() : nullptr; }
const uint64_t* ohp_schedule_stream_chunk_begin(const ohp_schedule* s) { return s ? s->chunkBegin.data() : nullptr; }
const uint64_t* ohp_schedule_stream_out_bytes(const ohp_schedule* s) { return s ? s->outBytes.data() : nullptr; }
const ohp_recent_audio* ohp_schedule_recent_audio(const ohp_schedule* s) { return s ? s->recent.data() : nullptr; }
const uint64_t* ohp_schedule_recent_begin(const ohp_schedule* s) { return s ? s->recentBegin.data() : nullptr; }
size_t ohp_schedule_num_starvations(const ohp_schedule* s) { return s ? s->starvations.size() : 0; }
const ohp_starvation* ohp_schedule_starvations(const ohp_schedule* s) { return s ? s->starvations.data() : nullptr; }
const char* ohp_schedule_last_error(void) { return g_error.c_str(); }
void ohp_schedule_free(ohp_schedule* s) { delete s; }

int ohp_flywheel_plan(const ohp_stream_spec* stream, const ohp_starvation* starvation,
                      uint64_t training_off, uint64_t generated_off, uint64_t out_off,
                      ohp_chunk_desc* prep, size_t* n_prep, ohp_flywheel_job* job, ohp_chunk_desc* blocks, size_t cap, size_t* n_blocks)
{
    if (!stream || !starvation || !prep || !n_prep || !job || (!blocks && cap) || !n_blocks) return OHP_E_INVALID_ARG;
    *n_blocks = 0;
    *n_prep = 0;
    const uint32_t jps = Jiffies::PerSampleOrZero(stream->sample_rate);
    const uint32_t B = stream->bit_depth / 8u;
    const uint32_t C = stream->channels;
    const uint32_t frameBytes = C * B;
    if (jps == 0 || frameBytes == 0 || !(stream->bit_depth == 8 || stream->bit_depth == 16 || stream->bit_depth == 24 || stream->bit_depth == 32)) {
        g_error = "flywheel plan: spec not representable";
        return OHP_E_INVALID_ARG;
    }
    if (C > OHP_FLYWHEEL_MAX_CHANNELS) {
        g_error = "flywheel plan: more channels than FlywheelRamperManager takes";
        return OHP_E_INVALID_DESC;
    }
    if (!starvation->plays) {
        g_error = "flywheel plan: this starvation plays nothing (the element was halted, muted or had not become audible)";
        return OHP_E_INVALID_ARG;
    }
    if (starvation->recent_jiffies < OHP_FLYWHEEL_TRAINING_JIFFIES || starvation->pcm_jiffies < OHP_FLYWHEEL_TRAINING_JIFFIES) {
        g_error = "flywheel plan: the last 1 ms the element played is not PCM of one attenuation throughout (silence or padding in the training block: not planned)";
        return OHP_E_INVALID_ARG;
    }
    // StarvationRamper::StartFlywheelRamp (StarvationRamper.cpp:491-536) cuts the recent audio to its last kTrainingJiffies;
    // MsgAudioPcm::CreatePlayable rounds both ends of every message down to a sample (Msg.cpp:2234-2243): the frames read are
    const uint64_t lastFrame = starvation->pcm_jiffies / jps;                                     // one past the last
    const uint64_t firstFrame = (starvation->pcm_jiffies - OHP_FLYWHEEL_TRAINING_JIFFIES) / jps;
    const uint32_t got = (uint32_t)(lastFrame - firstFrame);
    // ... and FlywheelInput::Prepare lays its planes out for Jiffies::ToSamples(kTrainingJiffies) of them (:90-98)
    const uint32_t train = OHP_FLYWHEEL_TRAINING_JIFFIES / jps;
    if (lastFrame > stream->total_frames || (got != train && got != train + 1) || train < 2) {
        g_error = "flywheel plan: starvation record does not fit the stream";
        return OHP_E_INVALID_ARG;
    }
    {
        // what ohp_flywheel_validate / the flywheel kernel refuse (csrc/ohp_flywheel_kernels.cuh, check_job): the reference's
        // fixed buffers -- FlywheelInput's 7680 bytes (StarvationRamper.cpp:76-83), RampGenerator's 6144 (:215-219) -- and
        // Burg's method wanting more samples than its degree (FlywheelRamper.cpp:180-195)
        const uint32_t decimation = (stream->sample_rate == 192000u || stream->sample_rate == 176400u) ? 4u
                                  : (stream->sample_rate == 88200u || stream->sample_rate == 96000u) ? 2u : 1u; // FlywheelRamper.cpp:330-345
        const uint32_t blockFrames = OHP_FLYWHEEL_BLOCK_JIFFIES / jps;
        if (train / decimation < OHP_FLYWHEEL_DEGREE + 1u || train * 4u * C > OHP_FLYWHEEL_MAX_INPUT_BYTES
            || blockFrames * frameBytes > OHP_FLYWHEEL_MAX_BLOCK_BYTES) {
            g_error = "flywheel plan: a rate / channel count / depth the reference's flywheel buffers do not hold";
            return OHP_E_INVALID_DESC;
        }
    }
    const uint8_t flags = (uint8_t)((stream->in_little_endian && B > 1) ? OHP_F_IN_LITTLE_ENDIAN : 0);
    auto planar = [&](uint64_t aSrc, uint64_t aDstSlot, uint32_t aBytes, uint32_t aChannels) {
        // FlywheelPlayableCreator clears the messages' ramps, not their attenuation (:61-74)
        ohp_chunk_desc& d = prep[(*n_prep)++];
        std::memset(&d, 0, sizeof d);
        d.src_off = aSrc;
        d.dst_off = training_off + aDstSlot * 4u;
        d.bytes = aBytes;
        d.ramp_start = (uint16_t)Ramp::kMax;
        d.ramp_end = (uint16_t)Ramp::kMax;
        d.attenuation = starvation->attenuation;
        d.bit_depth = (uint8_t)stream->bit_depth;
        d.channels = (uint8_t)aChannels;
        d.flags = flags;
        d.out_fmt = OHP_OUT_PLANAR32_BE;
        d.aux = (uint16_t)train;
    };
    const uint64_t src = stream->src_base + firstFrame * frameBytes;
    if (got == train || C == 1) {
        // mono with a frame too many: the plane's last subsample falls beyond the block (DoProcessFragment, :158-186)
        planar(src, 0, train * frameBytes, C);
    }
    else {
        // train + 1 frames into planes of train slots: channel c's last subsample is written, last of all, where channel
        // c + 1's first went; the last channel's falls beyond the block
        planar(src + frameBytes, 1, (train - 1) * frameBytes, C);
        planar(src, 0, B, 1);
        for (uint32_t c = 1; c < C; c++) {
            planar(src + (uint64_t)train * frameBytes + (c - 1) * B, (uint64_t)c * train, B, 1);
        }
    }
    // FlywheelRamperManager::Ramp for this stream: 20 ms from the 1 ms block (StarvationRamper.cpp:374-375, 422)
    std::memset(job, 0, sizeof *job);
    job->src_off = training_off;
    job->dst_off = generated_off;
    job->sample_rate = stream->sample_rate;
    job->out_frames = OHP_FLYWHEEL_RAMP_JIFFIES / jps;
    job->train_frames = (uint16_t)train;
    job->channels = (uint8_t)C;
    job->bit_depth = (uint8_t)stream->bit_depth;
    // RampGenerator plays it from the element's ramp value down (StarvationRamper.cpp:526-531)
    const int n = ohp_flywheel_ramp_chunks(job, starvation->ramp, generated_off, out_off, blocks, cap, nullptr);
    if (n < 0) return -n;
    *n_blocks = (size_t)n;
    return OHP_OK;
}

int ohp_flywheel_plan_recent(const ohp_stream_spec* stream, const ohp_starvation* starvation,
                             const ohp_recent_audio* recent, size_t n_recent,
                             uint64_t training_off, uint64_t generated_off, uint64_t out_off,
                             ohp_chunk_desc* prep, size_t prep_cap, size_t* n_prep, ohp_flywheel_job* job,
                             ohp_chunk_desc* blocks, size_t cap, size_t* n_blocks)
{
    if (!stream || !starvation || (!recent && n_recent) || !prep || !n_prep || !job || (!blocks && cap) || !n_blocks) return OHP_E_INVALID_ARG;
    *n_blocks = 0;
    *n_prep = 0;
    const uint32_t jps = Jiffies::PerSampleOrZero(stream->sample_rate);
    const uint32_t B = stream->bit_depth / 8u;
    const uint32_t C = stream->channels;
    const uint32_t frameBytes = C * B;
    if (jps == 0 || frameBytes == 0 || !(stream->bit_depth == 8 || stream->bit_depth == 16 || stream->bit_depth == 24 || stream->bit_depth == 32)) {
        g_error = "flywheel plan: spec not representable";
        return OHP_E_INVALID_ARG;
    }
    if (C > OHP_FLYWHEEL_MAX_CHANNELS) {
        g_error = "flywheel plan: more channels than FlywheelRamperManager takes";
        return OHP_E_INVALID_DESC;
    }
    if (!starvation->plays) {
        g_error = "flywheel plan: this starvation plays nothing (the element was halted, muted or had not become audible)";
        return OHP_E_INVALID_ARG;
    }
    const uint32_t train = OHP_FLYWHEEL_TRAINING_JIFFIES / jps;
    {
        const uint32_t decimation = (stream->sample_rate == 192000u || stream->sample_rate == 176400u) ? 4u
                                  : (stream->sample_rate == 88200u || stream->sample_rate == 96000u) ? 2u : 1u;
        const uint32_t blockFrames = OHP_FLYWHEEL_BLOCK_JIFFIES / jps;
        if (train < 2 || train / decimation < OHP_FLYWHEEL_DEGREE + 1u || train * 4u * C > OHP_FLYWHEEL_MAX_INPUT_BYTES
            || blockFrames * frameBytes > OHP_FLYWHEEL_MAX_BLOCK_BYTES) {
            g_error = "flywheel plan: a rate / channel count / depth the reference's flywheel buffers do not hold";
            return OHP_E_INVALID_DESC;
        }
    }
    // StartFlywheelRamp's cut (StarvationRamper.cpp:495-507): whole pieces go from the front while more than kTrainingJiffies
    // is left, the piece under the cut is split
    uint64_t total = 0;
    for (size_t i = 0; i < n_recent; i++) total += recent[i].jiffies;
    if (total < OHP_FLYWHEEL_TRAINING_JIFFIES) {
        g_error = "flywheel plan: less than 1 ms since the element's recent audio was emptied (the reference pads with silence: not planned)";
        return OHP_E_INVALID_ARG;
    }
    uint64_t excess = total - OHP_FLYWHEEL_TRAINING_JIFFIES;
    size_t first = 0;
    ohp_recent_audio head = {0, 0, 0, 0, 0};
    while (first < n_recent) {
        head = recent[first];
        if (excess == 0) break;
        if (head.jiffies > excess) {
            if (head.silence && excess % jps != 0) {
                // MsgSilence::SplitCompleted keeps the whole samples in front (Msg.cpp:2530-2535): less goes than was asked
                // for, the loop comes round with under a sample of excess and splits off messages of zero jiffies for ever
                g_error = "flywheel plan: a MsgSilence under the cut at a jiffy count that is not a whole sample: the reference does not return from this starvation";
                return OHP_E_INVALID_DESC;
            }
            head.jiffies -= (uint32_t)excess;
            if (!head.silence) head.pcm_jiffies += excess;
            excess = 0;
            break;
        }
        excess -= head.jiffies;
        first++;
    }
    // FlywheelInput::Prepare (:90-111): every piece through CreatePlayable -- both ends of a MsgAudioPcm rounded down to a
    // sample (Msg.cpp:2234-2243), a MsgSilence whole samples by construction -- frames in the order they are read
    struct Run { bool silence; uint64_t firstFrame; uint32_t frames; uint32_t attenuation; };
    std::vector<Run> runs;
    uint64_t got = 0;
    for (size_t i = first; i < n_recent; i++) {
        const ohp_recent_audio& p = (i == first) ? head : recent[i];
        Run r;
        r.silence = p.silence != 0;
        r.attenuation = p.silence ? OHP_UNITY_ATTENUATION : p.attenuation;
        if (p.silence) {
            r.firstFrame = 0;
            r.frames = p.jiffies / jps;
        }
        else {
            r.firstFrame = p.pcm_jiffies / jps;
            r.frames = (uint32_t)((p.pcm_jiffies + p.jiffies) / jps - r.firstFrame);
            if ((p.pcm_jiffies + p.jiffies) / jps > stream->total_frames) {
                g_error = "flywheel plan: a piece of recent audio outside the stream";
                return OHP_E_INVALID_ARG;
            }
        }
        if (r.frames == 0) continue;
        got += r.frames;
        runs.push_back(r);
    }
    if (got < train) {
        g_error = "flywheel plan: the pieces give FlywheelInput fewer frames than its planes have (the rest would be what an earlier starvation left there)";
        return OHP_E_INVALID_ARG;
    }
    if (got > (uint64_t)train + 1u) {
        g_error = "flywheel plan: recent audio does not fit a starvation record";
        return OHP_E_INVALID_ARG;
    }
    const uint8_t le = (uint8_t)((stream->in_little_endian && B > 1) ? OHP_F_IN_LITTLE_ENDIAN : 0);
    bool full = false;
    // frames [aFrom, aFrom + aCount) of run r, channels [aCh, aCh + aChannels), to slot aSlot of plane aCh and on
    auto emit = [&](const Run& r, uint32_t aFrom, uint32_t aCount, uint32_t aCh, uint32_t aChannels, uint64_t aSlot) {
        if (*n_prep == prep_cap) { full = true; return; }
        ohp_chunk_desc& d = prep[(*n_prep)++];
        std::memset(&d, 0, sizeof d);
        d.src_off = r.silence ? 0 : stream->src_base + (r.firstFrame + aFrom) * frameBytes + (uint64_t)aCh * B;
        d.dst_off = training_off + aSlot * 4u;
        d.bytes = aCount * aChannels * B;
        d.ramp_start = (uint16_t)Ramp::kMax;
        d.ramp_end = (uint16_t)Ramp::kMax;
        d.attenuation = (uint16_t)r.attenuation;
        d.bit_depth = (uint8_t)stream->bit_depth;
        d.channels = (uint8_t)aChannels;
        d.flags = (uint8_t)(r.silence ? OHP_F_SILENCE : le);
        d.out_fmt = OHP_OUT_PLANAR32_BE;
        d.aux = (uint16_t)train;
    };
    // which frames go out whole: all of them; or, with a frame too many and more than one channel, frames 1 .. train - 1
    // (every plane's first slot is written last by another frame: DoProcessFragment, :158-186); mono: frames 0 .. train - 1
    const bool over = got == (uint64_t)train + 1u;
    const uint64_t lo = (over && C > 1) ? 1 : 0, hi = train; // [lo, hi) in frames read
    uint64_t at = 0;
    const Run* firstRun = nullptr;
    const Run* lastRun = nullptr;
    for (const Run& r : runs) {
        if (firstRun == nullptr) firstRun = &r;
        lastRun = &r;
        const uint64_t a = at > lo ? at : lo, b = (at + r.frames) < hi ? (at + r.frames) : hi;
        if (b > a) emit(r, (uint32_t)(a - at), (uint32_t)(b - a), 0, C, a);
        at += r.frames;
    }
    if (over && C > 1) {
        emit(*firstRun, 0, 1, 0, 1, 0); // plane 0 keeps frame 0's subsample
        for (uint32_t c = 1; c < C; c++) emit(*lastRun, lastRun->frames - 1, 1, c - 1, 1, (uint64_t)c * train); // the last frame's, one plane on
    }
    if (full) {
        g_error = "flywheel plan: more descriptors than prep_cap";
        return OHP_E_INVALID_ARG;
    }
    std::memset(job, 0, sizeof *job);
    job->src_off = training_off;
    job->dst_off = generated_off;
    job->sample_rate = stream->sample_rate;
    job->out_frames = OHP_FLYWHEEL_RAMP_JIFFIES / jps;
    job->train_frames = (uint16_t)train;
    job->channels = (uint8_t)C;
    job->bit_depth = (uint8_t)stream->bit_depth;
    const int n = ohp_flywheel_ramp_chunks(job, starvation->ramp, generated_off, out_off, blocks, cap, nullptr);
    if (n < 0) return -n;
    *n_blocks = (size_t)n;
    return OHP_OK;
}

static int plan_batch(const ohp_stream_spec* streams, size_t n_streams, const ohp_starvation* starvations, size_t n_starvations,
                      const ohp_recent_audio* recent, const uint64_t* recent_begin,
                      uint64_t training_base, uint64_t generated_base, uint64_t out_base, ohp_flywheel_batch** out);

int ohp_flywheel_plan_batch(const ohp_stream_spec* streams, size_t n_streams, const ohp_starvation* starvations, size_t n_starvations,
                            uint64_t training_base, uint64_t generated_base, uint64_t out_base, ohp_flywheel_batch** out)
{
    return plan_batch(streams, n_streams, starvations, n_starvations, nullptr, nullptr, training_base, generated_base, out_base, out);
}

int ohp_flywheel_plan_batch_recent(const ohp_stream_spec* streams, size_t n_streams, const ohp_starvation* starvations, size_t n_starvations,
                                   const ohp_recent_audio* recent, const uint64_t* recent_begin,
                                   uint64_t training_base, uint64_t generated_base, uint64_t out_base, ohp_flywheel_batch** out)
{
    if (!recent_begin || (!recent && n_starvations && recent_begin[n_starvations] != 0)) return OHP_E_INVALID_ARG;
    return plan_batch(streams, n_streams, starvations, n_starvations, recent, recent_begin, training_base, generated_base, out_base, out);
}

static int plan_batch(const ohp_stream_spec* streams, size_t n_streams, const ohp_starvation* starvations, size_t n_starvations,
                      const ohp_recent_audio* recent, const uint64_t* recent_begin,
                      uint64_t training_base, uint64_t generated_base, uint64_t out_base, ohp_flywheel_batch** out)
{
    if (!out) return OHP_E_INVALID_ARG;
    *out = nullptr;
    if ((!streams && n_streams) || (!starvations && n_starvations) || n_starvations > 0xffffffffull) return OHP_E_INVALID_ARG;
    std::unique_ptr<ohp_flywheel_batch> b(new (std::nothrow) ohp_flywheel_batch());
    if (!b) return OHP_E_NO_MEMORY;
    auto align16 = [](uint64_t x) { return (x + 15u) & ~(uint64_t)15u; };
    uint64_t training = align16(training_base), generated = align16(generated_base), played = align16(out_base);
    for (size_t k = 0; k < n_starvations; k++) {
        const ohp_starvation& sv = starvations[k];
        if (sv.stream >= n_streams) {
            g_error = "flywheel plan: starvation " + std::to_string(k) + " names a stream outside the batch";
            return OHP_E_INVALID_ARG;
        }
        const ohp_stream_spec& sp = streams[sv.stream];
        ohp_chunk_desc prep[OHP_FLYWHEEL_MAX_PREP_RECENT];
        ohp_chunk_desc blocks[OHP_FLYWHEEL_RAMP_JIFFIES / OHP_FLYWHEEL_BLOCK_JIFFIES + 1];
        ohp_flywheel_job job;
        size_t n_prep = 0, n_blocks = 0;
        const int rc = recent_begin
            ? ohp_flywheel_plan_recent(&sp, &sv, recent + recent_begin[k], (size_t)(recent_begin[k + 1] - recent_begin[k]), training, generated,
                                       played, prep, sizeof prep / sizeof prep[0], &n_prep, &job, blocks, sizeof blocks / sizeof blocks[0], &n_blocks)
            : ohp_flywheel_plan(&sp, &sv, training, generated, played, prep, &n_prep, &job, blocks,
                                sizeof blocks / sizeof blocks[0], &n_blocks);
        if (rc == OHP_E_INVALID_ARG || rc == OHP_E_INVALID_DESC) continue; // plays nothing / not planned / the reference ASSERTs
        if (rc != OHP_OK) return rc;
        const uint64_t frame_bytes = (uint64_t)sp.channels * (sp.bit_depth / 8u);
        const uint64_t out_len = (uint64_t)job.out_frames * frame_bytes;
        b->planned.push_back((uint32_t)k);
        b->outOff.push_back(played);
        b->outLen.push_back(out_len);
        b->prep.insert(b->prep.end(), prep, prep + n_prep);
        b->jobs.push_back(job);
        b->blocks.insert(b->blocks.end(), blocks, blocks + n_blocks);
        training = align16(training + (uint64_t)job.train_frames * 4u * sp.channels);
        generated = align16(generated + out_len);
        played = align16(played + out_len);
    }
    b->arena[0] = training; b->arena[1] = generated; b->arena[2] = played;
    *out = b.release();
    return OHP_OK;
}

size_t ohp_flywheel_batch_num_planned(const ohp_flywheel_batch* b) { return b ? b->planned.size() : 0; }
const uint32_t* ohp_flywheel_batch_planned(const ohp_flywheel_batch* b) { return b ? b->planned.data() : nullptr; }
const uint64_t* ohp_flywheel_batch_out_off(const ohp_flywheel_batch* b) { return b ? b->outOff.data() : nullptr; }
const uint64_t* ohp_flywheel_batch_out_len(const ohp_flywheel_batch* b) { return b ? b->outLen.data() : nullptr; }
size_t ohp_flywheel_batch_num_prep(const ohp_flywheel_batch* b) { return b ? b->prep.size() : 0; }
const ohp_chunk_desc* ohp_flywheel_batch_prep(const ohp_flywheel_batch* b) { return b ? b->prep.data() : nullptr; }
const ohp_flywheel_job* ohp_flywheel_batch_jobs(const ohp_flywheel_batch* b) { return b ? b->jobs.data() : nullptr; }
size_t ohp_flywheel_batch_num_blocks(const ohp_flywheel_batch* b) { return b ? b->blocks.size() : 0; }
const ohp_chunk_desc* ohp_flywheel_batch_blocks(const ohp_flywheel_batch* b) { return b ? b->blocks.data() : nullptr; }
void ohp_flywheel_batch_arena_bytes(const ohp_flywheel_batch* b, uint64_t sizes[3])
{
    for (int i = 0; i < 3; i++) sizes[i] = b ? b->arena[i] : 0;
}
void ohp_flywheel_batch_free(ohp_flywheel_batch* b) { delete b; }

int ohp_flywheel_ramp_chunks(const ohp_flywheel_job* job, uint32_t current_ramp, uint64_t src_off, uint64_t dst_off,
                             ohp_chunk_desc* out, size_t cap, uint32_t* final_ramp)
{
    if (!job || (!out && cap)) return -OHP_E_INVALID_ARG;
    try {
        // RampGenerator::Start (StarvationRamper.cpp:235-247)
        const uint32_t jps = Jiffies::PerSample(job->sample_rate);
        const uint32_t frameBytes = job->channels * (job->bit_depth / 8u);
        const uint32_t blockFrames = OHP_FLYWHEEL_BLOCK_JIFFIES / jps;
        uint32_t remainingRamp = jps * job->out_frames;
        uint32_t remaining = job->out_frames;
        MsgFactory factory;
        size_t n = 0;
        while (remaining > 0) {
            const uint32_t frames = remaining > blockFrames ? blockFrames : remaining;
            remaining -= frames;
            if (n == cap) return -OHP_E_NO_MEMORY;
            // RampGenerator::EndBlock (StarvationRamper.cpp:351-364)
            MsgAudioPcm* audio = factory.CreateMsgAudioPcm(src_off, frames * frameBytes, job->channels, job->sample_rate,
                                                           job->bit_depth, AudioDataEndian::Big, MsgAudioPcm::kTrackOffsetInvalid);
            if (current_ramp == Ramp::kMin) {
                audio->SetMuted();
            }
            else {
                MsgAudio* split = nullptr;
                current_ramp = audio->SetRamp(current_ramp, remainingRamp, Ramp::EDown, split);
                if (split != nullptr) {
                    split->RemoveRef();
                    audio->RemoveRef();
                    OHP_ASSERT(false); // ASSERT(split == nullptr), StarvationRamper.cpp:359
                }
            }
            MsgPlayable* playable = audio->CreatePlayable();
            out[n++] = playable->Descriptor(dst_off, OHP_OUT_PACKED_BE);
            src_off += playable->Bytes();
            dst_off += playable->Bytes();
            playable->RemoveRef();
        }
        if (final_ramp) *final_ramp = current_ramp;
        return (int)n;
    }
    catch (const std::exception& e) {
        g_error = e.what();
        return -OHP_E_INVALID_DESC;
    }
}

uint32_t ohp_jiffies_per_sample(uint32_t sample_rate) { return Jiffies::PerSampleOrZero(sample_rate); }

int ohp_ramp_set(ohp_ramp* ramp, uint32_t start, uint32_t fragment_size, uint32_t remaining_duration, uint32_t direction,
                 ohp_ramp* split, uint32_t* split_pos)
{
    if (!ramp || !split || !split_pos) return -2;
    Ramp r = Ramp::FromAbi(*ramp);
    Ramp s;
    try {
        const bool ret = r.Set(start, fragment_size, remaining_duration, (Ramp::EDirection)direction, s, *split_pos);
        *ramp = r.ToAbi();
        *split = s.ToAbi();
        return ret ? 1 : 0;
    }
    catch (const AssertionFailed&) {
        return -1;
    }
}

int ohp_ramp_split(ohp_ramp* ramp, uint32_t new_size, uint32_t current_size, ohp_ramp* remaining)
{
    if (!ramp || !remaining) return -2;
    Ramp r = Ramp::FromAbi(*ramp);
    try {
        const Ramp rest = r.Split(new_size, current_size);
        *ramp = r.ToAbi();
        *remaining = rest.ToAbi();
        return 0;
    }
    catch (const AssertionFailed&) {
        return -1;
    }
}

} // extern "C"
