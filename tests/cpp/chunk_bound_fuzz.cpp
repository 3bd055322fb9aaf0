// sched::stream_chunk_bound -- the closed form that sizes ohp_run_streams_device's descriptor regions -- against the exact
// playables of run_stream<false>, the walk the device compiles.  Built and driven by tests/test_chunk_bound.py.
//
//   chunk_bound_fuzz fuzz <seed> <streams>   random streams, one at a time: every op, four stages, caps from one sample
//                                            up, codec reads, driver blocks, silence.  Prints a summary line, what it
//                                            covered, and every stream the bound does not cover.
//   chunk_bound_fuzz file <path>             the batches of <path> (u32 streams, u32 events, specs, events; repeated):
//                                            "status exact bound" per stream.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "../../ohpipeline_b200/host/schedule_walk.h"

using namespace ohp;

namespace {

struct Rng
{
    uint64_t s;
    uint64_t next()
    {
        uint64_t z = (s += 0x9E3779B97F4A7C15ull);
        z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
        z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
        return z ^ (z >> 31);
    }
    uint64_t below(uint64_t n) { return n ? next() % n : 0; }
    uint64_t in(uint64_t lo, uint64_t hi) { return lo + below(hi - lo + 1); } // [lo, hi]
    bool chance(unsigned percent) { return below(100) < percent; }
};

const uint32_t kRates[] = {7350, 8000, 11025, 12000, 14700, 16000, 22050, 24000, 29400, 32000,
                           44100, 48000, 88200, 96000, 176400, 192000, 352800, 384000};

// What a stage is for the whole stream: bare ramps (ops 1-4), or one of the reference's elements (ops 8-12).
enum Kind { kBare, kRamper, kMuter, kStarvation };

// A duration: a sample or less, a few samples, a message or so, or longer than the stream.
uint32_t duration(Rng& r, uint32_t jps, uint64_t msg_j, uint64_t total_j)
{
    switch (r.below(5)) {
    case 0: return (uint32_t)r.in(1, jps);
    case 1: return (uint32_t)(jps * r.in(1, 8) + r.below(jps));
    case 2: return (uint32_t)r.in(1, msg_j * 3 + 1);
    case 3: return (uint32_t)r.in(1, total_j + 1 < 0xffffffffull ? total_j + 1 : 0xffffffffull);
    default: return (uint32_t)(OHP_JIFFIES_PER_MS * r.in(1, 60));
    }
}

void random_stream(Rng& r, ohp_stream_spec& sp, std::vector<ohp_ramp_event>& ev)
{
    std::memset(&sp, 0, sizeof sp);
    sp.sample_rate = kRates[r.below(18)];
    sp.bit_depth = 8u * (uint32_t)r.in(1, 4);
    sp.channels = r.chance(90) ? (uint32_t)r.in(1, 8) : (uint32_t)r.in(9, 32);
    sp.in_little_endian = (uint32_t)r.below(2);
    sp.out_fmt = r.chance(50) ? OHP_OUT_PACKED_BE : OHP_OUT_PACKED_LE;
    const uint32_t fb = sp.channels * (sp.bit_depth / 8u);
    const uint32_t max_chunk = OHP_MAX_PCM_CHUNK_BYTES / fb;
    const uint32_t jps = core::jiffies_per_sample_or_zero(sp.sample_rate);
    sp.chunk_frames = (uint32_t)(r.chance(30) ? r.in(1, 8) : r.in(1, max_chunk));
    sp.total_frames = r.chance(5) ? r.below(3) : (r.chance(80) ? r.in(1, 3000) : r.in(3000, 20000));
    if (r.chance(35)) sp.codec_read_frames = (uint32_t)(r.chance(50) ? max_chunk : r.in(1, max_chunk));
    if (r.chance(35)) sp.driver_block_frames = (uint32_t)(r.chance(30) ? r.in(1, 4) : r.in(1, 2000));
    const uint64_t total_j = sp.total_frames * jps, msg_j = (uint64_t)sp.chunk_frames * jps;
    Kind kind[sched::kStages];
    for (int i = 0; i < sched::kStages; i++) kind[i] = (Kind)r.below(4);
    bool muted[sched::kStages] = {};
    const uint32_t n = (uint32_t)(r.chance(10) ? 0 : r.in(1, r.chance(20) ? 40 : 12));
    ev.clear();
    for (uint32_t k = 0; k < n; k++) {
        ohp_ramp_event e{};
        e.stage = (uint32_t)r.below(sched::kStages);
        // positions: anywhere, on a sample, on a message boundary, at either end
        const uint64_t span = total_j + total_j / 4 + 1;
        switch (r.below(4)) {
        case 0: e.at_jiffies = r.below(span); break;
        case 1: e.at_jiffies = r.below(span) / jps * jps; break;
        case 2: e.at_jiffies = msg_j ? r.below(span) / msg_j * msg_j : 0; break;
        default: e.at_jiffies = r.chance(50) ? 0 : total_j; break;
        }
        const uint32_t what = (uint32_t)r.below(10);
        if (what == 0) {
            e.op = OHP_EV_INSERT_SILENCE;
            e.stage = 0;
            e.at_jiffies = e.at_jiffies / jps * jps;
            e.arg = r.chance(60) ? jps * (uint32_t)r.in(1, 2000) : (uint32_t)r.in(1, 3 * OHP_JIFFIES_PER_MS);
        }
        else if (what == 1) {
            e.op = OHP_EV_MAX_MSG_JIFFIES; // caps from one sample up
            e.arg = r.chance(40) ? jps * (uint32_t)r.in(1, 4) : (uint32_t)r.in(jps, (uint64_t)jps * 3000);
        }
        else if (what == 2) {
            e.op = OHP_EV_SET_ATTENUATION;
            e.arg = (uint32_t)r.below(512);
        }
        else {
            switch (kind[e.stage]) {
            case kBare: {
                const uint32_t op = (uint32_t)r.in(1, 4);
                e.op = op;
                if (op <= 2) e.arg = duration(r, jps, msg_j, total_j);
                break;
            }
            case kRamper:
                e.op = r.chance(75) ? OHP_EV_RAMPER_STREAM : OHP_EV_HALT;
                if (e.op == OHP_EV_RAMPER_STREAM && r.chance(80)) e.arg = duration(r, jps, msg_j, total_j);
                break;
            case kMuter:
                if (r.chance(20)) { e.op = OHP_EV_HALT; break; }
                e.op = muted[e.stage] ? OHP_EV_MUTER_UNMUTE : OHP_EV_MUTER_MUTE; // never the same call twice: the reference ASSERTs
                muted[e.stage] = !muted[e.stage];
                e.arg = duration(r, jps, msg_j, total_j);
                break;
            case kStarvation:
                e.op = r.chance(80) ? OHP_EV_STARVATION : OHP_EV_HALT;
                if (e.op == OHP_EV_STARVATION) e.arg = duration(r, jps, msg_j, total_j);
                break;
            }
        }
        ev.push_back(e);
    }
    // sorted by position (stably: events at one position keep their order)
    for (size_t i = 1; i < ev.size(); i++) {
        for (size_t j = i; j > 0 && ev[j].at_jiffies < ev[j - 1].at_jiffies; j--) std::swap(ev[j], ev[j - 1]);
    }
    sp.first_event = 0;
    sp.num_events = (uint32_t)ev.size();
}

int fuzz(uint64_t seed, uint64_t count)
{
    Rng r{seed};
    ohp_stream_spec sp;
    std::vector<ohp_ramp_event> ev;
    uint64_t accepted = 0, refused = 0, violations = 0, playables = 0, bounds = 0, min_slack = ~0ull;
    uint64_t ops[13] = {}, codec = 0, driver = 0, one_sample_cap = 0, wide = 0;
    for (uint64_t k = 0; k < count; k++) {
        random_stream(r, sp, ev);
        uint64_t n = 0, bytes = 0;
        const ohp_ramp_event* e = ev.empty() ? nullptr : ev.data();
        const uint32_t rc = sched::run_stream<false>(sp, e, ev.size(), nullptr, nullptr, n, bytes);
        if (rc != sched::kOk) {
            refused++;
            continue;
        }
        const uint64_t bound = sched::stream_chunk_bound(sp, e, ev.size());
        accepted++;
        playables += n;
        bounds += bound;
        if (n > bound) {
            if (violations++ < 20) {
                std::printf("VIOLATION stream %llu: %llu playables, bound %llu (rate %u, %u-bit x %u, chunk %u, frames %llu, codec %u, "
                            "driver %u, %u events)\n", (unsigned long long)k, (unsigned long long)n, (unsigned long long)bound,
                            sp.sample_rate, sp.bit_depth, sp.channels, sp.chunk_frames, (unsigned long long)sp.total_frames,
                            sp.codec_read_frames, sp.driver_block_frames, sp.num_events);
            }
        }
        else if (bound - n < min_slack) {
            min_slack = bound - n;
        }
        bool seen[13] = {};
        for (const ohp_ramp_event& x : ev) {
            if (x.op < 13) seen[x.op] = true;
            if (x.op == OHP_EV_MAX_MSG_JIFFIES && x.arg == core::jiffies_per_sample_or_zero(sp.sample_rate)) seen[0] = true;
        }
        for (int i = 1; i < 13; i++) ops[i] += seen[i];
        one_sample_cap += seen[0];
        codec += sp.codec_read_frames != 0;
        driver += sp.driver_block_frames != 0;
        wide += sp.channels > 8;
    }
    std::printf("streams %llu accepted %llu refused %llu violations %llu playables %llu bounds %llu min_slack %llu\n",
                (unsigned long long)count, (unsigned long long)accepted, (unsigned long long)refused, (unsigned long long)violations,
                (unsigned long long)playables, (unsigned long long)bounds, (unsigned long long)min_slack);
    std::printf("covered");
    for (int i = 1; i < 13; i++) std::printf(" op%d %llu", i, (unsigned long long)ops[i]);
    std::printf(" one_sample_cap %llu codec %llu driver %llu wide %llu\n", (unsigned long long)one_sample_cap,
                (unsigned long long)codec, (unsigned long long)driver, (unsigned long long)wide);
    return 0;
}

int file(const char* path)
{
    FILE* f = std::fopen(path, "rb");
    if (!f) return 2;
    uint32_t hdr[2];
    while (std::fread(hdr, 4, 2, f) == 2) {
        std::vector<ohp_stream_spec> s(hdr[0]);
        std::vector<ohp_ramp_event> e(hdr[1] ? hdr[1] : 1);
        if (std::fread(s.data(), sizeof s[0], hdr[0], f) != hdr[0] || std::fread(e.data(), sizeof e[0], hdr[1], f) != hdr[1]) return 3;
        for (uint32_t k = 0; k < hdr[0]; k++) {
            uint64_t n = 0, bytes = 0;
            const uint32_t rc = sched::run_stream<false>(s[k], e.data(), hdr[1], nullptr, nullptr, n, bytes);
            const uint64_t bound = sched::stream_chunk_bound(s[k], e.data(), hdr[1]);
            std::printf("%u %llu %llu\n", rc, (unsigned long long)n, (unsigned long long)bound);
        }
    }
    std::fclose(f);
    return 0;
}

} // namespace

int main(int argc, char** argv)
{
    if (argc == 4 && std::strcmp(argv[1], "fuzz") == 0) return fuzz(std::strtoull(argv[2], nullptr, 0), std::strtoull(argv[3], nullptr, 0));
    if (argc == 3 && std::strcmp(argv[1], "file") == 0) return file(argv[2]);
    std::fprintf(stderr, "usage: %s fuzz <seed> <streams> | file <path>\n", argv[0]);
    return 2;
}
