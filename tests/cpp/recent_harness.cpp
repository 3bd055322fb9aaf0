// recent_harness.cpp -- the recent audio of the device walk and the device planner, on the host.  Built and run by
// tests/test_starvation_walk_recent.py.
//
//   recent_harness walk <in> <out>: <in> = uint64 n_streams, uint64 n_events, the streams (ohp_stream_spec), the events
//     (ohp_ramp_event).  Walks every stream with the recent audio kept (schedule_walk.h, RECENT: a team of one), once with
//     the bulk step and once without, and writes to <out>, per walk: the stream status words (uint32 x n_streams), the
//     records (ohp_starvation x n_events, all ones where an event left none), the piece counts (uint32 x n_events) and
//     the pieces (ohp_recent_audio x n_events x OHP_DEVICE_RECENT_PIECES, zero where unused).
//   recent_harness plan <in>: <in> = uint64 n, then n x (ohp_stream_spec, ohp_starvation, uint32 pieces, that many
//     ohp_recent_audio).  Holds flyplan::plan_recent against ohp_flywheel_plan_recent of libohp_host.so (prep room
//     OHP_FLYWHEEL_MAX_PREP_RECENT); prints one line per record that disagrees, then "checked <n> planned <k>".
#include "../../ohpipeline_b200/host/flywheel_plan.h"

#include <cstdio>
#include <cstring>
#include <vector>

using namespace ohp;

static int walk(const char* in, const char* out)
{
    FILE* f = std::fopen(in, "rb");
    if (!f) return 2;
    uint64_t ns = 0, ne = 0;
    if (std::fread(&ns, 8, 1, f) != 1 || std::fread(&ne, 8, 1, f) != 1) return 2;
    std::vector<ohp_stream_spec> streams(ns);
    std::vector<ohp_ramp_event> events(ne);
    if ((ns && std::fread(streams.data(), sizeof(ohp_stream_spec), ns, f) != ns) || (ne && std::fread(events.data(), sizeof(ohp_ramp_event), ne, f) != ne)) return 2;
    std::fclose(f);
    FILE* o = std::fopen(out, "wb");
    if (!o) return 2;
    for (int bulk = 1; bulk >= 0; bulk--) {
        std::vector<uint32_t> rcs(ns, 0);
        std::vector<ohp_starvation> rec(ne);
        std::memset(rec.data(), 0xff, ne * sizeof(ohp_starvation));
        std::vector<uint32_t> count(ne, 0);
        std::vector<ohp_recent_audio> pieces(ne * sched::kRecentPieces);
        std::memset(pieces.data(), 0, pieces.size() * sizeof(ohp_recent_audio));
        for (uint64_t s = 0; s < ns; s++) {
            const ohp_stream_spec& sp = streams[s];
            uint64_t n = 0, bytes = 0;
            ohp_starvation* r = rec.data() + sp.first_event;
            ohp_recent_audio* p = pieces.data() + sp.first_event * sched::kRecentPieces;
            uint32_t* c = count.data() + sp.first_event;
            rcs[s] = bulk ? sched::run_stream<false, 1, true, true, true>(sp, events.data(), ne, nullptr, nullptr, n, bytes, 0, ~0ull, r, s, false, nullptr, p, c)
                          : sched::run_stream<false, 1, false, true, true>(sp, events.data(), ne, nullptr, nullptr, n, bytes, 0, ~0ull, r, s, false, nullptr, p, c);
        }
        std::fwrite(rcs.data(), sizeof(uint32_t), ns, o);
        std::fwrite(rec.data(), sizeof(ohp_starvation), ne, o);
        std::fwrite(count.data(), sizeof(uint32_t), ne, o);
        std::fwrite(pieces.data(), sizeof(ohp_recent_audio), pieces.size(), o);
    }
    std::fclose(o);
    return 0;
}

static int plan(const char* in)
{
    FILE* f = std::fopen(in, "rb");
    if (!f) return 2;
    uint64_t n = 0;
    if (std::fread(&n, 8, 1, f) != 1) return 2;
    uint64_t planned = 0;
    for (uint64_t i = 0; i < n; i++) {
        ohp_stream_spec sp;
        ohp_starvation sv;
        uint32_t np = 0;
        if (std::fread(&sp, sizeof sp, 1, f) != 1 || std::fread(&sv, sizeof sv, 1, f) != 1 || std::fread(&np, 4, 1, f) != 1) return 2;
        std::vector<ohp_recent_audio> pieces(np ? np : 1);
        if (np && std::fread(pieces.data(), sizeof(ohp_recent_audio), np, f) != np) return 2;
        const uint64_t training = 1024 + 16 * i, generated = 4096 + 32 * i, out = 65536 + 48 * i;
        ohp_chunk_desc prepA[OHP_FLYWHEEL_MAX_PREP_RECENT], blocksA[64];
        ohp_flywheel_job jobA;
        size_t nPrepA = 0, nBlocksA = 0;
        std::memset(&jobA, 0, sizeof jobA);
        const int rcA = ohp_flywheel_plan_recent(&sp, &sv, np ? pieces.data() : nullptr, np, training, generated, out, prepA,
                                                 OHP_FLYWHEEL_MAX_PREP_RECENT, &nPrepA, &jobA, blocksA, 64, &nBlocksA);
        ohp_chunk_desc prepB[OHP_FLYWHEEL_MAX_PREP_RECENT], blocksB[flyplan::kMaxBlocks];
        ohp_flywheel_job jobB;
        uint32_t nPrepB = 0, nBlocksB = 0;
        std::memset(&jobB, 0, sizeof jobB);
        const int rcB = flyplan::plan_recent(sp, sv, pieces.data(), np, training, generated, out, prepB, nPrepB, jobB, blocksB, nBlocksB);
        bool same = rcA == rcB;
        if (same && rcA == OHP_OK) {
            planned++;
            same = nPrepA == nPrepB && nBlocksA == nBlocksB && std::memcmp(&jobA, &jobB, sizeof jobA) == 0
                && std::memcmp(prepA, prepB, nPrepA * sizeof(ohp_chunk_desc)) == 0
                && std::memcmp(blocksA, blocksB, nBlocksA * sizeof(ohp_chunk_desc)) == 0;
        }
        if (!same) {
            std::printf("record %llu: class-based rc %d (%zu prep, %zu blocks), device planner rc %d (%u prep, %u blocks)\n",
                        (unsigned long long)i, rcA, nPrepA, nBlocksA, rcB, nPrepB, nBlocksB);
        }
    }
    std::fclose(f);
    std::printf("checked %llu planned %llu\n", (unsigned long long)n, (unsigned long long)planned);
    return 0;
}

int main(int argc, char** argv)
{
    if (argc == 4 && std::strcmp(argv[1], "walk") == 0) return walk(argv[2], argv[3]);
    if (argc == 3 && std::strcmp(argv[1], "plan") == 0) return plan(argv[2]);
    return 2;
}
