// flywheel_plan_harness.cpp -- holds the planner the device compiles (ohpipeline_b200/host/flywheel_plan.h) against the
// class-based ohp_flywheel_plan of libohp_host.so, record by record.  Built and run by tests/test_starvation_walk.py.
// Input file: uint64 n, then n x (ohp_stream_spec, ohp_starvation).  Output: one line per record that disagrees, then
// "checked <n> planned <k>".
#include "../../ohpipeline_b200/host/flywheel_plan.h"

#include <cstdio>
#include <cstring>
#include <vector>

int main(int argc, char** argv)
{
    if (argc != 2) return 2;
    FILE* f = std::fopen(argv[1], "rb");
    if (!f) return 2;
    uint64_t n = 0;
    if (std::fread(&n, 8, 1, f) != 1) return 2;
    uint64_t planned = 0;
    for (uint64_t i = 0; i < n; i++) {
        ohp_stream_spec sp;
        ohp_starvation sv;
        if (std::fread(&sp, sizeof sp, 1, f) != 1 || std::fread(&sv, sizeof sv, 1, f) != 1) return 2;
        const uint64_t training = 1024 + 16 * i, generated = 4096 + 32 * i, out = 65536 + 48 * i;
        ohp_chunk_desc prepA[OHP_FLYWHEEL_MAX_PREP], blocksA[64];
        ohp_flywheel_job jobA;
        size_t nPrepA = 0, nBlocksA = 0;
        std::memset(&jobA, 0, sizeof jobA);
        const int rcA = ohp_flywheel_plan(&sp, &sv, training, generated, out, prepA, &nPrepA, &jobA, blocksA, 64, &nBlocksA);
        ohp_chunk_desc prepB[OHP_FLYWHEEL_MAX_PREP], blocksB[ohp::flyplan::kMaxBlocks];
        ohp_flywheel_job jobB;
        uint32_t nPrepB = 0, nBlocksB = 0;
        std::memset(&jobB, 0, sizeof jobB);
        const int rcB = ohp::flyplan::plan(sp, sv, training, generated, out, prepB, nPrepB, jobB, blocksB, nBlocksB);
        bool same = rcA == rcB;
        if (same && rcA == OHP_OK) {
            planned++;
            same = nPrepA == nPrepB && nBlocksA == nBlocksB && std::memcmp(&jobA, &jobB, sizeof jobA) == 0
                && std::memcmp(prepA, prepB, nPrepA * sizeof(ohp_chunk_desc)) == 0
                && std::memcmp(blocksA, blocksB, nBlocksA * sizeof(ohp_chunk_desc)) == 0;
            // ohp_flywheel_ramp_chunks on its own, from the plan's job and ramp
            ohp_chunk_desc chunksA[64], chunksB[ohp::flyplan::kMaxBlocks];
            uint32_t nB = 0;
            const int nA = ohp_flywheel_ramp_chunks(&jobA, sv.ramp, 7, 9, chunksA, 64, nullptr);
            const int rB = ohp::flyplan::ramp_chunks(jobB, sv.ramp, 7, 9, chunksB, nB);
            same = same && nA >= 0 && rB == OHP_OK && (uint32_t)nA == nB && std::memcmp(chunksA, chunksB, nB * sizeof(ohp_chunk_desc)) == 0;
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
