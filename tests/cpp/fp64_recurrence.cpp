// fp64_recurrence.cpp -- the device walk's FP64 ramp recurrence (ohpipeline_b200/host/schedule_walk.h, bulk_step, the
// STRIDE == kBulk branch that only the device compiles) restated on the host with std::fma, which rounds exactly as the
// GPU's DFMA does, and checked against the integer division every other walk uses (core::mul_add_div).  Built and run
// by tests/test_long_streams.py; tests/test_gpu_long_streams.py runs the real branch on the GPU.
//
//   fp64_recurrence <cases> <sweep>: <cases> = uint64 n, then n x (uint32 distance, size, remaining); then <sweep>
//   seeded adversarial cases.  Prints one line per disagreement, then "checked <n> edges <e>".
//   Build with -ffp-contract=off: the device code multiplies and adds where it says so, and nowhere else.
#include "../../ohpipeline_b200/host/ramp_core.h"

#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <random>

using namespace ohp;

// schedule_walk.h, bulk_step: one step of the chain, message with distance / remaining in front of it
static uint32_t fp64_step(uint32_t distance, uint32_t size, uint32_t remaining)
{
    const double sizeD = (double)size;
    const double inv = 1.0 / (double)remaining;
    const double remD = (double)remaining;
    const double distD = (double)distance;
    const double numd = std::fma(distD, sizeD, remD - 1.0);
    double qd = std::trunc(numd * inv);
    const double r = std::fma(-qd, remD, numd);
    // Only the upward correction is ever taken on these inputs: the numerator is below 2^36, so the product's error stays
    // below 1 / remaining and trunc never lands above the quotient.  The downward one is kept as the device code has it.
    if (r < 0.0) qd -= 1.0;
    else if (r >= remD) qd += 1.0;
    return (uint32_t)qd;
}

static uint64_t g_checked = 0, g_edges = 0, g_bad = 0;

static void check(uint32_t distance, uint32_t size, uint32_t remaining)
{
    // what the device loop ever sees: a message inside the ramp (remaining >= size), size < 2^21, distance <= kRampMax
    if (distance == 0 || distance > core::kRampMax || size == 0 || size >= (1u << 21) || remaining < size) return;
    const uint32_t want = core::mul_add_div(distance, size, remaining - 1, remaining);
    const uint32_t got = fp64_step(distance, size, remaining);
    const uint64_t num = (uint64_t)distance * size + remaining - 1;
    const uint64_t r = num % remaining;
    g_checked++;
    if (r == 0 || r == 1 || r == remaining - 1) g_edges++;
    if (got != want && g_bad++ < 20) {
        std::printf("distance %u size %u remaining %u: fp64 %u integer %u\n", distance, size, remaining, got, want);
    }
}

int main(int argc, char** argv)
{
    if (argc != 3) return 2;
    FILE* f = std::fopen(argv[1], "rb");
    if (!f) return 2;
    uint64_t n = 0;
    if (std::fread(&n, 8, 1, f) != 1) return 2;
    for (uint64_t i = 0; i < n; i++) {
        uint32_t c[3];
        if (std::fread(c, 4, 3, f) != 3) return 2;
        check(c[0], c[1], c[2]);
    }
    std::fclose(f);
    const uint64_t sweep = std::strtoull(argv[2], nullptr, 10);
    std::mt19937_64 rng(0x0F64);
    for (uint64_t i = 0; i < sweep; i++) {
        const uint32_t pick = (uint32_t)(rng() % 4);
        uint32_t size = pick == 0 ? (1u << 21) - 1 : (uint32_t)(rng() % ((1u << 21) - 1)) + 1;
        const uint32_t distance = (rng() & 1) ? core::kRampMax - (uint32_t)(rng() % 64) : (uint32_t)(rng() % core::kRampMax) + 1;
        uint64_t rem;
        if (pick == 1) {
            rem = 0xffffffffull - (rng() % 1024);                     // within 2^10 of 2^32 - 1
        } else {
            // an exact multiple of the divisor, or one beside it: distance * size + remaining - 1 = q * remaining + c - 1
            const uint64_t m = 1 + rng() % (pick == 3 ? 4096 : 8);
            const uint64_t c = rng() % 3;
            rem = ((uint64_t)distance * size - c) / m;
        }
        if (rem > 0xffffffffull) rem = 0xffffffffull - (rng() % 1024);
        if (rem < size) rem = size + (rng() % 1024);
        for (int d = -1; d <= 1; d++) check(distance, size, (uint32_t)(rem + d > 0xffffffffull ? rem : rem + d));
    }
    std::printf("checked %llu edges %llu\n", (unsigned long long)g_checked, (unsigned long long)g_edges);
    return g_bad ? 1 : 0;
}
