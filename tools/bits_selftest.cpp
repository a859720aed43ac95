// Host self-test of latok_b200/csrc/latok_bits.h (g++ only, no GPU): the bit-sliced ASCII classifier against the
// generated class table, the byte->plane transpose, squeeze_planes, chunk_carry (and when it must defer to the exact
// evaluation) and flood_down against scalar loops.
//   g++ -O1 -std=c++17 -I latok_b200/csrc tools/bits_selftest.cpp -o /tmp/bits_selftest && /tmp/bits_selftest
#include "latok_bits.h"
#include "_gen/latok_tables.h"
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <random>
using namespace latok;

static int fails = 0;
#define CHECK(c, ...) do { if (!(c)) { if (fails < 20) { printf("FAIL %s:%d: ", __FILE__, __LINE__); printf(__VA_ARGS__); printf("\n"); } ++fails; } } while (0)

int main()
{
    std::mt19937 rng(12345);
    // transpose + classifier: every byte value at every position
    for (int rep = 0; rep < 2000; ++rep) {
        uint8_t bytes[32];
        for (int j = 0; j < 32; ++j) bytes[j] = rep < 256 ? (uint8_t)((rep + j * 37) & 0xFF) : (uint8_t)(rng() & 0xFF);
        if (rep < 256) bytes[rep & 31] = (uint8_t)rep;
        uint32_t w[8], b[8], P[NBASE];
        memcpy(w, bytes, 32);
        bytes_to_planes(w, b);
        for (int j = 0; j < 32; ++j) for (int k = 0; k < 8; ++k)
            CHECK(((b[k] >> j) & 1u) == ((bytes[j] >> k) & 1u), "transpose byte %d bit %d", j, k);
        classify_ascii(b, P);
        for (int j = 0; j < 32; ++j) {
            const uint32_t want = bytes[j] < 128 ? LATOK_ASCII_FEAT[bytes[j]] : 0u;
            uint32_t got = 0;
            for (int f = 0; f < NBASE; ++f) got |= ((P[f] >> j) & 1u) << f;
            CHECK(got == want, "classify byte 0x%02X: got 0x%03X want 0x%03X", bytes[j], got, want);
        }
    }
    // squeeze
    for (int rep = 0; rep < 20000; ++rep) {
        uint32_t lead = (uint32_t)rng(), F = (uint32_t)rng(), P[3] = {(uint32_t)rng(), (uint32_t)rng(), (uint32_t)rng()};
        if (rep % 3 == 0) lead |= rng() | rng();
        const int vhi = rep % 5 == 0 ? (int)(rng() % 33) : 32;
        const uint32_t vmask = bits_low(vhi);
        lead &= vmask;
        uint32_t wantP[3] = {0, 0, 0}, wantF = 0; int o = 0;
        for (int j = 0; j < 32; ++j) if ((lead >> j) & 1u) {
            for (int f = 0; f < 3; ++f) wantP[f] |= ((P[f] >> j) & 1u) << o;
            wantF |= ((F >> j) & 1u) << o; ++o;
        }
        uint32_t Q[3] = {P[0], P[1], P[2]}, G = F;
        squeeze_planes<3>(Q, G, lead, vmask);
        const uint32_t nm = bits_low(o);
        if (lead) CHECK((Q[0] & nm) == wantP[0] && (Q[1] & nm) == wantP[1] && (Q[2] & nm) == wantP[2] && (G & nm) == wantF, "squeeze lead %08X", lead);
        uint32_t R[3] = {P[0], P[1], P[2]}, H = F;
        squeeze_planes_log<3>(R, H, lead);
        if (lead) CHECK(R[0] == wantP[0] && R[1] == wantP[1] && R[2] == wantP[2] && H == wantF, "squeeze (compress form) lead %08X", lead);
    }
    // chunk_carry / flood_down against the sequential definition (latok.c:218-244: a mark is taken before a closer at
    // the same position).  Marks may fall on closers (custom mask rows); chunk_carry is exact unless it flags the case
    // for the exact evaluation: a chunk with two marks pending, or a mark on a closer.
    int flagged_on_closer = 0;
    for (int rep = 0; rep < 200000; ++rep) {
        const int n = rep % 7 == 0 ? (int)(rng() % 33) : 32;
        const uint32_t nm = bits_low(n);
        uint32_t CL = rng() & rng() & nm, M = rng() & rng() & rng() & nm;
        if (rep % 4 == 0) M &= rng();
        if (rep % 3 != 0) M &= ~CL | (rng() & rng() & rng());    // mostly off the closers (all of them, under the default rules)
        const uint32_t cin = rng() & 1u, bin = rng() & 1u;
        // sequential
        int x = (int)cin; uint32_t hot = 0; bool dup = false;
        for (int j = 0; j < n; ++j) {
            if ((M >> j) & 1u) { if (x >= 1) dup = true; ++x; }
            if ((CL >> j) & 1u) { if (x >= 1) hot |= 1u << j; x = x > 0 ? x - 1 : 0; }
        }
        uint32_t cout;
        const uint32_t T = chunk_carry(M, CL, cin, cout);
        const bool dup2 = (M & ~CL & T) != 0u, flagged = dup2 || (M & CL) != 0u;
        if ((M & CL) == 0u) CHECK(dup == dup2, "dup M %08X CL %08X cin %u", M, CL, cin);
        else ++flagged_on_closer;
        CHECK(!dup || flagged, "two marks pending not flagged: M %08X CL %08X cin %u", M, CL, cin);
        if (!flagged) {
            CHECK((T & CL) == hot, "hot M %08X CL %08X cin %u: %08X vs %08X", M, CL, cin, T & CL, hot);
            CHECK(cout == (uint32_t)(x >= 1), "cout M %08X CL %08X cin %u", M, CL, cin);
            // flood
            uint32_t Z = 0; int nexthot = (int)bin;
            for (int j = n - 1; j >= 0; --j) {
                if ((CL >> j) & 1u) nexthot = (hot >> j) & 1u;
                if (nexthot) Z |= 1u << j;
            }
            const uint32_t Z2 = flood_down(hot, CL, bin) & nm;
            CHECK(Z == Z2, "flood hot %08X CL %08X bin %u n %d: %08X vs %08X", hot, CL, bin, n, Z2, Z);
        }
    }
    CHECK(flagged_on_closer > 10000, "only %d cases with a mark on a closer", flagged_on_closer);
    printf(fails ? "bits selftest: %d FAILURES\n" : "bits selftest ok\n", fails);
    return fails ? 1 : 0;
}
