// Per-source budgets through the C++ mirror (include/frequensee.hpp): three components with their own RaycastsPerTick and
// RaycastBounces in the 7 x 5 x 3 m shoebox, updated by ONE UAudioRayTracingSubsystem::UpdateSources() call.  Prints, per
// component, its histogram (FNV-1a 64 of the Q32.32 words of its slot) and its IR energy and peak, for
// tests/test_source_budgets.py to compare with the CPU reference.  "nogpu" mode only checks that context creation fails
// loudly without a device.
#include <cmath>
#include <cstdio>
#include <cstring>
#include <vector>
#include "frequensee.hpp"

using namespace FrequenSee;

int main(int argc, char** argv)
{
    auto ctx = FContext::Create();
    if (argc > 1 && !strcmp(argv[1], "nogpu")) {
        if (ctx) { printf("UNEXPECTED: context created without a GPU\n"); return 1; }
        printf("no-gpu: %s\n", fs_last_error(nullptr));
        return strstr(fs_last_error(nullptr), "no CPU fallback") ? 0 : 2;
    }
    if (!ctx) { printf("fs_create failed: %s\n", fs_last_error(nullptr)); return 3; }
    const float X = 7, Y = 5, Z = 3;
    const float quads[6][4][3] = {
        {{0,0,0},{0,Y,0},{0,Y,Z},{0,0,Z}}, {{X,0,0},{X,Y,0},{X,Y,Z},{X,0,Z}},
        {{0,0,0},{X,0,0},{X,0,Z},{0,0,Z}}, {{0,Y,0},{X,Y,0},{X,Y,Z},{0,Y,Z}},
        {{0,0,0},{X,0,0},{X,Y,0},{0,Y,0}}, {{0,0,Z},{X,0,Z},{X,Y,Z},{0,Y,Z}}};
    const float alpha[6] = {0.02f, 0.05f, 0.12f, 0.07f, 0.37f, 0.75f};
    UAudioRayTracingSubsystem sub(ctx);
    for (int f = 0; f < 6; ++f) {
        float tris[2][3][3];
        const int idx[2][3] = {{0, 1, 2}, {0, 2, 3}};
        for (int t = 0; t < 2; ++t) for (int v = 0; v < 3; ++v) memcpy(tris[t][v], quads[f][idx[t][v]], 12);
        FAcousticMaterial m; m.Absorption.assign(8, alpha[f]);
        sub.RegisterGeometry(&tris[0][0][0], 2, m);
    }
    // (position, RaycastsPerTick, RaycastBounces, convolver slot) of each component
    const float pos[3][3] = {{1.5f, 1.2f, 1.0f}, {6.0f, 4.0f, 2.0f}, {3.0f, 2.5f, 1.5f}};
    const int paths[3] = {4096, 700, 1500}, bounces[3] = {8, 0, 3};
    const uint32_t slot[3] = {5, 2, 9};
    std::vector<std::unique_ptr<UFrequenSeeAudioComponent>> comps;
    for (int s = 0; s < 3; ++s) {
        comps.emplace_back(new UFrequenSeeAudioComponent(ctx, slot[s], FVector3f{pos[s][0], pos[s][1], pos[s][2]}));
        comps[s]->RaycastsPerTick = paths[s]; comps[s]->RaycastBounces = bounces[s];
        sub.RegisterSource(comps[s].get());
    }
    sub.SetPlayerPawnLocation(FVector3f{5.0f, 3.5f, 1.6f});
    sub.Seed = 0x5EED;
    sub.UpdateSources();
    if (ctx->LastStatus != FS_OK) { printf("update failed: %s\n", ctx->LastError().c_str()); return 4; }
    uint32_t n = 0;
    fs_get_histogram_sources(ctx->Get(), &n);
    if (n != 3) { printf("histogram has %u sources\n", n); return 5; }
    const fs_config& c = ctx->Config();
    const size_t per = (size_t)c.n_bands * c.n_bins;
    std::vector<uint64_t> h(3 * per);
    if (fs_get_histogram(ctx->Get(), h.data()) != FS_OK) { printf("fs_get_histogram failed\n"); return 6; }
    printf("connected=%llu", (unsigned long long)sub.LastConnected);
    for (int s = 0; s < 3; ++s) {
        uint64_t f = 1469598103934665603ull;
        for (size_t i = 0; i < per; ++i) {
            uint64_t w = h[s * per + i];
            for (int b = 0; b < 8; ++b) { f ^= (w >> (8 * b)) & 0xffu; f *= 1099511628211ull; }
        }
        auto& ir = comps[s]->GetImpulseResponse();
        double e = 0; int peak = 0;
        for (int i = 0; i < c.sample_rate; ++i) { e += (double)ir[0][i] * ir[0][i]; if (ir[0][i] > ir[0][peak]) peak = i; }
        printf(" hist%d=%llu ir_energy%d=%.9g ir_peak%d=%d", s, (unsigned long long)f, s, e, s, peak);
    }
    printf("\n");
    return 0;
}
