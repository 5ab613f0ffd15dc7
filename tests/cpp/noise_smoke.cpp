// Automatic ray budgets through the C++ mirror (include/frequensee.hpp): three components in the 7 x 5 x 3 m shoebox share
// UAudioRayTracingSubsystem::TotalRaysPerTick on a context created with FS_FLAG_NOISE_STATS.  Two UpdateSources() calls:
// the first splits the total equally, the second by fs_allocate_paths from the first one's noise and the NoiseWeights.
// Prints, per update and component, the budget it traced and its LastNoise, for tests/test_gpu_noise_stats.py to compare
// with the CPU reference.  "nogpu" mode only checks that context creation fails loudly without a device.
#include <cstdio>
#include <cstring>
#include <memory>
#include <vector>
#include "frequensee.hpp"

using namespace FrequenSee;

int main(int argc, char** argv)
{
    fs_config cfg;
    fs_default_config(&cfg);
    cfg.flags |= FS_FLAG_NOISE_STATS;
    auto ctx = FContext::Create(&cfg);
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
    const float pos[3][3] = {{1.5f, 1.2f, 1.0f}, {6.0f, 4.0f, 2.0f}, {3.0f, 2.5f, 1.5f}};
    const int bounces[3] = {8, 4, 3};
    const float weight[3] = {1.0f, 2.0f, 0.5f};
    const uint32_t slot[3] = {5, 2, 9};
    std::vector<std::unique_ptr<UFrequenSeeAudioComponent>> comps;
    for (int s = 0; s < 3; ++s) {
        comps.emplace_back(new UFrequenSeeAudioComponent(ctx, slot[s], FVector3f{pos[s][0], pos[s][1], pos[s][2]}));
        comps[s]->RaycastsPerTick = 99;                      // ignored: the subsystem splits TotalRaysPerTick
        comps[s]->RaycastBounces = bounces[s];
        comps[s]->NoiseWeight = weight[s];
        sub.RegisterSource(comps[s].get());
    }
    sub.SetPlayerPawnLocation(FVector3f{5.0f, 3.5f, 1.6f});
    sub.Seed = 0x5EED;
    sub.TotalRaysPerTick = 6000;
    sub.MinRaysPerSource = 256;
    sub.MaxRaysPerSource = 4096;
    for (int u = 0; u < 2; ++u) {
        sub.UpdateSources();
        if (ctx->LastStatus != FS_OK) { printf("update %d failed: %s\n", u, ctx->LastError().c_str()); return 4; }
        printf("update=%d", u);
        for (int s = 0; s < 3; ++s) {
            const fs_noise_stats& n = comps[s]->LastNoise;
            printf(" n%d=%llu sig%d=%.17g var%d=%.17g", s, (unsigned long long)n.n_paths, s, n.signal, s, n.variance);
        }
        printf("\n");
    }
    return 0;
}
