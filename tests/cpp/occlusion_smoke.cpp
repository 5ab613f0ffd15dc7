// Direct-path occlusion through the C++ mirror (include/frequensee.hpp): the 7 x 5 x 3 m shoebox with a partition at x = 3.5
// over y in [0, 3] (a gap above y = 3), the player at (5, 1.5, 1.6) and three components -- one in the player's half, one
// behind the partition, and one as a 0.8 m ball by the partition's edge sampled by 512 rays.  One UpdateOcclusion(8, 77),
// then each component's LastOcclusion printed (%.9g: every float reads back exactly) for
// tests/test_gpu_occlusion.py to compare with the CPU reference.  "nogpu" mode only checks that context creation fails
// loudly without a device.
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
    auto ctx = FContext::Create(&cfg);
    if (argc > 1 && !strcmp(argv[1], "nogpu")) {
        if (ctx) { printf("UNEXPECTED: context created without a GPU\n"); return 1; }
        printf("no-gpu: %s\n", fs_last_error(nullptr));
        return strstr(fs_last_error(nullptr), "no CPU fallback") ? 0 : 2;
    }
    if (!ctx) { printf("fs_create failed: %s\n", fs_last_error(nullptr)); return 3; }
    const float X = 7, Y = 5, Z = 3, P = 3.5f, G = 3;
    const float quads[7][4][3] = {
        {{0,0,0},{0,Y,0},{0,Y,Z},{0,0,Z}}, {{X,0,0},{X,Y,0},{X,Y,Z},{X,0,Z}},
        {{0,0,0},{X,0,0},{X,0,Z},{0,0,Z}}, {{0,Y,0},{X,Y,0},{X,Y,Z},{0,Y,Z}},
        {{0,0,0},{X,0,0},{X,Y,0},{0,Y,0}}, {{0,0,Z},{X,0,Z},{X,Y,Z},{0,Y,Z}},
        {{P,0,0},{P,G,0},{P,G,Z},{P,0,Z}}};
    const float alpha[7] = {0.02f, 0.05f, 0.12f, 0.07f, 0.37f, 0.75f, 0.3f};
    UAudioRayTracingSubsystem sub(ctx);
    for (int f = 0; f < 7; ++f) {
        float tris[2][3][3];
        const int idx[2][3] = {{0, 1, 2}, {0, 2, 3}};
        for (int t = 0; t < 2; ++t) for (int v = 0; v < 3; ++v) memcpy(tris[t][v], quads[f][idx[t][v]], 12);
        FAcousticMaterial m; m.Absorption.assign(8, alpha[f]);
        sub.RegisterGeometry(&tris[0][0][0], 2, m);
    }
    const float pos[3][3] = {{6.0f, 1.0f, 1.2f}, {1.5f, 1.5f, 1.5f}, {2.8f, 2.9f, 1.5f}};
    const float radius[3] = {0.0f, 0.0f, 0.8f};
    std::vector<std::unique_ptr<UFrequenSeeAudioComponent>> comps;
    for (int s = 0; s < 3; ++s) {
        comps.emplace_back(new UFrequenSeeAudioComponent(ctx, (uint32_t)s, FVector3f{pos[s][0], pos[s][1], pos[s][2]}));
        comps[s]->OcclusionRadius = radius[s];
        comps[s]->OcclusionRays = 512;
        sub.RegisterSource(comps[s].get());
    }
    sub.SetPlayerPawnLocation(FVector3f{5.0f, 1.5f, 1.6f});
    sub.UpdateOcclusion(8, 77);
    if (ctx->LastStatus != FS_OK) { printf("UpdateOcclusion failed: %s\n", ctx->LastError().c_str()); return 4; }
    for (int s = 0; s < 3; ++s) {
        const fs_occlusion_result& r = comps[s]->LastOcclusion;
        printf("occlusion s%d n=%u visible=%.9g tr=", s, r.n_rays, r.visible);
        for (uint32_t b = 0; b < cfg.n_bands; ++b) printf(b ? ",%.9g" : "%.9g", r.transmission[b]);
        printf("\n");
    }
    return 0;
}
