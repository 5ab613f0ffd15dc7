// First-order edge diffraction through the C++ mirror (include/frequensee.hpp): a 4 x 4 m panel in the plane x = 0
// (y in [-2, 2], z in [0, 4], two triangles), the player at (2, 0, 1) behind it and two components -- one at (-2, 0, 1) in
// the panel's shadow, one at (1, 1, 1) in plain view.  One UpdateDiffraction(30), then each component's LastDiffraction
// printed (%.9g: every float reads back exactly) for tests/test_gpu_diffraction.py to compare with the CPU reference.
// "nogpu" mode only checks that context creation fails loudly without a device.
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
    const float tris[2][3][3] = {{{0, -2, 0}, {0, 2, 0}, {0, 2, 4}}, {{0, -2, 0}, {0, 2, 4}, {0, -2, 4}}};
    UAudioRayTracingSubsystem sub(ctx);
    FAcousticMaterial m; m.Absorption.assign(8, 0.3f);
    sub.RegisterGeometry(&tris[0][0][0], 2, m);
    const float pos[2][3] = {{-2.0f, 0.0f, 1.0f}, {1.0f, 1.0f, 1.0f}};
    std::vector<std::unique_ptr<UFrequenSeeAudioComponent>> comps;
    for (int s = 0; s < 2; ++s) {
        comps.emplace_back(new UFrequenSeeAudioComponent(ctx, (uint32_t)s, FVector3f{pos[s][0], pos[s][1], pos[s][2]}));
        sub.RegisterSource(comps[s].get());
    }
    sub.SetPlayerPawnLocation(FVector3f{2.0f, 0.0f, 1.0f});
    sub.UpdateDiffraction(30.0f);
    if (ctx->LastStatus != FS_OK) { printf("UpdateDiffraction failed: %s\n", ctx->LastError().c_str()); return 4; }
    for (int s = 0; s < 2; ++s) {
        const fs_diffraction_result& r = comps[s]->LastDiffraction;
        printf("diffraction s%d found=%u n=%u edge=%u,%u apex=%.9g,%.9g,%.9g length=%.9g z=%.9g gain=", s, r.found, r.n_paths,
               r.edge_tri, r.edge_k, r.apex[0], r.apex[1], r.apex[2], r.length, r.path_difference);
        for (uint32_t b = 0; b < cfg.n_bands; ++b) printf(b ? ",%.9g" : "%.9g", r.gain[b]);
        printf("\n");
    }
    return 0;
}
