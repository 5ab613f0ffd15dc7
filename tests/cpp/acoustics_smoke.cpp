// Room-acoustic parameters through the C++ mirror (include/frequensee.hpp): three components in the 7 x 5 x 3 m shoebox,
// one UpdateSources() with seed 0x5EED, then UpdateAcousticParams().  Prints, per component, the onset and valid bits and
// the broadband and band-0 EDT / T20 / T30, C50 / C80 / D50 and Ts of its LastAcoustics (%.17g: every double reads back
// exactly) for tests/test_gpu_acoustics.py to compare with the CPU reference.  A second UpdateAcousticParams() after a
// source has been unregistered must fail and leave LastAcoustics alone.  "nogpu" mode only checks that context creation
// fails loudly without a device.
#include <cstdio>
#include <cstring>
#include <memory>
#include <vector>
#include "frequensee.hpp"

using namespace FrequenSee;

static void print_slot(const char* name, int s, const fs_acoustic_slot& a)
{
    printf("acoustics s%d %s onset=%u valid=%u edt=%.17g t20=%.17g t30=%.17g r30=%.17g c50=%.17g c80=%.17g d50=%.17g ts=%.17g\n", s,
           name, a.onset_bin, a.valid, a.edt.time_s, a.t20.time_s, a.t30.time_s, a.t30.r, a.c50_db, a.c80_db, a.d50, a.ts_s);
}

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
    const int rays[3] = {20000, 12000, 8000};
    const int bounces[3] = {16, 8, 12};
    std::vector<std::unique_ptr<UFrequenSeeAudioComponent>> comps;
    for (int s = 0; s < 3; ++s) {
        comps.emplace_back(new UFrequenSeeAudioComponent(ctx, (uint32_t)s, FVector3f{pos[s][0], pos[s][1], pos[s][2]}));
        comps[s]->RaycastsPerTick = rays[s];
        comps[s]->RaycastBounces = bounces[s];
        sub.RegisterSource(comps[s].get());
    }
    sub.SetPlayerPawnLocation(FVector3f{5.0f, 3.5f, 1.6f});
    sub.Seed = 0x5EED;
    sub.UpdateSources();
    if (ctx->LastStatus != FS_OK) { printf("UpdateSources failed: %s\n", ctx->LastError().c_str()); return 4; }
    if (!sub.UpdateAcousticParams()) { printf("UpdateAcousticParams failed: %s\n", ctx->LastError().c_str()); return 5; }
    for (int s = 0; s < 3; ++s) {
        printf("acoustics s%d no_energy=%u\n", s, comps[s]->LastAcoustics.no_energy);
        print_slot("broadband", s, comps[s]->LastAcoustics.broadband);
        print_slot("band0", s, comps[s]->LastAcoustics.band[0]);
    }
    const fs_acoustic_params keep = comps[0]->LastAcoustics;
    sub.UnregisterSource(comps[2].get());
    if (sub.UpdateAcousticParams() || ctx->LastStatus != FS_ERR_STATE) { printf("UNEXPECTED: stale histogram accepted\n"); return 6; }
    if (memcmp(&keep, &comps[0]->LastAcoustics, sizeof(keep))) { printf("UNEXPECTED: LastAcoustics changed\n"); return 7; }
    printf("stale update refused\n");
    return 0;
}
