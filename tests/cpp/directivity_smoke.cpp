// Directional sources through the C++ mirror (include/frequensee.hpp): three components in the 7 x 5 x 3 m shoebox, two
// of them with a pattern of UAudioRayTracingSubsystem::SetDirectivityPatterns (a cardioid and a figure of eight from
// fs_directivity_polar) and the third omni.  One UpdateSources(), then UpdateSource() of component 0 alone, then
// UpdateSources() with every component omni (the orientations are cleared again).  After each update it prints, per
// histogram slot, the sum of its Q32.32 bins, for tests/test_gpu_source_directivity.py to compare with the CPU reference.
// "nogpu" mode only checks that context creation fails loudly without a device.
#include <cstdio>
#include <cstring>
#include <memory>
#include <vector>
#include "frequensee.hpp"

using namespace FrequenSee;

static int print_sums(const std::shared_ptr<FContext>& ctx, const char* tag)
{
    uint32_t S = 0;
    if (fs_get_histogram_sources(ctx->Get(), &S) != FS_OK) return 5;
    const fs_config& c = ctx->Config();
    std::vector<uint64_t> h((size_t)S * c.n_bands * c.n_bins);
    if (fs_get_histogram(ctx->Get(), h.data()) != FS_OK) return 6;
    printf("%s", tag);
    for (uint32_t s = 0; s < S; ++s) {
        unsigned long long sum = 0;
        for (size_t i = 0; i < (size_t)c.n_bands * c.n_bins; ++i) sum += h[(size_t)s * c.n_bands * c.n_bins + i];
        printf(" s%u=%llu", s, sum);
    }
    printf("\n");
    return 0;
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
    std::vector<fs_directivity> pats(2);
    const float card_w[8] = {0.5f, 0.5f, 0.5f, 0.5f, 0.5f, 0.5f, 0.5f, 0.5f}, eight_w[8] = {1, 1, 1, 1, 1, 1, 1, 1};
    const float one[8] = {1, 1, 1, 1, 1, 1, 1, 1};
    if (fs_directivity_polar(card_w, one, cfg.n_bands, &pats[0]) != FS_OK ||
        fs_directivity_polar(eight_w, one, cfg.n_bands, &pats[1]) != FS_OK) { printf("fs_directivity_polar failed\n"); return 4; }
    if (!sub.SetDirectivityPatterns(pats)) { printf("SetDirectivityPatterns failed: %s\n", ctx->LastError().c_str()); return 4; }
    const float pos[3][3] = {{1.5f, 1.2f, 1.0f}, {6.0f, 4.0f, 2.0f}, {3.0f, 2.5f, 1.5f}};
    const FVector3f fwd[3] = {{1.f, 0.f, 0.f}, {0.f, -2.f, 0.f}, {0.f, 0.f, 1.f}};
    const uint32_t pattern[3] = {0, 1, FS_OMNI};
    const uint32_t slot[3] = {5, 2, 9};
    std::vector<std::unique_ptr<UFrequenSeeAudioComponent>> comps;
    for (int s = 0; s < 3; ++s) {
        comps.emplace_back(new UFrequenSeeAudioComponent(ctx, slot[s], FVector3f{pos[s][0], pos[s][1], pos[s][2]}));
        comps[s]->RaycastsPerTick = 3000 + 1000 * s;
        comps[s]->RaycastBounces = 8 - 2 * s;
        comps[s]->Forward = fwd[s];
        comps[s]->DirectivityPattern = pattern[s];
        sub.RegisterSource(comps[s].get());
    }
    sub.SetPlayerPawnLocation(FVector3f{5.0f, 3.5f, 1.6f});
    sub.Seed = 0x5EED;
    sub.UpdateSources();                                     // seed 0x5EED
    if (ctx->LastStatus != FS_OK) { printf("UpdateSources failed: %s\n", ctx->LastError().c_str()); return 4; }
    if (int rc = print_sums(ctx, "sources")) return rc;
    sub.UpdateSource(*comps[0]);                             // seed 0x5EED + 1, one source in slot 0
    if (ctx->LastStatus != FS_OK) { printf("UpdateSource failed: %s\n", ctx->LastError().c_str()); return 4; }
    if (int rc = print_sums(ctx, "source0")) return rc;
    for (auto& c : comps) c->DirectivityPattern = FS_OMNI;
    sub.UpdateSources();                                     // seed 0x5EED + 2, all omni
    if (ctx->LastStatus != FS_OK) { printf("UpdateSources (omni) failed: %s\n", ctx->LastError().c_str()); return 4; }
    return print_sums(ctx, "omni");
}
