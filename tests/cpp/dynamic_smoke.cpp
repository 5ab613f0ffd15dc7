// Moving geometry through the C++ mirror (include/frequensee.hpp): a door actor is swung with MoveGeometry between two
// updates (UpdateSource refits the device BVH), and the result is compared with a second mirror on its own context that
// registered the door at its final position from the start (one full build).  Same seed: the impulse responses and the
// connected-path counts must be identical.  Prints one line of key=value pairs for tests/test_gpu_dynamic_scene.py.
#include <cmath>
#include <cstdio>
#include <cstring>
#include <vector>
#include "frequensee.hpp"

using namespace FrequenSee;

// axis-aligned box as 12 triangles
static std::vector<float> Box(const float lo[3], const float hi[3])
{
    const float c[8][3] = {{lo[0], lo[1], lo[2]}, {hi[0], lo[1], lo[2]}, {hi[0], hi[1], lo[2]}, {lo[0], hi[1], lo[2]},
                           {lo[0], lo[1], hi[2]}, {hi[0], lo[1], hi[2]}, {hi[0], hi[1], hi[2]}, {lo[0], hi[1], hi[2]}};
    const int q[6][4] = {{0, 3, 7, 4}, {1, 2, 6, 5}, {0, 1, 5, 4}, {3, 2, 6, 7}, {0, 1, 2, 3}, {4, 5, 6, 7}};
    std::vector<float> t;
    for (auto& f : q)
        for (int k : {0, 1, 2, 0, 2, 3}) t.insert(t.end(), c[f[k]], c[f[k]] + 3);
    return t;
}

// the door (a 4 cm slab in the doorway) rotated by Deg about its hinge, the vertical line (6.1, 3.5)
static std::vector<float> Door(double Deg)
{
    const float lo[3] = {6.08f, 3.5f, 0.0f}, hi[3] = {6.12f, 4.5f, 2.1f};
    std::vector<float> t = Box(lo, hi);
    const double a = Deg * 3.14159265358979323846 / 180.0, ca = std::cos(a), sa = std::sin(a);
    if (Deg != 0.0)
        for (size_t v = 0; v < t.size(); v += 3) {
            const double dx = t[v] - 6.1, dy = t[v + 1] - 3.5;
            t[v] = (float)(6.1 + dx * ca + dy * sa);
            t[v + 1] = (float)(3.5 - dx * sa + dy * ca);
        }
    return t;
}

// two 6 x 8 x 3 m rooms joined by a 1 x 2.1 m doorway: the shell, the dividing wall (three boxes around the opening), the door
static void Register(UAudioRayTracingSubsystem& Sub, double DoorDeg)
{
    FAcousticMaterial plaster; plaster.Absorption.assign(8, 0.05f);
    FAcousticMaterial carpet; carpet.Absorption.assign(8, 0.4f);
    FAcousticMaterial wood; wood.Absorption.assign(8, 0.1f);
    const float s0[3] = {0, 0, -0.1f}, s1[3] = {12.2f, 8, 0};
    std::vector<float> floor_ = Box(s0, s1);
    Sub.RegisterGeometry(floor_.data(), floor_.size() / 9, carpet);
    std::vector<float> shell;
    const float boxes[5][2][3] = {{{-0.1f, 0, 0}, {0, 8, 3}}, {{12.2f, 0, 0}, {12.3f, 8, 3}}, {{0, -0.1f, 0}, {12.2f, 0, 3}},
                                  {{0, 8, 0}, {12.2f, 8.1f, 3}}, {{0, 0, 3}, {12.2f, 8, 3.1f}}};
    for (auto& b : boxes) { std::vector<float> t = Box(b[0], b[1]); shell.insert(shell.end(), t.begin(), t.end()); }
    const float w[3][2][3] = {{{6, 0, 0}, {6.2f, 3.5f, 3}}, {{6, 4.5f, 0}, {6.2f, 8, 3}}, {{6, 3.5f, 2.1f}, {6.2f, 4.5f, 3}}};
    for (auto& b : w) { std::vector<float> t = Box(b[0], b[1]); shell.insert(shell.end(), t.begin(), t.end()); }
    Sub.RegisterGeometry(shell.data(), shell.size() / 9, plaster);
    std::vector<float> door = Door(DoorDeg);
    Sub.RegisterGeometry(door.data(), door.size() / 9, wood);          // actor 2
}

int main()
{
    auto ctx_a = FContext::Create(), ctx_b = FContext::Create();
    if (!ctx_a || !ctx_b) { printf("fs_create failed: %s\n", fs_last_error(nullptr)); return 3; }
    const FVector3f src{2.0f, 2.0f, 1.4f}, lis{10.0f, 6.0f, 1.6f};
    UAudioRayTracingSubsystem a(ctx_a), b(ctx_b);
    Register(a, 0.0);                      // closed
    Register(b, 70.0);                     // open from the start
    UFrequenSeeAudioComponent ca(ctx_a, 0, src), cb(ctx_b, 0, src);
    for (auto* c : {&ca, &cb}) { c->RaycastsPerTick = 1 << 16; c->RaycastBounces = 12; }
    a.RegisterSource(&ca); b.RegisterSource(&cb);
    a.SetPlayerPawnLocation(lis); b.SetPlayerPawnLocation(lis);
    a.Seed = 7;
    a.ForceUpdateSources();                // full build, door closed
    if (ctx_a->LastStatus != FS_OK) { printf("update failed: %s\n", ctx_a->LastError().c_str()); return 4; }
    const uint64_t closed_connected = a.LastConnected;
    std::vector<float> closed_ir = ca.GetImpulseResponse()[0];
    // swing the door open over a few ticks, then compare the last tick with the mirror built open
    for (double deg : {20.0, 45.0, 70.0}) {
        std::vector<float> door = Door(deg);
        if (!a.MoveGeometry(2, door.data())) { printf("MoveGeometry refused\n"); return 5; }
        a.Seed = 9;
        a.ForceUpdateSources();            // refit
        if (ctx_a->LastStatus != FS_OK) { printf("update failed: %s\n", ctx_a->LastError().c_str()); return 6; }
    }
    b.Seed = 9;
    b.ForceUpdateSources();
    if (ctx_b->LastStatus != FS_OK) { printf("update failed: %s\n", ctx_b->LastError().c_str()); return 7; }
    const auto& ia = ca.GetImpulseResponse();
    const auto& ib = cb.GetImpulseResponse();
    bool same = a.LastConnected == b.LastConnected;
    for (size_t c = 0; c < ia.size(); ++c) same = same && std::memcmp(ia[c].data(), ib[c].data(), sizeof(float) * ia[c].size()) == 0;
    double diff = 0;
    for (size_t i = 0; i < closed_ir.size(); ++i) diff += std::fabs((double)closed_ir[i] - ia[0][i]);
    printf("same=%d connected_open=%llu connected_ref=%llu connected_closed=%llu closed_differs=%d refits=%llu rebuilds=%llu ratio=%.6f\n",
           (int)same, (unsigned long long)a.LastConnected, (unsigned long long)b.LastConnected,
           (unsigned long long)closed_connected, (int)(diff > 0), (unsigned long long)a.Refits, (unsigned long long)a.Rebuilds,
           a.LastCostRatio);
    return 0;
}
