// frequensee.hpp -- C++ host-side mirror of the reference's interface for this path, over the C-ABI
// (include/frequensee.h).  Header-only, no Unreal dependency.  Same method names, argument meaning and
// (lack of) error behaviour as the reference classes, so a UE shim is a thin forwarding layer
// (INTEGRATION.md) and the tests read like the reference's call sites:
//
//   UFrequenSeeAudioComponent   COMP.h:19-154   EnergyBuffer, FlushEnergyBuffer, AddEnergyAtDelay,
//                                               ReconstructImpulseResponse, GetImpulseResponse
//   UAudioRayTracingSubsystem   SUB.h:86-197    RegisterGeometry, RegisterSource, UnregisterSource,
//                                               UpdateSource, ForceUpdateSources
//   FFrequenSeeAudioReverbPlugin REV.h:26-83    Initialize, OnInitSource, OnReleaseSource, ProcessSourceAudio
//
// The reference returns void everywhere and logs (SURVEY.md section 8b "Error convention"); here every
// method returns void too and failures are kept in LastStatus()/LastError() (never thrown), except the
// constructor helpers which return nullptr on failure.
#pragma once

#include <cmath>
#include <cstdint>
#include <cstring>
#include <memory>
#include <string>
#include <vector>

#include "frequensee.h"

namespace FrequenSee {

struct FVector3f { float X, Y, Z; };

// UAcousticMaterial (MAT.h:16-34): per-band absorption; Transmission / Scattering / ThicknessCm are part of the
// asset but no tracer of the reference reads them (SURVEY 8a/A10), they are carried and ignored.
struct FAcousticMaterial {
    std::vector<float> Absorption;     // [B]
    std::vector<float> Transmission, Scattering;
    float ThicknessCm = 2.5f;
};

class FContext {
public:
    static std::shared_ptr<FContext> Create(const fs_config* Config = nullptr)
    {
        fs_config c;
        if (Config) c = *Config; else fs_default_config(&c);
        fs_ctx* h = nullptr;
        if (fs_create(&c, &h) != FS_OK) return nullptr;
        return std::shared_ptr<FContext>(new FContext(h, c));
    }
    ~FContext() { fs_destroy(Handle); }
    fs_ctx* Get() const { return Handle; }
    const fs_config& Config() const { return Cfg; }
    int LastStatus = FS_OK;
    std::string LastError() const { const char* e = fs_last_error(Handle); return e ? e : ""; }
    int Check(int rc) { LastStatus = rc; return rc; }
private:
    FContext(fs_ctx* h, const fs_config& c) : Handle(h), Cfg(c) {}
    fs_ctx* Handle;
    fs_config Cfg;
};

// ---- UFrequenSeeAudioComponent (the contract object, COMP.h) --------------------------------------------------
class UFrequenSeeAudioComponent {
public:
    UFrequenSeeAudioComponent(std::shared_ptr<FContext> InCtx, uint32_t InSourceId, FVector3f InLocation)
        : Ctx(std::move(InCtx)), SourceId(InSourceId), Location(InLocation)
    {
        NumBins = (int)Ctx->Config().n_bins;                       // COMP.h:137-138
        SampleRate = (int)Ctx->Config().sample_rate;               // COMP.h:133
        NumChannels = (int)Ctx->Config().n_channels;               // COMP.h:135
        BinSizeMs = Ctx->Config().bin_ms;                          // COMP.h:72
        ImpulseBuffer.assign(NumChannels, std::vector<float>(SampleRate, 0.0f));   // COMP.h:143
        FlushEnergyBuffer();
    }
    // tunables (COMP.h:35-66)
    bool bApplyReverb = true;
    int RaycastsPerTick = 1 << 20;     // path pairs per update (reference USED_RAY_COUNT = 1000, SUB.h:176)
    int RaycastBounces = 16;           // max depth (reference RaycastBounces = 10 / unbounded RR)
    // weight of this emitter when UAudioRayTracingSubsystem::TotalRaysPerTick is split (fs_allocate_paths): a source of
    // weight 2 is given twice the SNR of one of weight 1; 0 = as few rays as the bounds allow
    float NoiseWeight = 1.0f;
    // FS_FLAG_NOISE_STATS: the noise of this source in the last UpdateSources() (fs_get_noise; n_paths = the budget it had)
    fs_noise_stats LastNoise{};

    std::vector<float> EnergyBuffer;   // COMP.h:70
    void FlushEnergyBuffer() { EnergyBuffer.assign(NumBins, 0.0f); bUseDeviceHistogram = false; }          // COMP.h:76-79
    void AddEnergyAtDelay(float DelaySeconds, float EnergyValue)                                            // COMP.h:87-91
    {
        int BinIndex = (int)std::floor((DelaySeconds * 1000.f) / BinSizeMs);
        if (BinIndex < 0) BinIndex = 0;
        if (BinIndex > NumBins - 1) BinIndex = NumBins - 1;
        EnergyBuffer[BinIndex] += EnergyValue;
    }
    // COMP.cpp:320-380.  Uses the device histogram left by UAudioRayTracingSubsystem::UpdateSource when there is
    // one, else the float EnergyBuffer filled through AddEnergyAtDelay (seam 1 of the reference taken literally).
    void ReconstructImpulseResponse()
    {
        std::vector<float> flat((size_t)NumChannels * SampleRate);
        int rc = bUseDeviceHistogram ? fs_build_ir_to(Ctx->Get(), 0, SourceId, flat.data())
                                     : fs_build_ir_from_energy(Ctx->Get(), SourceId, EnergyBuffer.data(), flat.data());
        if (Ctx->Check(rc) != FS_OK) return;
        for (int c = 0; c < NumChannels; ++c)
            std::memcpy(ImpulseBuffer[c].data(), flat.data() + (size_t)c * SampleRate, sizeof(float) * SampleRate);
    }
    // per-band synthesis from the device histogram (extends COMP.cpp:337-378; fs_build_ir_bands)
    void ReconstructImpulseResponsePerBand(uint64_t NoiseSeed)
    {
        std::vector<float> flat((size_t)NumChannels * SampleRate);
        if (Ctx->Check(fs_build_ir_bands(Ctx->Get(), 0, SourceId, NoiseSeed, flat.data())) != FS_OK) return;
        for (int c = 0; c < NumChannels; ++c)
            std::memcpy(ImpulseBuffer[c].data(), flat.data() + (size_t)c * SampleRate, sizeof(float) * SampleRate);
    }
    std::vector<std::vector<float>>& GetImpulseResponse() { return ImpulseBuffer; }                         // COMP.h:113
    // COMP.cpp:454-490: one float per line into Data (resized to the file's length)
    static bool LoadFloatArray(const std::string& FilePath, std::vector<float>& Data)
    {
        uint64_t n = 0;
        if (fs_load_float_array(FilePath.c_str(), nullptr, 0, &n) != FS_OK) return false;
        Data.resize((size_t)n);
        return fs_load_float_array(FilePath.c_str(), Data.data(), n, &n) == FS_OK;
    }
    // COMP.cpp:492-505
    static bool SaveArrayToFile(const std::vector<float>& Array, const std::string& FilePath)
    {
        return fs_save_float_array(FilePath.c_str(), Array.data(), Array.size()) == FS_OK;
    }
    // a loaded saved_ir.txt becomes this component's IR on both channels and is published to its convolver
    bool UseImpulseResponse(const std::vector<float>& Mono)
    {
        if ((int)Mono.size() != SampleRate) return false;
        std::vector<float> flat((size_t)NumChannels * SampleRate);
        for (int c = 0; c < NumChannels; ++c) {
            ImpulseBuffer[c] = Mono;
            std::memcpy(flat.data() + (size_t)c * SampleRate, Mono.data(), sizeof(float) * SampleRate);
        }
        return Ctx->Check(fs_set_ir(Ctx->Get(), SourceId, flat.data())) == FS_OK;
    }
    FVector3f GetActorLocation() const { return Location; }
    void SetActorLocation(FVector3f L) { Location = L; }
    uint32_t GetSourceId() const { return SourceId; }

    int SampleRate, NumChannels, NumBins;
    float BinSizeMs;
    std::vector<std::vector<float>> ImpulseBuffer;
    bool bUseDeviceHistogram = false;
private:
    std::shared_ptr<FContext> Ctx;
    uint32_t SourceId;
    FVector3f Location;
};

// ---- UAudioRayTracingSubsystem (SUB.h) ---------------------------------------------------------------------------
class UAudioRayTracingSubsystem {
public:
    explicit UAudioRayTracingSubsystem(std::shared_ptr<FContext> InCtx) : Ctx(std::move(InCtx)) {}

    // RegisterGeometry (SUB.h:99-100): one call per tagged actor = a triangle soup + its UAcousticMaterial.  Actors are
    // numbered in registration order (the ActorIndex of MoveGeometry).
    void RegisterGeometry(const float* Triangles /*[n][3][3] metres*/, uint64_t NumTriangles, const FAcousticMaterial& Material)
    {
        uint32_t id = (uint32_t)Materials.size();
        Materials.push_back(Material);
        Ranges.push_back({(uint64_t)TriMaterial.size(), NumTriangles});
        Moved.push_back(false);
        Verts.insert(Verts.end(), Triangles, Triangles + NumTriangles * 9);
        TriMaterial.insert(TriMaterial.end(), NumTriangles, id);
        bDirty = true;
    }
    // An actor moved (the reference's scene query sees WorldDynamic actors at their current transform, SUB.cpp:331-334):
    // its world-space triangles, same count as registered.  Takes effect at the next update: a refit of the device BVH
    // (fs_scene_update_vertices + fs_scene_refit), or a full rebuild once the refitted tree has degraded past
    // RebuildCostRatio.  Returns false for an unknown actor.
    bool MoveGeometry(uint32_t ActorIndex, const float* Triangles /*[n][3][3] metres*/)
    {
        if (ActorIndex >= Ranges.size()) return false;
        std::memcpy(Verts.data() + Ranges[ActorIndex].First * 9, Triangles, sizeof(float) * 9 * Ranges[ActorIndex].Count);
        Moved[ActorIndex] = true;
        return true;
    }
    // surface-area cost of the refitted tree over that of the last full build, above which Commit() rebuilds (DESIGN.md
    // section 3, "Moving geometry": measured trace time against this ratio)
    float RebuildCostRatio = 1.5f;
    float LastCostRatio = 1.0f;        // after the last refit (1 after a rebuild)
    uint64_t Refits = 0, Rebuilds = 0;
    void RegisterSource(UFrequenSeeAudioComponent* Src) { ActiveSources.push_back(Src); }                     // SUB.h:102
    void UnregisterSource(UFrequenSeeAudioComponent* Src)                                                      // SUB.h:103
    {
        for (size_t i = 0; i < ActiveSources.size(); ++i)
            if (ActiveSources[i] == Src) { ActiveSources.erase(ActiveSources.begin() + i); break; }
    }
    void SetPlayerPawnLocation(FVector3f L) { PawnLocation = L; }                                              // SUB.cpp:70-80
    uint64_t Seed = 0x5EED;

    // UpdateSource (SUB.cpp:128-195): GenerateFullPaths + EvaluatePath + Flush + AddEnergyAtDelay (on the
    // device, integer) + ReconstructImpulseResponse.  FIX: no second flush before the IR (SUB.cpp:191).
    void UpdateSource(UFrequenSeeAudioComponent& Src)
    {
        if (!Commit()) return;
        const FVector3f S = Src.GetActorLocation();
        const float src[3] = {S.X, S.Y, S.Z}, lis[3] = {PawnLocation.X, PawnLocation.Y, PawnLocation.Z};
        // one source per call: the device histogram of source slot 0 belongs to Src until the next update
        if (Ctx->Check(fs_trace(Ctx->Get(), src, 1, lis, (uint64_t)Src.RaycastsPerTick, (uint32_t)Src.RaycastBounces,
                                Seed++, nullptr)) != FS_OK) return;
        fs_stats st;
        if (fs_get_stats(Ctx->Get(), &st) == FS_OK) LastConnected = st.connected;   // "%d paths connected out of %d", SUB.cpp:232
        std::vector<float> flat((size_t)Src.NumChannels * Src.SampleRate);
        // histogram slot 0 of this trace -> the component's own convolver slot
        if (Ctx->Check(fs_build_ir_to(Ctx->Get(), 0, Src.GetSourceId(), flat.data())) != FS_OK) return;
        for (int c = 0; c < Src.NumChannels; ++c)
            std::memcpy(Src.ImpulseBuffer[c].data(), flat.data() + (size_t)c * Src.SampleRate, sizeof(float) * Src.SampleRate);
        Src.bUseDeviceHistogram = true;
    }
    void ForceUpdateSources() { for (auto* s : ActiveSources) UpdateSource(*s); }                              // SUB.cpp:883-886
    // Every active source in ONE trace, each with its own RaycastsPerTick and RaycastBounces (COMP.h:35-66): histogram slot
    // s belongs to ActiveSources[s] until the next update, and each IR is published to its component's own convolver slot.
    // The random streams differ from UpdateSource's (one flat work range over all sources, fs_trace_sources), so this is
    // a separate entry point; ForceUpdateSources keeps the reference's one-update-per-source sequence.
    //
    // Automatic budgets (the allocateSamples the reference declares, SUB.h:136, and never defines): with TotalRaysPerTick > 0
    // on a context created with FS_FLAG_NOISE_STATS, the components' RaycastsPerTick are ignored and TotalRaysPerTick is
    // split over the active sources, each between MinRaysPerSource and MaxRaysPerSource (0 = TotalRaysPerTick).  The first
    // update, and the first after the set of active sources has changed, splits it equally; every later one splits it with
    // fs_allocate_paths from the noise of the previous update (each component's LastNoise) and its NoiseWeight.
    // RaycastBounces stays per component.  A split the bounds make impossible fails the update (FS_ERR_INVALID in
    // Ctx->LastStatus).
    uint64_t TotalRaysPerTick = 0;     // 0: every source traces its own RaycastsPerTick
    uint64_t MinRaysPerSource = 1024, MaxRaysPerSource = 0;
    void UpdateSources()
    {
        if (ActiveSources.empty() || !Commit()) return;
        const float lis[3] = {PawnLocation.X, PawnLocation.Y, PawnLocation.Z};
        const uint32_t S = (uint32_t)ActiveSources.size();
        const bool noise = (Ctx->Config().flags & FS_FLAG_NOISE_STATS) != 0;
        std::vector<uint64_t> budget(S);
        for (uint32_t s = 0; s < S; ++s) budget[s] = (uint64_t)ActiveSources[s]->RaycastsPerTick;
        if (noise && TotalRaysPerTick > 0 && !SplitTotal(budget)) return;
        std::vector<fs_source_desc> desc(S);
        for (uint32_t s = 0; s < S; ++s) {
            const UFrequenSeeAudioComponent& c = *ActiveSources[s];
            const FVector3f L = c.GetActorLocation();
            desc[s].pos[0] = L.X; desc[s].pos[1] = L.Y; desc[s].pos[2] = L.Z;
            desc[s].max_depth = (uint32_t)c.RaycastBounces;
            desc[s].n_paths = budget[s];
        }
        NoiseSources.clear();
        if (Ctx->Check(fs_trace_sources(Ctx->Get(), desc.data(), S, lis, Seed++, nullptr)) != FS_OK) return;
        fs_stats st;
        if (fs_get_stats(Ctx->Get(), &st) == FS_OK) LastConnected = st.connected;
        if (noise) {
            std::vector<fs_noise_stats> ns(S);
            if (Ctx->Check(fs_get_noise(Ctx->Get(), ns.data(), S)) != FS_OK) return;
            for (uint32_t s = 0; s < S; ++s) ActiveSources[s]->LastNoise = ns[s];
            NoiseSources = ActiveSources;
        }
        for (size_t s = 0; s < ActiveSources.size(); ++s) {
            UFrequenSeeAudioComponent& c = *ActiveSources[s];
            std::vector<float> flat((size_t)c.NumChannels * c.SampleRate);
            if (Ctx->Check(fs_build_ir_to(Ctx->Get(), (uint32_t)s, c.GetSourceId(), flat.data())) != FS_OK) return;
            for (int ch = 0; ch < c.NumChannels; ++ch)
                std::memcpy(c.ImpulseBuffer[ch].data(), flat.data() + (size_t)ch * c.SampleRate, sizeof(float) * c.SampleRate);
            c.bUseDeviceHistogram = true;
        }
    }
    uint64_t LastConnected = 0;

private:
    // TotalRaysPerTick over the active sources: equally, or by fs_allocate_paths from the last update's noise when it
    // belongs to the same sources
    bool SplitTotal(std::vector<uint64_t>& budget)
    {
        const uint32_t S = (uint32_t)budget.size();
        const uint64_t lo = MinRaysPerSource, hi = MaxRaysPerSource ? MaxRaysPerSource : TotalRaysPerTick;
        if (NoiseSources == ActiveSources) {
            std::vector<fs_noise_stats> ns(S);
            std::vector<float> w(S);
            for (uint32_t s = 0; s < S; ++s) { ns[s] = ActiveSources[s]->LastNoise; w[s] = ActiveSources[s]->NoiseWeight; }
            return Ctx->Check(fs_allocate_paths(ns.data(), S, TotalRaysPerTick, lo, hi, w.data(), budget.data())) == FS_OK;
        }
        // equal split: fs_allocate_paths with the same demand everywhere
        std::vector<fs_noise_stats> eq(S);
        for (uint32_t s = 0; s < S; ++s) { eq[s] = fs_noise_stats{}; eq[s].n_paths = 1; eq[s].signal = 1.0; eq[s].variance = 1.0; }
        return Ctx->Check(fs_allocate_paths(eq.data(), S, TotalRaysPerTick, lo, hi, nullptr, budget.data())) == FS_OK;
    }
    std::vector<UFrequenSeeAudioComponent*> NoiseSources;   // the sources whose LastNoise the last update filled
    bool Commit()
    {
        if (!bDirty) return CommitMoves();
        const uint32_t B = Ctx->Config().n_bands;
        std::vector<float> ab(Materials.size() * B, 0.0f);
        for (size_t m = 0; m < Materials.size(); ++m)
            for (uint32_t b = 0; b < B; ++b)
                ab[m * B + b] = b < Materials[m].Absorption.size() ? Materials[m].Absorption[b] : 0.0f;
        if (Ctx->Check(fs_scene_set_triangles(Ctx->Get(), Verts.data(), TriMaterial.data(), TriMaterial.size())) != FS_OK) return false;
        if (Ctx->Check(fs_scene_set_materials(Ctx->Get(), ab.data(), (uint32_t)Materials.size(), B)) != FS_OK) return false;
        if (Ctx->Check(fs_scene_commit(Ctx->Get())) != FS_OK) return false;
        bDirty = false;
        Moved.assign(Moved.size(), false);
        LastCostRatio = 1.0f;
        ++Rebuilds;
        return true;
    }
    // moves only (topology unchanged): one fs_scene_update_vertices per moved actor, one refit
    bool CommitMoves()
    {
        bool any = false;
        for (size_t a = 0; a < Ranges.size(); ++a) {
            if (!Moved[a]) continue;
            if (Ctx->Check(fs_scene_update_vertices(Ctx->Get(), Verts.data() + Ranges[a].First * 9, Ranges[a].First,
                                                    Ranges[a].Count)) != FS_OK) return false;
            Moved[a] = false;
            any = true;
        }
        if (!any) return true;
        float ratio = 1.0f;
        if (Ctx->Check(fs_scene_refit(Ctx->Get(), &ratio)) != FS_OK) return false;
        ++Refits;
        LastCostRatio = ratio;
        if (ratio > RebuildCostRatio) {
            if (Ctx->Check(fs_scene_commit(Ctx->Get())) != FS_OK) return false;
            LastCostRatio = 1.0f;
            ++Rebuilds;
        }
        return true;
    }
    struct FRange { uint64_t First, Count; };
    std::vector<FRange> Ranges;        // per registered actor: its triangles in the scene
    std::vector<bool> Moved;
    std::shared_ptr<FContext> Ctx;
    std::vector<float> Verts;
    std::vector<uint32_t> TriMaterial;
    std::vector<FAcousticMaterial> Materials;
    std::vector<UFrequenSeeAudioComponent*> ActiveSources;
    FVector3f PawnLocation{0.f, 0.f, 0.f};
    bool bDirty = true;
};

// ---- FFrequenSeeAudioReverbPlugin (REV.h:26-83, IAudioReverb) -----------------------------------------------------
struct FAudioPluginInitializationParams { uint32_t NumSources; uint32_t NumOutputChannels; uint32_t SampleRate; uint32_t BufferLength; };

class FFrequenSeeAudioReverbPlugin {
public:
    explicit FFrequenSeeAudioReverbPlugin(std::shared_ptr<FContext> InCtx) : Ctx(std::move(InCtx)) {}
    void Initialize(const FAudioPluginInitializationParams P)                                                  // REV.cpp:74-102
    {
        SamplingRate = (int)P.SampleRate; FrameSize = (int)P.BufferLength;
        bValid = (P.SampleRate == Ctx->Config().sample_rate && P.BufferLength == Ctx->Config().conv_block);
    }
    void OnInitSource(uint32_t SourceId, uint32_t /*NumChannels*/) { Ctx->Check(fs_conv_init_source(Ctx->Get(), SourceId)); }      // REV.cpp:104-110
    void OnReleaseSource(uint32_t SourceId) { Ctx->Check(fs_conv_release_source(Ctx->Get(), SourceId)); }                           // REV.cpp:112-116
    // ProcessSourceAudio (REV.cpp:118-170): interleaved stereo in, interleaved stereo out; bApplyReverb == false -> passthrough
    void ProcessSourceAudio(const UFrequenSeeAudioComponent& Src, const float* InAudioBuffer, float* OutAudioBuffer)
    {
        if (!bValid) return;
        if (!Src.bApplyReverb) {                                                                                // REV.cpp:128-133
            std::memcpy(OutAudioBuffer, InAudioBuffer, sizeof(float) * FrameSize * Ctx->Config().n_channels);
            return;
        }
        Ctx->Check(fs_conv_process(Ctx->Get(), Src.GetSourceId(), InAudioBuffer, OutAudioBuffer, (uint32_t)FrameSize));
    }
private:
    std::shared_ptr<FContext> Ctx;
    int SamplingRate = 0, FrameSize = 0;
    bool bValid = false;
};

}  // namespace FrequenSee
