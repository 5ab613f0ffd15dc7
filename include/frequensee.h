/*
 * frequensee.h -- C-ABI of the B200-native FrequenSee propagation core.
 *
 * Drop-in boundary for ONE path of henreedev/audio-pathtracer: the per-frame BDPT sound
 * propagation update, its impulse-response stage and the FFT convolution.  Plain pointers and
 * sizes only: no Unreal types, no torch types.  Every entry point cites the reference
 * interface it replaces (paths relative to Plugins/FrequenSee/Source/FrequenSee/):
 *
 *   SUB.h/.cpp = Public/AudioRayTracingSubsystem.h, Private/AudioRayTracingSubsystem.cpp
 *   COMP.h/.cpp = Public/FrequenSeeAudioComponent.h, Private/FrequenSeeAudioComponent.cpp
 *   REV.h/.cpp  = Private/FrequenSeeAudioReverbPlugin.{h,cpp}
 *   GEO.h, MAT.h = Public/AcousticGeometryComponent.h, Public/AcousticMaterial.h
 *
 * Error convention: every function returns fs_status (0 = OK, negative = error);
 * fs_last_error(ctx) returns a human-readable message for the last failure ON THE CALLING THREAD
 * (thread-local: the game thread and the audio thread use one context concurrently).
 * Nothing throws across this boundary.  There is NO CPU fallback: if no CUDA device is usable
 * fs_create fails with FS_ERR_CUDA.
 *
 * Threading: fs_scene_*, fs_trace*, fs_build_ir*, fs_set_*, fs_get_* from one thread at a time
 * per context (the reference's game thread, SUB.cpp:55).  fs_conv_init_source /
 * fs_conv_release_source / fs_conv_process* may be called concurrently from other threads (the
 * reference's audio render thread and its source workers, REV.cpp:118): they run on a stream of
 * their own and never queue behind a trace.  The IR hand-off between the two is a
 * double-buffered set of partition spectra: an IR update writes the unpublished buffer on the
 * game thread's stream, and the convolver adopts it at the first callback (block boundary)
 * that finds the update complete -- a callback never waits for an update that is still being
 * computed, it keeps the previous IR (the reference shares ImpulseBuffer with no
 * synchronisation, COMP.cpp:378 vs REV.cpp:136).  With FS_FLAG_CONV_CROSSFADE the set is
 * triple-buffered: the published buffer, the buffer the source's last callback ended with
 * ("heard", which the next callback fades from) and the one an update writes, which is never
 * either of the other two.  An update is guaranteed to be in effect for
 * callbacks issued after a host-synchronising call of the game thread has returned
 * (fs_build_ir* with ir_out, fs_set_ir, fs_synchronize).  While at least one convolver source
 * is initialised, fs_trace* keeps to short kernels (one per bounce) so that a callback is
 * placed between two of them (measured p99 0.3 ms beside 5 ms updates); with no source
 * active, a large update runs as one persistent kernel per batch (5 % faster, but it holds
 * every SM for milliseconds).
 *
 * Ownership: the caller owns every host buffer passed in or out; the library copies at call
 * time and retains nothing.  Device memory is owned by the context.
 */
#ifndef FREQUENSEE_H
#define FREQUENSEE_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FS_MAX_BANDS 8

typedef enum fs_status {
    FS_OK = 0,
    FS_ERR_INVALID = -1,      /* bad argument / bad call order */
    FS_ERR_CUDA = -2,         /* CUDA runtime failure (message has the CUDA error string) */
    FS_ERR_NOMEM = -3,
    FS_ERR_STATE = -4,        /* e.g. fs_trace before fs_scene_commit */
    FS_ERR_OVERFLOW = -5      /* traversal stack overflow (BVH deeper than the kernel supports): the histogram of that trace is
                                 incomplete.  Reported by the trace call itself when it returns host data, otherwise by the
                                 next call on the context that can see the flag (fs_build_ir*, fs_trace*, fs_synchronize,
                                 fs_get_*) */
} fs_status;

/* flags for fs_config.flags */
#define FS_FLAG_COUNT_VISITS   1u   /* instrumented traversal: count BVH nodes popped / triangles tested */
#define FS_FLAG_NO_SPLAT_AGG   2u   /* plain one-atomic-per-lane splat instead of warp-aggregated */
#define FS_FLAG_SMEM_TREELET   4u   /* fused path only: stage the top BVH treelet in shared memory */
#define FS_FLAG_BRUTE_FORCE    8u   /* test every triangle (debug/parity only, tiny scenes) */
#define FS_FLAG_TIME_KERNELS  16u   /* CUDA events around each kernel class -> fs_stats.*_ms */
#define FS_FLAG_CONNECT_ALL   64u   /* SURVEY 8f rank 1: connect every source prefix s with every listener prefix t (the reference's
                                       unfinished Is_NaiveConnections, SUB.cpp:508-535), each connected path evaluated like the
                                       endpoint connection and weighted 1 / (s + t - 1); (1, 1) is the deterministic direct path.
                                       Up to (depth+1)^2 connection rays per pair: batches shrink to ~2^24 / (depth+1)^2 pairs */
#define FS_FLAG_MIS           512u   /* SURVEY 8f rank 1, second half: all prefix connections (as FS_FLAG_CONNECT_ALL) combined with the
                                       BALANCE HEURISTIC -- what the reference's unfinished getPdf / getExpectedWeight / MISEnergy aim
                                       at (SUB.cpp:537-597).  MIS needs one integrand for all strategies, which the reference's
                                       per-segment product (no cosines, pdf^0.1) is not: this mode evaluates the physically based
                                       contribution 1/(4 pi) prod_edges [cos cos / d^2 exp(-air d)] prod_vertices [rho / pi] and each
                                       visible connection (s, t) contributes f / sum_s' p_s' (area-measure densities of the walks).
                                       energy_clamp / energy_gain still apply (set 1e30 / 1 for physical units); pdf_exponent is unused;
                                       max_depth <= 32; diffuse surfaces only */
#define FS_FLAG_SHARE_LISTENER 128u  /* SURVEY 8f rank 4: the listener subpath of pair (source, i) is keyed by i only, so all
                                       sources of a multi-emitter update share one set of listener subpaths, traced once per
                                       fs_trace call (the reference regenerates it per source, SUB.cpp:215-230: different
                                       random numbers, hence a separate mode).  Nearly halves the rays of BASELINE configs[3] */
#define FS_FLAG_MATERIAL_MODEL 256u /* SURVEY 8f rank 3: the Transmission / Scattering / ThicknessCm fields of the material asset
                                       (MAT.h:26-33, set with fs_scene_set_materials_ex) drive the walk: at a surface the ray passes
                                       through (COMP.cpp:271-275), is mirrored (GetReflectionVector, COMP.cpp:186) or is scattered into
                                       the cosine lobe, with the authors' own energy split (MaterialAcousticProcessor.cpp:50-66:
                                       Refl = 1 - alpha, tau <= 1 - Refl, specular Refl (1 - sigma), diffuse Refl sigma, transmitted
                                       tau ^ (ThicknessCm / 2.5)).  Off by default: the reference's tracers read Absorption only */
#define FS_FLAG_IR_NORMALIZE 1024u  /* every IR that is built is scaled to unit L2 norm per channel before it is published to the
                                       convolver / returned: the normalisation the reference computes in NormalizeImpulseResponse
                                       (COMP.cpp:382-406) and then discards (":404 FIXME", :377-378).  A channel whose norm is below
                                       KINDA_SMALL_NUMBER (1e-4) is left alone (:394-397).  Off by default = the reference's effective
                                       behaviour */
#define FS_FLAG_CONV_CROSSFADE 2048u /* click-free IR updates in the convolver: a callback that adopts a newly published IR
                                       fades over its first block from the IR the source's previous callback ended with
                                       ("heard") to the new one:  y = (1 - w[i]) (history (*) IR_heard) + w[i] (history (*) IR_new),
                                       w[i] = 0.5 - 0.5 cos(pi (i+1) / conv_block), taken before clamp and wet/dry mix.  IRs
                                       published between two callbacks are skipped (the fade goes to the newest); every
                                       adoption fades, even of an identical IR; only block 0 of fs_conv_process_many can fade;
                                       the first callback after fs_conv_init_source never fades.  Costs a third set of
                                       partition spectra per source; a fade block reads 1.5x the spectra and runs one more
                                       inverse FFT.  Off by default: the IR switches at the block boundary */
#define FS_FLAG_NOISE_STATS  4096u  /* Monte Carlo noise of every update (fs_get_noise): the splat also accumulates the exact
                                       square of every path's Q32.32 value, per band q_b^2 and broadband (sum_b q_b)^2, into
                                       a 128-bit second-moment buffer [S][B+1][K] (fs_get_histogram_m2).  Each pair adds at
                                       most one path in the endpoint-connection mode, so the moments give an unbiased
                                       per-bin variance; sums are exact mod 2^128 (bit-identical for every batch split and
                                       device count) and cannot wrap below 2^128 / (B clamp gain 2^32)^2 pairs per bin:
                                       2^51 with the defaults (B = 8, clamp x gain = 10).  The statistics are exact as
                                       long as the histogram itself does not wrap: 2^64 / (clamp gain 2^32) pairs in one
                                       bin of a band, 2^28.7 with the defaults (the broadband sum is formed in 128 bits).
                                       The histogram itself is unchanged.  fs_create rejects it together with FS_FLAG_CONNECT_ALL / FS_FLAG_MIS,
                                       where one pair adds to several bins.  Off by default: the splat is the plain one */
#define FS_FLAG_FUSED_EXTEND  32u   /* A/B: fused RR+sample+traverse+shade kernel per bounce instead of the
                                       split shade/trace wavefront with per-lane ray replacement */

/* All tunables of the path in one POD: tier (i) UPROPERTYs (COMP.h:35-66) + tier (ii)
 * compile-time constants of the reference (SURVEY.md Appendix A), reference values as defaults
 * (fs_default_config), units converted from UE centimetres to metres. */
typedef struct fs_config {
    uint32_t n_bands;          /* B, 1..8.  Reference reads one band, Absorption[2] (SUB.cpp:385) */
    uint32_t n_bins;           /* K = NumBins = 1000 (COMP.h:137-138) */
    float    bin_ms;           /* BinSizeMs = 1 (COMP.h:72) */
    float    rr_prob;          /* RUSSIAN_ROULETTE_PROB = 0.9 (SUB.cpp:282); 1.0 disables */
    float    eps_offset;       /* ImpactPoint + 0.1 * ImpactNormal (SUB.cpp:345): 1e-3 m */
    float    eps_connect;      /* connection ray stops 0.1 short (SUB.cpp:253): 1e-3 m */
    float    min_seg;          /* "NodeDistance < 1.0 -> continue" glitch guard (SUB.cpp:375): 1e-2 m */
    float    sound_speed;      /* SoundSpeed = 343 (SUB.cpp:362) */
    float    pdf_exponent;     /* powf(Node.Probability, 0.1) (SUB.cpp:398) */
    float    energy_clamp;     /* FMath::Min(Energy, 1) (SUB.cpp:410) */
    float    energy_gain;      /* Energy *= 10 (SUB.cpp:413) */
    float    air_absorption[FS_MAX_BANDS]; /* per metre per band (AIR_ABSORPTION_FACTOR, SUB.cpp:395) */
    uint32_t sample_rate;      /* SampleRate = 48000 (COMP.h:133) */
    uint32_t n_channels;       /* NumChannels = 2 (COMP.h:135) */
    float    ir_threshold;     /* kEnergyThreshold = 1e-6 (COMP.cpp:322) */
    float    ir_lowpass;       /* FilterCoefficient = 0.25 (COMP.cpp:366) */
    uint32_t conv_block;       /* AudioCallbackBufferFrameSize = 1024 (Config/DefaultEngine.ini:15) */
    uint32_t conv_clamp;       /* clamp to +-1 (REV.cpp:162-168) */
    float    conv_wet;         /* MixAlpha = 1 (REV.cpp:161) */
    uint32_t max_batch_paths;  /* path pairs in flight per wavefront batch; 0 = default (1<<21) */
    uint32_t flags;            /* FS_FLAG_* */
    int32_t  device;           /* CUDA device ordinal; -1 = current device */
} fs_config;

/* counters of the last fs_trace* call; replaces the UE_LOG at SUB.cpp:232
 * ("%d paths connected out of %d") */
typedef struct fs_stats {
    uint64_t paths;
    uint64_t ext_rays;         /* extension rays traced (closest hit) */
    uint64_t shadow_rays;      /* connection rays traced (any hit) */
    uint64_t connected;
    uint64_t node_visits;      /* only with FS_FLAG_COUNT_VISITS: BVH nodes popped, all rays */
    uint64_t tri_tests;        /* only with FS_FLAG_COUNT_VISITS: triangles tested, all rays */
    uint64_t shadow_node_visits; /* the part of node_visits spent on connection rays */
    uint64_t shadow_tri_tests;
    uint64_t kernel_launches;  /* CUDA kernels launched by this context since fs_create */
    uint64_t bvh_nodes;        /* inner nodes of the committed BVH */
    uint64_t bvh_max_leaf;     /* triangles in the largest leaf */
    float    last_trace_ms;    /* device time of the last fs_trace*, CUDA events on the context stream */
    float    last_ir_ms;
    float    extend_ms;        /* only with FS_FLAG_TIME_KERNELS: extension stage (k_shade_gen + k_trace_closest, or k_extend) */
    float    connect_ms;       /*   "   k_connect */
    float    eval_ms;          /*   "   k_eval (evaluate + splat) */
    uint32_t extend_launches;  /* closest-hit traversal launches (k_trace_closest / k_extend) in the last trace */
    float    trace_ms;         /* only with FS_FLAG_TIME_KERNELS: sum over the k_trace_closest launches alone */
    uint32_t persistent_launches; /* of those, launches of the persistent per-batch kernel (k_path_q: every bounce of a batch -- traversal
                                  and shading -- in one launch); 0 = the per-bounce pipeline ran (small jobs, trivial scenes) */
    float    last_conv_ms;     /* device time of the k_conv_blocks launch(es) of the last fs_conv_process* call (CUDA events on the
                                  convolver's stream) */
} fs_stats;

/* per-path debug record, same layout as fso_path_dbg in oracle/fs_oracle.h */
typedef struct fs_path_dbg {
    uint32_t n_src_nodes, n_lis_nodes, connected;
    int32_t  bin;
    float    delay_s, total_dist;
    float    energy[FS_MAX_BANDS];
    float    src_end[3], lis_end[3];
} fs_path_dbg;

typedef struct fs_ctx fs_ctx;

/* ---- lifetime ---------------------------------------------------------------------------
 * replaces: UAudioRayTracingSubsystem construction + FFrequenSeeAudioReverbPlugin::Initialize
 * (REV.cpp:74-102) + plugin registration in StartupModule (MOD.cpp:12-23) */
void        fs_default_config(fs_config* cfg);
int         fs_create(const fs_config* cfg, fs_ctx** out);
void        fs_destroy(fs_ctx* ctx);
const char* fs_last_error(const fs_ctx* ctx);      /* ctx may be NULL: last fs_create failure */
/* run this context's work on an existing CUDA stream (cudaStream_t as void*), e.g. torch's
 * current stream; NULL restores the context's own stream */
int         fs_set_stream(fs_ctx* ctx, void* cuda_stream);
int         fs_synchronize(fs_ctx* ctx);

/* ---- scene -------------------------------------------------------------------------------
 * replaces: UAudioRayTracingSubsystem::RegisterGeometry (SUB.h:99-100), the per-hit
 * H.GetActor()->FindComponentByClass<UAcousticGeometryComponent>() (SUB.cpp:347) and
 * UAcousticMaterial::Absorption (MAT.h:22-24).
 * verts: [T][3][3] float32 metres; tri_material: [T]; absorption: [M][B] in [0,1]. */
int fs_scene_set_triangles(fs_ctx* ctx, const float* verts, const uint32_t* tri_material, uint64_t n_tris);
int fs_scene_set_materials(fs_ctx* ctx, const float* absorption, uint32_t n_materials, uint32_t n_bands);
/* the whole UAcousticMaterial asset (MAT.h:16-34).  Transmission [M][B], Scattering [M][B] and ThicknessCm [M] are validated
 * ([0,1]; thickness >= 0) and kept with the context.  Exactly like the reference's tracers the path tracer ignores them
 * (SURVEY 8a A10) unless the context was created with FS_FLAG_MATERIAL_MODEL (SURVEY 8f rank 3).  Any of the three may be
 * NULL (0, 1, 2.5 cm: a purely diffuse surface -- with these defaults the model reproduces the default mode bit for bit). */
int fs_scene_set_materials_ex(fs_ctx* ctx, const float* absorption, const float* transmission, const float* scattering,
                              const float* thickness_cm, uint32_t n_materials, uint32_t n_bands);
/* builds the BVH on the device: Morton codes, radix sort, PLOC agglomeration (search radius chosen by surface-area cost),
 * 4-wide quantised nodes in a dense breadth-first array.  One-time cost per scene: 0.2 s for 1 M triangles. */
int fs_scene_commit(fs_ctx* ctx);
/* moving geometry.  replaces: the engine's scene query seeing WorldDynamic actors at their current transform
 * (SUB.cpp:331-334: GeneratePath / ConnectSubpaths query Pawn + WorldStatic + WorldDynamic objects, so a door that swings is
 * heard by the next UpdateSource).
 * fs_scene_update_vertices overwrites the positions of triangles [first_tri, first_tri + n_tris) of the scene set by
 * fs_scene_set_triangles (verts: [n_tris][3][3] float metres; same count, same material ids).  Copies at call time,
 * enqueued on the context stream.  FS_ERR_STATE before fs_scene_set_triangles; FS_ERR_INVALID for a range outside the scene
 * or a non-finite / > 1e18 coordinate (checked before anything is copied: a rejected call changes nothing).
 * On a committed scene the positions take effect at the next fs_scene_refit (or fs_scene_commit = full rebuild); until
 * then fs_trace*, fs_update and fs_debug_*_hits return FS_ERR_STATE. */
int fs_scene_update_vertices(fs_ctx* ctx, const float* verts, uint64_t first_tri, uint64_t n_tris);
/* Refits the committed BVH to the current triangle positions: topology kept, every box and triangle record recomputed,
 * the quantisation grid re-derived.  Results are bit-identical to a fresh fs_scene_commit of the same positions (the
 * closest hit does not depend on the tree); only the traversal cost changes as the tree degrades.  FS_ERR_STATE if the
 * scene is not committed.  One host synchronisation (the grid is read back: trace parameters carry it by value).
 * cost_ratio_out (may be NULL): surface-area cost of the refitted BVH2 over that of the tree as committed, so the caller
 * can decide when a full fs_scene_commit pays off.  With the experiment knob FS_TUNE_W8 (8-wide nodes) this is a full
 * fs_scene_commit and the ratio is 1. */
int fs_scene_refit(fs_ctx* ctx, float* cost_ratio_out);

/* ---- BDPT update ---------------------------------------------------------------------------
 * replaces: UAudioRayTracingSubsystem::UpdateSource (SUB.cpp:128-195) = GenerateFullPaths
 * (:201-233) + ConnectSubpaths (:235-277) + EvaluatePath (:360-420) +
 * UFrequenSeeAudioComponent::FlushEnergyBuffer / AddEnergyAtDelay (COMP.h:76-79, 87-91).
 *
 * Traces n_paths path pairs per source (global work index g = source * n_paths + i, Philox
 * stream keyed by (seed, g)) and accumulates Q32.32 fixed-point energy into the context's
 * device histogram [S][B][K], which is zeroed first ("Flush").  hist_out (host, [S][B][K]
 * uint64) may be NULL to keep the result on the device only. */
int fs_trace(fs_ctx* ctx, const float* src_pos /*[S][3]*/, uint32_t n_sources, const float lis_pos[3],
             uint64_t n_paths, uint32_t max_depth, uint64_t seed, uint64_t* hist_out);

/* One whole update in one call, as the reference does it: UpdateSource (SUB.cpp:128-195) flushes, traces, splats AND calls
 * ReconstructImpulseResponse (:192).  = fs_trace (all sources) followed by fs_build_ir (one source) / fs_build_ir_all (several),
 * enqueued back to back with ONE synchronisation at the end.  hist_out ([S][B][K] uint64) and ir_out ([S][C][sample_rate]
 * float) are host buffers and may be NULL; page-locked ones (fs_host_alloc) are written by the copy engine directly.
 * If the traversal stack overflowed the call returns FS_ERR_OVERFLOW and the impulse responses it published are invalid until
 * the next successful update. */
int fs_update(fs_ctx* ctx, const float* src_pos /*[S][3]*/, uint32_t n_sources, const float lis_pos[3], uint64_t n_paths,
              uint32_t max_depth, uint64_t seed, uint64_t* hist_out, float* ir_out);

/* Shard form for multi-GPU: traces only g in [g_first, g_first + g_count) and ACCUMULATES into
 * a caller-provided DEVICE histogram d_hist [S][B][K] (uint64; e.g. a torch int64 tensor that
 * is then summed over ranks with one NCCL reduce).  zero_first != 0 clears it before. */
int fs_trace_range_device(fs_ctx* ctx, const float* src_pos, uint32_t n_sources, const float lis_pos[3],
                          uint64_t n_paths, uint64_t g_first, uint64_t g_count, uint32_t max_depth,
                          uint64_t seed, void* d_hist, int zero_first);
/* host-buffer shard form (accumulates into hist_inout) */
int fs_trace_range(fs_ctx* ctx, const float* src_pos, uint32_t n_sources, const float lis_pos[3],
                   uint64_t n_paths, uint64_t g_first, uint64_t g_count, uint32_t max_depth,
                   uint64_t seed, uint64_t* hist_inout);
/* debug: one record per path pair of the range (slow; parity localisation only) */
int fs_trace_debug(fs_ctx* ctx, const float* src_pos, uint32_t n_sources, const float lis_pos[3],
                   uint64_t n_paths, uint64_t g_first, uint64_t g_count, uint32_t max_depth,
                   uint64_t seed, fs_path_dbg* dbg_out);

/* ---- per-source budgets ----------------------------------------------------------------------
 * replaces: the per-component tunables RaycastsPerTick / RaycastBounces of UFrequenSeeAudioComponent (COMP.h:35-66), with
 * which the subsystem updates every active source (SUB.cpp:55-85, ForceUpdateSources SUB.cpp:883-886) -- in ONE call
 * instead of one fs_update per source.
 * Work range: G = sum of n_paths; source s owns g in [o_s, o_s + n_s) with o_s = sum_{s' < s} n_s'.  Philox is keyed by
 * (seed, g) for both subpaths as in fs_trace; with FS_FLAG_SHARE_LISTENER the listener subpath is keyed by i = g - o_s.
 * Both subpaths of a pair of source s stop at max_depth_s (0 = node 0 only, the direct-path pair).  The histogram has the
 * layout of fs_trace ([S][B][K] Q32.32, zeroed first) and every IR builder then normalises source s by 1 / n_s.
 * With every n_s = N and max_depth_s = D the result is bit-identical to fs_trace(pos, S, lis, N, D, seed).
 * Checked before anything is enqueued: n_sources >= 1, n_sources * n_bins < 2^32, every n_s >= 1, every depth <= 1024
 * (<= 63 with FS_FLAG_CONNECT_ALL, <= 32 with FS_FLAG_MIS).  FS_FLAG_SHARE_LISTENER needs equal depths: one shared
 * listener walk cannot serve two ray budgets (FS_ERR_INVALID otherwise).  fs_stats.paths = G. */
typedef struct fs_source_desc {
    float    pos[3];          /* metres */
    uint32_t max_depth;       /* RaycastBounces of this emitter: ray budget of BOTH subpaths of its pairs, 0..1024 */
    uint64_t n_paths;         /* RaycastsPerTick of this emitter, >= 1 */
} fs_source_desc;             /* 24 bytes */

int fs_trace_sources(fs_ctx* ctx, const fs_source_desc* src, uint32_t n_sources, const float lis_pos[3], uint64_t seed,
                     uint64_t* hist_out);
/* fs_update for per-source budgets: fs_trace_sources, then the IRs of fs_build_ir_all (published to convolver slots
 * 0 .. n_sources-1), one synchronisation */
int fs_update_sources(fs_ctx* ctx, const fs_source_desc* src, uint32_t n_sources, const float lis_pos[3], uint64_t seed,
                      uint64_t* hist_out, float* ir_out);
/* shard form (one process per GPU): traces g in [g_first, g_first + g_count) of [0, G) and ACCUMULATES into the device
 * histogram d_hist [S][B][K]; zero_first != 0 clears it before */
int fs_trace_sources_range_device(fs_ctx* ctx, const fs_source_desc* src, uint32_t n_sources, const float lis_pos[3],
                                  uint64_t g_first, uint64_t g_count, uint64_t seed, void* d_hist, int zero_first);
/* installs a reduced device histogram with per-source path counts (host [S]), e.g. after an NCCL reduce of
 * fs_trace_sources_range_device shards, so that fs_build_ir* normalise every source by its own count */
int fs_set_histogram_sources_device(fs_ctx* ctx, const void* d_hist, uint32_t n_sources, const uint64_t* n_paths);

/* ---- noise of an update and ray budgets (FS_FLAG_NOISE_STATS) --------------------------------
 * EXTENDS the reference: its subsystem declares allocateSamples (SUB.h:136) but never defines it, and every component's
 * RaycastsPerTick is fixed (COMP.h:35-66).  Cao et al. judge ray-based propagation by the SNR of the energy response and
 * distribute the next frame's samples by the previous frame's result; these entry points close that loop.
 * Per bin k of a source with n pairs: mu_k = S1_k / n, Var_k = (S2_k / n - mu_k^2) / (n - 1) (n - 1 taken as 1 for
 * n = 1), in energy units (histogram value x 2^-32).  signal = sum_k mu_k^2, variance = sum_k Var_k (the variance of the
 * histogram estimate), snr_db = 10 log10(signal / variance): +inf when variance = 0 < signal, -inf when signal = 0 (then
 * no_energy = 1 for the broadband values: nothing connected).  Broadband values are those of the band sum, the quantity
 * the default IR is built from. */
typedef struct fs_noise_stats {
    uint64_t n_paths;                   /* path pairs of the source in the update */
    uint32_t no_energy;                 /* 1: no path of the source connected (broadband signal 0) */
    uint32_t reserved;
    double   signal, variance, snr_db;  /* broadband */
    double   band_signal[FS_MAX_BANDS], band_variance[FS_MAX_BANDS], band_snr_db[FS_MAX_BANDS];   /* bands >= n_bands: 0 */
} fs_noise_stats;                       /* 232 bytes */

/* statistics of the last fs_trace / fs_trace_sources / fs_update* / fs_multi_trace* (on context 0 of the fs_multi), one per
 * source; n_sources must equal fs_get_histogram_sources (FS_ERR_INVALID otherwise).  FS_ERR_STATE without
 * FS_FLAG_NOISE_STATS, before any trace and after a call that leaves the histogram without its second moments
 * (fs_trace_range*, fs_trace_sources_range_device, fs_trace_debug, fs_set_histogram*).  One small kernel, one copy, synchronises. */
int fs_get_noise(fs_ctx* ctx, fs_noise_stats* out, uint32_t n_sources);
/* the raw second moments of the same update, host [S][B+1][K][2] uint64 (lo, hi): slot B is the broadband one.  Same
 * state rules as fs_get_noise. */
int fs_get_histogram_m2(fs_ctx* ctx, uint64_t* out);
/* ray budgets for the next update from the statistics of the last one.  Host only: no context, no GPU.
 * Policy: aim at equal weighted SNR.  Var ~ a_s / n with a_s = st[s].n_paths / snr_lin_s, so n_s ~ w_s a_s
 * (weight: [S] or NULL = 1), clamped to [min_paths, max_paths] by water-filling and rounded by largest remainder so that
 * sum n_s == total exactly.  Unclamped sources end with equal w_s a_s / n_s.  Priority when the bounds bind: a source whose
 * a_s overflows (signal far below its variance) is served first (equal shares, up to max_paths), then the sources with a
 * positive demand, then those without (variance 0 or weight 0), which get min_paths unless paths are left over.  A source
 * with no_energy keeps its previous count (clamped) and is taken out of the pool first; if the others cannot then take the
 * rest within the bounds, it joins the pool with no demand.  The SNR it predicts rests on one update's estimate of a_s:
 * measured on 16 tunnel emitters, one step narrowed the spread of snr_db by a factor 1.49, and repeated steps do not settle.
 * FS_ERR_INVALID for n_sources = 0, S min > total, S max < total, min = 0, min > max, a negative or non-finite weight. */
int fs_allocate_paths(const fs_noise_stats* st, uint32_t n_sources, uint64_t total, uint64_t min_paths, uint64_t max_paths,
                      const float* weight, uint64_t* n_out);

/* single rays through the device BVH (parity tests of the intersector):
 * rays: [n][6] (origin, direction); out_t [n] (inf on miss), out_tri [n] (0xffffffff on miss) */
int fs_debug_closest_hits(fs_ctx* ctx, const float* rays, uint64_t n, float* out_t, uint32_t* out_tri);
int fs_debug_any_hits(fs_ctx* ctx, const float* rays, const float* tmax, uint64_t n, uint8_t* out_hit);

/* ---- impulse response -----------------------------------------------------------------------
 * replaces: UFrequenSeeAudioComponent::ReconstructImpulseResponse (COMP.cpp:320-380) and
 * GetImpulseResponse (COMP.h:113).  Uses the histogram of `source` left by the last fs_trace
 * (or set by fs_set_histogram), normalised by 1/n_paths (SUB.cpp:164; after fs_trace_sources* by that source's own count).  Also refreshes that
 * source's convolver partition spectra.  ir_out: host [C][sample_rate] float, may be NULL. */
int fs_build_ir(fs_ctx* ctx, uint32_t source, float* ir_out);
/* same, with the histogram slot and the convolver slot named separately (a per-component update
 * traces one source into histogram slot 0 and publishes the IR to that component's own slot) */
int fs_build_ir_to(fs_ctx* ctx, uint32_t hist_source, uint32_t conv_source, float* ir_out);
/* multi-emitter update (BASELINE configs[3]: 64 sources): fs_build_ir for sources 0 .. n_sources-1 with the three IR kernels
 * launched once per 64 sources instead of once per source; same arithmetic.  ir_out: host [n_sources][C][sample_rate] or NULL. */
int fs_build_ir_all(fs_ctx* ctx, uint32_t n_sources, float* ir_out);
/* per-band synthesis (SURVEY.md 8f rank 2; EXTENDS the reference, whose IR is one low-passed broadband envelope,
 * COMP.cpp:337-378): each band keeps its envelope (the mapping of COMP.cpp:339-363 per band) and modulates a unit-RMS
 * octave-band noise carrier (f_b = 62.5 * 2^b Hz, Philox noise keyed by noise_seed through two RBJ band-pass biquads);
 * ir[c][t] = sum_b ramp_b[t] * carrier[c][b][t], no low-pass.  Publishes to conv_source's convolver like fs_build_ir_to. */
int fs_build_ir_bands(fs_ctx* ctx, uint32_t hist_source, uint32_t conv_source, uint64_t noise_seed, float* ir_out);
/* seam 1 of the reference taken literally: EnergyBuffer float[K] -> IR (AddEnergyAtDelay users) */
int fs_build_ir_from_energy(fs_ctx* ctx, uint32_t source, const float* energy /*[K]*/, float* ir_out);
/* install an already reduced histogram (host [S][B][K]) and its path count, e.g. after an NCCL reduce */
int fs_set_histogram(fs_ctx* ctx, const uint64_t* hist, uint32_t n_sources, uint64_t n_paths);
int fs_set_histogram_device(fs_ctx* ctx, const void* d_hist, uint32_t n_sources, uint64_t n_paths);
/* copies the histogram of the LAST fs_trace* / fs_set_histogram*: [S][B][K] with S = the source count of that call, which
 * fs_get_histogram_sources returns (size the buffer with it) */
int fs_get_histogram(fs_ctx* ctx, uint64_t* hist_out /*[S][B][K]*/);
int fs_get_histogram_sources(fs_ctx* ctx, uint32_t* n_sources_out);
/* install an external IR (host [C][sample_rate]) for `source`, e.g. a loaded saved_ir.txt
 * (COMP.cpp:454-490) */
int fs_set_ir(fs_ctx* ctx, uint32_t source, const float* ir);
/* text files with one float per line, the format of the reference's saved_ir.txt:
 * replaces UFrequenSeeAudioComponent::LoadFloatArray (COMP.cpp:454-490; FCString::Atof per line, empty lines
 * skipped) and SaveArrayToFile (COMP.cpp:492-505).  Host only: no context, no GPU.
 * fs_load_float_array: values are written to out[0 .. min(*n_out, cap)); *n_out = number of values in the file
 * (call with out = NULL, cap = 0 to size the buffer).  Returns FS_ERR_INVALID if the file cannot be read.
 * fs_save_float_array writes the shortest decimal form that reads back to the same float ("%.9g"). */
int fs_load_float_array(const char* path, float* out, uint64_t cap, uint64_t* n_out);

/* ---- page-locked host buffers ---------------------------------------------------------------
 * no reference counterpart (the reference's ImpulseBuffer is a TArray in the component, COMP.h:93).  An IR / histogram
 * destination that is page-locked -- allocated here, or registered by the caller with the CUDA runtime -- is written by
 * the copy engine directly; any other destination goes through the context's pinned staging buffer and one memcpy.
 * 64 emitters x 2 x 48 000 floats = 24.6 MB per update: the difference is the memcpy and the page faults of a fresh
 * buffer.  Usable before fs_create; free with fs_host_free. */
int  fs_host_alloc(size_t bytes, void** out);
void fs_host_free(void* p);
int fs_save_float_array(const char* path, const float* data, uint64_t n);

/* ---- convolution ----------------------------------------------------------------------------
 * replaces: IAudioReverb::OnInitSource / OnReleaseSource / ProcessSourceAudio (REV.h:39-47,
 * REV.cpp:104-170) and ConvolveFFT (REV.cpp:172-213), FCircularAudioBuffer (CIRC.cpp:43-75).
 * Uniformly partitioned overlap-save: output block = history (*) current IR, history initially
 * zero.  in/out: interleaved host [frames][C] float; frames must equal cfg.conv_block. */
int fs_conv_init_source(fs_ctx* ctx, uint32_t source);
int fs_conv_release_source(fs_ctx* ctx, uint32_t source);
int fs_conv_process(fs_ctx* ctx, uint32_t source, const float* in_interleaved, float* out_interleaved,
                    uint32_t frames);
/* multi-emitter callback (BASELINE configs[3]: 64 sources): one block of every listed source in ONE kernel launch
 * (grid = sources x channels) instead of n_sources serial calls.  sources: n_sources distinct initialised ids;
 * in / out: host [n_sources][frames][C] interleaved, in the order of `sources`. */
int fs_conv_process_multi(fs_ctx* ctx, const uint32_t* sources, uint32_t n_sources, const float* in_interleaved,
                          float* out_interleaved, uint32_t frames);
/* offline form: n_blocks consecutive callbacks in one call (config 3 bench); host buffers */
int fs_conv_process_many(fs_ctx* ctx, uint32_t source, const float* in_interleaved,
                         float* out_interleaved, uint32_t frames_per_block, uint32_t n_blocks);
/* real FFT of n samples on the device FFT kernel (n power of two, 64..4096); out [n/2+1][2] */
int fs_debug_rfft(fs_ctx* ctx, const float* in, uint32_t n, float* out_ri);

/* ---- several GPUs of one box -----------------------------------------------------------------
 * The reference is one process with one game thread (SUB.cpp:55-85); the independent unit of work is one iteration of its
 * pair loop (SUB.cpp:215-230).  fs_multi owns one context per device inside ONE host process (no Python, no MPI, no
 * collective library): the global work range g = source * n_paths + i is cut into contiguous shards, every device traces
 * its shard against its own copy of the BVH (one host thread per device enqueues it), the per-device Q32.32 histograms are
 * written into a staging buffer on device 0 by peer stores over NVLink and summed there.  Integer sums: bit-identical to
 * the single-device result for every device count.  The reduced histogram is that of context 0 (fs_multi_context(m, 0)):
 * fs_build_ir*, fs_conv_* and fs_get_histogram of the single-device API continue from it.
 * devices: CUDA ordinals (NULL = 0 .. n_devices-1); an ordinal may repeat (several contexts on one GPU).
 * Errors: fs_status; fs_multi_last_error() = message of the calling thread's last fs_multi_* failure. */
typedef struct fs_multi fs_multi;
int         fs_multi_create(const fs_config* cfg, const int* devices, uint32_t n_devices, fs_multi** out);
void        fs_multi_destroy(fs_multi* m);
const char* fs_multi_last_error(void);
uint32_t    fs_multi_device_count(const fs_multi* m);
fs_ctx*     fs_multi_context(fs_multi* m, uint32_t i);
/* the scene is replicated: every device builds its own (identical) BVH -- replaces RegisterGeometry (SUB.h:99-100) */
int fs_multi_scene_set_triangles(fs_multi* m, const float* verts, const uint32_t* tri_material, uint64_t n_tris);
int fs_multi_scene_set_materials(fs_multi* m, const float* absorption, uint32_t n_materials, uint32_t n_bands);
int fs_multi_scene_set_materials_ex(fs_multi* m, const float* absorption, const float* transmission, const float* scattering,
                                    const float* thickness_cm, uint32_t n_materials, uint32_t n_bands);
int fs_multi_scene_commit(fs_multi* m);
/* fs_scene_update_vertices / fs_scene_refit on every device (SUB.cpp:331-334); the ratio is that of device 0 */
int fs_multi_scene_update_vertices(fs_multi* m, const float* verts, uint64_t first_tri, uint64_t n_tris);
int fs_multi_scene_refit(fs_multi* m, float* cost_ratio_out);
/* fs_trace over all devices (UpdateSource, SUB.cpp:128-195).  Enqueues and returns; hist_out (host [S][B][K]) may be NULL,
 * non-NULL synchronises. */
int fs_multi_trace(fs_multi* m, const float* src_pos, uint32_t n_sources, const float lis_pos[3], uint64_t n_paths,
                   uint32_t max_depth, uint64_t seed, uint64_t* hist_out);
/* fs_trace_sources over all devices: [0, G) is cut into contiguous shards like fs_multi_trace; context 0 then holds the
 * reduced histogram and the per-source path counts */
int fs_multi_trace_sources(fs_multi* m, const fs_source_desc* src, uint32_t n_sources, const float lis_pos[3], uint64_t seed,
                           uint64_t* hist_out);
/* device time of the last fs_multi_trace (CUDA events on device 0's stream): the whole update, and the part after device
 * 0's own shard was done (waiting for the peers' stores + the sum).  Synchronises. */
int fs_multi_last_ms(fs_multi* m, float* total_ms, float* reduce_ms);
int fs_multi_synchronize(fs_multi* m);

/* ---- stats ------------------------------------------------------------------------------- */
int fs_get_stats(fs_ctx* ctx, fs_stats* out);

#ifdef __cplusplus
}
#endif
#endif
