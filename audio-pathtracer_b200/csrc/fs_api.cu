// fs_api.cu -- the extern "C" boundary (include/frequensee.h).  No CPU fallback anywhere: every
// entry point either runs the CUDA path or returns an error.
#include "fs_internal.h"
#include "fs_diffraction.h"

#include <nvtx3/nvToolsExt.h>          // header-only NVTX 3: named ranges per stage for nsys / ncu --nvtx (SURVEY section 5)
#include <algorithm>
#include <climits>
#include <cmath>
#include <stdio.h>
#include <utility>
#include <stdlib.h>
#include <new>
#include <vector>

// last failure message of the CALLING THREAD (the game thread and the audio thread use one context concurrently)
static thread_local std::string g_err;

#define CK(call)                                                                              \
    do {                                                                                      \
        cudaError_t e__ = (call);                                                             \
        if (e__ != cudaSuccess) return fail_cuda(ctx, e__, #call);                            \
    } while (0)

static int fail(fs_ctx* ctx, int code, const char* msg)
{
    (void)ctx;
    g_err = msg;
    return code;
}
static int fail_cuda(fs_ctx* ctx, cudaError_t e, const char* what)
{
    char buf[512];
    snprintf(buf, sizeof(buf), "CUDA error %d (%s) in %s", (int)e, cudaGetErrorString(e), what);
    (void)ctx;
    g_err = buf;
    (void)cudaGetLastError();
    return e == cudaErrorMemoryAllocation ? FS_ERR_NOMEM : FS_ERR_CUDA;
}

struct nvtx_range {                    // RAII range on the calling thread
    explicit nvtx_range(const char* name) { nvtxRangePushA(name); }
    ~nvtx_range() { nvtxRangePop(); }
};

struct dev_guard {
    int prev; bool ok;
    explicit dev_guard(int dev) : prev(-1), ok(false) { if (cudaGetDevice(&prev) == cudaSuccess) ok = (cudaSetDevice(dev) == cudaSuccess); }
    ~dev_guard() { if (prev >= 0) cudaSetDevice(prev); }
};

// the experiment knobs of a new context (defaults: fs_tune)
static fs_tune read_tune()
{
    fs_tune t;
    // the knob's value, if the variable is set and its value is within [lo, hi]
    auto env = [](const char* name, uint32_t& v, int lo = INT_MIN, int hi = INT_MAX) {
        if (const char* e = getenv(name)) { const int x = atoi(e); if (x >= lo && x <= hi) v = (uint32_t)x; }
    };
    env("FS_TUNE_REFILL", t.refill, 1, 32);
    env("FS_TUNE_LEAF_MAX", t.leaf_max, 1, 8);
    env("FS_TUNE_TEX", t.tex);
    env("FS_TUNE_BUILDER", t.builder);
    env("FS_TUNE_WIDE", t.wide);
    env("FS_TUNE_W8", t.w8);
    env("FS_TUNE_NODE_MIN", t.node_min);
    env("FS_TUNE_TRI_MIN", t.tri_min);
    env("FS_TUNE_COLLAPSE", t.collapse);
    env("FS_TUNE_L2PIN", t.l2pin_mb);
    env("FS_TUNE_TQ", t.tq);
    env("FS_TUNE_TQ_NODE_MIN", t.tq_node_min);
    env("FS_TUNE_TQ_FLUSH", t.tq_flush);
    t.tq_flush = std::min(std::max(t.tq_flush, 1u), 32u);
    env("FS_TUNE_MEGA", t.mega);
    env("FS_TUNE_MEGA_FROM", t.mega_from);
    env("FS_TUNE_MEGA_LANES", t.mega_lanes, 1, FS_MAX_LANES);
    env("FS_TUNE_STREAMS", t.streams, 1, FS_MAX_LANES);
    if (const char* e = getenv("FS_TUNE_CARVEOUT")) t.carveout = atoi(e);
    return t;
}

extern "C" {

void fs_default_config(fs_config* c)
{
    memset(c, 0, sizeof(*c));
    c->n_bands = 8; c->n_bins = 1000; c->bin_ms = 1.0f; c->rr_prob = 0.9f;
    c->eps_offset = 1e-3f; c->eps_connect = 1e-3f; c->min_seg = 1e-2f; c->sound_speed = 343.0f;
    c->pdf_exponent = 0.1f; c->energy_clamp = 1.0f; c->energy_gain = 10.0f;
    static const float air[FS_MAX_BANDS] = {0.0001f, 0.0003f, 0.0006f, 0.0010f, 0.0017f, 0.0035f, 0.0050f, 0.0120f};
    for (int b = 0; b < FS_MAX_BANDS; ++b) c->air_absorption[b] = air[b];
    c->sample_rate = 48000; c->n_channels = 2; c->ir_threshold = 1e-6f; c->ir_lowpass = 0.25f;
    c->conv_block = 1024; c->conv_clamp = 1; c->conv_wet = 1.0f;
    c->max_batch_paths = 0; c->flags = 0; c->device = -1;
}

const char* fs_last_error(const fs_ctx* ctx) { (void)ctx; return g_err.c_str(); }

int fs_create(const fs_config* cfg, fs_ctx** out)
{
    if (!cfg || !out) return fail(nullptr, FS_ERR_INVALID, "fs_create: null argument");
    *out = nullptr;
    if (cfg->n_bands < 1 || cfg->n_bands > FS_MAX_BANDS) return fail(nullptr, FS_ERR_INVALID, "n_bands must be 1..8");
    if (cfg->n_bins < 1 || cfg->n_bins > (1u << 20)) return fail(nullptr, FS_ERR_INVALID, "n_bins out of range");
    if (!(cfg->bin_ms > 0.f) || !(cfg->sound_speed > 0.f)) return fail(nullptr, FS_ERR_INVALID, "bin_ms/sound_speed must be > 0");
    if (!(cfg->rr_prob > 0.f) || cfg->rr_prob > 1.0f) return fail(nullptr, FS_ERR_INVALID, "rr_prob must be in (0,1]");
    if (cfg->n_channels < 1 || cfg->n_channels > 8) return fail(nullptr, FS_ERR_INVALID, "n_channels must be 1..8");
    if (cfg->conv_block < 32 || cfg->conv_block > 2048 || (cfg->conv_block & (cfg->conv_block - 1)))
        return fail(nullptr, FS_ERR_INVALID, "conv_block must be a power of two in 32..2048");
    if (cfg->sample_rate < cfg->conv_block) return fail(nullptr, FS_ERR_INVALID, "sample_rate < conv_block");
    if ((uint32_t)((double)cfg->bin_ms * 1e-3 * cfg->sample_rate + 0.5) < 1u)
        return fail(nullptr, FS_ERR_INVALID, "bin_ms * sample_rate / 1000 must be at least one sample");
    if (!(cfg->ir_lowpass > 0.0f) || cfg->ir_lowpass > 1.0f) return fail(nullptr, FS_ERR_INVALID, "ir_lowpass must be in (0,1]");
    // an empty bin passes a threshold <= 0 and maps to 0 / sqrt(0) = NaN; a NaN threshold silently zeroes the IR
    if (!(cfg->ir_threshold > 0.0f) || !isfinite(cfg->ir_threshold))
        return fail(nullptr, FS_ERR_INVALID, "ir_threshold must be finite and > 0");
    if ((cfg->flags & FS_FLAG_NOISE_STATS) && (cfg->flags & (FS_FLAG_CONNECT_ALL | FS_FLAG_MIS)))
        return fail(nullptr, FS_ERR_INVALID, "FS_FLAG_NOISE_STATS needs the endpoint connection (not with FS_FLAG_CONNECT_ALL / "
                                             "FS_FLAG_MIS: a pair adds to several bins there)");
    // warm-up window of the per-sample low-pass evaluation: (1 - a)^W <= 1e-12, a multiple of 32 taps
    uint32_t ir_window = 32;
    if (cfg->ir_lowpass < 1.0f) {
        const double w = ceil(log(1e-12) / log(1.0 - (double)cfg->ir_lowpass));
        if (!(w <= 8192.0)) return fail(nullptr, FS_ERR_INVALID, "ir_lowpass too small (needs a warm-up window above 8192 samples)");
        ir_window = ((uint32_t)w + 31u) & ~31u;
        if (ir_window < 32u) ir_window = 32u;
    }
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        char buf[256];
        snprintf(buf, sizeof(buf), "no usable CUDA device (%s); this library has no CPU fallback",
                 e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
        return fail(nullptr, FS_ERR_CUDA, buf);
    }
    int dev = cfg->device;
    if (dev < 0) { if (cudaGetDevice(&dev) != cudaSuccess) dev = 0; }
    if (dev >= ndev) return fail(nullptr, FS_ERR_INVALID, "device ordinal out of range");
    fs_ctx* ctx = new (std::nothrow) fs_ctx();
    if (!ctx) return fail(nullptr, FS_ERR_NOMEM, "out of host memory");
    ctx->cfg = *cfg;
    if (ctx->cfg.max_batch_paths == 0) ctx->cfg.max_batch_paths = 1u << 21;
    ctx->device = dev;
    ctx->ir_window = ir_window;
    ctx->launches.store(0); ctx->conv_active.store(0);
    ctx->tune = read_tune();
    dev_guard g(dev);
    int rc = FS_OK;
    do {
        cudaDeviceProp prop;
        if ((e = cudaGetDeviceProperties(&prop, dev)) != cudaSuccess) { rc = fail_cuda(nullptr, e, "cudaGetDeviceProperties"); break; }
        if (prop.major < 10) {
            char buf[256];
            snprintf(buf, sizeof(buf), "device %d is sm_%d%d; this library is built for sm_100a only", dev, prop.major, prop.minor);
            rc = fail(nullptr, FS_ERR_CUDA, buf); break;
        }
        ctx->sm_count = prop.multiProcessorCount;
        if ((e = cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking)) != cudaSuccess) { rc = fail_cuda(nullptr, e, "cudaStreamCreate"); break; }
        ctx->stream = ctx->own_stream;
        if ((e = cudaEventCreate(&ctx->ev0)) != cudaSuccess || (e = cudaEventCreate(&ctx->ev1)) != cudaSuccess ||
            (e = cudaEventCreate(&ctx->ev_ir0)) != cudaSuccess || (e = cudaEventCreate(&ctx->ev_ir1)) != cudaSuccess) { rc = fail_cuda(nullptr, e, "cudaEventCreate"); break; }
        if ((e = cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming)) != cudaSuccess) { rc = fail_cuda(nullptr, e, "cudaEventCreate"); break; }
        if ((e = cudaEventCreateWithFlags(&ctx->ev_overflow, cudaEventDisableTiming)) != cudaSuccess) { rc = fail_cuda(nullptr, e, "cudaEventCreate"); break; }
        if ((e = cudaEventCreate(&ctx->ev_c0)) != cudaSuccess || (e = cudaEventCreate(&ctx->ev_c1)) != cudaSuccess) { rc = fail_cuda(nullptr, e, "cudaEventCreate"); break; }
        if ((e = cudaMallocHost(&ctx->h_overflow, sizeof(uint32_t))) != cudaSuccess) { rc = fail_cuda(nullptr, e, "cudaMallocHost"); break; }
        *ctx->h_overflow = 0u;
        for (int l = 1; l < FS_MAX_LANES && e == cudaSuccess; ++l) {          // lane 0 runs on the context stream itself
            if ((e = cudaStreamCreateWithFlags(&ctx->lanes[l].stream, cudaStreamNonBlocking)) != cudaSuccess) break;
            e = cudaEventCreateWithFlags(&ctx->lanes[l].done, cudaEventDisableTiming);
        }
        if (e != cudaSuccess) { rc = fail_cuda(nullptr, e, "batch lanes"); break; }
        if ((e = cudaMalloc(&ctx->d_counters, sizeof(fs_dev_counters))) != cudaSuccess) { rc = fail_cuda(nullptr, e, "cudaMalloc counters"); break; }
        if ((e = cudaMemsetAsync(ctx->d_counters, 0, sizeof(fs_dev_counters), ctx->own_stream)) != cudaSuccess ||
            (e = cudaStreamSynchronize(ctx->own_stream)) != cudaSuccess) { rc = fail_cuda(nullptr, e, "cudaMemset"); break; }
        if ((e = cudaMalloc(&ctx->d_amp, sizeof(float) * cfg->n_bins)) != cudaSuccess) { rc = fail_cuda(nullptr, e, "cudaMalloc amp"); break; }
        if ((e = cudaMalloc(&ctx->d_energy, sizeof(float) * cfg->n_bins)) != cudaSuccess) { rc = fail_cuda(nullptr, e, "cudaMalloc energy"); break; }
        if ((e = fs_conv_setup(ctx)) != cudaSuccess) { rc = fail_cuda(nullptr, e, "fs_conv_setup"); break; }
    } while (0);
    if (rc != FS_OK) { fs_destroy(ctx); return rc; }
    *out = ctx;
    return FS_OK;
}

void fs_destroy(fs_ctx* ctx)
{
    if (!ctx) return;
    dev_guard g(ctx->device);
    cudaDeviceSynchronize();
    fs_conv_teardown(ctx);
    cudaFree(ctx->d_carriers); cudaFree(ctx->d_amp_bands); cudaFree(ctx->d_amp_all);
    cudaFree(ctx->lis_rec); cudaFree(ctx->lis_end);
    for (int l = 0; l < FS_MAX_LANES; ++l) {
        fs_wave_free(&ctx->lanes[l].wb);
        if (l && ctx->lanes[l].stream) cudaStreamDestroy(ctx->lanes[l].stream);
        if (ctx->lanes[l].done) cudaEventDestroy(ctx->lanes[l].done);
    }
    if (ctx->ev_fork) cudaEventDestroy(ctx->ev_fork);
    if (ctx->ev_overflow) cudaEventDestroy(ctx->ev_overflow);
    if (ctx->ev_c0) cudaEventDestroy(ctx->ev_c0);
    if (ctx->ev_c1) cudaEventDestroy(ctx->ev_c1);
    if (ctx->h_overflow) cudaFreeHost(ctx->h_overflow);
    cudaFree(ctx->d_bsdf_tab); cudaFree(ctx->d_lobes);
    fs_bvh_free(&ctx->bvh);
    cudaFree(ctx->d_verts); cudaFree(ctx->d_tri_mat); cudaFree(ctx->d_refl_over_pi);
    cudaFree(ctx->d_hist); cudaFree(ctx->d_m2); cudaFree(ctx->d_noise); cudaFree(ctx->d_acou); cudaFree(ctx->d_counters); cudaFree(ctx->d_src_pos); cudaFree(ctx->d_dbg); cudaFree(ctx->d_src_tab);
    cudaFree(ctx->d_dir_gain); cudaFree(ctx->d_dir_orient);
    cudaFree(ctx->d_occl_tau); cudaFree(ctx->d_occl);
    cudaFree(ctx->d_diff_edges); cudaFree(ctx->d_diff); cudaFree(ctx->d_diff_cand);
    cudaFree(ctx->d_amp); cudaFree(ctx->d_energy);
    for (cudaEvent_t e : ctx->kev) cudaEventDestroy(e);
    for (cudaEvent_t e : ctx->tev) cudaEventDestroy(e);
    if (ctx->ev0) cudaEventDestroy(ctx->ev0);
    if (ctx->ev1) cudaEventDestroy(ctx->ev1);
    if (ctx->ev_ir0) cudaEventDestroy(ctx->ev_ir0);
    if (ctx->ev_ir1) cudaEventDestroy(ctx->ev_ir1);
    if (ctx->own_stream) cudaStreamDestroy(ctx->own_stream);
    delete ctx;
}

static void apply_l2_policy(fs_ctx* ctx);

// Traversal-stack overflow of an earlier trace (fs_dev_counters::overflow, copied to pinned memory by one 4-byte async
// copy after every fs_trace*).  wait = false: look only if the copy has landed (never blocks); the flag stays on the
// device until the host has seen it, so it cannot be lost between two asynchronous traces.
static int check_overflow(fs_ctx* ctx, bool wait)
{
    if (!ctx->overflow_pending) return FS_OK;
    if (wait) { CK(cudaEventSynchronize(ctx->ev_overflow)); }
    else if (cudaEventQuery(ctx->ev_overflow) != cudaSuccess) { (void)cudaGetLastError(); return FS_OK; }
    ctx->overflow_pending = false;
    if (*ctx->h_overflow) {
        *ctx->h_overflow = 0u;
        return fail(ctx, FS_ERR_OVERFLOW, "BVH traversal stack overflow in the last trace (tree deeper than FS_STACK_SIZE): its histogram is incomplete");
    }
    return FS_OK;
}

int fs_set_stream(fs_ctx* ctx, void* cuda_stream)
{
    if (!ctx) return FS_ERR_INVALID;
    ctx->stream = cuda_stream ? (cudaStream_t)cuda_stream : ctx->own_stream;
    if (ctx->committed) { dev_guard g(ctx->device); apply_l2_policy(ctx); }
    return FS_OK;
}

int fs_synchronize(fs_ctx* ctx)
{
    if (!ctx) return FS_ERR_INVALID;
    dev_guard g(ctx->device);
    CK(cudaStreamSynchronize(ctx->stream));
    return check_overflow(ctx, true);
}

// ---- scene -----------------------------------------------------------------------------------
int fs_scene_set_triangles(fs_ctx* ctx, const float* verts, const uint32_t* tri_material, uint64_t n_tris)
{
    if (!ctx) return FS_ERR_INVALID;
    if (n_tris && (!verts || !tri_material)) return fail(ctx, FS_ERR_INVALID, "fs_scene_set_triangles: null array");
    if (n_tris >= (1ull << 27)) return fail(ctx, FS_ERR_INVALID, "too many triangles (< 2^27 supported)");
    dev_guard g(ctx->device);
    for (uint64_t i = 0; i < n_tris * 9; ++i)
        if (!(verts[i] == verts[i]) || fabsf(verts[i]) > 1e18f) return fail(ctx, FS_ERR_INVALID, "non-finite vertex");
    cudaFree(ctx->d_verts); cudaFree(ctx->d_tri_mat);
    ctx->d_verts = nullptr; ctx->d_tri_mat = nullptr;
    ctx->n_tris = n_tris; ctx->committed = false; ctx->tris_set = false; ctx->verts_dirty = false; ctx->diff_valid = false;
    if (n_tris) {
        CK(cudaMalloc(&ctx->d_verts, sizeof(float) * 9 * n_tris));
        CK(cudaMalloc(&ctx->d_tri_mat, sizeof(uint32_t) * n_tris));
        CK(cudaMemcpyAsync(ctx->d_verts, verts, sizeof(float) * 9 * n_tris, cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaMemcpyAsync(ctx->d_tri_mat, tri_material, sizeof(uint32_t) * n_tris, cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
    }
    // material ids are validated against the table at commit time
    ctx->tris_set = true;
    return FS_OK;
}

int fs_scene_set_materials(fs_ctx* ctx, const float* absorption, uint32_t n_materials, uint32_t n_bands)
{
    if (!ctx) return FS_ERR_INVALID;
    if (!absorption || n_materials == 0) return fail(ctx, FS_ERR_INVALID, "fs_scene_set_materials: empty table");
    if (n_bands != ctx->cfg.n_bands) return fail(ctx, FS_ERR_INVALID, "n_bands differs from fs_config.n_bands");
    dev_guard g(ctx->device);
    std::vector<float> r((size_t)n_materials * n_bands);
    ctx->mat_absorption.assign(absorption, absorption + r.size());
    ctx->mat_transmission.clear(); ctx->mat_scattering.clear(); ctx->mat_thickness_cm.clear();
    for (size_t i = 0; i < r.size(); ++i) {
        float a = absorption[i];
        if (!(a >= 0.0f && a <= 1.0f)) return fail(ctx, FS_ERR_INVALID, "absorption must be in [0,1]");
        // reflectivity / PI (SUB.cpp:381-386); the reference's "Absorption" asset field is used as
        // reflectivity there -- here absorption alpha means rho = 1 - alpha
        r[i] = (1.0f - a) / FS_PI;
    }
    cudaFree(ctx->d_refl_over_pi); ctx->d_refl_over_pi = nullptr;
    CK(cudaMalloc(&ctx->d_refl_over_pi, sizeof(float) * r.size()));
    CK(cudaMemcpyAsync(ctx->d_refl_over_pi, r.data(), sizeof(float) * r.size(), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->n_mats = n_materials; ctx->mats_set = true; ctx->committed = false;
    return FS_OK;
}

// The breadth-first wide-node array starts with the top of the tree: pin that prefix in L2 (persisting
// access-policy window on the context's stream) so the per-step streaming state (ray queues, node records:
// hundreds of MB) cannot evict the nodes every ray visits.  FS_TUNE_L2PIN = MB to pin (0 = off).
static void apply_l2_policy(fs_ctx* ctx)
{
    if (!ctx->bvh.wnodes) return;
    if (ctx->tune.l2pin_mb == 0xffffffffu) {
        // automatic (default): only for scenes whose nodes + triangles do not fit the L2 anyway -- there a 48 MB window over
        // the top of the tree is worth 2 % (concert hall, profiles/r2_experiments.md); scenes that fit need no help
        int l2 = 0;
        cudaDeviceGetAttribute(&l2, cudaDevAttrL2CacheSize, ctx->device);
        const size_t bvh_bytes = (size_t)ctx->bvh.n_wide * 64u + (size_t)ctx->bvh.n_tris * 64u;
        ctx->tune.l2pin_mb = (l2 > 0 && bvh_bytes > (size_t)l2) ? 48u : 0u;
    }
    if (!ctx->tune.l2pin_mb) return;
    int max_persist = 0, max_window = 0;
    cudaDeviceGetAttribute(&max_persist, cudaDevAttrMaxPersistingL2CacheSize, ctx->device);
    cudaDeviceGetAttribute(&max_window, cudaDevAttrMaxAccessPolicyWindowSize, ctx->device);
    size_t want = (size_t)ctx->tune.l2pin_mb << 20;
    const size_t have = (size_t)ctx->bvh.n_wide * 64u;
    if (want > have) want = have;
    if (want > (size_t)max_persist) want = (size_t)max_persist;
    if (want > (size_t)max_window) want = (size_t)max_window;
    if (!want) return;
    if (cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, want) != cudaSuccess) { (void)cudaGetLastError(); return; }
    cudaStreamAttrValue v; memset(&v, 0, sizeof(v));
    v.accessPolicyWindow.base_ptr = ctx->bvh.wnodes;
    v.accessPolicyWindow.num_bytes = want;
    v.accessPolicyWindow.hitRatio = 1.0f;
    v.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
    v.accessPolicyWindow.missProp = cudaAccessPropertyNormal;
    if (cudaStreamSetAttribute(ctx->stream, cudaStreamAttributeAccessPolicyWindow, &v) != cudaSuccess) (void)cudaGetLastError();
    for (int l = 1; l < FS_MAX_LANES; ++l)                 // the other batch lanes walk the same tree on streams of their own
        if (ctx->lanes[l].stream && cudaStreamSetAttribute(ctx->lanes[l].stream, cudaStreamAttributeAccessPolicyWindow, &v) != cudaSuccess)
            (void)cudaGetLastError();
    if (getenv("FS_VERBOSE")) fprintf(stderr, "[frequensee] L2 persisting window: %.1f MB of wide nodes (device max %d MB)\n", want / 1048576.0, max_persist >> 20);
}

int fs_scene_set_materials_ex(fs_ctx* ctx, const float* absorption, const float* transmission, const float* scattering,
                              const float* thickness_cm, uint32_t n_materials, uint32_t n_bands)
{
    int rc = fs_scene_set_materials(ctx, absorption, n_materials, n_bands);
    if (rc != FS_OK) return rc;
    const size_t n = (size_t)n_materials * n_bands;
    for (int which = 0; which < 2; ++which) {
        const float* v = which ? scattering : transmission;
        if (!v) continue;
        for (size_t i = 0; i < n; ++i)
            if (!(v[i] >= 0.0f && v[i] <= 1.0f)) return fail(ctx, FS_ERR_INVALID, which ? "scattering must be in [0,1]" : "transmission must be in [0,1]");
    }
    if (thickness_cm)
        for (uint32_t m = 0; m < n_materials; ++m)
            if (!(thickness_cm[m] >= 0.0f)) return fail(ctx, FS_ERR_INVALID, "thickness must be >= 0");
    ctx->mat_transmission.assign(transmission ? transmission : nullptr, transmission ? transmission + n : nullptr);
    ctx->mat_scattering.assign(scattering ? scattering : nullptr, scattering ? scattering + n : nullptr);
    ctx->mat_thickness_cm.assign(thickness_cm ? thickness_cm : nullptr, thickness_cm ? thickness_cm + n_materials : nullptr);
    ctx->committed = false;
    return FS_OK;
}

// Transmitted factor of one (material, band) of the material asset, for the material model and for fs_occlusion: tau is
// limited so that Refl + tau <= 1 (MaterialAcousticProcessor.cpp:59-60; limited in place, the lobe thresholds use it) and
// raised to ThicknessCm / 2.5 (ex), a Beer-Lambert layer with the asset's default 2.5 cm as the reference thickness.
static float transmitted_factor(float absorption, float& tau, float ex)
{
    const float refl = 1.0f - absorption;
    if (refl + tau > 1.0f) tau = 1.0f - refl;
    if (!(tau > 0.0f)) return 0.0f;
    return (ex == 1.0f) ? tau : fs_pow(tau, ex);
}

// fs_occlusion's table tau_eff [M][B], for every context (with or without FS_FLAG_MATERIAL_MODEL); materials set without
// Transmission have tau = 0: their surfaces block
static int build_occlusion_table(fs_ctx* ctx)
{
    const uint32_t M = ctx->n_mats, B = ctx->cfg.n_bands;
    std::vector<float> tab((size_t)M * B);
    const float* tr = ctx->mat_transmission.empty() ? nullptr : ctx->mat_transmission.data();
    const float* th = ctx->mat_thickness_cm.empty() ? nullptr : ctx->mat_thickness_cm.data();
    for (uint32_t m = 0; m < M; ++m) {
        const float ex = (th ? th[m] : 2.5f) / 2.5f;
        for (uint32_t b = 0; b < B; ++b) {
            float tau = tr ? tr[(size_t)m * B + b] : 0.0f;
            tab[(size_t)m * B + b] = transmitted_factor(ctx->mat_absorption[(size_t)m * B + b], tau, ex);
        }
    }
    cudaFree(ctx->d_occl_tau); ctx->d_occl_tau = nullptr;
    CK(cudaMalloc(&ctx->d_occl_tau, sizeof(float) * tab.size()));
    CK(cudaMemcpyAsync(ctx->d_occl_tau, tab.data(), sizeof(float) * tab.size(), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return FS_OK;
}

// FS_FLAG_MATERIAL_MODEL (SURVEY 8f rank 3): per (event, material, band) energy factors and per material lobe thresholds.
// Plain float arithmetic in a fixed order that the CPU harness restates (the tables must be
// bit-identical on both sides); fs_pow is the shared polynomial of fs_math.cuh.
static int build_material_model(fs_ctx* ctx)
{
    const uint32_t M = ctx->n_mats, B = ctx->cfg.n_bands;
    std::vector<float> tab((size_t)3 * M * B, 0.0f);
    std::vector<float4> lobes(M);
    const float* tr = ctx->mat_transmission.empty() ? nullptr : ctx->mat_transmission.data();
    const float* sc = ctx->mat_scattering.empty() ? nullptr : ctx->mat_scattering.data();
    const float* th = ctx->mat_thickness_cm.empty() ? nullptr : ctx->mat_thickness_cm.data();
    for (uint32_t m = 0; m < M; ++m) {
        float sum_r = 0.0f, sum_t = 0.0f, sum_s = 0.0f;
        const float thick = th ? th[m] : 2.5f;
        const float ex = thick / 2.5f;
        for (uint32_t b = 0; b < B; ++b) {
            const float a = ctx->mat_absorption[(size_t)m * B + b];
            const float refl = 1.0f - a;
            float tau = tr ? tr[(size_t)m * B + b] : 0.0f;
            const float tau_eff = transmitted_factor(a, tau, ex);
            const float sig = sc ? sc[(size_t)m * B + b] : 1.0f;
            tab[((size_t)0 * M + m) * B + b] = (refl * sig) / FS_PI;
            tab[((size_t)1 * M + m) * B + b] = refl * (1.0f - sig);
            tab[((size_t)2 * M + m) * B + b] = tau_eff;
            sum_r += refl; sum_t += tau; sum_s += sig;
        }
        const float mr = sum_r / (float)B, mt = sum_t / (float)B, ms = sum_s / (float)B;
        const float tot = mr + mt;
        const float t1 = (tot > 0.0f) ? mt / tot : 0.0f;
        const float ps = (1.0f - t1) * (1.0f - ms);
        const float t2 = t1 + ps;
        const float pd = 1.0f - t2;
        lobes[m] = make_float4(t1, t2, ps, pd);
    }
    cudaFree(ctx->d_bsdf_tab); cudaFree(ctx->d_lobes); ctx->d_bsdf_tab = nullptr; ctx->d_lobes = nullptr;
    CK(cudaMalloc(&ctx->d_bsdf_tab, sizeof(float) * tab.size()));
    CK(cudaMalloc(&ctx->d_lobes, sizeof(float4) * lobes.size()));
    CK(cudaMemcpyAsync(ctx->d_bsdf_tab, tab.data(), sizeof(float) * tab.size(), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(ctx->d_lobes, lobes.data(), sizeof(float4) * lobes.size(), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return FS_OK;
}

int fs_scene_commit(fs_ctx* ctx)
{
    if (!ctx) return FS_ERR_INVALID;
    if (!ctx->tris_set || !ctx->mats_set) return fail(ctx, FS_ERR_STATE, "fs_scene_commit: set triangles and materials first");
    nvtx_range nv("fs_scene_commit (BVH build)");
    dev_guard g(ctx->device);
    if (ctx->n_tris) {
        // validate material ids on the host copy-back of the id array (one-time, commit only)
        std::vector<uint32_t> m(ctx->n_tris);
        CK(cudaMemcpyAsync(m.data(), ctx->d_tri_mat, sizeof(uint32_t) * ctx->n_tris, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        for (uint64_t i = 0; i < ctx->n_tris; ++i)
            if (m[i] >= ctx->n_mats) return fail(ctx, FS_ERR_INVALID, "triangle material id out of range");
    }
    if (ctx->cfg.flags & FS_FLAG_MATERIAL_MODEL) {
        int rc = build_material_model(ctx);
        if (rc) return rc;
    }
    if (int rc = build_occlusion_table(ctx)) return rc;
    uint64_t bvh_launches = 0;
    CK(fs_bvh_build(ctx->stream, ctx->d_verts, ctx->d_tri_mat, ctx->n_tris, &ctx->bvh, &bvh_launches,
                    ctx->tune.leaf_max, ctx->tune.builder, ctx->tune.collapse | (ctx->tune.w8 ? 4u : 0u)));
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->launches.fetch_add(bvh_launches);
    ctx->stats.bvh_nodes = ctx->bvh.n_inner;
    if (getenv("FS_VERBOSE")) fprintf(stderr, "[frequensee] BVH: %u triangles, %u BVH2 nodes, %u reachable 4-wide nodes (%.1f MB)\n",
                                      ctx->bvh.n_tris, ctx->bvh.n_inner, ctx->bvh.n_wide, ctx->bvh.n_wide * 64.0 / 1e6);
    if (getenv("FS_VERBOSE") && ctx->bvh.w8nodes) fprintf(stderr, "[frequensee] BVH: %u 8-wide compressed nodes (%.1f MB)\n", ctx->bvh.n_w8, ctx->bvh.n_w8 * 80.0 / 1e6);
    ctx->stats.bvh_max_leaf = ctx->bvh.max_leaf;
    ctx->trav = fs_choose_traversal(ctx->tune, ctx->bvh);
    apply_l2_policy(ctx);
    ctx->committed = true;
    ctx->verts_dirty = false;
    ctx->diff_valid = false;
    return FS_OK;
}

static bool host_is_pinned(const void* p);

int fs_scene_update_vertices(fs_ctx* ctx, const float* verts, uint64_t first_tri, uint64_t n_tris)
{
    if (!ctx) return FS_ERR_INVALID;
    if (!ctx->tris_set) return fail(ctx, FS_ERR_STATE, "fs_scene_update_vertices: call fs_scene_set_triangles first");
    if (n_tris && !verts) return fail(ctx, FS_ERR_INVALID, "fs_scene_update_vertices: null array");
    if (first_tri > ctx->n_tris || n_tris > ctx->n_tris - first_tri)
        return fail(ctx, FS_ERR_INVALID, "fs_scene_update_vertices: triangle range outside the scene");
    for (uint64_t i = 0; i < n_tris * 9; ++i)
        if (!(verts[i] == verts[i]) || fabsf(verts[i]) > 1e18f) return fail(ctx, FS_ERR_INVALID, "non-finite vertex");
    if (!n_tris) return FS_OK;
    dev_guard g(ctx->device);
    // stream-ordered after any trace still in flight, before the next refit.  A pageable source is staged by the driver
    // before the call returns; a page-locked one is read by the copy engine later, so wait for it (the caller may reuse
    // the buffer as soon as this returns)
    CK(cudaMemcpyAsync(ctx->d_verts + first_tri * 9, verts, sizeof(float) * 9 * n_tris, cudaMemcpyHostToDevice, ctx->stream));
    if (host_is_pinned(verts)) CK(cudaStreamSynchronize(ctx->stream));
    if (ctx->committed) ctx->verts_dirty = true;
    return FS_OK;
}

int fs_scene_refit(fs_ctx* ctx, float* cost_ratio_out)
{
    if (!ctx) return FS_ERR_INVALID;
    if (!ctx->committed) return fail(ctx, FS_ERR_STATE, "fs_scene_refit: call fs_scene_commit first");
    nvtx_range nv("fs_scene_refit");
    if (ctx->tune.w8) {                 // the 8-wide nodes (experiment knob FS_TUNE_W8) are rebuilt, not refitted
        int rc = fs_scene_commit(ctx);
        if (rc == FS_OK && cost_ratio_out) *cost_ratio_out = 1.0f;
        return rc;
    }
    dev_guard g(ctx->device);
    uint64_t launches = 0;
    float ratio = 1.0f;
    CK(fs_bvh_refit(ctx->stream, ctx->d_verts, &ctx->bvh, &launches, &ratio));
    ctx->launches.fetch_add(launches);
    ctx->trav = fs_choose_traversal(ctx->tune, ctx->bvh);
    ctx->verts_dirty = false;
    ctx->diff_valid = false;
    if (cost_ratio_out) *cost_ratio_out = ratio;
    return FS_OK;
}

// ---- trace -----------------------------------------------------------------------------------
static void fill_params(fs_ctx* ctx, fs_trace_params* tp, const float lis[3], uint64_t n_paths, uint32_t max_depth,
                        uint64_t seed)
{
    const fs_config& c = ctx->cfg;
    memset(tp, 0, sizeof(*tp));
    const fs_traversal& tr = ctx->trav;
    tp->bv.nodes_tex = tr.tex ? (unsigned long long)ctx->bvh.nodes_tex : 0ull;
    tp->bv.tris_tex = tr.tex ? (unsigned long long)ctx->bvh.tris_tex : 0ull;
    tp->bv.wnodes = tr.nodes != FS_NODES_BVH2 ? ctx->bvh.wnodes : nullptr;
    tp->bv.wnodes_tex = tr.tex ? (unsigned long long)ctx->bvh.wnodes_tex : 0ull;
    const bool w8 = tr.nodes == FS_NODES_W8;
    tp->bv.w8nodes = w8 ? ctx->bvh.w8nodes : nullptr; tp->bv.tris8 = w8 ? ctx->bvh.tris8 : nullptr; tp->bv.tri8_map = w8 ? ctx->bvh.tri8_map : nullptr;
    tp->bv.w8_magic = 0x47000000u;
    for (int a = 0; a < 3; ++a) { tp->bv.qbase[a] = ctx->bvh.qbase[a]; tp->bv.qscale[a] = ctx->bvh.qscale[a]; }
    tp->bv.nodes = ctx->bvh.nodes; tp->bv.tris = ctx->bvh.tris; tp->bv.tri_orig = ctx->bvh.tri_orig;
    tp->bv.tri_mat = ctx->bvh.tri_mat; tp->bv.tri_nm = ctx->bvh.tri_nm; tp->bv.n_tris = ctx->bvh.n_tris; tp->bv.n_inner = ctx->bvh.n_inner;
    tp->top = ctx->bvh.top_nodes; tp->n_top = ctx->bvh.n_top;
    const bool model = (c.flags & FS_FLAG_MATERIAL_MODEL) && ctx->d_lobes;
    tp->refl_over_pi = model ? ctx->d_bsdf_tab : ctx->d_refl_over_pi; tp->n_mats = ctx->n_mats;
    tp->lobes = model ? ctx->d_lobes : nullptr;
    tp->ep.min_seg = c.min_seg; tp->ep.pdf_exponent = c.pdf_exponent; tp->ep.n_bands = c.n_bands;
    for (int b = 0; b < FS_MAX_BANDS; ++b) tp->ep.air[b] = c.air_absorption[b];
    tp->n_bins = c.n_bins; tp->bin_ms = c.bin_ms; tp->rr_prob = c.rr_prob; tp->eps_offset = c.eps_offset;
    tp->eps_connect = c.eps_connect; tp->sound_speed = c.sound_speed; tp->energy_clamp = c.energy_clamp;
    tp->energy_gain = c.energy_gain; tp->max_depth = max_depth;
    tp->seed_lo = (uint32_t)seed; tp->seed_hi = (uint32_t)(seed >> 32);
    tp->n_paths = n_paths;
    tp->src_pos = ctx->d_src_pos;
    if (lis) { tp->lis[0] = lis[0]; tp->lis[1] = lis[1]; tp->lis[2] = lis[2]; }
    tp->flags = c.flags;
    tp->dir_orient = ctx->dir_sources ? ctx->d_dir_orient : nullptr;
    tp->dir_gain = ctx->d_dir_gain; tp->n_dir_patterns = ctx->dir_patterns;
}

// with source orientations installed, a trace must name exactly that many sources; checked before anything is enqueued
static int check_dir_sources(fs_ctx* ctx, uint32_t n_sources, const char* who)
{
    if (!ctx->dir_sources || n_sources == ctx->dir_sources) return FS_OK;
    return fail(ctx, FS_ERR_INVALID, (std::string(who) + ": n_sources (" + std::to_string(n_sources) + ") differs from the " +
                                      std::to_string(ctx->dir_sources) + " source orientations installed by fs_set_source_directivity").c_str());
}

static int ensure_hist(fs_ctx* ctx, uint32_t n_sources)
{
    if (ctx->d_hist && ctx->hist_sources >= n_sources) return FS_OK;
    cudaFree(ctx->d_hist); ctx->d_hist = nullptr; ctx->hist_sources = 0; ctx->hist_cur_sources = 0;
    const size_t n = (size_t)n_sources * ctx->cfg.n_bands * ctx->cfg.n_bins;
    CK(cudaMalloc(&ctx->d_hist, 8 * n));
    ctx->hist_sources = n_sources;
    return FS_OK;
}

// FS_FLAG_NOISE_STATS: the second-moment buffer for n_sources, zeroed on the context stream like the histogram; null
// without the flag
static int prepare_m2(fs_ctx* ctx, uint32_t n_sources, ulonglong2** out)
{
    *out = nullptr;
    if (!(ctx->cfg.flags & FS_FLAG_NOISE_STATS)) return FS_OK;
    const size_t n = (size_t)n_sources * (ctx->cfg.n_bands + 1u) * ctx->cfg.n_bins;
    if (!ctx->d_m2 || ctx->m2_sources < n_sources) {
        cudaFree(ctx->d_m2); ctx->d_m2 = nullptr; ctx->m2_sources = 0;
        CK(cudaMalloc(&ctx->d_m2, sizeof(ulonglong2) * n));
        ctx->m2_sources = n_sources;
    }
    CK(cudaMemsetAsync(ctx->d_m2, 0, sizeof(ulonglong2) * n, ctx->stream));
    *out = ctx->d_m2;
    return FS_OK;
}

// bookkeeping of the histogram that fs_build_ir* read: its source count and the path count of every source (per_source:
// host [n_sources] after fs_trace_sources*, null = n_paths for all)
static void set_hist_counts(fs_ctx* ctx, uint32_t n_sources, uint64_t n_paths, const uint64_t* per_source)
{
    ctx->hist_n_paths = n_paths; ctx->hist_cur_sources = n_sources;
    if (per_source) ctx->hist_src_paths.assign(per_source, per_source + n_sources);
    else ctx->hist_src_paths.clear();
}
static uint64_t hist_paths(const fs_ctx* ctx, uint32_t source)
{
    return source < ctx->hist_src_paths.size() ? ctx->hist_src_paths[source] : ctx->hist_n_paths;
}

// per-source budgets (fs_trace_sources*) in the form trace_common takes: packed positions, offsets, depths, maxima
struct fs_src_table {
    std::vector<float> pos;          // [S][3]
    std::vector<uint64_t> off;       // [S+1]: off[s] = first work index of source s, off[S] = G
    std::vector<uint32_t> depth;     // [S]
    std::vector<uint64_t> n_paths;   // [S]
    uint64_t n_max; uint32_t d_max;
};

// validates a per-source call completely before anything is enqueued (the context is left as it was on every error)
static int prepare_sources(fs_ctx* ctx, const char* who, const fs_source_desc* src, uint32_t n_sources, const float lis_pos[3],
                           fs_src_table* t)
{
    std::string w(who);
    if (!ctx->committed) return fail(ctx, FS_ERR_STATE, (w + ": call fs_scene_commit first").c_str());
    if (ctx->verts_dirty) return fail(ctx, FS_ERR_STATE, (w + ": triangles were moved; call fs_scene_refit (or fs_scene_commit) first").c_str());
    if (!src || !lis_pos || n_sources == 0) return fail(ctx, FS_ERR_INVALID, (w + ": null sources / listener or no source").c_str());
    if ((uint64_t)n_sources * ctx->cfg.n_bins >= 0xffffffffull) return fail(ctx, FS_ERR_INVALID, (w + ": n_sources * n_bins too large").c_str());
    const uint32_t flags = ctx->cfg.flags;
    const uint32_t lim = (flags & FS_FLAG_MIS) ? 32u : (flags & FS_FLAG_CONNECT_ALL) ? 63u : 1024u;
    t->pos.resize(3ull * n_sources); t->off.resize(n_sources + 1ull); t->depth.resize(n_sources); t->n_paths.resize(n_sources);
    t->n_max = 0; t->d_max = 0;
    uint64_t G = 0;
    for (uint32_t s = 0; s < n_sources; ++s) {
        const fs_source_desc& d = src[s];
        if (d.n_paths == 0) return fail(ctx, FS_ERR_INVALID, (w + ": n_paths of source " + std::to_string(s) + " is 0").c_str());
        if (d.max_depth > lim)
            return fail(ctx, FS_ERR_INVALID, (w + ": max_depth of source " + std::to_string(s) + " > " + std::to_string(lim) +
                                              " (the limit of this flag mode)").c_str());
        if ((flags & FS_FLAG_SHARE_LISTENER) && d.max_depth != src[0].max_depth)
            return fail(ctx, FS_ERR_INVALID, (w + ": FS_FLAG_SHARE_LISTENER needs the same max_depth for every source "
                                                  "(one shared listener walk serves one ray budget)").c_str());
        if (G + d.n_paths < G) return fail(ctx, FS_ERR_INVALID, (w + ": total path count overflows").c_str());
        for (int a = 0; a < 3; ++a) t->pos[3ull * s + a] = d.pos[a];
        t->off[s] = G; t->depth[s] = d.max_depth; t->n_paths[s] = d.n_paths;
        G += d.n_paths;
        if (d.n_paths > t->n_max) t->n_max = d.n_paths;
        if (d.max_depth > t->d_max) t->d_max = d.max_depth;
    }
    t->off[n_sources] = G;
    return FS_OK;
}

// the listener cache is [max_depth + 2][n_paths] float4; without room for it the shared keying still holds, the listener
// subpaths are then simply traced in place by every batch
static bool lis_cache_fits(fs_ctx* ctx, uint64_t n_paths, uint32_t max_depth)
{
    if (ctx->lis_cache_n >= n_paths && ctx->lis_cache_depth >= max_depth) return true;
    size_t free_b = 0, total_b = 0;
    if (cudaMemGetInfo(&free_b, &total_b) != cudaSuccess) { (void)cudaGetLastError(); return false; }
    const double need = 16.0 * (double)n_paths * (double)(max_depth + 2u);
    return need < 0.25 * (double)free_b;
}

// tab (per-source budgets, fs_trace_sources*): src_pos = tab->pos, n_paths = the largest budget, max_depth = the largest depth,
// the work range is [0, G) with G = tab->off[S]; null = uniform budgets, G = n_sources * n_paths
static int trace_common(fs_ctx* ctx, const float* src_pos, uint32_t n_sources, const float lis_pos[3],
                        uint64_t n_paths, uint64_t g_first, uint64_t g_count, uint32_t max_depth, uint64_t seed,
                        unsigned long long* d_hist, fs_path_dbg* d_dbg, const fs_src_table* tab = nullptr,
                        ulonglong2* d_m2 = nullptr)
{
    nvtx_range nv("fs_trace");
    if (!ctx->committed) return fail(ctx, FS_ERR_STATE, "fs_trace: call fs_scene_commit first");
    if (ctx->verts_dirty) return fail(ctx, FS_ERR_STATE, "fs_trace: triangles were moved; call fs_scene_refit (or fs_scene_commit) first");
    if (!src_pos || !lis_pos || n_sources == 0) return fail(ctx, FS_ERR_INVALID, "fs_trace: null positions / no source");
    if (n_paths == 0) return fail(ctx, FS_ERR_INVALID, "fs_trace: n_paths must be > 0");
    if (max_depth > 1024) return fail(ctx, FS_ERR_INVALID, "fs_trace: max_depth > 1024");
    const uint64_t G = tab ? tab->off[n_sources] : (uint64_t)n_sources * n_paths;
    if (g_first + g_count > G || g_first + g_count < g_first) return fail(ctx, FS_ERR_INVALID, "fs_trace: work range exceeds the sources' paths");
    if ((uint64_t)n_sources * ctx->cfg.n_bins >= 0xffffffffull) return fail(ctx, FS_ERR_INVALID, "fs_trace: n_sources * n_bins too large");
    if (int rc = check_dir_sources(ctx, n_sources, "fs_trace")) return rc;
    // an overflow of the PREVIOUS trace that nobody has looked at yet: report it now if its flag has landed; if it is
    // still in flight the device flag is left set (reset_ovf = 0) so that this call's copy carries it
    int rc_ovf = check_overflow(ctx, false);
    if (rc_ovf) return rc_ovf;
    const int reset_ovf = ctx->overflow_pending ? 0 : 1;
    ctx->m2_valid = false;                    // the callers that pass d_m2 set it again once the trace is enqueued
    if (ctx->src_cap < n_sources) {
        cudaFree(ctx->d_src_pos); ctx->d_src_pos = nullptr;
        CK(cudaMalloc(&ctx->d_src_pos, sizeof(float) * 3 * n_sources));
        ctx->src_cap = n_sources;
    }
    CK(cudaMemcpyAsync(ctx->d_src_pos, src_pos, sizeof(float) * 3 * n_sources, cudaMemcpyHostToDevice, ctx->stream));
    if (tab) {
        if (ctx->src_tab_cap < n_sources) {
            cudaFree(ctx->d_src_tab); ctx->d_src_tab = nullptr; ctx->src_tab_cap = 0;
            CK(cudaMalloc(&ctx->d_src_tab, 12ull * n_sources + 8ull));
            ctx->src_tab_cap = n_sources;
        }
        CK(cudaMemcpyAsync(ctx->d_src_tab, tab->off.data(), 8ull * (n_sources + 1ull), cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaMemcpyAsync((char*)ctx->d_src_tab + 8ull * (n_sources + 1ull), tab->depth.data(), 4ull * n_sources,
                           cudaMemcpyHostToDevice, ctx->stream));
    }
    // equal batches: every bounce of a batch is a pair of launches whose cost has a fixed part (launch + the tail of the
    // slowest rays), so 1.25 M pairs run as 1 x 1.25 M or 2 x 0.63 M, never as 1 M + a 0.25 M remainder.
    // Batches alternate between up to tune.streams lanes (own stream + own wavefront buffers): a traversal launch ends
    // with a tail of a few long rays on an almost empty GPU, and the other lane's kernels fill it.  Histogram sums are
    // integer atomics, so the result does not depend on how batches interleave.  Per-kernel timing (FS_FLAG_TIME_KERNELS)
    // and the debug record path run on one lane so that every kernel is timed alone.
    uint32_t cap_cfg = ctx->cfg.max_batch_paths;
    uint32_t n_lanes = ctx->tune.streams;
    if ((ctx->cfg.flags & FS_FLAG_TIME_KERNELS) || d_dbg) n_lanes = 1;
    if ((ctx->cfg.flags & FS_FLAG_SHARE_LISTENER) && (ctx->cfg.flags & (FS_FLAG_FUSED_EXTEND | FS_FLAG_BRUTE_FORCE)))
        return fail(ctx, FS_ERR_INVALID, "FS_FLAG_SHARE_LISTENER needs the wavefront path");
    if ((ctx->cfg.flags & FS_FLAG_MATERIAL_MODEL) && (ctx->cfg.flags & (FS_FLAG_FUSED_EXTEND | FS_FLAG_BRUTE_FORCE)))
        return fail(ctx, FS_ERR_INVALID, "FS_FLAG_MATERIAL_MODEL needs the wavefront path");
    if (ctx->cfg.flags & FS_FLAG_MIS) {
        if (max_depth > 32) return fail(ctx, FS_ERR_INVALID, "FS_FLAG_MIS: max_depth <= 32");
        if (ctx->cfg.flags & FS_FLAG_MATERIAL_MODEL) return fail(ctx, FS_ERR_INVALID, "FS_FLAG_MIS: diffuse surfaces only (not with FS_FLAG_MATERIAL_MODEL)");
        if (ctx->cfg.flags & FS_FLAG_SHARE_LISTENER) return fail(ctx, FS_ERR_INVALID, "FS_FLAG_MIS: not with FS_FLAG_SHARE_LISTENER");
    }
    if (ctx->cfg.flags & (FS_FLAG_CONNECT_ALL | FS_FLAG_MIS)) {
        // up to (depth+1)^2 connection rays per pair: keep a batch's ray queue near 2^24 entries; ids are pair << 12 | s << 6 | t
        if (max_depth > 63) return fail(ctx, FS_ERR_INVALID, "FS_FLAG_CONNECT_ALL: max_depth <= 63");
        if (d_dbg) return fail(ctx, FS_ERR_INVALID, "FS_FLAG_CONNECT_ALL: no per-path debug records");
        if (ctx->cfg.flags & (FS_FLAG_FUSED_EXTEND | FS_FLAG_BRUTE_FORCE)) return fail(ctx, FS_ERR_INVALID, "FS_FLAG_CONNECT_ALL needs the wavefront path");
        uint32_t lim = (1u << 24) / ((max_depth + 1u) * (max_depth + 1u));
        if (lim < 256u) lim = 256u;
        if (lim > (1u << 20)) lim = 1u << 20;
        if (cap_cfg > lim) cap_cfg = lim;
        n_lanes = 1;
    }
    // a job that will use the persistent per-batch kernel runs on at most tune.mega_lanes lanes (same rule as in
    // launch_batch_split: batches of >= FS_MEGA_MIN_BATCH = 2^17 pairs on a scene of >= 4096 triangles, or FS_TUNE_MEGA=1)
    {
        const uint64_t nb1 = g_count ? (g_count + cap_cfg - 1) / cap_cfg : 1;
        const uint64_t cap1 = g_count ? (g_count + nb1 - 1) / nb1 : 1;
        const bool mega_job = !(ctx->cfg.flags & (FS_FLAG_COUNT_VISITS | FS_FLAG_CONNECT_ALL | FS_FLAG_MIS)) && max_depth >= 1 &&
                              (ctx->tune.mega == 1u || (ctx->tune.mega == 2u && cap1 >= FS_MEGA_MIN_BATCH && ctx->bvh.n_tris >= 4096u &&
                                                        ctx->conv_active.load() == 0));
        if (mega_job && n_lanes > ctx->tune.mega_lanes) n_lanes = ctx->tune.mega_lanes;
        // ... and on one lane when half of it would fall below the size from which the persistent kernel pays
        while (mega_job && ctx->tune.mega == 2u && n_lanes > 1 && g_count / n_lanes < FS_MEGA_MIN_BATCH) --n_lanes;
    }
    while (n_lanes > 1 && g_count / n_lanes < (1u << 17)) --n_lanes;            // small jobs: not worth a second set of launches
    uint64_t n_batches = g_count ? (g_count + cap_cfg - 1) / cap_cfg : 1;
    if (n_batches < n_lanes) n_batches = n_lanes;
    if (n_batches % n_lanes) n_batches += n_lanes - n_batches % n_lanes;
    const uint32_t cap = (uint32_t)(g_count ? (g_count + n_batches - 1) / n_batches : 1);
    ctx->lanes[0].stream = ctx->stream;                       // lane 0 = the caller's stream; nothing else is rebound
    ctx->cur_lanes = n_lanes;
    for (uint32_t l = 0; l < n_lanes; ++l) CK(fs_wave_alloc(ctx, &ctx->lanes[l], cap, max_depth));
    fs_trace_params tp;
    fill_params(ctx, &tp, lis_pos, n_paths, max_depth, seed);
    tp.n_src = n_sources;
    CK(cudaEventRecord(ctx->ev0, ctx->stream));
    ctx->kev_used = 0; ctx->tev_used = 0; ctx->stats.extend_launches = 0; ctx->stats.persistent_launches = 0;
    CK(fs_wave_reset_counters(ctx, reset_ovf));
    // FS_FLAG_SHARE_LISTENER with more than one source's worth of work: trace the n_paths listener subpaths once, now, and
    // let every source batch copy them in (smaller jobs just use the shared keying and trace them in place)
    if ((ctx->cfg.flags & FS_FLAG_SHARE_LISTENER) && !(ctx->cfg.flags & FS_FLAG_CONNECT_ALL) && !d_dbg && n_sources > 1 &&
        g_count > n_paths && max_depth > 0 && !(ctx->cfg.flags & (FS_FLAG_FUSED_EXTEND | FS_FLAG_BRUTE_FORCE)) &&
        lis_cache_fits(ctx, n_paths, max_depth)) {
        if (ctx->lis_cache_n < n_paths || ctx->lis_cache_depth < max_depth) {
            cudaFree(ctx->lis_rec); cudaFree(ctx->lis_end); ctx->lis_rec = ctx->lis_end = nullptr; ctx->lis_cache_n = 0;
            CK(cudaMalloc(&ctx->lis_rec, sizeof(float4) * (size_t)n_paths * (max_depth + 1ull)));
            CK(cudaMalloc(&ctx->lis_end, sizeof(float4) * (size_t)n_paths));
            ctx->lis_cache_n = n_paths; ctx->lis_cache_depth = max_depth;
        }
        tp.lis_rec = ctx->lis_rec; tp.lis_end = ctx->lis_end;
        tp.lis_mode = 1;
        for (uint64_t i0 = 0; i0 < n_paths; i0 += cap) {
            tp.g_first = i0;
            tp.batch = (uint32_t)(n_paths - i0 < cap ? n_paths - i0 : cap);
            CK(fs_wave_trace_batch(ctx, &ctx->lanes[0], tp, d_hist, nullptr, nullptr));
        }
        tp.lis_mode = 2;
    }
    // per-source budgets: set after the listener pass, which traces max n_s listener subpaths of one uniform source
    if (tab) {
        tp.src_off = (const uint64_t*)ctx->d_src_tab;
        tp.src_depth = (const uint32_t*)((const char*)ctx->d_src_tab + 8ull * (n_sources + 1ull));
    }
    if (n_lanes > 1) {
        CK(cudaEventRecord(ctx->ev_fork, ctx->stream));
        for (uint32_t l = 1; l < n_lanes; ++l) CK(cudaStreamWaitEvent(ctx->lanes[l].stream, ctx->ev_fork, 0));
    }
    uint32_t b = 0;
    for (uint64_t done = 0; done < g_count; ++b) {
        uint64_t nb = g_count - done;
        if (nb > cap) nb = cap;
        tp.g_first = g_first + done;
        tp.batch = (uint32_t)nb;
        const uint32_t l = b % n_lanes;
        CK(fs_wave_trace_batch(ctx, &ctx->lanes[l], tp, d_hist, (d_dbg && l == 0) ? d_dbg + done : nullptr, d_m2));
        done += nb;
    }
    for (uint32_t l = 1; l < n_lanes; ++l) {
        CK(cudaEventRecord(ctx->lanes[l].done, ctx->lanes[l].stream));
        CK(cudaStreamWaitEvent(ctx->stream, ctx->lanes[l].done, 0));
    }
    CK(cudaEventRecord(ctx->ev1, ctx->stream));
    // one 4-byte copy of the overflow flag on every return path (the async ones included)
    CK(cudaMemcpyAsync(ctx->h_overflow, &ctx->d_counters->overflow, sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaEventRecord(ctx->ev_overflow, ctx->stream));
    ctx->overflow_pending = true;
    ctx->timed = true;
    ctx->stats.paths = g_count;
    return FS_OK;
}

// synchronises the context stream and fills the host-side statistics of the last trace
static int finish_stats(fs_ctx* ctx)
{
    fs_dev_counters h;
    CK(cudaMemcpyAsync(&h, ctx->d_counters, sizeof(h), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->stats.ext_rays = h.ext_rays; ctx->stats.shadow_rays = h.shadow_rays; ctx->stats.connected = h.connected;
    ctx->stats.node_visits = h.node_visits; ctx->stats.tri_tests = h.tri_tests;
    ctx->stats.shadow_node_visits = h.shadow_node_visits; ctx->stats.shadow_tri_tests = h.shadow_tri_tests;
    if (getenv("FS_VERBOSE") && h.max_steps) {
        fprintf(stderr, "[frequensee] node steps per ray: max %u; rays by steps/8:", h.max_steps);
        for (int b = 0; b < 16; ++b) fprintf(stderr, " %u", h.steps_hist[b]);
        fprintf(stderr, "\n");
    }
    if (ctx->kev_used) {
        float ext = 0.f, con = 0.f, evl = 0.f, ms;
        for (size_t i = 0; i + 3 < ctx->kev_used; i += 4) {
            if (cudaEventElapsedTime(&ms, ctx->kev[i], ctx->kev[i + 1]) == cudaSuccess) ext += ms;
            if (cudaEventElapsedTime(&ms, ctx->kev[i + 1], ctx->kev[i + 2]) == cudaSuccess) con += ms;
            if (cudaEventElapsedTime(&ms, ctx->kev[i + 2], ctx->kev[i + 3]) == cudaSuccess) evl += ms;
        }
        (void)cudaGetLastError();
        ctx->stats.extend_ms = ext; ctx->stats.connect_ms = con; ctx->stats.eval_ms = evl;
        float tr = 0.f;
        const bool verbose = getenv("FS_VERBOSE") != nullptr;
        for (size_t i = 0; i + 1 < ctx->tev_used; i += 2)
            if (cudaEventElapsedTime(&ms, ctx->tev[i], ctx->tev[i + 1]) == cudaSuccess) {
                tr += ms;
                if (verbose) fprintf(stderr, "[frequensee] trace launch %zu: %.3f ms\n", i / 2, ms);
            }
        (void)cudaGetLastError();
        ctx->stats.trace_ms = tr;
    }
    if (ctx->timed) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1) == cudaSuccess) ctx->stats.last_trace_ms = ms;
        else (void)cudaGetLastError();
    }
    if (ctx->ir_timed) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, ctx->ev_ir0, ctx->ev_ir1) == cudaSuccess) ctx->stats.last_ir_ms = ms;
        else (void)cudaGetLastError();
    }
    return check_overflow(ctx, true);
}

int fs_trace(fs_ctx* ctx, const float* src_pos, uint32_t n_sources, const float lis_pos[3], uint64_t n_paths,
             uint32_t max_depth, uint64_t seed, uint64_t* hist_out)
{
    if (!ctx) return FS_ERR_INVALID;
    dev_guard g(ctx->device);
    if (n_sources == 0) return fail(ctx, FS_ERR_INVALID, "fs_trace: no source");
    int rc = check_dir_sources(ctx, n_sources, "fs_trace");
    if (rc) return rc;
    rc = ensure_hist(ctx, n_sources);
    if (rc) return rc;
    const size_t hn = (size_t)n_sources * ctx->cfg.n_bands * ctx->cfg.n_bins;
    CK(cudaMemsetAsync(ctx->d_hist, 0, 8 * hn, ctx->stream));            // FlushEnergyBuffer, COMP.h:76-79
    ulonglong2* d_m2 = nullptr;
    if ((rc = prepare_m2(ctx, n_sources, &d_m2))) return rc;
    rc = trace_common(ctx, src_pos, n_sources, lis_pos, n_paths, 0, (uint64_t)n_sources * n_paths, max_depth, seed,
                      ctx->d_hist, nullptr, nullptr, d_m2);
    if (rc) return rc;
    set_hist_counts(ctx, n_sources, n_paths, nullptr);
    ctx->m2_valid = d_m2 != nullptr;
    if (hist_out) {
        CK(cudaMemcpyAsync(hist_out, ctx->d_hist, 8 * hn, cudaMemcpyDeviceToHost, ctx->stream));
        return finish_stats(ctx);
    }
    return FS_OK;
}

// shard forms; d_m2 (device [S][B+1][K], null = none) accumulates the second moments like d_hist (fs_multi)
static int trace_range_device(fs_ctx* ctx, const float* src_pos, uint32_t n_sources, const float lis_pos[3],
                              uint64_t n_paths, uint64_t g_first, uint64_t g_count, uint32_t max_depth, uint64_t seed,
                              void* d_hist, ulonglong2* d_m2, int zero_first)
{
    if (!ctx) return FS_ERR_INVALID;
    if (!d_hist) return fail(ctx, FS_ERR_INVALID, "fs_trace_range_device: null histogram");
    if (int rc = check_dir_sources(ctx, n_sources, "fs_trace_range_device")) return rc;
    dev_guard g(ctx->device);
    const size_t hn = (size_t)n_sources * ctx->cfg.n_bands * ctx->cfg.n_bins;
    if (zero_first) CK(cudaMemsetAsync(d_hist, 0, 8 * hn, ctx->stream));
    if (zero_first && d_m2) CK(cudaMemsetAsync(d_m2, 0, sizeof(ulonglong2) * (size_t)n_sources * (ctx->cfg.n_bands + 1u) * ctx->cfg.n_bins, ctx->stream));
    return trace_common(ctx, src_pos, n_sources, lis_pos, n_paths, g_first, g_count, max_depth, seed,
                        (unsigned long long*)d_hist, nullptr, nullptr, d_m2);
}

int fs_trace_range_device(fs_ctx* ctx, const float* src_pos, uint32_t n_sources, const float lis_pos[3],
                          uint64_t n_paths, uint64_t g_first, uint64_t g_count, uint32_t max_depth, uint64_t seed,
                          void* d_hist, int zero_first)
{
    return trace_range_device(ctx, src_pos, n_sources, lis_pos, n_paths, g_first, g_count, max_depth, seed, d_hist, nullptr,
                              zero_first);
}

int fs_trace_range(fs_ctx* ctx, const float* src_pos, uint32_t n_sources, const float lis_pos[3], uint64_t n_paths,
                   uint64_t g_first, uint64_t g_count, uint32_t max_depth, uint64_t seed, uint64_t* hist_inout)
{
    if (!ctx) return FS_ERR_INVALID;
    if (!hist_inout) return fail(ctx, FS_ERR_INVALID, "fs_trace_range: null histogram");
    dev_guard g(ctx->device);
    int rc = check_dir_sources(ctx, n_sources, "fs_trace_range");
    if (rc) return rc;
    rc = ensure_hist(ctx, n_sources);
    if (rc) return rc;
    const size_t hn = (size_t)n_sources * ctx->cfg.n_bands * ctx->cfg.n_bins;
    CK(cudaMemcpyAsync(ctx->d_hist, hist_inout, 8 * hn, cudaMemcpyHostToDevice, ctx->stream));
    rc = trace_common(ctx, src_pos, n_sources, lis_pos, n_paths, g_first, g_count, max_depth, seed, ctx->d_hist, nullptr);
    if (rc) return rc;
    set_hist_counts(ctx, n_sources, n_paths, nullptr);
    CK(cudaMemcpyAsync(hist_inout, ctx->d_hist, 8 * hn, cudaMemcpyDeviceToHost, ctx->stream));
    return finish_stats(ctx);
}

int fs_trace_debug(fs_ctx* ctx, const float* src_pos, uint32_t n_sources, const float lis_pos[3], uint64_t n_paths,
                   uint64_t g_first, uint64_t g_count, uint32_t max_depth, uint64_t seed, fs_path_dbg* dbg_out)
{
    if (!ctx) return FS_ERR_INVALID;
    if (!dbg_out) return fail(ctx, FS_ERR_INVALID, "fs_trace_debug: null output");
    dev_guard g(ctx->device);
    int rc = check_dir_sources(ctx, n_sources, "fs_trace_debug");
    if (rc) return rc;
    rc = ensure_hist(ctx, n_sources);
    if (rc) return rc;
    if (ctx->dbg_cap < g_count) {
        cudaFree(ctx->d_dbg); ctx->d_dbg = nullptr; ctx->dbg_cap = 0;
        CK(cudaMalloc(&ctx->d_dbg, sizeof(fs_path_dbg) * g_count));
        ctx->dbg_cap = g_count;
    }
    const size_t hn = (size_t)n_sources * ctx->cfg.n_bands * ctx->cfg.n_bins;
    CK(cudaMemsetAsync(ctx->d_hist, 0, 8 * hn, ctx->stream));
    rc = trace_common(ctx, src_pos, n_sources, lis_pos, n_paths, g_first, g_count, max_depth, seed, ctx->d_hist, ctx->d_dbg);
    if (rc) return rc;
    set_hist_counts(ctx, n_sources, n_paths, nullptr);
    CK(cudaMemcpyAsync(dbg_out, ctx->d_dbg, sizeof(fs_path_dbg) * g_count, cudaMemcpyDeviceToHost, ctx->stream));
    return finish_stats(ctx);
}

static int debug_rays(fs_ctx* ctx, const float* rays, const float* tmax, uint64_t n, float* out_t, uint32_t* out_tri,
                      uint8_t* out_hit)
{
    if (!ctx) return FS_ERR_INVALID;
    if (!ctx->committed) return fail(ctx, FS_ERR_STATE, "commit the scene first");
    if (ctx->verts_dirty) return fail(ctx, FS_ERR_STATE, "triangles were moved; call fs_scene_refit (or fs_scene_commit) first");
    if (n == 0) return FS_OK;
    dev_guard g(ctx->device);
    float *d_rays = nullptr, *d_tmax = nullptr, *d_t = nullptr; uint32_t* d_tri = nullptr; uint8_t* d_hit = nullptr;
    int rc = FS_OK;
    cudaError_t e = cudaSuccess;
    cudaStream_t st = ctx->stream;
    fs_trace_params tp;
    fill_params(ctx, &tp, nullptr, 1, 1, 0);
    do {
        if ((e = cudaMalloc(&d_rays, sizeof(float) * 6 * n)) != cudaSuccess) break;
        if ((e = cudaMemcpyAsync(d_rays, rays, sizeof(float) * 6 * n, cudaMemcpyHostToDevice, st)) != cudaSuccess) break;
        if (out_hit) {
            if ((e = cudaMalloc(&d_tmax, sizeof(float) * n)) != cudaSuccess) break;
            if ((e = cudaMemcpyAsync(d_tmax, tmax, sizeof(float) * n, cudaMemcpyHostToDevice, st)) != cudaSuccess) break;
            if ((e = cudaMalloc(&d_hit, n)) != cudaSuccess) break;
        } else {
            if ((e = cudaMalloc(&d_t, sizeof(float) * n)) != cudaSuccess) break;
            if ((e = cudaMalloc(&d_tri, sizeof(uint32_t) * n)) != cudaSuccess) break;
        }
        if ((e = fs_wave_reset_counters(ctx, 1)) != cudaSuccess) break;
        if ((e = fs_wave_debug_rays(ctx, tp, d_rays, d_tmax, n, d_t, d_tri, d_hit)) != cudaSuccess) break;
        if (out_hit) { if ((e = cudaMemcpyAsync(out_hit, d_hit, n, cudaMemcpyDeviceToHost, st)) != cudaSuccess) break; }
        else {
            if ((e = cudaMemcpyAsync(out_t, d_t, sizeof(float) * n, cudaMemcpyDeviceToHost, st)) != cudaSuccess) break;
            if ((e = cudaMemcpyAsync(out_tri, d_tri, sizeof(uint32_t) * n, cudaMemcpyDeviceToHost, st)) != cudaSuccess) break;
        }
        if ((e = cudaStreamSynchronize(st)) != cudaSuccess) break;
    } while (0);
    if (e != cudaSuccess) cudaStreamSynchronize(st);
    cudaFree(d_rays); cudaFree(d_tmax); cudaFree(d_t); cudaFree(d_tri); cudaFree(d_hit);
    if (e != cudaSuccess) rc = fail_cuda(ctx, e, "fs_debug rays");
    return rc;
}

int fs_debug_closest_hits(fs_ctx* ctx, const float* rays, uint64_t n, float* out_t, uint32_t* out_tri)
{
    if (!rays || !out_t || !out_tri) return ctx ? fail(ctx, FS_ERR_INVALID, "null argument") : FS_ERR_INVALID;
    return debug_rays(ctx, rays, nullptr, n, out_t, out_tri, nullptr);
}
int fs_debug_any_hits(fs_ctx* ctx, const float* rays, const float* tmax, uint64_t n, uint8_t* out_hit)
{
    if (!rays || !tmax || !out_hit) return ctx ? fail(ctx, FS_ERR_INVALID, "null argument") : FS_ERR_INVALID;
    return debug_rays(ctx, rays, tmax, n, nullptr, nullptr, out_hit);
}

// ---- histogram / IR ---------------------------------------------------------------------------
int fs_set_histogram(fs_ctx* ctx, const uint64_t* hist, uint32_t n_sources, uint64_t n_paths)
{
    if (!ctx) return FS_ERR_INVALID;
    if (!hist || n_sources == 0 || n_paths == 0) return fail(ctx, FS_ERR_INVALID, "fs_set_histogram: bad argument");
    dev_guard g(ctx->device);
    int rc = ensure_hist(ctx, n_sources);
    if (rc) return rc;
    const size_t hn = (size_t)n_sources * ctx->cfg.n_bands * ctx->cfg.n_bins;
    CK(cudaMemcpyAsync(ctx->d_hist, hist, 8 * hn, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    set_hist_counts(ctx, n_sources, n_paths, nullptr);
    ctx->m2_valid = false;
    return FS_OK;
}

int fs_set_histogram_device(fs_ctx* ctx, const void* d_hist, uint32_t n_sources, uint64_t n_paths)
{
    if (!ctx) return FS_ERR_INVALID;
    if (!d_hist || n_sources == 0 || n_paths == 0) return fail(ctx, FS_ERR_INVALID, "fs_set_histogram_device: bad argument");
    dev_guard g(ctx->device);
    int rc = ensure_hist(ctx, n_sources);
    if (rc) return rc;
    const size_t hn = (size_t)n_sources * ctx->cfg.n_bands * ctx->cfg.n_bins;
    CK(cudaMemcpyAsync(ctx->d_hist, d_hist, 8 * hn, cudaMemcpyDeviceToDevice, ctx->stream));
    set_hist_counts(ctx, n_sources, n_paths, nullptr);
    ctx->m2_valid = false;
    return FS_OK;
}

int fs_set_histogram_sources_device(fs_ctx* ctx, const void* d_hist, uint32_t n_sources, const uint64_t* n_paths)
{
    if (!ctx) return FS_ERR_INVALID;
    if (!d_hist || !n_paths || n_sources == 0) return fail(ctx, FS_ERR_INVALID, "fs_set_histogram_sources_device: bad argument");
    uint64_t n_max = 0;
    for (uint32_t s = 0; s < n_sources; ++s) {
        if (n_paths[s] == 0) return fail(ctx, FS_ERR_INVALID, "fs_set_histogram_sources_device: a path count is 0");
        if (n_paths[s] > n_max) n_max = n_paths[s];
    }
    dev_guard g(ctx->device);
    int rc = ensure_hist(ctx, n_sources);
    if (rc) return rc;
    const size_t hn = (size_t)n_sources * ctx->cfg.n_bands * ctx->cfg.n_bins;
    CK(cudaMemcpyAsync(ctx->d_hist, d_hist, 8 * hn, cudaMemcpyDeviceToDevice, ctx->stream));
    set_hist_counts(ctx, n_sources, n_max, n_paths);
    ctx->m2_valid = false;
    return FS_OK;
}

int fs_get_histogram_sources(fs_ctx* ctx, uint32_t* n_sources_out)
{
    if (!ctx || !n_sources_out) return FS_ERR_INVALID;
    *n_sources_out = ctx->d_hist ? ctx->hist_cur_sources : 0u;
    return FS_OK;
}

int fs_get_histogram(fs_ctx* ctx, uint64_t* hist_out)
{
    if (!ctx) return FS_ERR_INVALID;
    if (!hist_out || !ctx->d_hist || ctx->hist_cur_sources == 0) return fail(ctx, FS_ERR_STATE, "fs_get_histogram: no histogram");
    dev_guard g(ctx->device);
    // the sources of the LAST trace / fs_set_histogram (not the high-water mark of the allocation)
    const size_t hn = (size_t)ctx->hist_cur_sources * ctx->cfg.n_bands * ctx->cfg.n_bins;
    CK(cudaMemcpyAsync(hist_out, ctx->d_hist, 8 * hn, cudaMemcpyDeviceToHost, ctx->stream));
    return finish_stats(ctx);
}

// the per-source convolver slot (it also holds the device IR): created on first use, under conv_mu
static int ensure_conv_source(fs_ctx* ctx, uint32_t source)
{
    if (source >= FS_MAX_SOURCES) return fail(ctx, FS_ERR_INVALID, "source id too large (< 4096)");
    std::lock_guard<std::mutex> lk(ctx->conv_mu);
    if (ctx->conv[source] && ctx->conv[source]->ir) return FS_OK;
    cudaError_t e = fs_conv_source_alloc(ctx, source, false);
    if (e != cudaSuccess) return fail_cuda(ctx, e, "fs_conv_source_alloc");
    return FS_OK;
}

static int ensure_pin_ir(fs_ctx* ctx, size_t n_floats)
{
    if (ctx->pin_ir_cap >= n_floats) return FS_OK;
    if (ctx->h_pin_ir) cudaFreeHost(ctx->h_pin_ir);
    ctx->h_pin_ir = nullptr; ctx->pin_ir_cap = 0;
    CK(cudaMallocHost(&ctx->h_pin_ir, sizeof(float) * n_floats));
    ctx->pin_ir_cap = n_floats;
    return FS_OK;
}

// page-locked destination (fs_host_alloc, or registered by the caller): the DMA engine can write it directly
static bool host_is_pinned(const void* p)
{
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { (void)cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeHost;
}

int fs_host_alloc(size_t bytes, void** out)
{
    if (!out || !bytes) return FS_ERR_INVALID;
    *out = nullptr;
    if (cudaMallocHost(out, bytes) != cudaSuccess) { (void)cudaGetLastError(); g_err = "fs_host_alloc: cudaMallocHost failed"; return FS_ERR_NOMEM; }
    return FS_OK;
}

void fs_host_free(void* p) { if (p) cudaFreeHost(p); }

static int ir_common(fs_ctx* ctx, uint32_t hist_source, uint32_t source, const float* energy, float* ir_out,
                     bool per_band = false, uint64_t noise_seed = 0)
{
    nvtx_range nv("fs_build_ir");
    const fs_config& c = ctx->cfg;
    int rc = check_overflow(ctx, false);            // never build an IR from a histogram known to be incomplete
    if (rc) return rc;
    if ((rc = ensure_conv_source(ctx, source)) != FS_OK) return rc;
    fs_conv_source* s = ctx->conv[source];
    CK(cudaEventRecord(ctx->ev_ir0, ctx->stream));
    const float* d_energy = nullptr;
    if (energy) {
        CK(cudaMemcpyAsync(ctx->d_energy, energy, sizeof(float) * c.n_bins, cudaMemcpyHostToDevice, ctx->stream));
        d_energy = ctx->d_energy;
    }
    const unsigned long long* hsrc = ctx->d_hist ? ctx->d_hist + (size_t)hist_source * c.n_bands * c.n_bins : nullptr;
    if (per_band) CK(fs_ir_build_bands(ctx, hsrc, hist_paths(ctx, hist_source), noise_seed, s->ir));
    else CK(fs_ir_build(ctx, hsrc, hist_paths(ctx, hist_source), d_energy, s->ir));
    { std::lock_guard<std::mutex> lk(ctx->conv_mu); CK(fs_conv_update_ir(ctx, source, ctx->stream)); }
    CK(cudaEventRecord(ctx->ev_ir1, ctx->stream));
    ctx->ir_timed = true;
    if (ir_out) {
        const size_t n = (size_t)c.n_channels * c.sample_rate;
        const bool direct = host_is_pinned(ir_out);
        if (!direct && (rc = ensure_pin_ir(ctx, n)) != FS_OK) return rc;
        CK(cudaMemcpyAsync(direct ? ir_out : ctx->h_pin_ir, s->ir, sizeof(float) * n, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        if (!direct) memcpy(ir_out, ctx->h_pin_ir, sizeof(float) * n);
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, ctx->ev_ir0, ctx->ev_ir1) == cudaSuccess) ctx->stats.last_ir_ms = ms;
        return check_overflow(ctx, true);
    }
    return FS_OK;
}

static bool have_hist(const fs_ctx* ctx, uint32_t source) { return ctx->d_hist && source < ctx->hist_cur_sources && ctx->hist_n_paths; }

int fs_build_ir(fs_ctx* ctx, uint32_t source, float* ir_out)
{
    if (!ctx) return FS_ERR_INVALID;
    if (!have_hist(ctx, source))
        return fail(ctx, FS_ERR_STATE, "fs_build_ir: no histogram for this source (call fs_trace or fs_set_histogram)");
    dev_guard g(ctx->device);
    return ir_common(ctx, source, source, nullptr, ir_out);
}

int fs_build_ir_to(fs_ctx* ctx, uint32_t hist_source, uint32_t conv_source, float* ir_out)
{
    if (!ctx) return FS_ERR_INVALID;
    if (!have_hist(ctx, hist_source))
        return fail(ctx, FS_ERR_STATE, "fs_build_ir_to: no histogram for this source (call fs_trace or fs_set_histogram)");
    dev_guard g(ctx->device);
    return ir_common(ctx, hist_source, conv_source, nullptr, ir_out);
}

int fs_build_ir_all(fs_ctx* ctx, uint32_t n_sources, float* ir_out)
{
    if (!ctx) return FS_ERR_INVALID;
    if (n_sources == 0 || !have_hist(ctx, n_sources - 1))
        return fail(ctx, FS_ERR_STATE, "fs_build_ir_all: no histogram for these sources (call fs_trace or fs_set_histogram)");
    if (n_sources > FS_MAX_SOURCES) return fail(ctx, FS_ERR_INVALID, "source id too large (< 4096)");
    dev_guard g(ctx->device);
    const fs_config& c = ctx->cfg;
    int rc = check_overflow(ctx, false);
    if (rc) return rc;
    for (uint32_t s = 0; s < n_sources; ++s)
        if ((rc = ensure_conv_source(ctx, s)) != FS_OK) return rc;
    CK(cudaEventRecord(ctx->ev_ir0, ctx->stream));
    for (uint32_t s0 = 0; s0 < n_sources; s0 += FS_PTR_TABLE) {
        const uint32_t n = n_sources - s0 < FS_PTR_TABLE ? n_sources - s0 : FS_PTR_TABLE;
        fs_ptr_table tab;
        fs_scale_table inv;
        for (uint32_t i = 0; i < n; ++i) {
            tab.p[i] = ctx->conv[s0 + i]->ir; tab.q[i] = nullptr;
            const uint64_t np = hist_paths(ctx, s0 + i);
            inv.v[i] = np ? 1.0 / (double)np : 0.0;
        }
        CK(fs_ir_build_multi(ctx, ctx->d_hist, s0, n, inv, tab));
        { std::lock_guard<std::mutex> lk(ctx->conv_mu); CK(fs_conv_update_ir_multi(ctx, s0, n, ctx->stream)); }
    }
    CK(cudaEventRecord(ctx->ev_ir1, ctx->stream));
    ctx->ir_timed = true;
    if (ir_out) {
        // straight into the caller's buffer when it is page-locked (fs_host_alloc); otherwise through one pinned staging
        // buffer (a pageable destination would be staged 64 KB at a time by the driver)
        const size_t per = (size_t)c.n_channels * c.sample_rate;
        const bool direct = host_is_pinned(ir_out);
        if (!direct && (rc = ensure_pin_ir(ctx, per * n_sources)) != FS_OK) return rc;
        float* dst = direct ? ir_out : ctx->h_pin_ir;
        for (uint32_t s = 0; s < n_sources; ++s)
            CK(cudaMemcpyAsync(dst + s * per, ctx->conv[s]->ir, sizeof(float) * per, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        if (!direct) memcpy(ir_out, ctx->h_pin_ir, sizeof(float) * per * n_sources);
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, ctx->ev_ir0, ctx->ev_ir1) == cudaSuccess) ctx->stats.last_ir_ms = ms;
        return check_overflow(ctx, true);
    }
    return FS_OK;
}

int fs_update(fs_ctx* ctx, const float* src_pos, uint32_t n_sources, const float lis_pos[3], uint64_t n_paths,
              uint32_t max_depth, uint64_t seed, uint64_t* hist_out, float* ir_out)
{
    if (!ctx) return FS_ERR_INVALID;
    nvtx_range nv("fs_update");
    int rc = fs_trace(ctx, src_pos, n_sources, lis_pos, n_paths, max_depth, seed, nullptr);      // enqueued, not synchronised
    if (rc) return rc;
    dev_guard g(ctx->device);
    if (hist_out) {
        const size_t hn = (size_t)n_sources * ctx->cfg.n_bands * ctx->cfg.n_bins;
        CK(cudaMemcpyAsync(hist_out, ctx->d_hist, 8 * hn, cudaMemcpyDeviceToHost, ctx->stream));
    }
    rc = (n_sources == 1) ? ir_common(ctx, 0, 0, nullptr, ir_out) : fs_build_ir_all(ctx, n_sources, ir_out);
    if (rc) return rc;
    if (!ir_out) return hist_out ? finish_stats(ctx) : FS_OK;      // with ir_out the IR read-back has synchronised already
    return FS_OK;
}

int fs_trace_sources(fs_ctx* ctx, const fs_source_desc* src, uint32_t n_sources, const float lis_pos[3], uint64_t seed,
                     uint64_t* hist_out)
{
    if (!ctx) return FS_ERR_INVALID;
    nvtx_range nv("fs_trace_sources");
    fs_src_table t;
    int rc = prepare_sources(ctx, "fs_trace_sources", src, n_sources, lis_pos, &t);
    if (rc || (rc = check_dir_sources(ctx, n_sources, "fs_trace_sources"))) return rc;
    dev_guard g(ctx->device);
    if ((rc = ensure_hist(ctx, n_sources))) return rc;
    const size_t hn = (size_t)n_sources * ctx->cfg.n_bands * ctx->cfg.n_bins;
    CK(cudaMemsetAsync(ctx->d_hist, 0, 8 * hn, ctx->stream));            // FlushEnergyBuffer, COMP.h:76-79
    ulonglong2* d_m2 = nullptr;
    if ((rc = prepare_m2(ctx, n_sources, &d_m2))) return rc;
    rc = trace_common(ctx, t.pos.data(), n_sources, lis_pos, t.n_max, 0, t.off[n_sources], t.d_max, seed, ctx->d_hist, nullptr, &t,
                      d_m2);
    if (rc) return rc;
    set_hist_counts(ctx, n_sources, t.n_max, t.n_paths.data());
    ctx->m2_valid = d_m2 != nullptr;
    if (hist_out) {
        CK(cudaMemcpyAsync(hist_out, ctx->d_hist, 8 * hn, cudaMemcpyDeviceToHost, ctx->stream));
        return finish_stats(ctx);
    }
    return FS_OK;
}

int fs_update_sources(fs_ctx* ctx, const fs_source_desc* src, uint32_t n_sources, const float lis_pos[3], uint64_t seed,
                      uint64_t* hist_out, float* ir_out)
{
    if (!ctx) return FS_ERR_INVALID;
    nvtx_range nv("fs_update_sources");
    if (n_sources > FS_MAX_SOURCES) return fail(ctx, FS_ERR_INVALID, "fs_update_sources: source id too large (< 4096)");
    int rc = fs_trace_sources(ctx, src, n_sources, lis_pos, seed, nullptr);      // enqueued, not synchronised
    if (rc) return rc;
    dev_guard g(ctx->device);
    if (hist_out) {
        const size_t hn = (size_t)n_sources * ctx->cfg.n_bands * ctx->cfg.n_bins;
        CK(cudaMemcpyAsync(hist_out, ctx->d_hist, 8 * hn, cudaMemcpyDeviceToHost, ctx->stream));
    }
    rc = (n_sources == 1) ? ir_common(ctx, 0, 0, nullptr, ir_out) : fs_build_ir_all(ctx, n_sources, ir_out);
    if (rc) return rc;
    if (!ir_out) return hist_out ? finish_stats(ctx) : FS_OK;
    return FS_OK;
}

static int trace_sources_range_device(fs_ctx* ctx, const fs_source_desc* src, uint32_t n_sources, const float lis_pos[3],
                                      uint64_t g_first, uint64_t g_count, uint64_t seed, void* d_hist, ulonglong2* d_m2,
                                      int zero_first)
{
    if (!ctx) return FS_ERR_INVALID;
    if (!d_hist) return fail(ctx, FS_ERR_INVALID, "fs_trace_sources_range_device: null histogram");
    fs_src_table t;
    int rc = prepare_sources(ctx, "fs_trace_sources_range_device", src, n_sources, lis_pos, &t);
    if (rc || (rc = check_dir_sources(ctx, n_sources, "fs_trace_sources_range_device"))) return rc;
    if (g_first + g_count > t.off[n_sources] || g_first + g_count < g_first)
        return fail(ctx, FS_ERR_INVALID, "fs_trace_sources_range_device: work range exceeds the sum of the path counts");
    dev_guard g(ctx->device);
    const size_t hn = (size_t)n_sources * ctx->cfg.n_bands * ctx->cfg.n_bins;
    if (zero_first) CK(cudaMemsetAsync(d_hist, 0, 8 * hn, ctx->stream));
    if (zero_first && d_m2) CK(cudaMemsetAsync(d_m2, 0, sizeof(ulonglong2) * (size_t)n_sources * (ctx->cfg.n_bands + 1u) * ctx->cfg.n_bins, ctx->stream));
    return trace_common(ctx, t.pos.data(), n_sources, lis_pos, t.n_max, g_first, g_count, t.d_max, seed,
                        (unsigned long long*)d_hist, nullptr, &t, d_m2);
}

int fs_trace_sources_range_device(fs_ctx* ctx, const fs_source_desc* src, uint32_t n_sources, const float lis_pos[3],
                                  uint64_t g_first, uint64_t g_count, uint64_t seed, void* d_hist, int zero_first)
{
    return trace_sources_range_device(ctx, src, n_sources, lis_pos, g_first, g_count, seed, d_hist, nullptr, zero_first);
}

int fs_build_ir_bands(fs_ctx* ctx, uint32_t hist_source, uint32_t conv_source, uint64_t noise_seed, float* ir_out)
{
    if (!ctx) return FS_ERR_INVALID;
    if (!have_hist(ctx, hist_source))
        return fail(ctx, FS_ERR_STATE, "fs_build_ir_bands: no histogram for this source (call fs_trace or fs_set_histogram)");
    dev_guard g(ctx->device);
    return ir_common(ctx, hist_source, conv_source, nullptr, ir_out, true, noise_seed);
}

int fs_build_ir_from_energy(fs_ctx* ctx, uint32_t source, const float* energy, float* ir_out)
{
    if (!ctx) return FS_ERR_INVALID;
    if (!energy) return fail(ctx, FS_ERR_INVALID, "fs_build_ir_from_energy: null energy");
    // a negative entry at or above the threshold maps to NaN, which the low-pass spreads over the rest of the IR
    for (uint32_t k = 0; k < ctx->cfg.n_bins; ++k)
        if (!(energy[k] >= 0.0f) || !isfinite(energy[k]))
            return fail(ctx, FS_ERR_INVALID, "fs_build_ir_from_energy: energy entries must be finite and >= 0");
    dev_guard g(ctx->device);
    return ir_common(ctx, 0, source, energy, ir_out);
}

int fs_set_ir(fs_ctx* ctx, uint32_t source, const float* ir)
{
    if (!ctx) return FS_ERR_INVALID;
    if (!ir) return fail(ctx, FS_ERR_INVALID, "fs_set_ir: null ir");
    dev_guard g(ctx->device);
    int rc = ensure_conv_source(ctx, source);
    if (rc) return rc;
    fs_conv_source* s = ctx->conv[source];
    const fs_config& c = ctx->cfg;
    CK(cudaMemcpyAsync(s->ir, ir, sizeof(float) * c.n_channels * c.sample_rate, cudaMemcpyHostToDevice, ctx->stream));
    { std::lock_guard<std::mutex> lk(ctx->conv_mu); CK(fs_conv_update_ir(ctx, source, ctx->stream)); }
    CK(cudaStreamSynchronize(ctx->stream));
    return FS_OK;
}

// ---- convolution (the audio thread; everything on conv_stream under conv_mu) --------------------------------------
int fs_conv_init_source(fs_ctx* ctx, uint32_t source)
{
    if (!ctx) return FS_ERR_INVALID;
    if (source >= FS_MAX_SOURCES) return fail(ctx, FS_ERR_INVALID, "source id too large (< 4096)");
    dev_guard g(ctx->device);
    std::lock_guard<std::mutex> lk(ctx->conv_mu);
    CK(fs_conv_source_alloc(ctx, source, true));
    return FS_OK;
}

int fs_conv_release_source(fs_ctx* ctx, uint32_t source)
{
    if (!ctx) return FS_ERR_INVALID;
    if (source >= FS_MAX_SOURCES) return fail(ctx, FS_ERR_INVALID, "source id too large (< 4096)");
    dev_guard g(ctx->device);
    std::lock_guard<std::mutex> lk(ctx->conv_mu);
    // Source.ClearBuffers(), REV.cpp:112-116: the history goes, the slot (and its IR, which the game thread may be
    // rebuilding right now on its own stream) stays until fs_destroy
    if (ctx->conv[source] && ctx->conv[source]->active) { ctx->conv[source]->active = false; ctx->conv_active.fetch_sub(1); }
    return FS_OK;
}

static int conv_process(fs_ctx* ctx, const uint32_t* sources, uint32_t n_src, const float* in, float* out, uint32_t frames,
                        uint32_t n_blocks)
{
    if (!ctx) return FS_ERR_INVALID;
    if (!in || !out || !sources) return fail(ctx, FS_ERR_INVALID, "fs_conv_process: null buffer");
    if (frames != ctx->cfg.conv_block) return fail(ctx, FS_ERR_INVALID, "fs_conv_process: frames must equal conv_block");
    if (n_blocks == 0 || n_src == 0) return FS_OK;
    nvtx_range nv("fs_conv_process");
    dev_guard g(ctx->device);
    std::lock_guard<std::mutex> lk(ctx->conv_mu);
    for (uint32_t i = 0; i < n_src; ++i) {
        if (sources[i] >= FS_MAX_SOURCES || !ctx->conv[sources[i]] || !ctx->conv[sources[i]]->active)
            return fail(ctx, FS_ERR_STATE, "fs_conv_process: source not initialised (fs_conv_init_source)");
        for (uint32_t j = 0; j < i; ++j)
            if (sources[j] == sources[i]) return fail(ctx, FS_ERR_INVALID, "fs_conv_process_multi: duplicate source id");
    }
    const fs_config& c = ctx->cfg;
    const size_t n = (size_t)n_src * n_blocks * frames * c.n_channels;
    cudaStream_t st = ctx->conv_stream;
    if (ctx->conv_io_cap < n) {
        cudaFree(ctx->d_conv_in); cudaFree(ctx->d_conv_out); ctx->d_conv_in = ctx->d_conv_out = nullptr;
        if (ctx->h_pin_in) cudaFreeHost(ctx->h_pin_in);
        if (ctx->h_pin_out) cudaFreeHost(ctx->h_pin_out);
        ctx->h_pin_in = ctx->h_pin_out = nullptr; ctx->conv_io_cap = 0;
        CK(cudaMalloc(&ctx->d_conv_in, sizeof(float) * n));
        CK(cudaMalloc(&ctx->d_conv_out, sizeof(float) * n));
        CK(cudaMallocHost(&ctx->h_pin_in, sizeof(float) * n));
        CK(cudaMallocHost(&ctx->h_pin_out, sizeof(float) * n));
        ctx->conv_io_cap = n;
    }
    memcpy(ctx->h_pin_in, in, sizeof(float) * n);
    CK(cudaMemcpyAsync(ctx->d_conv_in, ctx->h_pin_in, sizeof(float) * n, cudaMemcpyHostToDevice, st));
    CK(cudaEventRecord(ctx->ev_c0, st));
    CK(fs_conv_run(ctx, sources, n_src, ctx->d_conv_in, ctx->d_conv_out, n_blocks, st));
    CK(cudaEventRecord(ctx->ev_c1, st));
    CK(cudaMemcpyAsync(ctx->h_pin_out, ctx->d_conv_out, sizeof(float) * n, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    if (cudaEventElapsedTime(&ctx->last_conv_ms, ctx->ev_c0, ctx->ev_c1) != cudaSuccess) (void)cudaGetLastError();
    memcpy(out, ctx->h_pin_out, sizeof(float) * n);
    return FS_OK;
}

int fs_conv_process_many(fs_ctx* ctx, uint32_t source, const float* in, float* out, uint32_t frames, uint32_t n_blocks)
{
    return conv_process(ctx, &source, 1, in, out, frames, n_blocks);
}

int fs_conv_process(fs_ctx* ctx, uint32_t source, const float* in, float* out, uint32_t frames)
{
    return conv_process(ctx, &source, 1, in, out, frames, 1);
}

int fs_conv_process_multi(fs_ctx* ctx, const uint32_t* sources, uint32_t n_sources, const float* in, float* out, uint32_t frames)
{
    return conv_process(ctx, sources, n_sources, in, out, frames, 1);
}

int fs_debug_rfft(fs_ctx* ctx, const float* in, uint32_t n, float* out_ri)
{
    if (!ctx) return FS_ERR_INVALID;
    if (!in || !out_ri || n < 64 || n > 4096 || (n & (n - 1))) return fail(ctx, FS_ERR_INVALID, "fs_debug_rfft: n must be a power of two in 64..4096");
    dev_guard g(ctx->device);
    float* d_in = nullptr; float2* d_out = nullptr;
    CK(cudaMalloc(&d_in, sizeof(float) * n));
    cudaError_t e = cudaMalloc(&d_out, sizeof(float2) * (n / 2 + 1));
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_in, in, sizeof(float) * n, cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) e = fs_conv_rfft(ctx, d_in, n, d_out, ctx->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(out_ri, d_out, sizeof(float2) * (n / 2 + 1), cudaMemcpyDeviceToHost, ctx->stream);
    cudaError_t e2 = cudaStreamSynchronize(ctx->stream);
    cudaFree(d_in); cudaFree(d_out);
    if (e != cudaSuccess || e2 != cudaSuccess) return fail_cuda(ctx, e != cudaSuccess ? e : e2, "fs_debug_rfft");
    return FS_OK;
}

// the state rules of fs_get_noise / fs_get_histogram_m2
static int noise_state(fs_ctx* ctx, const char* who)
{
    std::string w(who);
    if (!(ctx->cfg.flags & FS_FLAG_NOISE_STATS)) return fail(ctx, FS_ERR_STATE, (w + ": the context was created without FS_FLAG_NOISE_STATS").c_str());
    if (!ctx->m2_valid || !ctx->d_hist || ctx->hist_cur_sources == 0)
        return fail(ctx, FS_ERR_STATE, (w + ": no second moments for the current histogram (trace with fs_trace / fs_trace_sources / "
                                            "fs_update* / fs_multi_trace* first)").c_str());
    return FS_OK;
}

static double snr_db(double signal, double variance)
{
    if (!(signal > 0.0)) return -INFINITY;
    if (!(variance > 0.0)) return INFINITY;
    return 10.0 * log10(signal / variance);
}

int fs_get_noise(fs_ctx* ctx, fs_noise_stats* out, uint32_t n_sources)
{
    if (!ctx) return FS_ERR_INVALID;
    if (!out) return fail(ctx, FS_ERR_INVALID, "fs_get_noise: null output");
    int rc = noise_state(ctx, "fs_get_noise");
    if (rc) return rc;
    const uint32_t S = ctx->hist_cur_sources, B = ctx->cfg.n_bands;
    if (n_sources != S) return fail(ctx, FS_ERR_INVALID, "fs_get_noise: n_sources differs from fs_get_histogram_sources");
    dev_guard g(ctx->device);
    const size_t n_out = (size_t)S * (B + 1u) * 2u;
    if (ctx->noise_cap < S) {
        cudaFree(ctx->d_noise); ctx->d_noise = nullptr; ctx->noise_cap = 0;
        CK(cudaMalloc(&ctx->d_noise, sizeof(double) * ((size_t)S + n_out)));
        ctx->noise_cap = S;
    }
    std::vector<uint64_t> n(S);
    for (uint32_t s = 0; s < S; ++s) n[s] = hist_paths(ctx, s);
    std::vector<double> h(n_out);
    uint64_t* d_n = (uint64_t*)ctx->d_noise;
    double* d_out = ctx->d_noise + S;
    CK(cudaMemcpyAsync(d_n, n.data(), 8ull * S, cudaMemcpyHostToDevice, ctx->stream));
    CK(fs_noise_reduce(ctx->d_hist, ctx->d_m2, d_n, S, B, ctx->cfg.n_bins, d_out, ctx->stream));
    ctx->launches.fetch_add(1);
    CK(cudaMemcpyAsync(h.data(), d_out, sizeof(double) * n_out, cudaMemcpyDeviceToHost, ctx->stream));
    if ((rc = finish_stats(ctx))) return rc;
    for (uint32_t s = 0; s < S; ++s) {
        fs_noise_stats& o = out[s];
        memset(&o, 0, sizeof(o));
        o.n_paths = n[s];
        const double* r = h.data() + (size_t)s * (B + 1u) * 2u;
        for (uint32_t b = 0; b < B; ++b) {
            o.band_signal[b] = r[2 * b]; o.band_variance[b] = r[2 * b + 1];
            o.band_snr_db[b] = snr_db(r[2 * b], r[2 * b + 1]);
        }
        o.signal = r[2 * B]; o.variance = r[2 * B + 1];
        o.snr_db = snr_db(o.signal, o.variance);
        o.no_energy = o.signal > 0.0 ? 0u : 1u;
    }
    return FS_OK;
}

int fs_get_histogram_m2(fs_ctx* ctx, uint64_t* out)
{
    if (!ctx) return FS_ERR_INVALID;
    if (!out) return fail(ctx, FS_ERR_INVALID, "fs_get_histogram_m2: null output");
    int rc = noise_state(ctx, "fs_get_histogram_m2");
    if (rc) return rc;
    dev_guard g(ctx->device);
    const size_t n = (size_t)ctx->hist_cur_sources * (ctx->cfg.n_bands + 1u) * ctx->cfg.n_bins;
    CK(cudaMemcpyAsync(out, ctx->d_m2, sizeof(ulonglong2) * n, cudaMemcpyDeviceToHost, ctx->stream));
    return finish_stats(ctx);
}

// ---- room-acoustic parameters ---------------------------------------------------------------------
int fs_get_acoustic_params(fs_ctx* ctx, fs_acoustic_params* out, uint32_t n_sources, float* edc_db_out)
{
    if (!ctx) return FS_ERR_INVALID;
    if (!out) return fail(ctx, FS_ERR_INVALID, "fs_get_acoustic_params: null output");
    if (!ctx->d_hist || ctx->hist_cur_sources == 0)
        return fail(ctx, FS_ERR_STATE, "fs_get_acoustic_params: no histogram (trace or fs_set_histogram first)");
    const uint32_t S = ctx->hist_cur_sources, B = ctx->cfg.n_bands, K = ctx->cfg.n_bins, W = B + 1u;
    if (n_sources != S) return fail(ctx, FS_ERR_INVALID, "fs_get_acoustic_params: n_sources differs from fs_get_histogram_sources");
    dev_guard g(ctx->device);
    const size_t n_rec = (size_t)S * W, rec_bytes = (sizeof(fs_acoustic_slot) * n_rec + 255u) & ~(size_t)255u;
    const size_t need = rec_bytes + (edc_db_out ? sizeof(float) * n_rec * K : 0u);
    if (ctx->acou_cap < need) {
        cudaFree(ctx->d_acou); ctx->d_acou = nullptr; ctx->acou_cap = 0;
        CK(cudaMalloc(&ctx->d_acou, need));
        ctx->acou_cap = need;
    }
    fs_acoustic_slot* d_rec = (fs_acoustic_slot*)ctx->d_acou;
    float* d_edc = edc_db_out ? (float*)((char*)ctx->d_acou + rec_bytes) : nullptr;
    std::vector<fs_acoustic_slot> h(n_rec);
    CK(fs_acoustics_run(ctx->d_hist, S, B, K, ctx->cfg.bin_ms, d_rec, d_edc, ctx->stream));
    ctx->launches.fetch_add(1);
    CK(cudaMemcpyAsync(h.data(), d_rec, sizeof(fs_acoustic_slot) * n_rec, cudaMemcpyDeviceToHost, ctx->stream));
    if (edc_db_out) CK(cudaMemcpyAsync(edc_db_out, d_edc, sizeof(float) * n_rec * K, cudaMemcpyDeviceToHost, ctx->stream));
    const int rc = finish_stats(ctx);
    if (rc != FS_OK && rc != FS_ERR_OVERFLOW) return rc;
    for (uint32_t s = 0; s < S; ++s) {
        fs_acoustic_params& o = out[s];
        memset(&o, 0, sizeof(o));
        const fs_acoustic_slot* r = h.data() + (size_t)s * W;
        for (uint32_t b = 0; b < B; ++b) o.band[b] = r[b];
        o.broadband = r[B];
        o.no_energy = r[B].onset_bin == 0xffffffffu ? 1u : 0u;
    }
    return rc;
}

// ---- directional sources ------------------------------------------------------------------------
// The tables live on the device and are replaced by stream-ordered copies on the context stream: a trace enqueued before a
// set call reads the old contents, one enqueued after it the new.  The host data is copied into a pageable vector first, so
// the caller's buffer is free when the call returns whatever memory it is.
int fs_set_directivity_patterns(fs_ctx* ctx, const fs_directivity* patterns, uint32_t n_patterns)
{
    if (!ctx) return FS_ERR_INVALID;
    if (!patterns || n_patterns < 1 || n_patterns > 256)
        return fail(ctx, FS_ERR_INVALID, "fs_set_directivity_patterns: 1..256 patterns needed");
    for (uint32_t p = 0; p < n_patterns; ++p)
        for (uint32_t b = 0; b < ctx->cfg.n_bands; ++b)
            for (int i = 0; i < FS_DIR_POINTS; ++i) {
                const float v = patterns[p].gain[b][i];
                if (!(v >= 0.0f) || !std::isfinite(v))
                    return fail(ctx, FS_ERR_INVALID, ("fs_set_directivity_patterns: gain of pattern " + std::to_string(p) + ", band " +
                                                      std::to_string(b) + " is negative or not finite").c_str());
            }
    dev_guard g(ctx->device);
    const size_t n = (size_t)n_patterns * FS_MAX_BANDS * FS_DIR_POINTS;
    std::vector<float> h(n);
    memcpy(h.data(), patterns, sizeof(float) * n);
    if (!ctx->d_dir_gain) CK(cudaMalloc(&ctx->d_dir_gain, sizeof(float) * FS_MAX_BANDS * FS_DIR_POINTS * 256));   // 270 KB, the largest table
    CK(cudaMemcpyAsync(ctx->d_dir_gain, h.data(), sizeof(float) * n, cudaMemcpyHostToDevice, ctx->stream));
    ctx->dir_patterns = n_patterns;
    ctx->dir_sources = 0;                        // the orientations named indices of the old table
    return FS_OK;
}

int fs_set_source_directivity(fs_ctx* ctx, const fs_source_orient* o, uint32_t n_sources)
{
    if (!ctx) return FS_ERR_INVALID;
    if (n_sources == 0) { ctx->dir_sources = 0; return FS_OK; }
    if (!o) return fail(ctx, FS_ERR_INVALID, "fs_set_source_directivity: null orientations");
    std::vector<float4> h(n_sources);
    for (uint32_t s = 0; s < n_sources; ++s) {
        const std::string who = "fs_set_source_directivity: source " + std::to_string(s);
        const uint32_t pat = o[s].pattern;
        if (pat != FS_OMNI && !ctx->dir_patterns)
            return fail(ctx, FS_ERR_INVALID, (who + ": pattern index without an installed pattern table (fs_set_directivity_patterns)").c_str());
        if (pat != FS_OMNI && pat >= ctx->dir_patterns)
            return fail(ctx, FS_ERR_INVALID, (who + ": pattern index " + std::to_string(pat) + " >= the " +
                                              std::to_string(ctx->dir_patterns) + " installed patterns").c_str());
        const double x = o[s].forward[0], y = o[s].forward[1], z = o[s].forward[2];
        const double len = sqrt(x * x + y * y + z * z);
        if (!std::isfinite(x) || !std::isfinite(y) || !std::isfinite(z) || !(len > 0.0))
            return fail(ctx, FS_ERR_INVALID, (who + ": forward must be a non-zero finite vector").c_str());
        h[s] = make_float4((float)(x / len), (float)(y / len), (float)(z / len), 0.0f);
        uint32_t bits = pat;
        memcpy(&h[s].w, &bits, 4);
    }
    dev_guard g(ctx->device);
    if (ctx->dir_orient_cap < n_sources) {
        cudaFree(ctx->d_dir_orient); ctx->d_dir_orient = nullptr; ctx->dir_orient_cap = 0; ctx->dir_sources = 0;
        CK(cudaMalloc(&ctx->d_dir_orient, sizeof(float4) * n_sources));
        ctx->dir_orient_cap = n_sources;
    }
    CK(cudaMemcpyAsync(ctx->d_dir_orient, h.data(), sizeof(float4) * n_sources, cudaMemcpyHostToDevice, ctx->stream));
    ctx->dir_sources = n_sources;
    return FS_OK;
}

int fs_directivity_polar(const float* dipole_weight, const float* power, uint32_t n_bands, fs_directivity* out)
{
    if (!dipole_weight || !power || !out || n_bands < 1 || n_bands > FS_MAX_BANDS)
        return fail(nullptr, FS_ERR_INVALID, "fs_directivity_polar: null argument or n_bands outside 1..8");
    for (uint32_t b = 0; b < n_bands; ++b) {
        if (!(dipole_weight[b] >= 0.0f && dipole_weight[b] <= 1.0f))
            return fail(nullptr, FS_ERR_INVALID, "fs_directivity_polar: dipole weight outside [0, 1]");
        if (!(power[b] >= 0.0f && power[b] <= 64.0f))
            return fail(nullptr, FS_ERR_INVALID, "fs_directivity_polar: power outside [0, 64]");
    }
    memset(out, 0, sizeof(*out));
    for (uint32_t b = 0; b < n_bands; ++b)
        for (int i = 0; i < FS_DIR_POINTS; ++i) {
            const double c = -1.0 + i / 16.0, w = dipole_weight[b];
            out->gain[b][i] = (float)pow(fabs((1.0 - w) + w * c), (double)power[b]);
        }
    return FS_OK;
}

// ---- direct-path occlusion ------------------------------------------------------------------------
int fs_occlusion(fs_ctx* ctx, const fs_occlusion_source* src, uint32_t n_sources, const float lis_pos[3], uint32_t max_crossings,
                 uint64_t seed, fs_occlusion_result* out)
{
    if (!ctx) return FS_ERR_INVALID;
    if (!ctx->committed) return fail(ctx, FS_ERR_STATE, "fs_occlusion: call fs_scene_commit first");
    if (ctx->verts_dirty) return fail(ctx, FS_ERR_STATE, "fs_occlusion: triangles were moved; call fs_scene_refit (or fs_scene_commit) first");
    if (!src || !lis_pos || !out) return fail(ctx, FS_ERR_INVALID, "fs_occlusion: null argument");
    if (n_sources == 0 || n_sources > FS_MAX_SOURCES) return fail(ctx, FS_ERR_INVALID, "fs_occlusion: n_sources must be 1..4096");
    if (max_crossings > 16) return fail(ctx, FS_ERR_INVALID, "fs_occlusion: max_crossings must be 0..16");
    auto bad_pos = [](const float* p) {
        for (int a = 0; a < 3; ++a) if (!std::isfinite(p[a]) || fabsf(p[a]) > 1e18f) return true;
        return false;
    };
    if (bad_pos(lis_pos)) return fail(ctx, FS_ERR_INVALID, "fs_occlusion: non-finite or > 1e18 listener position");
    const uint32_t S = n_sources, B = ctx->cfg.n_bands, W = B + 1u;
    // host staging of the upload: [S] float4 (centre, radius), then [S+1] u32 ray offsets
    std::vector<float4> hsrc(S + (S + 1u + 3u) / 4u);
    uint32_t* off = (uint32_t*)(hsrc.data() + S);
    uint32_t n_rays = 0;
    for (uint32_t s = 0; s < S; ++s) {
        const fs_occlusion_source& d = src[s];
        const std::string who = "fs_occlusion: source " + std::to_string(s);
        if (bad_pos(d.pos)) return fail(ctx, FS_ERR_INVALID, (who + ": non-finite or > 1e18 position").c_str());
        if (!(d.radius >= 0.0f) || !std::isfinite(d.radius)) return fail(ctx, FS_ERR_INVALID, (who + ": radius must be finite and >= 0").c_str());
        if (d.radius > 0.0f && (d.n_rays == 0 || d.n_rays > 65536u)) return fail(ctx, FS_ERR_INVALID, (who + ": n_rays must be 1..65536").c_str());
        if (d.reserved) return fail(ctx, FS_ERR_INVALID, (who + ": reserved field must be 0").c_str());
        hsrc[s] = make_float4(d.pos[0], d.pos[1], d.pos[2], d.radius);
        off[s] = n_rays;
        n_rays += d.radius > 0.0f ? d.n_rays : 1u;
    }
    off[S] = n_rays;
    dev_guard g(ctx->device);
    // device scratch: [S][B+1] u64 sums, one u64 slot for the overflow flag, then the staged sources and offsets
    const size_t acc_bytes = (8ull * S * W + 8ull + 15ull) & ~15ull, up_bytes = sizeof(float4) * hsrc.size();
    if (ctx->occl_cap < acc_bytes + up_bytes) {
        cudaFree(ctx->d_occl); ctx->d_occl = nullptr; ctx->occl_cap = 0;
        const size_t cap = 8ull * FS_MAX_SOURCES * (FS_MAX_BANDS + 1) + 16ull + sizeof(float4) * (FS_MAX_SOURCES + 1026);   // 0.35 MB: the largest call
        CK(cudaMalloc(&ctx->d_occl, cap));
        ctx->occl_cap = (uint32_t)cap;
    }
    unsigned long long* d_acc = (unsigned long long*)ctx->d_occl;
    uint32_t* d_overflow = (uint32_t*)(d_acc + (size_t)S * W);
    float4* d_src = (float4*)((char*)ctx->d_occl + acc_bytes);
    fs_trace_params tp;
    fill_params(ctx, &tp, nullptr, 1, 1, 0);
    std::vector<unsigned long long> h(acc_bytes / 8u);
    CK(cudaMemcpyAsync(d_src, hsrc.data(), up_bytes, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemsetAsync(d_acc, 0, acc_bytes, ctx->stream));
    CK(fs_occlusion_run(tp.bv, d_src, (const uint32_t*)(d_src + S), S, n_rays, lis_pos, ctx->d_occl_tau, B, max_crossings,
                        ctx->cfg.eps_connect, ctx->cfg.eps_offset, seed, d_acc, d_overflow, ctx->stream));
    ctx->launches.fetch_add(1);
    CK(cudaMemcpyAsync(h.data(), d_acc, acc_bytes, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    for (uint32_t s = 0; s < S; ++s) {
        const double n = (double)(off[s + 1] - off[s]);
        const unsigned long long* r = h.data() + (size_t)s * W;
        fs_occlusion_result& o = out[s];
        memset(&o, 0, sizeof(o));
        o.visible = (float)((double)r[B] / n);
        for (uint32_t b = 0; b < B; ++b) o.transmission[b] = (float)((double)r[b] * 0x1p-32 / n);
        o.n_rays = off[s + 1] - off[s];
    }
    if ((uint32_t)h[(size_t)S * W])
        return fail(ctx, FS_ERR_OVERFLOW, "fs_occlusion: BVH traversal stack overflow (tree deeper than FS_STACK_SIZE): the results are invalid");
    return FS_OK;
}

// ---- first-order edge diffraction -----------------------------------------------------------------
static_assert(sizeof(fs_diffraction_result) == 68, "fs_diffraction_result is part of the ABI");
static_assert(sizeof(fs_diff_edge) == 64, "fs_diff_edge is read as four 16-byte words");

// the checks every diffraction entry point shares; nothing is enqueued before they pass
static int diffraction_state(fs_ctx* ctx, const char* who, float min_fold_deg)
{
    if (!ctx->committed) return fail(ctx, FS_ERR_STATE, (std::string(who) + ": call fs_scene_commit first").c_str());
    if (ctx->verts_dirty)
        return fail(ctx, FS_ERR_STATE, (std::string(who) + ": triangles were moved; call fs_scene_refit (or fs_scene_commit) first").c_str());
    if (!std::isfinite(min_fold_deg) || min_fold_deg < 0.0f || min_fold_deg > 180.0f)
        return fail(ctx, FS_ERR_INVALID, (std::string(who) + ": min_fold_deg must be finite and in [0, 180]").c_str());
    return FS_OK;
}

// the edge set for min_fold_deg: built on first use after a commit, refit or threshold change
static int diffraction_edges(fs_ctx* ctx, float min_fold_deg)
{
    if (ctx->diff_valid && ctx->diff_fold_deg == min_fold_deg) return FS_OK;
    cudaFree(ctx->d_diff_edges); ctx->d_diff_edges = nullptr; ctx->n_diff_edges = 0; ctx->diff_valid = false;
    const float c_min = (float)(-cos((double)min_fold_deg * (M_PI / 180.0)));
    uint64_t launches = 0;
    const cudaError_t e = fs_diffraction_edges(ctx->stream, ctx->d_verts, (uint32_t)ctx->n_tris, c_min, &ctx->d_diff_edges,
                                               &ctx->n_diff_edges, &launches);
    ctx->launches.fetch_add(launches);
    CK(e);
    ctx->diff_fold_deg = min_fold_deg;
    ctx->diff_valid = true;
    return FS_OK;
}

int fs_diffraction(fs_ctx* ctx, const float* src_pos, uint32_t n_sources, const float lis_pos[3], float min_fold_deg,
                   const float* band_hz, fs_diffraction_result* out)
{
    if (!ctx) return FS_ERR_INVALID;
    if (int rc = diffraction_state(ctx, "fs_diffraction", min_fold_deg)) return rc;
    if (!src_pos || !lis_pos || !out) return fail(ctx, FS_ERR_INVALID, "fs_diffraction: null argument");
    if (n_sources == 0 || n_sources > FS_MAX_SOURCES) return fail(ctx, FS_ERR_INVALID, "fs_diffraction: n_sources must be 1..4096");
    auto bad_pos = [](const float* p) {
        for (int a = 0; a < 3; ++a) if (!std::isfinite(p[a]) || fabsf(p[a]) > 1e18f) return true;
        return false;
    };
    if (bad_pos(lis_pos)) return fail(ctx, FS_ERR_INVALID, "fs_diffraction: non-finite or > 1e18 listener position");
    const uint32_t S = n_sources, B = ctx->cfg.n_bands;
    for (uint32_t s = 0; s < S; ++s)
        if (bad_pos(src_pos + 3ull * s))
            return fail(ctx, FS_ERR_INVALID, ("fs_diffraction: source " + std::to_string(s) + ": non-finite or > 1e18 position").c_str());
    fs_diff_run a;
    memset(&a, 0, sizeof(a));
    for (uint32_t b = 0; b < B; ++b) {
        if (band_hz && !(std::isfinite(band_hz[b]) && band_hz[b] > 0.0f))
            return fail(ctx, FS_ERR_INVALID, "fs_diffraction: band_hz entries must be finite and > 0");
        a.band_hz[b] = band_hz ? band_hz[b] : fs_diff_default_hz(b);
    }
    dev_guard g(ctx->device);
    if (int rc = diffraction_edges(ctx, min_fold_deg)) return rc;
    // scratch: [S] float4 sources | [S] u64 best | [S] u32 path counts | u64 candidates, u64 rays, u32 overflow | [S] results
    const size_t o_best = 16ull * FS_MAX_SOURCES, o_np = o_best + 8ull * FS_MAX_SOURCES, o_misc = o_np + 4ull * FS_MAX_SOURCES,
                 o_out = o_misc + 32ull, cap = o_out + sizeof(fs_diffraction_result) * FS_MAX_SOURCES;   // 0.4 MB: the largest call
    if (!ctx->d_diff) {
        CK(cudaMalloc(&ctx->d_diff, cap));
        ctx->diff_cap = cap;
    }
    char* base = (char*)ctx->d_diff;
    std::vector<float4> hsrc(S);
    for (uint32_t s = 0; s < S; ++s) hsrc[s] = make_float4(src_pos[3 * s], src_pos[3 * s + 1], src_pos[3 * s + 2], 0.0f);
    fs_trace_params tp;
    fill_params(ctx, &tp, nullptr, 1, 1, 0);
    a.bv = tp.bv;
    a.edges = ctx->d_diff_edges; a.n_edges = ctx->n_diff_edges;
    a.src = (const float4*)base; a.n_src = S;
    for (int i = 0; i < 3; ++i) a.lis[i] = lis_pos[i];
    a.eps_offset = ctx->cfg.eps_offset; a.eps_connect = ctx->cfg.eps_connect; a.sound_speed = ctx->cfg.sound_speed;
    a.n_bands = B;
    a.cand = &ctx->d_diff_cand; a.cand_cap = &ctx->diff_cand_cap;
    a.best = (unsigned long long*)(base + o_best);
    a.n_paths = (uint32_t*)(base + o_np);
    a.d_count = (unsigned long long*)(base + o_misc);
    a.rays = a.d_count + 1;
    a.overflow = (uint32_t*)(a.d_count + 2);
    a.out = (fs_diffraction_result*)(base + o_out);
    CK(cudaMemcpyAsync(base, hsrc.data(), sizeof(float4) * S, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemsetAsync(a.best, 0xff, 8ull * S, ctx->stream));
    CK(cudaMemsetAsync(a.n_paths, 0, 4ull * S, ctx->stream));
    CK(cudaMemsetAsync(a.d_count, 0, 32, ctx->stream));
    uint64_t launches = 0;
    const cudaError_t e = fs_diffraction_run(a, ctx->stream, &launches, nullptr);
    ctx->launches.fetch_add(launches);
    CK(e);
    uint32_t overflow = 0;
    CK(cudaMemcpyAsync(out, a.out, sizeof(fs_diffraction_result) * S, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(&overflow, a.overflow, 4, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    if (overflow)
        return fail(ctx, FS_ERR_OVERFLOW, "fs_diffraction: BVH traversal stack overflow (tree deeper than FS_STACK_SIZE): the results are invalid");
    return FS_OK;
}

int fs_debug_diffraction_edges(fs_ctx* ctx, float min_fold_deg, uint32_t* out, uint64_t cap, uint64_t* n_out)
{
    if (!ctx) return FS_ERR_INVALID;
    if (int rc = diffraction_state(ctx, "fs_debug_diffraction_edges", min_fold_deg)) return rc;
    if (!n_out) return fail(ctx, FS_ERR_INVALID, "fs_debug_diffraction_edges: null n_out");
    dev_guard g(ctx->device);
    if (int rc = diffraction_edges(ctx, min_fold_deg)) return rc;
    const uint64_t n = ctx->n_diff_edges, m = out ? std::min<uint64_t>(n, cap) : 0;
    if (m) {
        std::vector<fs_diff_edge> h(m);
        CK(cudaMemcpyAsync(h.data(), ctx->d_diff_edges, sizeof(fs_diff_edge) * m, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        for (uint64_t i = 0; i < m; ++i) { out[2 * i] = h[i].tri; out[2 * i + 1] = h[i].k & 3u; }
    }
    *n_out = n;
    return FS_OK;
}

int fs_get_stats(fs_ctx* ctx, fs_stats* out)
{
    if (!ctx || !out) return FS_ERR_INVALID;
    dev_guard g(ctx->device);
    int rc = finish_stats(ctx);
    *out = ctx->stats;
    out->kernel_launches = ctx->launches.load();
    { std::lock_guard<std::mutex> lk(ctx->conv_mu); out->last_conv_ms = ctx->last_conv_ms; }
    return rc;
}

}  // extern "C"

// fs_multi.cu: make context 0's histogram the target of a multi-device update (allocated for n_sources, zeroed on the
// context stream, bookkeeping of fs_trace)
// per_source: host [n_sources] path counts of a per-source-budget update, or null (n_paths for every source)
// d_m2_out: context 0's second-moment buffer (zeroed), or null without FS_FLAG_NOISE_STATS
int fs_internal_hist_prepare(fs_ctx* ctx, uint32_t n_sources, uint64_t n_paths, const uint64_t* per_source,
                             unsigned long long** d_hist_out, ulonglong2** d_m2_out)
{
    dev_guard g(ctx->device);
    int rc = ensure_hist(ctx, n_sources);
    if (rc) return rc;
    const size_t hn = (size_t)n_sources * ctx->cfg.n_bands * ctx->cfg.n_bins;
    CK(cudaMemsetAsync(ctx->d_hist, 0, 8 * hn, ctx->stream));
    if ((rc = prepare_m2(ctx, n_sources, d_m2_out))) return rc;
    set_hist_counts(ctx, n_sources, n_paths, per_source);
    ctx->m2_valid = false;
    *d_hist_out = ctx->d_hist;
    return FS_OK;
}
// fs_multi.cu: the shard traces with second moments (d_m2 null = fs_trace_range_device / fs_trace_sources_range_device)
int fs_internal_trace_range(fs_ctx* ctx, const float* src_pos, uint32_t n_sources, const float lis_pos[3], uint64_t n_paths,
                            uint64_t g_first, uint64_t g_count, uint32_t max_depth, uint64_t seed, void* d_hist,
                            ulonglong2* d_m2, int zero_first)
{
    return trace_range_device(ctx, src_pos, n_sources, lis_pos, n_paths, g_first, g_count, max_depth, seed, d_hist, d_m2,
                              zero_first);
}
int fs_internal_trace_sources_range(fs_ctx* ctx, const fs_source_desc* src, uint32_t n_sources, const float lis_pos[3],
                                    uint64_t g_first, uint64_t g_count, uint64_t seed, void* d_hist, ulonglong2* d_m2,
                                    int zero_first)
{
    return trace_sources_range_device(ctx, src, n_sources, lis_pos, g_first, g_count, seed, d_hist, d_m2, zero_first);
}
// fs_multi.cu: the reduced second moments of context 0 belong to its histogram
void fs_internal_m2_valid(fs_ctx* ctx, bool valid) { ctx->m2_valid = valid; }
int fs_internal_check_dir_sources(fs_ctx* ctx, uint32_t n_sources, const char* who) { return check_dir_sources(ctx, n_sources, who); }

// ---- text float arrays (saved_ir.txt: one float per line, COMP.cpp:454-505); host only
int fs_load_float_array(const char* path, float* out, uint64_t cap, uint64_t* n_out)
{
    if (!path || !n_out) return FS_ERR_INVALID;
    FILE* f = fopen(path, "rb");
    if (!f) return FS_ERR_INVALID;
    uint64_t n = 0;
    char line[256];
    while (fgets(line, sizeof(line), f)) {
        const char* p = line;
        while (*p == ' ' || *p == '\t') ++p;
        if (*p == '\0' || *p == '\n' || *p == '\r') continue;            // ParseIntoArray(..., CullEmpty = true)
        char* end = nullptr;
        const float v = strtof(p, &end);                                // FCString::Atof: 0 for a non-numeric line
        if (out && n < cap) out[n] = (end == p) ? 0.0f : v;
        ++n;
    }
    fclose(f);
    *n_out = n;
    return FS_OK;
}

int fs_save_float_array(const char* path, const float* data, uint64_t n)
{
    if (!path || (!data && n)) return FS_ERR_INVALID;
    FILE* f = fopen(path, "wb");
    if (!f) return FS_ERR_INVALID;
    for (uint64_t i = 0; i < n; ++i) {
        char buf[48];
        snprintf(buf, sizeof(buf), "%.9g", (double)data[i]);
        if (!strpbrk(buf, ".eEn")) strcat(buf, ".0");                    // SanitizeFloat keeps one fractional digit ("1.0")
        if (fputs(buf, f) < 0 || (i + 1 < n && fputc('\n', f) == EOF)) { fclose(f); return FS_ERR_INVALID; }
    }
    return fclose(f) == 0 ? FS_OK : FS_ERR_INVALID;
}
