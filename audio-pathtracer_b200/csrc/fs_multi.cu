// fs_multi.cu -- several GPUs of one box behind the C-ABI (include/frequensee.h, fs_multi_*).
//
// SURVEY.md 8(b)/(e): "Multi-GPU is internal to the ctx".  The reference is one process with one game thread
// (SUB.cpp:55-85); the unit of parallel work is one iteration of its pair loop (SUB.cpp:215-230).  Here one host process
// owns one context per device: the global work range g = source * n_paths + i is cut into contiguous shards, every device
// traces its shard against its own copy of the BVH (enqueued by one host thread per device, so the launch work of the
// devices overlaps), and the per-device Q32.32 histograms are combined on device 0 WITHOUT a collective library:
//
//   k_hist_peer_store   on device i: vectorised stores of its histogram into slot i of a staging buffer that lives on device 0
//                       (peer-mapped memory: the stores travel over NVLink / NVSwitch), ordered by events
//   k_hist_sum          on device 0: hist0[j] += sum_i staging[i][j]
//
// Integer addition: the result is bit-identical for every device count and every shard order.  The reduced histogram is
// the histogram of context 0 (fs_multi_context(m, 0)), so fs_build_ir* / fs_conv_* of the single-device API continue from
// there.  A device may be listed more than once (two contexts on one GPU): that is how the path is tested on a one-GPU box.
#include "fs_internal.h"

#include <condition_variable>
#include <functional>
#include <new>
#include <thread>

// fs_api.cu
int fs_internal_hist_prepare(fs_ctx* ctx, uint32_t n_sources, uint64_t n_paths, const uint64_t* per_source,
                             unsigned long long** d_hist_out, ulonglong2** d_m2_out);
int fs_internal_trace_range(fs_ctx* ctx, const float* src_pos, uint32_t n_sources, const float lis_pos[3], uint64_t n_paths,
                            uint64_t g_first, uint64_t g_count, uint32_t max_depth, uint64_t seed, void* d_hist,
                            ulonglong2* d_m2, int zero_first);
int fs_internal_trace_sources_range(fs_ctx* ctx, const fs_source_desc* src, uint32_t n_sources, const float lis_pos[3],
                                    uint64_t g_first, uint64_t g_count, uint64_t seed, void* d_hist, ulonglong2* d_m2,
                                    int zero_first);
void fs_internal_m2_valid(fs_ctx* ctx, bool valid);
int fs_internal_check_dir_sources(fs_ctx* ctx, uint32_t n_sources, const char* who);

namespace {

__global__ void k_hist_peer_store(const ulonglong2* __restrict__ local, ulonglong2* __restrict__ remote, size_t n2)
{
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n2; i += (size_t)gridDim.x * blockDim.x) remote[i] = local[i];
    __threadfence_system();
}

__global__ void k_hist_sum(unsigned long long* __restrict__ hist, const unsigned long long* __restrict__ staging, size_t n, uint32_t n_slots,
                           size_t slot_stride)
{
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        unsigned long long s = hist[i];
        for (uint32_t k = 0; k < n_slots; ++k) s += staging[(size_t)k * slot_stride + i];
        hist[i] = s;
    }
}

// FS_FLAG_NOISE_STATS: m2[j] += sum_i staging[i][j] mod 2^128 (carry from the low word into the high word)
__global__ void k_m2_sum(ulonglong2* __restrict__ m2, const ulonglong2* __restrict__ staging, size_t n, uint32_t n_slots,
                         size_t slot_stride)
{
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        ulonglong2 s = m2[i];
        for (uint32_t k = 0; k < n_slots; ++k) {
            const ulonglong2 v = staging[(size_t)k * slot_stride + i];
            s.x += v.x;
            s.y += v.y + (s.x < v.x ? 1ull : 0ull);
        }
        m2[i] = s;
    }
}

// one persistent host thread per device: runs the closures the API thread hands it
struct worker {
    std::thread th;
    std::mutex mu;
    std::condition_variable cv;
    std::function<int()> job;
    bool has_job = false, done = true, quit = false;
    int rc = 0;
    void loop()
    {
        for (;;) {
            std::unique_lock<std::mutex> lk(mu);
            cv.wait(lk, [&] { return has_job || quit; });
            if (quit) return;
            std::function<int()> j = std::move(job);
            has_job = false;
            lk.unlock();
            const int r = j();
            lk.lock();
            rc = r; done = true;
            cv.notify_all();
        }
    }
    void post(std::function<int()> j)
    {
        std::lock_guard<std::mutex> lk(mu);
        job = std::move(j); has_job = true; done = false;
        cv.notify_all();
    }
    int wait()
    {
        std::unique_lock<std::mutex> lk(mu);
        cv.wait(lk, [&] { return done; });
        return rc;
    }
};

}  // namespace

struct fs_multi {
    uint32_t n = 0;
    std::vector<fs_ctx*> ctx;
    std::vector<int> dev;
    std::vector<worker*> wk;
    std::vector<unsigned long long*> d_local;      // [i] shard histogram on device i (i >= 1)
    std::vector<cudaEvent_t> ev_pushed;            // [i] recorded on device i's stream after its peer store
    unsigned long long* d_staging = nullptr;       // on device 0: [n - 1][cap] slots
    size_t cap = 0;                                // u64 elements per slot
    // FS_FLAG_NOISE_STATS: the same for the second moments, [S][B+1][K] (lo, hi) per slot
    std::vector<ulonglong2*> d_local_m2;
    ulonglong2* d_staging_m2 = nullptr;
    size_t cap_m2 = 0;                             // ulonglong2 elements per slot
    cudaEvent_t ev_ready = nullptr, ev_t0 = nullptr, ev_t1 = nullptr, ev_t2 = nullptr;
    float last_total_ms = 0.f, last_reduce_ms = 0.f;
    std::string err;
};

struct cur_dev_guard {                    // the API leaves the caller's current device as it found it
    int prev = -1;
    cur_dev_guard() { if (cudaGetDevice(&prev) != cudaSuccess) { prev = -1; (void)cudaGetLastError(); } }
    ~cur_dev_guard() { if (prev >= 0) cudaSetDevice(prev); }
};

static thread_local std::string g_multi_err;
static int mfail(int code, const std::string& msg) { g_multi_err = msg; return code; }

extern "C" {

const char* fs_multi_last_error(void) { return g_multi_err.c_str(); }

int fs_multi_create(const fs_config* cfg, const int* devices, uint32_t n_devices, fs_multi** out)
{
    if (!cfg || !out || n_devices == 0 || n_devices > 64) return mfail(FS_ERR_INVALID, "fs_multi_create: bad argument");
    *out = nullptr;
    cur_dev_guard guard;
    fs_multi* m = new (std::nothrow) fs_multi();
    if (!m) return mfail(FS_ERR_NOMEM, "out of host memory");
    m->n = n_devices;
    int rc = FS_OK;
    for (uint32_t i = 0; i < n_devices && rc == FS_OK; ++i) {
        fs_config c = *cfg;
        c.device = devices ? devices[i] : (int)i;
        fs_ctx* x = nullptr;
        rc = fs_create(&c, &x);
        if (rc != FS_OK) { mfail(rc, std::string("fs_multi_create: device ") + std::to_string(c.device) + ": " + fs_last_error(nullptr)); break; }
        m->ctx.push_back(x); m->dev.push_back(x->device);
    }
    if (rc == FS_OK) {
        // peer access towards device 0 (where the staging buffer lives)
        for (uint32_t i = 1; i < m->n && rc == FS_OK; ++i) {
            if (m->dev[i] == m->dev[0]) continue;
            int can = 0;
            cudaDeviceCanAccessPeer(&can, m->dev[i], m->dev[0]);
            if (!can) { rc = mfail(FS_ERR_CUDA, "fs_multi_create: no peer access between the devices (NVLink / PCIe P2P needed)"); break; }
            cudaSetDevice(m->dev[i]);
            cudaError_t e = cudaDeviceEnablePeerAccess(m->dev[0], 0);
            if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) rc = mfail(FS_ERR_CUDA, std::string("cudaDeviceEnablePeerAccess: ") + cudaGetErrorString(e));
            (void)cudaGetLastError();
        }
    }
    if (rc == FS_OK) {
        cudaSetDevice(m->dev[0]);
        if (cudaEventCreateWithFlags(&m->ev_ready, cudaEventDisableTiming) != cudaSuccess || cudaEventCreate(&m->ev_t0) != cudaSuccess ||
            cudaEventCreate(&m->ev_t1) != cudaSuccess || cudaEventCreate(&m->ev_t2) != cudaSuccess)
            rc = mfail(FS_ERR_CUDA, "cudaEventCreate");
        m->d_local.assign(m->n, nullptr); m->d_local_m2.assign(m->n, nullptr); m->ev_pushed.assign(m->n, nullptr);
        for (uint32_t i = 1; i < m->n && rc == FS_OK; ++i) {
            cudaSetDevice(m->dev[i]);
            if (cudaEventCreateWithFlags(&m->ev_pushed[i], cudaEventDisableTiming) != cudaSuccess) rc = mfail(FS_ERR_CUDA, "cudaEventCreate");
        }
        for (uint32_t i = 0; i < m->n; ++i) {
            worker* w = new worker();
            w->th = std::thread([w] { w->loop(); });
            m->wk.push_back(w);
        }
    }
    if (rc != FS_OK) { fs_multi_destroy(m); return rc; }
    *out = m;
    return FS_OK;
}

void fs_multi_destroy(fs_multi* m)
{
    if (!m) return;
    cur_dev_guard guard;
    for (worker* w : m->wk) {
        { std::lock_guard<std::mutex> lk(w->mu); w->quit = true; w->cv.notify_all(); }
        if (w->th.joinable()) w->th.join();
        delete w;
    }
    for (uint32_t i = 0; i < m->ctx.size(); ++i) {
        cudaSetDevice(m->dev[i]);
        cudaDeviceSynchronize();
        if (i < m->d_local.size()) cudaFree(m->d_local[i]);
        if (i < m->d_local_m2.size()) cudaFree(m->d_local_m2[i]);
        if (i < m->ev_pushed.size() && m->ev_pushed[i]) cudaEventDestroy(m->ev_pushed[i]);
    }
    if (!m->dev.empty()) {
        cudaSetDevice(m->dev[0]);
        cudaFree(m->d_staging); cudaFree(m->d_staging_m2);
        for (cudaEvent_t e : {m->ev_ready, m->ev_t0, m->ev_t1, m->ev_t2}) if (e) cudaEventDestroy(e);
    }
    for (fs_ctx* x : m->ctx) fs_destroy(x);
    delete m;
}

uint32_t fs_multi_device_count(const fs_multi* m) { return m ? m->n : 0; }
fs_ctx* fs_multi_context(fs_multi* m, uint32_t i) { return (m && i < m->n) ? m->ctx[i] : nullptr; }

// run f(i) on every device's host thread, return the first failure
static int on_all(fs_multi* m, const std::function<int(uint32_t)>& f)
{
    for (uint32_t i = 0; i < m->n; ++i) m->wk[i]->post([&f, i] { return f(i); });
    int rc = FS_OK;
    std::string msg;
    for (uint32_t i = 0; i < m->n; ++i) {
        const int r = m->wk[i]->wait();
        if (r != FS_OK && rc == FS_OK) rc = r;
    }
    return rc;
}

// the scene is replicated: every device commits its own BVH (the build is deterministic: identical trees)
int fs_multi_scene_set_triangles(fs_multi* m, const float* verts, const uint32_t* tri_material, uint64_t n_tris)
{
    if (!m) return FS_ERR_INVALID;
    std::vector<std::string> errs(m->n);
    int rc = on_all(m, [&](uint32_t i) { int r = fs_scene_set_triangles(m->ctx[i], verts, tri_material, n_tris); if (r) errs[i] = fs_last_error(m->ctx[i]); return r; });
    if (rc) for (auto& e : errs) if (!e.empty()) { mfail(rc, e); break; }
    return rc;
}
int fs_multi_scene_set_materials_ex(fs_multi* m, const float* absorption, const float* transmission, const float* scattering,
                                    const float* thickness_cm, uint32_t n_materials, uint32_t n_bands)
{
    if (!m) return FS_ERR_INVALID;
    std::vector<std::string> errs(m->n);
    int rc = on_all(m, [&](uint32_t i) {
        int r = fs_scene_set_materials_ex(m->ctx[i], absorption, transmission, scattering, thickness_cm, n_materials, n_bands);
        if (r) errs[i] = fs_last_error(m->ctx[i]);
        return r; });
    if (rc) for (auto& e : errs) if (!e.empty()) { mfail(rc, e); break; }
    return rc;
}
int fs_multi_scene_set_materials(fs_multi* m, const float* absorption, uint32_t n_materials, uint32_t n_bands)
{
    return fs_multi_scene_set_materials_ex(m, absorption, nullptr, nullptr, nullptr, n_materials, n_bands);
}
int fs_multi_scene_commit(fs_multi* m)
{
    if (!m) return FS_ERR_INVALID;
    std::vector<std::string> errs(m->n);
    int rc = on_all(m, [&](uint32_t i) { int r = fs_scene_commit(m->ctx[i]); if (r) errs[i] = fs_last_error(m->ctx[i]); return r; });
    if (rc) for (auto& e : errs) if (!e.empty()) { mfail(rc, e); break; }
    return rc;
}
int fs_multi_scene_update_vertices(fs_multi* m, const float* verts, uint64_t first_tri, uint64_t n_tris)
{
    if (!m) return FS_ERR_INVALID;
    std::vector<std::string> errs(m->n);
    int rc = on_all(m, [&](uint32_t i) { int r = fs_scene_update_vertices(m->ctx[i], verts, first_tri, n_tris); if (r) errs[i] = fs_last_error(m->ctx[i]); return r; });
    if (rc) for (auto& e : errs) if (!e.empty()) { mfail(rc, e); break; }
    return rc;
}
// every device refits its own copy (identical trees, identical results); the cost ratio is device 0's
int fs_multi_scene_refit(fs_multi* m, float* cost_ratio_out)
{
    if (!m) return FS_ERR_INVALID;
    std::vector<std::string> errs(m->n);
    std::vector<float> ratio(m->n, 1.0f);
    int rc = on_all(m, [&](uint32_t i) { int r = fs_scene_refit(m->ctx[i], &ratio[i]); if (r) errs[i] = fs_last_error(m->ctx[i]); return r; });
    if (rc) for (auto& e : errs) if (!e.empty()) { mfail(rc, e); break; }
    if (rc == FS_OK && cost_ratio_out) *cost_ratio_out = ratio[0];
    return rc;
}

// One IR update's trace over all devices (UpdateSource, SUB.cpp:128-195, for n_sources sources): shard, trace, peer-store,
// sum.  On return the work is ENQUEUED; the reduced histogram is context 0's (stream-ordered: fs_build_ir* on context 0
// follows without a host synchronisation).  hist_out (host [S][B][K]) may be NULL; non-NULL synchronises.
// G: the flat work range [0, G); trace(ctx, first, count, d_hist, zero_first) traces one shard; n_paths / per_source: the
// path counts context 0 records for its IR builders
// With FS_FLAG_NOISE_STATS the second moments travel the same way (trace's ulonglong2* argument: the shard's buffer) and are
// summed into context 0's with the carry.
static int multi_trace_common(fs_multi* m, uint32_t n_sources, uint64_t G, uint64_t n_paths, const uint64_t* per_source,
                              uint64_t* hist_out,
                              const std::function<int(fs_ctx*, uint64_t, uint64_t, void*, ulonglong2*, int)>& trace)
{
    cur_dev_guard guard;
    for (fs_ctx* c : m->ctx)                                  // before anything is enqueued on any device
        if (int r = fs_internal_check_dir_sources(c, n_sources, "fs_multi_trace")) return mfail(r, fs_last_error(c));
    fs_ctx* c0 = m->ctx[0];
    const size_t hn = (size_t)n_sources * c0->cfg.n_bands * c0->cfg.n_bins;
    const size_t cap = (hn + 1) & ~(size_t)1;                 // 16-byte vector stores
    if (m->cap < cap) {
        cudaSetDevice(m->dev[0]);
        cudaDeviceSynchronize();
        cudaFree(m->d_staging); m->d_staging = nullptr;
        if (m->n > 1 && cudaMalloc(&m->d_staging, 8 * cap * (m->n - 1)) != cudaSuccess) return mfail(FS_ERR_NOMEM, "fs_multi_trace: staging");
        for (uint32_t i = 1; i < m->n; ++i) {
            cudaSetDevice(m->dev[i]);
            cudaDeviceSynchronize();
            cudaFree(m->d_local[i]); m->d_local[i] = nullptr;
            if (cudaMalloc(&m->d_local[i], 8 * cap) != cudaSuccess) return mfail(FS_ERR_NOMEM, "fs_multi_trace: shard histogram");
            // (every update clears it on the device's own stream before tracing: zero_first below)
        }
        m->cap = cap;
    }
    const bool noise = (c0->cfg.flags & FS_FLAG_NOISE_STATS) != 0;
    const size_t mn = noise ? (size_t)n_sources * (c0->cfg.n_bands + 1u) * c0->cfg.n_bins : 0;
    if (m->cap_m2 < mn) {
        cudaSetDevice(m->dev[0]);
        cudaDeviceSynchronize();
        cudaFree(m->d_staging_m2); m->d_staging_m2 = nullptr;
        if (m->n > 1 && cudaMalloc(&m->d_staging_m2, sizeof(ulonglong2) * mn * (m->n - 1)) != cudaSuccess)
            return mfail(FS_ERR_NOMEM, "fs_multi_trace: staging");
        for (uint32_t i = 1; i < m->n; ++i) {
            cudaSetDevice(m->dev[i]);
            cudaDeviceSynchronize();
            cudaFree(m->d_local_m2[i]); m->d_local_m2[i] = nullptr;
            if (cudaMalloc(&m->d_local_m2[i], sizeof(ulonglong2) * mn) != cudaSuccess) return mfail(FS_ERR_NOMEM, "fs_multi_trace: shard moments");
        }
        m->cap_m2 = mn;
    }
    unsigned long long* d_hist0 = nullptr;
    ulonglong2* d_m20 = nullptr;
    {   // device 0: histogram of context 0, zeroed ("Flush", COMP.h:76-79)
        cudaSetDevice(m->dev[0]);
        if (cudaEventRecord(m->ev_t0, c0->stream) != cudaSuccess) return mfail(FS_ERR_CUDA, "cudaEventRecord");
        int rc = fs_internal_hist_prepare(c0, n_sources, n_paths, per_source, &d_hist0, &d_m20);
        if (rc) return mfail(rc, fs_last_error(c0));
    }
    std::vector<std::string> errs(m->n);
    int rc = on_all(m, [&](uint32_t i) {
        const uint64_t base = G / m->n, rem = G % m->n;
        const uint64_t first = i * base + (i < rem ? i : rem), count = base + (i < rem ? 1 : 0);
        fs_ctx* c = m->ctx[i];
        cudaSetDevice(m->dev[i]);
        int r = trace(c, first, count, i == 0 ? (void*)d_hist0 : (void*)m->d_local[i], i == 0 ? d_m20 : (noise ? m->d_local_m2[i] : nullptr),
                      i == 0 ? 0 : 1);
        if (r) { errs[i] = fs_last_error(c); return r; }
        if (i > 0) {
            // hand-written peer store: this device's shard histogram -> its slot of the staging buffer on device 0
            // (slot i - 1 is free again once device 0 has summed the previous update)
            if (cudaStreamWaitEvent(c->stream, m->ev_ready, 0) != cudaSuccess) { errs[i] = "cudaStreamWaitEvent"; return (int)FS_ERR_CUDA; }
            ulonglong2* remote = reinterpret_cast<ulonglong2*>(m->d_staging + (size_t)(i - 1) * m->cap);
            const size_t n2 = m->cap / 2;
            uint32_t grid = (uint32_t)((n2 + 255) / 256);
            if (grid > 4u * (uint32_t)c->sm_count) grid = 4u * (uint32_t)c->sm_count;
            k_hist_peer_store<<<grid, 256, 0, c->stream>>>(reinterpret_cast<const ulonglong2*>(m->d_local[i]), remote, n2);
            c->launches.fetch_add(1);
            if (noise) {
                uint32_t grid2 = (uint32_t)((mn + 255) / 256);
                if (grid2 > 4u * (uint32_t)c->sm_count) grid2 = 4u * (uint32_t)c->sm_count;
                k_hist_peer_store<<<grid2, 256, 0, c->stream>>>(m->d_local_m2[i], m->d_staging_m2 + (size_t)(i - 1) * m->cap_m2, mn);
                c->launches.fetch_add(1);
            }
            cudaError_t e = cudaGetLastError();
            if (e == cudaSuccess) e = cudaEventRecord(m->ev_pushed[i], c->stream);
            if (e != cudaSuccess) { errs[i] = std::string("peer store: ") + cudaGetErrorString(e); return (int)FS_ERR_CUDA; }
        }
        return (int)FS_OK; });
    if (rc) { for (auto& e : errs) if (!e.empty()) { mfail(rc, e); break; } return rc; }
    cudaSetDevice(m->dev[0]);
    cudaEventRecord(m->ev_t1, c0->stream);                    // device 0's own shard is traced
    for (uint32_t i = 1; i < m->n; ++i)
        if (cudaStreamWaitEvent(c0->stream, m->ev_pushed[i], 0) != cudaSuccess) return mfail(FS_ERR_CUDA, "cudaStreamWaitEvent");
    if (m->n > 1) {
        uint32_t grid = (uint32_t)((hn + 255) / 256);
        if (grid > 4u * (uint32_t)c0->sm_count) grid = 4u * (uint32_t)c0->sm_count;
        k_hist_sum<<<grid, 256, 0, c0->stream>>>(d_hist0, m->d_staging, hn, m->n - 1, m->cap);
        c0->launches.fetch_add(1);
        if (cudaGetLastError() != cudaSuccess) return mfail(FS_ERR_CUDA, "k_hist_sum");
        if (noise) {
            uint32_t grid2 = (uint32_t)((mn + 255) / 256);
            if (grid2 > 4u * (uint32_t)c0->sm_count) grid2 = 4u * (uint32_t)c0->sm_count;
            k_m2_sum<<<grid2, 256, 0, c0->stream>>>(d_m20, m->d_staging_m2, mn, m->n - 1, m->cap_m2);
            c0->launches.fetch_add(1);
            if (cudaGetLastError() != cudaSuccess) return mfail(FS_ERR_CUDA, "k_m2_sum");
        }
    }
    if (noise) fs_internal_m2_valid(c0, true);
    cudaEventRecord(m->ev_t2, c0->stream);
    cudaEventRecord(m->ev_ready, c0->stream);                 // the staging slots may be overwritten by the next update
    if (hist_out) {
        if (cudaMemcpyAsync(hist_out, d_hist0, 8 * hn, cudaMemcpyDeviceToHost, c0->stream) != cudaSuccess ||
            cudaStreamSynchronize(c0->stream) != cudaSuccess) return mfail(FS_ERR_CUDA, "fs_multi_trace: histogram read-back");
        for (uint32_t i = 0; i < m->n; ++i) {                 // a traversal overflow on any device invalidates the sum
            int r = fs_synchronize(m->ctx[i]);
            if (r) return mfail(r, fs_last_error(m->ctx[i]));
        }
    }
    return FS_OK;
}

int fs_multi_trace(fs_multi* m, const float* src_pos, uint32_t n_sources, const float lis_pos[3], uint64_t n_paths,
                   uint32_t max_depth, uint64_t seed, uint64_t* hist_out)
{
    if (!m) return FS_ERR_INVALID;
    if (!src_pos || !lis_pos || n_sources == 0 || n_paths == 0) return mfail(FS_ERR_INVALID, "fs_multi_trace: bad argument");
    return multi_trace_common(m, n_sources, (uint64_t)n_sources * n_paths, n_paths, nullptr, hist_out,
                              [&](fs_ctx* c, uint64_t first, uint64_t count, void* d_hist, ulonglong2* d_m2, int zero_first) {
                                  return fs_internal_trace_range(c, src_pos, n_sources, lis_pos, n_paths, first, count, max_depth,
                                                                 seed, d_hist, d_m2, zero_first); });
}

// fs_trace_sources over all devices: the flat range [0, sum n_s) is sharded like fs_multi_trace's
int fs_multi_trace_sources(fs_multi* m, const fs_source_desc* src, uint32_t n_sources, const float lis_pos[3], uint64_t seed,
                           uint64_t* hist_out)
{
    if (!m) return FS_ERR_INVALID;
    if (!src || !lis_pos || n_sources == 0) return mfail(FS_ERR_INVALID, "fs_multi_trace_sources: bad argument");
    std::vector<uint64_t> counts(n_sources);
    uint64_t G = 0, n_max = 0;
    for (uint32_t s = 0; s < n_sources; ++s) {
        // the full validation (depth limits, shared listener) is that of fs_trace_sources_range_device on every device
        if (src[s].n_paths == 0) return mfail(FS_ERR_INVALID, "fs_multi_trace_sources: a source has n_paths = 0");
        counts[s] = src[s].n_paths; G += src[s].n_paths;
        if (src[s].n_paths > n_max) n_max = src[s].n_paths;
    }
    return multi_trace_common(m, n_sources, G, n_max, counts.data(), hist_out,
                              [&](fs_ctx* c, uint64_t first, uint64_t count, void* d_hist, ulonglong2* d_m2, int zero_first) {
                                  return fs_internal_trace_sources_range(c, src, n_sources, lis_pos, first, count, seed, d_hist,
                                                                         d_m2, zero_first); });
}

// directional sources: every device weights its shard's paths with the same tables
int fs_multi_set_directivity_patterns(fs_multi* m, const fs_directivity* patterns, uint32_t n_patterns)
{
    if (!m) return FS_ERR_INVALID;
    std::vector<std::string> errs(m->n);
    int rc = on_all(m, [&](uint32_t i) { int r = fs_set_directivity_patterns(m->ctx[i], patterns, n_patterns); if (r) errs[i] = fs_last_error(m->ctx[i]); return r; });
    if (rc) for (auto& e : errs) if (!e.empty()) { mfail(rc, e); break; }
    return rc;
}
int fs_multi_set_source_directivity(fs_multi* m, const fs_source_orient* o, uint32_t n_sources)
{
    if (!m) return FS_ERR_INVALID;
    std::vector<std::string> errs(m->n);
    int rc = on_all(m, [&](uint32_t i) { int r = fs_set_source_directivity(m->ctx[i], o, n_sources); if (r) errs[i] = fs_last_error(m->ctx[i]); return r; });
    if (rc) for (auto& e : errs) if (!e.empty()) { mfail(rc, e); break; }
    return rc;
}

// device time of the last fs_multi_trace on device 0's stream: the whole update (it ends when the slowest device has
// delivered) and the part after device 0's own shard (waiting for the peers + the sum).  Synchronises.
int fs_multi_last_ms(fs_multi* m, float* total_ms, float* reduce_ms)
{
    if (!m) return FS_ERR_INVALID;
    cur_dev_guard guard;
    cudaSetDevice(m->dev[0]);
    if (cudaEventSynchronize(m->ev_t2) != cudaSuccess) return mfail(FS_ERR_CUDA, "cudaEventSynchronize");
    float a = 0.f, b = 0.f;
    cudaEventElapsedTime(&a, m->ev_t0, m->ev_t2);
    cudaEventElapsedTime(&b, m->ev_t1, m->ev_t2);
    (void)cudaGetLastError();
    if (total_ms) *total_ms = a;
    if (reduce_ms) *reduce_ms = b;
    return FS_OK;
}

int fs_multi_synchronize(fs_multi* m)
{
    if (!m) return FS_ERR_INVALID;
    for (uint32_t i = 0; i < m->n; ++i) {
        int r = fs_synchronize(m->ctx[i]);
        if (r) return mfail(r, fs_last_error(m->ctx[i]));
    }
    return FS_OK;
}

}  // extern "C"
