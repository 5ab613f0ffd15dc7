// fs_wavefront.cu -- wavefront BDPT: subpath extension, connection (shadow rays), path
// evaluation and fixed-point splatting.
//
// One batch = `batch` path pairs = 2*batch subpaths (side 0 from the source, side 1 from the
// listener; sp_id = 2*path + side).  Per bounce k one launch of k_extend consumes the queue of
// live subpaths and produces the next one, compacted with warp ballots (one atomic per warp), so
// warps stay full as Russian roulette / misses / max depth retire subpaths.  Kernels are
// persistent: grid = SMs x resident CTAs, each warp pulls 32 queue entries at a time from a
// device-side cursor, and queue lengths live on the device, so the whole update is enqueued
// without a host round trip.
//
//   k_extend  (GeneratePath, SUB.cpp:279-355)        RR, sample, closest hit, node record
//   k_connect (ConnectSubpaths, SUB.cpp:235-277)     any-hit ray between the two end nodes
//   k_eval    (EvaluatePath, SUB.cpp:360-420 + AddEnergyAtDelay, COMP.h:87-91)
//             energy product in path order, clamp/gain, Q32.32, warp-aggregated u64 atomics
//
// HBM layout (SoA, float4 granularity so every lane moves 16 B):
//   st_pos/st_nrm[2][2*cap]  ping-pong compacted subpath state
//   rec[k][sp_id]            node record k>=1 of subpath sp_id: (segment length, material, pdf, pdf^pdf_exponent)
//   end_pos[sp_id]           last node position + node count
#include "fs_internal.h"

namespace {

constexpr int WF_THREADS = 256;

// Per-step streaming state (ray queues / ray log, hit records, node records, end points: hundreds of MB per update) is written
// once and read once.  With FS_STREAM_HINTS the accesses carry the evict-first hint (st.global.cs / ld.global.cs) so that they
// do not push the BVH out of L2 -- it matters for scenes whose nodes + triangles do not fit the 126 MB L2 anyway.
#ifndef FS_STREAM_HINTS
#define FS_STREAM_HINTS 0      // measured (r2j): no effect on the room or the hall, left off
#endif
#if FS_STREAM_HINTS
#define FS_ST4(ptr, v) __stcs((ptr), (v))
#define FS_ST2(ptr, v) __stcs((ptr), (v))
#define FS_LD4(ptr) __ldcs(ptr)
#define FS_LD2(ptr) __ldcs(ptr)
#else
#define FS_ST4(ptr, v) (*(ptr) = (v))
#define FS_ST2(ptr, v) (*(ptr) = (v))
#define FS_LD4(ptr) (*(ptr))
#define FS_LD2(ptr) (*(ptr))
#endif

enum { MODE_BVH = 0, MODE_TOP = 1, MODE_BRUTE = 2 };

__device__ __forceinline__ uint32_t lane_id() { return threadIdx.x & 31u; }

// brute-force closest hit over the (sorted) triangle array; same (t, original id) rule
__device__ __forceinline__ int closest_brute(const fs_bvh_view& bv, fs_vec3 o, fs_vec3 d, float& best_t)
{
    int best = -1; uint32_t best_orig = 0xffffffffu;
    float bt = __int_as_float(0x7f800000);
    for (uint32_t i = 0; i < bv.n_tris; ++i) {
        const float4* tp = bv.tris + (size_t)i * 4;
        float4 a = fs_ldg4(tp), b = fs_ldg4(tp + 1), c = fs_ldg4(tp + 2);
        float t;
        if (fs_intersect_tri(o, d, fs_mk(a.x, a.y, a.z), fs_mk(b.x, b.y, b.z), fs_mk(c.x, c.y, c.z), t)) {
            uint32_t oi = __ldg(bv.tri_orig + i);
            if (t < bt || (t == bt && oi < best_orig)) { bt = t; best = (int)i; best_orig = oi; }
        }
    }
    best_t = bt;
    return best;
}
__device__ __forceinline__ bool any_brute(const fs_bvh_view& bv, fs_vec3 o, fs_vec3 d, float tmax)
{
    for (uint32_t i = 0; i < bv.n_tris; ++i) {
        const float4* tp = bv.tris + (size_t)i * 4;
        float4 a = fs_ldg4(tp), b = fs_ldg4(tp + 1), c = fs_ldg4(tp + 2);
        float t;
        if (fs_intersect_tri(o, d, fs_mk(a.x, a.y, a.z), fs_mk(b.x, b.y, b.z), fs_mk(c.x, c.y, c.z), t) && t < tmax)
            return true;
    }
    return false;
}

template <bool COUNT, int MODE>
__device__ __forceinline__ int trace_closest(const fs_trace_params& tp, const float4* top, fs_vec3 o, fs_vec3 d,
                                             float& t, fs_visit_counters* vc, uint32_t* overflow)
{
    if (MODE == MODE_BRUTE) return closest_brute(tp.bv, o, d, t);
    return fs_closest_hit<COUNT, MODE == MODE_TOP>(tp.bv, top, o, d, t, vc, overflow);
}
template <bool COUNT, int MODE>
__device__ __forceinline__ bool trace_any(const fs_trace_params& tp, const float4* top, fs_vec3 o, fs_vec3 d,
                                          float tmax, fs_visit_counters* vc, uint32_t* overflow)
{
    if (MODE == MODE_BRUTE) return any_brute(tp.bv, o, d, tmax);
    return fs_any_hit<COUNT, MODE == MODE_TOP>(tp.bv, top, o, d, tmax, vc, overflow);
}

__device__ __forceinline__ void stage_top(const fs_trace_params& tp, float4* smem_top)
{
    for (uint32_t i = threadIdx.x; i < tp.n_top * 4u; i += blockDim.x) smem_top[i] = tp.top[i];
    __syncthreads();
}

__device__ __forceinline__ void flush_counters(fs_dev_counters* dc, fs_visit_counters vc, bool shadow = false)
{
    uint32_t n = vc.nodes, t = vc.tris;
    for (int o = 16; o; o >>= 1) {
        n += __shfl_xor_sync(0xffffffffu, n, o);
        t += __shfl_xor_sync(0xffffffffu, t, o);
    }
    if (lane_id() == 0) {
        atomicAdd(&dc->node_visits, (unsigned long long)n);
        atomicAdd(&dc->tri_tests, (unsigned long long)t);
        if (shadow) {
            atomicAdd(&dc->shadow_node_visits, (unsigned long long)n);
            atomicAdd(&dc->shadow_tri_tests, (unsigned long long)t);
        }
    }
}

// ---------------------------------------------------------------------------------------------
// Source of pair p of the batch (work index g = g_first + p), its depth limit and the Philox key of its listener subpath
// under FS_FLAG_SHARE_LISTENER.  Uniform budgets: g = source * n_paths + i.  Per-source budgets (tp.src_off): source s owns
// g in [src_off[s], src_off[s+1]); k_resolve_sources has stored every pair's (source, depth) in wb.pair_src.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t pair_source(const fs_trace_params& tp, const fs_wave_buffers& wb, uint32_t p)
{
    return tp.src_off ? wb.pair_src[p].x : (uint32_t)((tp.g_first + p) / tp.n_paths);
}
__device__ __forceinline__ uint32_t pair_depth(const fs_trace_params& tp, const fs_wave_buffers& wb, uint32_t p)
{
    return tp.src_off ? wb.pair_src[p].y : tp.max_depth;
}
__device__ __forceinline__ uint64_t listener_key(const fs_trace_params& tp, const fs_wave_buffers& wb, uint32_t p)
{
    const uint64_t g = tp.g_first + p;
    return tp.src_off ? g - tp.src_off[wb.pair_src[p].x] : g % tp.n_paths;
}
__device__ __forceinline__ fs_vec3 source_pos(const fs_trace_params& tp, uint32_t s)
{
    return fs_mk(__ldg(tp.src_pos + 3 * s), __ldg(tp.src_pos + 3 * s + 1), __ldg(tp.src_pos + 3 * s + 2));
}

// per-source budgets: (source, depth) of every pair of the batch, by binary search over the offsets (once per batch)
__global__ void k_resolve_sources(const fs_trace_params tp, const fs_wave_buffers wb)
{
    const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= tp.batch) return;
    const uint64_t g = tp.g_first + p;
    uint32_t lo = 0, hi = tp.n_src;                       // src_off[lo] <= g < src_off[hi]
    while (hi - lo > 1u) {
        const uint32_t mid = (lo + hi) >> 1;
        if (__ldg(tp.src_off + mid) <= g) lo = mid; else hi = mid;
    }
    wb.pair_src[p] = make_uint2(lo, __ldg(tp.src_depth + lo));
}

// ---------------------------------------------------------------------------------------------
// k_extend: bounce k of every live subpath
// ---------------------------------------------------------------------------------------------
template <bool COUNT, int MODE>
__global__ void __launch_bounds__(WF_THREADS)
k_extend(const fs_trace_params tp, const fs_wave_buffers wb, uint32_t k, int in_buf,
         fs_dev_counters* __restrict__ dc)
{
    extern __shared__ float4 smem_top[];
    if (MODE == MODE_TOP) stage_top(tp, smem_top);
    const uint32_t lane = lane_id();
    const uint32_t count = (k == 0) ? 2u * tp.batch : wb.q_count[k];
    const float4* __restrict__ in_pos = wb.st_pos[in_buf];
    const float4* __restrict__ in_nrm = wb.st_nrm[in_buf];
    float4* __restrict__ out_pos = wb.st_pos[in_buf ^ 1];
    float4* __restrict__ out_nrm = wb.st_nrm[in_buf ^ 1];
    const uint32_t stride = 2u * wb.cap;             // rec[k][sp_id]: one plane per node index (writes of a bounce stay semi-coalesced)
    fs_visit_counters vc; vc.nodes = 0; vc.tris = 0;
    uint32_t rays_local = 0;
    for (;;) {
        uint32_t base = 0;
        if (lane == 0) base = atomicAdd(&wb.q_cursor[k], 32u);
        base = __shfl_sync(0xffffffffu, base, 0);
        if (base >= count) break;
        const uint32_t j = base + lane;
        const bool valid = j < count;
        bool alive = false;
        fs_vec3 pos = fs_mk(0.f, 0.f, 0.f), nrm = fs_mk(0.f, 0.f, 0.f);
        uint32_t sp_id = 0;
        if (valid) {
            if (k == 0) {
                // node 0: actor location, zero normal, no material, probability 1 (SUB.cpp:287-291)
                sp_id = j;
                if (sp_id & 1u) {
                    pos = fs_mk(tp.lis[0], tp.lis[1], tp.lis[2]);
                } else {
                    pos = source_pos(tp, pair_source(tp, wb, sp_id >> 1));
                }
            } else {
                float4 a = in_pos[j], b = in_nrm[j];
                pos = fs_mk(a.x, a.y, a.z); sp_id = __float_as_uint(a.w);
                nrm = fs_mk(b.x, b.y, b.z);
            }
            const uint64_t g = tp.g_first + (sp_id >> 1);
            uint32_t r[4];
            fs_philox4x32_10((uint32_t)g, (uint32_t)(g >> 32), k, sp_id & 1u, tp.seed_lo, tp.seed_hi, r);
            const float u0 = fs_u01(r[0]), u1 = fs_u01(r[1]), u2 = fs_u01(r[2]);
            bool terminated = true;
            uint32_t n_nodes = k + 1;                    // nodes pushed so far (SUB.cpp:297-298)
            const uint32_t depth = pair_depth(tp, wb, sp_id >> 1);
            if (k < depth && u0 < tp.rr_prob) {          // SUB.cpp:301-302 (k < depth: a depth-0 source traces no ray)
                fs_vec3 dir; float prob;
                if (k == 0) {                            // SUB.cpp:306-311
                    dir = fs_sample_sphere(u1, u2);
                    prob = FS_INV_4PI * tp.rr_prob;
                } else {                                 // SUB.cpp:312-318 (FIX: true cosine lobe)
                    float ct;
                    dir = fs_sample_cos_hemisphere(nrm, u1, u2, ct);
                    prob = (ct * FS_INV_PI) * tp.rr_prob;
                }
                ++rays_local;
                float t;
                uint32_t ovf_dummy = 0;
                int tri = trace_closest<COUNT, MODE>(tp, smem_top, pos, dir, t, &vc, &ovf_dummy);
                if (ovf_dummy) dc->overflow = 1u;
                if (tri >= 0) {                          // SUB.cpp:343-348
                    const float4* tq = tp.bv.tris + (size_t)tri * 4;
                    fs_vec3 fn = fs_mk(fs_ldg4(tq).w, fs_ldg4(tq + 1).w, fs_ldg4(tq + 2).w);
                    if (fs_dot(fn, dir) > 0.0f) { fn.x = -fn.x; fn.y = -fn.y; fn.z = -fn.z; }
                    fs_vec3 np;
                    np.x = fmaf(tp.eps_offset, fn.x, fmaf(t, dir.x, pos.x));
                    np.y = fmaf(tp.eps_offset, fn.y, fmaf(t, dir.y, pos.y));
                    np.z = fmaf(tp.eps_offset, fn.z, fmaf(t, dir.z, pos.z));
                    fs_vec3 dl = fs_sub(np, pos);
                    float seg = sqrtf(fs_dot(dl, dl));
                    uint32_t mat = __ldg(tp.bv.tri_mat + tri);
                    wb.rec[(size_t)(k + 1) * stride + sp_id] =
                        make_float4(seg, __uint_as_float(mat), prob, fs_pow(prob, tp.ep.pdf_exponent));
                    pos = np; nrm = fn;
                    n_nodes = k + 2;
                    terminated = (k + 1 >= depth);               // PARAM: ray budget per subpath
                }
                // miss: FIX -> subpath ends at the current node
            }
            if (terminated) wb.end_pos[sp_id] = make_float4(pos.x, pos.y, pos.z, __uint_as_float(n_nodes));
            alive = !terminated;
        }
        // ballot compaction into the next queue: one atomic per warp
        const uint32_t m = __ballot_sync(0xffffffffu, alive);
        if (m) {
            uint32_t slot = 0;
            if (lane == 0) slot = atomicAdd(&wb.q_count[k + 1], (uint32_t)__popc(m));
            slot = __shfl_sync(0xffffffffu, slot, 0);
            if (alive) {
                const uint32_t o = slot + __popc(m & ((1u << lane) - 1u));
                out_pos[o] = make_float4(pos.x, pos.y, pos.z, __uint_as_float(sp_id));
                out_nrm[o] = make_float4(nrm.x, nrm.y, nrm.z, 0.f);
            }
        }
    }
    for (int o = 16; o; o >>= 1) rays_local += __shfl_xor_sync(0xffffffffu, rays_local, o);
    if (lane == 0 && rays_local) atomicAdd(&dc->ext_rays, (unsigned long long)rays_local);
    if (COUNT) flush_counters(dc, vc);
}

// ---------------------------------------------------------------------------------------------
// k_connect: one visibility ray per path pair between the two LAST nodes
// ---------------------------------------------------------------------------------------------
template <bool COUNT, int MODE>
__global__ void __launch_bounds__(WF_THREADS)
k_connect(const fs_trace_params tp, const fs_wave_buffers wb, fs_dev_counters* __restrict__ dc,
          fs_path_dbg* __restrict__ dbg)
{
    extern __shared__ float4 smem_top[];
    if (MODE == MODE_TOP) stage_top(tp, smem_top);
    const uint32_t lane = lane_id();
    const uint32_t qi = tp.max_depth + 1;          // cursor / counter slot of this stage
    fs_visit_counters vc; vc.nodes = 0; vc.tris = 0;
    uint32_t rays_local = 0;
    for (;;) {
        uint32_t base = 0;
        if (lane == 0) base = atomicAdd(&wb.q_cursor[qi], 32u);
        base = __shfl_sync(0xffffffffu, base, 0);
        if (base >= tp.batch) break;
        const uint32_t p = base + lane;
        const bool valid = p < tp.batch;
        bool connected = false;
        float len = 0.f;
        if (valid) {
            float4 fe = wb.end_pos[2u * p], be = wb.end_pos[2u * p + 1u];
            fs_vec3 F = fs_mk(fe.x, fe.y, fe.z), Bp = fs_mk(be.x, be.y, be.z);
            fs_vec3 dl = fs_sub(Bp, F);
            len = sqrtf(fs_dot(dl, dl));
            float tmax = len - tp.eps_connect;              // SUB.cpp:253
            bool occluded = false;
            if (tmax > 0.0f) {
                float inv = 1.0f / len;
                fs_vec3 dir = fs_mk(dl.x * inv, dl.y * inv, dl.z * inv);
                ++rays_local;
                uint32_t ovf_dummy = 0;
                occluded = trace_any<COUNT, MODE>(tp, smem_top, F, dir, tmax, &vc, &ovf_dummy);
                if (ovf_dummy) dc->overflow = 1u;
            }
            connected = !occluded;
            if (dbg) {
                fs_path_dbg* q = dbg + p;
                q->n_src_nodes = __float_as_uint(fe.w); q->n_lis_nodes = __float_as_uint(be.w);
                q->connected = connected ? 1u : 0u; q->bin = -1; q->delay_s = 0.f; q->total_dist = 0.f;
                for (int b = 0; b < FS_MAX_BANDS; ++b) q->energy[b] = 0.f;
                q->src_end[0] = fe.x; q->src_end[1] = fe.y; q->src_end[2] = fe.z;
                q->lis_end[0] = be.x; q->lis_end[1] = be.y; q->lis_end[2] = be.z;
            }
        }
        const uint32_t m = __ballot_sync(0xffffffffu, connected);
        if (m) {
            uint32_t slot = 0;
            if (lane == 0) slot = atomicAdd(&wb.q_count[qi], (uint32_t)__popc(m));
            slot = __shfl_sync(0xffffffffu, slot, 0);
            if (connected) {
                const uint32_t o = slot + __popc(m & ((1u << lane) - 1u));
                wb.conn_queue[o] = p;
                wb.conn_len[p] = len;
            }
        }
    }
    for (int o = 16; o; o >>= 1) rays_local += __shfl_xor_sync(0xffffffffu, rays_local, o);
    if (lane == 0 && rays_local) atomicAdd(&dc->shadow_rays, (unsigned long long)rays_local);
    if (COUNT) flush_counters(dc, vc, true);
}

// ---------------------------------------------------------------------------------------------
// k_eval: EvaluatePath over F nodes ++ reverse(B nodes), then the splat
// ---------------------------------------------------------------------------------------------
// Sum of `v` over the lanes of `peers` (all lanes holding the same histogram address), result valid
// in the group's lowest lane.  Tree reduction over an arbitrary lane subset: in every round the
// even-ranked lanes absorb their next higher peer, odd-ranked lanes drop out.
__device__ __forceinline__ unsigned long long reduce_peers(uint32_t peers, unsigned long long v)
{
    const uint32_t group = peers;
    const uint32_t lane = lane_id();
    uint32_t rel = __popc(peers & ((1u << lane) - 1u));
    peers &= (0xfffffffeu << lane);                       // peers above me
    while (__any_sync(group, peers)) {
        const int next = __ffs(peers);                    // 1-based, 0 = none
        const unsigned long long t = __shfl_sync(group, v, next ? next - 1 : (int)lane);
        if (next) v += t;
        const bool done = rel & 1u;
        if (done) peers = 0;
        peers &= __ballot_sync(group, !done);
        rel >>= 1;
    }
    return v;
}

// reduce_peers for a 128-bit value (lo, hi): the second moment of FS_FLAG_NOISE_STATS.  Sums are taken mod 2^128.
__device__ __forceinline__ void reduce_peers_u128(uint32_t peers, unsigned long long& lo, unsigned long long& hi)
{
    const uint32_t group = peers;
    const uint32_t lane = lane_id();
    uint32_t rel = __popc(peers & ((1u << lane) - 1u));
    peers &= (0xfffffffeu << lane);
    while (__any_sync(group, peers)) {
        const int next = __ffs(peers);
        const int src = next ? next - 1 : (int)lane;
        const unsigned long long tl = __shfl_sync(group, lo, src), th = __shfl_sync(group, hi, src);
        if (next) { lo += tl; hi += th + (lo < tl ? 1ull : 0ull); }
        const bool done = rel & 1u;
        if (done) peers = 0;
        peers &= __ballot_sync(group, !done);
        rel >>= 1;
    }
}

// *p += (lo, hi) mod 2^128: one atomic on the low word, one on the high word with the carry of the first.  Every add is
// exact mod 2^128, so the sum does not depend on the order of the adds.
__device__ __forceinline__ void atomic_add_u128(ulonglong2* p, unsigned long long lo, unsigned long long hi)
{
    const unsigned long long old = atomicAdd(&p->x, lo);
    if (old + lo < old) ++hi;
    if (hi) atomicAdd(&p->y, hi);
}

// one band of one segment of EvaluatePath (SUB.cpp:368-399); P = prob^pdf_exponent comes from the node record
__device__ __forceinline__ void eval_seg_band(const fs_eval_params& ep, float bs, float P, float d, float air_b, float& E)
{
    if (d < ep.min_seg) return;                           // SUB.cpp:375-378 (the caller has already added d to the delay)
    const float G = 1.0f / (FS_FOUR_PI * (d * d));        // :391
    float e = E;
    e *= bs;                                              // :392
    e *= G;                                               // :393
    e *= fs_exp(-air_b * d);                              // :395-397
    e /= P;                                               // :398
    E = e;
}

// 8 lanes per connected path, one absorption band each (4 paths per warp): the walk over the node
// records is uniform across the 8 lanes of a path, so SIMD efficiency no longer depends on the band
// loop (the one-thread-per-path version ran at 8.9 of 32 lanes, profiles/r1e_summary.md).
// position of node k of subpath sp (node 0 = the source / the listener); FS_FLAG_CONNECT_ALL only
__device__ __forceinline__ fs_vec3 node_pos(const fs_trace_params& tp, const fs_wave_buffers& wb, uint32_t sp, uint32_t k, uint32_t stride)
{
    if (k == 0) {
        if (sp & 1u) return fs_mk(tp.lis[0], tp.lis[1], tp.lis[2]);
        return source_pos(tp, pair_source(tp, wb, sp >> 1));
    }
    const float4 v = wb.npos[(size_t)k * stride + sp];
    return fs_mk(v.x, v.y, v.z);
}

// Directional sources: energy gain of band b for a path of source s that leaves it along the unit direction (dx, dy, dz);
// 1 for an omni source (fs_directivity.h has the interpolation rule)
__device__ __forceinline__ float dir_gain(const fs_trace_params& tp, uint32_t s, uint32_t b, float dx, float dy, float dz)
{
    const float4 o = __ldg(tp.dir_orient + s);
    const uint32_t pat = __float_as_uint(o.w);
    if (pat == FS_OMNI) return 1.0f;
    float t;
    const uint32_t i = fs_dir_index(fs_dir_cos(dx, dy, dz, o.x, o.y, o.z), &t);
    const float* T = tp.dir_gain + ((size_t)pat * FS_MAX_BANDS + b) * FS_DIR_POINTS + i;
    return fs_dir_lerp(__ldg(T), __ldg(T + 1), t);
}

// bounce-0 direction of the source subpath of work index g: what choose_direction / k_extend drew at node 0
__device__ __forceinline__ fs_vec3 source_bounce0(const fs_trace_params& tp, uint64_t g)
{
    uint32_t r[4];
    fs_philox4x32_10((uint32_t)g, (uint32_t)(g >> 32), 0u, 0u, tp.seed_lo, tp.seed_hi, r);
    return fs_sample_sphere(fs_u01(r[1]), fs_u01(r[2]));
}

// M2 (FS_FLAG_NOISE_STATS, endpoint connection only): also splats the exact square of every Q32.32 value into
// m2 [S][B+1][K] (lo, hi): q_b^2 into slot b, and (sum_b q_b)^2 of the path into slot B (broadband)
// DIR (directional sources, tp.dir_orient set): every band starts at the gain of its source's pattern at the path's emission
// direction instead of 1.  The 8 lanes of a path compute that direction redundantly: they run in lockstep, so one lane
// doing it alone would cost the warp the same issue slots and add shuffles to hand the result out.
template <bool ALL, bool M2 = false, bool DIR = false>
__global__ void __launch_bounds__(WF_THREADS)
k_eval(const fs_trace_params tp, const fs_wave_buffers wb, unsigned long long* __restrict__ hist,
       fs_dev_counters* __restrict__ dc, fs_path_dbg* __restrict__ dbg, ulonglong2* __restrict__ m2)
{
    const uint32_t lane = lane_id();
    const uint32_t sub = lane >> 3, b = lane & 7u;
    const uint32_t qi = tp.max_depth + 1;
    const uint32_t count = wb.q_count[qi];
    const uint32_t stride = 2u * wb.cap;             // rec[k][sp_id]: one plane per node index (writes of a bounce stay semi-coalesced)
    const uint32_t NBr = tp.ep.n_bands;
    const bool band_on = b < NBr;
    const float air_b = band_on ? tp.ep.air[b] : 0.0f;
    if (blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(&dc->connected, (unsigned long long)count);
    const uint32_t warp_global = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint32_t n_warps = (gridDim.x * blockDim.x) >> 5;
    for (uint32_t base = warp_global * 4u; base < count; base += n_warps * 4u) {
        const uint32_t j = base + sub;
        const bool valid = (j < count) && band_on;
        unsigned long long q = 0ull;
        uint32_t key = 0xffffffffu;
        size_t hidx = 0, midx = 0;
        if (valid) {
            // ALL: the queue entry names a prefix pair (pair << 12 | (s-1) << 6 | (t-1)); the path is F[0..s) ++ reverse(B[0..t)),
            // its connecting segment is recomputed from the node positions, its weight is 1 / (s + t - 1)
            const uint32_t id = ALL ? wb.all_conn[j] : wb.conn_queue[j];
            const uint32_t p = ALL ? (id >> 12) : id;
            const uint32_t sf = 2u * p, sb = 2u * p + 1u;
            const uint32_t nf = ALL ? ((id >> 6) & 63u) + 1u : __float_as_uint(wb.end_pos[sf].w);
            const uint32_t nb = ALL ? (id & 63u) + 1u : __float_as_uint(wb.end_pos[sb].w);
            float len;
            fs_vec3 dl;
            if (ALL) {
                dl = fs_sub(node_pos(tp, wb, sb, nb - 1u, stride), node_pos(tp, wb, sf, nf - 1u, stride));
                len = sqrtf(fs_dot(dl, dl));
            } else len = wb.conn_len[p];
            float E = 1.0f, total = 0.0f;
            if (DIR) {
                // emission direction: the bounce-0 sample if the source prefix left node 0, else the connection ray's
                fs_vec3 d;
                if (nf >= 2u) d = source_bounce0(tp, tp.g_first + p);
                else {
                    if (!ALL) {
                        const float4 fe = wb.end_pos[sf], be = wb.end_pos[sb];
                        dl = fs_sub(fs_mk(be.x, be.y, be.z), fs_mk(fe.x, fe.y, fe.z));
                    }
                    const float inv = 1.0f / len;
                    d = fs_mk(dl.x * inv, dl.y * inv, dl.z * inv);
                }
                E = dir_gain(tp, pair_source(tp, wb, p), b, d.x, d.y, d.z);
            }
            float bs = 1.0f, P = 1.0f;                    // node 0 of the source subpath: no material, probability 1
            const float4* __restrict__ rf = wb.rec + sf;
            const float4* __restrict__ rb = wb.rec + sb;
            // records are fetched four at a time so their latencies overlap
            for (uint32_t i0 = 1; i0 < nf; i0 += 4) {     // segments F_{i-1} -> F_i
                float4 r[4];
#pragma unroll
                for (uint32_t u = 0; u < 4; ++u) r[u] = (i0 + u < nf) ? FS_LD4(rf + (size_t)(i0 + u) * stride) : make_float4(0.f, 0.f, 1.f, 1.f);
#pragma unroll
                for (uint32_t u = 0; u < 4; ++u) {
                    if (i0 + u < nf) {
                        total += r[u].x;                  // ScaledDistance += NodeDistance, SUB.cpp:374
                        eval_seg_band(tp.ep, bs, P, r[u].x, air_b, E);
                        // factor of node i0 + u for the segment that leaves it: the lobe the walk took there (top byte; always
                        // the diffuse one without the material model), the diffuse lobe where the prefix is cut for a connection
                        const uint32_t mw = __float_as_uint(r[u].y);
                        const uint32_t evn = (ALL && i0 + u == nf - 1u) ? 0u : (mw >> 24);
                        bs = __ldg(tp.refl_over_pi + ((size_t)evn * tp.n_mats + (mw & 0x00ffffffu)) * NBr + b);
                        P = r[u].w;
                    }
                }
            }
            total += len;
            eval_seg_band(tp.ep, bs, P, len, air_b, E);   // connection F_last -> B_last
            for (int i0 = (int)nb - 1; i0 >= 1; i0 -= 4) { // B_i -> B_{i-1}
                float4 r[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) r[u] = (i0 - u >= 1) ? FS_LD4(rb + (size_t)(i0 - u) * stride) : make_float4(0.f, 0.f, 1.f, 1.f);
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    if (i0 - u >= 1) {
                        total += r[u].x;
                        const uint32_t mw = __float_as_uint(r[u].y);
                        const uint32_t evn = (ALL && i0 - u == (int)nb - 1) ? 0u : (mw >> 24);
                        eval_seg_band(tp.ep, __ldg(tp.refl_over_pi + ((size_t)evn * tp.n_mats + (mw & 0x00ffffffu)) * NBr + b), r[u].w, r[u].x, air_b, E);
                    }
                }
            }
            const float delay = total / tp.sound_speed;                           // SUB.cpp:419
            const float fb = floorf((delay * 1000.0f) / tp.bin_ms);               // COMP.h:89
            uint32_t bin;
            if (!(fb >= 0.0f)) bin = 0;
            else if (fb >= (float)(tp.n_bins - 1)) bin = tp.n_bins - 1;
            else bin = (uint32_t)fb;
            const uint32_t s = pair_source(tp, wb, p);
            float e = E;
            e = (e < tp.energy_clamp) ? e : tp.energy_clamp;                      // SUB.cpp:410
            e = e * tp.energy_gain;                                               // SUB.cpp:413
            if (ALL && nf + nb > 2u) e = e * (1.0f / (float)(nf + nb - 1u));      // one over the strategies of this path length
            q = (unsigned long long)(e * 4294967296.0f);                          // Q32.32
            hidx = ((size_t)s * NBr + b) * tp.n_bins + bin;
            key = (s * tp.n_bins + bin) * 8u + b;
            if (M2) midx = ((size_t)s * (NBr + 1u) + b) * tp.n_bins + bin;
            if (dbg) {
                dbg[p].energy[b] = e;
                if (b == 0) { dbg[p].bin = (int32_t)bin; dbg[p].delay_s = delay; dbg[p].total_dist = total; }
            }
        }
        // broadband value of the path: its 8 lanes sum their q_b (lanes past n_bands and past the queue hold 0);
        // q_b <= clamp * gain * 2^32, so the sum fits 64 bits for clamp * gain < 2^29
        unsigned long long qs = 0ull;
        if (M2) {
            qs = q;
            qs += __shfl_xor_sync(0xffffffffu, qs, 4);
            qs += __shfl_xor_sync(0xffffffffu, qs, 2);
            qs += __shfl_xor_sync(0xffffffffu, qs, 1);
        }
        // splat: lanes with the same (source, band, bin) combine first, one RED.64 per group
        const uint32_t active = __ballot_sync(0xffffffffu, valid);
        if (valid) {
            if (tp.flags & FS_FLAG_NO_SPLAT_AGG) {
                atomicAdd(hist + hidx, q);
                if (M2) {
                    atomic_add_u128(m2 + midx, q * q, __umul64hi(q, q));
                    if (b == 0) atomic_add_u128(m2 + midx + (size_t)NBr * tp.n_bins, qs * qs, __umul64hi(qs, qs));
                }
            } else {
                const uint32_t peers = __match_any_sync(active, key);
                const bool leader = (uint32_t)(__ffs(peers) - 1) == lane;
                if (M2) {
                    unsigned long long lo = q * q, hi = __umul64hi(q, q);
                    if (peers != (1u << lane)) reduce_peers_u128(peers, lo, hi);
                    if (leader) atomic_add_u128(m2 + midx, lo, hi);
                }
                if (peers != (1u << lane)) q = reduce_peers(peers, q);
                if (leader) atomicAdd(hist + hidx, q);
                if (M2) {
                    // broadband: one lane per path (band 0), grouped by (source, bin)
                    const uint32_t bb_active = __ballot_sync(active, b == 0);
                    if (b == 0) {
                        const uint32_t bpeers = __match_any_sync(bb_active, key >> 3);
                        unsigned long long lo = qs * qs, hi = __umul64hi(qs, qs);
                        if (bpeers != (1u << lane)) reduce_peers_u128(bpeers, lo, hi);
                        if ((uint32_t)(__ffs(bpeers) - 1) == lane) atomic_add_u128(m2 + midx + (size_t)NBr * tp.n_bins, lo, hi);
                    }
                }
            }
        }
    }
}


// ---------------------------------------------------------------------------------------------
// k_eval_mis (FS_FLAG_MIS, SURVEY 8f rank 1): every visible prefix connection (s, t) contributes f / sum_{s'} p_{s'} -- the
// balance heuristic over all strategies that build a path of s + t vertices, for the physically based contribution
//     f = 1/(4 pi) * prod_edges [cos_a cos_b / d^2 * exp(-air d)] * prod_interior [rho / pi]
// with area-measure densities rr * D_a * cos_b / d^2 (D = 1/(4 pi) at the end points, cos_a / pi on surfaces).  This is what
// the reference's unfinished getPdf / getExpectedWeight / MISEnergy aim at (SUB.cpp:537-597).  8 lanes per connection (one
// band each); the geometry of the path is band independent and computed by all eight.  Same float operations in the same
// order as the CPU harness.
// ---------------------------------------------------------------------------------------------
#define FS_MIS_MAXV 66
__device__ __forceinline__ void mis_vertex(const fs_trace_params& tp, const fs_wave_buffers& wb, uint32_t sf, uint32_t sb, uint32_t s,
                                           uint32_t k, uint32_t i, uint32_t stride, fs_vec3& P, fs_vec3& N)
{
    const uint32_t sp = (i < s) ? sf : sb;
    const uint32_t node = (i < s) ? i : (k - 1u - i);
    P = node_pos(tp, wb, sp, node, stride);
    if (node == 0u) { N = fs_mk(0.f, 0.f, 0.f); return; }
    const float4 nv = wb.nnrm[(size_t)node * stride + sp];
    N = fs_mk(nv.x, nv.y, nv.z);
}

// DIR: f starts at the gain of the source's pattern at normalize(x1 - x0), the direction of the path's first edge
template <bool DIR = false>
__global__ void __launch_bounds__(WF_THREADS)
k_eval_mis(const fs_trace_params tp, const fs_wave_buffers wb, unsigned long long* __restrict__ hist, fs_dev_counters* __restrict__ dc)
{
    const uint32_t lane = lane_id();
    const uint32_t sub = lane >> 3, b = lane & 7u;
    const uint32_t qi = tp.max_depth + 1;
    const uint32_t count = wb.q_count[qi];
    const uint32_t stride = 2u * wb.cap;
    const uint32_t NBr = tp.ep.n_bands;
    const bool band_on = b < NBr;
    const float air_b = band_on ? tp.ep.air[b] : 0.0f;
    if (blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(&dc->connected, (unsigned long long)count);
    const uint32_t warp_global = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint32_t n_warps = (gridDim.x * blockDim.x) >> 5;
    float pf[FS_MIS_MAXV], pb[FS_MIS_MAXV], gg[FS_MIS_MAXV], dlen[FS_MIS_MAXV];
    for (uint32_t base = warp_global * 4u; base < count; base += n_warps * 4u) {
        const uint32_t j = base + sub;
        bool valid = (j < count) && band_on;
        unsigned long long q = 0ull;
        uint32_t key = 0xffffffffu;
        size_t hidx = 0;
        if (valid) {
            const uint32_t id = wb.all_conn[j];
            const uint32_t p = id >> 12;
            const uint32_t sf = 2u * p, sb = 2u * p + 1u;
            const uint32_t s = ((id >> 6) & 63u) + 1u, t = (id & 63u) + 1u;
            const uint32_t k = s + t;
            float total = 0.0f;
            bool ok = k <= (uint32_t)FS_MIS_MAXV;
            fs_vec3 Pa, Na, d0;
            if (ok) mis_vertex(tp, wb, sf, sb, s, k, 0u, stride, Pa, Na);
            for (uint32_t i = 0; ok && i + 1u < k; ++i) {
                fs_vec3 Pb, Nb;
                mis_vertex(tp, wb, sf, sb, s, k, i + 1u, stride, Pb, Nb);
                const fs_vec3 dl = fs_sub(Pb, Pa);
                const float d2 = fs_dot(dl, dl);
                const float d = sqrtf(d2);
                total += d;
                if (d < tp.ep.min_seg) { ok = false; break; }
                const float inv = 1.0f / d;
                const fs_vec3 dir = fs_mk(dl.x * inv, dl.y * inv, dl.z * inv);
                if (DIR && i == 0u) d0 = dir;
                const float cp = (i == 0u) ? 1.0f : fabsf(fs_dot(Na, dir));
                const float cm = (i + 2u == k) ? 1.0f : fabsf(fs_dot(Nb, dir));
                const float rd2 = 1.0f / d2;
                gg[i] = (cp * cm) * rd2;
                if (!(gg[i] > 0.0f)) { ok = false; break; }
                pf[i] = (tp.rr_prob * ((i == 0u) ? FS_INV_4PI : cp * FS_INV_PI)) * (cm * rd2);
                pb[i] = (tp.rr_prob * ((i + 2u == k) ? FS_INV_4PI : cm * FS_INV_PI)) * (cp * rd2);
                dlen[i] = d;
                Pa = Pb; Na = Nb;
            }
            if (ok) {
                const uint32_t depth = pair_depth(tp, wb, p);
                float sum = 1.0f, r = 1.0f;
                for (uint32_t sp = s; sp + 1u < k && sp <= depth; ++sp) { r = r * (pf[sp - 1u] / pb[sp]); sum += r; }
                r = 1.0f;
                for (uint32_t sp = s; sp > 1u && k - sp <= depth; --sp) { r = r * (pb[sp - 1u] / pf[sp - 2u]); sum += r; }
                float val = FS_INV_4PI;
                if (DIR) val = dir_gain(tp, pair_source(tp, wb, p), b, d0.x, d0.y, d0.z) * FS_INV_4PI;
                for (uint32_t i = 0; i + 1u < k; ++i) {
                    val = val * gg[i];
                    val = val * fs_exp(-air_b * dlen[i]);
                    const uint32_t jv = i + 1u;
                    if (jv + 1u < k) {
                        const uint32_t sp = (jv < s) ? sf : sb;
                        const uint32_t node = (jv < s) ? jv : (k - 1u - jv);
                        const uint32_t mw = __float_as_uint(wb.rec[(size_t)node * stride + sp].y) & 0x00ffffffu;
                        val = val * __ldg(tp.refl_over_pi + (size_t)mw * NBr + b);
                        val = val / ((jv < s) ? pf[jv - 1u] : pb[jv]);
                    }
                }
                float e = val / sum;
                const float delay = total / tp.sound_speed;
                const float fb = floorf((delay * 1000.0f) / tp.bin_ms);
                uint32_t bin;
                if (!(fb >= 0.0f)) bin = 0;
                else if (fb >= (float)(tp.n_bins - 1)) bin = tp.n_bins - 1;
                else bin = (uint32_t)fb;
                const uint32_t src = pair_source(tp, wb, p);
                e = (e < tp.energy_clamp) ? e : tp.energy_clamp;
                e = e * tp.energy_gain;
                q = (unsigned long long)(e * 4294967296.0f);
                hidx = ((size_t)src * NBr + b) * tp.n_bins + bin;
                key = (src * tp.n_bins + bin) * 8u + b;
            } else valid = false;
        }
        const uint32_t active = __ballot_sync(0xffffffffu, valid);
        if (valid) {
            const uint32_t peers = __match_any_sync(active, key);
            if (peers != (1u << lane)) q = reduce_peers(peers, q);
            if ((uint32_t)(__ffs(peers) - 1) == lane) atomicAdd(hist + hidx, q);
        }
    }
}

// =============================================================================================
// Split wavefront (default path): shading/generation kernels with every lane busy, and PURE
// traversal kernels with per-lane ray replacement.
//
// ncu on the fused k_extend showed smsp__thread_inst_executed_per_inst_executed = 7.5..8.9 of 32
// (profiles/r1a_ncu_k_extend_summary.txt): lanes whose ray ended early idle until the slowest
// lane of the warp finishes, and lanes at a leaf idle while others walk inner nodes.  Here
//   k_shade_gen(k)    consumes the hits of bounce k-1 (node record, offset, termination) and
//                     generates the rays of bounce k (Philox, Russian roulette, sampling) into a
//                     ballot-compacted ray queue: coherent, all 32 lanes busy;
//   k_trace_closest   persistent warps; a lane that retires its ray immediately pulls the next
//                     one from the queue (one atomicAdd per warp refill), so a warp always walks
//                     ~32 rays; "while-while" traversal with one postponed leaf per lane
//                     (speculative traversal) and one triangle test per lane per leaf-phase step;
//   k_connect_gen / k_trace_any  the same for the connection (shadow) rays.
// Ray record (32 B): (origin.xyz, sp_id | tmax) (dir.xyz, pdf | path id); hit record 8 B (t, tri).
// =============================================================================================
#ifndef FS_TR_THREADS
#define FS_TR_THREADS 256
#endif
constexpr int TR_THREADS = FS_TR_THREADS;
#ifndef FS_TR_MINBLOCKS
#define FS_TR_MINBLOCKS (1280 / FS_TR_THREADS)      // <= 51 registers: 1280 threads (40 warps) per SM
#endif
// refill a warp once this many lanes are idle (kernel argument, default FS_REFILL_DEFAULT)
#define FS_REFILL_DEFAULT 8u
constexpr uint32_t FULLM = 0xffffffffu;
#define TR_SENT 0x7fffffff

__device__ __forceinline__ void leaf_range(int leafnode, uint32_t& tc, uint32_t& te)
{
    const uint32_t payload = (uint32_t)(~leafnode);
    tc = payload >> 3;
    te = tc + (payload & 7u) + 1u;
}

// Russian roulette + direction of bounce k of subpath (g, side) at a node with normal nrm reached along d_in (GeneratePath,
// SUB.cpp:301-318).  Returns false when the walk ends here.  ev = the lobe taken (FS_EV_*), org = origin of the new ray.
// Without FS_FLAG_MATERIAL_MODEL every surface event is the cosine lobe (ev = 0, org = pos) -- the reference's model.
// With it (SURVEY 8f rank 3) the fourth word of the bounce's Philox block picks pass-through / mirror / cosine lobe by the
// per-material thresholds of tp.lobes (built in fs_scene_commit; the CPU harness restates the same arithmetic).
#define FS_EV_DIFFUSE 0u
#define FS_EV_SPECULAR 1u
#define FS_EV_TRANSMIT 2u
__device__ __forceinline__ bool choose_direction(const fs_trace_params& tp, uint32_t k, uint64_t g, uint32_t side, fs_vec3 nrm,
                                                 fs_vec3 d_in, uint32_t mat, fs_vec3 pos, fs_vec3& dir, float& prob, uint32_t& ev,
                                                 fs_vec3& org)
{
    uint32_t r[4];
    fs_philox4x32_10((uint32_t)g, (uint32_t)(g >> 32), k, side, tp.seed_lo, tp.seed_hi, r);
    const float u0 = fs_u01(r[0]), u1 = fs_u01(r[1]), u2 = fs_u01(r[2]);
    ev = FS_EV_DIFFUSE; org = pos;
    if (!(u0 < tp.rr_prob)) return false;                   // SUB.cpp:301-302
    if (k == 0) { dir = fs_sample_sphere(u1, u2); prob = FS_INV_4PI * tp.rr_prob; return true; }     // SUB.cpp:306-311
    if (tp.lobes) {
        const float4 lb = __ldg(tp.lobes + mat);            // (t1, t2, P_spec, P_diff)
        const float u3 = fs_u01(r[3]);
        if (u3 < lb.x) {                                    // pass through (COMP.cpp:271-275): continue from the far side
            ev = FS_EV_TRANSMIT; dir = d_in; prob = tp.rr_prob * lb.x;
            const float e2 = -2.0f * tp.eps_offset;
            org = fs_mk(fmaf(e2, nrm.x, pos.x), fmaf(e2, nrm.y, pos.y), fmaf(e2, nrm.z, pos.z));
            return true;
        }
        if (u3 < lb.y) {                                    // mirror (GetReflectionVector, COMP.cpp:186)
            ev = FS_EV_SPECULAR;
            const float sdn = -2.0f * fs_dot(d_in, nrm);
            dir = fs_mk(fmaf(sdn, nrm.x, d_in.x), fmaf(sdn, nrm.y, d_in.y), fmaf(sdn, nrm.z, d_in.z));
            prob = tp.rr_prob * lb.z;
            return true;
        }
        float ct; dir = fs_sample_cos_hemisphere(nrm, u1, u2, ct);
        prob = ((ct * FS_INV_PI) * tp.rr_prob) * lb.w;
        return true;
    }
    float ct; dir = fs_sample_cos_hemisphere(nrm, u1, u2, ct);      // SUB.cpp:312-318 (FIX: true cosine lobe)
    prob = (ct * FS_INV_PI) * tp.rr_prob;
    return true;
}

#ifndef FS_SG_THREADS
#define FS_SG_THREADS 256
#endif
#ifndef FS_SHADE_MINBLOCKS
#define FS_SHADE_MINBLOCKS (1536 / FS_SG_THREADS)
#endif
__global__ void __launch_bounds__(FS_SG_THREADS, FS_SHADE_MINBLOCKS)
k_shade_gen(const fs_trace_params tp, const fs_wave_buffers wb, uint32_t k, fs_dev_counters* __restrict__ dc)
{
    const uint32_t lane = lane_id();
    const uint32_t count_in = (k == 0) ? 2u * tp.batch : wb.q_count[k - 1];
    const int in = (int)((k + 1u) & 1u), out = (int)(k & 1u);
    const float4* __restrict__ in_o = wb.st_pos[in];
    const float4* __restrict__ in_d = wb.st_nrm[in];
    float4* __restrict__ out_o = wb.st_pos[out];
    float4* __restrict__ out_d = wb.st_nrm[out];
    const uint32_t stride = 2u * wb.cap;             // rec[k][sp_id]: one plane per node index (writes of a bounce stay semi-coalesced)
    // One queue-slot atomic per CTA tile, not per warp: ncu (r1i) had 43 % of this kernel's stall samples on the return
    // of the per-warp atomicAdd -- 10^5 same-address atomics per launch run at about one per nanosecond.
    __shared__ uint32_t s_cnt[FS_SG_THREADS / 32], s_base;
    const uint32_t warp = threadIdx.x >> 5;
    for (uint32_t tile = blockIdx.x * blockDim.x; tile < count_in; tile += gridDim.x * blockDim.x) {
        const uint32_t j = tile + threadIdx.x;
        bool emit = false;
        fs_vec3 pos = fs_mk(0.f, 0.f, 0.f), dir = fs_mk(0.f, 0.f, 0.f);
        uint32_t sp_id = 0; float prob = 1.0f;
        if (j < count_in) {
            fs_vec3 nrm = fs_mk(0.f, 0.f, 0.f), din = fs_mk(0.f, 0.f, 0.f);
            bool cont = true, hit = false;
            uint32_t nodes = 1, mat = 0;
            float seg = 0.f, pdf_in = 1.f;
            if (k == 0) {                         // node 0 (SUB.cpp:287-291)
                sp_id = j;
                if (tp.lis_mode && (sp_id & 1u) == tp.lis_mode - 1u) cont = false;   // shared listener: this side is not traced in this pass
                if (sp_id & 1u) pos = fs_mk(tp.lis[0], tp.lis[1], tp.lis[2]);
                else pos = source_pos(tp, pair_source(tp, wb, sp_id >> 1));
                if (tp.src_off && wb.pair_src[sp_id >> 1].y == 0u) cont = false;   // a depth-0 source among deeper ones: node 0 only
            } else {
                const float4 a = FS_LD4(in_o + j), b = FS_LD4(in_d + j);
                const float2 h = FS_LD2(wb.hit + j);
                sp_id = __float_as_uint(a.w);
                const fs_vec3 o = fs_mk(a.x, a.y, a.z), d = fs_mk(b.x, b.y, b.z);
                const int tri = __float_as_int(h.y);
                if (tri < 0) {                    // miss: FIX -> the subpath ends at the node the ray left
                    if (!tp.lobes) wb.end_pos[sp_id] = make_float4(o.x, o.y, o.z, __uint_as_float(k));
                    else if (k >= 2u) {
                        // material model: end_pos already holds that node (written when the ray was emitted: after a
                        // pass-through the ray origin is not the node); as an end node it connects through its diffuse lobe
                        float4* rp = wb.rec + (size_t)(k - 1u) * stride + sp_id;
                        float4 rv = *rp;
                        rv.y = __uint_as_float(__float_as_uint(rv.y) & 0x00ffffffu);
                        *rp = rv;
                    }
                    cont = false;
                } else {                          // SUB.cpp:343-348
                    const float t = h.x;
                    const float4 nm = fs_ldg4(tp.bv.tri_nm + tri);
                    fs_vec3 fn = fs_mk(nm.x, nm.y, nm.z);
                    if (fs_dot(fn, d) > 0.0f) { fn.x = -fn.x; fn.y = -fn.y; fn.z = -fn.z; }
                    pos.x = fmaf(tp.eps_offset, fn.x, fmaf(t, d.x, o.x));
                    pos.y = fmaf(tp.eps_offset, fn.y, fmaf(t, d.y, o.y));
                    pos.z = fmaf(tp.eps_offset, fn.z, fmaf(t, d.z, o.z));
                    const fs_vec3 dl = fs_sub(pos, o);
                    seg = sqrtf(fs_dot(dl, dl));
                    mat = __float_as_uint(nm.w);
                    pdf_in = b.w;
                    if (wb.npos) wb.npos[(size_t)k * stride + sp_id] = make_float4(pos.x, pos.y, pos.z, 0.0f);
                    if (wb.nnrm) wb.nnrm[(size_t)k * stride + sp_id] = make_float4(fn.x, fn.y, fn.z, 0.0f);
                    nrm = fn; din = d;
                    nodes = k + 1;
                    hit = true;
                    if (k >= pair_depth(tp, wb, sp_id >> 1)) cont = false;      // PARAM: ray budget per subpath exhausted
                }
            }
            uint32_t ev = FS_EV_DIFFUSE;
            fs_vec3 org = pos;
            if (cont) {
                uint64_t g = tp.g_first + (sp_id >> 1);
                if ((tp.flags & FS_FLAG_SHARE_LISTENER) && (sp_id & 1u)) g = listener_key(tp, wb, sp_id >> 1);   // keyed by the path index only
                emit = choose_direction(tp, k, g, sp_id & 1u, nrm, din, mat, pos, dir, prob, ev, org);
            }
            // node record of node k: the lobe the walk takes here rides in the top byte of the material word
            if (hit) FS_ST4(wb.rec + (size_t)k * stride + sp_id, make_float4(seg, __uint_as_float(mat | (ev << 24)), pdf_in, fs_pow(pdf_in, tp.ep.pdf_exponent)));
            // the walk ends at this node -- or, with the material model, may end here if the ray just emitted misses
            const bool at_node = (k == 0) ? !(tp.lis_mode && (sp_id & 1u) == tp.lis_mode - 1u) : hit;
            if (at_node && (!emit || tp.lobes)) FS_ST4(wb.end_pos + sp_id, make_float4(pos.x, pos.y, pos.z, __uint_as_float(nodes)));
            pos = org;                            // the ray starts at the node, or beyond its surface after a pass-through
        }
        const uint32_t m = __ballot_sync(FULLM, emit);
        if (lane == 0) s_cnt[warp] = (uint32_t)__popc(m);
        __syncthreads();
        if (threadIdx.x == 0) {
            uint32_t tot = 0;
#pragma unroll
            for (int w = 0; w < FS_SG_THREADS / 32; ++w) { const uint32_t c = s_cnt[w]; s_cnt[w] = tot; tot += c; }
            s_base = tot ? atomicAdd(&wb.q_count[k], tot) : 0u;      // ext_rays = sum of the queue lengths (k_connect_gen)
        }
        __syncthreads();
        if (emit) {
            const uint32_t o = s_base + s_cnt[warp] + __popc(m & ((1u << lane) - 1u));
            FS_ST4(out_o + o, make_float4(pos.x, pos.y, pos.z, __uint_as_float(sp_id)));
            FS_ST4(out_d + o, make_float4(dir.x, dir.y, dir.z, prob));
        }
        __syncthreads();                                   // s_cnt / s_base are rewritten by the next tile
    }
    (void)dc;
}

// per-lane traversal state shared by the two trace kernels
struct tr_state {
    fs_vec3 o, d;
    // BVH2 float nodes: (idir, o * idir).  4-wide quantised nodes: (s, b') with t(q) = fma(2^23 + q, s, b')
    float idx, idy, idz, oodx, oody, oodz;
    int node, leaf, sp;
    uint32_t tc, te;
    uint32_t oct;        // 8-wide nodes: bit a set = direction component a is >= 0 (near plane = low plane)
};

__device__ __forceinline__ float fs_rcp_fast(float x)
{
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}

template <bool WIDE>
__device__ __forceinline__ void tr_init(tr_state& s, const fs_bvh_view& bv, fs_vec3 o, fs_vec3 d)
{
    s.o = o; s.d = d;
    if (WIDE) {
        // 1 / d by MUFU.RCP (<= 1 ulp): the box test only has to be conservative, and a 2^-23 relative error of t is far
        // inside the spare quantum of the outward rounding (an IEEE division costs ~15 instructions per axis and ray)
        const float dx = (fabsf(d.x) > 1e-30f) ? d.x : ((d.x < 0.0f) ? -1e-30f : 1e-30f);
        const float dy = (fabsf(d.y) > 1e-30f) ? d.y : ((d.y < 0.0f) ? -1e-30f : 1e-30f);
        const float dz = (fabsf(d.z) > 1e-30f) ? d.z : ((d.z < 0.0f) ? -1e-30f : 1e-30f);
        const float ix = fs_rcp_fast(dx), iy = fs_rcp_fast(dy), iz = fs_rcp_fast(dz);
        s.idx = bv.qscale[0] * ix; s.idy = bv.qscale[1] * iy; s.idz = bv.qscale[2] * iz;
        // b' = (qbase - o) * idir - 2^23 * s: its rounding error is below half a quantum, which the spare quantum of
        // outward rounding at build time covers
        s.oodx = fmaf(-8388608.0f, s.idx, (bv.qbase[0] - o.x) * ix);
        s.oody = fmaf(-8388608.0f, s.idy, (bv.qbase[1] - o.y) * iy);
        s.oodz = fmaf(-8388608.0f, s.idz, (bv.qbase[2] - o.z) * iz);
    } else {
        const fs_ray_prep r = fs_prep_ray(o, d);
        s.idx = r.idx; s.idy = r.idy; s.idz = r.idz; s.oodx = r.oodx; s.oody = r.oody; s.oodz = r.oodz;
    }
    s.node = bv.n_tris ? 0 : TR_SENT; s.leaf = 0; s.sp = 0; s.tc = 0; s.te = 0;
}

// 2^23 + (16 bits of w chosen by the PRMT selector) as a float.  0x7410 = low half, 0x7432 = high half
__device__ __forceinline__ float q_sel(uint32_t w, uint32_t sel) { return __uint_as_float(__byte_perm(w, 0x4B000000u, sel)); }
__device__ __forceinline__ uint4 ldg_u4(const uint4* p)
{
    uint4 r;
    asm volatile("ld.global.nc.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return r;
}

// Traversal stack: the first FS_SSTACK entries of every thread live in shared memory (column
// layout [depth][thread]: bank-conflict free, ~30-cycle latency), deeper entries in local memory.
// ncu showed 12 % of the kernel's stall samples on the instruction consuming a local-memory pop
// (37 % of those loads missed L1, and the 256 B/thread stacks competed with BVH nodes for L1).
//
// DIST = true (closest-hit rays): an entry is (node, entry distance of its box).  A pop skips every
// entry whose box is entered beyond the current best hit (boxes are conservative, ties t == best are
// kept), so a subtree that became irrelevant after it was pushed costs one LDS instead of a 64 B node
// fetch + four slab tests that all miss.  ncu (r1h): 30 % of the node steps hit no child at all.
#ifndef FS_SSTACK
#define FS_SSTACK 12
#endif
template <bool DIST> struct tr_entry_t { typedef int type; };
template <> struct tr_entry_t<true> { typedef uint2 type; };
#ifndef FS_ANY_ORDERED
#define FS_ANY_ORDERED 0     // connection rays: visit the hit children near-to-far (1) or in slot order (0)
#endif
#ifndef FS_STACK_DIST
#define FS_STACK_DIST 0      // measured (r1i): culling removes only 2 % of the node visits, 8 B entries cost more than that
#endif
#define TR_SMEM_CLOSEST (FS_SSTACK * TR_THREADS * sizeof(tr_entry_t<FS_STACK_DIST != 0>::type))
#define TR_SMEM_ANY (FS_SSTACK * TR_THREADS * sizeof(int))
template <bool DIST>
struct tr_stack {
    typedef typename tr_entry_t<DIST>::type entry;
    entry* sh;        // &smem[threadIdx.x], stride blockDim.x
    entry* loc;       // per-thread local array for entries >= FS_SSTACK
    static __device__ __forceinline__ uint2 mk(int v, float d, uint2*) { return make_uint2((uint32_t)v, __float_as_uint(d)); }
    static __device__ __forceinline__ int mk(int v, float, int*) { return v; }
    static __device__ __forceinline__ int node_of(uint2 e) { return (int)e.x; }
    static __device__ __forceinline__ int node_of(int e) { return e; }
    static __device__ __forceinline__ bool live(uint2 e, float tbest) { return __uint_as_float(e.y) <= tbest; }
    static __device__ __forceinline__ bool live(int, float) { return true; }
    __device__ __forceinline__ void push(int& sp, int v, float d) const
    {
        const entry e = mk(v, d, (entry*)nullptr);
        if (sp < FS_SSTACK) sh[sp * TR_THREADS] = e; else loc[sp - FS_SSTACK] = e;
        ++sp;
    }
    // up to three entries at once, farthest first (e3, e2, e1; h3 implies h2 implies h1 = true)
    __device__ __forceinline__ void push3(int& sp, bool h2, bool h3, int v1, float d1, int v2, float d2, int v3, float d3,
                                          uint32_t* overflow) const
    {
        const int n = 1 + (int)h2 + (int)h3;
        if (sp + 3 <= FS_SSTACK) {                    // common case: straight-line predicated shared stores
            entry* q = sh + sp * TR_THREADS;
            if (h3) q[0] = mk(v3, d3, (entry*)nullptr);
            if (h2) q[h3 ? TR_THREADS : 0] = mk(v2, d2, (entry*)nullptr);
            q[(n - 1) * TR_THREADS] = mk(v1, d1, (entry*)nullptr);
            sp += n;
        } else if (sp + 3 <= FS_STACK_SIZE) {
            if (h3) push(sp, v3, d3);
            if (h2) push(sp, v2, d2);
            push(sp, v1, d1);
        } else *overflow = 1u;
    }
    // next entry that can still hold a hit not beyond tbest; TR_SENT when the stack is empty
    __device__ __forceinline__ int pop(int& sp, float tbest) const
    {
        while (sp > 0) {
            --sp;
            const entry e = (sp < FS_SSTACK) ? sh[sp * TR_THREADS] : loc[sp - FS_SSTACK];
            if (live(e, tbest)) return node_of(e);
        }
        return TR_SENT;
    }
};

// After a sorted 4-wide step (k0 <= k1 <= k2 <= k3, INF = no inner hit): push the 2nd..4th hit (farthest first), move on to the
// nearest, or pop when nothing was entered.  The three cases used to be three divergent blocks (push with 6.6 of 32 lanes in
// nine of ten warp steps, pop with 8.6, profiles/r2p_*): while the whole operation stays inside the shared-memory part of the
// stack it can be ONE predicated straight-line sequence for all lanes (FS_MERGED_ADVANCE=1).  Measured: ptxas turns it into 38
// instructions at full width against 24 + 9 in the divergent blocks, 24 B of spills in k_trace_q: room per-bounce 5.07 -> 5.18 ms,
// persistent kernel unchanged -- the branchy form (0) stays.
#ifndef FS_MERGED_ADVANCE
#define FS_MERGED_ADVANCE 0
#endif
__device__ __forceinline__ void w4_advance(tr_state& s, const tr_stack<false>& stack, float k0, float k1, float k2, float k3,
                                           int v0, int v1, int v2, int v3, uint32_t* overflow)
{
    const float INF = __int_as_float(0x7f800000);
    const bool h0 = k0 != INF, h1 = k1 != INF, h2 = k2 != INF, h3 = k3 != INF;
    if (FS_MERGED_ADVANCE && s.sp + 3 <= FS_SSTACK) {
        int* q = stack.sh + s.sp * TR_THREADS;
        int top = TR_SENT;
        if (!h0 && s.sp > 0) top = q[-TR_THREADS];
        if (h3) q[0] = v3;
        if (h2) q[h3 ? TR_THREADS : 0] = v2;
        if (h1) q[((int)h3 + (int)h2) * TR_THREADS] = v1;
        s.node = h0 ? v0 : top;
        s.sp += h0 ? ((int)h1 + (int)h2 + (int)h3) : (s.sp > 0 ? -1 : 0);
    } else {
        if (h1) stack.push3(s.sp, h2, h3, v1, k1, v2, k2, v3, k3, overflow);
        s.node = h0 ? v0 : stack.pop(s.sp, 0.f);
    }
}

// Speculative traversal (Aila & Laine): the first leaf a lane reaches is POSTPONED and the lane
// keeps walking; a second leaf makes it wait (node stays < 0) for the warp's triangle phase.
#define TR_POP (-0x7fffffff - 1)        // "take the next node from the stack" marker (never a valid leaf code)
template <bool DIST>
__device__ __forceinline__ void tr_advance(tr_state& s, const tr_stack<DIST>& stack, int cand, float tbest)
{
    for (;;) {
        if (cand == TR_POP) cand = stack.pop(s.sp, tbest);
        if (cand < 0 && s.leaf == 0) { s.leaf = cand; cand = TR_POP; continue; }   // one postponed leaf
        break;
    }
    s.node = cand;
}

template <bool ORDERED, int TEX, bool DIST>
__device__ __forceinline__ void tr_node_step(const fs_bvh_view& bv, tr_state& s, const tr_stack<DIST>& stack, float tlimit,
                                             uint32_t* overflow)
{
    const float4* p = bv.nodes + (size_t)s.node * 4;
    float4 n0, n1, n2, n3;
    if (TEX >= 2) {
        // The traversal is bound by the L1TEX LSU data pipe (one wavefront per lane per divergent
        // 16 B load).  Two of the four quarters of a node go through the texture data pipe instead,
        // which ncu/CUDA-event A/B measured ~8 % faster than four LSU loads; all four through TEX
        // is slower.
        const int b = s.node * 4;
        n0 = tex1Dfetch<float4>((cudaTextureObject_t)bv.nodes_tex, b);
        n1 = tex1Dfetch<float4>((cudaTextureObject_t)bv.nodes_tex, b + 1);
        n2 = fs_ldg4(p + 2); n3 = fs_ldg4(p + 3);
    } else {
        n0 = fs_ldg4(p); n1 = fs_ldg4(p + 1); n2 = fs_ldg4(p + 2); n3 = fs_ldg4(p + 3);
    }
    fs_ray_prep r;
    r.idx = s.idx; r.idy = s.idy; r.idz = s.idz; r.oodx = s.oodx; r.oody = s.oody; r.oodz = s.oodz;
    bool h0, h1; float t0, t1;
    fs_slab2(r, n0, n1, n2, tlimit, h0, h1, t0, t1);
    const int c0 = __float_as_int(n3.x), c1 = __float_as_int(n3.y);
    int cand = TR_POP;
    if (h0 || h1) {
        cand = h0 ? c0 : c1;
        if (h0 && h1) {
            int far_ = c1; float tfar = t1;
            if (ORDERED && t1 < t0) { far_ = c0; tfar = t0; cand = c1; }
            if (s.sp < FS_STACK_SIZE) stack.push(s.sp, far_, tfar); else *overflow = 1u;
        }
    }
    tr_advance(s, stack, cand, tlimit);
}


#define FS_CSWAP(ka, va, kb, vb) { const bool sw_ = kb < ka; const float tk_ = sw_ ? kb : ka; kb = sw_ ? ka : kb; ka = tk_; \
                                   const int tv_ = sw_ ? vb : va; vb = sw_ ? va : vb; va = tv_; }

// the four children of a 4-wide quantised node against the ray: near/far planes picked by the ray octant,
// entry distances k (INF = miss) and references v; ORDER 1: sorted near-to-far, 0: hits moved to the front, 2: slot order
template <int ORDER, int TEX>
__device__ __forceinline__ void wide_children(const fs_bvh_view& bv, const tr_state& s, float tlimit,
                                              float& k0, float& k1, float& k2, float& k3, int& v0, int& v1, int& v2, int& v3,
                                              const uint4* top = nullptr, int n_top = 0)
{
    const uint4* p = bv.wnodes + (size_t)s.node * 4;
    uint4 u0, u1, u2, u3;
    if (n_top && s.node < n_top) {       // FS_PQ_TOP: the top of the (breadth-first) node array staged in shared memory
        const uint4* q = top + s.node * 4;
        u0 = q[0]; u1 = q[1]; u2 = q[2]; u3 = q[3];
    } else if (TEX >= 2) {                      // two quarters through the texture data pipe, two through LSU
        const int b = s.node * 4;
        u0 = tex1Dfetch<uint4>((cudaTextureObject_t)bv.wnodes_tex, b);
        u1 = tex1Dfetch<uint4>((cudaTextureObject_t)bv.wnodes_tex, b + 1);
        u2 = ldg_u4(p + 2); u3 = ldg_u4(p + 3);
    } else {
        u0 = ldg_u4(p); u1 = ldg_u4(p + 1); u2 = ldg_u4(p + 2); u3 = ldg_u4(p + 3);
    }
    // ray octant (sign of s = sign of the direction): with a negative direction the HIGH plane is entered first
    const uint32_t nx = (s.idx < 0.0f) ? 0x7432u : 0x7410u, ny = (s.idy < 0.0f) ? 0x7432u : 0x7410u,
                   nz = (s.idz < 0.0f) ? 0x7432u : 0x7410u;
    const uint32_t fx = nx ^ 0x0022u, fy = ny ^ 0x0022u, fz = nz ^ 0x0022u;
    const float INF = __int_as_float(0x7f800000);
#define FS_CHILD(u, key, val)                                                                                         \
    {                                                                                                                 \
        const float tn = fmaxf(fmaxf(fmaxf(fmaf(q_sel(u.x, nx), s.idx, s.oodx), fmaf(q_sel(u.y, ny), s.idy, s.oody)), \
                                     fmaf(q_sel(u.z, nz), s.idz, s.oodz)), 0.0f);                                     \
        const float tf = fminf(fminf(fminf(fmaf(q_sel(u.x, fx), s.idx, s.oodx), fmaf(q_sel(u.y, fy), s.idy, s.oody)), \
                                     fmaf(q_sel(u.z, fz), s.idz, s.oodz)), tlimit);                                   \
        key = (tn <= tf) ? tn : INF;                                                                                  \
        val = (int)u.w;                                                                                               \
    }
    FS_CHILD(u0, k0, v0) FS_CHILD(u1, k1, v1) FS_CHILD(u2, k2, v2) FS_CHILD(u3, k3, v3)
#undef FS_CHILD
    if (ORDER == 1) {
        // 5-comparator network; misses (INF) sink to the end
        FS_CSWAP(k0, v0, k1, v1) FS_CSWAP(k2, v2, k3, v3) FS_CSWAP(k0, v0, k2, v2) FS_CSWAP(k1, v1, k3, v3) FS_CSWAP(k1, v1, k2, v2)
    } else if (ORDER == 0) {             // any-hit rays: only move the hits to the front
        if (k0 == INF) { k0 = k1; v0 = v1; k1 = INF; }
        if (k0 == INF) { k0 = k2; v0 = v2; k2 = INF; }
        if (k0 == INF) { k0 = k3; v0 = v3; k3 = INF; }
    }
}

// one step through a 4-wide node: test, push the farther hits, move on to the nearest (or pop)
template <bool ORDERED, int TEX, bool DIST>
__device__ __forceinline__ void tr_node_step4(const fs_bvh_view& bv, tr_state& s, const tr_stack<DIST>& stack, float tlimit,
                                              uint32_t* overflow)
{
    const float INF = __int_as_float(0x7f800000);
    float k0, k1, k2, k3; int v0, v1, v2, v3;
    wide_children<ORDERED ? 1 : 0, TEX>(bv, s, tlimit, k0, k1, k2, k3, v0, v1, v2, v3);
    if (ORDERED) {
        // hits are a prefix of the sorted order: push the 2nd..4th (farthest first, so the nearest is popped first)
        if (k1 != INF) stack.push3(s.sp, k2 != INF, k3 != INF, v1, k1, v2, k2, v3, k3, overflow);
    } else if (k0 != INF) {
        if (s.sp + 3 <= FS_STACK_SIZE) {
            if (k3 != INF) stack.push(s.sp, v3, k3);
            if (k2 != INF) stack.push(s.sp, v2, k2);
            if (k1 != INF) stack.push(s.sp, v1, k1);
        } else *overflow = 1u;
    }
    tr_advance(s, stack, (k0 != INF) ? v0 : TR_POP, tlimit);
}

// after a triangle step that exhausted the open range: open the postponed leaf, then re-settle
template <bool DIST>
__device__ __forceinline__ void tr_next_leaf(tr_state& s, const tr_stack<DIST>& stack, float tbest)
{
    if (s.tc == s.te) {
        if (s.leaf != 0) {
            leaf_range(s.leaf, s.tc, s.te); s.leaf = 0;
            if (s.node < 0) tr_advance(s, stack, s.node, tbest);      // a waiting second leaf becomes the postponed one
        }
    }
}

template <bool COUNT, int TEX, bool WIDE>
__global__ void __launch_bounds__(TR_THREADS, FS_TR_MINBLOCKS)
k_trace_closest(const fs_bvh_view bv, const float4* __restrict__ ray_o, const float4* __restrict__ ray_d,
                const uint32_t* __restrict__ count_ptr, uint32_t* __restrict__ cursor,
                float2* __restrict__ hits, fs_dev_counters* __restrict__ dc, const uint32_t REFILL_MIN,
                const uint32_t NODE_MIN, const uint32_t TRI_MIN)
{
    const uint32_t lane = lane_id();
    const uint32_t count = *count_ptr;
    typedef tr_stack<FS_STACK_DIST != 0> stack_t;
    extern __shared__ __align__(8) unsigned char smem_raw[];
    stack_t::entry lstack[FS_STACK_SIZE - FS_SSTACK];
    stack_t stack; stack.sh = reinterpret_cast<stack_t::entry*>(smem_raw) + threadIdx.x; stack.loc = lstack;
    tr_state s;
    s.node = TR_SENT; s.leaf = 0; s.sp = 0; s.tc = 0; s.te = 0;
    s.o = fs_mk(0.f, 0.f, 0.f); s.d = s.o; s.idx = s.idy = s.idz = s.oodx = s.oody = s.oodz = 0.f;
    bool running = false, exhausted = false;
    uint32_t j = 0, guard = 0;
    uint32_t* const ovf_p = &dc->overflow;       // rare: written straight to global memory, no register carried
    float bt = 0.f; int best = -1;
    fs_visit_counters vc; vc.nodes = 0; vc.tris = 0;
    for (;;) {
        // ---- refill idle lanes from the ray queue: one atomic per warp
        const uint32_t m_idle = __ballot_sync(FULLM, !running);
        if (!exhausted && ((uint32_t)__popc(m_idle) >= REFILL_MIN)) {
            const uint32_t n = (uint32_t)__popc(m_idle);
            uint32_t base = 0;
            if (lane == 0) base = atomicAdd(cursor, n);
            base = __shfl_sync(FULLM, base, 0);
            if (base + n >= count) exhausted = true;
            if (!running) {
                const uint32_t jj = base + (uint32_t)__popc(m_idle & ((1u << lane) - 1u));
                if (jj < count) {
                    const float4 a = ray_o[jj], b = ray_d[jj];
                    tr_init<WIDE>(s, bv, fs_mk(a.x, a.y, a.z), fs_mk(b.x, b.y, b.z));
                    bt = __int_as_float(0x7f800000); best = -1;
                    j = jj; running = true;
                }
            }
        }
        if (!__any_sync(FULLM, running)) break;
        // ---- walk until enough lanes have retired their ray ("while-while" with postponed leaves)
        for (;;) {
#if defined(FS_TRAVERSAL_GUARD)
            if (++guard > (1u << 22)) { *ovf_p = 2u; running = false; exhausted = true; break; }   // bring-up guard
#endif
            // inner nodes, until every lane that can still walk has triangle work pending
            for (;;) {
                const bool can = running && s.node >= 0 && s.node != TR_SENT;
                const uint32_t m_can = __ballot_sync(FULLM, can), m_leaf = __ballot_sync(FULLM, s.leaf != 0);
                if ((m_can & ~m_leaf) == 0u) break;
                // leave early for the triangle phase once too few lanes still walk and triangle work is waiting
                if (NODE_MIN && (uint32_t)__popc(m_can) < NODE_MIN && m_leaf != 0u) break;
                if (can) {
                    if (COUNT) vc.nodes++;
                    if (WIDE) tr_node_step4<true, TEX>(bv, s, stack, bt, ovf_p);
                    else tr_node_step<true, TEX>(bv, s, stack, bt, ovf_p);
                }
            }
            // triangles: one test per lane per step until every pending leaf of the warp is done
            tr_next_leaf(s, stack, bt);
            for (uint32_t it = 0;; ++it) {
                const bool has = s.tc < s.te;
                const uint32_t m_has = __ballot_sync(FULLM, has);
                if (m_has == 0u) break;
                // after at least one step: go back to walking once few lanes have triangles left and others can walk
                if (TRI_MIN && it && (uint32_t)__popc(m_has) < TRI_MIN &&
                    __any_sync(FULLM, running && s.node >= 0 && s.node != TR_SENT && s.leaf == 0)) break;
                if (has) {
                    const float4* tq = bv.tris + (size_t)s.tc * 4;
                    const float4 a = fs_ldg4(tq), b = fs_ldg4(tq + 1), c = fs_ldg4(tq + 2);
                    if (COUNT) vc.tris++;
                    float t;
                    if (fs_intersect_tri(s.o, s.d, fs_mk(a.x, a.y, a.z), fs_mk(b.x, b.y, b.z), fs_mk(c.x, c.y, c.z), t) && t <= bt) {
                        // tie: lower ORIGINAL triangle id wins (rare: ids are fetched only then)
                        if (t < bt || __float_as_uint(fs_ldg4(tq + 3).x) < __float_as_uint(fs_ldg4(bv.tris + (size_t)best * 4 + 3).x)) {
                            bt = t; best = (int)s.tc;
                        }
                    }
                    ++s.tc;
                    tr_next_leaf(s, stack, bt);
                }
            }
            // retire finished rays (8 B hit record), then decide whether to refill
            if (running && s.node == TR_SENT && s.leaf == 0 && s.tc == s.te) {
                hits[j] = make_float2(bt, __int_as_float(best));
                running = false;
            }
            const uint32_t m_run = __ballot_sync(FULLM, running);
            if (m_run == 0u) break;
            if (!exhausted && 32u - (uint32_t)__popc(m_run) >= REFILL_MIN) break;
        }
    }
    (void)guard;
    if (COUNT) flush_counters(dc, vc);
}


// =============================================================================================
// 8-wide compressed nodes (fs_bvh.cuh: w8nodes).  One step = one 80 B node: eight child boxes against the ray
// (near / far byte planes picked per axis by the ray octant, one PRMT + one FMA per plane), a hit mask instead of
// entry distances, no sorting network: the children sit in their slots by direction, the hit slots are visited in the
// order of (slot XOR octant).  The stack holds GROUPS -- (first child node, hits << 8 | inner mask), at most one entry per
// tree level -- so a step pushes one 8-byte entry instead of up to three, and an 8-wide tree is half as deep.
// =============================================================================================
#ifndef FS_W8_SSTACK
#define FS_W8_SSTACK 6                 // group-stack entries per thread in shared memory (8 B each); deeper ones in local memory
#endif
#define FS_W8_STACK_SIZE 40
struct w8_stack {
    uint2* sh;        // &smem[threadIdx.x], stride TR_THREADS
    uint2* loc;
    __device__ __forceinline__ void put(int i, uint2 e) const { if (i < FS_W8_SSTACK) sh[i * TR_THREADS] = e; else loc[i - FS_W8_SSTACK] = e; }
    __device__ __forceinline__ uint2 get(int i) const { return (i < FS_W8_SSTACK) ? sh[i * TR_THREADS] : loc[i - FS_W8_SSTACK]; }
};

__device__ __forceinline__ void tr_init8(tr_state& s, const fs_bvh_view& bv, fs_vec3 o, fs_vec3 d)
{
    s.o = o; s.d = d;
    const float dx = (fabsf(d.x) > 1e-30f) ? d.x : ((d.x < 0.0f) ? -1e-30f : 1e-30f);
    const float dy = (fabsf(d.y) > 1e-30f) ? d.y : ((d.y < 0.0f) ? -1e-30f : 1e-30f);
    const float dz = (fabsf(d.z) > 1e-30f) ? d.z : ((d.z < 0.0f) ? -1e-30f : 1e-30f);
    s.idx = fs_rcp_fast(dx); s.idy = fs_rcp_fast(dy); s.idz = fs_rcp_fast(dz);     // conservative boxes: 1 ulp is inside the padding
    s.oodx = s.oody = s.oodz = 0.0f;
    s.oct = ((~__float_as_uint(s.idx)) >> 31) | (((~__float_as_uint(s.idy)) >> 31) << 1) | (((~__float_as_uint(s.idz)) >> 31) << 2);
    s.node = bv.n_tris ? 0 : TR_SENT; s.leaf = 0; s.sp = 0; s.tc = 0; s.te = 0;
}

// 2^15 + (byte B of w) as a float: the byte goes to bits 8..15 of 0x47000000
#define FS_Q8(w, B) __uint_as_float(__byte_perm((w), magic, 0x7504u | ((B) << 4)))

// One step of lane state `s` through its node.  Returns the leaf slots the ray enters (hleaf, with the node's leaf mask
// and first triangle: triangle of slot b = tri_base + popc(lmask below b)) and moves s.node on to the next inner node
// (nearest hit child, else the next one of the newest group on the stack, else TR_SENT).
__device__ __forceinline__ void w8_step(const fs_bvh_view& bv, tr_state& s, const w8_stack& stack, const float tlimit,
                                        uint32_t& hleaf, uint32_t& lmask, uint32_t& tri_base, uint32_t* overflow)
{
    const uint32_t magic = bv.w8_magic;
    const uint4* p = bv.w8nodes + (size_t)s.node * 5;
    const uint4 u0 = ldg_u4(p), u1 = ldg_u4(p + 1), u2 = ldg_u4(p + 2), u3 = ldg_u4(p + 3), u4 = ldg_u4(p + 4);
    const float ax = __uint_as_float(u0.w & 0x7f800000u) * s.idx, ay = __uint_as_float(u1.x) * s.idy, az = __uint_as_float(u1.y) * s.idz;
    const float bx = fmaf(-32768.0f, ax, (__uint_as_float(u0.x) - s.o.x) * s.idx);
    const float by = fmaf(-32768.0f, ay, (__uint_as_float(u0.y) - s.o.y) * s.idy);
    const float bz = fmaf(-32768.0f, az, (__uint_as_float(u0.z) - s.o.z) * s.idz);
    const bool px = (s.oct & 1u) != 0u, py = (s.oct & 2u) != 0u, pz = (s.oct & 4u) != 0u;
    const uint32_t nx0 = px ? u2.x : u3.z, nx1 = px ? u2.y : u3.w, fx0 = px ? u3.z : u2.x, fx1 = px ? u3.w : u2.y;
    const uint32_t ny0 = py ? u2.z : u4.x, ny1 = py ? u2.w : u4.y, fy0 = py ? u4.x : u2.z, fy1 = py ? u4.y : u2.w;
    const uint32_t nz0 = pz ? u3.x : u4.z, nz1 = pz ? u3.y : u4.w, fz0 = pz ? u4.z : u3.x, fz1 = pz ? u4.w : u3.y;
    uint32_t H = 0u;
#define FS_W8_CHILD(J, W, B)                                                                                          \
    {                                                                                                                 \
        const float tn = fmaxf(fmaxf(fmaf(FS_Q8(nx##W, B), ax, bx), fmaf(FS_Q8(ny##W, B), ay, by)),                   \
                               fmaxf(fmaf(FS_Q8(nz##W, B), az, bz), 0.0f));                                           \
        const float tf = fminf(fminf(fmaf(FS_Q8(fx##W, B), ax, bx), fmaf(FS_Q8(fy##W, B), ay, by)),                   \
                               fminf(fmaf(FS_Q8(fz##W, B), az, bz), tlimit));                                         \
        if (tn <= tf) H |= 1u << (J);                                                                                 \
    }
    FS_W8_CHILD(0, 0, 0u) FS_W8_CHILD(1, 0, 1u) FS_W8_CHILD(2, 0, 2u) FS_W8_CHILD(3, 0, 3u)
    FS_W8_CHILD(4, 1, 0u) FS_W8_CHILD(5, 1, 1u) FS_W8_CHILD(6, 1, 2u) FS_W8_CHILD(7, 1, 3u)
#undef FS_W8_CHILD
    const uint32_t imask = u0.w & 0xffu;
    lmask = (u0.w >> 8) & 0xffu;
    hleaf = H & lmask;
    tri_base = u1.w;
    // inner hits, moved to traversal positions: position = slot XOR octant, highest first
    uint32_t P = H & imask;
    if (s.oct & 4u) P = ((P & 0x0fu) << 4) | (P >> 4);
    if (s.oct & 2u) P = ((P & 0x33u) << 2) | ((P >> 2) & 0x33u);
    if (s.oct & 1u) P = ((P & 0x55u) << 1) | ((P >> 1) & 0x55u);
    uint32_t gb = u1.z, gm = (P << 8) | imask;
    if (P == 0u) {                                   // nothing entered here: next child of the newest group on the stack
        if (s.sp == 0) { s.node = TR_SENT; return; }
        --s.sp;
        const uint2 e = stack.get(s.sp);
        gb = e.x; gm = e.y;
    }
    const uint32_t pbit = 31u - (uint32_t)__clz((int)gm);       // in 8..15
    gm ^= 1u << pbit;
    const uint32_t slot = (pbit - 8u) ^ s.oct;
    s.node = (int)(gb + (uint32_t)__popc(gm & ((1u << slot) - 1u)));        // slot <= 7: the mask only covers the inner-mask bits
    if (gm >> 8) {
        if (s.sp < FS_W8_STACK_SIZE) { stack.put(s.sp, make_uint2(gb, gm)); ++s.sp; } else *overflow = 1u;
    }
}

// =============================================================================================
// k_trace_q: traversal with a WARP-SHARED TRIANGLE QUEUE (closest hit of extension rays; any hit of connection rays).
//
// ncu on k_trace_closest (r1h/r1i, SASS-level counters): a ray needs ~2 550 thread-instructions, the kernel
// spends 3 100 -- but only 17.9 of 32 lanes are active per issued instruction.  The lost lanes are phase
// mismatch: in the node phase 11 lanes sit out (waiting at a second leaf, or done with a postponed leaf), and
// the triangle phase runs with 10.6 lanes because only the lanes that happen to hold a leaf take part.
//
// Here a lane never holds a leaf.  Every leaf child (one triangle) whose box the ray enters is appended as
// (owner lane, triangle) to a queue shared by the warp (shared memory, one ATOMS per node step) and the lane
// keeps walking; the traversal stack only holds inner nodes.  When >= FLUSH_MIN entries are waiting (or
// nobody can walk) the warp tests them CONVERGED: lane i takes entry i whoever owns it, fetches the owner's
// ray by shuffle, and merges a hit into the owner's best (t, triangle) -- a 64-bit key in shared memory,
// updated by compare-and-swap with the oracle's exact tie rule (equal t: lower original id).  The node phase
// loses only the lanes that are out of rays; the triangle phase runs at up to 32 of 32.
// Results are unchanged by construction: the closest hit is min (t, original id) over the triangles whose
// boxes the ray enters at or before the best t known so far -- any order, any delay.
// =============================================================================================
// at most FLUSH_MIN - 1 (<= 31) entries are waiting when a node-phase iteration starts and it adds at most 4 x 32
#define FS_TQ_CAP 160
#define TQ_INVALID 0xffffffffu
#define TQ_WARPS (TR_THREADS / 32)
#define TR_SMEM_TQ (FS_SSTACK * TR_THREADS * sizeof(int) + TR_THREADS * sizeof(unsigned long long) + \
                    TQ_WARPS * FS_TQ_CAP * sizeof(uint32_t) + TQ_WARPS * sizeof(uint32_t) + TR_THREADS * sizeof(uint32_t))

#ifndef FS_DRAIN_SPLIT
#define FS_DRAIN_SPLIT 1
#endif
#ifndef FS_PREFETCH_PUSHED
#define FS_PREFETCH_PUSHED 0
#endif
#ifndef FS_PREFETCH_TRIS
#define FS_PREFETCH_TRIS 0
#endif
#ifndef FS_TRI_TEX
#define FS_TRI_TEX 0
#endif
// ANY = false: closest hit of extension rays -> hits[j] = (t, triangle).
// ANY = true : connection rays (F.xyz, tmax) (dir.xyz, path id): any triangle closer than tmax occludes; the paths that
//              stay visible are appended to conn_queue.  Same node phase and queue; the "best key" of a lane degenerates
//              to an occluded flag (any store wins), and bt is the constant tmax.
// at most FLUSH_MIN - 1 (<= 31) entries wait when a node-phase iteration starts; an 8-wide step adds at most 8 x 32
#define FS_TQ8_CAP 288
#define TR_SMEM_TQ8 (FS_W8_SSTACK * TR_THREADS * sizeof(uint2) + TR_THREADS * sizeof(unsigned long long) + \
                     TQ_WARPS * FS_TQ8_CAP * sizeof(uint32_t) + TQ_WARPS * sizeof(uint32_t) + TR_THREADS * sizeof(uint32_t))
// W8 = true: 8-wide compressed nodes (w8_step), group stack, triangles in W8 order; false: 4-wide nodes (wide_children)
template <bool COUNT, int TEX, bool ANY, bool W8>
__global__ void __launch_bounds__(TR_THREADS, FS_TR_MINBLOCKS)
k_trace_q(const fs_bvh_view bv, const float4* __restrict__ ray_o, const float4* __restrict__ ray_d,
          const uint32_t* __restrict__ count_ptr, uint32_t* __restrict__ cursor,
          float2* __restrict__ hits, uint32_t* __restrict__ conn_queue, uint32_t* __restrict__ conn_count,
          fs_path_dbg* __restrict__ dbg, fs_dev_counters* __restrict__ dc, const uint32_t REFILL_MIN,
          const uint32_t NODE_MIN, const uint32_t FLUSH_MIN)
{
    constexpr bool DRAIN_SPLIT = FS_DRAIN_SPLIT != 0;
    constexpr uint32_t QCAP = W8 ? FS_TQ8_CAP : FS_TQ_CAP;
    constexpr int SST = W8 ? FS_W8_SSTACK : FS_SSTACK;         // stack entries per thread in shared memory
    const uint32_t lane = lane_id(), warp = threadIdx.x >> 5;
    const uint32_t count = *count_ptr;
    extern __shared__ __align__(8) unsigned char smem_raw[];
    int* const sstack = reinterpret_cast<int*>(smem_raw);
    uint2* const gstack = reinterpret_cast<uint2*>(smem_raw);
    unsigned long long* const skey = reinterpret_cast<unsigned long long*>(smem_raw + (W8 ? FS_W8_SSTACK * sizeof(uint2) : FS_SSTACK * sizeof(int)) * TR_THREADS);
    uint32_t* const squeue = reinterpret_cast<uint32_t*>(skey + TR_THREADS) + warp * QCAP;
    uint32_t* const sqcount = reinterpret_cast<uint32_t*>(skey + TR_THREADS) + TQ_WARPS * QCAP + warp;
    // helpers working for each lane's ray (drain splitting, below)
    uint32_t* const whelp = reinterpret_cast<uint32_t*>(skey + TR_THREADS) + TQ_WARPS * QCAP + TQ_WARPS + (threadIdx.x & ~31u);
    unsigned long long* const mykey = skey + threadIdx.x;
    unsigned long long* const wkey = skey + (threadIdx.x & ~31u);
    int lstack[W8 ? 1 : FS_STACK_SIZE - FS_SSTACK];
    uint2 lstack8[W8 ? FS_W8_STACK_SIZE - FS_W8_SSTACK : 1];
    tr_stack<false> stack; stack.sh = sstack + threadIdx.x; stack.loc = lstack;
    w8_stack stack8; stack8.sh = gstack + threadIdx.x; stack8.loc = lstack8;
    const float4* const tris = W8 ? bv.tris8 : bv.tris;
    const unsigned long long KEY_NONE = ((unsigned long long)0x7f800000u << 32) | 0xffffffffull;
    for (uint32_t i = lane; i < QCAP; i += 32) squeue[i] = TQ_INVALID;
    if (lane == 0) *sqcount = 0u;
    *mykey = KEY_NONE;
    whelp[lane] = 0u;
    uint32_t owner = lane;                           // lane whose ray this lane is walking (itself, except for drain helpers)
    __syncwarp();
    tr_state s;
    s.node = TR_SENT; s.leaf = 0; s.sp = 0; s.tc = 0; s.te = 0;
    s.o = fs_mk(0.f, 0.f, 0.f); s.d = s.o; s.idx = s.idy = s.idz = s.oodx = s.oody = s.oodz = 0.f;
    bool running = false, exhausted = false;
    uint32_t j = 0;
    uint32_t* const ovf_p = &dc->overflow;
    float bt = __int_as_float(0x7f800000);
    uint32_t qn = 0;                                 // entries in the warp's triangle queue (warp-uniform)
    uint32_t ray_steps = 0;                          // COUNT builds: node steps of the current ray
    fs_visit_counters vc; vc.nodes = 0; vc.tris = 0;
    for (;;) {
        // ---- refill idle lanes from the ray queue: one atomic per warp
        const uint32_t m_idle = __ballot_sync(FULLM, !running);
        if (!exhausted && ((uint32_t)__popc(m_idle) >= REFILL_MIN)) {
            const uint32_t n = (uint32_t)__popc(m_idle);
            uint32_t base = 0;
            if (lane == 0) base = atomicAdd(cursor, n);
            base = __shfl_sync(FULLM, base, 0);
            if (base + n >= count) exhausted = true;
            if (!running) {
                const uint32_t jj = base + (uint32_t)__popc(m_idle & ((1u << lane) - 1u));
                if (jj < count) {
                    const float4 a = FS_LD4(ray_o + jj), b = FS_LD4(ray_d + jj);
                    if (W8) tr_init8(s, bv, fs_mk(a.x, a.y, a.z), fs_mk(b.x, b.y, b.z));
                    else tr_init<true>(s, bv, fs_mk(a.x, a.y, a.z), fs_mk(b.x, b.y, b.z));
                    bt = ANY ? a.w : __int_as_float(0x7f800000); *mykey = KEY_NONE;
                    j = ANY ? __float_as_uint(b.w) : jj; running = true;
                    if (COUNT) ray_steps = 0;
                }
            }
        }
        if (!__any_sync(FULLM, running)) break;
        for (;;) {
            // ---- node phase: every lane with a ray walks; leaves go to the queue
            for (;;) {
                const bool can = running && s.node >= 0 && s.node != TR_SENT;
                const uint32_t m_can = __ballot_sync(FULLM, can);
                if (m_can == 0u || qn >= FLUSH_MIN) break;
                if (NODE_MIN && qn && (uint32_t)__popc(m_can) < NODE_MIN) break;   // few walkers left and triangle work waits
                uint32_t nl = 0;
                if (can) {
                    if (COUNT) { vc.nodes++; ray_steps++; }
                    if (W8) {
                        uint32_t hleaf, lmask, tri_base;
                        w8_step(bv, s, stack8, bt, hleaf, lmask, tri_base, ovf_p);
                        nl = (uint32_t)__popc(hleaf);
                        if (nl) {                     // entry = triangle << 5 | owner lane; triangle of slot b = tri_base + leaves below b
                            uint32_t* q = squeue + atomicAdd(sqcount, nl);
                            const uint32_t e0 = (tri_base << 5) | owner;
                            do {
                                const uint32_t bit = hleaf & (0u - hleaf);
                                *q++ = e0 + ((uint32_t)__popc(lmask & (bit - 1u)) << 5);
                                hleaf ^= bit;
                            } while (hleaf);
                        }
                    } else {
                        const float INF = __int_as_float(0x7f800000);
                        float k0, k1, k2, k3; int v0, v1, v2, v3;
                        wide_children<2, TEX>(bv, s, bt, k0, k1, k2, k3, v0, v1, v2, v3);
                        // every leaf child the ray enters goes to the queue right away (single-triangle leaves), so the
                        // stack only ever holds inner nodes and the step is straight-line code.
                        // leaf code v = ~(first << 3): entry = first << 5 | lane = -4 v + (lane - 4)
                        const bool l0 = k0 != INF && v0 < 0, l1 = k1 != INF && v1 < 0, l2 = k2 != INF && v2 < 0, l3 = k3 != INF && v3 < 0;
                        nl = (uint32_t)l0 + (uint32_t)l1 + (uint32_t)l2 + (uint32_t)l3;
                        if (nl) {
                            uint32_t* q = squeue + atomicAdd(sqcount, nl);
                            const uint32_t lm4 = owner - 4u;
#if FS_PREFETCH_TRIS
#define FS_PF_TRI(v) asm volatile("prefetch.global.L2 [%0];" :: "l"(bv.tris + (size_t)((uint32_t)(~(v)) >> 3) * 4))
#else
#define FS_PF_TRI(v)
#endif
                            if (l0) { *q = (uint32_t)v0 * 0xfffffffcu + lm4; FS_PF_TRI(v0); }
                            q += l0;
                            if (l1) { *q = (uint32_t)v1 * 0xfffffffcu + lm4; FS_PF_TRI(v1); }
                            q += l1;
                            if (l2) { *q = (uint32_t)v2 * 0xfffffffcu + lm4; FS_PF_TRI(v2); }
                            q += l2;
                            if (l3) { *q = (uint32_t)v3 * 0xfffffffcu + lm4; FS_PF_TRI(v3); }
#undef FS_PF_TRI
                        }
                        k0 = l0 ? INF : k0; k1 = l1 ? INF : k1; k2 = l2 ? INF : k2; k3 = l3 ? INF : k3;
                        FS_CSWAP(k0, v0, k1, v1) FS_CSWAP(k2, v2, k3, v3) FS_CSWAP(k0, v0, k2, v2) FS_CSWAP(k1, v1, k3, v3) FS_CSWAP(k1, v1, k2, v2)
                        w4_advance(s, stack, k0, k1, k2, k3, v0, v1, v2, v3, ovf_p);
                    }
                }
                qn += __reduce_add_sync(FULLM, nl);         // the queue length, tracked in a (uniform) register
            }
            // ---- triangle phase: the queue, 32 entries at a time, whoever owns them
            __syncwarp();
            const uint32_t total = qn;
            for (uint32_t base = 0; base < total; base += 32) {
                const uint32_t idx = base + lane;
                const uint32_t e = idx < total ? squeue[idx] : TQ_INVALID;
                const uint32_t eo = e & 31u;                       // lane that owns the entry's ray
                const float ox = __shfl_sync(FULLM, s.o.x, eo), oy = __shfl_sync(FULLM, s.o.y, eo), oz = __shfl_sync(FULLM, s.o.z, eo);
                const float dx = __shfl_sync(FULLM, s.d.x, eo), dy = __shfl_sync(FULLM, s.d.y, eo), dz = __shfl_sync(FULLM, s.d.z, eo);
                const float bto = __shfl_sync(FULLM, bt, eo);
                if (e != TQ_INVALID) {
                    const uint32_t tri = e >> 5;
                    const float4* tq = tris + (size_t)tri * 4;
#if FS_TRI_TEX
                    // one of the three triangle quarters through the texture data pipe (as for the nodes)
                    const bool ttex = TEX >= 2 && bv.tris_tex;
                    const float4 a = ttex ? tex1Dfetch<float4>((cudaTextureObject_t)bv.tris_tex, (int)(tri * 4u)) : fs_ldg4(tq);
                    const float4 b = (FS_TRI_TEX >= 2 && ttex) ? tex1Dfetch<float4>((cudaTextureObject_t)bv.tris_tex, (int)(tri * 4u + 1u)) : fs_ldg4(tq + 1);
                    const float4 c = fs_ldg4(tq + 2);
#else
                    const float4 a = fs_ldg4(tq), b = fs_ldg4(tq + 1), c = fs_ldg4(tq + 2);
#endif
                    if (COUNT) vc.tris++;
                    squeue[idx] = TQ_INVALID;
                    float t;
                    const bool hit = fs_intersect_tri(fs_mk(ox, oy, oz), fs_mk(dx, dy, dz), fs_mk(a.x, a.y, a.z), fs_mk(b.x, b.y, b.z),
                                                      fs_mk(c.x, c.y, c.z), t);
                    if (ANY) {
                        if (hit && t < bto) *(volatile unsigned long long*)(wkey + eo) = 0ull;      // occluded: any store wins
                    } else if (hit && t <= bto) {
                        // merge into the owner's best: min over (t, ORIGINAL triangle id); ids are fetched only on a tie
                        const unsigned long long mine = ((unsigned long long)__float_as_uint(t) << 32) | tri;
                        unsigned long long old = *(volatile unsigned long long*)(wkey + eo);
                        for (;;) {
                            const float told = __uint_as_float((uint32_t)(old >> 32));
                            bool better = t < told;
                            if (t == told) {
                                const uint32_t otri = (uint32_t)old;
                                better = otri == 0xffffffffu ||
                                         __float_as_uint(fs_ldg4(tq + 3).x) < __float_as_uint(fs_ldg4(tris + (size_t)otri * 4 + 3).x);
                            }
                            if (!better) break;
                            const unsigned long long prev = atomicCAS(wkey + eo, old, mine);
                            if (prev == old) break;
                            old = prev;
                        }
                    }
                }
            }
            __syncwarp();
            if (lane == 0) *sqcount = 0u;
            qn = 0u;
            const unsigned long long kk = *(volatile unsigned long long*)(wkey + owner);
            if (ANY) { if (running && kk != KEY_NONE) { s.node = TR_SENT; s.sp = 0; } }     // the owner's ray is occluded: stop walking
            else bt = __uint_as_float((uint32_t)(kk >> 32));
            __syncwarp();
            // ---- retire finished rays (nothing of theirs is left in the queue): helpers first, then the owners whose
            // helpers are all done
            const bool fin = running && s.node == TR_SENT;
            if (fin && owner != lane) { atomicSub(whelp + owner, 1u); running = false; owner = lane; }
            __syncwarp();
            const bool retire = fin && running && *(volatile uint32_t*)(whelp + lane) == 0u;
            if (ANY) {
                const bool conn = retire && kk == KEY_NONE;
                const uint32_t mc = __ballot_sync(FULLM, conn);
                if (mc) {                             // ballot-compacted append of the visible pairs
                    uint32_t slot = 0;
                    if (lane == 0) slot = atomicAdd(conn_count, (uint32_t)__popc(mc));
                    slot = __shfl_sync(FULLM, slot, 0);
                    if (conn) {
                        conn_queue[slot + (uint32_t)__popc(mc & ((1u << lane) - 1u))] = j;
                        if (dbg) dbg[j].connected = 1u;
                    }
                }
                if (retire) running = false;
            } else if (retire) {
                uint32_t ht = (uint32_t)kk;                      // 8-wide nodes: position in tris8 -> the index hit records carry
                if (W8 && ht != 0xffffffffu) ht = bv.tri8_map[ht];
                FS_ST2(hits + j, make_float2(bt, __int_as_float((int)ht)));
                running = false;
                if (COUNT) { atomicMax(&dc->max_steps, ray_steps); atomicAdd(&dc->steps_hist[ray_steps / 8u < 15u ? ray_steps / 8u : 15u], 1u); }
            }
            // ---- drain: once the ray queue is empty a launch lasts as long as its longest ray (up to 100 node steps in
            // the room, 400 in the hall, against 16 / 27 on average).  The subtrees on a ray's stack are independent, and
            // every triangle candidate ends up in the OWNER's key whoever found it -- so an idle lane takes the top half
            // of a busy lane's stack and walks it as a helper of the same ray.  The result is the same set of candidates.
            if (DRAIN_SPLIT && exhausted) {
                const uint32_t m_free = __ballot_sync(FULLM, !running);
                const bool give = running && s.node != TR_SENT && s.sp >= 1 && s.sp <= SST;
                const uint32_t m_give = __ballot_sync(FULLM, give);
                const uint32_t nf = (uint32_t)__popc(m_free), ng = (uint32_t)__popc(m_give);
                const uint32_t n = nf < ng ? nf : ng;
                if (n) {
                    const uint32_t lt = (1u << lane) - 1u;
                    const uint32_t rf = (uint32_t)__popc(m_free & lt), rg = (uint32_t)__popc(m_give & lt);
                    const bool take = !running && rf < n;
                    const uint32_t donor = take ? __fns(m_give, 0u, (int)rf + 1) : lane;      // k-th free lane <- k-th giver
                    const int dsp = __shfl_sync(FULLM, s.sp, donor);
                    const float ox = __shfl_sync(FULLM, s.o.x, donor), oy = __shfl_sync(FULLM, s.o.y, donor), oz = __shfl_sync(FULLM, s.o.z, donor);
                    const float dx = __shfl_sync(FULLM, s.d.x, donor), dy = __shfl_sync(FULLM, s.d.y, donor), dz = __shfl_sync(FULLM, s.d.z, donor);
                    const float ix = __shfl_sync(FULLM, s.idx, donor), iy = __shfl_sync(FULLM, s.idy, donor), iz = __shfl_sync(FULLM, s.idz, donor);
                    const float px = __shfl_sync(FULLM, s.oodx, donor), py = __shfl_sync(FULLM, s.oody, donor), pz = __shfl_sync(FULLM, s.oodz, donor);
                    const float dbt = __shfl_sync(FULLM, bt, donor);
                    const uint32_t down = __shfl_sync(FULLM, owner, donor);
                    if (take) {
                        const int h = (dsp + 1) >> 1;
                        s.o = fs_mk(ox, oy, oz); s.d = fs_mk(dx, dy, dz);
                        s.idx = ix; s.idy = iy; s.idz = iz; s.oodx = px; s.oody = py; s.oodz = pz;
                        bt = dbt; owner = down;
                        if (W8) {
                            const uint2* src = gstack + (threadIdx.x & ~31u) + donor;
                            for (int i = 0; i < h; ++i) stack8.sh[i * TR_THREADS] = src[(dsp - h + i) * TR_THREADS];
                            s.oct = ((~__float_as_uint(ix)) >> 31) | (((~__float_as_uint(iy)) >> 31) << 1) | (((~__float_as_uint(iz)) >> 31) << 2);
                            // next child of the newest group taken over (as the pop of w8_step)
                            s.sp = h - 1;
                            const uint2 e = stack8.sh[s.sp * TR_THREADS];
                            uint32_t gm = e.y;
                            const uint32_t pbit = 31u - (uint32_t)__clz((int)gm);
                            gm ^= 1u << pbit;
                            const uint32_t slot = (pbit - 8u) ^ s.oct;
                            s.node = (int)(e.x + (uint32_t)__popc(gm & ((1u << slot) - 1u)));
                            if (gm >> 8) { stack8.sh[s.sp * TR_THREADS] = make_uint2(e.x, gm); ++s.sp; }
                        } else {
                            const int* src = sstack + (threadIdx.x & ~31u) + donor;
                            for (int i = 0; i < h; ++i) stack.sh[i * TR_THREADS] = src[(dsp - h + i) * TR_THREADS];
                            s.sp = h;
                            s.node = stack.pop(s.sp, 0.f);
                        }
                        running = true;
                        atomicAdd(whelp + down, 1u);
                    }
                    __syncwarp();
                    if (give && rg < n) s.sp -= (s.sp + 1) >> 1;
                }
            }
            const uint32_t m_run = __ballot_sync(FULLM, running);
            if (m_run == 0u) break;
            if (!exhausted && 32u - (uint32_t)__popc(m_run) >= REFILL_MIN) break;
        }
    }
    if (COUNT) flush_counters(dc, vc, ANY);
}

// =============================================================================================
// k_path_q (EXPERIMENTAL, FS_TUNE_MEGA=1): ONE persistent launch per batch for the whole extension stage.
//
// The per-bounce pipeline pays a fixed cost per bounce -- the drain of the traversal launch (the slowest ray) plus the
// latency floor of k_shade_gen -- about 90 us x 16 bounces = 29 % of a room update.  Here a retired ray is not written
// out as a hit record: it goes to a per-warp SHADE QUEUE in shared memory, and when 24 have gathered the warp shades
// them converged (lane i takes entry i: node record, Russian roulette, next direction -- the arithmetic of
// k_shade_gen), appends the successor rays to a global RAY LOG and publishes each with an epoch flag.  Idle lanes of any
// warp take tickets (atomicAdd on the log head) and start a ray as soon as its flag shows the current epoch.  Rays of
// bounce k+1 therefore start while the long rays of bounce k are still walking; there is one drain per batch.
// Termination: `done` counts shaded rays, `tail` appended ones; a parent's successor is appended before the parent is
// counted done, so done == tail (done read first) means nothing is in flight and nothing can be appended any more.
// Every wait is bounded (a poll budget turns a protocol error into FS_ERR_OVERFLOW instead of a hang).
// =============================================================================================
struct pq_globals { uint32_t tail, head, done, error; };
#define PQ_NO_TICKET 0xffffffffu
#ifndef PQ_SHADE_MIN
#define PQ_SHADE_MIN 24u
#endif
#define PQ_SQ_CAP (PQ_SHADE_MIN + 32u)         // at most SHADE_MIN - 1 entries wait when up to 32 lanes retire
// shade queue entry = (ray-log index, t, triangle): the ray itself (origin, direction, subpath id, pdf) is re-read from the log
// when the entry is shaded -- 3 instead of 10 words per entry keeps a CTA at 25 KB of shared memory
#define PQ_SMEM (FS_SSTACK * TR_THREADS * sizeof(int) + TR_THREADS * sizeof(unsigned long long) + \
                 TQ_WARPS * FS_TQ_CAP * sizeof(uint32_t) + TQ_WARPS * sizeof(uint32_t) + \
                 TQ_WARPS * PQ_SQ_CAP * 3 * sizeof(uint32_t) + TR_THREADS * sizeof(uint32_t) + (size_t)FS_PQ_TOP * 64)

__device__ __forceinline__ void st_release_u32(uint32_t* p, uint32_t v) { asm volatile("st.release.gpu.global.u32 [%0], %1;" :: "l"(p), "r"(v) : "memory"); }
__device__ __forceinline__ uint32_t ld_cg_u32(const uint32_t* p) { uint32_t v; asm volatile("ld.global.cg.u32 %0, [%1];" : "=r"(v) : "l"(p)); return v; }
__device__ __forceinline__ float4 ld_cg_f4(const float4* p)
{
    float4 r;
    asm volatile("ld.global.cg.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p));
    return r;
}

// bounce-0 rays (written by k_shade_gen(0) into the ping-pong queue) become the first entries of the ray log
// the rays of bounce k0 (written by k_shade_gen(k0) into the ping-pong queue) become the first entries of the ray log
__global__ void k_pq_seed(const fs_wave_buffers wb, float4* __restrict__ log_o, float4* __restrict__ log_d,
                          uint32_t* __restrict__ log_flag, uint32_t epoch, pq_globals* __restrict__ g, uint32_t k0)
{
    const uint32_t n = wb.q_count[k0];
    const float4* __restrict__ so = wb.st_pos[k0 & 1u];
    const float4* __restrict__ sd = wb.st_nrm[k0 & 1u];
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        float4 a = so[i];                           // (pos, bits(sp_id)): the bounce index goes into the upper bits
        a.w = __uint_as_float(__float_as_uint(a.w) | (k0 << 22));
        log_o[i] = a;
        log_d[i] = sd[i];
        log_flag[i] = epoch;
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) { g->tail = n; g->head = 0u; g->done = 0u; g->error = 0u; }
}
// the number of extension rays of bounces >= k0, where k_connect_gen looks for it
__global__ void k_pq_finish(const fs_wave_buffers wb, const pq_globals* __restrict__ g, uint32_t max_depth, fs_dev_counters* dc, uint32_t k0)
{
    wb.q_count[k0] = g->tail;
    for (uint32_t k = k0 + 1u; k < max_depth; ++k) wb.q_count[k] = 0u;
    if (g->error) dc->overflow = 0x100u | g->error;
}

#ifndef PQ_IDLE_NS
#define PQ_IDLE_NS 256
#endif
#ifndef FS_PQ_TOP
#define FS_PQ_TOP 0             // nodes of the top of the tree staged in shared memory by k_path_q (experiment #68: no gain)
#endif
#ifndef PQ_DRAIN_SPLIT
#define PQ_DRAIN_SPLIT 0      // measured: hall +5 %, room -0.6 % (profiles/r2_experiments.md #67)
#endif
#ifndef PQ_TAIL_LANES
#define PQ_TAIL_LANES 16u    // measured: hall -1.7 %, room unchanged; 24: room +4 % (#66)
#endif
#ifndef PQ_AHEAD
#define PQ_AHEAD 0      // measured: no gain (room 4.42 vs 4.40 ms, hall 10.78 vs 10.72), profiles/r2_experiments.md
#endif
#ifndef FS_PQ_MINBLOCKS
#define FS_PQ_MINBLOCKS 4      // 62 registers, 32 warps/SM (3: 72 registers is slower, 5: spills and no L1 left)
#endif
#define PQ_SMEM8 (FS_W8_SSTACK * TR_THREADS * sizeof(uint2) + TR_THREADS * sizeof(unsigned long long) + \
                  TQ_WARPS * FS_TQ8_CAP * sizeof(uint32_t) + TQ_WARPS * sizeof(uint32_t) + \
                  TQ_WARPS * PQ_SQ_CAP * 3 * sizeof(uint32_t) + TR_THREADS * sizeof(uint32_t) + (size_t)FS_PQ_TOP * 64)
template <int TEX, bool W8>
__global__ void __launch_bounds__(TR_THREADS, FS_PQ_MINBLOCKS)
k_path_q(const fs_trace_params tp, const fs_wave_buffers wb, float4* __restrict__ log_o, float4* __restrict__ log_d,
         uint32_t* __restrict__ log_flag, const uint32_t epoch, const uint32_t log_cap, pq_globals* __restrict__ g,
         const uint32_t REFILL_MIN, const uint32_t NODE_MIN, const uint32_t FLUSH_MIN)
{
    const fs_bvh_view& bv = tp.bv;
    constexpr uint32_t QCAP = W8 ? FS_TQ8_CAP : FS_TQ_CAP;
    const uint32_t lane = lane_id(), warp = threadIdx.x >> 5;
    const uint32_t lt = (1u << lane) - 1u;
    extern __shared__ __align__(16) unsigned char smem_all[];
    // FS_PQ_TOP > 0 (experiment): the first FS_PQ_TOP nodes of the breadth-first array = the top of the tree, in shared memory
    constexpr int NTOP = W8 ? 0 : FS_PQ_TOP;
    const uint4* const stop = reinterpret_cast<const uint4*>(smem_all);
    unsigned char* const smem_raw = smem_all + (size_t)FS_PQ_TOP * 64;
    if (NTOP) {
        uint4* w = reinterpret_cast<uint4*>(smem_all);
        const uint32_t nn = (uint32_t)NTOP * 4u;
        for (uint32_t i = threadIdx.x; i < nn; i += TR_THREADS) w[i] = (i / 4u < bv.n_inner) ? bv.wnodes[i] : make_uint4(0x0000ffffu, 0x0000ffffu, 0x0000ffffu, 0x7fffffffu);
        __syncthreads();
    }
    int* const sstack = reinterpret_cast<int*>(smem_raw);
    uint2* const gstack = reinterpret_cast<uint2*>(smem_raw);
    unsigned long long* const skey = reinterpret_cast<unsigned long long*>(smem_raw + (W8 ? FS_W8_SSTACK * sizeof(uint2) : FS_SSTACK * sizeof(int)) * TR_THREADS);
    uint32_t* const w32 = reinterpret_cast<uint32_t*>(skey + TR_THREADS);
    uint32_t* const squeue = w32 + warp * QCAP;
    uint32_t* const sqcount = w32 + TQ_WARPS * QCAP + warp;
    uint32_t* const shq = w32 + TQ_WARPS * QCAP + TQ_WARPS + warp * (PQ_SQ_CAP * 3);   // shade queue, 3 planes
    // helpers working for each lane's ray (drain splitting, below)
    uint32_t* const whelp = w32 + TQ_WARPS * QCAP + TQ_WARPS + TQ_WARPS * (PQ_SQ_CAP * 3) + (threadIdx.x & ~31u);
    constexpr bool SPLIT = PQ_DRAIN_SPLIT != 0 && !W8;
    uint32_t my_ray = 0;                                                              // ray-log index of the ray this lane walks
    unsigned long long* const mykey = skey + threadIdx.x;
    unsigned long long* const wkey = skey + (threadIdx.x & ~31u);
    int lstack[W8 ? 1 : FS_STACK_SIZE - FS_SSTACK];
    uint2 lstack8[W8 ? FS_W8_STACK_SIZE - FS_W8_SSTACK : 1];
    tr_stack<false> stack; stack.sh = sstack + threadIdx.x; stack.loc = lstack;
    w8_stack stack8; stack8.sh = gstack + threadIdx.x; stack8.loc = lstack8;
    const float4* const tris = W8 ? bv.tris8 : bv.tris;
    const unsigned long long KEY_NONE = ((unsigned long long)0x7f800000u << 32) | 0xffffffffull;
    if (lane == 0) *sqcount = 0u;
    *mykey = KEY_NONE;
    whelp[lane] = 0u;
    uint32_t owner = lane;                            // lane whose ray this lane walks (itself, except for drain helpers)
    __syncwarp();
    tr_state s;
    s.node = TR_SENT; s.leaf = 0; s.sp = 0; s.tc = 0; s.te = 0;
    s.o = fs_mk(0.f, 0.f, 0.f); s.d = s.o; s.idx = s.idy = s.idz = s.oodx = s.oody = s.oodz = 0.f;
    bool running = false, ready = false;              // ready: the entry of `ticket` is published
    uint32_t ticket = PQ_NO_TICKET;
    uint32_t* const ovf_p = &g->error;                 // stack overflow lands in the same word (value 1)
    float bt = __int_as_float(0x7f800000);
    uint32_t qn = 0, sn = 0, polls = 0;
    const uint32_t stride = 2u * wb.cap;
    for (;;) {
        // ---- lanes without a ticket take one for the next entries of the ray log (one atomic per warp).  PQ_AHEAD: also while
        // they still walk a ray, and the ticket's flag is polled meanwhile, so that a ray start costs ONE round trip to the L2
        // (the entry) instead of three in a row (ticket, flag, entry) during which the lane sat out the warp's node steps
        const bool need = (PQ_AHEAD || !running) && ticket == PQ_NO_TICKET;
        const uint32_t m_need = __ballot_sync(FULLM, need);
        const uint32_t m_run0 = __ballot_sync(FULLM, running);
        if ((uint32_t)__popc(m_need) >= REFILL_MIN || (m_need && m_run0 == 0u)) {
            uint32_t base = 0;
            if (lane == 0) base = atomicAdd(&g->head, (uint32_t)__popc(m_need));
            base = __shfl_sync(FULLM, base, 0);
            if (need) ticket = base + (uint32_t)__popc(m_need & lt);
        }
        // ---- a ticket becomes a ray once its log entry is published
        // no fence on this side: the flag and the entry are both read at the L2 (ld.cg), the entry only after the flag's
        // value has come back (the branch needs it), and the writer released the flag after the entry.  __threadfence()
        // here was MEMBAR.SC + CCTL.IVALL -- an L1 flush of the BVH nodes at every ray start (6 % of the stall samples)
        if ((PQ_AHEAD || !running) && !ready && ticket != PQ_NO_TICKET && ticket < log_cap && ld_cg_u32(log_flag + ticket) == epoch) ready = true;
        if (!running && ready) {
            const float4 a = ld_cg_f4(log_o + ticket), b = ld_cg_f4(log_d + ticket);
            if (W8) tr_init8(s, bv, fs_mk(a.x, a.y, a.z), fs_mk(b.x, b.y, b.z));
            else tr_init<true>(s, bv, fs_mk(a.x, a.y, a.z), fs_mk(b.x, b.y, b.z));
            bt = __int_as_float(0x7f800000); *mykey = KEY_NONE;
            my_ray = ticket;
            running = true; ticket = PQ_NO_TICKET; ready = false;
        }
        const uint32_t m_run = __ballot_sync(FULLM, running);
        if (m_run == 0u && sn == 0u) {                // nothing to walk, nothing to shade: finished, or wait for rays
            const uint32_t dn = ld_cg_u32(&g->done);
            const uint32_t tl = ld_cg_u32(&g->tail);
            if (dn == tl || ld_cg_u32(&g->error)) break;
            if (++polls > (1u << 21)) { if (lane == 0) atomicMax(&g->error, 3u); break; }
            __nanosleep(PQ_IDLE_NS);
            continue;
        }
        if (m_run) {
            // ---- node phase (as k_trace_q)
            for (;;) {
                const bool can = running && s.node >= 0 && s.node != TR_SENT;
                const uint32_t m_can = __ballot_sync(FULLM, can);
                if (m_can == 0u || qn >= FLUSH_MIN) break;
                if (NODE_MIN && qn && (uint32_t)__popc(m_can) < NODE_MIN) break;
                uint32_t nl = 0;
                if (can) {
                    if (W8) {
                        uint32_t hleaf, lmask, tri_base;
                        w8_step(bv, s, stack8, bt, hleaf, lmask, tri_base, ovf_p);
                        nl = (uint32_t)__popc(hleaf);
                        if (nl) {
                            uint32_t* q = squeue + atomicAdd(sqcount, nl);
                            const uint32_t e0 = (tri_base << 5) | lane;
                            do {
                                const uint32_t bit = hleaf & (0u - hleaf);
                                *q++ = e0 + ((uint32_t)__popc(lmask & (bit - 1u)) << 5);
                                hleaf ^= bit;
                            } while (hleaf);
                        }
                    } else {
                        const float INF = __int_as_float(0x7f800000);
                        float k0, k1, k2, k3; int v0, v1, v2, v3;
                        wide_children<2, TEX>(bv, s, bt, k0, k1, k2, k3, v0, v1, v2, v3, stop, NTOP);
                        const bool l0 = k0 != INF && v0 < 0, l1 = k1 != INF && v1 < 0, l2 = k2 != INF && v2 < 0, l3 = k3 != INF && v3 < 0;
                        nl = (uint32_t)l0 + (uint32_t)l1 + (uint32_t)l2 + (uint32_t)l3;
                        if (nl) {
                            uint32_t* q = squeue + atomicAdd(sqcount, nl);
                            const uint32_t lm4 = owner - 4u;
                            if (l0) *q = (uint32_t)v0 * 0xfffffffcu + lm4;
                            q += l0;
                            if (l1) *q = (uint32_t)v1 * 0xfffffffcu + lm4;
                            q += l1;
                            if (l2) *q = (uint32_t)v2 * 0xfffffffcu + lm4;
                            q += l2;
                            if (l3) *q = (uint32_t)v3 * 0xfffffffcu + lm4;
                        }
                        k0 = l0 ? INF : k0; k1 = l1 ? INF : k1; k2 = l2 ? INF : k2; k3 = l3 ? INF : k3;
                        FS_CSWAP(k0, v0, k1, v1) FS_CSWAP(k2, v2, k3, v3) FS_CSWAP(k0, v0, k2, v2) FS_CSWAP(k1, v1, k3, v3) FS_CSWAP(k1, v1, k2, v2)
                        w4_advance(s, stack, k0, k1, k2, k3, v0, v1, v2, v3, ovf_p);
                    }
                }
                qn += __reduce_add_sync(FULLM, nl);
            }
            // ---- triangle phase
            __syncwarp();
            const uint32_t total = qn;
            for (uint32_t base = 0; base < total; base += 32) {
                const uint32_t idx = base + lane;
                const uint32_t e = idx < total ? squeue[idx] : TQ_INVALID;
                const uint32_t eo = e & 31u;
                const float ox = __shfl_sync(FULLM, s.o.x, eo), oy = __shfl_sync(FULLM, s.o.y, eo), oz = __shfl_sync(FULLM, s.o.z, eo);
                const float dx = __shfl_sync(FULLM, s.d.x, eo), dy = __shfl_sync(FULLM, s.d.y, eo), dz = __shfl_sync(FULLM, s.d.z, eo);
                const float bto = __shfl_sync(FULLM, bt, eo);
                if (e != TQ_INVALID) {
                    const uint32_t tri = e >> 5;
                    const float4* tq = tris + (size_t)tri * 4;
                    const float4 a = fs_ldg4(tq), b = fs_ldg4(tq + 1), c = fs_ldg4(tq + 2);
                    float t;
                    if (fs_intersect_tri(fs_mk(ox, oy, oz), fs_mk(dx, dy, dz), fs_mk(a.x, a.y, a.z), fs_mk(b.x, b.y, b.z), fs_mk(c.x, c.y, c.z), t)
                        && t <= bto) {
                        const unsigned long long mine = ((unsigned long long)__float_as_uint(t) << 32) | tri;
                        unsigned long long old = *(volatile unsigned long long*)(wkey + eo);
                        for (;;) {
                            const float told = __uint_as_float((uint32_t)(old >> 32));
                            bool better = t < told;
                            if (t == told) {
                                const uint32_t otri = (uint32_t)old;
                                better = otri == 0xffffffffu ||
                                         __float_as_uint(fs_ldg4(tq + 3).x) < __float_as_uint(fs_ldg4(tris + (size_t)otri * 4 + 3).x);
                            }
                            if (!better) break;
                            const unsigned long long prev = atomicCAS(wkey + eo, old, mine);
                            if (prev == old) break;
                            old = prev;
                        }
                    }
                }
            }
            __syncwarp();
            if (lane == 0) *sqcount = 0u;
            qn = 0u;
            const unsigned long long kk = *(volatile unsigned long long*)(wkey + owner);
            bt = __uint_as_float((uint32_t)(kk >> 32));
            __syncwarp();
            // ---- retire: helpers first, then the owners whose helpers are all done: the finished ray goes to the warp's shade queue
            bool fin = running && s.node == TR_SENT;
            if (SPLIT) {
                if (fin && owner != lane) { atomicSub(whelp + owner, 1u); running = false; owner = lane; fin = false; }
                __syncwarp();
                fin = fin && *(volatile uint32_t*)(whelp + lane) == 0u;
            }
            const uint32_t m_fin = __ballot_sync(FULLM, fin);
            if (fin) {
                const uint32_t q = sn + (uint32_t)__popc(m_fin & lt);
                shq[0 * PQ_SQ_CAP + q] = my_ray;
                shq[1 * PQ_SQ_CAP + q] = __float_as_uint(bt);
                uint32_t ht = (uint32_t)kk;                      // 8-wide nodes: position in tris8 -> index into tri_nm
                if (W8 && ht != 0xffffffffu) ht = bv.tri8_map[ht];
                shq[2 * PQ_SQ_CAP + q] = ht;
                running = false;
            }
            sn += (uint32_t)__popc(m_fin);
            // ---- drain (as in k_trace_q): a lane that has no ray and whose ticket is not published yet takes the top half of a
            // busy lane's stack and walks it as a helper of the same ray.  At the end of a batch the surviving paths are chains
            // of dependent rays on an almost empty GPU: the batch ends with its slowest chain, and a long ray (up to 435 node
            // steps in the hall against 27 on average) is walked by up to 32 lanes instead of one
            if (SPLIT) {
                // only a lane that HOLDS a ticket whose entry does not exist yet is out of work (a lane without a ticket is merely
                // waiting for the warp's next ticket request: splitting then fragments rays in the steady state, +25 %)
                const bool idle = !running && !ready && ticket != PQ_NO_TICKET;
                const uint32_t m_free = __ballot_sync(FULLM, idle);
                const bool give = running && owner == lane && s.node != TR_SENT && s.sp >= 1 && s.sp <= FS_SSTACK;
                const uint32_t m_give = __ballot_sync(FULLM, give);
                const uint32_t nf = (uint32_t)__popc(m_free), ng = (uint32_t)__popc(m_give);
                const uint32_t n = nf < ng ? nf : ng;
                if (n) {
                    const uint32_t rf = (uint32_t)__popc(m_free & lt), rg = (uint32_t)__popc(m_give & lt);
                    const bool take = idle && rf < n;
                    const uint32_t donor = take ? __fns(m_give, 0u, (int)rf + 1) : lane;      // k-th free lane <- k-th giver
                    const int dsp = __shfl_sync(FULLM, s.sp, donor);
                    const float ox = __shfl_sync(FULLM, s.o.x, donor), oy = __shfl_sync(FULLM, s.o.y, donor), oz = __shfl_sync(FULLM, s.o.z, donor);
                    const float dx = __shfl_sync(FULLM, s.d.x, donor), dy = __shfl_sync(FULLM, s.d.y, donor), dz = __shfl_sync(FULLM, s.d.z, donor);
                    const float ix = __shfl_sync(FULLM, s.idx, donor), iy = __shfl_sync(FULLM, s.idy, donor), iz = __shfl_sync(FULLM, s.idz, donor);
                    const float px = __shfl_sync(FULLM, s.oodx, donor), py = __shfl_sync(FULLM, s.oody, donor), pz = __shfl_sync(FULLM, s.oodz, donor);
                    const float dbt = __shfl_sync(FULLM, bt, donor);
                    if (take) {
                        const int h = (dsp + 1) >> 1;
                        const int* src = sstack + (threadIdx.x & ~31u) + donor;
                        for (int i = 0; i < h; ++i) stack.sh[i * TR_THREADS] = src[(dsp - h + i) * TR_THREADS];
                        s.o = fs_mk(ox, oy, oz); s.d = fs_mk(dx, dy, dz);
                        s.idx = ix; s.idy = iy; s.idz = iz; s.oodx = px; s.oody = py; s.oodz = pz;
                        s.sp = h; bt = dbt; owner = donor;
                        s.node = stack.pop(s.sp, 0.f);
                        running = true;
                        atomicAdd(whelp + donor, 1u);
                    }
                    __syncwarp();
                    if (give && rg < n) s.sp -= (s.sp + 1) >> 1;
                }
            }
        }
        // ---- shading phase: converged, lane i shades entry i (the arithmetic of k_shade_gen for node k = bounce + 1)
        // ... or, with PQ_TAIL_LANES, as soon as fewer than that many lanes of the warp still walk: at the end of a batch the few
        // surviving paths are chains of dependent rays, and a finished ray that waits for the slowest ray of its warp before it is
        // shaded lengthens every link of the chain
        if (sn >= PQ_SHADE_MIN || (sn && (uint32_t)__popc(__ballot_sync(FULLM, running)) < (PQ_TAIL_LANES ? PQ_TAIL_LANES : 1u))) {
            __syncwarp();
            for (uint32_t base = 0; base < sn; base += 32) {
                const uint32_t qi = base + lane;
                bool emit = false;
                fs_vec3 pos = fs_mk(0.f, 0.f, 0.f), dir = pos;
                float prob = 1.0f; uint32_t spk_out = 0;
                if (qi < sn) {
                    const uint32_t ri = shq[0 * PQ_SQ_CAP + qi];
                    const float4 ra = ld_cg_f4(log_o + ri), rb = ld_cg_f4(log_d + ri);      // the ray, back from the log (L2)
                    const uint32_t spk = __float_as_uint(ra.w);
                    const uint32_t sp_id = spk & 0x3fffffu, k = (spk >> 22) + 1u;
                    const float t = __uint_as_float(shq[1 * PQ_SQ_CAP + qi]);
                    const int tri = (int)shq[2 * PQ_SQ_CAP + qi];
                    const fs_vec3 o = fs_mk(ra.x, ra.y, ra.z);
                    const fs_vec3 d = fs_mk(rb.x, rb.y, rb.z);
                    const float pdf_in = rb.w;
                    fs_vec3 nrm = fs_mk(0.f, 0.f, 0.f);
                    bool cont = true, hit = false;
                    uint32_t nodes = k, mat = 0;
                    float seg = 0.f;
                    if (tri < 0) {                    // miss: the subpath ends at the node the ray left
                        if (!tp.lobes) wb.end_pos[sp_id] = make_float4(o.x, o.y, o.z, __uint_as_float(k));
                        else if (k >= 2u) {           // material model: see k_shade_gen
                            float4* rp = wb.rec + (size_t)(k - 1u) * stride + sp_id;
                            // written earlier in THIS launch, possibly by another SM, and its 32-byte sector also holds the
                            // record of the pair's other subpath: read at the L2, never through a (possibly stale) L1 line
                            float4 rv = ld_cg_f4(rp);
                            rv.y = __uint_as_float(__float_as_uint(rv.y) & 0x00ffffffu);
                            *rp = rv;
                        }
                        cont = false;
                    } else {                          // SUB.cpp:343-348
                        const float4 nm = fs_ldg4(bv.tri_nm + tri);
                        fs_vec3 fn = fs_mk(nm.x, nm.y, nm.z);
                        if (fs_dot(fn, d) > 0.0f) { fn.x = -fn.x; fn.y = -fn.y; fn.z = -fn.z; }
                        pos.x = fmaf(tp.eps_offset, fn.x, fmaf(t, d.x, o.x));
                        pos.y = fmaf(tp.eps_offset, fn.y, fmaf(t, d.y, o.y));
                        pos.z = fmaf(tp.eps_offset, fn.z, fmaf(t, d.z, o.z));
                        const fs_vec3 dl = fs_sub(pos, o);
                        seg = sqrtf(fs_dot(dl, dl));
                        mat = __float_as_uint(nm.w);
                        nrm = fn;
                        nodes = k + 1u;
                        hit = true;
                        if (k >= pair_depth(tp, wb, sp_id >> 1)) cont = false;
                    }
                    uint32_t ev = FS_EV_DIFFUSE;
                    fs_vec3 org = pos;
                    if (cont) {
                        uint64_t gg = tp.g_first + (sp_id >> 1);
                        if ((tp.flags & FS_FLAG_SHARE_LISTENER) && (sp_id & 1u)) gg = listener_key(tp, wb, sp_id >> 1);
                        emit = choose_direction(tp, k, gg, sp_id & 1u, nrm, d, mat, pos, dir, prob, ev, org);
                        spk_out = sp_id | (k << 22);
                    }
                    if (hit) {
                        FS_ST4(wb.rec + (size_t)k * stride + sp_id, make_float4(seg, __uint_as_float(mat | (ev << 24)), pdf_in, fs_pow(pdf_in, tp.ep.pdf_exponent)));
                        if (!emit || tp.lobes) FS_ST4(wb.end_pos + sp_id, make_float4(pos.x, pos.y, pos.z, __uint_as_float(nodes)));
                    }
                    pos = org;
                }
                const uint32_t m_emit = __ballot_sync(FULLM, emit);
                if (m_emit) {
                    uint32_t slot = 0;
                    if (lane == 0) slot = atomicAdd(&g->tail, (uint32_t)__popc(m_emit));
                    slot = __shfl_sync(FULLM, slot, 0);
                    if (emit) {
                        const uint32_t w = slot + (uint32_t)__popc(m_emit & lt);
                        if (w < log_cap) {
                            log_d[w] = make_float4(dir.x, dir.y, dir.z, prob);
                            log_o[w] = make_float4(pos.x, pos.y, pos.z, __uint_as_float(spk_out));
                            st_release_u32(log_flag + w, epoch);      // MEMBAR.ALL.GPU + ST.STRONG: no L1 invalidation
                        } else atomicMax(&g->error, 2u);        // the log is sized for the worst case: cannot happen
                    }
                }
            }
            __syncwarp();
            // lane 0 made every tail increment of this batch itself and used the returned slots: they are performed before this
            if (lane == 0) atomicAdd(&g->done, sn);            // after the successors were appended
            sn = 0u;
        }
    }
}

// connection rays: (F.xyz, tmax) (dir.xyz, path id); unoccluded paths are appended to conn_queue
template <bool COUNT, int TEX, bool WIDE>
__global__ void __launch_bounds__(TR_THREADS, FS_TR_MINBLOCKS)
k_trace_any(const fs_bvh_view bv, const float4* __restrict__ ray_o, const float4* __restrict__ ray_d,
            const uint32_t* __restrict__ count_ptr, uint32_t* __restrict__ cursor,
            uint32_t* __restrict__ conn_queue, uint32_t* __restrict__ conn_count,
            fs_dev_counters* __restrict__ dc, fs_path_dbg* __restrict__ dbg, const uint32_t REFILL_MIN,
            const uint32_t NODE_MIN)
{
    const uint32_t lane = lane_id();
    const uint32_t count = *count_ptr;
    extern __shared__ int smem_stack[];
    int lstack[FS_STACK_SIZE - FS_SSTACK];
    tr_stack<false> stack; stack.sh = smem_stack + threadIdx.x; stack.loc = lstack;
    tr_state s;
    s.node = TR_SENT; s.leaf = 0; s.sp = 0; s.tc = 0; s.te = 0;
    s.o = fs_mk(0.f, 0.f, 0.f); s.d = s.o; s.idx = s.idy = s.idz = s.oodx = s.oody = s.oodz = 0.f;
    bool running = false, exhausted = false, occluded = false;
    uint32_t path = 0, guard = 0;
    uint32_t* const ovf_p = &dc->overflow;
    float tmax = 0.f;
    fs_visit_counters vc; vc.nodes = 0; vc.tris = 0;
    for (;;) {
        const uint32_t m_idle = __ballot_sync(FULLM, !running);
        if (!exhausted && ((uint32_t)__popc(m_idle) >= REFILL_MIN)) {
            const uint32_t n = (uint32_t)__popc(m_idle);
            uint32_t base = 0;
            if (lane == 0) base = atomicAdd(cursor, n);
            base = __shfl_sync(FULLM, base, 0);
            if (base + n >= count) exhausted = true;
            if (!running) {
                const uint32_t jj = base + (uint32_t)__popc(m_idle & ((1u << lane) - 1u));
                if (jj < count) {
                    const float4 a = ray_o[jj], b = ray_d[jj];
                    tr_init<WIDE>(s, bv, fs_mk(a.x, a.y, a.z), fs_mk(b.x, b.y, b.z));
                    tmax = a.w; path = __float_as_uint(b.w); occluded = false; running = true;
                }
            }
        }
        if (!__any_sync(FULLM, running)) break;
        for (;;) {
#if defined(FS_TRAVERSAL_GUARD)
            if (++guard > (1u << 22)) { *ovf_p = 2u; running = false; exhausted = true; break; }   // bring-up guard
#endif
            for (;;) {
                const bool can = running && s.node >= 0 && s.node != TR_SENT;
                if (!__any_sync(FULLM, can && s.leaf == 0)) break;
                if (NODE_MIN && (uint32_t)__popc(__ballot_sync(FULLM, can)) < NODE_MIN && __any_sync(FULLM, s.leaf != 0)) break;
                if (can) {
                    if (COUNT) vc.nodes++;
                    if (WIDE) tr_node_step4<FS_ANY_ORDERED != 0, (TEX ? 2 : 0)>(bv, s, stack, tmax, ovf_p);
                    else tr_node_step<false, (TEX ? 2 : 0)>(bv, s, stack, tmax, ovf_p);
                }
            }
            tr_next_leaf(s, stack, tmax);
            for (;;) {
                const bool has = s.tc < s.te;
                if (!__any_sync(FULLM, has)) break;
                if (has) {
                    const float4* tq = bv.tris + (size_t)s.tc * 4;
                    const float4 a = fs_ldg4(tq), b = fs_ldg4(tq + 1), c = fs_ldg4(tq + 2);
                    if (COUNT) vc.tris++;
                    float t;
                    ++s.tc;
                    if (fs_intersect_tri(s.o, s.d, fs_mk(a.x, a.y, a.z), fs_mk(b.x, b.y, b.z), fs_mk(c.x, c.y, c.z), t)
                        && t < tmax) {           // any hit ends the ray
                        occluded = true; s.tc = s.te; s.node = TR_SENT; s.leaf = 0; s.sp = 0;
                    } else tr_next_leaf(s, stack, tmax);
                }
            }
            const bool done = running && s.node == TR_SENT && s.leaf == 0;
            const bool conn = done && !occluded;
            const uint32_t mc = __ballot_sync(FULLM, conn);
            if (mc) {                             // ballot-compacted append of the visible pairs
                uint32_t slot = 0;
                if (lane == 0) slot = atomicAdd(conn_count, (uint32_t)__popc(mc));
                slot = __shfl_sync(FULLM, slot, 0);
                if (conn) {
                    conn_queue[slot + (uint32_t)__popc(mc & ((1u << lane) - 1u))] = path;
                    if (dbg) dbg[path].connected = 1u;
                }
            }
            if (done) running = false;
            const uint32_t m_run = __ballot_sync(FULLM, running);
            if (m_run == 0u) break;
            if (!exhausted && 32u - (uint32_t)__popc(m_run) >= REFILL_MIN) break;
        }
    }
    (void)guard;
    if (COUNT) flush_counters(dc, vc, true);
}

// builds the connection ray of every pair; pairs closer than eps_connect are visible by definition
__global__ void __launch_bounds__(WF_THREADS)
k_connect_gen(const fs_trace_params tp, const fs_wave_buffers wb, fs_dev_counters* __restrict__ dc,
              fs_path_dbg* __restrict__ dbg)
{
    const uint32_t lane = lane_id();
    const uint32_t qc = tp.max_depth + 1, qs = tp.max_depth + 2;
    float4* __restrict__ sh_o = wb.st_pos[0];
    float4* __restrict__ sh_d = wb.st_nrm[0];
    if (blockIdx.x == 0 && threadIdx.x == 0) {              // extension rays of this batch = the lengths of its ray queues
        unsigned long long ext = 0;
        for (uint32_t k = 0; k < tp.max_depth; ++k) ext += wb.q_count[k];
        atomicAdd(&dc->ext_rays, ext);
    }
    // one shadow-queue atomic per CTA tile (as in k_shade_gen: per-warp atomics on one address ran at ~1 per ns and were
    // 63 % of this kernel's stall samples); the shadow-ray count is added once per CTA
    __shared__ uint32_t s_cnt[WF_THREADS / 32], s_base;
    const uint32_t warp = threadIdx.x >> 5;
    for (uint32_t tile = blockIdx.x * blockDim.x; tile < tp.batch; tile += gridDim.x * blockDim.x) {
        const uint32_t p = tile + threadIdx.x;
        bool shadow = false, direct = false;
        fs_vec3 F = fs_mk(0.f, 0.f, 0.f), dir = F;
        float tmax = 0.f;
        if (p < tp.batch) {
            const float4 fe = wb.end_pos[2u * p], be = wb.end_pos[2u * p + 1u];
            F = fs_mk(fe.x, fe.y, fe.z);
            const fs_vec3 dl = fs_sub(fs_mk(be.x, be.y, be.z), F);
            const float len = sqrtf(fs_dot(dl, dl));
            wb.conn_len[p] = len;
            tmax = len - tp.eps_connect;                    // SUB.cpp:253
            if (tmax > 0.0f) {
                const float inv = 1.0f / len;
                dir = fs_mk(dl.x * inv, dl.y * inv, dl.z * inv);
                shadow = true;
            } else direct = true;
            if (dbg) {
                fs_path_dbg* q = dbg + p;
                q->n_src_nodes = __float_as_uint(fe.w); q->n_lis_nodes = __float_as_uint(be.w);
                q->connected = direct ? 1u : 0u; q->bin = -1; q->delay_s = 0.f; q->total_dist = 0.f;
                for (int b = 0; b < FS_MAX_BANDS; ++b) q->energy[b] = 0.f;
                q->src_end[0] = fe.x; q->src_end[1] = fe.y; q->src_end[2] = fe.z;
                q->lis_end[0] = be.x; q->lis_end[1] = be.y; q->lis_end[2] = be.z;
            }
        }
        const uint32_t ms = __ballot_sync(FULLM, shadow), md = __ballot_sync(FULLM, direct);
        if (lane == 0) s_cnt[warp] = (uint32_t)__popc(ms);
        __syncthreads();
        if (threadIdx.x == 0) {
            uint32_t tot = 0;
#pragma unroll
            for (int w = 0; w < WF_THREADS / 32; ++w) { const uint32_t c = s_cnt[w]; s_cnt[w] = tot; tot += c; }
            s_base = 0u;
            if (tot) { s_base = atomicAdd(&wb.q_count[qs], tot); atomicAdd(&dc->shadow_rays, (unsigned long long)tot); }
        }
        __syncthreads();
        if (shadow) {
            const uint32_t o = s_base + s_cnt[warp] + (uint32_t)__popc(ms & ((1u << lane) - 1u));
            sh_o[o] = make_float4(F.x, F.y, F.z, tmax);
            sh_d[o] = make_float4(dir.x, dir.y, dir.z, __uint_as_float(p));
        }
        if (md) {                                               // coincident end points: rare
            uint32_t slot_d = 0;
            if (lane == 0) slot_d = atomicAdd(&wb.q_count[qc], (uint32_t)__popc(md));
            slot_d = __shfl_sync(FULLM, slot_d, 0);
            if (direct) wb.conn_queue[slot_d + (uint32_t)__popc(md & ((1u << lane) - 1u))] = p;
        }
        __syncthreads();
    }
}

// FS_FLAG_CONNECT_ALL / FS_FLAG_MIS: the connection ray of every prefix pair (s, t) of every path pair.  One WARP per path
// pair: lane 0 reserves the pair's nf * nb queue slots, the 32 lanes build the (s, t) rays side by side (a pair has up to
// (depth + 1)^2 of them; one thread per pair left 31 lanes idle behind the longest pair of the warp).  A pair closer than
// eps_connect is visible by definition and travels as a ray with tmax = 0 (no triangle has t < 0), so every (s, t) has
// exactly one queue entry.
__global__ void __launch_bounds__(WF_THREADS)
k_connect_all_gen(const fs_trace_params tp, const fs_wave_buffers wb, fs_dev_counters* __restrict__ dc)
{
    const uint32_t qs = tp.max_depth + 2;
    const uint32_t stride = 2u * wb.cap;
    const uint32_t lane = lane_id();
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        unsigned long long ext = 0;
        for (uint32_t k = 0; k < tp.max_depth; ++k) ext += wb.q_count[k];
        atomicAdd(&dc->ext_rays, ext);
    }
    unsigned long long n_shadow = 0;
    const uint32_t warp_global = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint32_t n_warps = (gridDim.x * blockDim.x) >> 5;
    for (uint32_t p = warp_global; p < tp.batch; p += n_warps) {
        const uint32_t nf = __float_as_uint(wb.end_pos[2u * p].w), nb = __float_as_uint(wb.end_pos[2u * p + 1u].w);
        const uint32_t n = nf * nb;
        uint32_t o = 0;
        if (lane == 0) o = atomicAdd(&wb.q_count[qs], n);
        o = __shfl_sync(0xffffffffu, o, 0);
        for (uint32_t idx = lane; idx < n; idx += 32u) {
            const uint32_t s = idx / nb + 1u, t = idx - (s - 1u) * nb + 1u;
            const fs_vec3 F = node_pos(tp, wb, 2u * p, s - 1u, stride);
            const fs_vec3 B = node_pos(tp, wb, 2u * p + 1u, t - 1u, stride);
            const fs_vec3 dl = fs_sub(B, F);
            const float len = sqrtf(fs_dot(dl, dl));
            float tmax = len - tp.eps_connect;                  // SUB.cpp:253
            fs_vec3 dir = fs_mk(1.0f, 0.0f, 0.0f);
            if (tmax > 0.0f) {
                const float inv = 1.0f / len;
                dir = fs_mk(dl.x * inv, dl.y * inv, dl.z * inv);
                ++n_shadow;
            } else tmax = 0.0f;
            wb.all_o[o + idx] = make_float4(F.x, F.y, F.z, tmax);
            wb.all_d[o + idx] = make_float4(dir.x, dir.y, dir.z, __uint_as_float((p << 12) | ((s - 1u) << 6) | (t - 1u)));
        }
    }
    for (int of = 16; of; of >>= 1) n_shadow += __shfl_xor_sync(0xffffffffu, n_shadow, of);
    if (lane == 0 && n_shadow) atomicAdd(&dc->shadow_rays, n_shadow);
}

// FS_FLAG_SHARE_LISTENER: the listener subpaths of a call are traced once (lis_mode 1), kept as [D+1][n_paths] records +
// end points, and copied into the side-1 slots of every source batch (lis_mode 2) before its connection stage
__global__ void k_lis_store(const fs_trace_params tp, const fs_wave_buffers wb, fs_dev_counters* __restrict__ dc)
{
    const uint32_t stride = 2u * wb.cap;
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        unsigned long long ext = 0;
        for (uint32_t k = 0; k < tp.max_depth; ++k) ext += wb.q_count[k];
        atomicAdd(&dc->ext_rays, ext);
    }
    for (uint32_t p = blockIdx.x * blockDim.x + threadIdx.x; p < tp.batch; p += gridDim.x * blockDim.x) {
        const uint64_t i = tp.g_first + p;
        const float4 e = wb.end_pos[2u * p + 1u];
        tp.lis_end[i] = e;
        const uint32_t n = __float_as_uint(e.w);
        for (uint32_t k = 1; k < n; ++k) tp.lis_rec[(size_t)k * tp.n_paths + i] = wb.rec[(size_t)k * stride + 2u * p + 1u];
    }
}
__global__ void k_lis_load(const fs_trace_params tp, const fs_wave_buffers wb)
{
    const uint32_t stride = 2u * wb.cap;
    for (uint32_t p = blockIdx.x * blockDim.x + threadIdx.x; p < tp.batch; p += gridDim.x * blockDim.x) {
        const uint64_t i = listener_key(tp, wb, p);
        const float4 e = tp.lis_end[i];
        wb.end_pos[2u * p + 1u] = e;
        const uint32_t n = __float_as_uint(e.w);
        for (uint32_t k = 1; k < n; ++k) wb.rec[(size_t)k * stride + 2u * p + 1u] = tp.lis_rec[(size_t)k * tp.n_paths + i];
    }
}

// max_depth == 0: no ray is ever extended, both subpaths consist of node 0 only
__global__ void k_init_ends(const fs_trace_params tp, const fs_wave_buffers wb)
{
    uint32_t sp = blockIdx.x * blockDim.x + threadIdx.x;
    if (sp >= 2u * tp.batch) return;
    float x, y, z;
    if (sp & 1u) { x = tp.lis[0]; y = tp.lis[1]; z = tp.lis[2]; }
    else {
        const uint32_t s = pair_source(tp, wb, sp >> 1);
        x = tp.src_pos[3 * s]; y = tp.src_pos[3 * s + 1]; z = tp.src_pos[3 * s + 2];
    }
    wb.end_pos[sp] = make_float4(x, y, z, __uint_as_float(1u));
}

// reset_dc: bit 0 = the per-call counters, bit 1 = the overflow flag too (left alone while the host has not yet seen the
// flag of the previous call)
__global__ void k_reset_queues(uint32_t* q_count, uint32_t* q_cursor, uint32_t n, fs_dev_counters* dc, int reset_dc)
{
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) { q_count[i] = 0u; q_cursor[i] = 0u; }
    if (reset_dc && i == 0) {
        dc->ext_rays = 0; dc->shadow_rays = 0; dc->connected = 0; dc->node_visits = 0; dc->tri_tests = 0;
        dc->shadow_node_visits = 0; dc->shadow_tri_tests = 0;
        if (reset_dc & 2) dc->overflow = 0;
        dc->max_steps = 0;
        for (int b = 0; b < 16; ++b) dc->steps_hist[b] = 0;
    }
}

// single rays (intersector parity tests)
template <int MODE>
__global__ void __launch_bounds__(WF_THREADS)
k_debug_rays(const fs_trace_params tp, const float* __restrict__ rays, const float* __restrict__ tmax,
             uint64_t n, float* __restrict__ out_t, uint32_t* __restrict__ out_tri, uint8_t* __restrict__ out_hit,
             fs_dev_counters* __restrict__ dc)
{
    extern __shared__ float4 smem_top[];
    if (MODE == MODE_TOP) stage_top(tp, smem_top);
    fs_visit_counters vc; vc.nodes = 0; vc.tris = 0;
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        fs_vec3 o = fs_mk(rays[i * 6 + 0], rays[i * 6 + 1], rays[i * 6 + 2]);
        fs_vec3 d = fs_mk(rays[i * 6 + 3], rays[i * 6 + 4], rays[i * 6 + 5]);
        uint32_t ovf = 0;
        if (out_hit) {
            out_hit[i] = trace_any<false, MODE>(tp, smem_top, o, d, tmax[i], &vc, &ovf) ? 1 : 0;
        } else {
            float t;
            int tri = trace_closest<false, MODE>(tp, smem_top, o, d, t, &vc, &ovf);
            out_t[i] = t;
            out_tri[i] = tri >= 0 ? __ldg(tp.bv.tri_orig + tri) : 0xffffffffu;
        }
        if (ovf) dc->overflow = 1u;
    }
}


// ---- debug rays through the PRODUCTION traversal kernels (intersector parity tests) ----
__global__ void k_dbg_pack(const float* __restrict__ rays, const float* __restrict__ tmax, uint64_t n,
                           float4* __restrict__ ro, float4* __restrict__ rd, uint32_t* __restrict__ count, uint8_t* __restrict__ out_hit)
{
    const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (i == 0) *count = (uint32_t)n;
    if (i >= n) return;
    const float w0 = tmax ? tmax[i] : __uint_as_float((uint32_t)i);
    ro[i] = make_float4(rays[i * 6 + 0], rays[i * 6 + 1], rays[i * 6 + 2], w0);
    rd[i] = make_float4(rays[i * 6 + 3], rays[i * 6 + 4], rays[i * 6 + 5], tmax ? __uint_as_float((uint32_t)i) : 0.f);
    if (out_hit) out_hit[i] = 1;          // any-hit: rays the kernel reports as unoccluded are cleared afterwards
}
__global__ void k_dbg_unpack_closest(const fs_bvh_view bv, const float2* __restrict__ hits, uint64_t n,
                                     float* __restrict__ out_t, uint32_t* __restrict__ out_tri)
{
    const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int tri = __float_as_int(hits[i].y);
    out_t[i] = hits[i].x;
    out_tri[i] = tri >= 0 ? bv.tri_orig[tri] : 0xffffffffu;
}
__global__ void k_dbg_unpack_any(const uint32_t* __restrict__ conn, const uint32_t* __restrict__ conn_count, uint8_t* __restrict__ out_hit)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < *conn_count) out_hit[conn[i]] = 0;
}

template <typename K>
int resident_ctas(const fs_ctx* ctx, K kernel, int threads, size_t smem)
{
    int n = 0;
    if (smem > 48 * 1024) cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    // experiment knob: shared-memory carve-out in percent of the 228 KB (the rest is L1); default = the driver's choice
    if (ctx->tune.carveout != -1) cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, ctx->tune.carveout);
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, kernel, threads, smem) != cudaSuccess || n < 1) n = 1;
    return n;
}

// Grid of a persistent traversal launch: `kernel`'s resident CTAs on every SM (shared by `lanes` batch lanes that run at
// the same time), at most `max_ctas`, at least one.  Each instantiation's occupancy is looked up once per context.
template <typename K>
uint32_t tr_grid(fs_ctx* ctx, K kernel, size_t smem, uint32_t max_ctas, uint32_t lanes = 1)
{
    int& occ = ctx->resident[reinterpret_cast<const void*>(kernel)];
    if (!occ) occ = resident_ctas(ctx, kernel, TR_THREADS, smem);
    const uint32_t grid = (uint32_t)(ctx->sm_count * occ) / lanes;
    return grid > max_ctas ? (max_ctas ? max_ctas : 1) : grid;
}

// FS_FLAG_TIME_KERNELS: the next n events of one of a context's event pools, which grows as needed
cudaEvent_t* take_events(std::vector<cudaEvent_t>& pool, size_t& used, size_t n)
{
    if (pool.size() < used + n) {
        const size_t old = pool.size();
        pool.resize(used + n);
        for (size_t i = old; i < pool.size(); ++i) cudaEventCreate(&pool[i]);
    }
    cudaEvent_t* ev = &pool[used];
    used += n;
    return ev;
}

// Closest-hit rays (origin, direction + tmax; ray count and work cursor on the device) through the kernel `tr` names;
// (t, triangle) records to `hit`
template <bool COUNT>
void launch_closest(fs_ctx* ctx, const fs_traversal& tr, uint32_t max_ctas, cudaStream_t st, const fs_bvh_view& bv,
                    const float4* ro, const float4* rd, const uint32_t* count, uint32_t* cursor, float2* hit)
{
    const fs_tune& t = ctx->tune;
    auto queue = [&](auto kernel, size_t smem) {
        kernel<<<tr_grid(ctx, kernel, smem, max_ctas), TR_THREADS, smem, st>>>(bv, ro, rd, count, cursor, hit, nullptr, nullptr, nullptr,
                                                                             ctx->d_counters, t.refill, t.tq_node_min, t.tq_flush);
    };
    auto phased = [&](auto kernel) {
        kernel<<<tr_grid(ctx, kernel, TR_SMEM_CLOSEST, max_ctas), TR_THREADS, TR_SMEM_CLOSEST, st>>>(bv, ro, rd, count, cursor, hit,
                                                                             ctx->d_counters, t.refill, t.node_min, t.tri_min);
    };
    const bool tex = tr.closest_tex == 2;
    if (tr.closest_q && tr.nodes == FS_NODES_W8) queue(k_trace_q<COUNT, 0, false, true>, TR_SMEM_TQ8);
    else if (tr.closest_q) tex ? queue(k_trace_q<COUNT, 2, false, false>, TR_SMEM_TQ) : queue(k_trace_q<COUNT, 0, false, false>, TR_SMEM_TQ);
    else if (tr.nodes != FS_NODES_BVH2) tex ? phased(k_trace_closest<COUNT, 2, true>) : phased(k_trace_closest<COUNT, 0, true>);
    else tex ? phased(k_trace_closest<COUNT, 2, false>) : phased(k_trace_closest<COUNT, 0, false>);
}

// Any-hit rays (origin, direction + tmax; ray count and work cursor on the device) through the kernel `tr` names; the ids of
// the unoccluded rays are appended to conn[], counted by *conn_count
template <bool COUNT>
void launch_any(fs_ctx* ctx, const fs_traversal& tr, uint32_t max_ctas, cudaStream_t st, const fs_bvh_view& bv,
                const float4* ro, const float4* rd, const uint32_t* count, uint32_t* cursor, uint32_t* conn, uint32_t* conn_count,
                fs_path_dbg* dbg)
{
    const fs_tune& t = ctx->tune;
    auto queue = [&](auto kernel, size_t smem) {
        kernel<<<tr_grid(ctx, kernel, smem, max_ctas), TR_THREADS, smem, st>>>(bv, ro, rd, count, cursor, nullptr, conn, conn_count, dbg,
                                                                             ctx->d_counters, t.refill, t.tq_node_min, t.tq_flush);
    };
    auto phased = [&](auto kernel) {
        kernel<<<tr_grid(ctx, kernel, TR_SMEM_ANY, max_ctas), TR_THREADS, TR_SMEM_ANY, st>>>(bv, ro, rd, count, cursor, conn, conn_count,
                                                                             ctx->d_counters, dbg, t.refill, t.node_min);
    };
    const bool tex = tr.any_tex == 2;
    if (tr.any_q && tr.nodes == FS_NODES_W8) queue(k_trace_q<COUNT, 0, true, true>, TR_SMEM_TQ8);
    else if (tr.any_q) tex ? queue(k_trace_q<COUNT, 2, true, false>, TR_SMEM_TQ) : queue(k_trace_q<COUNT, 0, true, false>, TR_SMEM_TQ);
    else if (tr.nodes != FS_NODES_BVH2) tex ? phased(k_trace_any<COUNT, 2, true>) : phased(k_trace_any<COUNT, 0, true>);
    else tex ? phased(k_trace_any<COUNT, 2, false>) : phased(k_trace_any<COUNT, 0, false>);
}

int pick_mode(const fs_trace_params& tp)
{
    if (tp.flags & FS_FLAG_BRUTE_FORCE) return MODE_BRUTE;
    if ((tp.flags & FS_FLAG_SMEM_TREELET) && tp.n_top >= 2) return MODE_TOP;
    return MODE_BVH;
}

}  // namespace

fs_traversal fs_choose_traversal(const fs_tune& t, const fs_bvh_device& b)
{
    fs_traversal c = {};
    c.tex = t.tex != 0;
    c.nodes = !(t.wide && b.wnodes) ? FS_NODES_BVH2 : (t.w8 && b.w8nodes) ? FS_NODES_W8 : FS_NODES_W4;
    // queue entries are single triangles: 4-wide nodes with single-triangle leaves, or the 8-wide nodes (such leaves by construction)
    c.closest_q = t.tq && (c.nodes == FS_NODES_W8 || (c.nodes == FS_NODES_W4 && b.max_leaf == 1));
    c.any_q = c.closest_q && t.tq >= 2;
    // TEX 2 needs the texture handle of the node array the kernel walks; the 8-wide kernels have no texture path
    const bool w8q = c.closest_q && c.nodes == FS_NODES_W8;
    const bool has_tex = (c.nodes == FS_NODES_BVH2 ? b.nodes_tex : b.wnodes_tex) != 0;
    c.closest_tex = (has_tex && !w8q && t.tex >= 2) ? 2 : 0;
    c.any_tex = (has_tex && !(w8q && c.any_q) && t.tex != 0) ? 2 : 0;
    return c;
}

cudaError_t fs_wave_alloc(fs_ctx* ctx, fs_lane* lane, uint32_t cap, uint32_t max_depth)
{
    fs_wave_buffers* wb = &lane->wb;
    if (wb->cap >= cap && wb->depth_cap >= max_depth && wb->rec) return cudaSuccess;
    if (cap < wb->cap) cap = wb->cap;
    if (max_depth < wb->depth_cap) max_depth = wb->depth_cap;
    fs_wave_free(wb);
    cudaError_t e;
    const size_t n2 = 2ull * cap;
    for (int i = 0; i < 2; ++i) {
        if ((e = cudaMalloc(&wb->st_pos[i], sizeof(float4) * n2)) != cudaSuccess) return e;
        if ((e = cudaMalloc(&wb->st_nrm[i], sizeof(float4) * n2)) != cudaSuccess) return e;
    }
    if ((e = cudaMalloc(&wb->rec, sizeof(float4) * n2 * (max_depth + 1ull))) != cudaSuccess) return e;
    if ((e = cudaMalloc(&wb->end_pos, sizeof(float4) * n2)) != cudaSuccess) return e;
    if ((e = cudaMalloc(&wb->conn_queue, 4ull * cap)) != cudaSuccess) return e;
    if ((e = cudaMalloc(&wb->conn_len, 4ull * cap)) != cudaSuccess) return e;
    if ((e = cudaMalloc(&wb->hit, sizeof(float2) * n2)) != cudaSuccess) return e;
    if ((e = cudaMalloc(&wb->q_count, 4ull * (max_depth + 4))) != cudaSuccess) return e;
    if ((e = cudaMalloc(&wb->q_cursor, 4ull * (max_depth + 4))) != cudaSuccess) return e;
    if ((e = cudaMalloc(&wb->pair_src, sizeof(uint2) * cap)) != cudaSuccess) return e;
    if (ctx->cfg.flags & (FS_FLAG_CONNECT_ALL | FS_FLAG_MIS)) {
        const uint64_t per = (uint64_t)(max_depth + 1) * (max_depth + 1);
        wb->all_cap = (uint64_t)cap * per;
        if ((e = cudaMalloc(&wb->npos, sizeof(float4) * n2 * (max_depth + 1ull))) != cudaSuccess) return e;
        if ((ctx->cfg.flags & FS_FLAG_MIS) && (e = cudaMalloc(&wb->nnrm, sizeof(float4) * n2 * (max_depth + 1ull))) != cudaSuccess) return e;
        if ((e = cudaMalloc(&wb->all_o, sizeof(float4) * wb->all_cap)) != cudaSuccess) return e;
        if ((e = cudaMalloc(&wb->all_d, sizeof(float4) * wb->all_cap)) != cudaSuccess) return e;
        if ((e = cudaMalloc(&wb->all_conn, 4ull * wb->all_cap)) != cudaSuccess) return e;
    }
    const bool mega_alloc = ctx->tune.mega == 1u || (ctx->tune.mega == 2u && cap >= FS_MEGA_MIN_BATCH && ctx->bvh.n_tris >= 4096u);
    if (mega_alloc && max_depth >= 1 && cap <= (1u << 21) && !(ctx->cfg.flags & (FS_FLAG_CONNECT_ALL | FS_FLAG_MIS | FS_FLAG_COUNT_VISITS))) {
        const uint64_t lc = (uint64_t)n2 * max_depth;                  // every subpath traces at most max_depth rays
        if (lc < 0xffffffffull) {
            wb->log_cap = (uint32_t)lc;
            if ((e = cudaMalloc(&wb->log_o, sizeof(float4) * lc)) != cudaSuccess) return e;
            if ((e = cudaMalloc(&wb->log_d, sizeof(float4) * lc)) != cudaSuccess) return e;
            if ((e = cudaMalloc(&wb->log_flag, 4ull * lc)) != cudaSuccess) return e;
            if ((e = cudaMemsetAsync(wb->log_flag, 0, 4ull * lc, lane->stream)) != cudaSuccess) return e;
            if ((e = cudaStreamSynchronize(lane->stream)) != cudaSuccess) return e;
            if ((e = cudaMalloc(&wb->pq, 16)) != cudaSuccess) return e;
            wb->pq_epoch = 0;
        }
    }
    wb->cap = cap; wb->depth_cap = max_depth;
    return cudaSuccess;
}

void fs_wave_free(fs_wave_buffers* wb)
{
    for (int i = 0; i < 2; ++i) { cudaFree(wb->st_pos[i]); cudaFree(wb->st_nrm[i]); }
    cudaFree(wb->rec); cudaFree(wb->end_pos); cudaFree(wb->conn_queue); cudaFree(wb->conn_len);
    cudaFree(wb->q_count); cudaFree(wb->q_cursor); cudaFree(wb->hit); cudaFree(wb->pair_src);
    cudaFree(wb->npos); cudaFree(wb->nnrm); cudaFree(wb->all_o); cudaFree(wb->all_d); cudaFree(wb->all_conn);
    cudaFree(wb->log_o); cudaFree(wb->log_d); cudaFree(wb->log_flag); cudaFree(wb->pq);
    memset(wb, 0, sizeof(*wb));
}

template <bool COUNT, int MODE>
static cudaError_t launch_batch(fs_ctx* ctx, fs_lane* lane, const fs_trace_params& tp, unsigned long long* d_hist,
                                fs_path_dbg* d_dbg, ulonglong2* d_m2)
{
    cudaStream_t st = lane->stream;
    const fs_wave_buffers& wb = lane->wb;
    const size_t smem = (MODE == MODE_TOP) ? (size_t)tp.n_top * 64 : 0;
    // occupancy depends on the instantiation (COUNT, MODE) and on the treelet size: queried per call, it is a host-only lookup
    const int occ_ext = resident_ctas(ctx, k_extend<COUNT, MODE>, WF_THREADS, smem);
    const int occ_con = resident_ctas(ctx, k_connect<COUNT, MODE>, WF_THREADS, smem);
    if (smem > 48 * 1024) {
        cudaFuncSetAttribute(k_extend<COUNT, MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        cudaFuncSetAttribute(k_connect<COUNT, MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    }
    const bool timing = (tp.flags & FS_FLAG_TIME_KERNELS) != 0;
    cudaEvent_t* ev = timing ? take_events(ctx->kev, ctx->kev_used, 4) : nullptr;
    const uint32_t nq = tp.max_depth + 4;
    k_reset_queues<<<(nq + 63) / 64, 64, 0, st>>>(wb.q_count, wb.q_cursor, nq, ctx->d_counters, 0);
    ctx->launches.fetch_add(1);
    // persistent grids: SMs x resident CTAs, capped by the work available
    const uint32_t warps_needed = (2u * tp.batch + 31u) / 32u;
    uint32_t grid_ext = (uint32_t)(ctx->sm_count * occ_ext);
    uint32_t ctas_needed = (warps_needed + WF_THREADS / 32 - 1) / (WF_THREADS / 32);
    if (grid_ext > ctas_needed) grid_ext = ctas_needed ? ctas_needed : 1;
    if (timing) cudaEventRecord(ev[0], st);
    if (tp.max_depth == 0) {
        k_init_ends<<<(2u * tp.batch + 255u) / 256u, 256, 0, st>>>(tp, wb);
        ctx->launches.fetch_add(1);
    }
    for (uint32_t k = 0; k < tp.max_depth; ++k) {
        k_extend<COUNT, MODE><<<grid_ext, WF_THREADS, smem, st>>>(tp, wb, k, (int)(k & 1u), ctx->d_counters);
        ctx->launches.fetch_add(1);
        ++ctx->stats.extend_launches;
    }
    if (timing) cudaEventRecord(ev[1], st);
    uint32_t grid_con = (uint32_t)(ctx->sm_count * occ_con);
    uint32_t ctas_con = ((tp.batch + 31u) / 32u + WF_THREADS / 32 - 1) / (WF_THREADS / 32);
    if (grid_con > ctas_con) grid_con = ctas_con ? ctas_con : 1;
    k_connect<COUNT, MODE><<<grid_con, WF_THREADS, smem, st>>>(tp, wb, ctx->d_counters, d_dbg);
    ctx->launches.fetch_add(1);
    if (timing) cudaEventRecord(ev[2], st);
    uint32_t grid_ev = (uint32_t)ctx->sm_count * 8u;
    const uint32_t ctas_ev = (tp.batch / 4u + WF_THREADS / 32 - 1) / (WF_THREADS / 32) + 1;
    if (grid_ev > ctas_ev) grid_ev = ctas_ev;
    const bool dir = tp.dir_orient != nullptr;
    if (dir && d_m2) k_eval<false, true, true><<<grid_ev, WF_THREADS, 0, st>>>(tp, wb, d_hist, ctx->d_counters, d_dbg, d_m2);
    else if (dir) k_eval<false, false, true><<<grid_ev, WF_THREADS, 0, st>>>(tp, wb, d_hist, ctx->d_counters, d_dbg, nullptr);
    else if (d_m2) k_eval<false, true><<<grid_ev, WF_THREADS, 0, st>>>(tp, wb, d_hist, ctx->d_counters, d_dbg, d_m2);
    else k_eval<false><<<grid_ev, WF_THREADS, 0, st>>>(tp, wb, d_hist, ctx->d_counters, d_dbg, nullptr);
    ctx->launches.fetch_add(1);
    if (timing) cudaEventRecord(ev[3], st);
    return cudaGetLastError();
}


// ---------------------------------------------------------------------------------------------
// split wavefront: shade_gen(0) trace(0) shade_gen(1) ... trace(D-1) shade_gen(D) connect_gen
// trace_any eval
// ---------------------------------------------------------------------------------------------
template <bool COUNT>
static cudaError_t launch_batch_split(fs_ctx* ctx, fs_lane* lane, const fs_trace_params& tp, unsigned long long* d_hist,
                                      fs_path_dbg* d_dbg, ulonglong2* d_m2)
{
    cudaStream_t st = lane->stream;
    fs_wave_buffers& wb = lane->wb;
    const fs_traversal& tr = ctx->trav;
    const fs_tune& t = ctx->tune;
    const bool timing = (tp.flags & FS_FLAG_TIME_KERNELS) != 0;
    cudaEvent_t* ev = timing ? take_events(ctx->kev, ctx->kev_used, 4) : nullptr;
    const uint32_t nq = tp.max_depth + 4;
    k_reset_queues<<<(nq + 63) / 64, 64, 0, st>>>(wb.q_count, wb.q_cursor, nq, ctx->d_counters, 0);
    ctx->launches.fetch_add(1);
    const uint32_t D = tp.max_depth;
    const uint32_t n_sub = 2u * tp.batch;
    uint32_t grid_sh = (n_sub + FS_SG_THREADS - 1) / FS_SG_THREADS;
    if (grid_sh > (uint32_t)ctx->sm_count * (2048u / FS_SG_THREADS)) grid_sh = (uint32_t)ctx->sm_count * (2048u / FS_SG_THREADS);
    const uint32_t ctas_needed = (n_sub + TR_THREADS - 1) / TR_THREADS;
    if (timing) cudaEventRecord(ev[0], st);
    if (D == 0) {
        k_init_ends<<<(n_sub + 255u) / 256u, 256, 0, st>>>(tp, wb);
        ctx->launches.fetch_add(1);
    } else {
        // Bounces 0 .. k0-1 run as one k_shade_gen + k_trace_q pair each.  With the persistent per-batch kernel enabled
        // (FS_TUNE_MEGA), every bounce from k0 on runs inside ONE k_path_q launch: those are the bounces where few rays are
        // left and the fixed cost of a launch pair (the drain of its slowest rays + the latency floor of k_shade_gen)
        // outweighs the work.  The timing / counting contexts keep the per-bounce pipeline for every bounce.
        // FS_TUNE_MEGA: 0 = never, 1 = always, 2 (default) = when it pays: large batches on scenes where traversal dominates
        // (measured, profiles/r2_experiments.md: room 2^20 pairs -5.7 %, hall -2.2 %; 2^16-pair jobs and the 12-triangle
        // shoebox +16 ... +32 %: one long persistent launch has a longer tail than it saves, in-kernel shading at partial warps)
        // ... and only while no convolver source is active: a persistent grid holds every SM for the whole batch (4-5 ms), an
        // audio callback issued meanwhile would wait for it (measured p99 3.6 ms); between per-bounce kernels it waits 0.3 ms
        const bool mega_ok = t.mega == 1u || (t.mega == 2u && tp.batch >= FS_MEGA_MIN_BATCH && tp.bv.n_tris >= 4096u &&
                                              ctx->conv_active.load() == 0);
        const bool mega = !COUNT && tr.closest_q && wb.log_o && mega_ok && (uint64_t)n_sub * D <= wb.log_cap;
        const uint32_t k0 = mega ? (t.mega_from < D ? t.mega_from : D) : D;
        for (uint32_t k = 0; k <= D; ++k) {
            k_shade_gen<<<grid_sh, FS_SG_THREADS, 0, st>>>(tp, wb, k, ctx->d_counters);
            ctx->launches.fetch_add(1);
            if (k == D) break;
            if (k == k0) {
                const uint32_t epoch = ++wb.pq_epoch;
                pq_globals* g = (pq_globals*)wb.pq;
                k_pq_seed<<<ctx->sm_count * 4, 256, 0, st>>>(wb, wb.log_o, wb.log_d, wb.log_flag, epoch, g, k0);
                cudaEvent_t* te = timing ? take_events(ctx->tev, ctx->tev_used, 2) : nullptr;
                if (timing) cudaEventRecord(te[0], st);   // the persistent launch is the "traversal launch" of this batch
                // the flag / ticket protocol does not need the whole grid resident (any resident warp can take any ray);
                // with several batch lanes each lane's persistent grid gets its share of the SMs
                auto path_q = [&](auto kernel, size_t smem) {
                    const uint32_t grid = tr_grid(ctx, kernel, smem, ctas_needed, ctx->cur_lanes ? ctx->cur_lanes : 1u);
                    kernel<<<grid, TR_THREADS, smem, st>>>(tp, wb, wb.log_o, wb.log_d, wb.log_flag, epoch, wb.log_cap, g,
                                                           t.refill, t.tq_node_min, t.tq_flush);
                };
                if (tr.nodes == FS_NODES_W8) path_q(k_path_q<0, true>, PQ_SMEM8);
                else tr.closest_tex == 2 ? path_q(k_path_q<2, false>, PQ_SMEM) : path_q(k_path_q<0, false>, PQ_SMEM);
                if (timing) cudaEventRecord(te[1], st);
                ctx->stats.persistent_launches += 1;
                k_pq_finish<<<1, 1, 0, st>>>(wb, g, D, ctx->d_counters, k0);
                ctx->launches.fetch_add(3);
                ctx->stats.extend_launches += 1;
                break;
            }
            cudaEvent_t* te = timing ? take_events(ctx->tev, ctx->tev_used, 2) : nullptr;
            if (timing) cudaEventRecord(te[0], st);
            launch_closest<COUNT>(ctx, tr, ctas_needed, st, tp.bv, wb.st_pos[k & 1u], wb.st_nrm[k & 1u], wb.q_count + k,
                                  wb.q_cursor + k, wb.hit);
            if (timing) cudaEventRecord(te[1], st);
            ctx->launches.fetch_add(1);
            ++ctx->stats.extend_launches;
        }
    }
    if (timing) cudaEventRecord(ev[1], st);
    uint32_t grid_cg = (tp.batch + WF_THREADS - 1) / WF_THREADS;
    if (grid_cg > (uint32_t)ctx->sm_count * 8u) grid_cg = (uint32_t)ctx->sm_count * 8u;
    if (!grid_cg) grid_cg = 1;
    if (tp.lis_mode == 1) {                       // listener pass: keep the subpaths, no connection
        k_lis_store<<<grid_cg, WF_THREADS, 0, st>>>(tp, wb, ctx->d_counters);
        ctx->launches.fetch_add(1);
        if (timing) { cudaEventRecord(ev[2], st); cudaEventRecord(ev[3], st); }
        return cudaGetLastError();
    }
    if (tp.lis_mode == 2) { k_lis_load<<<grid_cg, WF_THREADS, 0, st>>>(tp, wb); ctx->launches.fetch_add(1); }
    const bool all = (tp.flags & (FS_FLAG_CONNECT_ALL | FS_FLAG_MIS)) != 0;        // every prefix pair (s, t) instead of the two end points
    if (all) {
        uint32_t grid_ca = (tp.batch + WF_THREADS / 32 - 1) / (WF_THREADS / 32);          // one warp per path pair
        if (grid_ca > (uint32_t)ctx->sm_count * 8u) grid_ca = (uint32_t)ctx->sm_count * 8u;
        k_connect_all_gen<<<grid_ca ? grid_ca : 1, WF_THREADS, 0, st>>>(tp, wb, ctx->d_counters);
    }
    else k_connect_gen<<<grid_cg, WF_THREADS, 0, st>>>(tp, wb, ctx->d_counters, d_dbg);
    const uint32_t ctas_any = all ? ~0u : (tp.batch + TR_THREADS - 1) / TR_THREADS;   // `all`: the ray count is known on the device only
    const float4* any_o = all ? wb.all_o : wb.st_pos[0];
    const float4* any_d = all ? wb.all_d : wb.st_nrm[0];
    uint32_t* any_conn = all ? wb.all_conn : wb.conn_queue;
    launch_any<COUNT>(ctx, tr, ctas_any, st, tp.bv, any_o, any_d, wb.q_count + (D + 2), wb.q_cursor + (D + 2), any_conn,
                      wb.q_count + (D + 1), all ? nullptr : d_dbg);
    ctx->launches.fetch_add(2);
    if (timing) cudaEventRecord(ev[2], st);
    uint32_t grid_ev = (uint32_t)ctx->sm_count * 8u;
    const uint32_t ctas_ev = (tp.batch / 4u + WF_THREADS / 32 - 1) / (WF_THREADS / 32) + 1;   // 4 paths per warp
    if (!all && grid_ev > ctas_ev) grid_ev = ctas_ev;
    if (tp.dir_orient) {                          // directional sources: the same kernels, each band starting at its gain
        if (tp.flags & FS_FLAG_MIS) k_eval_mis<true><<<grid_ev, WF_THREADS, 0, st>>>(tp, wb, d_hist, ctx->d_counters);
        else if (all) k_eval<true, false, true><<<grid_ev, WF_THREADS, 0, st>>>(tp, wb, d_hist, ctx->d_counters, nullptr, nullptr);
        else if (d_m2) k_eval<false, true, true><<<grid_ev, WF_THREADS, 0, st>>>(tp, wb, d_hist, ctx->d_counters, d_dbg, d_m2);
        else k_eval<false, false, true><<<grid_ev, WF_THREADS, 0, st>>>(tp, wb, d_hist, ctx->d_counters, d_dbg, nullptr);
    }
    else if (tp.flags & FS_FLAG_MIS) k_eval_mis<false><<<grid_ev, WF_THREADS, 0, st>>>(tp, wb, d_hist, ctx->d_counters);
    else if (all) k_eval<true><<<grid_ev, WF_THREADS, 0, st>>>(tp, wb, d_hist, ctx->d_counters, nullptr, nullptr);
    else if (d_m2) k_eval<false, true><<<grid_ev, WF_THREADS, 0, st>>>(tp, wb, d_hist, ctx->d_counters, d_dbg, d_m2);
    else k_eval<false><<<grid_ev, WF_THREADS, 0, st>>>(tp, wb, d_hist, ctx->d_counters, d_dbg, nullptr);
    ctx->launches.fetch_add(1);
    if (timing) cudaEventRecord(ev[3], st);
    return cudaGetLastError();
}

cudaError_t fs_wave_trace_batch(fs_ctx* ctx, fs_lane* lane, const fs_trace_params& tp, unsigned long long* d_hist,
                                fs_path_dbg* d_dbg, ulonglong2* d_m2)
{
    const bool count = (tp.flags & FS_FLAG_COUNT_VISITS) != 0;
    if (tp.src_off) {
        k_resolve_sources<<<(tp.batch + 255u) / 256u, 256, 0, lane->stream>>>(tp, lane->wb);
        ctx->launches.fetch_add(1);
    }
    if (!(tp.flags & (FS_FLAG_FUSED_EXTEND | FS_FLAG_BRUTE_FORCE)))
        return count ? launch_batch_split<true>(ctx, lane, tp, d_hist, d_dbg, d_m2)
                     : launch_batch_split<false>(ctx, lane, tp, d_hist, d_dbg, d_m2);
    switch (pick_mode(tp)) {
    case MODE_BRUTE: return launch_batch<false, MODE_BRUTE>(ctx, lane, tp, d_hist, d_dbg, d_m2);
    case MODE_TOP:
        return count ? launch_batch<true, MODE_TOP>(ctx, lane, tp, d_hist, d_dbg, d_m2)
                     : launch_batch<false, MODE_TOP>(ctx, lane, tp, d_hist, d_dbg, d_m2);
    default:
        return count ? launch_batch<true, MODE_BVH>(ctx, lane, tp, d_hist, d_dbg, d_m2)
                     : launch_batch<false, MODE_BVH>(ctx, lane, tp, d_hist, d_dbg, d_m2);
    }
}

// reset of the per-call device counters (first batch of a trace call)
cudaError_t fs_wave_reset_counters(fs_ctx* ctx, int reset_overflow)
{
    k_reset_queues<<<1, 64, 0, ctx->stream>>>(nullptr, nullptr, 0, ctx->d_counters, reset_overflow ? 3 : 1);
    ctx->launches.fetch_add(1);
    return cudaGetLastError();
}

cudaError_t fs_wave_debug_rays(fs_ctx* ctx, const fs_trace_params& tp, const float* d_rays, const float* d_tmax,
                               uint64_t n, float* d_t, uint32_t* d_tri, uint8_t* d_hit)
{
    cudaStream_t st = ctx->stream;
    const int mode = pick_mode(tp);
    if (!(tp.flags & (FS_FLAG_FUSED_EXTEND | FS_FLAG_BRUTE_FORCE)) && n < 0xffffffffull) {
        // default: the traversal kernels the trace chose for this tree and these knobs (ctx->trav)
        float4 *ro = nullptr, *rd = nullptr; float2* hits = nullptr; uint32_t *misc = nullptr, *conn = nullptr;
        cudaError_t e;
        if ((e = cudaMalloc(&ro, sizeof(float4) * n)) != cudaSuccess) return e;
        if ((e = cudaMalloc(&rd, sizeof(float4) * n)) != cudaSuccess) { cudaFree(ro); return e; }
        if ((e = cudaMalloc(&hits, sizeof(float2) * n)) != cudaSuccess) { cudaFree(ro); cudaFree(rd); return e; }
        if ((e = cudaMalloc(&conn, 4 * n)) != cudaSuccess) { cudaFree(ro); cudaFree(rd); cudaFree(hits); return e; }
        if ((e = cudaMalloc(&misc, 4 * 4)) != cudaSuccess) { cudaFree(ro); cudaFree(rd); cudaFree(hits); cudaFree(conn); return e; }
        cudaMemsetAsync(misc, 0, 16, st);            // [0] ray count, [1] cursor, [2] connected count
        const uint32_t g = (uint32_t)((n + 255) / 256);
        k_dbg_pack<<<g, 256, 0, st>>>(d_rays, d_hit ? d_tmax : nullptr, n, ro, rd, misc, d_hit);
        const uint32_t ctas = (uint32_t)((n + TR_THREADS - 1) / TR_THREADS);
        if (d_hit) {
            launch_any<false>(ctx, ctx->trav, ctas, st, tp.bv, ro, rd, misc, misc + 1, conn, misc + 2, nullptr);
            k_dbg_unpack_any<<<g, 256, 0, st>>>(conn, misc + 2, d_hit);
        } else {
            launch_closest<false>(ctx, ctx->trav, ctas, st, tp.bv, ro, rd, misc, misc + 1, hits);
            k_dbg_unpack_closest<<<g, 256, 0, st>>>(tp.bv, hits, n, d_t, d_tri);
        }
        ctx->launches.fetch_add(3);
        e = cudaStreamSynchronize(st);
        cudaFree(ro); cudaFree(rd); cudaFree(hits); cudaFree(conn); cudaFree(misc);
        return e != cudaSuccess ? e : cudaGetLastError();
    }
    const size_t smem = (mode == MODE_TOP) ? (size_t)tp.n_top * 64 : 0;
    uint32_t grid = (uint32_t)((n + WF_THREADS - 1) / WF_THREADS);
    if (grid > (uint32_t)ctx->sm_count * 8u) grid = (uint32_t)ctx->sm_count * 8u;
    if (!grid) grid = 1;
    if (mode == MODE_BRUTE) k_debug_rays<MODE_BRUTE><<<grid, WF_THREADS, 0, st>>>(tp, d_rays, d_tmax, n, d_t, d_tri, d_hit, ctx->d_counters);
    else if (mode == MODE_TOP) {
        if (smem > 48 * 1024) cudaFuncSetAttribute(k_debug_rays<MODE_TOP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        k_debug_rays<MODE_TOP><<<grid, WF_THREADS, smem, st>>>(tp, d_rays, d_tmax, n, d_t, d_tri, d_hit, ctx->d_counters);
    } else k_debug_rays<MODE_BVH><<<grid, WF_THREADS, 0, st>>>(tp, d_rays, d_tmax, n, d_t, d_tri, d_hit, ctx->d_counters);
    ctx->launches.fetch_add(1);
    return cudaGetLastError();
}
