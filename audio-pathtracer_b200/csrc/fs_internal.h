// fs_internal.h -- context and cross-translation-unit declarations (not part of the ABI).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <string.h>
#include <string>
#include <atomic>
#include <mutex>
#include <unordered_map>
#include <vector>

#include "../../include/frequensee.h"
#include "fs_math.cuh"
#include "fs_bvh.cuh"
#include "fs_directivity.h"

#define FS_TOP_CAP 1024          // nodes of the shared-memory treelet (64 KB)

struct fs_diff_edge;             // fs_diffraction.h

struct fs_bvh_device {
    float4* nodes;
    float4* tris;
    uint32_t* tri_orig;
    uint32_t* tri_mat;
    float4* tri_nm;
    float4* top_nodes;
    cudaTextureObject_t nodes_tex, tris_tex, wnodes_tex;
    uint4* wnodes;
    float qbase[3], qscale[3];
    uint32_t n_tris, n_inner, n_top, max_leaf;
    uint32_t n_wide;             // wide nodes reachable from the root (dense breadth-first array)
    uint4* w8nodes;              // 8-wide compressed nodes (80 B each), dense breadth-first; null if not built
    float4* tris8;               // triangle records in the order the 8-wide nodes address them
    uint32_t* tri8_map;          // position in tris8 -> position in tris (the index hit records carry)
    uint32_t n_w8;
    float extent;
    int* wsrc;                   // [n_wide][4] provenance of each wide-node slot: BVH2 node * 2 + side (-1: empty slot)
    // fs_bvh_refit scratch, allocated at the first refit (callers that never refit pay nothing)
    struct refit_scratch {
        int* parent;             // [n_inner] BVH2 parent (-1: root)
        uint32_t* need;          // [n_inner] inner children
        uint32_t* arrive;        // [n_inner] arrival counters of the bottom-up pass
        float4* ubox;            // [n_inner][2] unpadded box of every inner node
        int* queue;              // [FS_TOP_CAP] k_top_treelet
        void* misc;              // double cost[2] (as committed, refitted) | float grid[8] | uint32 n_top
        double cost0;            // surface-area cost of the tree as committed
    } rf;
};

cudaError_t fs_bvh_build(cudaStream_t st, const float* d_verts, const uint32_t* d_mats, uint64_t n_tris,
                         fs_bvh_device* out, uint64_t* launches, uint32_t leaf_max, uint32_t builder /*0 LBVH, 1 PLOC*/,
                         uint32_t collapse /*wide nodes: bit 0 greedy by surface area (else grandchildren), bit 1 keep the sparse layout,
                                                    bit 2 also build the 8-wide compressed nodes, bit 3 greedy instead of optimal 8-wide collapse,
                                                    bit 4 optimal (dynamic programme) instead of greedy 4-wide collapse*/);
void fs_bvh_free(fs_bvh_device* b);
// Refits the committed tree `b` to new positions of its triangles (d_verts, same count and order as at the build): topology
// kept, triangle records, BVH2 boxes, quantisation grid, 4-wide node boxes and the treelet recomputed; one host
// synchronisation (the grid).  *cost_ratio = surface-area cost of the refitted BVH2 / that of the tree as committed.
cudaError_t fs_bvh_refit(cudaStream_t st, const float* d_verts, fs_bvh_device* b, uint64_t* launches, float* cost_ratio);

// device-side counters of one trace call
struct fs_dev_counters {
    unsigned long long ext_rays, shadow_rays, connected, node_visits, tri_tests;
    unsigned long long shadow_node_visits, shadow_tri_tests;
    uint32_t overflow, max_steps;      // max_steps: longest ray of the call in node steps (FS_FLAG_COUNT_VISITS builds)
    uint32_t steps_hist[16];           // rays by node steps: [8 i, 8 i + 8), last bucket open-ended (same builds)
};

// constant-ish parameters every wavefront kernel needs
struct fs_trace_params {
    fs_bvh_view bv;
    const float4* top;          // global copy of the treelet (staged to smem by each CTA)
    uint32_t n_top;
    const float* refl_over_pi;  // [E][M][B] factor per (event, material, band); E = 1 (reflectivity / pi) without the material model, else 3
    const float4* lobes;        // [M] (t1, t2, P_spec, P_diff) event thresholds / probabilities; null without FS_FLAG_MATERIAL_MODEL
    uint32_t n_mats;
    fs_eval_params ep;
    uint32_t n_bins;
    float bin_ms, rr_prob, eps_offset, eps_connect, sound_speed, energy_clamp, energy_gain;
    uint32_t max_depth;         // per-source budgets: the largest depth (it sizes the records, queues and bounce loops)
    uint32_t seed_lo, seed_hi;
    uint64_t n_paths;           // per source; per-source budgets: the largest budget (stride of the listener cache)
    // per-source budgets (fs_trace_sources): null = uniform, source of work index g = g / n_paths.  Otherwise every batch
    // resolves each pair's (source, depth) once into fs_wave_buffers::pair_src.
    const uint64_t* src_off;    // device [S+1]: first work index of every source, src_off[S] = G
    const uint32_t* src_depth;  // device [S]: ray budget per subpath of every source
    uint32_t n_src;
    uint64_t g_first;           // first global work index of this batch
    uint32_t batch;             // path pairs in this batch
    uint32_t cap;               // allocated path pairs (stride of per-node records = 2 * cap)
    const float* src_pos;       // device [S][3]
    float lis[3];
    uint32_t flags;
    // FS_FLAG_SHARE_LISTENER: 0 = both subpaths traced; 1 = listener pass (only side 1 is traced, then stored in the cache);
    // 2 = source pass (only side 0 is traced, side 1 is loaded from the cache before the connection)
    uint32_t lis_mode;
    float4* lis_rec;            // cache [max_depth+1][n_paths]: node records of listener subpath i
    float4* lis_end;            // cache [n_paths]: (end.xyz, bits(n_nodes))
    // directional sources (fs_set_source_directivity): null = none (k_eval<..., false>).  dir_orient [S]: (unit forward.xyz,
    // bits(pattern index or FS_OMNI)); dir_gain [P][FS_MAX_BANDS][FS_DIR_POINTS] energy gains (fs_directivity.h)
    const float4* dir_orient;
    const float* dir_gain;
    uint32_t n_dir_patterns;
};

struct fs_wave_buffers {
    float4* st_pos[2];          // ping-pong subpath state: (pos.xyz, bits(sp_id))
    float4* st_nrm[2];          //                          (nrm.xyz, bits(depth))
    float4* rec;                // [max_depth+1][2*cap]: (segment length, bits(mat), pdf, pdf^pdf_exponent) of node k of subpath sp_id
    float4* end_pos;            // [2*cap]: (end.xyz, bits(n_nodes))
    float2* hit;                // [2*cap]: closest-hit records (t, bits(sorted triangle index or -1))
    uint32_t* conn_queue;       // [cap] path ids whose connection is unoccluded
    float* conn_len;            // [cap] connection segment length, indexed by path
    uint32_t* q_count;          // [max_depth+4]: [k] rays of bounce k, [D+1] connected pairs, [D+2] shadow rays
    uint32_t* q_cursor;         // [max_depth+4] work cursors of the persistent kernels
    uint2* pair_src;            // [cap] (source, depth limit) of every pair of the batch; per-source budgets only
    uint32_t cap, depth_cap;
    // FS_FLAG_CONNECT_ALL: node positions of every subpath and the (s, t) connection rays of a batch
    float4* npos;               // [max_depth+1][2*cap]: position of node k >= 1 of subpath sp_id
    float4* nnrm;               // FS_FLAG_MIS: [max_depth+1][2*cap] surface normal (facing the arriving ray) at node k >= 1
    float4 *all_o, *all_d;      // [all_cap] connection rays (F.xyz, tmax) (dir.xyz, bits(pair << 12 | (s-1) << 6 | (t-1)))
    uint32_t* all_conn;         // [all_cap] ids of the visible connections
    uint64_t all_cap;
    // FS_TUNE_MEGA: ray log of the persistent per-batch kernel (k_path_q)
    float4 *log_o, *log_d; uint32_t* log_flag; void* pq; uint32_t log_cap, pq_epoch;
};

struct fs_conv_source {
    bool active;
    float2* fdl;                // [P][C][NF] input spectra ring
    float2* H[3];               // IR partition spectra [P][C][NF]: two buffers, a third (H[2]) only with FS_FLAG_CONV_CROSSFADE
    float* prev;                // [C][Bk] previous input block
    float* ir;                  // [C][sample_rate] device IR of this source
    // IR hand-off (game thread -> audio thread), all under fs_ctx::conv_mu: `pub` is the buffer the convolver reads;
    // `pending` (or -1) was written by the last IR update and becomes `pub` at the first callback that finds its
    // h_ready event complete -- the audio thread never waits for a trace that is still running.
    // With FS_FLAG_CONV_CROSSFADE, `heard` (or -1 after fs_conv_init_source) is the buffer the last callback ended with;
    // a callback whose `pub` differs from it fades from H[heard] to H[pub] over its first block and then sets heard = pub.
    // Invariant: an IR update writes neither `pub` nor `heard` (pending is always a third buffer), and the callback
    // reads both only under conv_mu, which it holds until the stream has synchronised.  Without the flag heard stays -1.
    int pub, pending, heard;
    cudaEvent_t h_ready[3];
    uint32_t head;              // FDL head slot
};

// smallest batch (path pairs) the persistent per-batch kernel is chosen for automatically (FS_TUNE_MEGA=2): measured break-even
// in the furnished room (2^17 pairs: 1.47 vs 1.49 ms; 2^16: 1.35 vs 1.23 ms), -14 % already at 164 k pairs in the concert hall
#define FS_MEGA_MIN_BATCH (1u << 17)
#define FS_MAX_LANES 4
#define FS_MAX_SOURCES 4096
#define FS_PTR_TABLE 64
struct fs_ptr_table { void* p[FS_PTR_TABLE]; void* q[FS_PTR_TABLE]; };   // per-source device pointers passed by value

// one batch lane: a stream and its own wavefront buffers.  Lane 0 runs on the context stream itself.
struct fs_lane { cudaStream_t stream; fs_wave_buffers wb; cudaEvent_t done; };

// Experiment knobs: the FS_TUNE_* environment variables, read once by fs_create (DESIGN.md appendix).  Out-of-range values
// of refill, leaf_max, streams and mega_lanes are ignored; tq_flush is clamped to 1..32.
struct fs_tune {
    uint32_t refill = 4;            // refill a warp once this many lanes are idle, 1..32
    uint32_t leaf_max = FS_LEAF_MAX;   // LBVH leaf size, 1..8
    uint32_t tex = 2;               // node fetches through the texture pipe: 0 none, 1 any-hit kernels, 2 every 4-wide / BVH2 kernel
    uint32_t builder = 1;           // 0 LBVH, 1 PLOC
    uint32_t wide = 1;              // 0: BVH2 float nodes
    uint32_t w8 = 0;                // 1: 8-wide compressed nodes (measured 5-10 % slower than the 4-wide nodes, profiles/r2_experiments.md)
    uint32_t node_min = 14, tri_min = 4;   // thresholds of the phased kernels
    uint32_t collapse = 17;         // bit 4: optimal (dynamic-programme) collapse of the BVH2 into 4-wide nodes: -22 % nodes, -4 % node steps
    uint32_t l2pin_mb = 0xffffffffu;   // MB of wide nodes in the persisting L2 window; 0xffffffff automatic (resolved at the first commit)
    uint32_t tq = 2;                // 0 phased kernels, 1 queue kernel for extension rays only, 2 also for connection rays
    uint32_t tq_node_min = 10;
    uint32_t tq_flush = 24;         // FS_TQ_CAP assumes <= 31 entries carried into a node step
    uint32_t mega = 2;              // one persistent launch per batch for the extension stage (k_path_q): 0 never, 1 always, 2 when it pays
    uint32_t mega_from = 0;         // first bounce inside the persistent kernel
    uint32_t mega_lanes = 2;        // batch lanes with it (2: each lane's persistent grid on half of the SMs -- one batch's connect /
                                    // evaluate stage and tail overlap the other's walk: room -2.5 %), 1..FS_MAX_LANES
    uint32_t streams = 2;           // batch lanes of the per-bounce pipeline, 1..FS_MAX_LANES
    int carveout = -1;              // shared-memory carve-out of the traversal kernels in percent (-1: the driver's choice)
};

// Node format and traversal kernels of the split wavefront and of the debug rays, chosen by fs_choose_traversal from the
// knobs and the built tree after every fs_scene_commit and fs_scene_refit
enum fs_node_format : uint8_t { FS_NODES_BVH2, FS_NODES_W4, FS_NODES_W8 };
struct fs_traversal {
    fs_node_format nodes;           // node arrays fs_bvh_view exposes: `nodes`, + `wnodes` (W4), + `w8nodes` (W8)
    bool tex;                       // fs_bvh_view carries the texture handles
    bool closest_q;                 // closest-hit rays: queue kernel k_trace_q and, per batch, k_path_q (else k_trace_closest)
    bool any_q;                     // any-hit rays: k_trace_q<ANY> (else k_trace_any)
    uint8_t closest_tex, any_tex;   // TEX of each instantiation: 2 node fetches through the texture pipe, 0 none
};
fs_traversal fs_choose_traversal(const fs_tune& t, const fs_bvh_device& b);

struct fs_ctx {
    fs_config cfg;
    int device;
    cudaStream_t own_stream, stream;
    cudaStream_t conv_stream;   // the audio thread's stream: fs_conv_process* never queues behind a trace
    // scene
    float* d_verts; uint32_t* d_tri_mat; uint64_t n_tris;
    float* d_refl_over_pi; uint32_t n_mats;
    float* d_bsdf_tab; float4* d_lobes;   // FS_FLAG_MATERIAL_MODEL: [3][M][B] diffuse / specular / transmitted factors, [M] lobe thresholds
    std::vector<float> mat_absorption;
    std::vector<float> mat_transmission, mat_scattering, mat_thickness_cm;
    bool mats_set, tris_set, committed;
    bool verts_dirty;           // fs_scene_update_vertices on a committed scene, not yet refitted: the tree no longer bounds the triangles
    fs_bvh_device bvh;
    // trace: batches alternate between lanes -- while one batch's traversal launch drains its slowest rays, the other
    // lane's kernels fill the SMs
    fs_lane lanes[FS_MAX_LANES];
    cudaEvent_t ev_fork;
    float4 *lis_rec, *lis_end; uint64_t lis_cache_n; uint32_t lis_cache_depth;   // FS_FLAG_SHARE_LISTENER cache
    unsigned long long* d_hist; uint32_t hist_sources;   // [S][B][K]; hist_sources = allocated, hist_cur_sources = valid
    uint32_t hist_cur_sources;
    uint64_t hist_n_paths;
    std::vector<uint64_t> hist_src_paths;   // per-source path counts after fs_trace_sources* (empty: every source has hist_n_paths)
    // FS_FLAG_NOISE_STATS: exact second moments of the per-pair Q32.32 contributions, [S][B+1][K] (lo, hi) mod 2^128, slot B
    // broadband.  Allocated at the first trace with the flag; m2_valid = they belong to the histogram in d_hist (set by
    // fs_trace / fs_trace_sources / fs_update* / fs_multi_trace*, cleared by every other call that writes d_hist)
    ulonglong2* d_m2; uint32_t m2_sources; bool m2_valid;
    double* d_noise; uint32_t noise_cap;    // fs_get_noise scratch: [S] path counts (u64), then [S][B+1] (signal, variance)
    void* d_acou; size_t acou_cap;          // fs_get_acoustic_params scratch: [S][B+1] records, then the [S][B+1][K] float EDC
    void* d_src_tab; uint32_t src_tab_cap;  // per-source budgets on the device: [S+1] u64 offsets, then [S] u32 depths
    // directional sources: the installed pattern table [P][FS_MAX_BANDS][FS_DIR_POINTS] and orientations [dir_sources]
    // (float4: unit forward, bits(pattern)); dir_sources = 0: none installed, every source omni
    float* d_dir_gain; uint32_t dir_patterns;
    float4* d_dir_orient; uint32_t dir_sources, dir_orient_cap;
    // fs_occlusion: transmitted factor tau_eff [M][B] of every material (built by every fs_scene_commit), and the scratch of
    // one call: [S][B+1] u64 sums, the call's own overflow flag (one u64 slot), [S] float4 sources, [S+1] u32 ray offsets
    float* d_occl_tau;
    void* d_occl; uint32_t occl_cap;
    // fs_diffraction: the edge set, built by the first call after a commit, refit or threshold change (diff_valid false
    // until then), for diff_fold_deg; and the scratch of one call: [S] float4 sources, [S] u64 best, [S] u32 path counts,
    // u64 candidate count, u64 rays, u32 overflow, [S] results; the candidate pairs
    fs_diff_edge* d_diff_edges; uint32_t n_diff_edges; float diff_fold_deg; bool diff_valid;
    void* d_diff; size_t diff_cap;
    uint2* d_diff_cand; unsigned long long diff_cand_cap;
    fs_dev_counters* d_counters;
    // traversal-stack overflow of the last trace: one 4-byte async copy into pinned memory after every fs_trace*, looked at
    // by the next call that can (sticky until reported)
    uint32_t* h_overflow; cudaEvent_t ev_overflow; bool overflow_pending;
    float* d_src_pos; uint32_t src_cap;
    fs_path_dbg* d_dbg; uint64_t dbg_cap;
    fs_stats stats;                      // game-thread fields only; kernel launches are counted in `launches`
    std::atomic<uint64_t> launches;
    std::atomic<int> conv_active;        // initialised convolver sources: while > 0 the tracer keeps to short per-bounce kernels
    cudaEvent_t ev0, ev1, ev_ir0, ev_ir1; bool timed, ir_timed;
    std::vector<cudaEvent_t> kev; size_t kev_used;   // FS_FLAG_TIME_KERNELS: 4 events per batch
    std::vector<cudaEvent_t> tev; size_t tev_used;   //   + one (begin, end) pair per k_trace_closest launch
    int sm_count;
    std::unordered_map<const void*, int> resident;   // resident CTAs per SM of every traversal kernel launched (per context = per device)
    fs_tune tune;
    fs_traversal trav;
    uint32_t cur_lanes;                  // batch lanes of the running trace call
    // IR / conv
    float* d_energy;            // [K] scratch
    float* d_amp;               // [K]
    float* d_amp_all; uint32_t amp_all_cap;   // [FS_PTR_TABLE][K]: multi-source IR build
    float* d_carriers; float* d_amp_bands; uint64_t carrier_seed;   // per-band IR synthesis: [C][B][fs] noise carriers, [B][K]
    float2* d_twiddle;          // [conv fft size / 2]
    float* d_xfade;             // FS_FLAG_CONV_CROSSFADE: [Bk] fade-in window w[i] = 0.5 - 0.5 cos(pi (i+1) / Bk)
    uint32_t fft_n, n_part, n_freq, ir_window;
    // per-source convolver state: FS_MAX_SOURCES stable slots (never reallocated: the audio thread may hold one while the
    // game thread creates another); creation, release and the IR hand-off fields are guarded by conv_mu
    std::vector<fs_conv_source*> conv;
    float *d_conv_in, *d_conv_out; size_t conv_io_cap;   // device staging [sources][blocks][frames][C]
    float *h_pin_in, *h_pin_out;
    cudaEvent_t ev_c0, ev_c1; float last_conv_ms;        // device time of the last callback's k_conv_blocks (under conv_mu)
    float* h_pin_ir; size_t pin_ir_cap;  // pinned staging for IR read-back (fs_build_ir_all: one copy for all sources)
    std::mutex conv_mu;
};

// fs_wavefront.cu
cudaError_t fs_wave_alloc(fs_ctx* ctx, fs_lane* lane, uint32_t cap, uint32_t max_depth);
void fs_wave_free(fs_wave_buffers* wb);
// d_m2: FS_FLAG_NOISE_STATS second moments [S][B+1][K] (lo, hi), accumulated by k_eval<false, true>; null = none
cudaError_t fs_wave_trace_batch(fs_ctx* ctx, fs_lane* lane, const fs_trace_params& tp, unsigned long long* d_hist,
                                fs_path_dbg* d_dbg, ulonglong2* d_m2);
cudaError_t fs_wave_reset_counters(fs_ctx* ctx, int reset_overflow);
cudaError_t fs_wave_debug_rays(fs_ctx* ctx, const fs_trace_params& tp, const float* d_rays, const float* d_tmax,
                               uint64_t n, float* d_t, uint32_t* d_tri, uint8_t* d_hit);

// fs_occlusion.cu: k_occlusion over n_rays = d_off[n_src] flat rays; d_acc [n_src][n_bands+1] must be zeroed
cudaError_t fs_occlusion_run(const fs_bvh_view& bv, const float4* d_src, const uint32_t* d_off, uint32_t n_src, uint32_t n_rays,
                             const float lis[3], const float* d_tau, uint32_t n_bands, uint32_t max_crossings, float eps_connect,
                             float eps_offset, uint64_t seed, unsigned long long* d_acc, uint32_t* d_overflow, cudaStream_t st);

// fs_bvh_build.cu: the stable LSD radix sort of the build (8 passes of 8 bits over (u64 key, u32 value); the result is back in
// keys / vals; block_hist holds 256 fs_radix_sort_blocks(n) words) and the exclusive scan (tile_sums: ceil(n / 1024) + 1
// words, *total = the sum)
uint32_t fs_radix_sort_blocks(uint32_t n);
void fs_radix_sort_u64(cudaStream_t st, uint64_t* keys, uint32_t* vals, uint64_t* keys_tmp, uint32_t* vals_tmp, uint32_t n,
                       uint32_t* block_hist, uint64_t* launches);
void fs_scan_u32(cudaStream_t st, const uint32_t* in, uint32_t* out, uint32_t n, uint32_t* tile_sums, uint32_t* total,
                 uint64_t* launches);

// fs_diffraction.cu: the edge set of the triangles d_verts [n_tris][3][3] for the fold threshold c_min, in ascending
// (tri, k) (cudaMalloc'ed into *d_edges when not empty), and one query over it
cudaError_t fs_diffraction_edges(cudaStream_t st, const float* d_verts, uint32_t n_tris, float c_min, fs_diff_edge** d_edges,
                                 uint32_t* n_out, uint64_t* launches);
#define FS_DIFF_CAND_MAX (1ull << 27)   // candidate pairs held at once (1 GB); a larger edge range is split
struct fs_diff_run {
    fs_bvh_view bv;
    const fs_diff_edge* edges; uint32_t n_edges;
    const float4* src; uint32_t n_src;            // [S] (position, -)
    float lis[3];
    float eps_offset, eps_connect, sound_speed;
    float band_hz[FS_MAX_BANDS]; uint32_t n_bands;
    uint2** cand; unsigned long long* cand_cap;   // the context's candidate buffer, grown on demand
    unsigned long long* d_count;                  // candidates of one edge range
    unsigned long long* best;                     // [S] min (bits(length) << 32 | edge rank), set to ~0 by the caller
    uint32_t* n_paths;                            // [S] zeroed by the caller
    unsigned long long* rays;                     // leg rays traced
    uint32_t* overflow;
    fs_diffraction_result* out;                   // [S] device
};
cudaError_t fs_diffraction_run(const fs_diff_run& a, cudaStream_t st, uint64_t* launches, uint64_t* n_cand_out);

// fs_ir.cu
struct fs_scale_table { double v[FS_PTR_TABLE]; };   // per-source 1 / n_paths, passed by value
cudaError_t fs_ir_build_multi(fs_ctx* ctx, const unsigned long long* d_hist, uint32_t s0, uint32_t n, const fs_scale_table& inv_scale,
                              const fs_ptr_table& d_ir);
cudaError_t fs_conv_update_ir_multi(fs_ctx* ctx, uint32_t s0, uint32_t n, cudaStream_t st);
cudaError_t fs_ir_build_bands(fs_ctx* ctx, const unsigned long long* d_hist_src, uint64_t n_paths, uint64_t noise_seed,
                              float* d_ir_out);
cudaError_t fs_ir_build(fs_ctx* ctx, const unsigned long long* d_hist_src, uint64_t n_paths,
                        const float* d_energy_in, float* d_ir_out);

// fs_noise.cu: per (source, band or broadband) sum over bins of mu^2 and of Var(mu_hat) from the histogram, the second
// moments and the per-source pair counts d_n [S]; out [S][B+1][2] (signal, variance), energy units.  Fixed-order double sums.
cudaError_t fs_noise_reduce(const unsigned long long* d_hist, const ulonglong2* d_m2, const uint64_t* d_n, uint32_t n_sources,
                            uint32_t n_bands, uint32_t n_bins, double* d_out, cudaStream_t st);

// fs_acoustics.cu: k_acoustics, one CTA per (source, band or broadband slot) of the histogram [S][B][K]; records d_out
// [S][B+1] and, when d_edc is not null, the decay curves d_edc [S][B+1][K] in dB
cudaError_t fs_acoustics_run(const unsigned long long* d_hist, uint32_t n_sources, uint32_t n_bands, uint32_t n_bins, float bin_ms,
                             fs_acoustic_slot* d_out, float* d_edc, cudaStream_t st);

// fs_conv.cu
cudaError_t fs_conv_setup(fs_ctx* ctx);
void fs_conv_teardown(fs_ctx* ctx);
// all three: conv_mu held by the caller
cudaError_t fs_conv_source_alloc(fs_ctx* ctx, uint32_t source, bool reset_history);
void fs_conv_source_free(fs_ctx* ctx, uint32_t source);
cudaError_t fs_conv_update_ir(fs_ctx* ctx, uint32_t source, cudaStream_t st);
// n_src sources x n_blocks callbacks in ONE launch (grid = sources x channels); d_in / d_out: [n_src][n_blocks][Bk][C]
cudaError_t fs_conv_run(fs_ctx* ctx, const uint32_t* sources, uint32_t n_src, const float* d_in, float* d_out, uint32_t n_blocks,
                        cudaStream_t st);
cudaError_t fs_conv_rfft(fs_ctx* ctx, const float* d_in, uint32_t n, float2* d_out, cudaStream_t st);
