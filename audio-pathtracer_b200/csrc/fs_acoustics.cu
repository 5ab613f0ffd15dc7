// fs_acoustics.cu -- room-acoustic parameters of the energy histogram (fs_get_acoustic_params): Schroeder decay curve,
// EDT / T20 / T30 fits, C50 / C80 / D50 and centre time per (source, band or broadband slot).  Semantics in
// include/frequensee.h, finishing arithmetic in fs_acoustics.h.
//
// One CTA per slot.  Thread t owns the contiguous bins [t c, (t + 1) c), c = ceil(K / AP_THREADS), so any K up to 2^20 works:
//   pass 1: exact 128-bit chunk sum and the chunk's first non-empty bin; a suffix scan over the threads gives every chunk
//           R at its start, thread 0's is S0; the onset k0 is a min reduction;
//   pass 2: R_k walked through the chunk; ka / kb of every fit are min / max reductions of the per-chunk candidates;
//   pass 3: R_k again; the fit sums sum w L, sum L, sum L^2 (levels relative to R_ka, fs_ap_fit_level), the exact
//           early-window and centre-time sums, the EDC.
// Integer sums are exact; the double sums are reduced by one fixed tree, so a histogram gives the same bytes every time.
#include "fs_internal.h"
#include "fs_acoustics.h"

namespace {

constexpr int AP_THREADS = 256;

struct u128 { unsigned long long lo, hi; };

__device__ __forceinline__ void add128(u128& a, u128 b) { a.lo += b.lo; a.hi += b.hi + (a.lo < b.lo ? 1ull : 0ull); }
__device__ __forceinline__ void sub128(u128& a, u128 b) { const unsigned long long br = a.lo < b.lo ? 1ull : 0ull; a.lo -= b.lo; a.hi -= b.hi + br; }

// E_k of slot c: band c, or the 128-bit band sum for c == B
__device__ __forceinline__ u128 load_e(const unsigned long long* __restrict__ h, uint32_t c, uint32_t B, uint32_t K, uint32_t k)
{
    u128 e{0ull, 0ull};
    if (c < B) { e.lo = h[(size_t)c * K + k]; return e; }
    for (uint32_t b = 0; b < B; ++b) add128(e, u128{h[(size_t)b * K + k], 0ull});
    return e;
}

__device__ __forceinline__ u128 reduce128(u128 v, unsigned long long* sh_lo, unsigned long long* sh_hi)
{
    __syncthreads();
    sh_lo[threadIdx.x] = v.lo; sh_hi[threadIdx.x] = v.hi;
    __syncthreads();
    for (int w = AP_THREADS / 2; w > 0; w >>= 1) {
        if ((int)threadIdx.x < w) {
            u128 a{sh_lo[threadIdx.x], sh_hi[threadIdx.x]};
            add128(a, u128{sh_lo[threadIdx.x + w], sh_hi[threadIdx.x + w]});
            sh_lo[threadIdx.x] = a.lo; sh_hi[threadIdx.x] = a.hi;
        }
        __syncthreads();
    }
    return u128{sh_lo[0], sh_hi[0]};
}

// min (is_max = false) or max of a signed value over the CTA
__device__ __forceinline__ int reduce_ext(int v, bool is_max, int* sh)
{
    __syncthreads();
    sh[threadIdx.x] = v;
    __syncthreads();
    for (int w = AP_THREADS / 2; w > 0; w >>= 1) {
        if ((int)threadIdx.x < w) {
            const int o = sh[threadIdx.x + w];
            sh[threadIdx.x] = is_max ? max(sh[threadIdx.x], o) : min(sh[threadIdx.x], o);
        }
        __syncthreads();
    }
    return sh[0];
}

__device__ __forceinline__ double reduce_d(double v, double* sh)
{
    __syncthreads();
    sh[threadIdx.x] = v;
    __syncthreads();
    for (int w = AP_THREADS / 2; w > 0; w >>= 1) {
        if ((int)threadIdx.x < w) sh[threadIdx.x] += sh[threadIdx.x + w];
        __syncthreads();
    }
    return sh[0];
}

__global__ void __launch_bounds__(AP_THREADS)
k_acoustics(const unsigned long long* __restrict__ hist, uint32_t n_bands, uint32_t n_bins, double delta, uint32_t n50,
            uint32_t n80, fs_acoustic_slot* __restrict__ out, float* __restrict__ edc)
{
    __shared__ unsigned long long sh_lo[AP_THREADS], sh_hi[AP_THREADS];
    __shared__ double sh_d[AP_THREADS];
    __shared__ int sh_i[AP_THREADS];
    __shared__ unsigned long long sh_ra[2 * FS_AP_FITS];   // R at the first point of every fit
    const uint32_t B = n_bands, K = n_bins, t = threadIdx.x;
    const uint32_t s = blockIdx.x / (B + 1u), c = blockIdx.x % (B + 1u);
    const unsigned long long* h = hist + (size_t)s * B * K;
    float* e_out = edc ? edc + (size_t)blockIdx.x * K : nullptr;
    const uint32_t chunk = (K + AP_THREADS - 1u) / AP_THREADS;
    const uint32_t k_beg = min(t * chunk, K), k_end = min(k_beg + chunk, K);

    // pass 1: chunk sums and onset candidates
    u128 sum{0ull, 0ull};
    int first = INT_MAX;
    for (uint32_t k = k_beg; k < k_end; ++k) {
        const u128 e = load_e(h, c, B, K, k);
        if (first == INT_MAX && (e.lo | e.hi)) first = (int)k;
        add128(sum, e);
    }
    // inclusive suffix scan of the chunk sums: R at the start of every chunk
    sh_lo[t] = sum.lo; sh_hi[t] = sum.hi;
    __syncthreads();
    for (uint32_t off = 1; off < AP_THREADS; off <<= 1) {
        u128 v{0ull, 0ull};
        if (t + off < AP_THREADS) v = u128{sh_lo[t + off], sh_hi[t + off]};
        __syncthreads();
        u128 a{sh_lo[t], sh_hi[t]};
        add128(a, v);
        sh_lo[t] = a.lo; sh_hi[t] = a.hi;
        __syncthreads();
    }
    const u128 r0{sh_lo[t], sh_hi[t]}, s0{sh_lo[0], sh_hi[0]};
    const int k0 = reduce_ext(first, false, sh_i);
    if (k0 == INT_MAX) {                                   // no energy: the record of an empty slot
        if (e_out) for (uint32_t k = k_beg; k < k_end; ++k) e_out[k] = __int_as_float(0x7fc00000);
        if (t == 0) {
            fs_ap_sums a{};
            a.k0 = FS_AP_NO_ONSET; a.n_bins = K; a.n50 = n50; a.n80 = n80;
            fs_acoustic_slot o;
            fs_ap_finish(&a, delta, &o);
            out[blockIdx.x] = o;
        }
        return;
    }
    const double s0d = fs_ap_u128(s0.hi, s0.lo);
    double thr_hi[FS_AP_FITS], thr_lo[FS_AP_FITS];
#pragma unroll
    for (int i = 0; i < FS_AP_FITS; ++i) { thr_hi[i] = s0d * fs_ap_c_hi(i); thr_lo[i] = s0d * fs_ap_c_lo(i); }

    // pass 2: fit points
    int ka[FS_AP_FITS], kb[FS_AP_FITS];
#pragma unroll
    for (int i = 0; i < FS_AP_FITS; ++i) { ka[i] = (int)K; kb[i] = -1; }
    {
        u128 r = r0;
        for (uint32_t k = k_beg; k < k_end; ++k) {
            const double rd = fs_ap_u128(r.hi, r.lo);
#pragma unroll
            for (int i = 0; i < FS_AP_FITS; ++i) {
                if ((int)k >= k0 && ka[i] == (int)K && rd <= thr_hi[i]) ka[i] = (int)k;
                if (k + 2u <= K && rd >= thr_lo[i]) kb[i] = (int)k;
            }
            sub128(r, load_e(h, c, B, K, k));
        }
    }
#pragma unroll
    for (int i = 0; i < FS_AP_FITS; ++i) { ka[i] = reduce_ext(ka[i], false, sh_i); kb[i] = reduce_ext(kb[i], true, sh_i); }
    for (int i = 0; i < FS_AP_FITS; ++i)
        if (ka[i] >= (int)k_beg && ka[i] < (int)k_end) {
            u128 r = r0;
            for (uint32_t k = k_beg; k < (uint32_t)ka[i]; ++k) sub128(r, load_e(h, c, B, K, k));
            sh_ra[2 * i] = r.lo; sh_ra[2 * i + 1] = r.hi;
        }
    __syncthreads();

    // pass 3: fit sums, early windows, centre-time moment, EDC
    double fs[FS_AP_FITS][3];
#pragma unroll
    for (int i = 0; i < FS_AP_FITS; ++i) fs[i][0] = fs[i][1] = fs[i][2] = 0.0;
    u128 e50{0ull, 0ull}, e80{0ull, 0ull}, ts{0ull, 0ull};
    {
        u128 r = r0;
        for (uint32_t k = k_beg; k < k_end; ++k) {
            const u128 e = load_e(h, c, B, K, k);
            const double L = fs_ap_level_db(fs_ap_u128(r.hi, r.lo), s0d);
            if ((int)k >= k0) {
                const unsigned long long d = k - (uint32_t)k0;
                if (d < n50) add128(e50, e);
                if (d < n80) add128(e80, e);
                add128(ts, u128{e.lo * d, __umul64hi(e.lo, d) + e.hi * d});
            }
#pragma unroll
            for (int i = 0; i < FS_AP_FITS; ++i)
                if ((int)k >= ka[i] && (int)k <= kb[i]) {
                    const u128 ra{sh_ra[2 * i], sh_ra[2 * i + 1]};
                    u128 drop = ra;
                    sub128(drop, r);
                    const double l = fs_ap_fit_level(fs_ap_u128(drop.hi, drop.lo), fs_ap_u128(ra.hi, ra.lo));
                    const double w = (double)(2 * (int)k - ka[i] - kb[i]);
                    fs[i][0] += w * l; fs[i][1] += l; fs[i][2] += l * l;
                }
            if (e_out) e_out[k] = (int)k < k0 ? 0.0f : (float)L;
            sub128(r, e);
        }
    }
    fs_ap_sums a;
#pragma unroll
    for (int i = 0; i < FS_AP_FITS; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) a.fit[i][j] = reduce_d(fs[i][j], sh_d);
    const u128 e50s = reduce128(e50, sh_lo, sh_hi), e80s = reduce128(e80, sh_lo, sh_hi), tss = reduce128(ts, sh_lo, sh_hi);
    if (t == 0) {
        const u128 last = load_e(h, c, B, K, K - 1u);
        a.k0 = (uint32_t)k0; a.n_bins = K; a.n50 = n50; a.n80 = n80;
#pragma unroll
        for (int i = 0; i < FS_AP_FITS; ++i) { a.ka[i] = (uint32_t)ka[i]; a.kb[i] = kb[i]; }
        a.s0_hi = s0.hi; a.s0_lo = s0.lo; a.last_hi = last.hi; a.last_lo = last.lo;
        a.e50_hi = e50s.hi; a.e50_lo = e50s.lo; a.e80_hi = e80s.hi; a.e80_lo = e80s.lo; a.ts_hi = tss.hi; a.ts_lo = tss.lo;
        fs_acoustic_slot o;
        fs_ap_finish(&a, delta, &o);
        out[blockIdx.x] = o;
    }
}

}  // namespace

cudaError_t fs_acoustics_run(const unsigned long long* d_hist, uint32_t n_sources, uint32_t n_bands, uint32_t n_bins, float bin_ms,
                             fs_acoustic_slot* d_out, float* d_edc, cudaStream_t st)
{
    k_acoustics<<<n_sources * (n_bands + 1u), AP_THREADS, 0, st>>>(d_hist, n_bands, n_bins, (double)bin_ms * 1e-3,
                                                                   fs_ap_window(50.0, bin_ms), fs_ap_window(80.0, bin_ms), d_out, d_edc);
    return cudaGetLastError();
}
