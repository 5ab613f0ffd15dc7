// fs_noise.cu -- Monte Carlo noise of an update (FS_FLAG_NOISE_STATS) and the ray budgets allocated from it.
//
// In the endpoint-connection mode every path pair adds at most one connected path, i.e. one Q32.32 value q_b to exactly one
// bin of every band.  The histogram S1 is the sum of q over the pairs, k_eval<false, true> accumulates the exact sum of q^2
// (S2, 128 bits).  With n pairs of a source, per bin:
//     mu = S1 / n,   Var(mu_hat) = (S2 / n - mu^2) / (n - 1) = (n S2 - S1^2) / (n^2 (n - 1))
// (the numerator is formed exactly in 192-bit integers, so it is never negative), converted to energy units (2^-32 for
// S1, 2^-64 for S2).  signal = sum_k mu_k^2, variance = sum_k Var_k.  This is the sample-based SNR by which Cao et al.
// judge ray-based propagation and distribute the next frame's samples.
#include "fs_internal.h"

#include <algorithm>
#include <cmath>
#include <vector>

namespace {

constexpr int NOISE_THREADS = 256;

// one CTA per (source, band or broadband slot): a fixed-order double reduction over the bins
__global__ void __launch_bounds__(NOISE_THREADS)
k_noise_reduce(const unsigned long long* __restrict__ hist, const ulonglong2* __restrict__ m2, const uint64_t* __restrict__ n_src,
               uint32_t n_bands, uint32_t n_bins, double* __restrict__ out)
{
    __shared__ double sh_sig[NOISE_THREADS], sh_var[NOISE_THREADS];
    const uint32_t s = blockIdx.x / (n_bands + 1u), c = blockIdx.x % (n_bands + 1u);
    const uint64_t n = n_src[s];
    const double dn = (double)n;
    const double den = dn * dn * (double)(n > 1 ? n - 1 : 1);
    const unsigned long long* h = hist + (size_t)s * n_bands * n_bins;
    const ulonglong2* q = m2 + ((size_t)s * (n_bands + 1u) + c) * n_bins;
    double sig = 0.0, var = 0.0;
    for (uint32_t k = threadIdx.x; k < n_bins; k += NOISE_THREADS) {
        // S1 as (s1, s1h): the broadband S1 is the sum of the band histograms, which can pass 2^64 before any band does
        unsigned long long s1 = 0ull, s1h = 0ull;
        if (c < n_bands) s1 = h[(size_t)c * n_bins + k];
        else for (uint32_t b = 0; b < n_bands; ++b) { const unsigned long long v = h[(size_t)b * n_bins + k]; s1 += v; s1h += s1 < v ? 1ull : 0ull; }
        const ulonglong2 s2 = q[k];
        // n * S2 (192 bits) - S1^2 (192 bits: s1h <= 7)
        const unsigned long long p0 = n * s2.x, c0 = __umul64hi(n, s2.x);
        unsigned long long p1 = n * s2.y + c0;
        unsigned long long p2 = __umul64hi(n, s2.y) + (p1 < c0 ? 1ull : 0ull);
        unsigned long long a0 = s1 * s1, a1 = __umul64hi(s1, s1), a2 = s1h * s1h;
        const unsigned long long t0 = s1 * (2ull * s1h), t1 = __umul64hi(s1, 2ull * s1h);   // 2 s1 s1h 2^64
        a1 += t0; a2 += t1 + (a1 < t0 ? 1ull : 0ull);
        const unsigned long long d0 = p0 - a0;
        unsigned long long br = p0 < a0 ? 1ull : 0ull;
        const unsigned long long d1 = p1 - a1 - br;
        br = (p1 < a1 || (p1 == a1 && br)) ? 1ull : 0ull;
        const unsigned long long d2 = p2 - a2 - br;
        const bool neg = p2 < a2 || (p2 == a2 && br);   // only if a sum has wrapped: no estimate rather than a wrong one
        const double num = neg ? 0.0 : ((double)d2 * 0x1p128 + (double)d1 * 0x1p64 + (double)d0);
        const double mu = ((double)s1h * 0x1p64 + (double)s1) * 0x1p-32 / dn;
        sig += mu * mu;
        var += num * 0x1p-64 / den;
    }
    sh_sig[threadIdx.x] = sig; sh_var[threadIdx.x] = var;
    __syncthreads();
    for (int w = NOISE_THREADS / 2; w > 0; w >>= 1) {
        if ((int)threadIdx.x < w) { sh_sig[threadIdx.x] += sh_sig[threadIdx.x + w]; sh_var[threadIdx.x] += sh_var[threadIdx.x + w]; }
        __syncthreads();
    }
    if (threadIdx.x == 0) { out[2 * blockIdx.x] = sh_sig[0]; out[2 * blockIdx.x + 1] = sh_var[0]; }
}

}  // namespace

cudaError_t fs_noise_reduce(const unsigned long long* d_hist, const ulonglong2* d_m2, const uint64_t* d_n, uint32_t n_sources,
                            uint32_t n_bands, uint32_t n_bins, double* d_out, cudaStream_t st)
{
    k_noise_reduce<<<n_sources * (n_bands + 1u), NOISE_THREADS, 0, st>>>(d_hist, d_m2, d_n, n_bands, n_bins, d_out);
    return cudaGetLastError();
}

extern "C" int fs_allocate_paths(const fs_noise_stats* st, uint32_t n_sources, uint64_t total, uint64_t min_paths,
                                 uint64_t max_paths, const float* weight, uint64_t* n_out)
{
    const uint32_t S = n_sources;
    if (!st || !n_out || S == 0 || min_paths == 0 || min_paths > max_paths) return FS_ERR_INVALID;
    if ((unsigned __int128)S * min_paths > total || (unsigned __int128)S * max_paths < total) return FS_ERR_INVALID;
    if (weight)
        for (uint32_t s = 0; s < S; ++s)
            if (!std::isfinite(weight[s]) || weight[s] < 0.0f) return FS_ERR_INVALID;
    auto clampn = [&](uint64_t v) { return v < min_paths ? min_paths : v > max_paths ? max_paths : v; };
    // a source with no energy keeps its previous count (clamped) as long as the others can still take the rest
    std::vector<char> pool(S, 1);
    uint64_t kept = 0, n_kept = 0;
    for (uint32_t s = 0; s < S; ++s)
        if (st[s].no_energy) { pool[s] = 0; kept += clampn(st[s].n_paths); ++n_kept; }
    uint64_t R = total - (kept <= total ? kept : total);
    const uint64_t n_pool = S - n_kept;
    if (kept > total || (unsigned __int128)n_pool * min_paths > R || (unsigned __int128)n_pool * max_paths < R) {
        std::fill(pool.begin(), pool.end(), 1);   // no feasible split that keeps them: every source joins the pool
        R = total;
    } else {
        for (uint32_t s = 0; s < S; ++s) if (!pool[s]) n_out[s] = clampn(st[s].n_paths);
    }
    // demand d_s = w_s a_s with a_s = n_s / snr_lin_s = n_s variance_s / signal_s: Var ~ a_s / n, so n_s ~ d_s equalises
    // the weighted SNR.  Sources without energy that are in the pool (see above), noise-free sources and sources of weight 0
    // demand 0; a source whose a_s overflows (signal far below its variance) demands the most there is: it is served first.
    std::vector<double> d(S, 0.0);
    std::vector<char> inf_demand(S, 0);
    for (uint32_t s = 0; s < S; ++s) {
        if (!pool[s] || st[s].no_energy || !(st[s].signal > 0.0)) continue;
        const double w = weight ? (double)weight[s] : 1.0;
        const double a = (double)st[s].n_paths * st[s].variance / st[s].signal;
        if (w > 0.0 && !std::isfinite(a)) inf_demand[s] = 1;
        else d[s] = w * a;
    }
    // water-filling over a set M: x_s = clamp(lambda dd_s, min, max) with sum x_s = budget.  The sum is monotone in lambda;
    // lambda is found by bisection on log(lambda) between "all at min" and "all at max", which stays finite for any
    // positive demands (a denormal one included).  When even every member at max does not reach the budget, all are at max.
    std::vector<double> x(S, 0.0);
    auto fill = [&](const std::vector<uint32_t>& M, const std::vector<double>& dd, double budget) {
        if (M.empty()) return;
        double lmin = INFINITY, lmax = -INFINITY;
        for (uint32_t s : M) { lmin = std::min(lmin, std::log(dd[s])); lmax = std::max(lmax, std::log(dd[s])); }
        auto xs = [&](double t, uint32_t s) { return std::min(std::max(std::exp(t + std::log(dd[s])), (double)min_paths), (double)max_paths); };
        auto f = [&](double t) { double v = 0.0; for (uint32_t s : M) v += xs(t, s); return v; };
        double lo = std::log((double)min_paths) - lmax, hi = std::log((double)max_paths) - lmin;
        for (int it = 0; it < 200; ++it) {
            const double mid = 0.5 * (lo + hi);
            if (f(mid) < budget) lo = mid; else hi = mid;
        }
        for (uint32_t s : M) x[s] = xs(hi, s);
    };
    // the pool in priority order: I (infinite demand), P (positive demand), Z (no demand); each class takes what is left
    // once the classes after it hold min_paths, and at most max_paths per source
    std::vector<uint32_t> I, P, Z;
    for (uint32_t s = 0; s < S; ++s) if (pool[s]) (inf_demand[s] ? I : d[s] > 0.0 ? P : Z).push_back(s);
    const std::vector<double> ones(S, 1.0);
    double left = (double)R;
    const std::vector<uint32_t>* cls[3] = {&I, &P, &Z};
    for (int k = 0; k < 3; ++k) {
        double after = 0.0;
        for (int j = k + 1; j < 3; ++j) after += (double)cls[j]->size() * (double)min_paths;
        const double cap = (double)cls[k]->size() * (double)max_paths;
        const double budget = std::min(cap, left - after);
        fill(*cls[k], k == 1 ? d : ones, budget);
        for (uint32_t s : *cls[k]) left -= x[s];
    }
    // largest remainder: floors, then one more path to the largest fractional parts until the sum is R exactly
    std::vector<uint32_t> idx;
    int64_t rem = (int64_t)R;
    for (uint32_t s = 0; s < S; ++s) if (pool[s]) {
        uint64_t v = (uint64_t)std::floor(x[s]);
        v = clampn(v);
        n_out[s] = v; rem -= (int64_t)v;
        idx.push_back(s);
    }
    std::stable_sort(idx.begin(), idx.end(), [&](uint32_t a, uint32_t b) { return x[a] - std::floor(x[a]) > x[b] - std::floor(x[b]); });
    while (rem > 0) {                             // one pass normally; more only if the bisection left a whole path over
        bool moved = false;
        for (uint32_t s : idx) if (rem > 0 && n_out[s] < max_paths) { ++n_out[s]; --rem; moved = true; }
        if (!moved) break;
    }
    while (rem < 0) {
        bool moved = false;
        for (auto it = idx.rbegin(); it != idx.rend(); ++it) if (rem < 0 && n_out[*it] > min_paths) { --n_out[*it]; ++rem; moved = true; }
        if (!moved) break;
    }
    return rem == 0 ? FS_OK : FS_ERR_INVALID;
}
