// fs_ir.cu -- energy histogram -> impulse response.
//
// Replaces UFrequenSeeAudioComponent::ReconstructImpulseResponse (COMP.cpp:320-380):
//   k_energy : E_k = (sum_b hist[b][k]) * 2^-32 / n_paths   (1/N of SUB.cpp:164 applied after the
//              integer reduction), a_k = E_k / sqrt(E_k * sqrt(4 pi)) if |E_k| >= threshold else 0
//              (COMP.cpp:339-346)
//   k_ir     : sample j of bin k: (1-w) a_{k-1} + w a_k, w = j/48 (COMP.cpp:347-363; FIX: 48
//              samples per bin, the reference's ceil(0.001f*48000.f) is 49); one-pole low-pass
//              y_i = 0.25 x_i + 0.75 y_{i-1}, y_0 = x_0 (COMP.cpp:366-375) evaluated per output
//              sample over a warm-up window of W taps, (1 - a)^W <= 1e-12 (a = 0.25: W = 128; fs_ctx::ir_window);
//              output = filtered, un-normalised (COMP.cpp:377-378); every channel gets the same
//              mono IR (COMP.cpp:327-330).
// Algorithmic bytes per update: read B*K*8, write C*sample_rate*4.
#include "fs_internal.h"
#include <math.h>
#include <vector>

namespace {

__global__ void k_energy(const unsigned long long* __restrict__ hist, uint32_t n_bands, uint32_t n_bins,
                         double inv_scale, const float* __restrict__ energy_in, float threshold,
                         float* __restrict__ amp)
{
    uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n_bins) return;
    float e;
    if (energy_in) e = energy_in[k];
    else {
        unsigned long long s = 0;
        for (uint32_t b = 0; b < n_bands; ++b) s += hist[(size_t)b * n_bins + k];
        e = (float)(((double)s * (1.0 / 4294967296.0)) * inv_scale);
    }
    const float Pi4 = sqrtf(4.0f * FS_PI);
    float a = 0.0f;
    if (fabsf(e) >= threshold) a = e / sqrtf(e * Pi4);
    amp[k] = a;
}

__device__ __forceinline__ float raw_sample(const float* __restrict__ amp, uint32_t i, uint32_t spb, uint32_t n_bins)
{
    uint32_t bin = i / spb, jj = i - bin * spb;
    if (bin >= n_bins) return 0.0f;
    float e = amp[bin];
    float pe = bin ? amp[bin - 1] : e;
    float w = (float)jj / (float)spb;
    return (1.0f - w) * pe + w * e;
}

// One CTA = IR_TILE consecutive samples.  The raw (ramp) samples of the tile and of the IR_WINDOW samples before it are
// computed once into shared memory (one integer + one float division each), then every thread runs its W-tap low-pass
// recurrence from shared memory -- same operations in the same order as evaluating raw_sample() per tap, 8x faster.
constexpr int IR_TILE = 256;
__device__ __forceinline__ void ir_tile(const float* __restrict__ amp, uint32_t n_bins, uint32_t spb, uint32_t n_samples,
                                        uint32_t n_channels, float a, float* __restrict__ ir, float* sraw, const uint32_t IR_WINDOW)
{
    const uint32_t t0 = blockIdx.x * IR_TILE;
    const uint32_t first = t0 >= (uint32_t)IR_WINDOW ? t0 - IR_WINDOW : 0u;      // first sample held in sraw
    const uint32_t cnt = t0 + IR_TILE - first;
    for (uint32_t q = threadIdx.x; q < cnt; q += blockDim.x) sraw[q] = raw_sample(amp, first + q, spb, n_bins);
    __syncthreads();
    const uint32_t i = t0 + threadIdx.x;
    if (i >= n_samples) return;
    const uint32_t j0 = i >= (uint32_t)IR_WINDOW ? i - IR_WINDOW : 0u;
    float y = sraw[j0 - first];
    if (j0 > 0) y = a * y;
    for (uint32_t j = j0 + 1; j <= i; ++j) y = a * sraw[j - first] + (1.0f - a) * y;
    for (uint32_t c = 0; c < n_channels; ++c) ir[(size_t)c * n_samples + i] = y;
}

__global__ void __launch_bounds__(IR_TILE)
k_ir(const float* __restrict__ amp, uint32_t n_bins, uint32_t spb, uint32_t n_samples,
     uint32_t n_channels, float a, float* __restrict__ ir, uint32_t win)
{
    extern __shared__ float sraw[];                        // [IR_TILE + win]
    ir_tile(amp, n_bins, spb, n_samples, n_channels, a, ir, sraw, win);
}

// ---- per-band synthesis (SURVEY 8f rank 2): band envelopes x band-limited noise carriers ------------------------
// amp[b][k] = the mapping of COMP.cpp:339-346 applied to band b alone
__global__ void k_energy_bands(const unsigned long long* __restrict__ hist, uint32_t n_bands, uint32_t n_bins,
                               double inv_scale, float threshold, float* __restrict__ amp)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_bands * n_bins) return;
    const float e = (float)(((double)hist[i] * (1.0 / 4294967296.0)) * inv_scale);
    const float Pi4 = sqrtf(4.0f * FS_PI);
    amp[i] = (fabsf(e) >= threshold) ? e / sqrtf(e * Pi4) : 0.0f;
}

// ir[c][t] = sum_b ramp_b[t] * carrier[c][b][t]; the ramp is COMP.cpp:347-363 per band, no low-pass (band-limited carriers)
__global__ void k_ir_bands(const float* __restrict__ amp, const float* __restrict__ carriers, uint32_t n_bands,
                           uint32_t n_bins, uint32_t spb, uint32_t n_samples, uint32_t n_channels, float* __restrict__ ir)
{
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_samples) return;
    const uint32_t bin = t / spb, j = t - bin * spb;
    const float w = (float)j / (float)spb;
    for (uint32_t c = 0; c < n_channels; ++c) {
        float acc = 0.0f;
        if (bin < n_bins)
            for (uint32_t b = 0; b < n_bands; ++b) {
                const float e = amp[b * n_bins + bin], pe = bin ? amp[b * n_bins + bin - 1] : e;
                const float raw = (1.0f - w) * pe + w * e;
                acc = acc + raw * carriers[((size_t)c * n_bands + b) * n_samples + t];
            }
        ir[(size_t)c * n_samples + t] = acc;
    }
}

// ---- all sources of a multi-emitter update in one launch each (config 4: 64 sources x 58 us of tiny serial launches) ----
__global__ void k_energy_multi(const unsigned long long* __restrict__ hist, uint32_t n_bands, uint32_t n_bins, fs_scale_table inv_scale,
                               float threshold, float* __restrict__ amp /*[S][K]*/)
{
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x, src = blockIdx.y;
    if (k >= n_bins) return;
    const unsigned long long* h = hist + (size_t)src * n_bands * n_bins;
    unsigned long long sum = 0;
    for (uint32_t b = 0; b < n_bands; ++b) sum += h[(size_t)b * n_bins + k];
    const float e = (float)(((double)sum * (1.0 / 4294967296.0)) * inv_scale.v[src]);
    const float Pi4 = sqrtf(4.0f * FS_PI);
    amp[(size_t)src * n_bins + k] = (fabsf(e) >= threshold) ? e / sqrtf(e * Pi4) : 0.0f;
}

__global__ void __launch_bounds__(IR_TILE)
k_ir_multi(const float* __restrict__ amp, uint32_t n_bins, uint32_t spb, uint32_t n_samples,
           uint32_t n_channels, float a, fs_ptr_table tab, uint32_t win)
{
    extern __shared__ float sraw[];                        // [IR_TILE + win]
    const uint32_t src = blockIdx.y;
    ir_tile(amp + (size_t)src * n_bins, n_bins, spb, n_samples, n_channels, a, (float*)tab.p[src], sraw, win);
}

// FS_FLAG_IR_NORMALIZE (NormalizeImpulseResponse, COMP.cpp:382-406): one CTA per (channel, source); sum of squares in double
// over a fixed tree, then every sample divided by the float norm; a channel below 1e-4 is left alone
__global__ void __launch_bounds__(1024)
k_ir_normalize(fs_ptr_table tab, float* single, uint32_t n_samples)
{
    __shared__ double red[1024];
    float* ir = (single ? single : (float*)tab.p[blockIdx.y]) + (size_t)blockIdx.x * n_samples;
    double s = 0.0;
    for (uint32_t i = threadIdx.x; i < n_samples; i += 1024) { const double v = (double)ir[i]; s += v * v; }
    red[threadIdx.x] = s;
    __syncthreads();
    for (uint32_t w = 512; w; w >>= 1) {
        if (threadIdx.x < w) red[threadIdx.x] += red[threadIdx.x + w];
        __syncthreads();
    }
    const float norm = (float)sqrt(red[0]);
    if (norm < 1e-4f) return;
    for (uint32_t i = threadIdx.x; i < n_samples; i += 1024) ir[i] = ir[i] / norm;
}

static void ir_normalize(fs_ctx* ctx, const fs_ptr_table* tab, uint32_t n, float* single)
{
    if (!(ctx->cfg.flags & FS_FLAG_IR_NORMALIZE)) return;
    fs_ptr_table t0; memset(&t0, 0, sizeof(t0));
    k_ir_normalize<<<dim3(ctx->cfg.n_channels, n), 1024, 0, ctx->stream>>>(tab ? *tab : t0, single, ctx->cfg.sample_rate);
    ctx->launches.fetch_add(1);
}

}  // namespace

// same arithmetic as fs_ir_build, for sources [s0, s0 + n) (n <= FS_PTR_TABLE): d_ir[i] = device IR of source s0 + i,
// normalised by inv_scale.v[i] (1 / the path count of that source)
cudaError_t fs_ir_build_multi(fs_ctx* ctx, const unsigned long long* d_hist, uint32_t s0, uint32_t n, const fs_scale_table& inv_scale,
                              const fs_ptr_table& d_ir)
{
    const fs_config& c = ctx->cfg;
    cudaError_t e;
    if (ctx->amp_all_cap < n) {
        cudaFree(ctx->d_amp_all); ctx->d_amp_all = nullptr;
        if ((e = cudaMalloc(&ctx->d_amp_all, sizeof(float) * (size_t)FS_PTR_TABLE * c.n_bins)) != cudaSuccess) return e;
        ctx->amp_all_cap = FS_PTR_TABLE;
    }
    const uint32_t spb = (uint32_t)((double)c.bin_ms * 1e-3 * c.sample_rate + 0.5);
    k_energy_multi<<<dim3((c.n_bins + 255) / 256, n), 256, 0, ctx->stream>>>(d_hist + (size_t)s0 * c.n_bands * c.n_bins, c.n_bands,
                                                                            c.n_bins, inv_scale, c.ir_threshold, ctx->d_amp_all);
    k_ir_multi<<<dim3((c.sample_rate + IR_TILE - 1) / IR_TILE, n), IR_TILE, sizeof(float) * (IR_TILE + ctx->ir_window), ctx->stream>>>(
        ctx->d_amp_all, c.n_bins, spb, c.sample_rate, c.n_channels, c.ir_lowpass, d_ir, ctx->ir_window);
    ctx->launches.fetch_add(2);
    ir_normalize(ctx, &d_ir, n, nullptr);
    return cudaGetLastError();
}

// Noise carriers [C][B][sample_rate]: white noise from Philox4x32-10 (counter (t/4, 'IRNZ', channel, band), key = seed)
// through two cascaded RBJ band-pass biquads (0 dB peak gain, Q = sqrt 2) at f_b = 62.5 * 2^b Hz (capped at 0.45 fs), in
// double precision on the host, scaled to unit RMS.  Depends on (seed, B, C, fs) only: built once, cached on the device.
static void band_carriers_host(const fs_config& c, uint64_t seed, std::vector<float>& out)
{
    const uint32_t NS = c.sample_rate, B = c.n_bands, Cn = c.n_channels;
    const double fs = (double)c.sample_rate;
    out.assign((size_t)Cn * B * NS, 0.0f);
    std::vector<double> y(NS);
    for (uint32_t ch = 0; ch < Cn; ++ch)
        for (uint32_t b = 0; b < B; ++b) {
            double fc = 62.5 * (double)(1u << b);
            if (fc > 0.45 * fs) fc = 0.45 * fs;
            const double w0 = 2.0 * 3.14159265358979323846 * fc / fs, q = 1.4142135623730951;
            const double alpha = sin(w0) / (2.0 * q), a0 = 1.0 + alpha;
            const double b0 = alpha / a0, b2 = -alpha / a0, a1 = -2.0 * cos(w0) / a0, a2 = (1.0 - alpha) / a0;
            double x1 = 0, x2 = 0, u1 = 0, u2 = 0, v1 = 0, v2 = 0, ss = 0;
            uint32_t r[4] = {0, 0, 0, 0};
            for (uint32_t t = 0; t < NS; ++t) {
                if ((t & 3u) == 0) fs_philox4x32_10(t >> 2, 0x49524E5Au, ch, b, (uint32_t)seed, (uint32_t)(seed >> 32), r);
                const double x = (double)r[t & 3u] * (2.0 / 4294967296.0) - 1.0;
                const double u = b0 * x + b2 * x2 - a1 * u1 - a2 * u2;
                const double v = b0 * u + b2 * u2 - a1 * v1 - a2 * v2;
                x2 = x1; x1 = x; u2 = u1; u1 = u; v2 = v1; v1 = v;
                y[t] = v; ss += v * v;
            }
            const double g = ss > 0.0 ? 1.0 / sqrt(ss / (double)NS) : 0.0;
            float* o = out.data() + ((size_t)ch * B + b) * NS;
            for (uint32_t t = 0; t < NS; ++t) o[t] = (float)(y[t] * g);
        }
}

cudaError_t fs_ir_build_bands(fs_ctx* ctx, const unsigned long long* d_hist_src, uint64_t n_paths, uint64_t noise_seed,
                              float* d_ir_out)
{
    const fs_config& c = ctx->cfg;
    cudaError_t e;
    const size_t ncar = (size_t)c.n_channels * c.n_bands * c.sample_rate;
    if (!ctx->d_carriers || ctx->carrier_seed != noise_seed) {
        std::vector<float> h;
        band_carriers_host(c, noise_seed, h);
        if (!ctx->d_carriers) {
            if ((e = cudaMalloc(&ctx->d_carriers, sizeof(float) * ncar)) != cudaSuccess) return e;
            if ((e = cudaMalloc(&ctx->d_amp_bands, sizeof(float) * c.n_bands * c.n_bins)) != cudaSuccess) return e;
        }
        if ((e = cudaMemcpyAsync(ctx->d_carriers, h.data(), sizeof(float) * ncar, cudaMemcpyHostToDevice, ctx->stream)) != cudaSuccess) return e;
        if ((e = cudaStreamSynchronize(ctx->stream)) != cudaSuccess) return e;     // h goes out of scope
        ctx->carrier_seed = noise_seed;
    }
    const uint32_t spb = (uint32_t)((double)c.bin_ms * 1e-3 * c.sample_rate + 0.5);
    const double inv_scale = n_paths ? 1.0 / (double)n_paths : 0.0;
    const uint32_t nbk = c.n_bands * c.n_bins;
    k_energy_bands<<<(nbk + 255) / 256, 256, 0, ctx->stream>>>(d_hist_src, c.n_bands, c.n_bins, inv_scale, c.ir_threshold,
                                                              ctx->d_amp_bands);
    k_ir_bands<<<(c.sample_rate + 255) / 256, 256, 0, ctx->stream>>>(ctx->d_amp_bands, ctx->d_carriers, c.n_bands, c.n_bins, spb,
                                                                      c.sample_rate, c.n_channels, d_ir_out);
    ctx->launches.fetch_add(2);
    ir_normalize(ctx, nullptr, 1, d_ir_out);
    return cudaGetLastError();
}

cudaError_t fs_ir_build(fs_ctx* ctx, const unsigned long long* d_hist_src, uint64_t n_paths,
                        const float* d_energy_in, float* d_ir_out)
{
    const fs_config& c = ctx->cfg;
    const uint32_t spb = (uint32_t)((double)c.bin_ms * 1e-3 * c.sample_rate + 0.5);
    const double inv_scale = n_paths ? 1.0 / (double)n_paths : 0.0;
    k_energy<<<(c.n_bins + 255) / 256, 256, 0, ctx->stream>>>(d_hist_src, c.n_bands, c.n_bins, inv_scale,
                                                              d_energy_in, c.ir_threshold, ctx->d_amp);
    k_ir<<<(c.sample_rate + IR_TILE - 1) / IR_TILE, IR_TILE, sizeof(float) * (IR_TILE + ctx->ir_window), ctx->stream>>>(
        ctx->d_amp, c.n_bins, spb, c.sample_rate, c.n_channels, c.ir_lowpass, d_ir_out, ctx->ir_window);
    ctx->launches.fetch_add(2);
    ir_normalize(ctx, nullptr, 1, d_ir_out);
    return cudaGetLastError();
}
