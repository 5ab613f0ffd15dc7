// fs_conv.cu -- uniformly partitioned overlap-save FFT convolution of dry audio with the IR.
//
// Replaces FFrequenSeeAudioReverbPlugin::ProcessSourceAudio + ConvolveFFT (REV.cpp:118-213) and
// FCircularAudioBuffer (CIRC.cpp:43-75).  The reference transforms a 49 023-sample history and
// the whole 48 000-tap IR with three 65 536-point KissFFTs per channel per callback; here the IR
// is cut into P = ceil(ir_len / Bk) partitions of one callback block (Bk = 1024) whose 2Bk-point
// spectra H_p are computed once per IR refresh, the input spectra X_k live in a frequency-domain
// delay line, and one callback costs one 2Bk FFT, a P-term spectral multiply-accumulate and one
// inverse FFT:   y_block = IFFT( sum_p X_{k-p} * H_p )[Bk .. 2Bk)
// which equals "history (*) current IR" on the newest block, exactly the reference's result
// (history initially zero, CIRC.cpp:15-21).  FIX: channels are de-interleaved (REV.cpp:147-148
// copies interleaved samples into both channel tails).
//
// Kernels: k_ir_spectra / k_ir_spectra_multi (grid P x C [x sources]) and k_conv_blocks (grid = sources x channels: every
// emitter of a multi-source callback in ONE launch; each CTA loops over its blocks), both on a shared-memory Stockham
// FFT with radix-4 passes (a 2048-point transform = one radix-2 + five radix-4 passes instead of eleven radix-2).
// Algorithmic bytes per block, source and channel: (P+1)*(Bk+1)*8*2 (H_p and X_{k-p} spectra) + 2*Bk*4*2.
//
// Threads: everything here that touches a source's FDL / head / published spectra runs on fs_ctx::conv_stream under
// fs_ctx::conv_mu (the audio thread); IR updates are enqueued on the context stream by the game thread and handed over
// through the (pub, pending, heard, h_ready) fields of fs_conv_source -- see fs_internal.h.
//
// FS_FLAG_CONV_CROSSFADE: a callback that adopts a new IR fades over its first block from the IR the source's previous
// callback ended with:  y = (1 - w) * IFFT(sum_p X_{k-p} G_p) + w * IFFT(sum_p X_{k-p} H_p),  w[i] = 0.5 - 0.5 cos(pi (i+1)/Bk)
// (table d_xfade).  One MAC pass reads each X_{k-p} once against both spectra sets: (P+1)(Bk+1)*8*3 + 2*Bk*4*2 bytes.
#include "fs_internal.h"

#include <math.h>
#include <new>
#include <vector>

namespace {

__device__ __forceinline__ float2 cmul(float2 a, float2 b)
{
    return make_float2(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x);
}
__device__ __forceinline__ float2 cadd(float2 a, float2 b) { return make_float2(a.x + b.x, a.y + b.y); }
__device__ __forceinline__ float2 csub(float2 a, float2 b) { return make_float2(a.x - b.x, a.y - b.y); }

// In-block Stockham autosort FFT of n = 2^logn points between two shared buffers: one radix-2 pass when logn is odd, then
// radix-4 passes.  tw[m] = exp(-2 pi i m / tw_n), m < tw_n (full circle, so the 3k-th twiddle needs no folding).
// Returns the buffer holding the result.  Inverse = conjugated twiddles and butterflies, unnormalised.
__device__ float2* fft_stockham(float2* a, float2* b, uint32_t n, const float2* __restrict__ tw, uint32_t tw_n, bool inverse)
{
    float2* in = a; float2* out = b;
    uint32_t ns = 1;
    const float sgn = inverse ? -1.0f : 1.0f;
    if (__popc(n - 1u) & 1u) {                                  // odd log2 n: one radix-2 pass (ns = 1: all twiddles are 1)
        const uint32_t half = n >> 1;
        for (uint32_t j = threadIdx.x; j < half; j += blockDim.x) {
            const float2 x0 = in[j], x1 = in[j + half];
            out[2u * j] = cadd(x0, x1);
            out[2u * j + 1u] = csub(x0, x1);
        }
        __syncthreads();
        float2* t = in; in = out; out = t;
        ns = 2;
    }
    const uint32_t quarter = n >> 2;
    for (; ns < n; ns <<= 2) {
        const uint32_t tstep = tw_n / (4u * ns);
        for (uint32_t j = threadIdx.x; j < quarter; j += blockDim.x) {
            const uint32_t k = j & (ns - 1u);
            float2 w1 = tw[k * tstep], w2 = tw[2u * k * tstep], w3 = tw[3u * k * tstep];
            w1.y *= sgn; w2.y *= sgn; w3.y *= sgn;
            const float2 x0 = in[j];
            const float2 x1 = cmul(in[j + quarter], w1);
            const float2 x2 = cmul(in[j + 2u * quarter], w2);
            const float2 x3 = cmul(in[j + 3u * quarter], w3);
            const float2 s02 = cadd(x0, x2), d02 = csub(x0, x2), s13 = cadd(x1, x3), d13 = csub(x1, x3);
            // -i * d13 (forward) / +i * d13 (inverse)
            const float2 r = make_float2(sgn * d13.y, -sgn * d13.x);
            const uint32_t j0 = ((j - k) << 2) + k;
            out[j0] = cadd(s02, s13);
            out[j0 + ns] = cadd(d02, r);
            out[j0 + 2u * ns] = csub(s02, s13);
            out[j0 + 3u * ns] = csub(d02, r);
        }
        __syncthreads();
        float2* t = in; in = out; out = t;
    }
    return in;
}

// H[p][c][f] = FFT_2Bk( ir[c][p*Bk .. (p+1)*Bk) zero-padded ) for up to FS_PTR_TABLE sources in one launch:
// tab.p[s] = device IR, tab.q[s] = destination H of source s (blockIdx.z)
__global__ void k_ir_spectra(fs_ptr_table tab, uint32_t ir_len, uint32_t bk, uint32_t n_ch,
                             const float2* __restrict__ tw, uint32_t tw_n)
{
    extern __shared__ float2 sm[];
    const uint32_t n = 2u * bk, nf = bk + 1u;
    float2* a = sm; float2* b = sm + n;
    const uint32_t p = blockIdx.x, c = blockIdx.y;
    const float* ir = (const float*)tab.p[blockIdx.z];
    float2* H = (float2*)tab.q[blockIdx.z];
    for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) {
        const uint32_t src = p * bk + i;
        float v = (i < bk && src < ir_len) ? ir[(size_t)c * ir_len + src] : 0.0f;
        a[i] = make_float2(v, 0.0f);
    }
    __syncthreads();
    float2* r = fft_stockham(a, b, n, tw, tw_n, false);
    float2* dst = H + ((size_t)p * n_ch + c) * nf;
    for (uint32_t f = threadIdx.x; f < nf; f += blockDim.x) dst[f] = r[f];
}

struct conv_src {
    float2* fdl;            // [P][C][NF]
    const float2* H;        // [P][C][NF]
    const float2* H_prev;   // FS_FLAG_CONV_CROSSFADE: the heard IR's spectra when block 0 fades from it, else null
    float* prev;            // [C][Bk] previous input block
    uint32_t head, pad;
};
struct conv_args {
    conv_src src[FS_PTR_TABLE];
    const float* in;        // [n_src][n_blocks][Bk][C] interleaved
    float* out;
    const float2* tw;
    const float* xfade;     // [Bk] fade-in window (FS_FLAG_CONV_CROSSFADE)
    uint32_t bk, n_part, n_ch, n_blocks, tw_n;
    float wet; int clamp;
};

// Spectral multiply-accumulate of bin f over partitions 1 .. P-1: acc += sum_p X_{k-p}[f] H_p[f], and with TWO also
// acc2 += sum_p X_{k-p}[f] G_p[f] from the same X loads.  The P - 1 (X, H) pairs of a bin are independent loads: four
// partitions in flight per thread.
template <bool TWO>
__device__ __forceinline__ void mac_history(const float2* __restrict__ fdl_c, const float2* __restrict__ Hc,
                                            const float2* __restrict__ Gc, size_t pstride, uint32_t P, uint32_t head,
                                            uint32_t f, float2& acc, float2& acc2)
{
    uint32_t s = head;
    uint32_t p = 1;
    for (; p + 4u <= P; p += 4u) {
        float2 xv[4], hv[4], gv[4];
#pragma unroll
        for (uint32_t u = 0; u < 4; ++u) {
            s = s ? s - 1u : P - 1u;
            xv[u] = fdl_c[(size_t)s * pstride + f];
            hv[u] = Hc[(size_t)(p + u) * pstride + f];
            if (TWO) gv[u] = Gc[(size_t)(p + u) * pstride + f];
        }
#pragma unroll
        for (uint32_t u = 0; u < 4; ++u) {
            acc.x += xv[u].x * hv[u].x - xv[u].y * hv[u].y;
            acc.y += xv[u].x * hv[u].y + xv[u].y * hv[u].x;
            if (TWO) {
                acc2.x += xv[u].x * gv[u].x - xv[u].y * gv[u].y;
                acc2.y += xv[u].x * gv[u].y + xv[u].y * gv[u].x;
            }
        }
    }
    for (; p < P; ++p) {
        s = s ? s - 1u : P - 1u;
        const float2 xv = fdl_c[(size_t)s * pstride + f];
        const float2 hv = Hc[(size_t)p * pstride + f];
        acc.x += xv.x * hv.x - xv.y * hv.y;
        acc.y += xv.x * hv.y + xv.y * hv.x;
        if (TWO) {
            const float2 gv = Gc[(size_t)p * pstride + f];
            acc2.x += xv.x * gv.x - xv.y * gv.y;
            acc2.y += xv.x * gv.y + xv.y * gv.x;
        }
    }
}

// FADE = false: the plain callback (two shared buffers).  FADE = true (FS_FLAG_CONV_CROSSFADE, launched only when some
// source of the chunk fades): a source with H_prev set computes block 0 against both IRs -- one MAC pass with two
// accumulators, two inverse FFTs, the old IR's output tail held in registers -- in three shared buffers; every other
// block, and every source without H_prev, runs the plain code.  The H_prev branch is uniform per CTA.
template <bool FADE>
__global__ void k_conv_blocks(const __grid_constant__ conv_args a)
{
    extern __shared__ float2 sm[];
    const uint32_t bk = a.bk, n = 2u * bk, nf = bk + 1u, C = a.n_ch, P = a.n_part;
    float2* s0 = sm; float2* s1 = sm + n;
    const uint32_t c = blockIdx.x, si = blockIdx.y;
    const conv_src& S = a.src[si];
    uint32_t head = S.head;
    float* prev = S.prev + (size_t)c * bk;
    const float2* __restrict__ Hc = S.H + (size_t)c * nf;
    float2* fdl_c = S.fdl + (size_t)c * nf;
    const size_t pstride = (size_t)C * nf;                   // one partition
    for (uint32_t blk = 0; blk < a.n_blocks; ++blk) {
        const bool fade = FADE && blk == 0 && S.H_prev != nullptr;
        const float* in = a.in + ((size_t)si * a.n_blocks + blk) * bk * C;
        float* out = a.out + ((size_t)si * a.n_blocks + blk) * bk * C;
        // window = previous block ++ current block (de-interleaved)
        for (uint32_t i = threadIdx.x; i < bk; i += blockDim.x) {
            const float cur = in[(size_t)i * C + c];
            s0[i] = make_float2(prev[i], 0.0f);
            s0[bk + i] = make_float2(cur, 0.0f);
            prev[i] = cur;
        }
        __syncthreads();
        float2* X = fft_stockham(s0, s1, n, a.tw, a.tw_n, false);
        float2* Y = (X == s0) ? s1 : s0;
        float2* slot = fdl_c + (size_t)head * pstride;
        // spectral multiply-accumulate over the partitions; X_k itself comes from shared memory
        if (fade) {                                               // Y = spectrum against the new IR, Z = against the heard one
            const float2* __restrict__ Gc = S.H_prev + (size_t)c * nf;
            float2* Z = sm + 2u * n;
            for (uint32_t f = threadIdx.x; f < nf; f += blockDim.x) {
                const float2 x = X[f];
                slot[f] = x;
                float2 acc = cmul(x, Hc[f]), acc2 = cmul(x, Gc[f]);
                mac_history<true>(fdl_c, Hc, Gc, pstride, P, head, f, acc, acc2);
                Y[f] = acc;
                Z[f] = acc2;
                if (f > 0 && f < bk) { Y[n - f] = make_float2(acc.x, -acc.y); Z[n - f] = make_float2(acc2.x, -acc2.y); }
            }
        } else {
            for (uint32_t f = threadIdx.x; f < nf; f += blockDim.x) {
                const float2 x = X[f];
                slot[f] = x;
                float2 acc = cmul(x, Hc[f]), unused;
                mac_history<false>(fdl_c, Hc, nullptr, pstride, P, head, f, acc, unused);
                Y[f] = acc;
                if (f > 0 && f < bk) Y[n - f] = make_float2(acc.x, -acc.y);
            }
        }
        __syncthreads();
        const float scale = 1.0f / (float)n;
        // fade: the heard IR's output tail, at most 2 samples per thread (Bk <= 2048, blockDim = min(Bk, 1024)); X is free
        float y_old[2];
        if (fade) {
            const float2* yz = fft_stockham(sm + 2u * n, X, n, a.tw, a.tw_n, true);
#pragma unroll
            for (uint32_t r = 0; r < 2; ++r) {
                const uint32_t i = threadIdx.x + r * blockDim.x;
                if (i < bk) y_old[r] = yz[bk + i].x * scale;
            }
            __syncthreads();
        }
        float2* X2 = (Y == s0) ? s1 : s0;
        float2* y = fft_stockham(Y, X2, n, a.tw, a.tw_n, true);
        if (fade) {
#pragma unroll
            for (uint32_t r = 0; r < 2; ++r) {
                const uint32_t i = threadIdx.x + r * blockDim.x;
                if (i >= bk) continue;
                const float w = a.xfade[i];
                float v = (1.0f - w) * y_old[r] + w * (y[bk + i].x * scale);
                if (a.clamp) v = fminf(fmaxf(v, -1.0f), 1.0f);
                const float dry = in[(size_t)i * C + c];
                out[(size_t)i * C + c] = v * a.wet + dry * (1.0f - a.wet);
            }
        } else {
            for (uint32_t i = threadIdx.x; i < bk; i += blockDim.x) {
                float v = y[bk + i].x * scale;
                if (a.clamp) v = fminf(fmaxf(v, -1.0f), 1.0f);               // REV.cpp:162-168
                const float dry = in[(size_t)i * C + c];
                out[(size_t)i * C + c] = v * a.wet + dry * (1.0f - a.wet);   // MixAlpha, REV.cpp:161
            }
        }
        __syncthreads();
        head = (head + 1u == P) ? 0u : head + 1u;
    }
}

__global__ void k_rfft(const float* __restrict__ in, uint32_t n, const float2* __restrict__ tw, uint32_t tw_n,
                       float2* __restrict__ out)
{
    extern __shared__ float2 sm[];
    float2* a = sm; float2* b = sm + n;
    for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) a[i] = make_float2(in[i], 0.0f);
    __syncthreads();
    float2* r = fft_stockham(a, b, n, tw, tw_n, false);
    for (uint32_t f = threadIdx.x; f <= n / 2; f += blockDim.x) out[f] = r[f];
}

size_t spectra_elems(const fs_ctx* ctx) { return (size_t)ctx->n_part * ctx->cfg.n_channels * ctx->n_freq; }
uint32_t tw_len(const fs_ctx* ctx) { return ctx->fft_n > 4096u ? ctx->fft_n : 4096u; }
int n_ir_buffers(const fs_ctx* ctx) { return (ctx->cfg.flags & FS_FLAG_CONV_CROSSFADE) ? 3 : 2; }

}  // namespace

cudaError_t fs_conv_setup(fs_ctx* ctx)
{
    const fs_config& c = ctx->cfg;
    ctx->fft_n = 2u * c.conv_block;
    ctx->n_freq = c.conv_block + 1u;
    ctx->n_part = (c.sample_rate + c.conv_block - 1u) / c.conv_block;   // IRSize = SampleRate * 1 s (REV.cpp:79)
    ctx->conv.assign(FS_MAX_SOURCES, nullptr);
    // twiddles of a 4096-point circle (covers every n <= 4096 by striding), computed in double
    const uint32_t tn = tw_len(ctx);
    std::vector<float2> tw(tn);
    for (uint32_t m = 0; m < tn; ++m) {
        double ang = -2.0 * 3.14159265358979323846 * (double)m / (double)tn;
        tw[m] = make_float2((float)cos(ang), (float)sin(ang));
    }
    cudaError_t e;
    {   // the audio thread's stream: highest priority, so its CTAs are placed first whenever a trace kernel frees an SM
        int lo = 0, hi = 0;
        if (cudaDeviceGetStreamPriorityRange(&lo, &hi) != cudaSuccess) { lo = hi = 0; (void)cudaGetLastError(); }
        if ((e = cudaStreamCreateWithPriority(&ctx->conv_stream, cudaStreamNonBlocking, hi)) != cudaSuccess) return e;
    }
    if ((e = cudaMalloc(&ctx->d_twiddle, sizeof(float2) * tw.size())) != cudaSuccess) return e;
    if ((e = cudaMemcpyAsync(ctx->d_twiddle, tw.data(), sizeof(float2) * tw.size(), cudaMemcpyHostToDevice, ctx->conv_stream)) != cudaSuccess) return e;
    if (c.flags & FS_FLAG_CONV_CROSSFADE) {   // fade-in window, computed in double: w[i] = 0.5 - 0.5 cos(pi (i+1) / Bk)
        std::vector<float> w(c.conv_block);
        for (uint32_t i = 0; i < c.conv_block; ++i)
            w[i] = (float)(0.5 - 0.5 * cos(3.14159265358979323846 * (double)(i + 1u) / (double)c.conv_block));
        if ((e = cudaMalloc(&ctx->d_xfade, sizeof(float) * w.size())) != cudaSuccess) return e;
        if ((e = cudaMemcpyAsync(ctx->d_xfade, w.data(), sizeof(float) * w.size(), cudaMemcpyHostToDevice, ctx->conv_stream)) != cudaSuccess) return e;
    }
    if ((e = cudaStreamSynchronize(ctx->conv_stream)) != cudaSuccess) return e;
    const size_t smem = sizeof(float2) * 2 * ctx->fft_n;
    if (smem > 48 * 1024) {
        if ((e = cudaFuncSetAttribute(k_ir_spectra, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)) != cudaSuccess) return e;
        if ((e = cudaFuncSetAttribute(k_conv_blocks<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)) != cudaSuccess) return e;
    }
    const size_t smem_fade = sizeof(float2) * 3 * ctx->fft_n;     // 48 KB at Bk = 1024, 96 KB at 2048
    if ((c.flags & FS_FLAG_CONV_CROSSFADE) && smem_fade > 48 * 1024)
        if ((e = cudaFuncSetAttribute(k_conv_blocks<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_fade)) != cudaSuccess) return e;
    if ((e = cudaFuncSetAttribute(k_rfft, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024)) != cudaSuccess) return e;
    return cudaSuccess;
}

void fs_conv_teardown(fs_ctx* ctx)
{
    for (uint32_t s = 0; s < ctx->conv.size(); ++s) fs_conv_source_free(ctx, s);
    cudaFree(ctx->d_twiddle); ctx->d_twiddle = nullptr;
    cudaFree(ctx->d_xfade); ctx->d_xfade = nullptr;
    cudaFree(ctx->d_conv_in); cudaFree(ctx->d_conv_out); ctx->d_conv_in = ctx->d_conv_out = nullptr;
    if (ctx->h_pin_in) cudaFreeHost(ctx->h_pin_in);
    if (ctx->h_pin_out) cudaFreeHost(ctx->h_pin_out);
    if (ctx->h_pin_ir) cudaFreeHost(ctx->h_pin_ir);
    ctx->h_pin_in = ctx->h_pin_out = ctx->h_pin_ir = nullptr;
    if (ctx->conv_stream) cudaStreamDestroy(ctx->conv_stream);
    ctx->conv_stream = nullptr;
}

// Creates the slot of `source` on first use (zero IR, zero spectra); reset_history = OnInitSource (REV.cpp:104-110;
// SetSize zeroes the ring, CIRC.cpp:15-21).  conv_mu is held by the caller.  The memsets run on conv_stream and are
// complete on return, so no later kernel on any stream can see the buffers before they are cleared.
cudaError_t fs_conv_source_alloc(fs_ctx* ctx, uint32_t source, bool reset_history)
{
    if (source >= ctx->conv.size()) return cudaErrorInvalidValue;
    cudaError_t e;
    const fs_config& c = ctx->cfg;
    const size_t sp = spectra_elems(ctx);
    cudaStream_t st = ctx->conv_stream;
    fs_conv_source* s = ctx->conv[source];
    if (!s) {
        s = new (std::nothrow) fs_conv_source();
        if (!s) return cudaErrorMemoryAllocation;
        memset(s, 0, sizeof(*s));
        s->pending = -1; s->heard = -1;
        ctx->conv[source] = s;
    }
    if (!s->fdl) {
        const int nbuf = n_ir_buffers(ctx);
        if ((e = cudaMalloc(&s->fdl, sizeof(float2) * sp)) != cudaSuccess) return e;
        for (int i = 0; i < nbuf; ++i)
            if ((e = cudaMalloc(&s->H[i], sizeof(float2) * sp)) != cudaSuccess) return e;
        if ((e = cudaMalloc(&s->prev, sizeof(float) * c.n_channels * c.conv_block)) != cudaSuccess) return e;
        if ((e = cudaMalloc(&s->ir, sizeof(float) * c.n_channels * c.sample_rate)) != cudaSuccess) return e;
        for (int i = 0; i < nbuf; ++i)
            if ((e = cudaEventCreateWithFlags(&s->h_ready[i], cudaEventDisableTiming)) != cudaSuccess) return e;
        for (int i = 0; i < nbuf; ++i)
            if ((e = cudaMemsetAsync(s->H[i], 0, sizeof(float2) * sp, st)) != cudaSuccess) return e;
        if ((e = cudaMemsetAsync(s->ir, 0, sizeof(float) * c.n_channels * c.sample_rate, st)) != cudaSuccess) return e;
        s->pub = 0; s->pending = -1; s->heard = -1;
        if ((e = cudaMemsetAsync(s->fdl, 0, sizeof(float2) * sp, st)) != cudaSuccess) return e;
        if ((e = cudaMemsetAsync(s->prev, 0, sizeof(float) * c.n_channels * c.conv_block, st)) != cudaSuccess) return e;
        s->head = 0;
    }
    if (reset_history) {                  // fs_conv_init_source: the slot becomes an audio source (an IR build alone does not)
        if ((e = cudaMemsetAsync(s->fdl, 0, sizeof(float2) * sp, st)) != cudaSuccess) return e;
        if ((e = cudaMemsetAsync(s->prev, 0, sizeof(float) * c.n_channels * c.conv_block, st)) != cudaSuccess) return e;
        s->head = 0;
        s->heard = -1;                    // the first callback of a new source starts on the published IR: no fade
        if (!s->active) ctx->conv_active.fetch_add(1);
        s->active = true;
    }
    return cudaStreamSynchronize(st);
}

void fs_conv_source_free(fs_ctx* ctx, uint32_t source)
{
    if (source >= ctx->conv.size() || !ctx->conv[source]) return;
    fs_conv_source* s = ctx->conv[source];
    if (s->active) ctx->conv_active.fetch_sub(1);
    cudaFree(s->fdl); cudaFree(s->prev); cudaFree(s->ir);
    for (int i = 0; i < 3; ++i) {
        cudaFree(s->H[i]);
        if (s->h_ready[i]) cudaEventDestroy(s->h_ready[i]);
    }
    delete s;
    ctx->conv[source] = nullptr;
}

// The buffer an IR update may write: never the published one, nor (FS_FLAG_CONV_CROSSFADE) the heard one.  A pending
// buffer whose spectra are already complete is adopted first; one that is still being computed is simply written again
// (same stream: ordered).  conv_mu held.
static int writable_buffer(fs_conv_source* s)
{
    if (s->pending >= 0 && cudaEventQuery(s->h_ready[s->pending]) == cudaSuccess) { s->pub = s->pending; s->pending = -1; }
    (void)cudaGetLastError();
    if (s->pending >= 0) return s->pending;
    int b = 0;
    while (b == s->pub || b == s->heard) ++b;      // 1 - pub without the flag (heard = -1); at most 2 with it
    return b;
}

// partition spectra of the sources' current device IRs (k_ir_spectra on `st`, the game thread's stream) into their
// unpublished buffers; the audio thread adopts each one at the first callback after its event has completed.
// sources [s0, s0 + n), n <= FS_PTR_TABLE.  conv_mu held by the caller.
cudaError_t fs_conv_update_ir_multi(fs_ctx* ctx, uint32_t s0, uint32_t n, cudaStream_t st)
{
    const fs_config& c = ctx->cfg;
    fs_ptr_table tab;
    int nxt[FS_PTR_TABLE];
    for (uint32_t i = 0; i < n; ++i) {
        fs_conv_source* s = ctx->conv[s0 + i];
        nxt[i] = writable_buffer(s);
        tab.p[i] = s->ir; tab.q[i] = s->H[nxt[i]];
    }
    const size_t smem = sizeof(float2) * 2 * ctx->fft_n;
    uint32_t threads = c.conv_block < 1024u ? c.conv_block : 1024u;
    k_ir_spectra<<<dim3(ctx->n_part, c.n_channels, n), threads, smem, st>>>(tab, c.sample_rate, c.conv_block, c.n_channels,
                                                                             ctx->d_twiddle, tw_len(ctx));
    ctx->launches.fetch_add(1);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    for (uint32_t i = 0; i < n; ++i) {
        fs_conv_source* s = ctx->conv[s0 + i];
        if ((e = cudaEventRecord(s->h_ready[nxt[i]], st)) != cudaSuccess) return e;
        s->pending = nxt[i];
    }
    return cudaSuccess;
}

cudaError_t fs_conv_update_ir(fs_ctx* ctx, uint32_t source, cudaStream_t st)
{
    return fs_conv_update_ir_multi(ctx, source, 1, st);
}

// one launch for all sources of the call (chunks of FS_PTR_TABLE); conv_mu held by the caller; st = conv_stream
cudaError_t fs_conv_run(fs_ctx* ctx, const uint32_t* sources, uint32_t n_src, const float* d_in, float* d_out, uint32_t n_blocks,
                        cudaStream_t st)
{
    const fs_config& c = ctx->cfg;
    const bool xfade = (c.flags & FS_FLAG_CONV_CROSSFADE) != 0;
    const uint32_t threads = c.conv_block < 1024u ? c.conv_block : 1024u;
    const size_t per_src = (size_t)n_blocks * c.conv_block * c.n_channels;
    for (uint32_t i0 = 0; i0 < n_src; i0 += FS_PTR_TABLE) {
        const uint32_t n = n_src - i0 < FS_PTR_TABLE ? n_src - i0 : FS_PTR_TABLE;
        conv_args a;
        bool any_fade = false;
        for (uint32_t i = 0; i < n; ++i) {
            fs_conv_source* s = ctx->conv[sources[i0 + i]];
            // adopt a finished IR update at this block boundary (never wait for one that is still being computed)
            if (s->pending >= 0 && cudaEventQuery(s->h_ready[s->pending]) == cudaSuccess) { s->pub = s->pending; s->pending = -1; }
            (void)cudaGetLastError();
            a.src[i].fdl = s->fdl; a.src[i].H = s->H[s->pub]; a.src[i].prev = s->prev; a.src[i].head = s->head; a.src[i].pad = 0;
            // fade from the IR this source's last callback ended with; both buffers stay untouched until the stream has
            // synchronised (conv_mu is held until then, and writable_buffer never returns pub or heard)
            a.src[i].H_prev = (xfade && s->heard >= 0 && s->heard != s->pub) ? s->H[s->heard] : nullptr;
            any_fade |= a.src[i].H_prev != nullptr;
            if (xfade) s->heard = s->pub;
            s->head = (s->head + n_blocks) % ctx->n_part;
        }
        a.in = d_in + i0 * per_src; a.out = d_out + i0 * per_src; a.tw = ctx->d_twiddle; a.xfade = ctx->d_xfade;
        a.bk = c.conv_block; a.n_part = ctx->n_part; a.n_ch = c.n_channels; a.n_blocks = n_blocks; a.tw_n = tw_len(ctx);
        a.wet = c.conv_wet; a.clamp = (int)c.conv_clamp;
        if (any_fade)
            k_conv_blocks<true><<<dim3(c.n_channels, n), threads, sizeof(float2) * 3 * ctx->fft_n, st>>>(a);
        else
            k_conv_blocks<false><<<dim3(c.n_channels, n), threads, sizeof(float2) * 2 * ctx->fft_n, st>>>(a);
        ctx->launches.fetch_add(1);
        cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) return e;
    }
    return cudaSuccess;
}

cudaError_t fs_conv_rfft(fs_ctx* ctx, const float* d_in, uint32_t n, float2* d_out, cudaStream_t st)
{
    uint32_t threads = n / 4 < 1024u ? n / 4 : 1024u;
    if (threads < 32u) threads = 32u;
    k_rfft<<<1, threads, sizeof(float2) * 2 * n, st>>>(d_in, n, ctx->d_twiddle, tw_len(ctx), d_out);
    ctx->launches.fetch_add(1);
    return cudaGetLastError();
}
