// b200sd -- layout conversion, small-M linear, timestep embedding, fused CFG + scheduler step and
// image post-processing kernels (HBM / latency bound; vectorised, coalesced, one launch each).
#include "common.cuh"
#include "../../include/b200sd.h"

#include <algorithm>

namespace b200sd {

extern void count_launch(int n);

static inline int grid_for(size_t n, int threads) {
    return static_cast<int>(std::min<size_t>((n + threads - 1) / threads, static_cast<size_t>(num_sms()) * 16));
}

// ---- NCHW -> NHWC fp16 (pad channels) -------------------------------------------------------
template <typename T>
__global__ void nchw_to_nhwc_kernel(const T* __restrict__ in, __half* __restrict__ out, int n, int c, int hw,
                                    int c_pad) {
    pdl_trigger();  // no TMEM / large shared memory here: dependents may start their prologue at once
    pdl_wait();
    const size_t total = static_cast<size_t>(n) * hw * c_pad;
    for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total;
         i += static_cast<size_t>(gridDim.x) * blockDim.x) {
        const int ch = static_cast<int>(i % c_pad);
        const size_t px = i / c_pad;
        const int p = static_cast<int>(px % hw);
        const int b = static_cast<int>(px / hw);
        float v = 0.f;
        if (ch < c) v = static_cast<float>(in[(static_cast<size_t>(b) * c + ch) * hw + p]);
        out[i] = __float2half_rn(v);
    }
}

template <typename T>
__global__ void nhwc_to_nchw_f32_kernel(const T* __restrict__ in, float* __restrict__ out, int n, int c, int hw,
                                        int c_pad) {
    pdl_trigger();  // no TMEM / large shared memory here: dependents may start their prologue at once
    pdl_wait();
    const size_t total = static_cast<size_t>(n) * c * hw;
    for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total;
         i += static_cast<size_t>(gridDim.x) * blockDim.x) {
        const int p = static_cast<int>(i % hw);
        const size_t r = i / hw;
        const int ch = static_cast<int>(r % c);
        const int b = static_cast<int>(r / c);
        out[i] = static_cast<float>(in[(static_cast<size_t>(b) * hw + p) * c_pad + ch]);
    }
}

// ---- (B, D, 1, S) -> [B*S, D] fp16 (tiled transpose through shared memory) -------------------
template <typename T>
__global__ void ctx_to_tokens_kernel(const T* __restrict__ in, __half* __restrict__ out, int d, int s) {
    pdl_trigger();  // no TMEM / large shared memory here: dependents may start their prologue at once
    pdl_wait();
    __shared__ float tile[32][33];
    const int b = blockIdx.z;
    const int d0 = blockIdx.y * 32, s0 = blockIdx.x * 32;
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        const int dd = d0 + r, ss = s0 + threadIdx.x;
        if (dd < d && ss < s) tile[r][threadIdx.x] = static_cast<float>(in[(static_cast<size_t>(b) * d + dd) * s + ss]);
    }
    __syncthreads();
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        const int ss = s0 + r, dd = d0 + threadIdx.x;
        if (dd < d && ss < s) out[(static_cast<size_t>(b) * s + ss) * d + dd] = __float2half_rn(tile[threadIdx.x][r]);
    }
}

// ---- CLIP text embeddings: out[b*s + t, :] = token_embedding[ids[b, t]] + position_embedding[t] -----------
// ids arrive as float32 (the reference feeds input_ids as floats, pipeline.py:173); out-of-range ids clamp.
__global__ void embed_tokens_kernel(const float* __restrict__ ids, const uint4* __restrict__ tok,
                                    const uint4* __restrict__ pos, uint4* __restrict__ out, int rows, int s, int vecs,
                                    int vocab) {
    pdl_trigger();  // no TMEM / large shared memory here: dependents may start their prologue at once
    pdl_wait();
    const size_t total = static_cast<size_t>(rows) * vecs;
    for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total;
         i += static_cast<size_t>(gridDim.x) * blockDim.x) {
        const int r = static_cast<int>(i / vecs), v = static_cast<int>(i - static_cast<size_t>(r) * vecs);
        const int id = min(max(__float2int_rn(ids[r]), 0), vocab - 1);
        uint4 a = tok[static_cast<size_t>(id) * vecs + v];
        const uint4 b = pos[static_cast<size_t>(r % s) * vecs + v];
        __half2* ah = reinterpret_cast<__half2*>(&a);
        const __half2* bh = reinterpret_cast<const __half2*>(&b);
#pragma unroll
        for (int q = 0; q < 4; ++q) ah[q] = __hadd2(ah[q], bh[q]);
        out[i] = a;
    }
}

// ---- nearest x2 upsample, NHWC fp16, 16-byte vectors ------------------------------------------
__global__ void upsample2x_kernel(const uint4* __restrict__ in, uint4* __restrict__ out, int n, int h, int w,
                                  int vecs) {
    pdl_trigger();  // no TMEM / large shared memory here: dependents may start their prologue at once
    pdl_wait();
    const size_t total = static_cast<size_t>(n) * (2 * h) * (2 * w) * vecs;
    for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total;
         i += static_cast<size_t>(gridDim.x) * blockDim.x) {
        const int v = static_cast<int>(i % vecs);
        size_t r = i / vecs;
        const int ox = static_cast<int>(r % (2 * w));
        r /= (2 * w);
        const int oy = static_cast<int>(r % (2 * h));
        const int b = static_cast<int>(r / (2 * h));
        out[i] = in[((static_cast<size_t>(b) * h + (oy >> 1)) * w + (ox >> 1)) * vecs + v];
    }
}

__global__ void add_kernel(const __half2* __restrict__ a, const __half2* __restrict__ b, __half2* __restrict__ out,
                           size_t n2) {
    pdl_trigger();  // no TMEM / large shared memory here: dependents may start their prologue at once
    pdl_wait();
    for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < n2;
         i += static_cast<size_t>(gridDim.x) * blockDim.x) {
        const float2 x = __half22float2(a[i]), y = __half22float2(b[i]);
        out[i] = __floats2half2_rn(x.x + y.x, x.y + y.y);
    }
}

// ---- small-M linear: one warp per output column, all M rows at once (M <= 8) -------------------
// The (optionally SiLU-activated) input rows are staged in shared memory ONCE per block -- every column warp used to
// re-read and re-activate them (the 20 800-column time-embedding projection was MUFU-bound on 20 800 redundant SiLU
// passes) -- and a warp requests four weight vectors per lane before the first one is consumed.
template <int kM>
__global__ void __launch_bounds__(256) linear_small_kernel(const float* __restrict__ x, const __half* __restrict__ w,
                                                           const float* __restrict__ bias,
                                                           const float* __restrict__ add, float* __restrict__ out,
                                                           int m, int n, int k, int act_in, int act_out) {
    extern __shared__ __align__(16) float xs[];  // [kM][k]
    pdl_trigger();  // no TMEM / large shared memory here: dependents may start their prologue at once
    pdl_wait();
    for (int i = threadIdx.x; i < kM * k; i += blockDim.x) {
        const int r = i / k;
        float v = r < m ? x[i] : 0.f;
        if (act_in) v = silu_f(v);
        xs[i] = v;
    }
    __syncthreads();
    const int col = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (col >= n) return;
    const __half* wr = w + static_cast<size_t>(col) * k;
    float acc[kM];
#pragma unroll
    for (int r = 0; r < kM; ++r) acc[r] = 0.f;
    constexpr int kInFlight = 4;
    for (int kb = lane * 8; kb < k; kb += 32 * 8 * kInFlight) {
        uint4 raw[kInFlight];
#pragma unroll
        for (int i = 0; i < kInFlight; ++i) {
            const int kk = kb + i * 256;
            raw[i] = kk < k ? __ldg(reinterpret_cast<const uint4*>(wr + kk)) : make_uint4(0, 0, 0, 0);
        }
#pragma unroll
        for (int i = 0; i < kInFlight; ++i) {
            const int kk = kb + i * 256;
            if (kk >= k) break;
            const __half2* h2 = reinterpret_cast<const __half2*>(&raw[i]);
            float wf[8];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const float2 t = __half22float2(h2[q]);
                wf[2 * q] = t.x;
                wf[2 * q + 1] = t.y;
            }
#pragma unroll
            for (int r = 0; r < kM; ++r) {
                const float4 x0 = *reinterpret_cast<const float4*>(xs + r * k + kk);
                const float4 x1 = *reinterpret_cast<const float4*>(xs + r * k + kk + 4);
                acc[r] += x0.x * wf[0] + x0.y * wf[1] + x0.z * wf[2] + x0.w * wf[3] + x1.x * wf[4] + x1.y * wf[5] + x1.z * wf[6] +
                          x1.w * wf[7];
            }
        }
    }
#pragma unroll
    for (int r = 0; r < kM; ++r) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) acc[r] += __shfl_xor_sync(0xffffffffu, acc[r], o);
    }
    if (lane == 0) {
        const float b = (bias ? bias[col] : 0.f) + (add ? add[col] : 0.f);
        for (int r = 0; r < m && r < kM; ++r) {
            float v = acc[r] + b;
            if (act_out) v = silu_f(v);
            out[static_cast<size_t>(r) * n + col] = v;
        }
    }
}

// ---- sinusoidal timestep embedding (unet.py:703-728) -------------------------------------------
__global__ void timestep_embedding_kernel(const float* __restrict__ t, float* __restrict__ out, int m, int dim,
                                          int flip, float freq_shift) {
    pdl_trigger();  // no TMEM / large shared memory here: dependents may start their prologue at once
    pdl_wait();
    const int half = dim / 2;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m * half) return;
    const int r = i / half, j = i % half;
    const float freq = expf(-logf(10000.0f) * static_cast<float>(j) / (static_cast<float>(half) - freq_shift));
    const float ang = t[r] * freq;
    const float s = sinf(ang), c = cosf(ang);
    float* o = out + static_cast<size_t>(r) * dim;
    if (flip) {
        o[j] = c;
        o[half + j] = s;
    } else {
        o[j] = s;
        o[half + j] = c;
    }
}

// ---- fused CFG + scheduler step ------------------------------------------------------------------
// Philox-4x32-10 normal (rng.py NvRandomSource, the Swift pipeline's nvidiaRNG): counter (draw, 0, idx, 0), Box-Muller on
// the first two output words in double precision, rounded once to fp32.  The explicit _rn intrinsics keep the compiler
// from contracting the uniform maps into FMAs, which the host twin does not do.
__device__ __forceinline__ float philox_normal(uint32_t k0, uint32_t k1, uint32_t draw, uint32_t idx) {
    uint32_t c0 = draw, c1 = 0u, c2 = idx, c3 = 0u;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint64_t v1 = static_cast<uint64_t>(c0) * 0xD2511F53ull;
        const uint64_t v2 = static_cast<uint64_t>(c2) * 0xCD9E8D57ull;
        c0 = static_cast<uint32_t>(v2 >> 32) ^ c1 ^ k0;
        c1 = static_cast<uint32_t>(v2);
        c2 = static_cast<uint32_t>(v1 >> 32) ^ c3 ^ k1;
        c3 = static_cast<uint32_t>(v1);
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    const double u = __dadd_rn(__dmul_rn(static_cast<double>(c0), 1.0 / 4294967296.0), 1.0 / 8589934592.0);
    const double v = __dadd_rn(__dmul_rn(static_cast<double>(c1), 3.141592653589793 / 2147483648.0),
                               3.141592653589793 / 4294967296.0);
    return static_cast<float>(__dmul_rn(sqrt(-2.0 * log(u)), sin(v)));
}

// One thread per latent element (n*c*h*w, NCHW fp32).  See include/b200sd.h for the algebra.  kExt = false is the
// plain CFG + scheduler step (b200sd_cfg_scheduler_step); kExt = true adds the sampler terms (input scale, noise,
// input-only mode) of b200sd_sampler_step.
template <bool kExt>
__global__ void cfg_step_kernel(const float* __restrict__ noise_pred, float* __restrict__ latents,
                                float* __restrict__ hist, float* __restrict__ denoised, __half* __restrict__ unet_in,
                                int c_pad, int n, int c, int hw, b200sd_sampler_coeffs sk,
                                const uint32_t* __restrict__ rng_key) {
    pdl_trigger();  // no TMEM / large shared memory here: dependents may start their prologue at once
    pdl_wait();
    const b200sd_step_coeffs& k = sk.step;
    const int numel = n * c * hw;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= numel) return;
    if (kExt && !noise_pred) {  // input-only mode: the first UNet input of a loop
        const int p = i % hw;
        const int ch = (i / hw) % c;
        const int b = i / (hw * c);
        const __half hv = __float2half_rn(sk.in_scale * latents[i]);
        unet_in[(static_cast<size_t>(b) * hw + p) * c_pad + ch] = hv;
        unet_in[(static_cast<size_t>(n + b) * hw + p) * c_pad + ch] = hv;
        return;
    }
    int ni = i;  // index of this element inside one CFG half of noise_pred
    if (k.noise_pred_nhwc) {  // the UNet's conv_out output as it leaves the epilogue: [2n, h*w, c]
        const int p = i % hw;
        const int ch = (i / hw) % c;
        const int b = i / (hw * c);
        ni = (b * hw + p) * c + ch;
    }
    const float eu = noise_pred[ni];
    const float ec = noise_pred[numel + ni];
    const float eps = eu + k.guidance * (ec - eu);
    const float x = latents[i];
    float xp = k.cx * x + k.ce * eps;
    float x0 = k.x0_cx * x + k.x0_ce * eps;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        if (j < k.n_hist) {
            const float hv = hist[static_cast<size_t>(j) * numel + i];
            xp += k.ch[j] * hv;
            x0 += k.x0_ch[j] * hv;
        }
    }
    if (kExt && sk.noise_scale != 0.f) {  // no "+ 0 * z": that would turn a -0 into +0
        const int per = c * hw;
        const int b = i / per;
        const float z = philox_normal(rng_key[0], rng_key[1], sk.noise_draw + static_cast<uint32_t>(b),
                                      static_cast<uint32_t>(i - b * per));
        xp += sk.noise_scale * z;
    }
    if (k.push_eps_slot >= 0) hist[static_cast<size_t>(k.push_eps_slot) * numel + i] = eps;
    if (k.push_x0_slot >= 0) hist[static_cast<size_t>(k.push_x0_slot) * numel + i] = x0;
    if (k.push_x_slot >= 0) hist[static_cast<size_t>(k.push_x_slot) * numel + i] = x;
    if (denoised) denoised[i] = x0;
    latents[i] = xp;
    if (unet_in) {
        // NCHW index -> NHWC, duplicated for the (uncond, cond) batch halves
        const int p = i % hw;
        const int ch = (i / hw) % c;
        const int b = i / (hw * c);
        const __half hv = __float2half_rn(kExt && sk.in_scale != 1.f ? sk.in_scale * xp : xp);
        unet_in[(static_cast<size_t>(b) * hw + p) * c_pad + ch] = hv;
        unet_in[(static_cast<size_t>(n + b) * hw + p) * c_pad + ch] = hv;
    }
}

// ---- image post-process: clip(x/2+0.5, 0, 1), NHWC(c_pad) -> NHWC(c) fp32 and/or u8 -------------
template <typename T>
__global__ void image_post_kernel(const T* __restrict__ in, int c_pad, float* __restrict__ of, uint8_t* __restrict__ ou,
                                  size_t pixels, int c) {
    pdl_trigger();  // no TMEM / large shared memory here: dependents may start their prologue at once
    pdl_wait();
    const size_t total = pixels * c;
    for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total;
         i += static_cast<size_t>(gridDim.x) * blockDim.x) {
        const size_t px = i / c;
        const int ch = static_cast<int>(i % c);
        float v = static_cast<float>(in[px * c_pad + ch]) * 0.5f + 0.5f;
        v = fminf(fmaxf(v, 0.f), 1.f);
        if (of) of[i] = v;
        if (ou) ou[i] = static_cast<uint8_t>(__float2int_rn(v * 255.f));
    }
}


// ---- latent prep for the VAE decoder: z/scaling -> post_quant_conv (1x1, <= 8 channels) -> NHWC fp16 ----
__global__ void latent_prep_kernel(const float* __restrict__ z, const float* __restrict__ w /* [c, c] */,
                                   const float* __restrict__ b, float inv_scale, __half* __restrict__ out, int n, int c,
                                   int hw, int c_pad) {
    pdl_trigger();  // no TMEM / large shared memory here: dependents may start their prologue at once
    pdl_wait();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n * hw) return;
    const int p = i % hw, img = i / hw;
    float v[8];
#pragma unroll
    for (int ci = 0; ci < 8; ++ci) v[ci] = ci < c ? z[(static_cast<size_t>(img) * c + ci) * hw + p] * inv_scale : 0.f;
    for (int co = 0; co < c_pad; ++co) {
        float acc = 0.f;
        if (co < c) {
            acc = b ? b[co] : 0.f;
            for (int ci = 0; ci < c; ++ci) acc += w[co * c + ci] * v[ci];
        }
        out[static_cast<size_t>(i) * c_pad + co] = __float2half_rn(acc);
    }
}

}  // namespace b200sd

using namespace b200sd;

extern "C" int b200sd_nchw_to_nhwc(const void* in, int32_t in_f32, void* out, int32_t n, int32_t c, int32_t h,
                                   int32_t w, int32_t c_pad, void* stream_) {
    if (!b200sd::launch_class_enabled(8)) return 0;  // bench.py's per-class timing graphs
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    B200SD_REQUIRE(in && out && c_pad >= c, "b200sd_nchw_to_nhwc: bad arguments");
    const size_t total = static_cast<size_t>(n) * h * w * c_pad;
    if (in_f32)
        B200SD_CHECK_CUDA(launch_kernel(nchw_to_nhwc_kernel<float>, dim3(grid_for(total, 256)), dim3(256), 0, stream, reinterpret_cast<const float*>(in),
                                                                             reinterpret_cast<__half*>(out), n, c,
                                                                             h * w, c_pad));
    else
        B200SD_CHECK_CUDA(launch_kernel(nchw_to_nhwc_kernel<__half>, dim3(grid_for(total, 256)), dim3(256), 0, stream, reinterpret_cast<const __half*>(in),
                                                                              reinterpret_cast<__half*>(out), n, c,
                                                                              h * w, c_pad));
    B200SD_CHECK_CUDA(cudaGetLastError());
    count_launch(1);
    return 0;
}

extern "C" int b200sd_nhwc_to_nchw_f32(const void* in, int32_t in_f32, float* out, int32_t n, int32_t c, int32_t h,
                                       int32_t w, int32_t c_pad, void* stream_) {
    if (!b200sd::launch_class_enabled(8)) return 0;  // bench.py's per-class timing graphs
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    B200SD_REQUIRE(in && out && c_pad >= c, "b200sd_nhwc_to_nchw_f32: bad arguments");
    const size_t total = static_cast<size_t>(n) * c * h * w;
    if (in_f32)
        B200SD_CHECK_CUDA(launch_kernel(nhwc_to_nchw_f32_kernel<float>, dim3(grid_for(total, 256)), dim3(256), 0, stream, reinterpret_cast<const float*>(in),
                                                                                 out, n, c, h * w, c_pad));
    else
        B200SD_CHECK_CUDA(launch_kernel(nhwc_to_nchw_f32_kernel<__half>, dim3(grid_for(total, 256)), dim3(256), 0, stream, reinterpret_cast<const __half*>(in),
                                                                                  out, n, c, h * w, c_pad));
    B200SD_CHECK_CUDA(cudaGetLastError());
    count_launch(1);
    return 0;
}

extern "C" int b200sd_ctx_to_tokens(const void* in, int32_t in_f32, void* out, int32_t b, int32_t d, int32_t s,
                                    void* stream_) {
    if (!b200sd::launch_class_enabled(8)) return 0;  // bench.py's per-class timing graphs
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    B200SD_REQUIRE(in && out, "b200sd_ctx_to_tokens: null pointer");
    dim3 grid((s + 31) / 32, (d + 31) / 32, b), block(32, 8);
    if (in_f32)
        B200SD_CHECK_CUDA(launch_kernel(ctx_to_tokens_kernel<float>, dim3(grid), dim3(block), 0, stream, reinterpret_cast<const float*>(in),
                                                                reinterpret_cast<__half*>(out), d, s));
    else
        B200SD_CHECK_CUDA(launch_kernel(ctx_to_tokens_kernel<__half>, dim3(grid), dim3(block), 0, stream, reinterpret_cast<const __half*>(in),
                                                                 reinterpret_cast<__half*>(out), d, s));
    B200SD_CHECK_CUDA(cudaGetLastError());
    count_launch(1);
    return 0;
}

extern "C" int b200sd_embed_tokens(const float* ids, const void* token_embedding, const void* position_embedding,
                                   void* out, int32_t batch, int32_t s, int32_t d, int32_t vocab, void* stream_) {
    if (!b200sd::launch_class_enabled(8)) return 0;  // bench.py's per-class timing graphs
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    B200SD_REQUIRE(ids && token_embedding && position_embedding && out && d % 8 == 0 && vocab > 0,
                   "b200sd_embed_tokens: bad arguments (d=%d must be a multiple of 8)", d);
    const size_t total = static_cast<size_t>(batch) * s * (d / 8);
    B200SD_CHECK_CUDA(launch_kernel(embed_tokens_kernel, dim3(grid_for(total, 256)), dim3(256), 0, stream, ids,
                                    reinterpret_cast<const uint4*>(token_embedding),
                                    reinterpret_cast<const uint4*>(position_embedding), reinterpret_cast<uint4*>(out),
                                    batch * s, s, d / 8, vocab));
    B200SD_CHECK_CUDA(cudaGetLastError());
    count_launch(1);
    return 0;
}

extern "C" int b200sd_upsample2x(const void* in, void* out, int32_t n, int32_t h, int32_t w, int32_t c,
                                 void* stream_) {
    if (!b200sd::launch_class_enabled(8)) return 0;  // bench.py's per-class timing graphs
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    B200SD_REQUIRE(in && out && c % 8 == 0, "b200sd_upsample2x: c=%d must be a multiple of 8", c);
    const size_t total = static_cast<size_t>(n) * 4 * h * w * (c / 8);
    B200SD_CHECK_CUDA(launch_kernel(upsample2x_kernel, dim3(grid_for(total, 256)), dim3(256), 0, stream, reinterpret_cast<const uint4*>(in),
                                                                reinterpret_cast<uint4*>(out), n, h, w, c / 8));
    B200SD_CHECK_CUDA(cudaGetLastError());
    count_launch(1);
    return 0;
}

extern "C" int b200sd_add(const void* a, const void* b, void* out, size_t numel, void* stream_) {
    if (!b200sd::launch_class_enabled(8)) return 0;  // bench.py's per-class timing graphs
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    B200SD_REQUIRE(a && b && out && numel % 2 == 0, "b200sd_add: bad arguments");
    B200SD_CHECK_CUDA(launch_kernel(add_kernel, dim3(grid_for(numel / 2, 256)), dim3(256), 0, stream, reinterpret_cast<const __half2*>(a),
                                                             reinterpret_cast<const __half2*>(b),
                                                             reinterpret_cast<__half2*>(out), numel / 2));
    B200SD_CHECK_CUDA(cudaGetLastError());
    count_launch(1);
    return 0;
}

extern "C" int b200sd_linear_small(const float* x, const void* wgt, const float* bias, const float* add, float* out,
                                   int32_t m, int32_t n, int32_t k, int32_t act_in, int32_t act_out, void* stream_) {
    if (!b200sd::launch_class_enabled(8)) return 0;  // bench.py's per-class timing graphs
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    B200SD_REQUIRE(x && wgt && out, "b200sd_linear_small: null pointer");
    B200SD_REQUIRE(m >= 1 && m <= 32 && k % 8 == 0, "b200sd_linear_small: need 1 <= m <= 32 and k %% 8 == 0 (m=%d k=%d)",
                   m, k);
    const int blocks = (n + 7) / 8;
    const __half* w = reinterpret_cast<const __half*>(wgt);
    for (int r0 = 0; r0 < m; r0 += 8) {
        const int mm = std::min(8, m - r0);
        const float* xr = x + static_cast<size_t>(r0) * k;
        float* orow = out + static_cast<size_t>(r0) * n;
        const size_t smem = static_cast<size_t>(mm <= 2 ? 2 : 8) * k * sizeof(float);
        B200SD_REQUIRE(smem <= 160 * 1024, "b200sd_linear_small: k = %d too large for the staged input rows", k);
        static bool attr = false;
        if (!attr) {
            B200SD_CHECK_CUDA(cudaFuncSetAttribute(linear_small_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024));
            B200SD_CHECK_CUDA(cudaFuncSetAttribute(linear_small_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024));
            attr = true;
        }
        if (mm <= 2)
            B200SD_CHECK_CUDA(launch_kernel(linear_small_kernel<2>, dim3(blocks), dim3(256), smem, stream, xr, w, bias, add, orow, mm, n, k, act_in, act_out));
        else
            B200SD_CHECK_CUDA(launch_kernel(linear_small_kernel<8>, dim3(blocks), dim3(256), smem, stream, xr, w, bias, add, orow, mm, n, k, act_in, act_out));
        B200SD_CHECK_CUDA(cudaGetLastError());
        count_launch(1);
    }
    return 0;
}

extern "C" int b200sd_timestep_embedding(const float* timesteps, float* out, int32_t m, int32_t dim,
                                         int32_t flip_sin_to_cos, float freq_shift, void* stream_) {
    if (!b200sd::launch_class_enabled(8)) return 0;  // bench.py's per-class timing graphs
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    B200SD_REQUIRE(timesteps && out && dim % 2 == 0, "b200sd_timestep_embedding: bad arguments");
    const int total = m * (dim / 2);
    B200SD_CHECK_CUDA(launch_kernel(timestep_embedding_kernel, dim3((total + 127) / 128), dim3(128), 0, stream, timesteps, out, m, dim, flip_sin_to_cos,
                                                                      freq_shift));
    B200SD_CHECK_CUDA(cudaGetLastError());
    count_launch(1);
    return 0;
}

static int launch_step(const char* what, const float* noise_pred, float* latents, float* hist, float* denoised,
                       void* unet_in, int32_t c_pad, int32_t n, int32_t c, int32_t h, int32_t w,
                       const b200sd_sampler_coeffs& sk, const uint32_t* rng_key, bool ext, cudaStream_t stream) {
    const b200sd_step_coeffs* coeffs = &sk.step;
    if (noise_pred) {  // the input-only mode reads no history
    B200SD_REQUIRE(coeffs->n_hist >= 0 && coeffs->n_hist <= 4 && (coeffs->n_hist == 0 || hist),
                   "%s: bad history arguments", what);
    B200SD_REQUIRE(coeffs->push_eps_slot < 4 && coeffs->push_x0_slot < 4 && coeffs->push_x_slot < 4 &&
                       (hist || (coeffs->push_eps_slot < 0 && coeffs->push_x0_slot < 0 && coeffs->push_x_slot < 0)),
                   "%s: bad history ring slot", what);
    }
    const int numel = n * c * h * w;
    B200SD_CHECK_CUDA(launch_kernel(ext ? cfg_step_kernel<true> : cfg_step_kernel<false>, dim3((numel + 255) / 256),
                                    dim3(256), 0, stream, noise_pred, latents, hist, denoised,
                                    reinterpret_cast<__half*>(unet_in), c_pad, n, c, h * w, sk, rng_key));
    B200SD_CHECK_CUDA(cudaGetLastError());
    count_launch(1);
    return 0;
}

extern "C" int b200sd_cfg_scheduler_step(const float* noise_pred, float* latents, float* hist, float* denoised,
                                         void* unet_in, int32_t c_pad, int32_t n, int32_t c, int32_t h, int32_t w,
                                         const b200sd_step_coeffs* coeffs, void* stream_) {
    if (!b200sd::launch_class_enabled(8)) return 0;  // bench.py's per-class timing graphs
    B200SD_REQUIRE(noise_pred && latents && coeffs, "b200sd_cfg_scheduler_step: null pointer");
    b200sd_sampler_coeffs sk{};
    sk.step = *coeffs;
    sk.in_scale = 1.f;
    return launch_step("b200sd_cfg_scheduler_step", noise_pred, latents, hist, denoised, unet_in, c_pad, n, c, h, w, sk,
                       nullptr, false, static_cast<cudaStream_t>(stream_));
}

extern "C" int b200sd_sampler_step(const float* noise_pred, float* latents, float* hist, float* denoised, void* unet_in,
                                   int32_t c_pad, int32_t n, int32_t c, int32_t h, int32_t w,
                                   const b200sd_sampler_coeffs* coeffs, const uint32_t* rng_key, void* stream_) {
    if (!b200sd::launch_class_enabled(8)) return 0;  // bench.py's per-class timing graphs
    B200SD_REQUIRE(latents && coeffs, "b200sd_sampler_step: null pointer");
    B200SD_REQUIRE(noise_pred || (unet_in && c_pad >= c), "b200sd_sampler_step: the input-only mode needs unet_in");
    B200SD_REQUIRE(coeffs->noise_scale == 0.f || !noise_pred || rng_key,
                   "b200sd_sampler_step: noise_scale != 0 needs rng_key");
    // with the sampler terms off this is the plain step kernel, so those samplers keep its arithmetic exactly
    const bool ext = !noise_pred || coeffs->in_scale != 1.f || coeffs->noise_scale != 0.f;
    return launch_step("b200sd_sampler_step", noise_pred, latents, hist, denoised, unet_in, c_pad, n, c, h, w, *coeffs,
                       rng_key, ext, static_cast<cudaStream_t>(stream_));
}

extern "C" int b200sd_image_postprocess(const void* in, int32_t in_f32, int32_t c_pad, float* out_f32,
                                        uint8_t* out_u8, int32_t n, int32_t h, int32_t w, int32_t c, void* stream_) {
    if (!b200sd::launch_class_enabled(8)) return 0;  // bench.py's per-class timing graphs
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    B200SD_REQUIRE(in && (out_f32 || out_u8), "b200sd_image_postprocess: null pointer");
    const size_t pixels = static_cast<size_t>(n) * h * w;
    if (in_f32)
        B200SD_CHECK_CUDA(launch_kernel(image_post_kernel<float>, dim3(grid_for(pixels * c, 256)), dim3(256), 0, stream, reinterpret_cast<const float*>(in),
                                                                                c_pad, out_f32, out_u8, pixels, c));
    else
        B200SD_CHECK_CUDA(launch_kernel(image_post_kernel<__half>, dim3(grid_for(pixels * c, 256)), dim3(256), 0, stream, reinterpret_cast<const __half*>(in),
                                                                                 c_pad, out_f32, out_u8, pixels, c));
    B200SD_CHECK_CUDA(cudaGetLastError());
    count_launch(1);
    return 0;
}

extern "C" int b200sd_latent_prep(const float* z, const float* w, const float* b, float inv_scale, void* out,
                                  int32_t n, int32_t c, int32_t h, int32_t wd, int32_t c_pad, void* stream_) {
    if (!b200sd::launch_class_enabled(8)) return 0;  // bench.py's per-class timing graphs
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    B200SD_REQUIRE(z && w && out && c >= 1 && c <= 8 && c_pad >= c, "b200sd_latent_prep: bad arguments");
    const int total = n * h * wd;
    B200SD_CHECK_CUDA(launch_kernel(latent_prep_kernel, dim3((total + 255) / 256), dim3(256), 0, stream, z, w, b, inv_scale, reinterpret_cast<__half*>(out), n,
                                                               c, h * wd, c_pad));
    B200SD_CHECK_CUDA(cudaGetLastError());
    count_launch(1);
    return 0;
}
