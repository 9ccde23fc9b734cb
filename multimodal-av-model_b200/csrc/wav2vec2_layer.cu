// wav2vec2_layer.cu — Wav2Vec2EncoderLayerStableLayerNorm under bf16 autocast, around torch's attention core, as two host
// calls per direction (transformers/models/wav2vec2/modeling_wav2vec2.py, Wav2Vec2EncoderLayerStableLayerNorm.forward):
//
//   attn_in      : ln1 = LayerNorm(x) (fp32 math, bf16 out); q, k, v = ln1 . W^T + b (one grouped GEMM launch)
//   [SDPA stays torch: the caller runs the attention interface HF runs, with its own dropout stream]
//   attn_out_ffn : h1 = x + drop(attn . Wo^T + bo); y = h1 + drop(gelu_drop(LayerNorm(h1) . W1^T + b1) . W2^T + b2)
//
// Every value the module path materialises in bf16 (LayerNorm outputs, Linear outputs, GELU output, dropout outputs,
// residual sums) is rounded to bf16 here at the same point, so native and module paths differ only in GEMM and
// LayerNorm summation order.  Dropout reproduces ATen's CUDA native_dropout bit for bit (see Drop below); the caller
// reserves the generator offsets.  Backward regenerates the masks from (seed, offset) and recomputes GELU from the saved
// pre-activation.  LayerNorm weight and bias gradients and the bias column sums are reduced from per-CTA partials in a
// fixed order (no float atomics); the weight-gradient GEMMs use the library's split-K.
#include <curand_kernel.h>

#include <initializer_list>

#include "common.cuh"
#include "gemm_internal.h"

namespace avctc {
namespace {

constexpr int kRowsPerCta = 8;     // warp-per-row kernels: 8 warps, one row each
constexpr int kLnBwdCtas = 148;    // CTAs of the LayerNorm backward = rows of its weight/bias partials
constexpr int kColParts = 32;      // row chunks of the bias column sums

// ATen's fused dropout (aten/src/ATen/native/cuda/Dropout.cu, fused_dropout_kernel_vec) on a contiguous, 16-byte
// aligned bf16 tensor whose size is a multiple of 8 runs with VEC = 8: a grid of min(ceil(n/256), SMs *
// maxThreadsPerSM/256) blocks of 256 threads; thread t calls curand_init(seed, t, offset) and, per grid-stride step,
// handles the 8 elements 8*(t + step*threads) .. +7 with two curand_uniform4 draws; an element is kept when its uniform
// is < keep (float) and then scaled in float.  The draws of step s are Philox counters offset/4 + 2s and + 2s + 1 of
// subsequence t, which curand_init(seed, t, offset + 8*s) followed by two curand_uniform4 yields directly.
struct Drop {
    unsigned long long seed, offset;
    unsigned long long threads;
    float keep, scale;
    int active;
};

// v[0..8) are elements i..i+8 (i % 8 == 0): dropped -> 0, kept -> v * scale (float; the caller rounds)
__device__ __forceinline__ void drop8(const Drop& d, long long i, float* v) {
    if (!d.active) return;
    const unsigned long long g = (unsigned long long)i >> 3;
    curandStatePhilox4_32_10_t st;
    curand_init(d.seed, g % d.threads, d.offset + 8ull * (g / d.threads), &st);
    const float4 r0 = curand_uniform4(&st), r1 = curand_uniform4(&st);
    const float u[8] = {r0.x, r0.y, r0.z, r0.w, r1.x, r1.y, r1.z, r1.w};
#pragma unroll
    for (int k = 0; k < 8; ++k) v[k] = u[k] < d.keep ? v[k] * d.scale : 0.f;
}

__device__ __forceinline__ float rbf(float x) { return __bfloat162float(__float2bfloat16(x)); }

__device__ __forceinline__ void load8(const __nv_bfloat16* p, float* v) {
    const uint4 u = *reinterpret_cast<const uint4*>(p);
    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&u);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const float2 f = __bfloat1622float2(h[k]);
        v[2 * k] = f.x; v[2 * k + 1] = f.y;
    }
}
__device__ __forceinline__ void store8(__nv_bfloat16* p, const float* v) {
    uint4 u;
    __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&u);
#pragma unroll
    for (int k = 0; k < 4; ++k) h[k] = __floats2bfloat162_rn(v[2 * k], v[2 * k + 1]);
    *reinterpret_cast<uint4*>(p) = u;
}
__device__ __forceinline__ void load8f(const float* p, float* v) {
    const float4 a = *reinterpret_cast<const float4*>(p), b = *reinterpret_cast<const float4*>(p + 4);
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}

// exact-erf GELU and its derivative as ATen's CUDA kernels compute them (float opmath)
__device__ __forceinline__ float gelu_f(float x) { return x * 0.5f * (1.f + erff(x * (float)M_SQRT1_2)); }
__device__ __forceinline__ float gelu_grad(float dy, float x) {
    constexpr float kBeta = (float)(M_2_SQRTPI * M_SQRT1_2 * 0.5);
    const float cdf = 0.5f * (1.f + erff(x * (float)M_SQRT1_2));
    const float pdf = expf(-0.5f * x * x) * kBeta;
    return dy * (cdf + x * pdf);
}

// LayerNorm over rows of E = 256*NC bf16 values, one warp per row (lane owns 8-element chunks lane, lane+32, ...).
// RESID: the row is first formed as h = bf16(res + bf16(drop(a))) and h is written out.  Writes y = bf16(LN(row)) and
// the row's mean and 1/sqrt(var + eps) for backward.
template <int NC, bool RESID>
__global__ void __launch_bounds__(256) ln_fwd_kernel(const __nv_bfloat16* __restrict__ a, const __nv_bfloat16* __restrict__ res,
                                                     Drop d, long long M, const float* __restrict__ g,
                                                     const float* __restrict__ b, float eps, __nv_bfloat16* h_out,
                                                     __nv_bfloat16* y, float* mean_out, float* rstd_out) {
    constexpr int E = NC * 256;
    const int lane = threadIdx.x & 31;
    const long long row = (long long)blockIdx.x * kRowsPerCta + (threadIdx.x >> 5);
    if (row >= M) return;
    float v[NC][8];
    float s = 0.f;
#pragma unroll
    for (int j = 0; j < NC; ++j) {
        const long long idx = row * E + (lane + 32 * j) * 8;
        load8(a + idx, v[j]);
        if (RESID) {
            float r[8];
            drop8(d, idx, v[j]);
            load8(res + idx, r);
#pragma unroll
            for (int k = 0; k < 8; ++k) v[j][k] = rbf(r[k] + rbf(v[j][k]));
            store8(h_out + idx, v[j]);
        }
#pragma unroll
        for (int k = 0; k < 8; ++k) s += v[j][k];
    }
    const float mean = warp_sum(s) / E;
    float q = 0.f;
#pragma unroll
    for (int j = 0; j < NC; ++j)
#pragma unroll
        for (int k = 0; k < 8; ++k) { const float t = v[j][k] - mean; q += t * t; }
    const float rstd = rsqrtf(warp_sum(q) / E + eps);
#pragma unroll
    for (int j = 0; j < NC; ++j) {
        const int col = (lane + 32 * j) * 8;
        float gg[8], bb[8], o[8];
        load8f(g + col, gg);
        load8f(b + col, bb);
#pragma unroll
        for (int k = 0; k < 8; ++k) o[k] = (v[j][k] - mean) * rstd * gg[k] + bb[k];
        store8(y + row * E + col, o);
    }
    if (lane == 0) { mean_out[row] = mean; rstd_out[row] = rstd; }
}

// LayerNorm backward, one warp per row, rows grid-strided over a fixed grid.  dxn = d LN / d x for the bf16 incoming
// gradient dy (the module path's fp32 LayerNorm sees the bf16 gradient of the Linear input).
// RESID = false: out = bf16(dxn).
// RESID = true:  out = dh = bf16(res + bf16(dxn)) (the residual branch's gradient joins), out2 = bf16(drop_bwd(dh)).
// part != NULL: part[0][cta][E] = sum over the CTA's rows of dy * xhat (weight), part[1][cta][E] = sum of dy (bias),
// warps combined in a fixed order.
template <int NC, bool RESID>
__global__ void __launch_bounds__(256) ln_bwd_kernel(const __nv_bfloat16* __restrict__ dy, const __nv_bfloat16* __restrict__ x,
                                                     const float* __restrict__ mean, const float* __restrict__ rstd,
                                                     const float* __restrict__ g, long long M,
                                                     const __nv_bfloat16* __restrict__ res, Drop d, __nv_bfloat16* out,
                                                     __nv_bfloat16* out2, float* part) {
    constexpr int E = NC * 256;
    __shared__ float red[kRowsPerCta][E];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float ag[NC][8], ab[NC][8];
#pragma unroll
    for (int j = 0; j < NC; ++j)
#pragma unroll
        for (int k = 0; k < 8; ++k) ag[j][k] = ab[j][k] = 0.f;
    for (long long row = (long long)blockIdx.x * kRowsPerCta + warp; row < M; row += (long long)gridDim.x * kRowsPerCta) {
        const float mu = mean[row], rs = rstd[row];
        float gy[NC][8], xh[NC][8];
        float s1 = 0.f, s2 = 0.f;
#pragma unroll
        for (int j = 0; j < NC; ++j) {
            const int col = (lane + 32 * j) * 8;
            float dv[8], gg[8];
            load8(dy + row * E + col, dv);
            load8(x + row * E + col, xh[j]);
            load8f(g + col, gg);
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                xh[j][k] = (xh[j][k] - mu) * rs;
                gy[j][k] = dv[k] * gg[k];
                s1 += gy[j][k];
                s2 += gy[j][k] * xh[j][k];
                if (part) { ag[j][k] += dv[k] * xh[j][k]; ab[j][k] += dv[k]; }
            }
        }
        s1 = warp_sum(s1) / E;
        s2 = warp_sum(s2) / E;
#pragma unroll
        for (int j = 0; j < NC; ++j) {
            const long long idx = row * E + (lane + 32 * j) * 8;
            float o[8];
#pragma unroll
            for (int k = 0; k < 8; ++k) o[k] = rs * (gy[j][k] - s1 - xh[j][k] * s2);
            if (RESID) {
                float r[8];
                load8(res + idx, r);
#pragma unroll
                for (int k = 0; k < 8; ++k) o[k] = rbf(r[k] + rbf(o[k]));
                store8(out + idx, o);
                drop8(d, idx, o);
                store8(out2 + idx, o);
            } else {
                store8(out + idx, o);
            }
        }
    }
    if (part == nullptr) return;     // uniform across the block
    for (int pass = 0; pass < 2; ++pass) {
#pragma unroll
        for (int j = 0; j < NC; ++j)
#pragma unroll
            for (int k = 0; k < 8; ++k) red[warp][(lane + 32 * j) * 8 + k] = pass ? ab[j][k] : ag[j][k];
        __syncthreads();
        for (int c = threadIdx.x; c < E; c += blockDim.x) {
            float s = 0.f;
#pragma unroll
            for (int w = 0; w < kRowsPerCta; ++w) s += red[w][c];
            part[((long long)pass * gridDim.x + blockIdx.x) * E + c] = s;
        }
        __syncthreads();
    }
}

// act = bf16(drop(bf16(gelu(pre)))), n % 8 == 0
__global__ void gelu_drop_kernel(const __nv_bfloat16* __restrict__ pre, long long n, Drop d, __nv_bfloat16* act) {
    for (long long i = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 8; i < n; i += (long long)gridDim.x * blockDim.x * 8) {
        float v[8];
        load8(pre + i, v);
#pragma unroll
        for (int k = 0; k < 8; ++k) v[k] = rbf(gelu_f(v[k]));
        drop8(d, i, v);
        store8(act + i, v);
    }
}

// y = bf16(h + bf16(drop(z)))
__global__ void resid_drop_kernel(const __nv_bfloat16* __restrict__ z, const __nv_bfloat16* __restrict__ h, long long n, Drop d,
                                  __nv_bfloat16* y) {
    for (long long i = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 8; i < n; i += (long long)gridDim.x * blockDim.x * 8) {
        float v[8], r[8];
        load8(z + i, v);
        drop8(d, i, v);
        load8(h + i, r);
#pragma unroll
        for (int k = 0; k < 8; ++k) v[k] = rbf(r[k] + rbf(v[k]));
        store8(y + i, v);
    }
}

// out = bf16(drop_bwd(g)); GELU = true: out = bf16(gelu'(pre) * bf16(drop_bwd(g))) (out may alias g)
template <bool GELU>
__global__ void drop_bwd_kernel(const __nv_bfloat16* g, const __nv_bfloat16* __restrict__ pre, long long n, Drop d,
                                __nv_bfloat16* out) {
    for (long long i = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 8; i < n; i += (long long)gridDim.x * blockDim.x * 8) {
        float v[8];
        load8(g + i, v);
        drop8(d, i, v);
        if (GELU) {
            float p[8];
            load8(pre + i, p);
#pragma unroll
            for (int k = 0; k < 8; ++k) v[k] = gelu_grad(rbf(v[k]), p[k]);
        }
        store8(out + i, v);
    }
}

// out [M, 3E] = [a | b | c], each [M, E] contiguous, E % 8 == 0
__global__ void pack3_kernel(const __nv_bfloat16* __restrict__ a, const __nv_bfloat16* __restrict__ b,
                             const __nv_bfloat16* __restrict__ c, long long M, int E, __nv_bfloat16* out) {
    const long long per_row = 3ll * E / 8, total = M * per_row;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const long long row = i / per_row;
        const int col = (int)(i - row * per_row) * 8, which = col / E, cc = col - which * E;
        const __nv_bfloat16* src = which == 0 ? a : (which == 1 ? b : c);
        *reinterpret_cast<uint4*>(out + row * 3 * E + col) = *reinterpret_cast<const uint4*>(src + row * E + cc);
    }
}

// bias gradients, pass 1: part[p][n] = sum of x[m][n] over row chunk p (two columns per thread)
struct ColJob { const __nv_bfloat16* x; int N; float* part; };
struct ColJobs { ColJob j[3]; int count; long long M; };
__global__ void colsum_part_kernel(const ColJobs js) {
    const ColJob jb = js.j[blockIdx.z];
    const int n = (blockIdx.x * blockDim.x + threadIdx.x) * 2;
    if (n >= jb.N) return;
    const long long per = (js.M + kColParts - 1) / kColParts;
    const long long m0 = (long long)blockIdx.y * per, m1 = m0 + per < js.M ? m0 + per : js.M;
    float s0 = 0.f, s1 = 0.f;
    for (long long m = m0; m < m1; ++m) {
        const float2 f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(jb.x + m * jb.N + n));
        s0 += f.x; s1 += f.y;
    }
    jb.part[(long long)blockIdx.y * jb.N + n] = s0;
    jb.part[(long long)blockIdx.y * jb.N + n + 1] = s1;
}

// pass 2 (also LayerNorm weight/bias): out[n] = sum over p in order of part[p][n]
struct SumJob { const float* part; int P, N; float* out; };
struct SumJobs { SumJob j[5]; int count; };
__global__ void sum_parts_kernel(const SumJobs js) {
    const SumJob jb = js.j[blockIdx.y];
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= jb.N) return;
    float s = 0.f;
    for (int p = 0; p < jb.P; ++p) s += jb.part[(long long)p * jb.N + n];
    jb.out[n] = s;
}

struct Dims { long long M; int E, F; };
bool make_dims(long long M, int E, int F, Dims* d) {
    if (M <= 0 || E <= 0 || F <= 0 || E % 256 || E > 1024 || F % 8) return false;
    d->M = M; d->E = E; d->F = F;
    return true;
}

struct Carver {
    char* base; size_t off;
    template <typename T> T* take(size_t n) {
        T* p = base ? reinterpret_cast<T*>(base + off) : nullptr;
        off = (off + n * sizeof(T) + 255) / 256 * 256;
        return p;
    }
};
using bf = __nv_bfloat16;
struct InSaved { bf* ln; float *mean, *rstd; size_t total; };
InSaved carve_in_saved(void* base, const Dims& d) {
    Carver c{reinterpret_cast<char*>(base), 0};
    InSaved s;
    s.ln = c.take<bf>(d.M * d.E); s.mean = c.take<float>(d.M); s.rstd = c.take<float>(d.M);
    s.total = c.off;
    return s;
}
struct OutSaved { bf *ao, *h, *ln, *pre, *act, *z; float *mean, *rstd; size_t total; };
OutSaved carve_out_saved(void* base, const Dims& d) {
    Carver c{reinterpret_cast<char*>(base), 0};
    OutSaved s;
    s.ao = c.take<bf>(d.M * d.E); s.h = c.take<bf>(d.M * d.E); s.ln = c.take<bf>(d.M * d.E);
    s.pre = c.take<bf>(d.M * d.F); s.act = c.take<bf>(d.M * d.F); s.z = c.take<bf>(d.M * d.E);
    s.mean = c.take<float>(d.M); s.rstd = c.take<float>(d.M);
    s.total = c.off;
    return s;
}
struct InScratch { bf *dqkv, *dln; float *lnpart, *colpart; size_t total; };
InScratch carve_in_scratch(void* base, const Dims& d) {
    Carver c{reinterpret_cast<char*>(base), 0};
    InScratch s;
    s.dqkv = c.take<bf>(d.M * 3 * d.E); s.dln = c.take<bf>(d.M * d.E);
    s.lnpart = c.take<float>(2ull * kLnBwdCtas * d.E); s.colpart = c.take<float>((size_t)kColParts * 3 * d.E);
    s.total = c.off;
    return s;
}
struct OutScratch { bf *dz, *da, *dln, *dzo; float *lnpart, *colpart; size_t total; };
OutScratch carve_out_scratch(void* base, const Dims& d) {
    Carver c{reinterpret_cast<char*>(base), 0};
    OutScratch s;
    s.dz = c.take<bf>(d.M * d.E); s.da = c.take<bf>(d.M * d.F); s.dln = c.take<bf>(d.M * d.E); s.dzo = c.take<bf>(d.M * d.E);
    s.lnpart = c.take<float>(2ull * kLnBwdCtas * d.E); s.colpart = c.take<float>((size_t)kColParts * (2 * d.E + d.F));
    s.total = c.off;
    return s;
}

// ATen's launch geometry for a dropout over n elements on the current device: threads of the grid and the generator
// offset increment ((n-1) / (256 * grid * 4) + 1) * 4
int dropout_geometry(long long n, unsigned long long* threads, long long* incr) {
    static int sms[64], max_threads[64];
    int dev = 0;
    AVCTC_CUDA_RETURN(cudaGetDevice(&dev));
    if (dev < 0 || dev >= 64) return AVCTC_ERR_UNSUPPORTED;
    if (sms[dev] == 0) {
        AVCTC_CUDA_RETURN(cudaDeviceGetAttribute(&max_threads[dev], cudaDevAttrMaxThreadsPerMultiProcessor, dev));
        AVCTC_CUDA_RETURN(cudaDeviceGetAttribute(&sms[dev], cudaDevAttrMultiProcessorCount, dev));
    }
    long long grid = (n + 255) / 256;
    const long long cap = (long long)sms[dev] * (max_threads[dev] / 256);
    if (grid > cap) grid = cap;
    if (threads) *threads = (unsigned long long)grid * 256;
    if (incr) *incr = ((n - 1) / (256 * grid * 4) + 1) * 4;
    return 0;
}

// One dropout over n elements as native_dropout runs it; a training dropout with p > 0 reserves its generator offset
// increment from `offset`.  backward: the scale native_dropout_backward uses.
int make_drop(long long n, double p, int training, unsigned long long seed, unsigned long long offset, bool backward,
              Drop* o, long long* incr) {
    o->seed = seed; o->offset = offset; o->threads = 1; o->keep = 1.f; o->scale = 1.f; o->active = 0;
    *incr = 0;
    if (!(p >= 0.0 && p < 1.0)) return AVCTC_ERR_BAD_ARG;
    if (!training || p == 0.0) return 0;
    AVCTC_TRY(dropout_geometry(n, &o->threads, incr));
    o->active = 1;
    o->keep = (float)(1.0 - p);
    o->scale = backward ? (float)(1.0 / (1.0 - p)) : (float)(1.0 / (double)o->keep);
    return 0;
}

// The three dropouts of attn_out_ffn in module order (hidden after out_proj, intermediate, output) on consecutive
// generator offsets from `offset`.
int make_drops(const Dims& d, const double p[3], int training, unsigned long long seed, unsigned long long offset,
               bool backward, Drop out[3], long long* total_incr) {
    const long long n[3] = {d.M * d.E, d.M * d.F, d.M * d.E};
    long long total = 0;
    for (int i = 0; i < 3; ++i) {
        long long incr = 0;
        AVCTC_TRY(make_drop(n[i], p[i], training, seed, offset + (unsigned long long)total, backward, &out[i], &incr));
        total += incr;
    }
    if (total_incr) *total_incr = total;
    return 0;
}

int elementwise_grid(long long n) {
    long long g = (n / 8 + 255) / 256;
    return (int)(g < 148 * 8 ? (g > 0 ? g : 1) : 148 * 8);
}

template <bool RESID>
int launch_ln_fwd(const bf* a, const bf* res, const Drop& dr, const Dims& d, const float* g, const float* b, float eps,
                  bf* h, bf* y, float* mean, float* rstd, cudaStream_t st) {
    const dim3 grid((unsigned)((d.M + kRowsPerCta - 1) / kRowsPerCta));
    switch (d.E / 256) {
        case 1: ln_fwd_kernel<1, RESID><<<grid, 256, 0, st>>>(a, res, dr, d.M, g, b, eps, h, y, mean, rstd); break;
        case 2: ln_fwd_kernel<2, RESID><<<grid, 256, 0, st>>>(a, res, dr, d.M, g, b, eps, h, y, mean, rstd); break;
        case 3: ln_fwd_kernel<3, RESID><<<grid, 256, 0, st>>>(a, res, dr, d.M, g, b, eps, h, y, mean, rstd); break;
        default: ln_fwd_kernel<4, RESID><<<grid, 256, 0, st>>>(a, res, dr, d.M, g, b, eps, h, y, mean, rstd); break;
    }
    AVCTC_CUDA_RETURN(cudaGetLastError());
    return 0;
}

int ln_bwd_ctas(long long M) {
    const long long need = (M + kRowsPerCta - 1) / kRowsPerCta;
    return (int)(need < kLnBwdCtas ? need : kLnBwdCtas);
}

template <bool RESID>
int launch_ln_bwd(const bf* dy, const bf* x, const float* mean, const float* rstd, const float* g, const Dims& d,
                  const bf* res, const Drop& dr, bf* out, bf* out2, float* part, cudaStream_t st) {
    const int grid = ln_bwd_ctas(d.M);
    switch (d.E / 256) {
        case 1: ln_bwd_kernel<1, RESID><<<grid, 256, 0, st>>>(dy, x, mean, rstd, g, d.M, res, dr, out, out2, part); break;
        case 2: ln_bwd_kernel<2, RESID><<<grid, 256, 0, st>>>(dy, x, mean, rstd, g, d.M, res, dr, out, out2, part); break;
        case 3: ln_bwd_kernel<3, RESID><<<grid, 256, 0, st>>>(dy, x, mean, rstd, g, d.M, res, dr, out, out2, part); break;
        default: ln_bwd_kernel<4, RESID><<<grid, 256, 0, st>>>(dy, x, mean, rstd, g, d.M, res, dr, out, out2, part); break;
    }
    AVCTC_CUDA_RETURN(cudaGetLastError());
    return 0;
}

bool misaligned(std::initializer_list<const void*> ps) {
    for (const void* p : ps)
        if (reinterpret_cast<uintptr_t>(p) & 15) return true;
    return false;
}

}  // namespace
}  // namespace avctc

using namespace avctc;

extern "C" size_t avctc_w2v_workspace_bytes(long long M, int E, int F, int which) {
    Dims d;
    if (!make_dims(M, E, F, &d)) return 0;
    switch (which) {
        case 0: return carve_in_saved(nullptr, d).total;
        case 1: return carve_out_saved(nullptr, d).total;
        case 2: return carve_in_scratch(nullptr, d).total;
        case 3: return carve_out_scratch(nullptr, d).total;
        default: return 0;
    }
}

extern "C" long long avctc_w2v_dropout_increment(long long M, int E, int F, double p_hidden, double p_act, double p_out,
                                                 int training) {
    Dims d;
    if (!make_dims(M, E, F, &d)) return AVCTC_ERR_UNSUPPORTED;
    const double p[3] = {p_hidden, p_act, p_out};
    Drop dr[3];
    long long total = 0;
    const int rc = make_drops(d, p, training, 0, 0, false, dr, &total);
    return rc ? (rc > 0 ? -rc : rc) : total;
}

extern "C" int avctc_w2v_dropout(const void* x, long long n, double p, unsigned long long seed, unsigned long long offset,
                                 void* y, void* stream) {
    if (!x || !y || n <= 0 || n % 8) return AVCTC_ERR_BAD_ARG;
    if (misaligned({x, y})) return AVCTC_ERR_ALIGNMENT;
    Drop dr;
    long long incr = 0;
    AVCTC_TRY(make_drop(n, p, 1, seed, offset, false, &dr, &incr));
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    drop_bwd_kernel<false><<<elementwise_grid(n), 256, 0, st>>>(reinterpret_cast<const bf*>(x), nullptr, n, dr,
                                                                 reinterpret_cast<bf*>(y));
    AVCTC_CUDA_RETURN(cudaGetLastError());
    return 0;
}

extern "C" int avctc_w2v_attn_in_forward(const void* x, long long M, int E, const float* ln_w, const float* ln_b, float eps,
                                         const void* wqkv, const float* bqkv, void* q, void* k, void* v, void* saved,
                                         size_t saved_bytes, void* stream) {
    Dims d;
    if (!make_dims(M, E, 8, &d)) return AVCTC_ERR_UNSUPPORTED;
    if (!x || !ln_w || !ln_b || !wqkv || !bqkv || !q || !k || !v || !saved) return AVCTC_ERR_BAD_ARG;
    if (misaligned({x, ln_w, ln_b, wqkv, q, k, v, saved})) return AVCTC_ERR_ALIGNMENT;
    InSaved s = carve_in_saved(saved, d);
    if (saved_bytes < s.total) return AVCTC_ERR_WORKSPACE;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    Drop none{};
    AVCTC_TRY(launch_ln_fwd<false>(reinterpret_cast<const bf*>(x), nullptr, none, d, ln_w, ln_b, eps, nullptr, s.ln, s.mean,
                                   s.rstd, st));
    const bf* w = reinterpret_cast<const bf*>(wqkv);
    const size_t EE = (size_t)E * E;
    AvctcGemmJob g[3] = {linear_job(s.ln, E, w, bqkv, M, E, E, q, AVCTC_BF16, E),
                         linear_job(s.ln, E, w + EE, bqkv + E, M, E, E, k, AVCTC_BF16, E),
                         linear_job(s.ln, E, w + 2 * EE, bqkv + 2 * E, M, E, E, v, AVCTC_BF16, E)};
    return avctc_gemm_launch_group(g, 3, stream);
}

extern "C" int avctc_w2v_attn_in_backward(const void* dq, const void* dk, const void* dv, const void* x, long long M, int E,
                                          const float* ln_w, const void* wqkv, void* dx, float* g_wqkv, float* g_bqkv,
                                          float* g_lnw, float* g_lnb, const void* saved, size_t saved_bytes, void* scratch,
                                          size_t scratch_bytes, void* stream) {
    Dims d;
    if (!make_dims(M, E, 8, &d)) return AVCTC_ERR_UNSUPPORTED;
    if (!dq || !dk || !dv || !x || !ln_w || !wqkv || !dx || !saved || !scratch) return AVCTC_ERR_BAD_ARG;
    const bool wg = g_wqkv != nullptr;
    if (wg != (g_bqkv != nullptr) || wg != (g_lnw != nullptr) || wg != (g_lnb != nullptr)) return AVCTC_ERR_BAD_ARG;
    if (misaligned({dq, dk, dv, x, ln_w, wqkv, dx, saved, scratch})) return AVCTC_ERR_ALIGNMENT;
    InSaved s = carve_in_saved(const_cast<void*>(saved), d);
    InScratch w = carve_in_scratch(scratch, d);
    if (saved_bytes < s.total || scratch_bytes < w.total) return AVCTC_ERR_WORKSPACE;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    const int E3 = 3 * E;
    pack3_kernel<<<elementwise_grid(M * E3), 256, 0, st>>>(reinterpret_cast<const bf*>(dq), reinterpret_cast<const bf*>(dk),
                                                          reinterpret_cast<const bf*>(dv), M, E, w.dqkv);
    AVCTC_CUDA_RETURN(cudaGetLastError());
    {   // input gradient of the three projections (one K = 3E GEMM) and, when trained, their weight gradient
        AvctcGemmJob g[2] = {dgrad_job(w.dqkv, E3, reinterpret_cast<const bf*>(wqkv), M, E3, E, w.dln),
                             wgrad_job(w.dqkv, E3, s.ln, E, M, E3, E, g_wqkv, E, false, tiles_of(M, E))};
        AVCTC_TRY(avctc_gemm_launch_group(g, wg ? 2 : 1, stream));
    }
    Drop none{};
    AVCTC_TRY(launch_ln_bwd<false>(w.dln, reinterpret_cast<const bf*>(x), s.mean, s.rstd, ln_w, d, nullptr, none,
                                   reinterpret_cast<bf*>(dx), nullptr, wg ? w.lnpart : nullptr, st));
    if (wg) {
        ColJobs cj{};
        cj.count = 1; cj.M = M;
        cj.j[0] = {w.dqkv, E3, w.colpart};
        colsum_part_kernel<<<dim3((E3 / 2 + 255) / 256, kColParts, 1), 256, 0, st>>>(cj);
        AVCTC_CUDA_RETURN(cudaGetLastError());
        const int P = ln_bwd_ctas(M);
        SumJobs sj{};
        sj.count = 3;
        sj.j[0] = {w.colpart, kColParts, E3, g_bqkv};
        sj.j[1] = {w.lnpart, P, E, g_lnw};
        sj.j[2] = {w.lnpart + (size_t)P * E, P, E, g_lnb};
        sum_parts_kernel<<<dim3((E3 + 255) / 256, 3), 256, 0, st>>>(sj);
        AVCTC_CUDA_RETURN(cudaGetLastError());
    }
    return AVCTC_OK;
}

extern "C" int avctc_w2v_attn_out_ffn_forward(const void* attn, const void* x, long long M, int E, int F, const void* wo,
                                              const float* bo, const float* ln_w, const float* ln_b, float eps,
                                              const void* w1, const float* b1, const void* w2, const float* b2,
                                              double p_hidden, double p_act, double p_out, int training,
                                              unsigned long long seed, unsigned long long offset, void* y, void* saved,
                                              size_t saved_bytes, void* stream) {
    Dims d;
    if (!make_dims(M, E, F, &d)) return AVCTC_ERR_UNSUPPORTED;
    if (!attn || !x || !wo || !bo || !ln_w || !ln_b || !w1 || !b1 || !w2 || !b2 || !y || !saved) return AVCTC_ERR_BAD_ARG;
    if (misaligned({attn, x, wo, ln_w, ln_b, w1, w2, y, saved})) return AVCTC_ERR_ALIGNMENT;
    OutSaved s = carve_out_saved(saved, d);
    if (saved_bytes < s.total) return AVCTC_ERR_WORKSPACE;
    const double p[3] = {p_hidden, p_act, p_out};
    Drop dr[3];
    AVCTC_TRY(make_drops(d, p, training, seed, offset, false, dr, nullptr));
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    const bf* xb = reinterpret_cast<const bf*>(x);
    AvctcGemmJob j = linear_job(reinterpret_cast<const bf*>(attn), E, reinterpret_cast<const bf*>(wo), bo, M, E, E, s.ao,
                                AVCTC_BF16, E);
    AVCTC_TRY(avctc_gemm_launch_group(&j, 1, stream));
    AVCTC_TRY(launch_ln_fwd<true>(s.ao, xb, dr[0], d, ln_w, ln_b, eps, s.h, s.ln, s.mean, s.rstd, st));
    j = linear_job(s.ln, E, reinterpret_cast<const bf*>(w1), b1, M, F, E, s.pre, AVCTC_BF16, F);
    AVCTC_TRY(avctc_gemm_launch_group(&j, 1, stream));
    gelu_drop_kernel<<<elementwise_grid(M * F), 256, 0, st>>>(s.pre, M * F, dr[1], s.act);
    AVCTC_CUDA_RETURN(cudaGetLastError());
    j = linear_job(s.act, F, reinterpret_cast<const bf*>(w2), b2, M, E, F, s.z, AVCTC_BF16, E);
    AVCTC_TRY(avctc_gemm_launch_group(&j, 1, stream));
    resid_drop_kernel<<<elementwise_grid(M * E), 256, 0, st>>>(s.z, s.h, M * E, dr[2], reinterpret_cast<bf*>(y));
    AVCTC_CUDA_RETURN(cudaGetLastError());
    return AVCTC_OK;
}

extern "C" int avctc_w2v_attn_out_ffn_backward(const void* dy, const void* attn, long long M, int E, int F, const void* wo,
                                               const float* ln_w, const void* w1, const void* w2, double p_hidden,
                                               double p_act, double p_out, int training, unsigned long long seed,
                                               unsigned long long offset, void* dattn, void* dx, float* g_wo, float* g_bo,
                                               float* g_lnw, float* g_lnb, float* g_w1, float* g_b1, float* g_w2,
                                               float* g_b2, const void* saved, size_t saved_bytes, void* scratch,
                                               size_t scratch_bytes, void* stream) {
    Dims d;
    if (!make_dims(M, E, F, &d)) return AVCTC_ERR_UNSUPPORTED;
    if (!dy || !attn || !wo || !ln_w || !w1 || !w2 || !dattn || !dx || !saved || !scratch) return AVCTC_ERR_BAD_ARG;
    const bool wg = g_wo != nullptr;
    for (const float* p : {g_bo, g_lnw, g_lnb, g_w1, g_b1, g_w2, g_b2})
        if ((p != nullptr) != wg) return AVCTC_ERR_BAD_ARG;
    if (misaligned({dy, attn, wo, ln_w, w1, w2, dattn, dx, saved, scratch})) return AVCTC_ERR_ALIGNMENT;
    OutSaved s = carve_out_saved(const_cast<void*>(saved), d);
    OutScratch w = carve_out_scratch(scratch, d);
    if (saved_bytes < s.total || scratch_bytes < w.total) return AVCTC_ERR_WORKSPACE;
    const double p[3] = {p_hidden, p_act, p_out};
    Drop dr[3];
    AVCTC_TRY(make_drops(d, p, training, seed, offset, true, dr, nullptr));
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    const bf* dyb = reinterpret_cast<const bf*>(dy);
    const int tE = tiles_of(M, E), tF = tiles_of(M, F);
    drop_bwd_kernel<false><<<elementwise_grid(M * E), 256, 0, st>>>(dyb, nullptr, M * E, dr[2], w.dz);
    AVCTC_CUDA_RETURN(cudaGetLastError());
    {   // output_dense
        AvctcGemmJob g[2] = {dgrad_job(w.dz, E, reinterpret_cast<const bf*>(w2), M, E, F, w.da),
                             wgrad_job(w.dz, E, s.act, F, M, E, F, g_w2, F, false, tF)};
        AVCTC_TRY(avctc_gemm_launch_group(g, wg ? 2 : 1, stream));
    }
    drop_bwd_kernel<true><<<elementwise_grid(M * F), 256, 0, st>>>(w.da, s.pre, M * F, dr[1], w.da);
    AVCTC_CUDA_RETURN(cudaGetLastError());
    {   // intermediate_dense
        AvctcGemmJob g[2] = {dgrad_job(w.da, F, reinterpret_cast<const bf*>(w1), M, F, E, w.dln),
                             wgrad_job(w.da, F, s.ln, E, M, F, E, g_w1, E, false, tE)};
        AVCTC_TRY(avctc_gemm_launch_group(g, wg ? 2 : 1, stream));
    }
    AVCTC_TRY(launch_ln_bwd<true>(w.dln, s.h, s.mean, s.rstd, ln_w, d, dyb, dr[0], reinterpret_cast<bf*>(dx), w.dzo,
                                  wg ? w.lnpart : nullptr, st));
    {   // out_proj
        AvctcGemmJob g[2] = {dgrad_job(w.dzo, E, reinterpret_cast<const bf*>(wo), M, E, E, reinterpret_cast<bf*>(dattn)),
                             wgrad_job(w.dzo, E, reinterpret_cast<const bf*>(attn), E, M, E, E, g_wo, E, false, tE)};
        AVCTC_TRY(avctc_gemm_launch_group(g, wg ? 2 : 1, stream));
    }
    if (wg) {
        ColJobs cj{};
        cj.count = 3; cj.M = M;
        float* cp = w.colpart;
        cj.j[0] = {w.dz, E, cp};
        cj.j[1] = {w.da, F, cp + (size_t)kColParts * E};
        cj.j[2] = {w.dzo, E, cp + (size_t)kColParts * (E + F)};
        const int maxN = E > F ? E : F;
        colsum_part_kernel<<<dim3((maxN / 2 + 255) / 256, kColParts, 3), 256, 0, st>>>(cj);
        AVCTC_CUDA_RETURN(cudaGetLastError());
        const int P = ln_bwd_ctas(M);
        SumJobs sj{};
        sj.count = 5;
        sj.j[0] = {cj.j[0].part, kColParts, E, g_b2};
        sj.j[1] = {cj.j[1].part, kColParts, F, g_b1};
        sj.j[2] = {cj.j[2].part, kColParts, E, g_bo};
        sj.j[3] = {w.lnpart, P, E, g_lnw};
        sj.j[4] = {w.lnpart + (size_t)P * E, P, E, g_lnb};
        sum_parts_kernel<<<dim3((maxN + 255) / 256, 5), 256, 0, st>>>(sj);
        AVCTC_CUDA_RETURN(cudaGetLastError());
    }
    return AVCTC_OK;
}
