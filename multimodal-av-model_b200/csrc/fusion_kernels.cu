// fusion_kernels.cu — the non-GEMM steps of CrossAttentionFusion / CTCDecoder on sm_100a.
//
//  resample   /root/reference/model/fusion_module.py:40-55,66 : speech-frame select (mask not in {0,3}),
//             per-sample compaction, zero pad to the batch max, linear(align_corners=True) resample of the
//             audio features to T_v frames, nearest resample of the mask, input_lengths = count(mask != 0).
//             The reference does this with B Python iterations, boolean indexing and B .item() syncs; here
//             it is two launches with every length kept on the device.
//  softmax    nn.MultiheadAttention's softmax over ALL T keys (no padding mask, fusion_module.py:61) and its
//             backward; rows live in a [Z, T, Tp] buffer (Tp = T rounded up to 8 for TMA), pad columns zero.
//  colsum     bias gradients.
//  log_softmax  CTCDecoder (model/decoder.py:25) forward/backward over the V classes.
#include "common.cuh"

namespace avctc {

// ------------------------------------------------------------------------------------------ resample
// pass 1: one CTA per sample. rank[b][j] = position of frame j among the speech frames (or -1),
// src[b][i] = original index of the i-th speech frame, cnt[b] = number of speech frames.
__global__ void resample_index_kernel(const int64_t* __restrict__ mask, int B, int Ta, int* __restrict__ rank,
                                      int* __restrict__ src, int* __restrict__ cnt) {
    const int b = blockIdx.x;
    __shared__ int warp_tot[32];
    __shared__ int base_s;
    if (threadIdx.x == 0) base_s = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    for (int j0 = 0; j0 < Ta; j0 += blockDim.x) {
        const int j = j0 + threadIdx.x;
        bool sp = false;
        if (j < Ta) {
            const long long m = mask[(size_t)b * Ta + j];
            sp = (m != 0) && (m != 3);
        }
        const unsigned bal = __ballot_sync(kFullMask, sp);
        const int within = __popc(bal & ((1u << lane) - 1));
        if (lane == 0) warp_tot[warp] = __popc(bal);
        __syncthreads();
        int before = base_s;
        for (int w = 0; w < warp; ++w) before += warp_tot[w];
        if (j < Ta) {
            const int r = sp ? before + within : -1;
            rank[(size_t)b * Ta + j] = r;
            if (sp) src[(size_t)b * Ta + r] = j;
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            int tot = 0;
            for (int w = 0; w < nw; ++w) tot += warp_tot[w];
            base_s += tot;
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) cnt[b] = base_s;
}

struct LerpCoef { int i0, i1; float w0, w1; };
// ATen upsample_linear1d, align_corners=True: src = dst * (in-1)/(out-1) in fp32
__device__ __forceinline__ LerpCoef lerp_coef(int t, int Tp, int Tv) {
    LerpCoef c;
    if (Tp == Tv) { c.i0 = t; c.i1 = t; c.w0 = 1.f; c.w1 = 0.f; return c; }
    const float scale = (Tv > 1) ? (float)(Tp - 1) / (float)(Tv - 1) : 0.f;
    const float s = scale * (float)t;
    c.i0 = (int)s;
    c.i1 = c.i0 + ((c.i0 < Tp - 1) ? 1 : 0);
    c.w1 = s - (float)c.i0;
    c.w0 = 1.f - c.w1;
    return c;
}
// ATen upsample_nearest1d: src = min(floor(dst * float(in)/out), in-1)
__device__ __forceinline__ int nearest_src(int t, int Tp, int Tv) {
    if (Tp == Tv) return t;
    const float scale = (float)Tp / (float)Tv;
    int s = (int)floorf((float)t * scale);
    return s < Tp - 1 ? s : Tp - 1;
}
__device__ __forceinline__ int batch_max(const int* cnt, int B) {
    int m = 0;
    for (int i = threadIdx.x & 31; i < B; i += 32) m = max(m, cnt[i]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(kFullMask, m, o));
    return m;
}

// 8 consecutive elements of a row (nullptr -> zeros) as floats; the row start is 16-byte aligned when D % 8 == 0
__device__ __forceinline__ void load8(const float* r, int d, float (&x)[8]) {
    if (!r) {
#pragma unroll
        for (int k = 0; k < 8; ++k) x[k] = 0.f;
        return;
    }
    const float4 a = *reinterpret_cast<const float4*>(r + d), b = *reinterpret_cast<const float4*>(r + d + 4);
    x[0] = a.x; x[1] = a.y; x[2] = a.z; x[3] = a.w; x[4] = b.x; x[5] = b.y; x[6] = b.z; x[7] = b.w;
}
__device__ __forceinline__ void load8(const __nv_bfloat16* r, int d, float (&x)[8]) {
    if (!r) {
#pragma unroll
        for (int k = 0; k < 8; ++k) x[k] = 0.f;
        return;
    }
    const uint4 raw = *reinterpret_cast<const uint4*>(r + d);
    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&raw);
#pragma unroll
    for (int k = 0; k < 4; ++k) { const float2 f = __bfloat1622float2(h[k]); x[2 * k] = f.x; x[2 * k + 1] = f.y; }
}

template <typename TIn>
__global__ void resample_apply_kernel(const TIn* __restrict__ audio, const int64_t* __restrict__ mask, int B, int Ta,
                                      int D, int Tv, const int* __restrict__ src, const int* __restrict__ cnt,
                                      __nv_bfloat16* __restrict__ out, int64_t* __restrict__ mask_out,
                                      int64_t* __restrict__ input_lengths) {
    const int b = blockIdx.y, t = blockIdx.x;
    const int Tp = batch_max(cnt, B);
    const int nb = cnt[b];
    __nv_bfloat16* orow = out + ((size_t)b * Tv + t) * D;
    if (Tp == 0) {   // no speech anywhere in the batch (the reference raises inside F.interpolate)
        for (int d = threadIdx.x; d < D; d += blockDim.x) orow[d] = __float2bfloat16(0.f);
        if (threadIdx.x == 0) mask_out[(size_t)b * Tv + t] = 0;
        return;
    }
    const LerpCoef c = lerp_coef(t, Tp, Tv);
    const TIn* r0 = (c.i0 < nb) ? audio + ((size_t)b * Ta + src[(size_t)b * Ta + c.i0]) * D : nullptr;
    const TIn* r1 = (c.i1 < nb && c.w1 != 0.f) ? audio + ((size_t)b * Ta + src[(size_t)b * Ta + c.i1]) * D : nullptr;
    if ((D & 7) == 0) {          // 8 elements per thread: 16-byte (bf16) / 2 x 16-byte (fp32) loads, 16-byte stores
        for (int d = threadIdx.x * 8; d < D; d += blockDim.x * 8) {
            float x0[8], x1[8];
            load8(r0, d, x0);
            load8(r1, d, x1);
            uint4 pk;
            __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&pk);
#pragma unroll
            for (int k = 0; k < 4; ++k)
                h[k] = __floats2bfloat162_rn(c.w0 * x0[2 * k] + c.w1 * x1[2 * k], c.w0 * x0[2 * k + 1] + c.w1 * x1[2 * k + 1]);
            *reinterpret_cast<uint4*>(orow + d) = pk;
        }
    } else {
        for (int d = threadIdx.x; d < D; d += blockDim.x) {
            const float x0 = r0 ? to_float(r0[d]) : 0.f;
            const float x1 = r1 ? to_float(r1[d]) : 0.f;
            orow[d] = __float2bfloat16(c.w0 * x0 + c.w1 * x1);
        }
    }
    if (threadIdx.x == 0) {
        const int s = nearest_src(t, Tp, Tv);
        const long long m = (s < nb) ? mask[(size_t)b * Ta + src[(size_t)b * Ta + s]] : 0;
        mask_out[(size_t)b * Tv + t] = m;
        if (m != 0) atomicAdd(reinterpret_cast<unsigned long long*>(input_lengths + b), 1ull);
    }
}

// backward (deterministic gather): d_audio[b][j] = sum_t w(t -> rank j) * d_out[b][t]
template <typename TOut>
__global__ void resample_bwd_kernel(const __nv_bfloat16* __restrict__ dout, int B, int Ta, int D, int Tv,
                                    const int* __restrict__ rank, const int* __restrict__ cnt, TOut* __restrict__ daudio) {
    const int b = blockIdx.y, j = blockIdx.x;
    const int Tp = batch_max(cnt, B);
    const int r = rank[(size_t)b * Ta + j];
    TOut* drow = daudio + ((size_t)b * Ta + j) * D;
    auto put = [](TOut* p, float v) {
        if constexpr (sizeof(TOut) == 4) *p = v; else *p = __float2bfloat16(v);
    };
    if (r < 0 || Tp == 0) {
        if ((D & 7) == 0) {
            for (int d = threadIdx.x * 8; d < D; d += blockDim.x * 8) {
                if constexpr (sizeof(TOut) == 4) {
                    *reinterpret_cast<float4*>(drow + d) = make_float4(0.f, 0.f, 0.f, 0.f);
                    *reinterpret_cast<float4*>(drow + d + 4) = make_float4(0.f, 0.f, 0.f, 0.f);
                } else {
                    *reinterpret_cast<uint4*>(drow + d) = make_uint4(0, 0, 0, 0);
                }
            }
        } else {
            for (int d = threadIdx.x; d < D; d += blockDim.x) put(drow + d, 0.f);
        }
        return;
    }
    // output frames whose stencil can touch padded index r
    int t_lo = 0, t_hi = Tv - 1;
    if (Tp != Tv && Tv > 1 && Tp > 1) {
        const float inv = (float)(Tv - 1) / (float)(Tp - 1);
        t_lo = max(0, (int)floorf((float)(r - 1) * inv) - 1);
        t_hi = min(Tv - 1, (int)ceilf((float)(r + 1) * inv) + 1);
    } else if (Tp == Tv) {
        t_lo = t_hi = r;
    }
    // every output frame of [t_lo, t_hi] whose stencil touches padded index r contributes; the weight is recomputed per
    // frame (uniform across the CTA), so any up-sampling ratio works — Tp == 1 has all Tv frames on index 0
    auto weight = [&](int t) {
        const LerpCoef c = lerp_coef(t, Tp, Tv);
        float w = 0.f;
        if (c.i0 == r) w += c.w0;
        if (c.i1 == r && c.w1 != 0.f) w += c.w1;
        return w;
    };
    if ((D & 7) == 0) {
        for (int d = threadIdx.x * 8; d < D; d += blockDim.x * 8) {
            float acc[8];
#pragma unroll
            for (int k = 0; k < 8; ++k) acc[k] = 0.f;
            for (int t = t_lo; t <= t_hi; ++t) {
                const float w = weight(t);
                if (w == 0.f) continue;
                float x[8];
                load8(dout + ((size_t)b * Tv + t) * D, d, x);
#pragma unroll
                for (int k = 0; k < 8; ++k) acc[k] += w * x[k];
            }
            if constexpr (sizeof(TOut) == 4) {
                *reinterpret_cast<float4*>(drow + d) = make_float4(acc[0], acc[1], acc[2], acc[3]);
                *reinterpret_cast<float4*>(drow + d + 4) = make_float4(acc[4], acc[5], acc[6], acc[7]);
            } else {
                uint4 pk;
                __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&pk);
#pragma unroll
                for (int k = 0; k < 4; ++k) h[k] = __floats2bfloat162_rn(acc[2 * k], acc[2 * k + 1]);
                *reinterpret_cast<uint4*>(drow + d) = pk;
            }
        }
        return;
    }
    for (int d = threadIdx.x; d < D; d += blockDim.x) {
        float acc = 0.f;
        for (int t = t_lo; t <= t_hi; ++t) {
            const float w = weight(t);
            if (w != 0.f) acc += w * __bfloat162float(dout[((size_t)b * Tv + t) * D + d]);
        }
        put(drow + d, acc);
    }
}

// ------------------------------------------------------------------------------------------ softmax
// one warp per row; S fp32 [rows][Tp] (first T valid) -> P bf16 [rows][Tp], pad columns written as 0
__global__ void softmax_fwd_kernel(const float* __restrict__ S, __nv_bfloat16* __restrict__ P, long long rows, int T,
                                   int Tp) {
    pdl_launch_dependents();
    pdl_wait();
    const long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (row >= rows) return;
    const int lane = threadIdx.x & 31;
    const float* s = S + row * Tp;
    float m = AVCTC_NEG_INF;
    for (int c = lane; c < T; c += 32) m = fmaxf(m, s[c]);
    m = warp_max(m);
    float sum = 0.f;
    for (int c = lane; c < T; c += 32) sum += __expf(s[c] - m);
    sum = warp_sum(sum);
    const float inv = 1.f / sum;
    __nv_bfloat16* p = P + row * Tp;
    for (int c = lane; c < Tp; c += 32) p[c] = __float2bfloat16(c < T ? __expf(s[c] - m) * inv : 0.f);
}
// dS = P * (dP - sum_k dP*P)
__global__ void softmax_bwd_kernel(const __nv_bfloat16* __restrict__ P, const float* __restrict__ dP,
                                   __nv_bfloat16* __restrict__ dS, long long rows, int T, int Tp) {
    pdl_launch_dependents();
    pdl_wait();
    const long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (row >= rows) return;
    const int lane = threadIdx.x & 31;
    const __nv_bfloat16* p = P + row * Tp;
    const float* dp = dP + row * Tp;
    float dot = 0.f;
    for (int c = lane; c < T; c += 32) dot += __bfloat162float(p[c]) * dp[c];
    dot = warp_sum(dot);
    __nv_bfloat16* ds = dS + row * Tp;
    for (int c = lane; c < Tp; c += 32)
        ds[c] = __float2bfloat16(c < T ? __bfloat162float(p[c]) * (dp[c] - dot) : 0.f);
}

// ------------------------------------------------------------------------------------------ colsum
// out[n] (+)= sum_m X[m][n]; block = 32 columns x 8 row-lanes over one of gridDim.y row chunks; chunk sums are
// added with fp32 atomics into an `out` the host zeroed (the sum order of the <= 64 chunk totals is not fixed).
template <typename TIn>
__global__ void colsum_kernel(const TIn* __restrict__ X, long long M, int N, long long ld, float* __restrict__ out) {
    __shared__ float part[8][33];
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int n = blockIdx.x * 32 + tx;
    const long long per = (M + gridDim.y - 1) / gridDim.y;
    const long long m0 = (long long)blockIdx.y * per, m1 = (m0 + per < M) ? m0 + per : M;
    float acc = 0.f;
    if (n < N)
        for (long long m = m0 + ty; m < m1; m += 8) acc += to_float(X[m * ld + n]);
    part[ty][tx] = acc;
    __syncthreads();
    if (ty == 0 && n < N) {
        float s = 0.f;
#pragma unroll
        for (int i = 0; i < 8; ++i) s += part[i][tx];
        atomicAdd(out + n, s);
    }
}

// ------------------------------------------------------------------------------------------ log_softmax
// one warp per row of V classes; logits fp32 or bf16 -> log-probs (same or fp32)
template <typename TIn, typename TOut>
__global__ void log_softmax_fwd_kernel(const TIn* __restrict__ X, TOut* __restrict__ Y, long long rows, int V) {
    const long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (row >= rows) return;
    const int lane = threadIdx.x & 31;
    const TIn* x = X + row * V;
    float m = AVCTC_NEG_INF;
    for (int c = lane; c < V; c += 32) m = fmaxf(m, to_float(x[c]));
    m = warp_max(m);
    float sum = 0.f;
    for (int c = lane; c < V; c += 32) sum += expf(to_float(x[c]) - m);
    sum = warp_sum(sum);
    const float lse = m + logf(sum);
    TOut* y = Y + row * V;
    for (int c = lane; c < V; c += 32) {
        const float v = to_float(x[c]) - lse;
        if constexpr (sizeof(TOut) == 4) y[c] = v; else y[c] = __float2bfloat16(v);
    }
}
// dX = dY - exp(Y) * sum(dY)   (dX written as bf16 for the following tcgen05 GEMMs)
template <typename TY>
__global__ void log_softmax_bwd_kernel(const TY* __restrict__ Y, const TY* __restrict__ dY,
                                       __nv_bfloat16* __restrict__ dX, long long rows, int V, long long ldx) {
    const long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (row >= rows) return;
    const int lane = threadIdx.x & 31;
    const TY* y = Y + row * V;
    const TY* dy = dY + row * V;
    float s = 0.f;
    for (int c = lane; c < V; c += 32) s += to_float(dy[c]);
    s = warp_sum(s);
    __nv_bfloat16* dx = dX + row * ldx;
    for (int c = lane; c < V; c += 32) dx[c] = __float2bfloat16(to_float(dy[c]) - expf(to_float(y[c])) * s);
}

}  // namespace avctc

using namespace avctc;

extern "C" size_t avctc_resample_workspace_bytes(int B, int Ta) {
    if (B < 0 || Ta < 0) return 0;
    return ((size_t)2 * B * Ta + B) * sizeof(int) + 256;
}

extern "C" int avctc_resample_forward(const void* audio, int dtype, const int64_t* mask, int B, int Ta, int D, int Tv,
                                      void* out_bf16, int64_t* mask_out, int64_t* input_lengths, void* workspace,
                                      size_t workspace_bytes, void* stream) {
    if (B <= 0 || Ta <= 0 || D <= 0 || Tv <= 0) return AVCTC_ERR_BAD_ARG;
    if (!audio || !mask || !out_bf16 || !mask_out || !input_lengths || !workspace) return AVCTC_ERR_BAD_ARG;
    if (workspace_bytes < avctc_resample_workspace_bytes(B, Ta)) return AVCTC_ERR_WORKSPACE;
    if (dtype != AVCTC_F32 && dtype != AVCTC_BF16) return AVCTC_ERR_BAD_ARG;
    if ((D & 7) == 0 && ((reinterpret_cast<uintptr_t>(audio) | reinterpret_cast<uintptr_t>(out_bf16)) & 15))
        return AVCTC_ERR_ALIGNMENT;      // the 8-wide path uses 16-byte accesses
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    int* rank = reinterpret_cast<int*>(workspace);
    int* src = rank + (size_t)B * Ta;
    int* cnt = src + (size_t)B * Ta;
    AVCTC_CUDA_RETURN(cudaMemsetAsync(input_lengths, 0, sizeof(int64_t) * B, st));
    resample_index_kernel<<<B, 256, 0, st>>>(mask, B, Ta, rank, src, cnt);
    dim3 grid(Tv, B);
    if (dtype == AVCTC_F32)
        resample_apply_kernel<float><<<grid, 128, 0, st>>>(reinterpret_cast<const float*>(audio), mask, B, Ta, D, Tv, src,
                                                          cnt, reinterpret_cast<__nv_bfloat16*>(out_bf16), mask_out,
                                                          input_lengths);
    else if (dtype == AVCTC_BF16)
        resample_apply_kernel<__nv_bfloat16><<<grid, 128, 0, st>>>(reinterpret_cast<const __nv_bfloat16*>(audio), mask, B,
                                                                  Ta, D, Tv, src, cnt,
                                                                  reinterpret_cast<__nv_bfloat16*>(out_bf16), mask_out,
                                                                  input_lengths);
    return (int)cudaGetLastError();
}

extern "C" int avctc_resample_backward(const void* dout_bf16, int B, int Ta, int D, int Tv, const void* workspace,
                                       void* daudio, int dtype, void* stream) {
    if (B <= 0 || Ta <= 0 || D <= 0 || Tv <= 0 || !dout_bf16 || !workspace || !daudio) return AVCTC_ERR_BAD_ARG;
    if ((D & 7) == 0 && ((reinterpret_cast<uintptr_t>(dout_bf16) | reinterpret_cast<uintptr_t>(daudio)) & 15))
        return AVCTC_ERR_ALIGNMENT;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    const int* rank = reinterpret_cast<const int*>(workspace);
    const int* cnt = rank + (size_t)2 * B * Ta;
    dim3 grid(Ta, B);
    const __nv_bfloat16* d = reinterpret_cast<const __nv_bfloat16*>(dout_bf16);
    if (dtype == AVCTC_F32)
        resample_bwd_kernel<float><<<grid, 128, 0, st>>>(d, B, Ta, D, Tv, rank, cnt, reinterpret_cast<float*>(daudio));
    else if (dtype == AVCTC_BF16)
        resample_bwd_kernel<__nv_bfloat16><<<grid, 128, 0, st>>>(d, B, Ta, D, Tv, rank, cnt,
                                                                reinterpret_cast<__nv_bfloat16*>(daudio));
    else return AVCTC_ERR_BAD_ARG;
    return (int)cudaGetLastError();
}

extern "C" int avctc_softmax_forward(const float* S, void* P_bf16, long long rows, int T, int Tp, void* stream) {
    if (!S || !P_bf16 || rows <= 0 || T <= 0 || Tp < T) return AVCTC_ERR_BAD_ARG;
    const int wpb = 8;
    return (int)avctc_launch_pdl(softmax_fwd_kernel, dim3((unsigned)((rows + wpb - 1) / wpb)), dim3(wpb * 32), 0,
                                 reinterpret_cast<cudaStream_t>(stream), S, reinterpret_cast<__nv_bfloat16*>(P_bf16), rows, T, Tp);
}
extern "C" int avctc_softmax_backward(const void* P_bf16, const float* dP, void* dS_bf16, long long rows, int T, int Tp,
                                      void* stream) {
    if (!P_bf16 || !dP || !dS_bf16 || rows <= 0 || T <= 0 || Tp < T) return AVCTC_ERR_BAD_ARG;
    const int wpb = 8;
    return (int)avctc_launch_pdl(softmax_bwd_kernel, dim3((unsigned)((rows + wpb - 1) / wpb)), dim3(wpb * 32), 0,
                                 reinterpret_cast<cudaStream_t>(stream), reinterpret_cast<const __nv_bfloat16*>(P_bf16), dP,
                                 reinterpret_cast<__nv_bfloat16*>(dS_bf16), rows, T, Tp);
}

extern "C" int avctc_colsum(const void* X, int dtype, long long M, int N, long long ld, float* out, int accumulate,
                            void* stream) {
    if (!X || !out || M <= 0 || N <= 0 || ld < N) return AVCTC_ERR_BAD_ARG;
    if (dtype != AVCTC_F32 && dtype != AVCTC_BF16) return AVCTC_ERR_BAD_ARG;   // before the memset: out stays intact
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    int chunks = (int)((M + 127) / 128);
    if (chunks > 64) chunks = 64;
    const dim3 grid((N + 31) / 32, chunks);
    if (!accumulate) AVCTC_CUDA_RETURN(cudaMemsetAsync(out, 0, sizeof(float) * (size_t)N, st));
    if (dtype == AVCTC_F32) colsum_kernel<float><<<grid, 256, 0, st>>>(reinterpret_cast<const float*>(X), M, N, ld, out);
    else if (dtype == AVCTC_BF16)
        colsum_kernel<__nv_bfloat16><<<grid, 256, 0, st>>>(reinterpret_cast<const __nv_bfloat16*>(X), M, N, ld, out);
    return (int)cudaGetLastError();
}

extern "C" int avctc_log_softmax_forward(const void* X, int in_dtype, void* Y, int out_dtype, long long rows, int V,
                                         void* stream) {
    if (!X || !Y || rows <= 0 || V <= 0) return AVCTC_ERR_BAD_ARG;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    const int wpb = 8;
    const unsigned grid = (unsigned)((rows + wpb - 1) / wpb);
    if (in_dtype == AVCTC_F32 && out_dtype == AVCTC_F32)
        log_softmax_fwd_kernel<float, float><<<grid, wpb * 32, 0, st>>>(reinterpret_cast<const float*>(X), reinterpret_cast<float*>(Y), rows, V);
    else if (in_dtype == AVCTC_BF16 && out_dtype == AVCTC_F32)
        log_softmax_fwd_kernel<__nv_bfloat16, float><<<grid, wpb * 32, 0, st>>>(reinterpret_cast<const __nv_bfloat16*>(X), reinterpret_cast<float*>(Y), rows, V);
    else if (in_dtype == AVCTC_F32 && out_dtype == AVCTC_BF16)
        log_softmax_fwd_kernel<float, __nv_bfloat16><<<grid, wpb * 32, 0, st>>>(reinterpret_cast<const float*>(X), reinterpret_cast<__nv_bfloat16*>(Y), rows, V);
    else if (in_dtype == AVCTC_BF16 && out_dtype == AVCTC_BF16)
        log_softmax_fwd_kernel<__nv_bfloat16, __nv_bfloat16><<<grid, wpb * 32, 0, st>>>(reinterpret_cast<const __nv_bfloat16*>(X), reinterpret_cast<__nv_bfloat16*>(Y), rows, V);
    else return AVCTC_ERR_BAD_ARG;
    return (int)cudaGetLastError();
}
extern "C" int avctc_log_softmax_backward(const void* Y, const void* dY, int dtype, void* dX_bf16, long long rows, int V,
                                          long long ldx, void* stream) {
    if (!Y || !dY || !dX_bf16 || rows <= 0 || V <= 0 || ldx < V) return AVCTC_ERR_BAD_ARG;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    const int wpb = 8;
    const unsigned grid = (unsigned)((rows + wpb - 1) / wpb);
    if (dtype == AVCTC_F32)
        log_softmax_bwd_kernel<float><<<grid, wpb * 32, 0, st>>>(reinterpret_cast<const float*>(Y), reinterpret_cast<const float*>(dY), reinterpret_cast<__nv_bfloat16*>(dX_bf16), rows, V, ldx);
    else if (dtype == AVCTC_BF16)
        log_softmax_bwd_kernel<__nv_bfloat16><<<grid, wpb * 32, 0, st>>>(reinterpret_cast<const __nv_bfloat16*>(Y), reinterpret_cast<const __nv_bfloat16*>(dY), reinterpret_cast<__nv_bfloat16*>(dX_bf16), rows, V, ldx);
    else return AVCTC_ERR_BAD_ARG;
    return (int)cudaGetLastError();
}
