// visual_encoder.cu — the frozen VisualEncoder forward (encoders.py) around cuDNN's 3x3 / 1x1 trunk convolutions:
// the front end (temporal taps + 7x7/2 convolution) as one implicit-GEMM kernel, train-mode BatchNorm statistics as
// per-CTA partials combined in a fixed order, and fused BatchNorm-apply / PReLU / residual / pooling passes.
//
// Layout: every activation is NHWC bf16 ([rows, C], C contiguous), math in fp32.  Each kernel rounds to bf16 where the
// eager module path materialises a bf16 tensor (after BN, after PReLU, after the residual add), so results differ
// from eager only by the order of the statistics reductions.  Statistics partials are (count, mean, M2) per channel
// in a [3][C][P] fp32 buffer (P = number of producing CTAs), merged with Chan's formula in a fixed order: no float
// atomics, every run is bit-identical.
#include "common.cuh"

namespace {

constexpr int kFrontC = 64;                   // output channels of the front-end convolution
constexpr int kTaps = 5, kKH = 7, kKW = 7;    // (5,7,7) kernel, stride (1,2,2), padding (2,3,3)
constexpr int kK = kTaps * kKH * kKW;         // 245
constexpr int kKPad = 256;                    // K padded to 16 x k16 steps (weights zero beyond 245)
constexpr int kWStride = 264;                 // smem row stride of the weights (bf16): conflict-free B fragments
constexpr int kTileH = 16, kTileW = 48;       // output pixels per CTA: 16 rows x 48 columns = 48 m16 tiles
constexpr int kHaloH = 2 * (kTileH - 1) + kKH;  // 37 input rows
constexpr int kHaloW = 104;                   // 2 * (48 - 1) + 7 = 101 input columns, padded
constexpr int kFrontThreads = 256;            // 8 warps x 6 m16 tiles each, two at a time
constexpr int kStatThreads = 256;

struct Stat {
    float n, mean, m2;
};

__device__ __forceinline__ Stat chan_merge(Stat a, Stat b) {
    if (b.n == 0.f) return a;
    if (a.n == 0.f) return b;
    const float n = a.n + b.n;
    const float d = b.mean - a.mean;
    const float f = b.n / n;
    return Stat{n, a.mean + d * f, a.m2 + b.m2 + d * d * a.n * f};
}

__device__ __forceinline__ float bf16r(float v) { return __bfloat162float(__float2bfloat16_rn(v)); }

__device__ __forceinline__ float prelu_bf16(float z, float slope) { return z > 0.f ? z : bf16r(slope * z); }

__device__ __forceinline__ void unpack8(const uint4& u, float* f) {
    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&u);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const float2 v = __bfloat1622float2(h[i]);
        f[2 * i] = v.x;
        f[2 * i + 1] = v.y;
    }
}

__device__ __forceinline__ uint4 pack8(const float* f) {
    uint4 u;
    __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&u);
#pragma unroll
    for (int i = 0; i < 4; ++i) h[i] = __floats2bfloat162_rn(f[2 * i], f[2 * i + 1]);
    return u;
}

__device__ __forceinline__ void mma_bf16_16816(float* c, const uint32_t* a, uint32_t b0, uint32_t b1) {
    asm volatile(
        "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, "
        "{%0,%1,%2,%3};"
        : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

__device__ __forceinline__ uint32_t pack2(unsigned short lo, unsigned short hi) {
    return (uint32_t)lo | ((uint32_t)hi << 16);
}

}  // namespace

// ---------------------------------------------------------------------------------------------------------------
// Front end: y[n, oh, ow, co] = sum_{kt,kh,kw} w[co, kt, kh, kw] * bf16(x[b, t+kt-2, 2oh+kh-3, 2ow+kw-3]), n = b*T+t,
// zero outside the clip.  One CTA = one frame x 16 output rows x 48 output columns.  The 5 temporal taps of its input
// halo are staged in shared memory, rounded to bf16 as autocast rounds the taps; the GEMM (M = 768 pixels, N = 64,
// K = 245 -> 256) runs on mma.sync with A fragments gathered through a k -> smem offset table.  The epilogue writes
// bf16 y and the CTA's per-channel (count, mean, M2) of the bf16-rounded outputs (partials == nullptr: no statistics).
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kFrontThreads, 2)
vis_frontend_conv_kernel(const float* __restrict__ x, int T, int H, int W, int Ho, int Wo,
                         const __nv_bfloat16* __restrict__ wts, __nv_bfloat16* __restrict__ y,
                         float* __restrict__ partials, int P) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __nv_bfloat16* w_s = reinterpret_cast<__nv_bfloat16*>(smem_raw);                  // [64][kWStride]
    unsigned short* halo = reinterpret_cast<unsigned short*>(w_s + kFrontC * kWStride);  // [5][kHaloH][kHaloW]
    int* koff = reinterpret_cast<int*>(halo + kTaps * kHaloH * kHaloW);               // [256]
    Stat* wstat = reinterpret_cast<Stat*>(koff + kKPad);                               // [8 warps][64]

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int ow0 = blockIdx.x * kTileW, oh0 = blockIdx.y * kTileH;
    const int n = blockIdx.z, b = n / T, t = n - b * T;
    const int ih0 = 2 * oh0 - 3, iw0 = 2 * ow0 - 3;

    {   // weights: 64 x 256 bf16, 16-byte copies
        const uint4* src = reinterpret_cast<const uint4*>(wts);
        for (int i = tid; i < kFrontC * kKPad / 8; i += kFrontThreads) {
            const int r = i / (kKPad / 8), c = i - r * (kKPad / 8);
            *reinterpret_cast<uint4*>(w_s + r * kWStride + c * 8) = src[i];
        }
    }
    for (int k = tid; k < kKPad; k += kFrontThreads) {
        int off = 0;                            // k >= 245: any finite element (its weight is zero)
        if (k < kK) {
            const int kt = k / (kKH * kKW), r = k - kt * kKH * kKW, kh = r / kKW, kw = r - kh * kKW;
            off = (kt * kHaloH + kh) * kHaloW + kw;
        }
        koff[k] = off;
    }
    for (int i = tid; i < 8 * kFrontC; i += kFrontThreads) wstat[i] = Stat{0.f, 0.f, 0.f};
    for (int row = warp; row < kTaps * kHaloH; row += kFrontThreads / 32) {     // one warp per halo row
        const int kt = row / kHaloH, hr = row - kt * kHaloH;
        const int tt = t + kt - 2, ih = ih0 + hr;
        const bool in = tt >= 0 && tt < T && ih >= 0 && ih < H;
        const float* src = x + ((size_t)(b * T + (in ? tt : 0)) * H + (in ? ih : 0)) * W;
        for (int wc = lane; wc < kHaloW; wc += 32) {
            const int iw = iw0 + wc;
            const float v = (in && iw >= 0 && iw < W) ? __ldg(src + iw) : 0.f;
            halo[row * kHaloW + wc] = __bfloat16_as_ushort(__float2bfloat16_rn(v));
        }
    }
    __syncthreads();

    const int r0 = lane >> 2, q = lane & 3;
    const int rows_valid = min(kTileH, Ho - oh0), cols_valid = min(kTileW, Wo - ow0);
    // 48 m16 tiles (16 rows x 3 column tiles), 6 per warp, two at a time
#pragma unroll 1
    for (int pair = 0; pair < 3; ++pair) {
        int base[2][2], cnt[2], prow[2], pcol[2];
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            const int id = warp * 6 + pair * 2 + j;
            prow[j] = id / 3;
            pcol[j] = (id - prow[j] * 3) * 16;
            base[j][0] = 2 * prow[j] * kHaloW + 2 * (pcol[j] + r0);
            base[j][1] = base[j][0] + 16;          // pixel + 8 -> 16 input columns further
            cnt[j] = prow[j] < rows_valid ? max(0, min(16, cols_valid - pcol[j])) : 0;
        }
        float acc[2][8][4];
#pragma unroll
        for (int j = 0; j < 2; ++j)
#pragma unroll
            for (int nt = 0; nt < 8; ++nt)
#pragma unroll
                for (int e = 0; e < 4; ++e) acc[j][nt][e] = 0.f;
        if (cnt[0] + cnt[1] > 0) {
#pragma unroll 2
            for (int ks = 0; ks < kKPad / 16; ++ks) {
                const int k0 = ks * 16 + 2 * q;
                const int o0 = koff[k0], o1 = koff[k0 + 1], o8 = koff[k0 + 8], o9 = koff[k0 + 9];
                uint32_t a[2][4];
#pragma unroll
                for (int j = 0; j < 2; ++j) {
                    a[j][0] = pack2(halo[base[j][0] + o0], halo[base[j][0] + o1]);
                    a[j][1] = pack2(halo[base[j][1] + o0], halo[base[j][1] + o1]);
                    a[j][2] = pack2(halo[base[j][0] + o8], halo[base[j][0] + o9]);
                    a[j][3] = pack2(halo[base[j][1] + o8], halo[base[j][1] + o9]);
                }
#pragma unroll
                for (int nt = 0; nt < 8; ++nt) {
                    const __nv_bfloat16* wr = w_s + (nt * 8 + r0) * kWStride + k0;
                    const uint32_t b0 = *reinterpret_cast<const uint32_t*>(wr);
                    const uint32_t b1 = *reinterpret_cast<const uint32_t*>(wr + 8);
                    mma_bf16_16816(acc[0][nt], a[0], b0, b1);
                    mma_bf16_16816(acc[1][nt], a[1], b0, b1);
                }
            }
        }
        // epilogue: bf16 store + statistics of the rounded values
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            if (cnt[j] == 0) continue;                          // warp-uniform
            const bool v0 = r0 < cnt[j], v1 = r0 + 8 < cnt[j];
            const int oh = oh0 + prow[j];
            const size_t row0 = ((size_t)n * Ho + oh) * Wo + ow0 + pcol[j] + r0;
            const float inv = 1.f / (float)cnt[j];
#pragma unroll
            for (int nt = 0; nt < 8; ++nt) {
                const int co = nt * 8 + 2 * q;
                const __nv_bfloat162 h0 = __floats2bfloat162_rn(acc[j][nt][0], acc[j][nt][1]);
                const __nv_bfloat162 h1 = __floats2bfloat162_rn(acc[j][nt][2], acc[j][nt][3]);
                if (v0) *reinterpret_cast<__nv_bfloat162*>(y + row0 * kFrontC + co) = h0;
                if (v1) *reinterpret_cast<__nv_bfloat162*>(y + (row0 + 8) * kFrontC + co) = h1;
                if (partials == nullptr) continue;
                const float2 f0 = __bfloat1622float2(h0), f1 = __bfloat1622float2(h1);
                float s0 = (v0 ? f0.x : 0.f) + (v1 ? f1.x : 0.f);
                float s1 = (v0 ? f0.y : 0.f) + (v1 ? f1.y : 0.f);
#pragma unroll
                for (int o = 4; o < 32; o <<= 1) {
                    s0 += __shfl_xor_sync(avctc::kFullMask, s0, o);
                    s1 += __shfl_xor_sync(avctc::kFullMask, s1, o);
                }
                const float m0 = s0 * inv, m1 = s1 * inv;
                float d0 = (v0 ? (f0.x - m0) * (f0.x - m0) : 0.f) + (v1 ? (f1.x - m0) * (f1.x - m0) : 0.f);
                float d1 = (v0 ? (f0.y - m1) * (f0.y - m1) : 0.f) + (v1 ? (f1.y - m1) * (f1.y - m1) : 0.f);
#pragma unroll
                for (int o = 4; o < 32; o <<= 1) {
                    d0 += __shfl_xor_sync(avctc::kFullMask, d0, o);
                    d1 += __shfl_xor_sync(avctc::kFullMask, d1, o);
                }
                if (r0 == 0) {
                    Stat* ws = wstat + warp * kFrontC + co;
                    ws[0] = chan_merge(ws[0], Stat{(float)cnt[j], m0, d0});
                    ws[1] = chan_merge(ws[1], Stat{(float)cnt[j], m1, d1});
                }
            }
        }
    }
    if (partials == nullptr) return;
    __syncthreads();
    if (tid < kFrontC) {
        Stat s = wstat[tid];
        for (int w = 1; w < kFrontThreads / 32; ++w) s = chan_merge(s, wstat[w * kFrontC + tid]);
        const int p = (blockIdx.z * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x;
        partials[(size_t)(0 * kFrontC + tid) * P + p] = s.n;
        partials[(size_t)(1 * kFrontC + tid) * P + p] = s.mean;
        partials[(size_t)(2 * kFrontC + tid) * P + p] = s.m2;
    }
}

// ---------------------------------------------------------------------------------------------------------------
// Statistics of a cuDNN convolution output x [M, C] bf16: CTA p covers rows [p*chunk, (p+1)*chunk); thread = one
// 8-channel group x every R-th row (Welford), the R row lanes merged in order through shared memory.
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kStatThreads)
vis_bn_stats_kernel(const __nv_bfloat16* __restrict__ x, long long M, int C, long long chunk,
                    float* __restrict__ partials, int P) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    Stat* st = reinterpret_cast<Stat*>(smem_raw);        // [R][C]
    const int G = C / 8, R = kStatThreads / G;
    const int tid = threadIdx.x, g = tid % G, r = tid / G;
    const long long lo = (long long)blockIdx.x * chunk, hi = min(M, lo + chunk);
    float mean[8], m2[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) mean[i] = m2[i] = 0.f;
    float cnt = 0.f;
    if (r < R) {
        for (long long row = lo + r; row < hi; row += R) {
            const uint4 u = __ldg(reinterpret_cast<const uint4*>(x + row * C) + g);
            float v[8];
            unpack8(u, v);
            cnt += 1.f;
            const float inv = 1.f / cnt;
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const float d = v[i] - mean[i];
                mean[i] += d * inv;
                m2[i] += d * (v[i] - mean[i]);
            }
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) st[r * C + g * 8 + i] = Stat{cnt, mean[i], m2[i]};
    }
    __syncthreads();
    for (int c = tid; c < C; c += kStatThreads) {
        Stat s = st[c];
        for (int k = 1; k < R; ++k) s = chan_merge(s, st[k * C + c]);
        partials[(size_t)(0 * C + c) * P + blockIdx.x] = s.n;
        partials[(size_t)(1 * C + c) * P + blockIdx.x] = s.mean;
        partials[(size_t)(2 * C + c) * P + blockIdx.x] = s.m2;
    }
}

// ---------------------------------------------------------------------------------------------------------------
// One CTA per channel.  training: merge the P partials (thread i takes i, i+256, ..., then a fixed tree), normalise
// with the biased variance, update the running statistics as ATen does (momentum, unbiased variance n/(n-1)).
// eval: scale / shift from the running statistics.  Writes scale_shift[c] = gamma/sqrt(var+eps),
// scale_shift[C+c] = beta - mean*scale.
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
vis_bn_finalize_kernel(const float* __restrict__ partials, int P, int C, const float* __restrict__ weight,
                       const float* __restrict__ bias, float* __restrict__ running_mean,
                       float* __restrict__ running_var, float momentum, float eps, int training,
                       float* __restrict__ scale_shift) {
    __shared__ Stat red[256];
    const int c = blockIdx.x, tid = threadIdx.x;
    float mean, var;
    if (training) {
        Stat s{0.f, 0.f, 0.f};
        const float* pn = partials + (size_t)(0 * C + c) * P;
        const float* pm = partials + (size_t)(1 * C + c) * P;
        const float* p2 = partials + (size_t)(2 * C + c) * P;
        for (int i = tid; i < P; i += 256) s = chan_merge(s, Stat{pn[i], pm[i], p2[i]});
        red[tid] = s;
        __syncthreads();
        for (int h = 128; h > 0; h >>= 1) {
            if (tid < h) red[tid] = chan_merge(red[tid], red[tid + h]);
            __syncthreads();
        }
        if (tid != 0) return;
        s = red[0];
        mean = s.mean;
        var = s.n > 0.f ? s.m2 / s.n : 0.f;
        const float unbiased = s.n > 1.f ? s.m2 / (s.n - 1.f) : var;
        running_mean[c] = momentum * mean + (1.f - momentum) * running_mean[c];
        running_var[c] = momentum * unbiased + (1.f - momentum) * running_var[c];
    } else {
        if (tid != 0) return;
        mean = running_mean[c];
        var = running_var[c];
    }
    const float invstd = 1.f / sqrtf(var + eps);
    const float sc = (weight ? weight[c] : 1.f) * invstd;
    scale_shift[c] = sc;
    scale_shift[C + c] = (bias ? bias[c] : 0.f) - mean * sc;
}

// ---------------------------------------------------------------------------------------------------------------
// Front-end BN apply + PReLU + 3x3/2 max pool (padding 1, -inf): out [N, Hp, Wp, 64] from y [N, H, W, 64].
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
vis_frontend_pool_kernel(const __nv_bfloat16* __restrict__ y, long long N, int H, int W, int Hp, int Wp,
                         const float* __restrict__ scale_shift, const __nv_bfloat16* __restrict__ slope,
                         __nv_bfloat16* __restrict__ out) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long total = N * Hp * Wp * (kFrontC / 8);
    if (i >= total) return;
    const int g = (int)(i % (kFrontC / 8));
    const long long pix = i / (kFrontC / 8);
    const int pw = (int)(pix % Wp), ph = (int)((pix / Wp) % Hp);
    const long long n = pix / ((long long)Wp * Hp);
    float sc[8], sh[8], sl[8], mx[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        sc[k] = scale_shift[g * 8 + k];
        sh[k] = scale_shift[kFrontC + g * 8 + k];
        sl[k] = __bfloat162float(slope[g * 8 + k]);
        mx[k] = AVCTC_NEG_INF;
    }
    for (int dh = -1; dh <= 1; ++dh) {
        const int h = 2 * ph + dh;
        if (h < 0 || h >= H) continue;
        for (int dw = -1; dw <= 1; ++dw) {
            const int w = 2 * pw + dw;
            if (w < 0 || w >= W) continue;
            const uint4 u = __ldg(reinterpret_cast<const uint4*>(y + ((n * H + h) * W + w) * kFrontC) + g);
            float v[8];
            unpack8(u, v);
#pragma unroll
            for (int k = 0; k < 8; ++k) mx[k] = fmaxf(mx[k], prelu_bf16(bf16r(fmaf(v[k], sc[k], sh[k])), sl[k]));
        }
    }
    reinterpret_cast<uint4*>(out + pix * kFrontC)[g] = pack8(mx);
}

// ---------------------------------------------------------------------------------------------------------------
// Trunk BN apply [+ residual] + PReLU over x [M, C]:  z = bf16(x*scale+shift); with a residual r (identity bf16, or
// the downsample conv's raw output with its own scale / shift -> bf16) z = bf16(z + r); out = bf16(PReLU(z)).
// pool_hw > 0: rows are frames of pool_hw pixels and out [M/pool_hw, C] = bf16(mean of the activated bf16 values).
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
vis_bn_act_kernel(const __nv_bfloat16* __restrict__ x, long long M, int C, const float* __restrict__ scale_shift,
                  const __nv_bfloat16* __restrict__ slope, const __nv_bfloat16* __restrict__ res,
                  const float* __restrict__ res_scale_shift, int pool_hw, __nv_bfloat16* __restrict__ out) {
    const int G = C / 8;
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long outer = pool_hw > 0 ? M / pool_hw : M;
    if (i >= outer * G) return;
    const int g = (int)(i % G);
    const long long o = i / G;
    float sc[8], sh[8], sl[8], rsc[8], rsh[8], acc[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        sc[k] = scale_shift[g * 8 + k];
        sh[k] = scale_shift[C + g * 8 + k];
        sl[k] = __bfloat162float(slope[g * 8 + k]);
        rsc[k] = res_scale_shift ? res_scale_shift[g * 8 + k] : 1.f;
        rsh[k] = res_scale_shift ? res_scale_shift[C + g * 8 + k] : 0.f;
        acc[k] = 0.f;
    }
    const int rows = pool_hw > 0 ? pool_hw : 1;
    const long long row0 = pool_hw > 0 ? o * pool_hw : o;
    for (int rr = 0; rr < rows; ++rr) {
        const long long off = (row0 + rr) * C;
        float v[8];
        unpack8(__ldg(reinterpret_cast<const uint4*>(x + off) + g), v);
#pragma unroll
        for (int k = 0; k < 8; ++k) v[k] = bf16r(fmaf(v[k], sc[k], sh[k]));
        if (res) {
            float r[8];
            unpack8(__ldg(reinterpret_cast<const uint4*>(res + off) + g), r);
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                if (res_scale_shift) r[k] = bf16r(fmaf(r[k], rsc[k], rsh[k]));
                v[k] = bf16r(v[k] + r[k]);
            }
        }
#pragma unroll
        for (int k = 0; k < 8; ++k) v[k] = prelu_bf16(v[k], sl[k]);
        if (pool_hw > 0) {
#pragma unroll
            for (int k = 0; k < 8; ++k) acc[k] += v[k];
        } else {
            reinterpret_cast<uint4*>(out + off)[g] = pack8(v);
        }
    }
    if (pool_hw > 0) {
#pragma unroll
        for (int k = 0; k < 8; ++k) acc[k] /= (float)pool_hw;
        reinterpret_cast<uint4*>(out + o * C)[g] = pack8(acc);
    }
}

// ------------------------------------------------------------------------------------------------ C ABI
static inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }
static inline bool channels_ok(int C) { return C >= 8 && C <= 2048 && C % 8 == 0 && kStatThreads % (C / 8) == 0; }

static size_t frontend_smem_bytes() {
    return (size_t)kFrontC * kWStride * 2 + (size_t)kTaps * kHaloH * kHaloW * 2 + kKPad * 4 +
           (size_t)(kFrontThreads / 32) * kFrontC * sizeof(Stat);
}

extern "C" {

AVCTC_API int avctc_visual_frontend_ctas(int B, int T, int H, int W) {
    if (B < 1 || T < 1 || H < 1 || W < 1) return 0;
    const long long Ho = (H - 1) / 2 + 1, Wo = (W - 1) / 2 + 1;
    const long long p = ((Wo + kTileW - 1) / kTileW) * ((Ho + kTileH - 1) / kTileH) * (long long)B * T;
    return p > (1LL << 30) ? 0 : (int)p;
}

AVCTC_API int avctc_visual_frontend(const float* x, int B, int T, int H, int W, const void* w_bf16, void* y_bf16,
                                    float* partials, int P, void* stream) {
    if (!x || !w_bf16 || !y_bf16) return AVCTC_ERR_BAD_ARG;
    const int p = avctc_visual_frontend_ctas(B, T, H, W);
    if (p == 0 || (long long)B * T > 65535) return AVCTC_ERR_UNSUPPORTED;
    if (partials && P != p) return AVCTC_ERR_WORKSPACE;
    if (!aligned16(w_bf16) || !aligned16(y_bf16)) return AVCTC_ERR_ALIGNMENT;
    const int Ho = (H - 1) / 2 + 1, Wo = (W - 1) / 2 + 1;
    static bool attr_set[64] = {};            // per device, set on the first (uncaptured) call
    int dev = 0;
    AVCTC_CUDA_RETURN(cudaGetDevice(&dev));
    const size_t smem = frontend_smem_bytes();
    if (dev >= 64 || !attr_set[dev]) {
        AVCTC_CUDA_RETURN(cudaFuncSetAttribute(vis_frontend_conv_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                               (int)smem));
        if (dev < 64) attr_set[dev] = true;
    }
    const dim3 grid((Wo + kTileW - 1) / kTileW, (Ho + kTileH - 1) / kTileH, B * T);
    vis_frontend_conv_kernel<<<grid, kFrontThreads, smem, (cudaStream_t)stream>>>(
        x, T, H, W, Ho, Wo, (const __nv_bfloat16*)w_bf16, (__nv_bfloat16*)y_bf16, partials, P);
    return (int)cudaGetLastError();
}

AVCTC_API int avctc_bn_stats_ctas(long long M, int C) {
    if (M < 1 || !channels_ok(C)) return 0;
    const int R = kStatThreads / (C / 8);
    const long long want = (M + 4LL * R - 1) / (4LL * R);        // at least 4 rows per thread
    return (int)(want < 4 * 148 ? want : 4 * 148);
}

AVCTC_API int avctc_bn_stats(const void* x_bf16, long long M, int C, float* partials, int P, void* stream) {
    if (!x_bf16 || !partials) return AVCTC_ERR_BAD_ARG;
    if (!channels_ok(C) || M < 1) return AVCTC_ERR_UNSUPPORTED;
    if (P != avctc_bn_stats_ctas(M, C)) return AVCTC_ERR_WORKSPACE;
    if (!aligned16(x_bf16)) return AVCTC_ERR_ALIGNMENT;
    const long long chunk = (M + P - 1) / P;
    const size_t smem = (size_t)kStatThreads / (C / 8) * C * sizeof(Stat);
    if (smem > 48 * 1024) return AVCTC_ERR_UNSUPPORTED;
    vis_bn_stats_kernel<<<P, kStatThreads, smem, (cudaStream_t)stream>>>((const __nv_bfloat16*)x_bf16, M, C, chunk,
                                                                         partials, P);
    return (int)cudaGetLastError();
}

AVCTC_API int avctc_bn_finalize(const float* partials, int P, int C, const float* weight, const float* bias,
                                float* running_mean, float* running_var, float momentum, float eps, int training,
                                float* scale_shift, void* stream) {
    if (!running_mean || !running_var || !scale_shift || (training && (!partials || P < 1))) return AVCTC_ERR_BAD_ARG;
    if (C < 1) return AVCTC_ERR_UNSUPPORTED;
    vis_bn_finalize_kernel<<<C, 256, 0, (cudaStream_t)stream>>>(partials, P, C, weight, bias, running_mean,
                                                                running_var, momentum, eps, training, scale_shift);
    return (int)cudaGetLastError();
}

AVCTC_API int avctc_visual_frontend_pool(const void* y_bf16, long long N, int H, int W, const float* scale_shift,
                                         const void* slope_bf16, void* out_bf16, void* stream) {
    if (!y_bf16 || !scale_shift || !slope_bf16 || !out_bf16) return AVCTC_ERR_BAD_ARG;
    if (N < 1 || H < 1 || W < 1) return AVCTC_ERR_UNSUPPORTED;
    if (!aligned16(y_bf16) || !aligned16(out_bf16)) return AVCTC_ERR_ALIGNMENT;
    const int Hp = (H - 1) / 2 + 1, Wp = (W - 1) / 2 + 1;
    const long long total = N * Hp * Wp * (kFrontC / 8);
    vis_frontend_pool_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        (const __nv_bfloat16*)y_bf16, N, H, W, Hp, Wp, scale_shift, (const __nv_bfloat16*)slope_bf16,
        (__nv_bfloat16*)out_bf16);
    return (int)cudaGetLastError();
}

AVCTC_API int avctc_bn_act(const void* x_bf16, long long M, int C, const float* scale_shift, const void* slope_bf16,
                           const void* res_bf16, const float* res_scale_shift, int pool_hw, void* out_bf16,
                           void* stream) {
    if (!x_bf16 || !scale_shift || !slope_bf16 || !out_bf16 || (res_scale_shift && !res_bf16)) return AVCTC_ERR_BAD_ARG;
    if (M < 1 || C < 8 || C % 8 != 0 || pool_hw < 0 || (pool_hw > 0 && M % pool_hw != 0)) return AVCTC_ERR_UNSUPPORTED;
    if (!aligned16(x_bf16) || !aligned16(out_bf16) || (res_bf16 && !aligned16(res_bf16))) return AVCTC_ERR_ALIGNMENT;
    const long long threads = (pool_hw > 0 ? M / pool_hw : M) * (C / 8);
    vis_bn_act_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        (const __nv_bfloat16*)x_bf16, M, C, scale_shift, (const __nv_bfloat16*)slope_bf16,
        (const __nv_bfloat16*)res_bf16, res_scale_shift, pool_hw, (__nv_bfloat16*)out_bf16);
    return (int)cudaGetLastError();
}

}  // extern "C"
