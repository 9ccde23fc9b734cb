// fusion_path.cu — CrossAttentionFusion forward / backward up to fusion_proj as ONE host call each.
//
// Replaces /root/reference/model/fusion_module.py:40-63 (speech-frame select + resample, visual_proj, audio_proj,
// nn.MultiheadAttention(query=audio, key=value=visual), fusion_proj) and its autograd.  Every step is one of this
// library's kernels; enqueuing them from C++ instead of one Python/ctypes round trip per kernel removes ~20 us of host
// time per launch (21.6 GFLOP forward is ~13 us of tensor work).  Round 2: GEMMs that do not depend on each other share
// a launch (grouped GEMM: the two input projections; q and k|v projections; each layer's dgrad + wgrad; ...), the
// attention core is one tcgen05 kernel per direction (attention.cu), the bf16 weight copies live in a buffer the module
// owns and are refreshed only when a parameter changed, TMA descriptors are memoised.  Forward: 7 launches (8 when the
// weights changed), backward: 7 (+1 when df is fp32, +1 for d_audio).  Weight gradients use split-K so that their
// 16-48 output tiles spread over the SMs their launch leaves free.
#include "common.cuh"
#include "gemm_internal.h"

int avctc_attention_supported(int T, int E, int H);
int avctc_attention_launch(int forward, const void* q, const void* kv, const void* dout, void* o, float* lse2, void* dq,
                           void* dkv, int B, int T, int H, int E, void* stream);

namespace avctc {

struct CastJob { const float* src; __nv_bfloat16* dst; long long n; };
struct CastJobs { CastJob j[8]; int count; };

// fp32 -> bf16 for up to 8 tensors in one launch: one flat index space over all tensors (4 elements per step)
__global__ void multi_cast_kernel(const CastJobs jobs) {
    long long total4 = 0;
    for (int t = 0; t < jobs.count; ++t) total4 += (jobs.j[t].n + 3) >> 2;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total4; i += (long long)gridDim.x * blockDim.x) {
        long long r = i;
        int t = 0;
        while (r >= ((jobs.j[t].n + 3) >> 2)) { r -= (jobs.j[t].n + 3) >> 2; ++t; }
        const CastJob jb = jobs.j[t];
        const long long e = r << 2;
        if (e + 4 <= jb.n && ((reinterpret_cast<uintptr_t>(jb.src) & 15) == 0) && ((reinterpret_cast<uintptr_t>(jb.dst) & 7) == 0)) {
            const float4 v = *reinterpret_cast<const float4*>(jb.src + e);
            __nv_bfloat162* d = reinterpret_cast<__nv_bfloat162*>(jb.dst + e);
            d[0] = __floats2bfloat162_rn(v.x, v.y);
            d[1] = __floats2bfloat162_rn(v.z, v.w);
        } else {
            for (long long k = e; k < jb.n && k < e + 4; ++k) jb.dst[k] = __float2bfloat16(jb.src[k]);
        }
    }
}

struct ColsumJob { const __nv_bfloat16* x; long long M; int N; long long ld; float* out; };
struct ColsumJobs { ColsumJob j[6]; int count; };
// bias gradients of every linear in one launch: out[n] += sum_m x[m][n] (outs zeroed by the caller); grid (N/32, row
// chunks, jobs), fp32 atomics across row chunks
__global__ void multi_colsum_kernel(const ColsumJobs jobs) {
    __shared__ float part[8][33];
    const ColsumJob jb = jobs.j[blockIdx.z];
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int n = blockIdx.x * 32 + tx;
    if (blockIdx.x * 32 >= jb.N) return;
    const long long per = (jb.M + gridDim.y - 1) / gridDim.y;
    const long long m0 = (long long)blockIdx.y * per, m1 = (m0 + per < jb.M) ? m0 + per : jb.M;
    float acc = 0.f;
    if (n < jb.N)
        for (long long m = m0 + ty; m < m1; m += 8) acc += __bfloat162float(jb.x[m * jb.ld + n]);
    part[ty][tx] = acc;
    __syncthreads();
    if (ty == 0 && n < jb.N) {
        float s = 0.f;
#pragma unroll
        for (int i = 0; i < 8; ++i) s += part[i][tx];
        atomicAdd(jb.out + n, s);
    }
}

struct FusionDims { int B, T, Ta, Dv, Da, E, H, hd, Tp; long long M, BH; };

static bool make_dims(int B, int T, int Ta, int Dv, int Da, int E, int H, FusionDims* d) {
    if (B <= 0 || T <= 0 || Ta <= 0 || Dv <= 0 || Da <= 0 || E <= 0 || H <= 0) return false;
    if (E % H) return false;
    d->B = B; d->T = T; d->Ta = Ta; d->Dv = Dv; d->Da = Da; d->E = E; d->H = H; d->hd = E / H;
    if (d->hd % 64 || Dv % 8 || Da % 8) return false;      // head slices are addressed as 64-wide K blocks
    d->Tp = (T + 7) / 8 * 8;
    d->M = (long long)B * T; d->BH = (long long)B * H;
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

struct Weights {    // bf16 copies of the five weight matrices: a persistent buffer owned by the module (refreshed by
    __nv_bfloat16 *w_vp, *w_ap, *w_in, *w_o, *w_f; size_t total;      // forward only when a parameter changed)
};
static Weights carve_weights(void* base, const FusionDims& d) {
    Carver c{reinterpret_cast<char*>(base), 0};
    Weights w;
    const size_t E = d.E;
    w.w_vp = c.take<__nv_bfloat16>(E * d.Dv); w.w_ap = c.take<__nv_bfloat16>(E * d.Da);
    w.w_in = c.take<__nv_bfloat16>(3 * E * E); w.w_o = c.take<__nv_bfloat16>(E * E); w.w_f = c.take<__nv_bfloat16>(E * E);
    w.total = c.off;
    return w;
}
struct Saved {      // written by forward, read by backward
    __nv_bfloat16 *xa, *v, *a, *q, *kv, *P, *o, *ao; float* lse2;
    void* rs_ws; size_t rs_bytes; size_t total;
};
static Saved carve_saved(void* base, const FusionDims& d) {
    Carver c{reinterpret_cast<char*>(base), 0};
    Saved s;
    const size_t E = d.E, M = d.M;
    const bool fused = avctc_attention_supported(d.T, d.E, d.H) != 0;
    s.xa = c.take<__nv_bfloat16>(M * d.Da);
    s.v = c.take<__nv_bfloat16>(M * E); s.a = c.take<__nv_bfloat16>(M * E); s.q = c.take<__nv_bfloat16>(M * E);
    s.kv = c.take<__nv_bfloat16>(M * 2 * E);
    s.P = fused ? nullptr : c.take<__nv_bfloat16>((size_t)d.BH * d.T * d.Tp);     // unfused attention route only
    s.lse2 = c.take<float>((size_t)d.BH * d.T);
    s.o = c.take<__nv_bfloat16>(M * E); s.ao = c.take<__nv_bfloat16>(M * E);
    s.rs_bytes = avctc_resample_workspace_bytes(d.B, d.Ta);
    s.rs_ws = c.take<char>(s.rs_bytes);
    s.total = c.off;
    return s;
}
struct Scratch {    // S (forward, unfused attention) and every backward intermediate
    float* S; __nv_bfloat16 *dfb, *dao, *dout, *dS, *dq, *dkv, *da, *dv, *dxa; size_t total;
};
static Scratch carve_scratch(void* base, const FusionDims& d, bool backward) {
    Carver c{reinterpret_cast<char*>(base), 0};
    Scratch s{};
    const size_t E = d.E, M = d.M;
    const bool fused = avctc_attention_supported(d.T, d.E, d.H) != 0;
    s.S = fused ? c.take<float>(64) : c.take<float>((size_t)d.BH * d.T * d.Tp);           // forward: scores; backward: dP
    if (backward) {
        s.dfb = c.take<__nv_bfloat16>(M * E); s.dao = c.take<__nv_bfloat16>(M * E); s.dout = c.take<__nv_bfloat16>(M * E);
        s.dS = fused ? nullptr : c.take<__nv_bfloat16>((size_t)d.BH * d.T * d.Tp);
        s.dq = c.take<__nv_bfloat16>(M * E); s.dkv = c.take<__nv_bfloat16>(M * 2 * E);
        s.da = c.take<__nv_bfloat16>(M * E); s.dv = c.take<__nv_bfloat16>(M * E);
        s.dxa = c.take<__nv_bfloat16>(M * d.Da);
    }
    s.total = c.off;
    return s;
}


}  // namespace avctc

using namespace avctc;

extern "C" size_t avctc_fusion_workspace_bytes(int B, int T, int Ta, int Dv, int Da, int E, int H, int which) {
    FusionDims d;
    if (!make_dims(B, T, Ta, Dv, Da, E, H, &d)) return 0;
    if (which == 0) return carve_saved(nullptr, d).total;
    if (which == 3) return carve_weights(nullptr, d).total;
    return carve_scratch(nullptr, d, which == 2).total;
}

extern "C" int avctc_fusion_forward(const void* visual_bf16, const void* audio, int audio_dtype, const int64_t* mask,
                                    const float* w_vp, const float* b_vp, const float* w_ap, const float* b_ap,
                                    const float* w_in, const float* b_in, const float* w_o, const float* b_o,
                                    const float* w_f, const float* b_f, int B, int T, int Ta, int Dv, int Da, int E, int H,
                                    void* out, int out_dtype, int64_t* mask_out, int64_t* input_lengths,
                                    void* wbf16, size_t wbf16_bytes, int refresh_weights, void* saved, size_t saved_bytes,
                                    void* scratch, size_t scratch_bytes, void* stream) {
    FusionDims d;
    if (!make_dims(B, T, Ta, Dv, Da, E, H, &d)) return AVCTC_ERR_UNSUPPORTED;
    if (!visual_bf16 || !audio || !mask || !w_vp || !b_vp || !w_ap || !b_ap || !w_in || !b_in || !w_o || !b_o || !w_f ||
        !b_f || !out || !mask_out || !input_lengths || !saved || !scratch || !wbf16)
        return AVCTC_ERR_BAD_ARG;
    if (out_dtype != AVCTC_F32 && out_dtype != AVCTC_BF16) return AVCTC_ERR_BAD_ARG;
    if ((reinterpret_cast<uintptr_t>(saved) | reinterpret_cast<uintptr_t>(scratch) | reinterpret_cast<uintptr_t>(wbf16)) & 255)
        return AVCTC_ERR_ALIGNMENT;
    Saved s = carve_saved(saved, d);
    Scratch w = carve_scratch(scratch, d, false);
    Weights wt = carve_weights(wbf16, d);
    if (saved_bytes < s.total || scratch_bytes < w.total || wbf16_bytes < wt.total) return AVCTC_ERR_WORKSPACE;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    const long long M = d.M;
    const int Eh = d.E, hd = d.hd, Tp = d.Tp;
    if (refresh_weights) {
        CastJobs cj;
        cj.count = 5;
        cj.j[0] = {w_vp, wt.w_vp, (long long)Eh * Dv}; cj.j[1] = {w_ap, wt.w_ap, (long long)Eh * Da};
        cj.j[2] = {w_in, wt.w_in, 3ll * Eh * Eh}; cj.j[3] = {w_o, wt.w_o, (long long)Eh * Eh}; cj.j[4] = {w_f, wt.w_f, (long long)Eh * Eh};
        multi_cast_kernel<<<592, 256, 0, st>>>(cj);
        AVCTC_CUDA_RETURN(cudaGetLastError());
    }
    AVCTC_TRY(avctc_resample_forward(audio, audio_dtype, mask, B, Ta, Da, T, s.xa, mask_out, input_lengths, s.rs_ws,
                                     s.rs_bytes, stream));
    const __nv_bfloat16* xv = reinterpret_cast<const __nv_bfloat16*>(visual_bf16);
    {   // visual_proj and audio_proj share a launch; so do the query and the key|value projections
        AvctcGemmJob g1[2] = {linear_job(xv, Dv, wt.w_vp, b_vp, M, Eh, Dv, s.v, AVCTC_BF16, Eh),
                              linear_job(s.xa, Da, wt.w_ap, b_ap, M, Eh, Da, s.a, AVCTC_BF16, Eh)};
        AVCTC_TRY(avctc_gemm_launch_group(g1, 2, stream));
        AvctcGemmJob g2[2] = {linear_job(s.a, Eh, wt.w_in, b_in, M, Eh, Eh, s.q, AVCTC_BF16, Eh),
                              linear_job(s.v, Eh, wt.w_in + (size_t)Eh * Eh, b_in + Eh, M, 2 * Eh, Eh, s.kv, AVCTC_BF16, 2 * Eh)};
        AVCTC_TRY(avctc_gemm_launch_group(g2, 2, stream));
    }
    if (avctc_attention_supported(T, Eh, H)) {
        AVCTC_TRY(avctc_attention_launch(1, s.q, s.kv, nullptr, s.o, s.lse2, nullptr, nullptr, B, T, H, Eh, stream));
    } else {
        const float alpha = 1.f / sqrtf((float)hd);
        {   // S[b,h] = alpha * q_h . k_h^T
            avctc_gemm_operand A = opnd(s.q, M, Eh, Eh), Bo = opnd(s.kv, M, 2 * Eh, 2 * Eh);
            A.k_inner = hd; A.r_outer = T; Bo.k_inner = hd; Bo.r_outer = T;
            AVCTC_TRY(avctc_gemm_launch(&A, &Bo, T, T, hd, (int)d.BH, H, w.S, AVCTC_F32, Tp, (long long)H * T * Tp,
                                        (long long)T * Tp, nullptr, 0, alpha, 0, 1, stream));
        }
        AVCTC_TRY(avctc_softmax_forward(w.S, s.P, d.BH * T, T, Tp, stream));
        {   // o[b,:,h] = P[b,h] . v_h
            avctc_gemm_operand A = opnd(s.P, T, T, Tp, false, d.BH, (long long)T * Tp);
            A.z_outer = H; A.z_inner = 1;
            avctc_gemm_operand Bo = opnd(s.kv + Eh, 2 * Eh - Eh, M, 2 * Eh, true);    // values: columns [E,2E) of kv
            Bo.rows = Eh; Bo.k_outer = T; Bo.r_inner = hd;
            AVCTC_TRY(avctc_gemm_launch(&A, &Bo, T, hd, T, (int)d.BH, H, s.o, AVCTC_BF16, Eh, (long long)T * Eh, hd, nullptr, 0,
                                        1.f, 0, 1, stream));
        }
    }
    {
        AvctcGemmJob j = linear_job(s.o, Eh, wt.w_o, b_o, M, Eh, Eh, s.ao, AVCTC_BF16, Eh);
        AVCTC_TRY(avctc_gemm_launch_group(&j, 1, stream));
        j = linear_job(s.ao, Eh, wt.w_f, b_f, M, Eh, Eh, out, out_dtype, Eh);
        AVCTC_TRY(avctc_gemm_launch_group(&j, 1, stream));
    }
    return AVCTC_OK;
}

extern "C" int avctc_fusion_backward(const void* df, int df_dtype, const void* visual_bf16, int B, int T, int Ta, int Dv,
                                     int Da, int E, int H, float* g_wvp, float* g_bvp, float* g_wap, float* g_bap,
                                     float* g_win, float* g_bin, float* g_wo, float* g_bo, float* g_wf, float* g_bf,
                                     void* d_visual_bf16, void* d_audio, int d_audio_dtype, const void* wbf16,
                                     size_t wbf16_bytes, const void* saved, size_t saved_bytes, void* scratch,
                                     size_t scratch_bytes, int grads_zeroed, void* stream) {
    FusionDims d;
    if (!make_dims(B, T, Ta, Dv, Da, E, H, &d)) return AVCTC_ERR_UNSUPPORTED;
    if (!df || !visual_bf16 || !g_wvp || !g_bvp || !g_wap || !g_bap || !g_win || !g_bin || !g_wo || !g_bo || !g_wf || !g_bf ||
        !saved || !scratch || !wbf16)
        return AVCTC_ERR_BAD_ARG;
    if (df_dtype != AVCTC_F32 && df_dtype != AVCTC_BF16) return AVCTC_ERR_BAD_ARG;
    Saved s = carve_saved(const_cast<void*>(saved), d);
    Scratch w = carve_scratch(scratch, d, true);
    Weights wt = carve_weights(const_cast<void*>(wbf16), d);
    if (saved_bytes < s.total || scratch_bytes < w.total || wbf16_bytes < wt.total) return AVCTC_ERR_WORKSPACE;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    const long long M = d.M;
    const int Eh = d.E, hd = d.hd, Tp = d.Tp;
    const float alpha = 1.f / sqrtf((float)hd);
    const __nv_bfloat16* dfb = reinterpret_cast<const __nv_bfloat16*>(df);
    if (df_dtype == AVCTC_F32) {
        CastJobs cj;
        cj.count = 1;
        cj.j[0] = {reinterpret_cast<const float*>(df), w.dfb, M * Eh};
        multi_cast_kernel<<<148, 256, 0, st>>>(cj);
        AVCTC_CUDA_RETURN(cudaGetLastError());
        dfb = w.dfb;
    }
    const __nv_bfloat16* xv = reinterpret_cast<const __nv_bfloat16*>(visual_bf16);
    const bool pz = grads_zeroed != 0;     // all ten gradient tensors are views of one buffer the caller zeroed once
    const int t512 = tiles_of(M, Eh);
    {   // fusion_proj: weight gradient and input gradient depend on df only -> one launch
        AvctcGemmJob g[2] = {dgrad_job(dfb, Eh, wt.w_f, M, Eh, Eh, w.dao),
                             wgrad_job(dfb, Eh, s.ao, Eh, M, Eh, Eh, g_wf, Eh, pz, t512)};
        AVCTC_TRY(avctc_gemm_launch_group(g, 2, stream));
    }
    {   // out_proj
        AvctcGemmJob g[2] = {dgrad_job(w.dao, Eh, wt.w_o, M, Eh, Eh, w.dout),
                             wgrad_job(w.dao, Eh, s.o, Eh, M, Eh, Eh, g_wo, Eh, pz, t512)};
        AVCTC_TRY(avctc_gemm_launch_group(g, 2, stream));
    }
    if (avctc_attention_supported(T, Eh, H)) {
        AVCTC_TRY(avctc_attention_launch(0, s.q, s.kv, w.dout, s.o, s.lse2, w.dq, w.dkv, B, T, H, Eh, stream));
    } else {
        // attention core: dP = do_h . v_h^T ; dS = P * (dP - sum(dP*P)) ; dq = alpha dS.k ; dk = alpha dS^T.q ; dv = P^T.do
        const __nv_bfloat16* kk = s.kv;
        const __nv_bfloat16* vv = s.kv + Eh;
        {
            avctc_gemm_operand A = opnd(w.dout, M, Eh, Eh), Bo = opnd(vv, M, Eh, 2 * Eh);
            A.k_inner = hd; A.r_outer = T; Bo.k_inner = hd; Bo.r_outer = T;
            AVCTC_TRY(avctc_gemm_launch(&A, &Bo, T, T, hd, (int)d.BH, H, w.S, AVCTC_F32, Tp, (long long)H * T * Tp,
                                        (long long)T * Tp, nullptr, 0, 1.f, 0, 1, stream));
        }
        AVCTC_TRY(avctc_softmax_backward(s.P, w.S, w.dS, d.BH * T, T, Tp, stream));
        {
            avctc_gemm_operand A = opnd(w.dS, T, T, Tp, false, d.BH, (long long)T * Tp);
            A.z_outer = H; A.z_inner = 1;
            avctc_gemm_operand Bo = opnd(kk, Eh, M, 2 * Eh, true);
            Bo.k_outer = T; Bo.r_inner = hd;
            AVCTC_TRY(avctc_gemm_launch(&A, &Bo, T, hd, T, (int)d.BH, H, w.dq, AVCTC_BF16, Eh, (long long)T * Eh, hd, nullptr, 0,
                                        alpha, 0, 1, stream));
        }
        {
            avctc_gemm_operand A = opnd(w.dS, T, T, Tp, true, d.BH, (long long)T * Tp);
            A.z_outer = H; A.z_inner = 1;
            avctc_gemm_operand Bo = opnd(s.q, Eh, M, Eh, true);
            Bo.k_outer = T; Bo.r_inner = hd;
            AVCTC_TRY(avctc_gemm_launch(&A, &Bo, T, hd, T, (int)d.BH, H, w.dkv, AVCTC_BF16, 2 * Eh, (long long)T * 2 * Eh, hd,
                                        nullptr, 0, alpha, 0, 1, stream));
        }
        {
            avctc_gemm_operand A = opnd(s.P, T, T, Tp, true, d.BH, (long long)T * Tp);
            A.z_outer = H; A.z_inner = 1;
            avctc_gemm_operand Bo = opnd(w.dout, Eh, M, Eh, true);
            Bo.k_outer = T; Bo.r_inner = hd;
            AVCTC_TRY(avctc_gemm_launch(&A, &Bo, T, hd, T, (int)d.BH, H, w.dkv + Eh, AVCTC_BF16, 2 * Eh, (long long)T * 2 * Eh, hd,
                                        nullptr, 0, 1.f, 0, 1, stream));
        }
    }
    {   // in_proj (rows [0,E) = query projection of a; rows [E,3E) = key|value projections of v): 4 GEMMs, one launch
        const int dg = 2 * t512;
        AvctcGemmJob g[4] = {dgrad_job(w.dq, Eh, wt.w_in, M, Eh, Eh, w.da),
                             dgrad_job(w.dkv, 2 * Eh, wt.w_in + (size_t)Eh * Eh, M, 2 * Eh, Eh, w.dv),
                             wgrad_job(w.dq, Eh, s.a, Eh, M, Eh, Eh, g_win, Eh, pz, dg + 64),
                             wgrad_job(w.dkv, 2 * Eh, s.v, Eh, M, 2 * Eh, Eh, g_win + (size_t)Eh * Eh, Eh, pz, dg + 64)};
        AVCTC_TRY(avctc_gemm_launch_group(g, 4, stream));
    }
    {   // audio_proj / visual_proj: weight gradients + (when the inputs need them) input gradients, one launch
        AvctcGemmJob g[4];
        int n = 0, dg = 0;
        if (d_visual_bf16) { g[n++] = dgrad_job(w.dv, Eh, wt.w_vp, M, Eh, Dv, reinterpret_cast<__nv_bfloat16*>(d_visual_bf16)); dg += tiles_of(M, Dv); }
        if (d_audio) { g[n++] = dgrad_job(w.da, Eh, wt.w_ap, M, Eh, Da, w.dxa); dg += tiles_of(M, Da); }
        g[n++] = wgrad_job(w.da, Eh, s.xa, Da, M, Eh, Da, g_wap, Da, pz, dg + 32);
        g[n++] = wgrad_job(w.dv, Eh, xv, Dv, M, Eh, Dv, g_wvp, Dv, pz, dg + 64);
        AVCTC_TRY(avctc_gemm_launch_group(g, n, stream));
    }
    {   // the six bias gradients (column sums of the six dY tensors) in one launch
        if (!pz) {
            AVCTC_CUDA_RETURN(cudaMemsetAsync(g_bf, 0, sizeof(float) * Eh, st));
            AVCTC_CUDA_RETURN(cudaMemsetAsync(g_bo, 0, sizeof(float) * Eh, st));
            AVCTC_CUDA_RETURN(cudaMemsetAsync(g_bin, 0, sizeof(float) * 3 * Eh, st));
            AVCTC_CUDA_RETURN(cudaMemsetAsync(g_bap, 0, sizeof(float) * Eh, st));
            AVCTC_CUDA_RETURN(cudaMemsetAsync(g_bvp, 0, sizeof(float) * Eh, st));
        }
        ColsumJobs cj;
        cj.count = 6;
        cj.j[0] = {dfb, M, Eh, Eh, g_bf};
        cj.j[1] = {w.dao, M, Eh, Eh, g_bo};
        cj.j[2] = {w.dq, M, Eh, Eh, g_bin};
        cj.j[3] = {w.dkv, M, 2 * Eh, 2 * Eh, g_bin + Eh};
        cj.j[4] = {w.da, M, Eh, Eh, g_bap};
        cj.j[5] = {w.dv, M, Eh, Eh, g_bvp};
        int chunks = (int)((M + 127) / 128);
        if (chunks > 32) chunks = 32;
        multi_colsum_kernel<<<dim3((2 * Eh + 31) / 32, chunks, 6), 256, 0, st>>>(cj);
        AVCTC_CUDA_RETURN(cudaGetLastError());
    }
    if (d_audio)
        AVCTC_TRY(avctc_resample_backward(w.dxa, B, Ta, Da, T, s.rs_ws, d_audio, d_audio_dtype, stream));
    return AVCTC_OK;
}
