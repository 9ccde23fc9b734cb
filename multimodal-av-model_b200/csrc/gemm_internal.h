// gemm_internal.h — library-internal launch interface of the tcgen05 GEMM (gemm_tcgen05.cu), shared with the host
// orchestration of the fusion path (fusion_path.cu).  Not part of the public C ABI.
#pragma once
#include <cuda_bf16.h>

#include "../../include/avctc_b200.h"

struct AvctcGemmJob {
    avctc_gemm_operand a, b;
    int M, N, K, batch, inner_count;
    void* C; int out_dtype; long long ldc, c_outer, c_inner;
    const float* bias; int bias_mode;
    float alpha; int accumulate;
    int splits;        // > 1: split-K with fp32 red.add into a C this call zeroes; < -1: the caller zeroed C already
};

// One launch for up to 6 independent GEMMs (see GemmGroup in gemm_tcgen05.cu).
int avctc_gemm_launch_group(const AvctcGemmJob* jobs, int njobs, void* stream);

int avctc_gemm_launch(const avctc_gemm_operand* a, const avctc_gemm_operand* b, int M, int N, int K, int batch,
                      int inner_count, void* C, int out_dtype, long long ldc, long long c_outer, long long c_inner,
                      const float* bias, int bias_mode, float alpha, int accumulate, int splits, void* stream);

// 3-D bf16 TMA descriptor (dim0 contiguous; dim1 stride ld elements; dim2 stride zstride elements), 128-byte swizzle,
// memoised by (pointer, extents, strides, box): encoding costs ~1 us of host time per map and the fusion path needs ~40
// per step on pointers the caching allocator hands back every step.
#include <cuda.h>
int avctc_tensor_map(CUtensorMap* out, const void* ptr, long long dim0, long long dim1, long long dim2, long long ld,
                     long long zstride, int box0, int box1);

// Job builders shared by the host orchestrations (fusion_path.cu, wav2vec2_layer.cu).
namespace avctc {
inline avctc_gemm_operand opnd(const void* ptr, long long rows, long long kdim, long long ld, bool mn = false,
                               long long zdim = 1, long long zstride = 0) {
    avctc_gemm_operand o;
    o.ptr = ptr; o.rows = rows; o.kdim = kdim; o.zdim = zdim; o.ld = ld; o.zstride = zstride;
    o.k_outer = o.k_inner = o.r_outer = o.r_inner = o.z_outer = o.z_inner = 0;
    o.mn_major = mn ? 1 : 0;
    return o;
}

#define AVCTC_TRY(expr) do { const int rc_ = (expr); if (rc_) return rc_; } while (0)

inline AvctcGemmJob job(const avctc_gemm_operand& A, const avctc_gemm_operand& Bo, int M, int N, int K, void* C, int dtype,
                        long long ldc, const float* bias = nullptr, int splits = 1) {
    AvctcGemmJob j;
    j.a = A; j.b = Bo; j.M = M; j.N = N; j.K = K; j.batch = 1; j.inner_count = 1;
    j.C = C; j.out_dtype = dtype; j.ldc = ldc; j.c_outer = 0; j.c_inner = 0;
    j.bias = bias; j.bias_mode = bias ? 1 : 0; j.alpha = 1.f; j.accumulate = 0; j.splits = splits;
    return j;
}
// y[M,N] = x[M,K] . w[N,K]^T + b
inline AvctcGemmJob linear_job(const __nv_bfloat16* x, long long ldx, const __nv_bfloat16* w, const float* b, long long M,
                               int N, int K, void* y, int ydtype, long long ldy) {
    return job(opnd(x, M, K, ldx), opnd(w, N, K, K), (int)M, N, K, y, ydtype, ldy, b);
}
// dx[M,K] = dy[M,N] . w[N,K]
inline AvctcGemmJob dgrad_job(const __nv_bfloat16* dy, long long ldy, const __nv_bfloat16* w, long long M, int N, int K,
                              __nv_bfloat16* dx) {
    return job(opnd(dy, M, N, ldy), opnd(w, K, N, K, true), (int)M, K, N, dx, AVCTC_BF16, K);
}
// g[N,K] (fp32) = dy[M,N]^T . x[M,K], split-K over M with red.add into g (zeroed here unless the caller did)
inline AvctcGemmJob wgrad_job(const __nv_bfloat16* dy, long long ldy, const __nv_bfloat16* x, long long ldx, long long M,
                              int N, int K, float* g, long long ldg, bool prezeroed, int other_ctas) {
    const int tiles = ((N + 127) / 128) * ((K + 127) / 128);
    // the launch should put ~2 CTAs on every SM together with its other jobs; 16-byte vector red.add epilogue
    int splits = (296 - other_ctas + tiles - 1) / tiles;
    if (splits < 1) splits = 1;
    if (splits > 8) splits = 8;
    return job(opnd(dy, N, M, ldy, true), opnd(x, K, M, ldx, true), N, K, (int)M, g, AVCTC_F32, ldg, nullptr,
               prezeroed ? -splits : splits);
}
inline int tiles_of(long long M, int N) { return (int)((M + 127) / 128) * ((N + 127) / 128); }
}  // namespace avctc
