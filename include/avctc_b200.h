/*
 * avctc_b200.h — C ABI of libavctc_b200.so: the B200 (sm_100a) implementation of the AV-CTC hot path
 * of limeorange1102/multimodal-av-model.
 *
 * The reference has no FFI/operator interface of its own (it is pure Python over PyTorch, SURVEY.md
 * §8b); each entry point below replaces the PyTorch op (or Python loop) the reference reaches at the
 * cited call site.  Conventions (SURVEY.md §8b "C-ABI underneath"):
 *   - plain pointers + sizes only, no torch types; every pointer is DEVICE memory unless it says host
 *   - the caller owns every buffer (inputs, outputs, workspace); the library never allocates device
 *     memory, never frees, never retains pointers, and never synchronises the host
 *   - all work is enqueued on `stream` (a cudaStream_t passed as void*)
 *   - return 0 on success, a negative avctc_status on bad arguments, or a positive cudaError_t passed
 *     through; nothing throws across the boundary (the Python host raises RuntimeError)
 *   - dtype enums: AVCTC_F32 = 0, AVCTC_BF16 = 1
 */
#ifndef AVCTC_B200_H_
#define AVCTC_B200_H_

#include <stddef.h>
#include <stdint.h>

#if defined(__GNUC__)
#define AVCTC_API __attribute__((visibility("default")))
#else
#define AVCTC_API
#endif

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
    AVCTC_OK = 0,
    AVCTC_ERR_BAD_ARG = -1,       /* null pointer, negative size, bad enum */
    AVCTC_ERR_UNSUPPORTED = -2,   /* shape outside what the kernels are built for */
    AVCTC_ERR_WORKSPACE = -3,     /* workspace_bytes too small */
    AVCTC_ERR_ALIGNMENT = -4      /* pointer/stride alignment requirement violated */
} avctc_status;

enum { AVCTC_F32 = 0, AVCTC_BF16 = 1 };
enum { AVCTC_REDUCE_NONE = 0, AVCTC_REDUCE_MEAN = 1, AVCTC_REDUCE_SUM = 2 };

/* Library identification / build check. Returns e.g. "avctc_b200 0.1 sm_100a". Host pointer. */
AVCTC_API const char* avctc_version(void);
/* Human-readable text for a status returned by any entry point (host pointer, static storage). */
AVCTC_API const char* avctc_status_string(int status);
/* Tuning knobs for benchmarking and A/B measurements (host-side process-global ints; no knob changes a result).
 * key: "ctc_lin" (1 = probability-domain CTC scan when 2L+1 <= 512, 0 = log-domain scan),
 * "ctc_ws" (1 = warp-specialised TMA-fed scan, 0 = single-warp scan), "ctc_k" (log-domain scan, states per lane:
 * 0 = auto, 2/4/8/16), "ctc_pf" (gradient pass: L2 prefetch distance in rows, 0 = off, +4 = also alpha/beta),
 * "ctc_overlap" (1 = a gradient pass launched right behind the scan starts on each sample as soon as that sample's
 * alpha/beta rows are complete, 0 = it waits for the whole scan grid), "ctc_stage" (1 = the fp32 gradient pass stages each log-prob row in
 * shared memory with cp.async, 0 = register streaming), "ctc_stamp" (1 = the CTC kernels leave
 * globaltimer stamps in the workspace's flag block: debug / tests), "ctc_grad_warps", "beam_fast" (1 = threshold top-k fast path), "beam_two_phase" (1 = top-k for all rows first),
 * "beam_pf" (1 = L2 prefetch of the next row), "beam_fused" (-1 = auto: one fused top-k + recurrence kernel for short utterances
 * up to 16 x SMs of them per call, 0 = never, 1 = whenever the shape is eligible), "beam_fused_grid" (cap on its CTAs: tests), "pdl" (1 = programmatic dependent launch for the GEMM / softmax / CTC
 * kernel chains), "lstm_tag" (BiLSTM step exchange: 0 counter barrier, 1 sentinel polling in the forward pass when
 * B <= 8, 2 forward always, 3 forward and backward), "lstm_groups" (batch groups of the BiLSTM kernels: 0 auto, n = n
 * groups), "gemm_dbg" (per-CTA timestamps).  Unknown keys return
 * AVCTC_ERR_BAD_ARG. */
AVCTC_API int avctc_set_tuning(const char* key, int value);

/* ------------------------------------------------------------------------------------------------
 * CTC loss — replaces nn.CTCLoss(blank, zero_infinity=True) = ATen _ctc_loss/_ctc_loss_backward
 *   constructed /root/reference/model/trainer.py:25 (also model/decoder.py:12)
 *   called      /root/reference/model/trainer.py:116-117, 224-225; model/decoder.py:28-33
 * log_probs is the [T,B,V] VIEW the reference passes (a transpose of [B,T,V]): element (t,b,c) at
 * log_probs[t*stride_t + b*stride_b + c] (strides in elements, class stride must be 1).
 * targets: int64, sample b's labels start at targets[b*target_stride] (2-D padded) or at
 * targets[target_offsets[b]] when target_offsets != NULL (1-D concatenated).  Lengths are int64 DEVICE
 * tensors and are read on the device (no host sync; values are clamped to [0,T] / [0,max_target_len]).
 * ---------------------------------------------------------------------------------------------- */
AVCTC_API size_t avctc_ctc_workspace_bytes(int T, int B, int max_target_len);

/* alpha (and, when need_grad != 0, beta) lattice scan.  Writes nll[b] (fp32, +inf when infeasible)
 * and fills `workspace` for avctc_ctc_backward. */
AVCTC_API int avctc_ctc_forward(const void* log_probs, int dtype, int64_t stride_t, int64_t stride_b,
                      int T, int B, int V,
                      const int64_t* targets, int64_t target_stride, const int64_t* target_offsets,
                      const int64_t* input_lengths, const int64_t* target_lengths,
                      int max_target_len, int blank, int need_grad,
                      float* nll, void* workspace, size_t workspace_bytes, void* stream);

/* loss[0] = reduction over nll (mean: mean_b(nll_b / max(L_b,1)); sum), with inf -> 0 first when
 * zero_infinity.  For AVCTC_REDUCE_NONE writes loss[b] (B floats). */
AVCTC_API int avctc_ctc_reduce(const float* nll, const int64_t* target_lengths, int B, int reduction,
                     int zero_infinity, float* loss, void* stream);

/* grad[T,B,V] (contiguous, dtype = log_probs dtype) = d loss / d log_probs in ATen's softmax-folded
 * convention: (exp(lp) - posterior) * g_b for t < input_length, 0 elsewhere and 0 for infeasible
 * samples when zero_infinity.  g_b = grad_out[b*grad_out_stride] * (mean: 1/(B*max(L_b,1)); else 1);
 * grad_out is a DEVICE fp32 scalar (stride 0) or [B] vector.
 * `workspace` is the one avctc_ctc_forward(need_grad=1) filled, untouched in between, on the same stream (or ordered
 * behind it); it is declared const because alpha/beta are only read, but the kernel does update a few control words in
 * its last block and leaves them as it found them.  The call may be enqueued directly behind avctc_ctc_forward
 * (avctc_ctc_reduce in between is fine): the gradient of each utterance then starts as soon as that utterance's
 * lattice rows are complete, under the scans of the longer ones; grad_out must in that case have been written
 * before avctc_ctc_forward was enqueued (anything else on the stream between the two calls orders them fully). */
AVCTC_API int avctc_ctc_backward(const void* log_probs, int dtype, int64_t stride_t, int64_t stride_b,
                       int T, int B, int V,
                       const int64_t* targets, int64_t target_stride, const int64_t* target_offsets,
                       const int64_t* input_lengths, const int64_t* target_lengths,
                       int max_target_len, int blank, int reduction, int zero_infinity,
                       const float* nll, const float* grad_out, int64_t grad_out_stride,
                       void* grad, const void* workspace, size_t workspace_bytes, void* stream);

/* avctc_ctc_forward(need_grad=1) + avctc_ctc_reduce + avctc_ctc_backward enqueued back to back by one call (same
 * arguments, same results): the form in which the gradient pass overlaps the scan. */
AVCTC_API int avctc_ctc_forward_backward(const void* log_probs, int dtype, int64_t stride_t, int64_t stride_b,
                               int T, int B, int V,
                               const int64_t* targets, int64_t target_stride, const int64_t* target_offsets,
                               const int64_t* input_lengths, const int64_t* target_lengths,
                               int max_target_len, int blank, int reduction, int zero_infinity,
                               float* nll, float* loss, const float* grad_out, int64_t grad_out_stride,
                               void* grad, void* workspace, size_t workspace_bytes, void* stream);

/* grad[t][b][:] *= grad_out[b*grad_out_stride], in place (rows whose factor is exactly 1 are left alone).  The autograd
 * host uses it to run the gradient pass at forward time: avctc_ctc_backward with a unit grad_out goes out directly behind
 * avctc_ctc_forward (so it overlaps the scan, see above) and loss.backward() only applies the incoming factor — the
 * chain rule step of torch's CtcLossBackward (/root/reference/model/trainer.py:121 `scaler.scale(loss_total).backward()`). */
AVCTC_API int avctc_ctc_scale_grad(void* grad, int dtype, int T, int B, int V, const float* grad_out,
                         int64_t grad_out_stride, void* stream);

/* ------------------------------------------------------------------------------------------------
 * CTC forced alignment — torchaudio.functional.forced_align (Viterbi over the CTC lattice) for a padded batch
 * log_probs: utterance n, frame t, class c at log_probs[n*stride_n + t*stride_t + c] (fp32 or bf16 per dtype,
 * class stride 1; the [T,N,V] view the CTC loss takes is stride_n = V, stride_t = N*V).  targets int64, utterance
 * n's labels at targets[n*target_stride ..]; input_lengths / target_lengths are int64 DEVICE tensors read on the
 * device (no host sync).
 * Outputs (caller-owned, written for every utterance): paths[n*T + t] (int32) = the label aligned to frame t,
 * scores[n*T + t] (log_probs dtype) = log_probs of that label at frame t, an exact copy; frames t >= input_lengths[n]
 * get blank and 0.  status[n] (int32): 0 aligned; 1 a label among the first target_lengths[n] is blank or outside
 * [0,V); 2 infeasible: input_lengths[n] < L + R (R = adjacent repeats); 3 a length outside [0,T] / [0,max_target_len].
 * A non-zero status leaves the row blank / 0.  Results are bit-identical to torchaudio's CPU forced_align run on the
 * utterance alone (same float32 sums, same comparison order on ties).  target_lengths[n] = 0 aligns every frame to
 * blank (torchaudio cannot express it).
 * Supported: 2*max_target_len+1 <= 511 and T x 128 bytes of back-pointers in shared memory (T up to ~1700);
 * AVCTC_ERR_UNSUPPORTED otherwise.  avctc_ctc_align_supported is the host-side query (1 = supported, 0 = not).
 * ---------------------------------------------------------------------------------------------- */
AVCTC_API int avctc_ctc_align_supported(int T, int max_target_len);
AVCTC_API int avctc_ctc_align(const void* log_probs, int dtype, int64_t stride_n, int64_t stride_t, int N, int T, int V,
                    const int64_t* targets, int64_t target_stride, const int64_t* input_lengths,
                    const int64_t* target_lengths, int max_target_len, int blank, int32_t* paths, void* scores,
                    int32_t* status, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Beam-search decode — replaces simple_beam_search(log_probs[T,V], beam_width, blank)
 *   /root/reference/beam_search.py:2-42, called per utterance at model/trainer.py:230,237
 * Batched: one CTA per utterance.  log_probs fp32, utterance n frame t class c at
 * log_probs[n*stride_n + t*stride_t + c].  lengths (int64 device, may be NULL = all T frames, which is
 * what the reference does) gives the number of frames to decode per utterance.
 * out_ids[n*T .. ] int32 receives the collapsed token ids, out_len[n] their count.
 * Token lists are bit-exact with the reference on CPU, including torch.topk's tie order.
 * Optional debug export (may be NULL): final beam scores dbg_scores[n*beam + i] (double) and raw
 * (uncollapsed) best-beam-first paths dbg_paths[(n*beam + i)*T + t] (int32).
 * ---------------------------------------------------------------------------------------------- */
AVCTC_API size_t avctc_beam_workspace_bytes(int N, int T, int V, int beam);
/* Which kernels avctc_beam_search will launch for this shape on the current device (148 SMs assumed without one) and
 * the current "beam_fused" / "beam_two_phase" knobs: host-side query, launches nothing. */
#define AVCTC_BEAM_ROUTE_NONE 0       /* shape not supported */
#define AVCTC_BEAM_ROUTE_SINGLE 1     /* one kernel, one warp per utterance does top-k and recurrence (V > 1024) */
#define AVCTC_BEAM_ROUTE_TWO_PHASE 2  /* top-k kernel over all N*T rows, then the recurrence kernel */
#define AVCTC_BEAM_ROUTE_FUSED 3      /* one persistent kernel: top-k warps feed recurrence warps through shared memory */
AVCTC_API int avctc_beam_route(int N, int T, int V, int beam);
AVCTC_API int avctc_beam_search(const float* log_probs, int64_t stride_n, int64_t stride_t, int N, int T, int V,
                      const int64_t* lengths, int beam, int blank,
                      int32_t* out_ids, int32_t* out_len, double* dbg_scores, int32_t* dbg_paths,
                      void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------------
 * CTC prefix beam search with N-best hypotheses (csrc/ctc_prefix_beam.cu; the search is defined in DESIGN.md §4.13 and
 * restated in oracle/prefix_beam_oracle.py, whose results it reproduces bit for bit).  Prefixes are scored by the
 * probability of all their alignments (fp64 natural logs).  log_probs fp32, utterance n frame t class c at
 * log_probs[n*stride_n + t*stride_t + c]; lengths int64 device (NULL = all T frames), read on the device.
 * beam in 1..15, nbest in 1..beam, blank in [0,V); V <= 1024 (AVCTC_ERR_UNSUPPORTED otherwise).
 * Outputs: hypothesis i of utterance n (best first) has out_len[n*nbest + i] tokens at out_tokens[(n*nbest + i)*T ..]
 * (entries past out_len are left untouched) and log-probability out_scores[n*nbest + i] (double).  Unused slots get
 * length 0 and score -inf.  status[n] (int32): 0 decoded; 1 a frame's log-probs contain NaN; 2 lengths[n] outside [0,T].
 * A failed utterance has no hypotheses.  lengths[n] = 0 gives one empty hypothesis of score 0.
 * Two kernel launches, no host sync.  The workspace query returns 0 for an unsupported shape.
 * ---------------------------------------------------------------------------------------------- */
AVCTC_API size_t avctc_ctc_prefix_beam_workspace_bytes(int N, int T, int V, int beam);
AVCTC_API int avctc_ctc_prefix_beam(const float* log_probs, int64_t stride_n, int64_t stride_t, int N, int T, int V,
                                    const int64_t* lengths, int beam, int nbest, int blank, int32_t* out_tokens,
                                    int32_t* out_len, double* out_scores, int32_t* status, void* workspace,
                                    size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------------
 * The same search with shallow fusion of a token-level back-off n-gram LM (DESIGN.md §4.14, restated in
 * oracle/prefix_beam_lm_oracle.py, whose results it reproduces bit for bit).  Each prefix carries an LM score L
 * (fp64 natural log): an extension s+c adds lm_weight * ln P(c | <s> s) + token_bonus, and candidates are ranked by
 * acoustic + L.  After the last frame lm_weight * ln P(</s> | <s> s) is added and the beam re-ranked.
 * LM words have ids 0..num_words-1 (num_words <= 2048, 11 bits).  An n-gram w1..wn is the key
 * sum_i w_i << 11*(n-i); the order-n table (n = 2..5) is table[n-2], `capacity` 16-byte entries {uint64 key; float
 * log10 p; float log10 back-off}, empty slots keyed ~0, at most half full, probed linearly from
 * slot = h & (capacity-1), h = key * 0x9E3779B97F4A7C15 (mod 2^64), h ^= h >> 29.  Unigrams are dense.
 * `lm` is a HOST pointer to the descriptor (read during the call); the pointers inside it are device memory.
 * lm_weight finite and >= 0, token_bonus finite, order 1..5, map_len == V; AVCTC_ERR_BAD_ARG otherwise, before any
 * launch.  Outputs as avctc_ctc_prefix_beam, with out_scores = out_acoustic + out_lm per hypothesis (unused slots
 * -inf in all three).  Same workspace query, two kernel launches, no host sync.
 * ---------------------------------------------------------------------------------------------- */
typedef struct avctc_ngram_lm {
    int order;                   /* 1..5 */
    int num_words;               /* LM word ids are 0..num_words-1, num_words <= 2048 */
    int bos, eos;                /* word ids of <s> and </s> */
    int map_len;                 /* entries of token_word: must equal V */
    const int32_t* token_word;   /* device [map_len]: model token -> LM word id (<unk>'s id for a piece the LM lacks) */
    const float* unigram;        /* device [num_words][2]: log10 p, log10 back-off (0 when absent) */
    const void* table[4];        /* device tables of orders 2..5 (unused past `order`) */
    uint64_t capacity[4];        /* entries of each table: a power of two >= 2 */
} avctc_ngram_lm;
AVCTC_API int avctc_ctc_prefix_beam_lm(const float* log_probs, int64_t stride_n, int64_t stride_t, int N, int T, int V,
                                       const int64_t* lengths, int beam, int nbest, int blank, const avctc_ngram_lm* lm,
                                       double lm_weight, double token_bonus, int32_t* out_tokens, int32_t* out_len,
                                       double* out_scores, double* out_acoustic, double* out_lm, int32_t* status,
                                       void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------------
 * The same search with contextual biasing towards a phrase list, with or without the n-gram LM (DESIGN.md §4.15,
 * restated in oracle/context_graph_oracle.py, whose results it reproduces bit for bit).  The phrases form an
 * Aho-Corasick automaton: node 0 is the root, node v has the depth potential phi(v) (the sum of its path's per-token
 * weights) and the completion credit omega(v) (phi of the first node on v's fail chain that ends a phrase, else 0).
 * Each prefix carries a node u and a bias score G (root and 0 for the empty prefix): an extension s+c moves to
 * v = delta(u, c) and adds (phi(v) - phi(u)) + omega(v) to G; candidates are ranked by (acoustic + L) + G, or
 * acoustic + G without an LM.  After the last frame bias = G - phi(u) and score = (acoustic + lm) + bias.
 * Candidates still come from the acoustic top-(2B+1) list of each frame: a phrase token outside it cannot be boosted.
 * Tables (device memory, `ctx` a HOST pointer read during the call): token_sym[map_len] maps a model token to its
 * context-alphabet symbol 0..alphabet-1, or -1 for a token of no phrase (which always returns to the root);
 * delta[num_nodes * alphabet] is the dense transition table, row-major by node; node[num_nodes] = (phi, omega).
 * `lm` NULL = no LM (lm_weight and token_bonus are ignored; out_lm gets 0 per hypothesis), else it is checked as by
 * avctc_ctc_prefix_beam_lm.  ctx non-NULL with num_nodes >= 1, map_len == V and alphabet in 1..V; AVCTC_ERR_BAD_ARG
 * otherwise, before any launch.  Outputs as avctc_ctc_prefix_beam_lm plus out_bias, with out_scores =
 * (out_acoustic + out_lm) + out_bias per hypothesis (unused slots -inf in all four).  Same workspace query, two
 * kernel launches, no host sync.
 * ---------------------------------------------------------------------------------------------- */
typedef struct avctc_context_graph {
    int num_nodes;               /* automaton nodes, root = 0 */
    int alphabet;                /* distinct phrase tokens: 1..V */
    const int32_t* token_sym;    /* device [map_len]: model token -> symbol, -1 when no phrase uses the token */
    int map_len;                 /* entries of token_sym: must equal V */
    const int32_t* delta;        /* device [num_nodes][alphabet]: next node */
    const double* node;          /* device [num_nodes][2]: phi, omega (16-byte aligned) */
} avctc_context_graph;
AVCTC_API int avctc_ctc_prefix_beam_biased(const float* log_probs, int64_t stride_n, int64_t stride_t, int N, int T,
                                           int V, const int64_t* lengths, int beam, int nbest, int blank,
                                           const avctc_ngram_lm* lm, double lm_weight, double token_bonus,
                                           const avctc_context_graph* ctx, int32_t* out_tokens, int32_t* out_len,
                                           double* out_scores, double* out_acoustic, double* out_lm, double* out_bias,
                                           int32_t* status, void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Fusion path dense contraction (tcgen05 + TMEM + TMA) — replaces the cuBLAS GEMMs under
 *   nn.Linear x4            /root/reference/model/fusion_module.py:57,58,63; model/decoder.py:24
 *   nn.MultiheadAttention   /root/reference/model/fusion_module.py:61 (in/out projections, Q.K^T, P.V)
 * and their backward passes.   C[z] = alpha * A[z] . B[z]^T (+ bias),   A: M x K,  B: N x K, bf16 in, fp32
 * accumulate.  An operand is a 3-D bf16 tensor described by avctc_gemm_operand:
 *   mn_major = 0: element (row r, k) at ptr[z*zstride + r*ld + k]   (row-major rows x K, e.g. activations, weights)
 *   mn_major = 1: element (row r, k) at ptr[z*zstride + k*ld + r]   (the transposed view; no copy is made)
 * rows/kdim/zdim are the tensor's full extents (TMA zero-fills reads outside them).  Batch entry
 * z in [0,batch) is split as outer = z / inner_count, inner = z % inner_count and reads its slice at
 * element offsets (k: outer*k_outer + inner*k_inner, row: outer*r_outer + inner*r_inner,
 * z: outer*z_outer + inner*z_inner); C[z] starts at C + outer*c_outer + inner*c_inner, row stride ldc.
 * ptr must be 16-byte aligned and ld, zstride multiples of 8 elements.
 * bias_mode: 0 none, 1 bias[n] per output column, 2 bias[m] per output row (fp32).  accumulate != 0 adds
 * into an fp32 C.
 * ---------------------------------------------------------------------------------------------- */
typedef struct {
    const void* ptr;
    long long rows, kdim, zdim, ld, zstride;
    int k_outer, k_inner, r_outer, r_inner, z_outer, z_inner;
    int mn_major;
} avctc_gemm_operand;

AVCTC_API int avctc_gemm_bf16(const avctc_gemm_operand* a, const avctc_gemm_operand* b, int M, int N, int K, int batch,
                    int inner_count, void* C, int out_dtype, long long ldc, long long c_outer, long long c_inner,
                    const float* bias, int bias_mode, float alpha, int accumulate, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Fusion glue — replaces the Python/ATen glue of CrossAttentionFusion.forward
 *   /root/reference/model/fusion_module.py:40-55 (speech-frame select, pad_sequence, F.interpolate linear
 *   align_corners=True for audio / nearest for the mask) and :66 (input_lengths), without host syncs.
 * audio [B,Ta,D] (fp32 or bf16, contiguous), mask [B,Ta] int64 in {0,1,2,3} -> out [B,Tv,D] bf16,
 * mask_out [B,Tv] int64, input_lengths [B] int64.  workspace keeps the compaction maps for backward.
 * If no frame of the whole batch is speech the reference raises inside F.interpolate; here out = 0 and
 * input_lengths = 0 (documented deviation, no host sync is spent on detecting it).
 * ---------------------------------------------------------------------------------------------- */
AVCTC_API size_t avctc_resample_workspace_bytes(int B, int Ta);
AVCTC_API int avctc_resample_forward(const void* audio, int dtype, const int64_t* mask, int B, int Ta, int D, int Tv,
                           void* out_bf16, int64_t* mask_out, int64_t* input_lengths, void* workspace,
                           size_t workspace_bytes, void* stream);
/* d_audio [B,Ta,D] (dtype fp32/bf16) from d_out [B,Tv,D] bf16; deterministic gather, zero for non-speech frames. */
AVCTC_API int avctc_resample_backward(const void* dout_bf16, int B, int Ta, int D, int Tv, const void* workspace,
                            void* daudio, int dtype, void* stream);

/* softmax over the first T entries of each Tp-strided row (nn.MultiheadAttention, no key mask):
 * S fp32 [rows,Tp] -> P bf16 [rows,Tp] with zero pad columns; backward dS = P*(dP - sum(dP*P)). */
AVCTC_API int avctc_softmax_forward(const float* S, void* P_bf16, long long rows, int T, int Tp, void* stream);
AVCTC_API int avctc_softmax_backward(const void* P_bf16, const float* dP, void* dS_bf16, long long rows, int T, int Tp,
                           void* stream);
/* out[n] (+)= sum_m X[m*ld + n]  (bias gradients).  ld >= N; AVCTC_ERR_BAD_ARG otherwise, and for a bad dtype, with
 * out left untouched. */
AVCTC_API int avctc_colsum(const void* X, int dtype, long long M, int N, long long ld, float* out, int accumulate,
                 void* stream);
/* CTC head: F.log_softmax over V classes (/root/reference/model/decoder.py:25) and its backward
 * dX = dY - exp(Y)*sum(dY), dX written as bf16 with row stride ldx. */
AVCTC_API int avctc_log_softmax_forward(const void* X, int in_dtype, void* Y, int out_dtype, long long rows, int V,
                              void* stream);
AVCTC_API int avctc_log_softmax_backward(const void* Y, const void* dY, int dtype, void* dX_bf16, long long rows, int V,
                               long long ldx, void* stream);

/* ------------------------------------------------------------------------------------------------
 * CTC head — CTCDecoder.forward, /root/reference/model/decoder.py:24-25: log_softmax(x . W^T + b) as ONE kernel
 * (csrc/ctc_head.cu): a thread-block cluster owns 128 rows x all V classes, the fp32 logits stay in tensor memory and
 * the per-row softmax statistics are exchanged through distributed shared memory, so the log-probs are the only
 * [M,V] tensor that touches HBM.  passes = 2 additionally applies the second F.log_softmax of evaluate()
 * (/root/reference/model/trainer.py:212,221) in the same kernel.
 * x: bf16 [M,K]; w: bf16 [V,K] (nn.Linear weight); bias: fp32 [V]; log_probs: fp32 [M,V].  V <= 1024, K % 8 == 0.
 * backward: dlog_probs fp32 [M,V] (+ the forward's log_probs) -> g_w fp32 [V,K], g_b fp32 [V] and, if non-NULL,
 * dx bf16 [M,K]; dz is caller-owned bf16 scratch of M * round_up(V, 8) elements.
 * ---------------------------------------------------------------------------------------------- */
AVCTC_API int avctc_ctc_head_forward(const void* x_bf16, const void* w_bf16, const float* bias, int M, int V, int K,
                           float* log_probs, int passes, void* stream);
AVCTC_API int avctc_ctc_head_backward(const float* log_probs, const float* dlog_probs, const void* x_bf16,
                            const void* w_bf16, int M, int V, int K, void* dz_bf16, float* g_w, float* g_b,
                            void* dx_bf16, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Attention core (tcgen05 + TMEM, scores never leave the SM) — replaces, inside nn.MultiheadAttention
 *   /root/reference/model/fusion_module.py:61 -> torch/nn/functional.py:6630-6652,
 * bmm(q / sqrt(hd), k^T) -> softmax over all T keys (no mask) -> bmm(P, v), and its autograd.
 * q: bf16 [B,T,E] (the projected queries, head h in columns [h*128, h*128+128)); kv: bf16 [B,T,2E] (keys | values).
 * o: bf16 [B,T,E] (heads already merged); lse2: fp32 [B*H,T] = log2 sum_j exp(s_ij / sqrt(hd)) (kept for backward).
 * backward: dout bf16 [B,T,E] plus the forward's o and lse2 -> dq bf16 [B,T,E], dkv bf16 [B,T,2E] (dk | dv).
 * Requires E == 128*H and T <= 192 (AVCTC_ERR_UNSUPPORTED otherwise); pointers 16-byte aligned.
 * ---------------------------------------------------------------------------------------------- */
AVCTC_API int avctc_attention_forward(const void* q, const void* kv, void* o, float* lse2, int B, int T, int H, int E,
                            void* stream);
AVCTC_API int avctc_attention_backward(const void* q, const void* kv, const void* dout, const void* o, const float* lse2,
                             void* dq, void* dkv, int B, int T, int H, int E, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Fused fusion path — CrossAttentionFusion.forward up to and including fusion_proj, and its backward,
 *   /root/reference/model/fusion_module.py:40-63 (resample, visual_proj, audio_proj, cross_attn_audio, fusion_proj)
 * as ONE host call each: the call enqueues the resample, the (grouped) tcgen05 GEMMs, the fused attention kernel
 * (csrc/attention.cu: Q.K^T -> softmax -> P.V with the scores in tensor memory; T <= 192 and head_dim 128, other shapes
 * run it as GEMM + softmax + GEMM) and the bias column sums on `stream`.  Requires fused_dim/num_heads to be a multiple
 * of 64 and Dv, Da multiples of 8.
 * visual: bf16 [B*T,Dv]; audio: fp32/bf16 [B,Ta,Da]; mask int64 [B,Ta]; weights and biases are the fp32 nn.Module
 * parameters (w_in/b_in = MultiheadAttention.in_proj_weight/bias [3E,E]/[3E]).  out: [B*T,E] fp32 or bf16 (out_dtype).
 * `wbf16` (which=3 bytes) holds the bf16 copies of the five weight matrices; the caller keeps it across calls and sets
 * refresh_weights != 0 whenever a weight changed since the buffer was last filled (first call, optimizer step) — the
 * library then re-casts them first.  backward must see the buffer as forward left it.
 * `saved` (which=0 bytes) carries the activations from forward to backward; `scratch` (which=1 for forward, which=2
 * for backward) is free after the call's kernels ran.  backward writes fp32 parameter gradients and, when the pointers
 * are non-NULL, d_visual (bf16 [B*T,Dv]) and d_audio ([B,Ta,Da], fp32 or bf16).  grads_zeroed != 0 promises that all
 * ten gradient tensors were zeroed by the caller (e.g. views of one zero-filled buffer): the library then skips its
 * own per-tensor memsets.
 * ---------------------------------------------------------------------------------------------- */
AVCTC_API size_t avctc_fusion_workspace_bytes(int B, int T, int Ta, int Dv, int Da, int E, int H, int which);
AVCTC_API int avctc_fusion_forward(const void* visual_bf16, const void* audio, int audio_dtype, const int64_t* mask,
                         const float* w_vp, const float* b_vp, const float* w_ap, const float* b_ap,
                         const float* w_in, const float* b_in, const float* w_o, const float* b_o,
                         const float* w_f, const float* b_f, int B, int T, int Ta, int Dv, int Da, int E, int H,
                         void* out, int out_dtype, int64_t* mask_out, int64_t* input_lengths,
                         void* wbf16, size_t wbf16_bytes, int refresh_weights, void* saved, size_t saved_bytes,
                         void* scratch, size_t scratch_bytes, void* stream);
AVCTC_API int avctc_fusion_backward(const void* df, int df_dtype, const void* visual_bf16, int B, int T, int Ta, int Dv,
                          int Da, int E, int H, float* g_wvp, float* g_bvp, float* g_wap, float* g_bap,
                          float* g_win, float* g_bin, float* g_wo, float* g_bo, float* g_wf, float* g_bf,
                          void* d_visual_bf16, void* d_audio, int d_audio_dtype, const void* wbf16, size_t wbf16_bytes,
                          const void* saved, size_t saved_bytes, void* scratch, size_t scratch_bytes, int grads_zeroed,
                          void* stream);

/* ------------------------------------------------------------------------------------------------
 * temporal_model — nn.LSTM(E, E, num_layers=2, batch_first=True, bidirectional=True), zero initial state,
 *   /root/reference/model/fusion_module.py:21-27, called at :64 over all padded frames
 * as persistent cooperative kernels (csrc/lstm.cu).  H in {256, 512}, B <= 64 (H = 512) / 128 (H = 256), In % 8 == 0;
 * calls with more than 8 sequences run as independent batch groups side by side in one launch.
 * x: bf16 [B,T,In]; params / grads: HOST arrays of 16 DEVICE fp32 pointers in nn.LSTM's flat parameter order
 * (weight_ih_l0 [4H,In], weight_hh_l0 [4H,H], bias_ih_l0 [4H], bias_hh_l0 [4H], the same four "_reverse", then the
 * four + four of layer 1 with In = 2H); gate order i,f,g,o.  y: bf16 [B,T,2H].  `saved` (which=0) carries weights in
 * bf16, gates and cell states from forward to backward (written only when need_grad); scratch which=1 forward,
 * which=2 backward.  backward: dy bf16 [B,T,2H] -> 16 parameter gradients and, if non-NULL, dx bf16 [B,T,In].
 * The kernels use a cooperative launch (groups * 2*H/16 <= 128 CTAs must be co-resident).
 * ---------------------------------------------------------------------------------------------- */
AVCTC_API size_t avctc_bilstm_workspace_bytes(int B, int T, int In, int H, int which);
AVCTC_API int avctc_bilstm_forward(const void* x_bf16, int B, int T, int In, int H, const float* const* params,
                         void* y_bf16, void* saved, size_t saved_bytes, void* scratch, size_t scratch_bytes,
                         int need_grad, void* stream);
AVCTC_API int avctc_bilstm_backward(const void* dy_bf16, const void* x_bf16, int B, int T, int In, int H,
                          float* const* grads, void* dx_bf16, const void* saved, size_t saved_bytes,
                          void* scratch, size_t scratch_bytes, void* stream);

/* ------------------------------------------------------------------------------------------------
 * InfoNCE — replaces contrastive_loss_with_mask after its optional projection
 *   /root/reference/contrastive.py:13-44 (valid-row select, F.normalize, index sets, sim/TEMPERATURE,
 *   -log_softmax(.).mean() for (weak,strong) * w_pos and (weak,neg) * w_neg), called at model/trainer.py:108-109.
 * y [N,P] (fp32 or bf16, row stride ld): the projected (or raw) features of ALL B*T rows; flat_mask [N] int64 in
 * {0,1,2,3}.  loss: 1 fp32.  Nothing is gathered on the host and no count leaves the device.  P <= 256.
 * backward writes dy [N,P] (zero rows for mask==3) given the DEVICE scalar grad_out.
 * ---------------------------------------------------------------------------------------------- */
AVCTC_API size_t avctc_infonce_workspace_bytes(int N, int P);
AVCTC_API int avctc_infonce_forward(const void* y, int dtype, long long ld, const int64_t* flat_mask, int N, int P,
                          float temperature, float w_pos, float w_neg, float* loss, void* workspace,
                          size_t workspace_bytes, void* stream);
AVCTC_API int avctc_infonce_backward(const int64_t* flat_mask, int N, int P, float temperature, float w_pos, float w_neg,
                           const float* grad_out, void* dy, int dtype, long long ld, void* workspace,
                           size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Visual encoder forward (encoders.py VisualEncoder, frozen, bf16 autocast) around cuDNN's trunk convolutions.
 * Activations are NHWC bf16 ([rows, C], C contiguous, 16-byte aligned); statistics partials are fp32 [3][C][P]
 * (count, mean, M2 per channel and producing CTA), combined in a fixed order (bit-identical runs).
 * avctc_visual_frontend: x [B,1,T,H,W] fp32 -> y [B*T, Ho, Wo, 64] bf16, Ho = (H-1)/2+1, Wo = (W-1)/2+1: the (5,7,7)
 *   Conv3d, stride (1,2,2), padding (2,3,3), over the bf16-rounded clip; w_bf16 [64][256] = weight[:,0] as
 *   [64, 5*7*7] zero-padded to 256.  partials [3][64][P], P = avctc_visual_frontend_ctas(), or NULL (no statistics).
 * avctc_bn_stats: partials of x [M, C] (C % 8 == 0, 256 % (C/8) == 0), P = avctc_bn_stats_ctas(M, C).
 * avctc_bn_finalize: scale_shift [2][C] = {gamma/sqrt(var+eps), beta - mean*scale}; training = 1: batch statistics
 *   from the partials (biased variance) and running_mean/var updated in place (momentum, unbiased variance);
 *   training = 0: from the running statistics, nothing updated.  weight / bias may be NULL (1 / 0).
 * avctc_visual_frontend_pool: out [N, (H-1)/2+1, (W-1)/2+1, 64] = 3x3/2 max pool (padding 1) of
 *   bf16(PReLU(bf16(y*scale+shift))), y [N, H, W, 64].
 * avctc_bn_act: out = bf16(PReLU(z)), z = bf16(x*scale+shift) [+ residual: z = bf16(z + r), r = res or, with
 *   res_scale_shift, bf16(res*res_scale+res_shift)]; pool_hw > 0: out [M/pool_hw, C] = bf16(mean over each
 *   group of pool_hw rows).  slope_bf16: PReLU slope per channel.
 * ---------------------------------------------------------------------------------------------- */
AVCTC_API int avctc_visual_frontend_ctas(int B, int T, int H, int W);
AVCTC_API int avctc_visual_frontend(const float* x, int B, int T, int H, int W, const void* w_bf16, void* y_bf16,
                                    float* partials, int P, void* stream);
AVCTC_API int avctc_bn_stats_ctas(long long M, int C);
AVCTC_API int avctc_bn_stats(const void* x_bf16, long long M, int C, float* partials, int P, void* stream);
AVCTC_API int avctc_bn_finalize(const float* partials, int P, int C, const float* weight, const float* bias,
                                float* running_mean, float* running_var, float momentum, float eps, int training,
                                float* scale_shift, void* stream);
AVCTC_API int avctc_visual_frontend_pool(const void* y_bf16, long long N, int H, int W, const float* scale_shift,
                                         const void* slope_bf16, void* out_bf16, void* stream);
AVCTC_API int avctc_bn_act(const void* x_bf16, long long M, int C, const float* scale_shift, const void* slope_bf16,
                           const void* res_bf16, const float* res_scale_shift, int pool_hw, void* out_bf16,
                           void* stream);

/* ------------------------------------------------------------------------------------------------
 * wav2vec2 encoder layer (Wav2Vec2EncoderLayerStableLayerNorm, bf16 autocast, train or eval) around torch's attention
 * core (csrc/wav2vec2_layer.cu).  Rows M = B*T, hidden E (multiple of 256, <= 1024), intermediate F (multiple of 8).
 * Activations are contiguous bf16 [M, E] / [M, F], 16-byte aligned; LayerNorm weights/biases fp32; weights bf16 in
 * nn.Linear layout; biases fp32 holding the bf16-rounded values autocast would add.  Every tensor the module path
 * materialises in bf16 is rounded at the same point.
 * avctc_w2v_attn_in_forward: ln1 = LayerNorm(x) (fp32 math), q/k/v = ln1 . W^T + b into three [M, E] tensors;
 *   wqkv = [Wq; Wk; Wv] [3E, E], bqkv [3E].
 * avctc_w2v_attn_out_ffn_forward: attn [M, E] = the attention output HF feeds out_proj; x = the layer input;
 *   h = bf16(x + drop_h(attn . Wo^T + bo)); y = bf16(h + drop_o(drop_a(gelu(LayerNorm(h) . W1^T + b1)) . W2^T + b2)).
 *   Dropouts (training != 0, p > 0) reproduce ATen's CUDA native_dropout for Philox (seed, offset) bit for bit; the three
 *   take consecutive offsets from `offset` in that order, together avctc_w2v_dropout_increment(): the caller advances
 *   its generator by that much.
 * Backward entries take the forward's `saved` buffer unchanged plus a scratch buffer, regenerate the dropout masks from
 *   the same (seed, offset), and write bf16 input gradients.  The fp32 parameter gradients (all NULL or all set) are
 *   written, not accumulated; LayerNorm and bias gradients are reduced in a fixed order.
 *   attn_in_backward: dq, dk, dv contiguous [M, E] -> dx (the LayerNorm branch's share of d x).
 *   attn_out_ffn_backward: dy -> dattn and dx (the residual branch's share of d x).
 * avctc_w2v_workspace_bytes: which = 0 attn_in saved, 1 attn_out_ffn saved, 2 attn_in scratch, 3 attn_out_ffn scratch.
 * avctc_w2v_dropout: y = native_dropout(x, p) for a contiguous bf16 x of n elements (n % 8 == 0) at (seed, offset).
 * ---------------------------------------------------------------------------------------------- */
AVCTC_API size_t avctc_w2v_workspace_bytes(long long M, int E, int F, int which);
AVCTC_API long long avctc_w2v_dropout_increment(long long M, int E, int F, double p_hidden, double p_act, double p_out,
                                                int training);
AVCTC_API int avctc_w2v_dropout(const void* x, long long n, double p, unsigned long long seed, unsigned long long offset,
                                void* y, void* stream);
AVCTC_API int avctc_w2v_attn_in_forward(const void* x, long long M, int E, const float* ln_w, const float* ln_b, float eps,
                                        const void* wqkv, const float* bqkv, void* q, void* k, void* v, void* saved,
                                        size_t saved_bytes, void* stream);
AVCTC_API int avctc_w2v_attn_in_backward(const void* dq, const void* dk, const void* dv, const void* x, long long M, int E,
                                         const float* ln_w, const void* wqkv, void* dx, float* g_wqkv, float* g_bqkv,
                                         float* g_lnw, float* g_lnb, const void* saved, size_t saved_bytes, void* scratch,
                                         size_t scratch_bytes, void* stream);
AVCTC_API int avctc_w2v_attn_out_ffn_forward(const void* attn, const void* x, long long M, int E, int F, const void* wo,
                                             const float* bo, const float* ln_w, const float* ln_b, float eps,
                                             const void* w1, const float* b1, const void* w2, const float* b2,
                                             double p_hidden, double p_act, double p_out, int training,
                                             unsigned long long seed, unsigned long long offset, void* y, void* saved,
                                             size_t saved_bytes, void* stream);
AVCTC_API int avctc_w2v_attn_out_ffn_backward(const void* dy, const void* attn, long long M, int E, int F, const void* wo,
                                              const float* ln_w, const void* w1, const void* w2, double p_hidden,
                                              double p_act, double p_out, int training, unsigned long long seed,
                                              unsigned long long offset, void* dattn, void* dx, float* g_wo, float* g_bo,
                                              float* g_lnw, float* g_lnb, float* g_w1, float* g_b1, float* g_w2,
                                              float* g_b2, const void* saved, size_t saved_bytes, void* scratch,
                                              size_t scratch_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* AVCTC_B200_H_ */
