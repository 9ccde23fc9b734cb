// beam_internal.h — library-internal launch interface of the per-frame top-k pass (beam_search.cu), shared with the
// CTC prefix beam search (ctc_prefix_beam.cu).  Not part of the public C ABI.
#pragma once
#include <stdint.h>

// torch.topk(log_probs[n, t], k) for every frame t < lengths[n] (all T when lengths is NULL) of every utterance, in
// torch's CPU order including ties: values to tk_val[(n*T + t)*k + j], classes to tk_idx[...].  One launch of
// beam_topk_kernel.  V <= 1024, k + 1 <= 32, k <= V and N*T < 2^31, else AVCTC_ERR_UNSUPPORTED (nothing launched).
int avctc_beam_topk_lists(const float* log_probs, int64_t stride_n, int64_t stride_t, int N, int T, int V,
                          const int64_t* lengths, int k, float* tk_val, int32_t* tk_idx, void* stream);
