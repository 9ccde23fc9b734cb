"""CTC prefix beam search: ranked transcription hypotheses with their log-probabilities.

    ctc_prefix_beam_search(log_probs[N,T,V], lengths=None, beam_width=5, nbest=1, blank=0,
                           lm=None, lm_weight=0.5, token_bonus=0.0, context=None) -> list[list[Hypothesis]]

Unlike simple_beam_search, which keeps raw alignment paths and so returns the greedy collapse, the prefix beam search
scores each prefix by the sum over all of its alignments and merges the alignments that collapse to the same text.
The search is defined in DESIGN.md §4.13; the kernel (csrc/ctc_prefix_beam.cu) reproduces the CPU restatement in
oracle/prefix_beam_oracle.py bit for bit, scores included.  Two kernel launches and one host sync per call.  CUDA
tensors only.

With an n-gram LM (ngram_lm.NgramLM), the search fuses it shallowly (DESIGN.md §4.14, oracle/prefix_beam_lm_oracle.py):
prefixes are ranked by acoustic + lm_weight * ln P_LM + token_bonus * length, </s> included at the end, and each
hypothesis is an LMHypothesis carrying both parts.

With a phrase list (context_graph.ContextGraph), the search biases towards those phrases (DESIGN.md §4.15,
oracle/context_graph_oracle.py), with or without an LM: prefixes are ranked by acoustic (+ lm) + bias, a completed
phrase earns the sum of its per-token weights, and each hypothesis is a BiasedHypothesis.
"""
from __future__ import annotations

import ctypes
import math
from dataclasses import dataclass
from typing import List

import numpy as np
import torch

from . import _lib
from .context_graph import ContextGraph
from .ngram_lm import NgramLM

MAX_BEAM = 15


@dataclass
class Hypothesis:
    """One decoded prefix: token ids (blanks and repeats already merged) and its natural-log probability."""
    tokens: List[int]
    score: float


@dataclass
class LMHypothesis(Hypothesis):
    """A hypothesis of the LM-fused search: score = acoustic_score + lm_score (one fp64 add), where acoustic_score is
    the CTC log-probability and lm_score = lm_weight * ln P_LM(tokens </s>) + token_bonus * len(tokens)."""
    acoustic_score: float
    lm_score: float


@dataclass
class BiasedHypothesis(LMHypothesis):
    """A hypothesis of the biased search: score = (acoustic_score + lm_score) + bias_score, where bias_score is the
    sum of the per-token weights of every phrase the tokens complete (lm_score is 0.0 without an LM)."""
    bias_score: float


def ctc_prefix_beam_search(log_probs, lengths=None, beam_width: int = 5, nbest: int = 1, blank: int = 0,
                           lm: NgramLM = None, lm_weight: float = 0.5, token_bonus: float = 0.0,
                           context: ContextGraph = None) -> List[List[Hypothesis]]:
    """log_probs: CUDA [N,T,V] log-probabilities (any float dtype; read as fp32).  lengths: frames to decode per
    utterance (default T).  Returns, per utterance, up to nbest hypotheses, best first.  V <= 1024.  With `lm`, an
    NgramLM built for this model's V pieces, hypotheses are LMHypothesis ranked by the fused score; lm_weight must be
    finite and >= 0, token_bonus finite.  With `context`, a ContextGraph built for V pieces and this blank, hypotheses
    are BiasedHypothesis ranked by the biased score, with or without `lm`."""
    _lib.require_cuda(log_probs, "log_probs")
    if log_probs.dim() != 3:
        raise RuntimeError("log_probs must be (N, T, V)")
    N, T, V = log_probs.shape
    B, nbest, blank = int(beam_width), int(nbest), int(blank)
    if not 1 <= B <= MAX_BEAM:
        raise ValueError(f"beam_width must be in [1, {MAX_BEAM}], got {B}")
    if not 1 <= nbest <= B:
        raise ValueError(f"nbest must be in [1, beam_width={B}], got {nbest}")
    if not 0 <= blank < V:
        raise ValueError(f"blank must be in [0, {V}), got {blank}")
    if lm is not None:
        if not isinstance(lm, NgramLM):
            raise TypeError(f"lm must be an NgramLM, got {type(lm).__name__}")
        if lm.vocab_size != V:
            raise ValueError(f"the LM was built for {lm.vocab_size} pieces, log_probs have V={V} classes")
        alpha, beta = float(lm_weight), float(token_bonus)
        if not (math.isfinite(alpha) and alpha >= 0.0):
            raise ValueError(f"lm_weight must be finite and >= 0, got {lm_weight}")
        if not math.isfinite(beta):
            raise ValueError(f"token_bonus must be finite, got {token_bonus}")
    if context is not None:
        if not isinstance(context, ContextGraph):
            raise TypeError(f"context must be a ContextGraph, got {type(context).__name__}")
        if context.vocab_size != V:
            raise ValueError(f"the context graph was built for {context.vocab_size} pieces, log_probs have V={V} classes")
        if context.blank != blank:
            raise ValueError(f"the context graph was built for blank {context.blank}, the search uses blank {blank}")
    lp = log_probs.detach()
    if lp.dtype != torch.float32:
        lp = lp.float()
    if lp.stride(2) != 1:
        lp = lp.contiguous()
    dev = lp.device
    L = _lib.lib()
    ws_bytes = int(L.avctc_ctc_prefix_beam_workspace_bytes(N, T, V, B))
    if ws_bytes == 0:
        raise RuntimeError(f"ctc_prefix_beam_search: shape N={N}, T={T}, V={V} is not supported (V <= 1024)")
    if lengths is not None:
        lengths = torch.as_tensor(lengths).to(device=dev, dtype=torch.int64).contiguous()
        if lengths.shape != (N,):
            raise RuntimeError("lengths must be a 1-D tensor of one entry per utterance")
    Tp = max(T, 1)
    # every output in one device buffer, so that results and statuses come back with one copy; with an LM the scores
    # are [3][N][nbest]: fused, acoustic, LM; with a context graph [4][N][nbest]: fused, acoustic, LM, bias
    nsc = 4 if context is not None else 1 if lm is None else 3
    n_sc, n_len, n_st, n_tok = nsc * N * nbest * 8, N * nbest * 4, N * 4, N * nbest * Tp * 4
    o_len = n_sc
    o_st = o_len + n_len
    o_tok = (o_st + n_st + 7) // 8 * 8
    out = torch.empty(o_tok + n_tok, dtype=torch.uint8, device=dev)
    scores = out[:o_len].view(torch.float64)
    lens = out[o_len:o_st].view(torch.int32)
    status = out[o_st:o_st + n_st].view(torch.int32)
    tokens = out[o_tok:].view(torch.int32)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    with _lib.device_guard(dev):
        if context is not None:
            sc4 = scores.view(4, N * nbest)
            _lib.check(L.avctc_ctc_prefix_beam_biased(
                lp.data_ptr(), lp.stride(0), lp.stride(1), N, T, V, lengths.data_ptr() if lengths is not None else None,
                B, nbest, blank, ctypes.addressof(lm.descriptor(dev)) if lm is not None else None,
                alpha if lm is not None else 0.0, beta if lm is not None else 0.0,
                ctypes.addressof(context.descriptor(dev)), tokens.data_ptr(), lens.data_ptr(), sc4[0].data_ptr(),
                sc4[1].data_ptr(), sc4[2].data_ptr(), sc4[3].data_ptr(), status.data_ptr(), ws.data_ptr(), ws_bytes,
                _lib.stream_ptr(dev)), "avctc_ctc_prefix_beam_biased")
        elif lm is None:
            _lib.check(L.avctc_ctc_prefix_beam(
                lp.data_ptr(), lp.stride(0), lp.stride(1), N, T, V, lengths.data_ptr() if lengths is not None else None,
                B, nbest, blank, tokens.data_ptr(), lens.data_ptr(), scores.data_ptr(), status.data_ptr(),
                ws.data_ptr(), ws_bytes, _lib.stream_ptr(dev)), "avctc_ctc_prefix_beam")
        else:
            desc = lm.descriptor(dev)
            sc3 = scores.view(3, N * nbest)
            _lib.check(L.avctc_ctc_prefix_beam_lm(
                lp.data_ptr(), lp.stride(0), lp.stride(1), N, T, V, lengths.data_ptr() if lengths is not None else None,
                B, nbest, blank, ctypes.addressof(desc), alpha, beta, tokens.data_ptr(), lens.data_ptr(),
                sc3[0].data_ptr(), sc3[1].data_ptr(), sc3[2].data_ptr(), status.data_ptr(), ws.data_ptr(), ws_bytes,
                _lib.stream_ptr(dev)), "avctc_ctc_prefix_beam_lm")
    host = out.cpu().numpy()                              # the one host sync
    sc_all = host[:o_len].view(np.float64).reshape(nsc, N, nbest)
    sc = sc_all[0]
    ln = host[o_len:o_st].view(np.int32).reshape(N, nbest)
    st = host[o_st:o_st + n_st].view(np.int32)
    tk = host[o_tok:].view(np.int32).reshape(N, nbest, Tp)
    bad = np.flatnonzero(st)
    if len(bad):
        n = int(bad[0])
        if st[n] == 1:
            raise RuntimeError(f"ctc_prefix_beam_search: utterance {n}: log_probs contain NaN")
        raise RuntimeError(f"ctc_prefix_beam_search: utterance {n}: length {int(lengths[n])} outside [0, {T}]")
    res = []
    for n in range(N):
        row = []
        for i in range(nbest):
            if not sc[n, i] > -np.inf:                    # unused slot
                break
            if context is not None:
                row.append(BiasedHypothesis(tk[n, i, :ln[n, i]].tolist(), float(sc[n, i]), float(sc_all[1, n, i]),
                                            float(sc_all[2, n, i]), float(sc_all[3, n, i])))
            elif lm is None:
                row.append(Hypothesis(tk[n, i, :ln[n, i]].tolist(), float(sc[n, i])))
            else:
                row.append(LMHypothesis(tk[n, i, :ln[n, i]].tolist(), float(sc[n, i]), float(sc_all[1, n, i]),
                                        float(sc_all[2, n, i])))
        res.append(row)
    return res
