"""CTC forced alignment: where in the recording each token of a KNOWN transcript was spoken.

    forced_align(log_probs[N,T,V], targets[N,L], input_lengths=None, target_lengths=None, blank=0) -> (paths, scores)
    merge_tokens(tokens[T], scores[T], blank=0) -> list[TokenSpan]
    merge_tokens_batch(paths, scores, input_lengths=None, blank=0) -> list[list[TokenSpan]]

forced_align has torchaudio.functional.forced_align's signature, defaults, return dtypes and results, but takes a
padded batch: row n on frames [0, input_lengths[n]) is bit-identical to torchaudio's CPU forced_align run on that
utterance alone (paths, and scores as exact copies of the input values); frames past an utterance's input length get
blank and 0.  One kernel launch (csrc/ctc_align.cu) and one host sync, to read the per-utterance status.
A target length of 0 aligns every frame to blank, which torchaudio cannot express.  CUDA tensors only.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import List

import torch

from . import _lib


def forced_align(log_probs, targets, input_lengths=None, target_lengths=None, blank: int = 0):
    _lib.require_cuda(log_probs, "log_probs")
    _lib.require_cuda(targets, "targets")
    if log_probs.dim() != 3:
        raise RuntimeError("log_probs must be a 3-D tensor")
    if targets.dim() != 2:
        raise RuntimeError("targets must be a 2-D tensor")
    if targets.dtype not in (torch.int32, torch.int64):
        raise RuntimeError("targets must be int32 or int64 type")
    N, T, V = log_probs.shape
    if targets.shape[0] != N:
        raise RuntimeError(f"targets has {targets.shape[0]} rows, log_probs has {N} utterances")
    if not 0 <= blank < V:
        raise RuntimeError("blank must be within [0, num classes)")
    dt = _lib.dtype_enum(log_probs)
    dev = log_probs.device
    Lmax = targets.shape[1]
    if log_probs.stride(2) != 1:
        log_probs = log_probs.contiguous()
    tg = targets.to(device=dev, dtype=torch.int64)
    if tg.stride(1) != 1:
        tg = tg.contiguous()
    if input_lengths is None:
        input_lengths = torch.full((N,), T, dtype=torch.int64, device=dev)
    if target_lengths is None:
        target_lengths = torch.full((N,), Lmax, dtype=torch.int64, device=dev)
    il = input_lengths.to(device=dev, dtype=torch.int64).contiguous()
    tl = target_lengths.to(device=dev, dtype=torch.int64).contiguous()
    if il.shape != (N,) or tl.shape != (N,):
        raise RuntimeError("input_lengths and target_lengths must be 1-D tensors of one entry per utterance")
    paths = torch.empty((N, T), dtype=torch.int32, device=dev)
    scores = torch.empty((N, T), dtype=log_probs.dtype, device=dev)
    status = torch.empty((N,), dtype=torch.int32, device=dev)
    with _lib.device_guard(dev):
        _lib.check(_lib.lib().avctc_ctc_align(log_probs.data_ptr(), dt, log_probs.stride(0), log_probs.stride(1), N, T, V,
                                              tg.data_ptr(), tg.stride(0), il.data_ptr(), tl.data_ptr(), Lmax, blank,
                                              paths.data_ptr(), scores.data_ptr(), status.data_ptr(),
                                              _lib.stream_ptr(dev)), "avctc_ctc_align")
    st = status.cpu()                                    # the one host sync
    bad = torch.nonzero(st).flatten()
    if len(bad):
        _raise_for(int(bad[0]), int(st[bad[0]]), tg, il, tl, T, V, blank)
    return paths.to(targets.dtype), scores


def _raise_for(n, code, tg, il, tl, T, V, blank):
    """torchaudio's message for the first rejected utterance, prefixed with its index (host reads on the error path)."""
    if code == 3:
        raise RuntimeError(f"utterance {n}: input length {int(il[n])} outside [0, {T}] or target length {int(tl[n])} "
                           f"outside [0, {tg.shape[1]}]")
    row = tg[n, :int(tl[n])].cpu()
    if code == 1:
        if bool((row == blank).any()):
            raise ValueError(f"utterance {n}: targets Tensor shouldn't contain blank index. Found {row}.")
        raise ValueError(f"utterance {n}: targets values must be less than the CTC dimension (and not negative)")
    R = int((row[1:] == row[:-1]).sum()) if len(row) > 1 else 0
    raise RuntimeError(f"utterance {n}: targets length is too long for CTC. Found log_probs length: {int(il[n])}, "
                       f"targets length: {len(row)}, and number of repeats: {R}")


@dataclass
class TokenSpan:
    """torchaudio.functional.TokenSpan: one token with frame span [start, end) and the mean of its frame scores."""
    token: int
    start: int
    end: int
    score: float

    def __len__(self) -> int:
        return self.end - self.start


def merge_tokens(tokens, scores, blank: int = 0) -> List[TokenSpan]:
    """torchaudio.functional.merge_tokens: collapse one utterance's frame labels into token spans (blank dropped,
    end exclusive, score = scores[start:end].mean() in the scores' dtype)."""
    if tokens.ndim != 1 or scores.ndim != 1:
        raise ValueError("`tokens` and `scores` must be 1D Tensor.")
    if len(tokens) != len(scores):
        raise ValueError("`tokens` and `scores` must be the same length.")
    edge = torch.tensor([-1], device=tokens.device, dtype=tokens.dtype)
    diff = torch.diff(tokens, prepend=edge, append=edge)
    changes = torch.nonzero(diff != 0).flatten().tolist()
    toks = tokens.tolist()
    return [TokenSpan(token=toks[s], start=s, end=e, score=scores[s:e].mean().item())
            for s, e in zip(changes[:-1], changes[1:]) if toks[s] != blank]


def merge_tokens_batch(paths, scores, input_lengths=None, blank: int = 0) -> List[List[TokenSpan]]:
    """merge_tokens for every row of a forced_align result, each cut at its input length, after ONE device-to-host
    copy (paths, scores and lengths packed into one float64 block: every value is exact in it)."""
    N, T = paths.shape
    if input_lengths is None:
        input_lengths = torch.full((N,), T, dtype=torch.int64, device=paths.device)
    block = torch.cat([paths.to(torch.float64), scores.to(torch.float64),
                       input_lengths.to(device=paths.device, dtype=torch.float64).view(N, 1)], dim=1).cpu()
    p = block[:, :T].to(paths.dtype)
    s = block[:, T:2 * T].to(scores.dtype)
    lens = block[:, 2 * T].to(torch.int64).tolist()
    return [merge_tokens(p[n, :lens[n]], s[n, :lens[n]], blank) for n in range(N)]


# ------------------------------------------------------------------------------------------------ fused frames -> time
def nearest_src_index(out_size: int, in_size: int) -> torch.Tensor:
    """F.interpolate(mode='nearest') source index, float32 like ATen: min(floor(dst * float32(in/out)), in-1).  The map
    the fusion module's mask resample applies (avctc_resample_forward) from T_v fused frames to speech-frame ranks."""
    scale = torch.tensor(in_size, dtype=torch.float32) / torch.tensor(out_size, dtype=torch.float32)
    src = torch.floor(torch.arange(out_size, dtype=torch.float32) * scale).to(torch.int64)
    return torch.clamp(src, max=in_size - 1)


def fused_frame_encoder_index(mask_ds, t_v: int):
    """For a speaker's downsampled mask [B, T_enc] (host tensor; speech = value not in {0, 3}): the encoder frame of
    every fused frame, [B, T_v] int64 (-1 where the fused frame is padding).  The fusion compacts each utterance's
    speech frames, pads them to Tp = the batch's largest speech count and resamples Tp -> T_v with nearest_src_index;
    this inverts that map."""
    mask_ds = torch.as_tensor(mask_ds)
    speech = (mask_ds != 0) & (mask_ds != 3)
    counts = speech.sum(1)
    B = mask_ds.shape[0]
    out = torch.full((B, t_v), -1, dtype=torch.int64)
    Tp = int(counts.max()) if B else 0
    if Tp == 0:
        return out
    rank = nearest_src_index(t_v, Tp)
    for b in range(B):
        frames = torch.nonzero(speech[b]).flatten()
        ok = rank < len(frames)
        out[b, ok] = frames[rank[ok]]
    return out


@dataclass
class TimedTokenSpan(TokenSpan):
    """A TokenSpan with its piece text and its time in the mixed recording: [start_sec, end_sec]."""
    piece: str = ""
    start_sec: float = 0.0
    end_sec: float = 0.0
