"""float64 restatement of the fusion-path kernels of csrc/fusion_kernels.cu, csrc/attention.cu and csrc/gemm_tcgen05.cu,
forward and backward written out step by step (no autograd), on plain torch ops.

  resample     speech-frame select -> zero pad to the batch max Tp -> linear interpolation (align_corners=True) to Tv
               frames; nearest-neighbour resample of the mask; input_lengths = count(mask_out != 0).  The backward is
               the adjoint of the forward: the [Tv, Tp] interpolation matrix transposed, scattered back to each
               sample's speech frames.
  softmax      over the first T of Tp columns (pad columns 0); the backward takes the bf16 P the forward wrote.
  colsum       column sums (bias gradients).
  log_softmax  over V classes, and dX = dY - exp(Y) * sum(dY).
  attention    softmax(q k^T / sqrt(128)) v per head of 128 columns, and its backward.  With ``round_bf16=True`` the
               values the kernel materialises in bf16 are rounded at the same points: the unnormalised P before P.V,
               P and dS in the backward, and the outputs; D = rowsum(dO * O) is taken from the bf16 O the caller
               passes.
  gemm         C = alpha * A . B^T (+ bias per column or per row) (+ C).

Every function takes and returns torch tensors on any device; it computes in float64.

TEST INFRASTRUCTURE ONLY: nothing in the package imports this module."""
from __future__ import annotations

import math

import torch

f64 = torch.float64
LN2 = math.log(2.0)


def _rbf(t, on):
    return t.to(torch.bfloat16).to(f64) if on else t


# ----------------------------------------------------------------------------------------------------- resample
def speech_index(mask):
    """-> (src [B, Ta] int64: original index of the i-th speech frame in its first cnt[b] entries, cnt [B])."""
    speech = (mask != 0) & (mask != 3)
    cnt = speech.sum(1)
    src = torch.argsort((~speech).to(torch.int8), dim=1, stable=True)
    return src, cnt


def lerp_coef(Tp, Tv, device=None, dtype=f64):
    """(i0, i1, w0, w1) [Tv] of ATen's upsample_linear1d with align_corners=True; (t, t, 1, 0) when Tp == Tv.  The
    scale (Tp-1)/(Tv-1), the source index and the weights are computed in `dtype`, as ATen does in the tensor's opmath
    type (float32 for float32 and bf16 tensors); the weights are returned as float64."""
    t = torch.arange(Tv, device=device)
    if Tp == Tv:
        return t, t, torch.ones(Tv, dtype=f64, device=device), torch.zeros(Tv, dtype=f64, device=device)
    scale = (torch.tensor(Tp - 1, dtype=dtype) / (Tv - 1)).to(device) if Tv > 1 else torch.zeros((), dtype=dtype,
                                                                                                   device=device)
    s = t.to(dtype) * scale
    i0 = s.floor().long()
    w1 = s - i0.to(dtype)
    return i0, i0 + (i0 < Tp - 1).long(), (1 - w1).to(f64), w1.to(f64)


def lerp_matrix(Tp, Tv, device=None, coef=None, dtype=f64):
    """[Tv, Tp] float64 interpolation weights from lerp_coef (or the given coefficients)."""
    i0, i1, w0, w1 = lerp_coef(Tp, Tv, device, dtype) if coef is None else coef
    W = torch.zeros(Tv, Tp, dtype=f64, device=i0.device)
    rows = torch.arange(Tv, device=i0.device)
    W.index_put_((rows, i0), w0, accumulate=True)
    W.index_put_((rows, i1), w1, accumulate=True)
    return W


def nearest_index(Tp, Tv, device=None):
    """[Tv] source frame of ATen's upsample_nearest1d: min(floor(t * float(Tp / Tv)), Tp - 1) in float32 arithmetic."""
    t = torch.arange(Tv, device=device)
    if Tp == Tv:
        return t
    scale = torch.tensor(Tp, dtype=torch.float32) / torch.tensor(Tv, dtype=torch.float32)
    return torch.clamp(torch.floor(t.to(torch.float32) * scale.to(t.device)).long(), max=Tp - 1)


def _pad(audio, src, cnt, Tp):
    """[B, Tp, D] float64: each sample's speech frames in order, zero past cnt[b]."""
    B, Ta, D = audio.shape
    a = torch.gather(audio.to(f64), 1, src[:, :Tp, None].expand(B, Tp, D))
    keep = torch.arange(Tp, device=audio.device)[None, :] < cnt[:, None]
    return a * keep[:, :, None]


def resample_forward(audio, mask, Tv, W=None, coef_dtype=f64):
    """audio [B, Ta, D], mask [B, Ta] int64 -> (out [B, Tv, D] float64, mask_out [B, Tv] int64, input_lengths [B]).
    A batch without any speech frame gives zeros.  coef_dtype: see lerp_coef; W overrides the interpolation matrix
    (mutation tests)."""
    B, Ta, D = audio.shape
    src, cnt = speech_index(mask)
    Tp = int(cnt.max())
    if Tp == 0:
        z = torch.zeros(B, Tv, dtype=torch.int64, device=audio.device)
        return torch.zeros(B, Tv, D, dtype=f64, device=audio.device), z, z.sum(1)
    a = _pad(audio, src, cnt, Tp)
    m = torch.gather(mask, 1, src[:, :Tp]) * (torch.arange(Tp, device=mask.device)[None, :] < cnt[:, None])
    out = (lerp_matrix(Tp, Tv, audio.device, dtype=coef_dtype) if W is None else W) @ a
    mask_out = m[:, nearest_index(Tp, Tv, mask.device)]
    return out, mask_out, (mask_out != 0).sum(1)


def resample_backward(dout, mask, W=None, coef_dtype=f64):
    """dout [B, Tv, D] -> d_audio [B, Ta, D] float64: (W^T dout) scattered to each sample's speech frames, 0 elsewhere."""
    B, Tv, D = dout.shape
    Ta = mask.shape[1]
    src, cnt = speech_index(mask)
    Tp = int(cnt.max())
    da = torch.zeros(B, Ta, D, dtype=f64, device=dout.device)
    if Tp == 0:
        return da
    g = (lerp_matrix(Tp, Tv, dout.device, dtype=coef_dtype) if W is None else W).T @ dout.to(f64)
    keep = (torch.arange(Tp, device=dout.device)[None, :] < cnt[:, None]).to(f64)
    da.scatter_add_(1, src[:, :Tp, None].expand(B, Tp, D), g * keep[:, :, None])
    return da


# ----------------------------------------------------------------------------------------------------- softmax
def softmax_forward(S, T):
    """S [rows, Tp] -> P [rows, Tp] float64: softmax over the first T columns, pad columns 0."""
    s = S[:, :T].to(f64)
    P = torch.zeros(S.shape, dtype=f64, device=S.device)
    e = torch.exp(s - s.max(1, keepdim=True).values)
    P[:, :T] = e / e.sum(1, keepdim=True)
    return P


def softmax_backward(P, dP, T):
    """dS = P * (dP - sum_k dP * P) over the first T columns, pad columns 0.  P is the bf16 P of the forward."""
    p, dp = P[:, :T].to(f64), dP[:, :T].to(f64)
    dS = torch.zeros(P.shape, dtype=f64, device=P.device)
    dS[:, :T] = p * (dp - (p * dp).sum(1, keepdim=True))
    return dS


# ----------------------------------------------------------------------------------------------------- colsum
def colsum(X, N):
    """X [M, ld] -> [N] float64 sums of the first N columns."""
    return X[:, :N].to(f64).sum(0)


# ----------------------------------------------------------------------------------------------------- log_softmax
def log_softmax_forward(X):
    x = X.to(f64)
    m = x.max(1, keepdim=True).values
    return x - (m + torch.log(torch.exp(x - m).sum(1, keepdim=True)))


def log_softmax_backward(Y, dY):
    y, dy = Y.to(f64), dY.to(f64)
    return dy - torch.exp(y) * dy.sum(1, keepdim=True)


# ----------------------------------------------------------------------------------------------------- attention
def _heads(x, B, T, H):
    return x.to(f64).reshape(B, T, H, 128).transpose(1, 2)          # [B, H, T, 128]


def _merge(x):
    B, H, T, _ = x.shape
    return x.transpose(1, 2).reshape(B, T, H * 128)


def attention_forward(q, kv, H, round_bf16=True, key_mask=None):
    """q [B, T, E], kv [B, T, 2E] (keys | values), E = 128 H -> (o [B, T, E], lse2 [B*H, T] = log2 sum_j exp(s_ij)),
    s = q k^T / sqrt(128).  key_mask [T] bool drops the keys where it is False (mutation tests)."""
    B, T, E = q.shape
    qh, kh, vh = _heads(q, B, T, H), _heads(kv[..., :E], B, T, H), _heads(kv[..., E:], B, T, H)
    s = qh @ kh.transpose(-1, -2) / math.sqrt(128.0)
    if key_mask is not None:
        s = s.masked_fill(~key_mask, -math.inf)
    m = s.max(-1, keepdim=True).values
    e = torch.exp(s - m)
    l = e.sum(-1, keepdim=True)
    o = (_rbf(e, round_bf16) @ vh) / l
    lse2 = ((m + torch.log(l)) / LN2).reshape(B * H, T)
    return _rbf(_merge(o), round_bf16), lse2


def attention_backward(q, kv, dout, o, lse2, H, round_bf16=True, zero_D=False, key_mask=None):
    """-> (dq [B, T, E], dk [B, T, E], dv [B, T, E]).  o and lse2 are the forward's outputs (o as the kernel stores it).
    zero_D takes D = 0 and key_mask drops keys (mutation tests)."""
    B, T, E = q.shape
    rb = round_bf16
    qh, kh, vh = _heads(q, B, T, H), _heads(kv[..., :E], B, T, H), _heads(kv[..., E:], B, T, H)
    doh, oh = _heads(dout, B, T, H), _heads(o, B, T, H)
    alpha = 1.0 / math.sqrt(128.0)
    s = qh @ kh.transpose(-1, -2) * alpha
    if key_mask is not None:
        s = s.masked_fill(~key_mask, -math.inf)
    P = torch.exp(s - lse2.to(f64).reshape(B, H, T, 1) * LN2)
    dP = doh @ vh.transpose(-1, -2)
    D = torch.zeros_like(dP[..., :1]) if zero_D else (doh * oh).sum(-1, keepdim=True)
    dS = _rbf(P * (dP - D) * alpha, rb)
    dq = dS @ kh
    dk = dS.transpose(-1, -2) @ qh
    dv = _rbf(P, rb).transpose(-1, -2) @ doh
    return tuple(_rbf(_merge(x), rb) for x in (dq, dk, dv))


# ----------------------------------------------------------------------------------------------------- gemm
def gemm(A, Bm, alpha=1.0, bias=None, bias_mode=0, C0=None):
    """A [.., M, K], Bm [.., N, K] -> alpha * A . B^T (+ bias[n] for bias_mode 1, bias[m] for 2) (+ C0)."""
    C = alpha * (A.to(f64) @ Bm.to(f64).transpose(-1, -2))
    M, N = C.shape[-2:]
    if bias_mode == 1:
        C = C + bias[:N].to(f64)
    elif bias_mode == 2:
        C = C + bias[:M].to(f64)[:, None]
    if C0 is not None:
        C = C + C0.to(f64)
    return C
