"""float64 restatement of the two halves of Wav2Vec2EncoderLayerStableLayerNorm that csrc/wav2vec2_layer.cu runs around
torch's attention core, forward and backward written out step by step (no autograd), on plain torch ops.

  attn_in      : ln1 = LN(x); q, k, v = ln1 . W^T + b                (W = [Wq; Wk; Wv], [3E, E])
  attn_out_ffn : h = x + drop_h(attn . Wo^T + bo)
                 y = h + drop_o(drop_a(gelu(LN(h) . W1^T + b1)) . W2^T + b2)

Rows are flattened: x, attn, dy are [M, E].  With ``round_bf16=True`` every value the bf16-autocast module path
materialises in bf16 is rounded to bf16 at the same point (LayerNorm outputs, Linear outputs, the GELU output, dropout
outputs, residual sums, every bf16 input gradient); the parameter gradients stay unrounded, as the library writes them
in fp32.  With ``round_bf16=False`` everything is float64.

Dropout masks come from the caller (0/1 tensors, or None for no dropout).  They are applied as ATen does: forward
``v * (1 / keep)`` with keep = 1 - p as float, backward ``g * 1 / (1 - p)``.

TEST INFRASTRUCTURE ONLY: nothing in the package imports this module."""
from __future__ import annotations

import math

import torch

f64 = torch.float64


def _rbf(t, on):
    return t.to(torch.bfloat16).to(f64) if on else t


def _fwd_scale(p, round_bf16):
    """native_dropout's forward scale: 1 / keep with keep = 1 - p in float (fp32) on the bf16 path."""
    if not round_bf16:
        return 1.0 / (1.0 - p)
    keep = float(torch.tensor(1.0 - p, dtype=torch.float32))
    return float(torch.tensor(1.0 / keep, dtype=torch.float32))


def _bwd_scale(p, round_bf16):
    s = 1.0 / (1.0 - p)
    return float(torch.tensor(s, dtype=torch.float32)) if round_bf16 else s


def _drop(v, mask, scale, rb):
    if mask is None:
        return v
    return _rbf(v * mask.to(f64) * scale, rb)


def _ln_fwd(x, w, b, eps):
    mean = x.mean(-1, keepdim=True)
    var = (x - mean).pow(2).mean(-1, keepdim=True)
    rstd = 1.0 / torch.sqrt(var + eps)
    xhat = (x - mean) * rstd
    return xhat * w + b, xhat, rstd


def _ln_bwd(dy, xhat, rstd, w):
    """d LN / d x for incoming dy, and the per-column weight and bias gradients."""
    gy = dy * w
    s1 = gy.mean(-1, keepdim=True)
    s2 = (gy * xhat).mean(-1, keepdim=True)
    dx = rstd * (gy - s1 - xhat * s2)
    return dx, (dy * xhat).sum(0), dy.sum(0)


def gelu(x):
    return 0.5 * x * (1.0 + torch.erf(x / math.sqrt(2.0)))


def gelu_grad(x):
    return 0.5 * (1.0 + torch.erf(x / math.sqrt(2.0))) + x * torch.exp(-0.5 * x * x) / math.sqrt(2.0 * math.pi)


def attn_in_forward(x, ln_w, ln_b, eps, wqkv, bqkv, round_bf16=True):
    """-> (q, k, v, saved).  x [M, E]; wqkv [3E, E]; bqkv [3E]."""
    rb = round_bf16
    x, ln_w, ln_b, wqkv, bqkv = (t.to(f64) for t in (x, ln_w, ln_b, wqkv, bqkv))
    E = x.shape[1]
    ln, xhat, rstd = _ln_fwd(x, ln_w, ln_b, eps)
    ln = _rbf(ln, rb)
    qkv = _rbf(ln @ wqkv.T + bqkv, rb)
    saved = dict(round_bf16=rb, ln=ln, xhat=xhat, rstd=rstd, ln_w=ln_w, wqkv=wqkv)
    return qkv[:, :E], qkv[:, E:2 * E], qkv[:, 2 * E:], saved


def attn_in_backward(dq, dk, dv, saved):
    """-> dict(dx, g_wqkv, g_bqkv, g_lnw, g_lnb, and the intermediates dqkv, dln)."""
    rb = saved["round_bf16"]
    dqkv = torch.cat([t.to(f64) for t in (dq, dk, dv)], 1)
    dln = _rbf(dqkv @ saved["wqkv"], rb)
    dxn, g_lnw, g_lnb = _ln_bwd(dln, saved["xhat"], saved["rstd"], saved["ln_w"])
    return dict(dx=_rbf(dxn, rb), g_wqkv=dqkv.T @ saved["ln"], g_bqkv=dqkv.sum(0), g_lnw=g_lnw, g_lnb=g_lnb,
                dqkv=dqkv, dln=dln)


def attn_out_ffn_forward(attn, x, wo, bo, ln_w, ln_b, eps, w1, b1, w2, b2, masks=(None, None, None),
                         probs=(0.0, 0.0, 0.0), round_bf16=True):
    """-> (y, saved).  attn, x [M, E]; w1 [F, E]; w2 [E, F]; masks = (hidden [M, E], intermediate [M, F],
    output [M, E]) 0/1 tensors or None; probs = their dropout probabilities."""
    rb = round_bf16
    attn, x, wo, bo, ln_w, ln_b, w1, b1, w2, b2 = (t.to(f64) for t in (attn, x, wo, bo, ln_w, ln_b, w1, b1, w2, b2))
    sc = [_fwd_scale(p, rb) for p in probs]
    ao = _rbf(attn @ wo.T + bo, rb)
    h = _rbf(x + _drop(ao, masks[0], sc[0], rb), rb)
    ln, xhat, rstd = _ln_fwd(h, ln_w, ln_b, eps)
    ln = _rbf(ln, rb)
    pre = _rbf(ln @ w1.T + b1, rb)
    act = _drop(_rbf(gelu(pre), rb), masks[1], sc[1], rb)
    z = _rbf(act @ w2.T + b2, rb)
    y = _rbf(h + _drop(z, masks[2], sc[2], rb), rb)
    saved = dict(round_bf16=rb, masks=masks, probs=probs, attn=attn, ln=ln, xhat=xhat, rstd=rstd, ln_w=ln_w, pre=pre,
                 act=act, wo=wo, w1=w1, w2=w2)
    return y, saved


def attn_out_ffn_backward(dy, saved):
    """-> dict(dattn, dx, g_wo, g_bo, g_lnw, g_lnb, g_w1, g_b1, g_w2, g_b2, and the intermediates dz, dpre, dln, dh,
    dzo: the gradients of the output dropout's input, of the intermediate Linear's output, of the final LayerNorm's
    output, of h, and of the hidden dropout's input)."""
    rb = saved["round_bf16"]
    masks = saved["masks"]
    sc = [_bwd_scale(p, rb) for p in saved["probs"]]
    dy = dy.to(f64)
    dz = _drop(dy, masks[2], sc[2], rb)
    da = _drop(_rbf(dz @ saved["w2"], rb), masks[1], sc[1], rb)
    dpre = _rbf(gelu_grad(saved["pre"]) * da, rb)
    dln = _rbf(dpre @ saved["w1"], rb)
    dxn, g_lnw, g_lnb = _ln_bwd(dln, saved["xhat"], saved["rstd"], saved["ln_w"])
    dh = _rbf(dy + _rbf(dxn, rb), rb)
    dzo = _drop(dh, masks[0], sc[0], rb)
    dattn = _rbf(dzo @ saved["wo"], rb)
    return dict(dattn=dattn, dx=dh, g_wo=dzo.T @ saved["attn"], g_bo=dzo.sum(0), g_lnw=g_lnw, g_lnb=g_lnb,
                g_w1=dpre.T @ saved["ln"], g_b1=dpre.sum(0), g_w2=dz.T @ saved["act"], g_b2=dz.sum(0),
                dz=dz, dpre=dpre, dln=dln, dh=dh, dzo=dzo)
