"""CPU: oracle/w2v_oracle.py (round_bf16=False) is HF's Wav2Vec2EncoderLayerStableLayerNorm in float64.  The oracle's
attn_in -> SDPA -> attn_out_ffn chain, with its hand-written backward, must give the module's output and, against
autograd through the module, the input gradient and all sixteen parameter gradients, in eval mode and in train mode
with the three dropouts replaced by fixed masks (which checks where each dropout sits)."""
import pytest
import torch
import torch.nn.functional as F

from oracle import w2v_oracle as wo

f64 = torch.float64


class _MaskDrop(torch.nn.Module):
    """nn.Dropout with a fixed mask: x * mask / (1 - p)."""

    def __init__(self, mask, p):
        super().__init__()
        self.mask, self.p = mask, p

    def forward(self, x):
        return x * self.mask.view_as(x) / (1.0 - self.p)


def _layer(E, F_, seed):
    from transformers.models.wav2vec2.modeling_wav2vec2 import Wav2Vec2EncoderLayerStableLayerNorm
    from multimodal_av_model_b200.encoders import xlsr_large_config
    cfg = xlsr_large_config(hidden_size=E, intermediate_size=F_, num_attention_heads=E // 64, attention_dropout=0.0)
    cfg._attn_implementation = "sdpa"
    torch.manual_seed(seed)
    layer = Wav2Vec2EncoderLayerStableLayerNorm(cfg).to(f64)
    with torch.no_grad():                                   # non-trivial LayerNorm affine parameters
        for ln in (layer.layer_norm, layer.final_layer_norm):
            ln.weight.uniform_(0.5, 1.5)
            ln.bias.uniform_(-0.2, 0.2)
    return layer


def _oracle_layer(layer, x, mask4d, dy, masks, probs):
    """The oracle chain around float64 SDPA -> (y, dx, {parameter name: gradient})."""
    a, ff = layer.attention, layer.feed_forward
    ln1, ln2 = layer.layer_norm, layer.final_layer_norm
    B, T, E = x.shape
    M, H = B * T, a.num_heads
    xm = x.reshape(M, E)
    wqkv = torch.cat([a.q_proj.weight, a.k_proj.weight, a.v_proj.weight]).detach()
    bqkv = torch.cat([a.q_proj.bias, a.k_proj.bias, a.v_proj.bias]).detach()
    q, k, v, s_in = wo.attn_in_forward(xm, ln1.weight.detach(), ln1.bias.detach(), ln1.eps, wqkv, bqkv, round_bf16=False)
    q4, k4, v4 = (t.reshape(B, T, H, -1).transpose(1, 2).requires_grad_() for t in (q, k, v))
    o = F.scaled_dot_product_attention(q4, k4, v4, attn_mask=mask4d, scale=a.scaling)
    attn = o.transpose(1, 2).reshape(M, E)
    lin = lambda m: (m.weight.detach(), m.bias.detach())
    y, s_out = wo.attn_out_ffn_forward(attn.detach(), xm, *lin(a.out_proj), ln2.weight.detach(), ln2.bias.detach(),
                                       ln2.eps, *lin(ff.intermediate_dense), *lin(ff.output_dense), masks=masks,
                                       probs=probs, round_bf16=False)
    g_out = wo.attn_out_ffn_backward(dy.reshape(M, E), s_out)
    dq, dk, dv = torch.autograd.grad(attn, (q4, k4, v4), g_out["dattn"])
    g_in = wo.attn_in_backward(*(t.transpose(1, 2).reshape(M, E) for t in (dq, dk, dv)), s_in)
    gw, gb = g_in["g_wqkv"], g_in["g_bqkv"]
    grads = {"attention.q_proj.weight": gw[:E], "attention.q_proj.bias": gb[:E],
             "attention.k_proj.weight": gw[E:2 * E], "attention.k_proj.bias": gb[E:2 * E],
             "attention.v_proj.weight": gw[2 * E:], "attention.v_proj.bias": gb[2 * E:],
             "attention.out_proj.weight": g_out["g_wo"], "attention.out_proj.bias": g_out["g_bo"],
             "layer_norm.weight": g_in["g_lnw"], "layer_norm.bias": g_in["g_lnb"],
             "final_layer_norm.weight": g_out["g_lnw"], "final_layer_norm.bias": g_out["g_lnb"],
             "feed_forward.intermediate_dense.weight": g_out["g_w1"], "feed_forward.intermediate_dense.bias": g_out["g_b1"],
             "feed_forward.output_dense.weight": g_out["g_w2"], "feed_forward.output_dense.bias": g_out["g_b2"]}
    return y.reshape(B, T, E), (g_in["dx"] + g_out["dx"]).reshape(B, T, E), grads


def _close(a, b, what):
    """float64 agreement: ~1e-10 of the reference's scale (the key bias gradient is zero up to rounding)."""
    scale = max(b.abs().max().item(), 1.0)
    err = (a - b).abs().max().item()
    assert err <= 1e-10 * scale, (what, err, scale)


def _inputs(B, T, E, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B, T, E, generator=g, dtype=f64)
    lens = torch.tensor([T, T - 5, 3][:B])
    valid = torch.arange(T)[None, :] < lens[:, None]
    x = x.masked_fill(~valid[..., None], 0)                 # padded frames are 0, as upstream
    x[0, 1] = 50 + 0.1 * x[0, 1]                            # a row with a large offset
    mask4d = valid[:, None, None, :].expand(B, 1, T, T)
    dy = torch.randn(B, T, E, generator=g, dtype=f64)
    return x, mask4d, dy


@pytest.mark.parametrize("E,F_", [(256, 1024), (768, 3072)])
@pytest.mark.parametrize("train", [False, True])
def test_oracle_is_the_module(E, F_, train):
    B, T = 3, 16
    layer = _layer(E, F_, seed=E + train)
    x, mask4d, dy = _inputs(B, T, E, seed=E)
    masks, probs = (None, None, None), (0.0, 0.0, 0.0)
    if train:
        layer.train()
        g = torch.Generator().manual_seed(7)
        probs = (0.1, 0.3, 0.2)                              # three different p, so a swapped scale shows
        masks = tuple((torch.rand(B * T, n, generator=g) >= p).to(f64) for n, p in zip((E, F_, E), probs))
        ff = layer.feed_forward
        layer.dropout = _MaskDrop(masks[0], probs[0])
        ff.intermediate_dropout = _MaskDrop(masks[1], probs[1])
        ff.output_dropout = _MaskDrop(masks[2], probs[2])
    else:
        layer.eval()
    y, dx, grads = _oracle_layer(layer, x, mask4d, dy, masks, probs)
    xr = x.clone().requires_grad_()
    z = layer(xr, attention_mask=mask4d)[0]
    z.backward(dy)
    _close(y, z.detach(), "y")
    _close(dx, xr.grad, "dx")
    ref = {n: p.grad for n, p in layer.named_parameters()}
    assert sorted(ref) == sorted(grads)
    for n in ref:
        _close(grads[n], ref[n], n)
    if train:   # the masks matter: without them the oracle is far from the module
        y0, _, _ = _oracle_layer(layer, x, mask4d, dy, (None, masks[1], masks[2]), probs)
        assert (y0 - z.detach()).abs().max().item() > 1e-3


@pytest.mark.parametrize("p", [0.0, 0.1])
def test_oracle_bf16_rounding_is_on_the_grid(p):
    """round_bf16=True: every tensor the module path materialises in bf16 is exactly representable in bf16, and the
    result stays within bf16 rounding of the float64 one."""
    M, E, F_ = 40, 256, 264
    g = torch.Generator().manual_seed(3)
    r = lambda *s: torch.randn(*s, generator=g, dtype=f64)
    x, attn, dy = (r(M, E).to(torch.bfloat16).to(f64) for _ in range(3))     # the kernels' inputs are bf16
    lnw, lnb = 1 + 0.2 * r(E), 0.1 * r(E)
    w = dict(wo=r(E, E) / 16, bo=0.1 * r(E), w1=r(F_, E) / 16, b1=0.1 * r(F_), w2=r(E, F_) / 16, b2=0.1 * r(E))
    masks = tuple((torch.rand(M, n, generator=g) >= p).to(f64) if p else None for n in (E, F_, E))
    out = {}
    for rb in (True, False):
        y, s = wo.attn_out_ffn_forward(attn, x, w["wo"], w["bo"], lnw, lnb, 1e-5, w["w1"], w["b1"], w["w2"], w["b2"],
                                       masks=masks, probs=(p, p, p), round_bf16=rb)
        out[rb] = dict(y=y, ln=s["ln"], pre=s["pre"], act=s["act"], **wo.attn_out_ffn_backward(dy, s))
    on_grid = lambda t: torch.equal(t, t.to(torch.bfloat16).to(f64))
    for n in ("y", "ln", "pre", "act", "dattn", "dx", "dz", "dpre", "dln", "dzo"):
        assert on_grid(out[True][n]), n
        assert n == "dz" and not p or not on_grid(out[False][n]), n       # without dropout, dz is dy itself
        rel = ((out[True][n] - out[False][n]).norm() / out[False][n].norm()).item()
        assert rel < 2e-2, (n, rel)
