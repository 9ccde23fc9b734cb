"""GPU: the native wav2vec2 encoder layer (csrc/wav2vec2_layer.cu around torch's attention interface) against HF's module
path on the same GPU, same weights, same CUDA generator state: dropout draws identical to ATen's native_dropout, outputs
and gradients within bf16 rounding, the generator offset advanced exactly as the module path advances it, eval mode,
bit-identical repeats, and the cases that must stay on the module path."""
import copy

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

B, T = 8, 249


def _enc():
    from multimodal_av_model_b200 import encoders
    return encoders


def _gen():
    return torch.cuda.default_generators[torch.cuda.current_device()]


def _layer(seed=0, trainable=True, train=True, **cfg_overrides):
    from transformers.models.wav2vec2.modeling_wav2vec2 import Wav2Vec2EncoderLayerStableLayerNorm
    from multimodal_av_model_b200.encoders import xlsr_large_config
    cfg = xlsr_large_config(**cfg_overrides)
    cfg._attn_implementation = "sdpa"
    torch.manual_seed(seed)
    layer = Wav2Vec2EncoderLayerStableLayerNorm(cfg).cuda()
    with torch.no_grad():                                   # non-trivial LayerNorm affine parameters
        for ln in (layer.layer_norm, layer.final_layer_norm):
            ln.weight.uniform_(0.5, 1.5)
            ln.bias.uniform_(-0.2, 0.2)
    layer.requires_grad_(trainable)
    return layer.train(train)


def _inputs(seed=1, e=1024):
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randn(B, T, e, device="cuda", generator=g).to(torch.bfloat16)
    lens = torch.tensor([249, 200, 131, 249, 17, 90, 248, 160])
    m = torch.arange(T)[None, :] < lens[:, None]
    x = x.masked_fill(~m.cuda()[..., None], 0)                                   # padded frames are 0, as upstream
    mask4d = m.cuda()[:, None, None, :].expand(B, 1, T, T)
    return x, mask4d


def _run(layer, x, mask4d, native, seed=5):
    torch.manual_seed(seed)
    x = x.detach().clone().requires_grad_()
    with torch.autocast("cuda", dtype=torch.bfloat16):
        if native:
            assert _enc()._w2v_native_applies(layer, x)
            y = _enc()._w2v_native_layer(layer, x, mask4d)
        else:
            y = layer(x, attention_mask=mask4d, output_attentions=False)[0]
    offset = _gen().get_offset()
    r = torch.randn(y.shape, device="cuda", generator=torch.Generator(device="cuda").manual_seed(9))
    (y.float() * r).sum().backward()
    grads = {n: p.grad.clone() for n, p in layer.named_parameters() if p.grad is not None}
    layer.zero_grad(set_to_none=True)
    return y.detach(), offset, x.grad, grads


def _grads_close(g, g_ref, rel):
    """Parameter gradients within bf16 rounding.  The key projection's bias has a true gradient of exactly zero (the
    same shift of every key's score leaves softmax unchanged); both paths return rounding noise there, so the native
    one is only held to the module path's noise level."""
    assert sorted(g) == sorted(g_ref)
    for n in g_ref:
        if n.endswith("k_proj.bias"):
            assert g[n].norm().item() <= 2 * g_ref[n].norm().item() + 1e-6, (n, g[n].norm().item(), g_ref[n].norm().item())
        else:
            _close(g[n], g_ref[n], n, rel=rel)


def _close(y, z, what, rel=2e-2):
    """Within bf16 rounding: a small relative error overall, no element off by more than a few percent of the tensor's
    scale, and (what a wrong dropout mask would break) almost no element off by more than a tenth of the RMS."""
    y, z = y.float(), z.float()
    d = (y - z).abs()
    rms = z.pow(2).mean().sqrt().item()
    assert (d.norm() / z.norm()).item() <= rel, (what, (d.norm() / z.norm()).item())
    assert d.max().item() <= 0.05 * z.abs().max().item() + 1e-6, (what, d.max().item(), z.abs().max().item())
    assert (d > 0.1 * rms).float().mean().item() <= 1e-3, (what, (d > 0.1 * rms).float().mean().item())


@pytest.mark.parametrize("n", [1992 * 1024, 1992 * 4096, 8 * 1000, 4096])
def test_dropout_draws_equal_aten_native_dropout(n):
    from multimodal_av_model_b200 import _lib
    L = _lib.lib()
    x = torch.randn(n, device="cuda").to(torch.bfloat16)
    torch.manual_seed(3)
    gen = _gen()
    seed, off = gen.initial_seed(), gen.get_offset()
    ref, _ = torch.native_dropout(x, 0.1, True)
    incr = gen.get_offset() - off
    y = torch.empty_like(x)
    _lib.check(L.avctc_w2v_dropout(x.data_ptr(), n, 0.1, seed, off, y.data_ptr(), _lib.stream_ptr(x.device)),
               "avctc_w2v_dropout")
    assert torch.equal(y, ref)
    if n % 1024 == 0:                 # the offset the library reserves for a dropout over n = M*E elements
        assert L.avctc_w2v_dropout_increment(n // 1024, 1024, 8, 0.1, 0.0, 0.0, 1) == incr


@pytest.mark.parametrize("trainable", [False, True])
def test_native_layer_matches_module_path_train(trainable):
    layer = _layer(trainable=trainable)
    x, mask4d = _inputs()
    y, off, dx, g = _run(layer, x, mask4d, native=True)
    z, off_ref, dx_ref, g_ref = _run(layer, x, mask4d, native=False)
    assert off == off_ref
    _close(y, z, "y", rel=1e-2)
    _close(dx, dx_ref, "dx")
    assert (len(g) == 16) == trainable
    _grads_close(g, g_ref, 3e-2)


def test_native_layer_matches_module_path_train_768():
    """A 768-wide layer (a base model's width) takes the native path too: three 256-column chunks per LayerNorm row."""
    layer = _layer(7, hidden_size=768, intermediate_size=3072, num_attention_heads=12)
    x, mask4d = _inputs(7, e=768)
    y, off, dx, g = _run(layer, x, mask4d, native=True)
    z, off_ref, dx_ref, g_ref = _run(layer, x, mask4d, native=False)
    assert off == off_ref
    _close(y, z, "y", rel=1e-2)
    _close(dx, dx_ref, "dx")
    assert len(g) == 16
    _grads_close(g, g_ref, 3e-2)


def test_native_layer_follows_fused_adam_steps():
    """Adam(fused=True), the trainer's optimizer on CUDA, updates the weights without advancing their version counters;
    the native path's bf16 weight copies must still follow every step."""
    layer = _layer(6, trainable=True)
    x, mask4d = _inputs(6)
    opt = torch.optim.Adam(layer.parameters(), lr=1e-2, fused=True)
    for _ in range(2):
        _, _, _, g = _run(layer, x, mask4d, native=True)
        for n, p in layer.named_parameters():
            p.grad = g[n]
        opt.step()
        opt.zero_grad(set_to_none=True)
    layer.eval()
    y, _, _, _ = _run(layer, x, mask4d, native=True)
    z, _, _, _ = _run(layer, x, mask4d, native=False)
    _close(y, z, "y after two optimizer steps", rel=1e-2)


def test_native_layer_matches_module_path_eval():
    layer = _layer(trainable=False, train=False)
    x, mask4d = _inputs(2)
    y, off, dx, _ = _run(layer, x, mask4d, native=True)
    z, off_ref, dx_ref, _ = _run(layer, x, mask4d, native=False)
    assert off == off_ref
    _close(y, z, "y", rel=1e-2)
    _close(dx, dx_ref, "dx")


def test_native_layer_forward_is_bit_identical_from_equal_states():
    layer = _layer(3)
    x, mask4d = _inputs(3)
    outs = []
    for _ in range(2):
        torch.manual_seed(11)
        with torch.autocast("cuda", dtype=torch.bfloat16):
            outs.append(_enc()._w2v_native_layer(layer, x, mask4d))
    assert torch.equal(outs[0], outs[1])


def test_native_path_not_taken_under_capture_in_fp32_or_on_cpu():
    enc = _enc()
    layer = _layer(4, trainable=False)
    x, _ = _inputs(4)
    with torch.autocast("cuda", dtype=torch.bfloat16):
        assert enc._w2v_native_applies(layer, x)
        assert not enc._w2v_native_applies(layer, x.float())
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        graph, seen = torch.cuda.CUDAGraph(), []
        with torch.cuda.stream(s):
            with torch.cuda.graph(graph, stream=s):
                seen.append(enc._w2v_native_applies(layer, x))
                x.add(1)
        torch.cuda.current_stream().wait_stream(s)
        assert seen == [False]
    assert not enc._w2v_native_applies(layer, x)                       # no autocast
    cpu = copy.deepcopy(layer).cpu()
    with torch.autocast("cpu", dtype=torch.bfloat16):
        assert not enc._w2v_native_applies(cpu, x.cpu())


def _audio_run(aud, wav, mask, lens, native, monkeypatch):
    enc = _enc()
    with monkeypatch.context() as mp:
        if not native:
            mp.setattr(enc, "_w2v_native_applies", lambda layer, hidden: False)
        from multimodal_av_model_b200 import _lib
        c0 = _lib.launch_count
        np.random.seed(21)
        torch.manual_seed(21)
        aud.begin_step()
        with torch.autocast("cuda", dtype=torch.bfloat16):
            last, middle = aud(wav, attention_mask=mask, host_lengths=lens)
        launched = _lib.launch_count - c0
    offset = _gen().get_offset()
    g = torch.Generator(device="cuda").manual_seed(5)
    loss = (last.float() * torch.randn(last.shape, device="cuda", generator=g)).sum() \
        + (middle.float() * torch.randn(middle.shape, device="cuda", generator=g)).sum()
    loss.backward()
    grads = {n: p.grad.clone() for n, p in aud.named_parameters() if p.grad is not None}
    aud.zero_grad(set_to_none=True)
    return last.detach(), middle.detach(), offset, grads, launched


def test_audio_encoder_native_matches_module_path_train(monkeypatch):
    """Full AudioEncoder, train mode (SpecAugment and LayerDrop active, seeded), layers 6-9 trainable, ragged masks.
    Each path runs on its own copy, so that both meet the graphed layers 0-5 in the same capture state."""
    import multimodal_av_model_b200 as pkg
    from multimodal_av_model_b200.encoders import unfreeze_middle_layers, xlsr_large_config
    torch.manual_seed(0)
    aud = pkg.AudioEncoder(freeze=True, config=xlsr_large_config()).cuda().train()
    unfreeze_middle_layers(aud.model)
    n = 32000
    wav = torch.randn(4, n, device="cuda")
    lens = torch.tensor([n, 25000, 12000, 31000])
    mask = (torch.arange(n)[None, :] < lens[:, None]).long().cuda()
    ref = copy.deepcopy(aud)
    a = _audio_run(aud, wav, mask, lens, True, monkeypatch)
    b = _audio_run(ref, wav, mask, lens, False, monkeypatch)
    assert a[4] > b[4]                                                  # the library's layer kernels ran
    assert a[2] == b[2]                                                 # generator offset
    _close(a[0], b[0], "last_hidden_state", rel=3e-2)
    _close(a[1], b[1], "middle", rel=3e-2)
    assert len(a[3]) == 4 * 16
    _grads_close(a[3], b[3], 6e-2)
