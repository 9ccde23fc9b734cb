"""Producers that feed the hot path: VisualEncoder and AudioEncoder (SURVEY.md §8 row a15).

The third-party wav2vec2 stays HF/PyTorch.  The frozen visual encoder's bf16-autocast forward on CUDA runs on this
library's kernels (csrc/visual_encoder.cu: front end, BatchNorm, PReLU, residual and pooling passes) around cuDNN's trunk
convolutions; its module path is the CPU path and the reference the tests compare against.  Module and
parameter names follow /root/reference/model/encoder.py:6-100 so reference checkpoints load unchanged
(`frontend3D.*`, `trunk.layer{1..4}.*`, `model.*`).
"""
from __future__ import annotations

import torch
import torch.nn as nn


def _act(kind, channels):
    return nn.PReLU(channels) if kind == "prelu" else nn.ReLU(inplace=True)


class BasicBlock(nn.Module):
    """3x3-3x3 residual block with a per-channel PReLU (encoder.py:6-22)."""

    def __init__(self, inplanes, planes, stride=1, downsample=None, relu_type="prelu"):
        super().__init__()
        self.conv1 = nn.Conv2d(inplanes, planes, kernel_size=3, stride=stride, padding=1, bias=False)
        self.bn1 = nn.BatchNorm2d(planes)
        self.relu = _act(relu_type, planes)
        self.conv2 = nn.Conv2d(planes, planes, kernel_size=3, stride=1, padding=1, bias=False)
        self.bn2 = nn.BatchNorm2d(planes)
        self.downsample = downsample

    def forward(self, x):
        skip = x if self.downsample is None else self.downsample(x)
        y = self.bn2(self.conv2(self.relu(self.bn1(self.conv1(x)))))
        return self.relu(y + skip)


class ResNet(nn.Module):
    """ResNet trunk without stem: four stages of `layers[i]` blocks, widths 64/128/256/512 (encoder.py:24-53)."""

    def __init__(self, block, layers, relu_type="prelu"):
        super().__init__()
        self.inplanes = 64
        widths, strides = (64, 128, 256, 512), (1, 2, 2, 2)
        for i, (w, s, n) in enumerate(zip(widths, strides, layers), start=1):
            setattr(self, f"layer{i}", self._stage(block, w, n, s, relu_type))
        self.avgpool = nn.AdaptiveAvgPool2d((1, 1))

    def _stage(self, block, planes, blocks, stride, relu_type):
        down = None
        if stride != 1 or self.inplanes != planes:
            down = nn.Sequential(nn.Conv2d(self.inplanes, planes, kernel_size=1, stride=stride, bias=False),
                                 nn.BatchNorm2d(planes))
        mods = [block(self.inplanes, planes, stride, down, relu_type)]
        self.inplanes = planes
        mods += [block(planes, planes, relu_type=relu_type) for _ in range(blocks - 1)]
        return nn.Sequential(*mods)

    def forward(self, x):
        for i in range(1, 5):
            x = getattr(self, f"layer{i}")(x)
        return torch.flatten(self.avgpool(x), 1)


class VisualEncoder(nn.Module):
    """[B,1,T,96,96] -> [B,T,512]: Conv3d(1->64,(5,7,7),s(1,2,2)) + BN + PReLU + MaxPool3d, then a per-frame
    ResNet-18 trunk (encoder.py:57-75)."""

    def __init__(self, relu_type="prelu"):
        super().__init__()
        self.frontend3D = nn.Sequential(
            nn.Conv3d(1, 64, kernel_size=(5, 7, 7), stride=(1, 2, 2), padding=(2, 3, 3), bias=False),
            nn.BatchNorm3d(64),
            _act(relu_type, 64),
            nn.MaxPool3d(kernel_size=(1, 3, 3), stride=(1, 2, 2), padding=(0, 1, 1)))
        self.trunk = ResNet(BasicBlock, [2, 2, 2, 2], relu_type=relu_type)
        self.output_dim = 512

    def _channels_last(self):
        """cuDNN's NHWC tensor-core kernels and ATen's channels-last BatchNorm are ~2x faster here than NCHW on B200
        (measured: 20.4 -> 10.8 ms per [8,1,150,96,96] call); values are unchanged up to bf16 rounding."""
        if not getattr(self, "_cl_done", False):
            self.trunk.to(memory_format=torch.channels_last)
            self._cl_done = True

    def _frontend_as_2d(self, x):
        """frontend3D (encoder.py:57-62) evaluated frame-wise with 2-D kernels, same parameters and same arithmetic:
        a (5,7,7) Conv3d over ONE input channel with stride (1,2,2) is a 7x7 Conv2d whose 5 input channels are the
        temporal taps t-2..t+2 (zero padded); BatchNorm3d over (B,T,H,W) equals BatchNorm2d over (B*T,H,W);
        MaxPool3d((1,3,3)) is MaxPool2d(3) per frame.  cuDNN has bf16 tensor-core kernels for the 2-D form (the 3-D
        form falls back to a TF32 kernel plus layout conversions) and the [B,64,T,H,W] -> [B*T,64,H,W] transpose copy
        disappears.  Returns [B*T,64,H',W'] channels-last."""
        import torch.nn.functional as F
        conv, bn, act, pool = self.frontend3D[0], self.frontend3D[1], self.frontend3D[2], self.frontend3D[3]
        b, _, t, h, w = x.shape
        kt = conv.kernel_size[0]
        pt = conv.padding[0]
        xp = F.pad(x[:, 0], (0, 0, 0, 0, pt, pt))                                   # [B, T+2pt, H, W]
        taps = xp.unfold(1, kt, 1)                                                    # [B, T, H, W, kt] (view)
        taps = taps.permute(0, 1, 4, 2, 3).reshape(b * t, kt, h, w)                   # temporal taps as channels
        taps = taps.contiguous(memory_format=torch.channels_last)
        w2 = conv.weight
        if not w2.requires_grad and torch.is_autocast_enabled(w2.device.type) and w2.dtype == torch.float32:
            key = (w2._version, w2.data_ptr(), torch.get_autocast_dtype(w2.device.type))
            if getattr(self, "_front_w", (None,))[0] != key:                          # frozen: cast once, not per step
                self._front_w = (key, w2.detach().to(key[2]))
            w2 = self._front_w[1]
        w2 = w2[:, 0]                                                                 # [64, kt, 7, 7]
        y = F.conv2d(taps, w2, None, stride=conv.stride[1:], padding=conv.padding[1:])
        if bn.training and bn.track_running_stats and bn.num_batches_tracked is not None:
            bn.num_batches_tracked.add_(1)
        y = F.batch_norm(y, bn.running_mean, bn.running_var, bn.weight, bn.bias,
                         bn.training or not bn.track_running_stats, bn.momentum if bn.momentum is not None else 0.1, bn.eps)
        y = act(y)
        return F.max_pool2d(y, pool.kernel_size[1:], pool.stride[1:], pool.padding[1:])

    def forward(self, x):
        # main.py:100-103 freezes every parameter of this encoder: for a fixed clip shape its forward is a fixed kernel
        # sequence whose output needs no gradient -> replayed from a CUDA graph (graphed.py), ~170 launches -> 1
        if x.is_cuda and x.shape[1] == 1:
            self._channels_last()
        seg = getattr(self, "_graph_seg", None)
        if seg is None:
            from .graphed import GraphedSegment
            seg = self._graph_seg = GraphedSegment(self._forward_impl, list(self.parameters()), list(self.buffers()),
                                                   modules=list(self.modules()))
        if seg.usable(x):
            return seg(x)
        return self._forward_impl(x)

    def _native_applies(self, x):
        """The frozen bf16-autocast forward on CUDA runs on this library's kernels (csrc/visual_encoder.cu) around
        cuDNN's trunk convolutions; everything else (CPU, fp32, ReLU variant, trainable weights, BatchNorm without
        running statistics) takes the module path, which is also the reference the native path is tested against."""
        if not (x.is_cuda and x.dim() == 5 and x.shape[1] == 1 and x.dtype == torch.float32
                and x.shape[0] * x.shape[2] <= 65535 and torch.is_autocast_enabled("cuda")
                and torch.get_autocast_dtype("cuda") == torch.bfloat16):
            return False
        if torch.is_grad_enabled() and x.requires_grad or any(p.requires_grad for p in self.parameters()):
            return False
        conv, pool = self.frontend3D[0], self.frontend3D[3]
        if ((conv.kernel_size, conv.stride, conv.padding, conv.dilation, conv.groups, conv.bias is None)
                != ((5, 7, 7), (1, 2, 2), (2, 3, 3), (1, 1, 1), 1, True)
                or (pool.kernel_size, pool.stride, pool.padding, pool.dilation) != ((1, 3, 3), (1, 2, 2), (0, 1, 1), 1)):
            return False
        for m in self.modules():
            if isinstance(m, nn.ReLU) or (isinstance(m, nn.modules.batchnorm._BatchNorm)
                                          and (not m.track_running_stats or m.momentum is None)):
                return False
        return True

    def _native_params(self):
        """bf16 copies the kernels read, made once per parameter version: the front-end weight as [64, 5*7*7] padded
        to K = 256, and every PReLU slope (the rounding autocast applies to them in the module path)."""
        params = list(self.parameters())
        key = tuple((p._version, p.data_ptr()) for p in params)
        hit = getattr(self, "_native_cache", None)
        if hit is None or hit[0] != key:
            w = self.frontend3D[0].weight.detach().to(torch.bfloat16).reshape(64, -1)
            w = torch.nn.functional.pad(w, (0, 256 - w.shape[1])).contiguous()
            slopes = {m: m.weight.detach().to(torch.bfloat16).contiguous() for m in self.modules()
                      if isinstance(m, nn.PReLU)}
            hit = self._native_cache = (key, {"front_w": w, "slopes": slopes})
        return hit[1]

    def _forward_native(self, x):
        from . import _lib
        L = _lib.lib()
        dev = x.device
        cl = torch.channels_last
        self._channels_last()
        prm = self._native_params()
        with _lib.device_guard(dev):
            st = _lib.stream_ptr(dev)
            tracked = []

            def scale_shift(bn, parts, p, c):
                ss = torch.empty(2 * c, device=dev, dtype=torch.float32)
                _lib.check(L.avctc_bn_finalize(
                    parts.data_ptr() if bn.training else None, p, c,
                    bn.weight.data_ptr() if bn.weight is not None else None,
                    bn.bias.data_ptr() if bn.bias is not None else None, bn.running_mean.data_ptr(),
                    bn.running_var.data_ptr(), float(bn.momentum), float(bn.eps), int(bn.training), ss.data_ptr(), st),
                    "avctc_bn_finalize")
                if bn.training:
                    tracked.append(bn.num_batches_tracked)
                return ss

            def conv_bn(conv, bn, inp):
                """cuDNN convolution (module call: channels-last bf16, cached weights), then its BatchNorm scale/shift."""
                y = conv(inp).contiguous(memory_format=cl)
                n, c, h, w = y.shape
                p = L.avctc_bn_stats_ctas(n * h * w, c)
                parts = None
                if bn.training:
                    parts = torch.empty(3 * c * p, device=dev, dtype=torch.float32)
                    _lib.check(L.avctc_bn_stats(y.data_ptr(), n * h * w, c, parts.data_ptr(), p, st), "avctc_bn_stats")
                return y, scale_shift(bn, parts, p, c)

            b, _, t, h, w = x.shape
            x = x.contiguous()
            ho, wo = (h - 1) // 2 + 1, (w - 1) // 2 + 1
            bn0 = self.frontend3D[1]
            p = L.avctc_visual_frontend_ctas(b, t, h, w)
            parts = torch.empty(3 * 64 * p, device=dev, dtype=torch.float32) if bn0.training else None
            y = torch.empty((b * t, ho, wo, 64), device=dev, dtype=torch.bfloat16)
            _lib.check(L.avctc_visual_frontend(x.data_ptr(), b, t, h, w, prm["front_w"].data_ptr(), y.data_ptr(),
                                               parts.data_ptr() if parts is not None else None, p, st),
                       "avctc_visual_frontend")
            ss = scale_shift(bn0, parts, p, 64)
            cur = torch.empty((b * t, (ho - 1) // 2 + 1, (wo - 1) // 2 + 1, 64), device=dev, dtype=torch.bfloat16)
            _lib.check(L.avctc_visual_frontend_pool(y.data_ptr(), b * t, ho, wo, ss.data_ptr(),
                                                    prm["slopes"][self.frontend3D[2]].data_ptr(), cur.data_ptr(), st),
                       "avctc_visual_frontend_pool")
            cur = cur.permute(0, 3, 1, 2)                                    # NCHW view of the NHWC tensor
            blocks = [blk for i in range(1, 5) for blk in getattr(self.trunk, f"layer{i}")]
            for blk in blocks:
                slope = prm["slopes"][blk.relu].data_ptr()
                y1, ss1 = conv_bn(blk.conv1, blk.bn1, cur)
                a1 = torch.empty_like(y1, memory_format=cl)
                _lib.check(L.avctc_bn_act(y1.data_ptr(), y1.numel() // y1.shape[1], y1.shape[1], ss1.data_ptr(), slope,
                                          None, None, 0, a1.data_ptr(), st), "avctc_bn_act")
                y2, ss2 = conv_bn(blk.conv2, blk.bn2, a1)
                res, res_ss = cur, None
                if blk.downsample is not None:
                    res, res_ss = conv_bn(blk.downsample[0], blk.downsample[1], cur)
                n, c, hh, ww = y2.shape
                last = blk is blocks[-1]                         # fused global average pool: [N, C] directly
                out = (torch.empty((n, c), device=dev, dtype=torch.bfloat16) if last
                       else torch.empty_like(y2, memory_format=cl))
                _lib.check(L.avctc_bn_act(y2.data_ptr(), n * hh * ww, c, ss2.data_ptr(), slope,
                                          res.contiguous(memory_format=cl).data_ptr(),
                                          res_ss.data_ptr() if res_ss is not None else None, hh * ww if last else 0,
                                          out.data_ptr(), st), "avctc_bn_act")
                cur = out
            if tracked:
                torch._foreach_add_(tracked, 1)
        return cur.view(b, t, 512)

    def _forward_impl(self, x):
        if self._native_applies(x):
            return self._forward_native(x)
        b, t = x.shape[0], x.shape[2]
        conv = self.frontend3D[0]
        if (x.is_cuda and x.shape[1] == 1 and conv.stride[0] == 1 and conv.dilation == (1, 1, 1)
                and isinstance(self.frontend3D[1], nn.BatchNorm3d) and self.frontend3D[1].momentum is not None):
            self._channels_last()
            y = self._frontend_as_2d(x)
            return self.trunk(y).view(b, t, 512)
        y = self.frontend3D(x)                                   # [B,64,T,H',W']
        t, h, w = y.shape[2:]
        y = y.transpose(1, 2).reshape(b * t, 64, h, w)
        return self.trunk(y).view(b, t, 512)


def xlsr_large_config(**overrides):
    """Wav2Vec2 XLSR-53-large layout (what kresnik/wav2vec2-large-xlsr-korean uses), for offline random init."""
    from transformers import Wav2Vec2Config
    cfg = dict(hidden_size=1024, num_hidden_layers=24, num_attention_heads=16, intermediate_size=4096,
               feat_extract_norm="layer", do_stable_layer_norm=True, conv_bias=True, num_conv_pos_embeddings=128,
               num_conv_pos_embedding_groups=16)
    cfg.update(overrides)
    return Wav2Vec2Config(**cfg)


class AudioEncoder(nn.Module):
    """HF Wav2Vec2Model wrapper (encoder.py:80-100): returns (last_hidden_state, mean of hidden_states[6:10]).
    `config=` builds a randomly initialised model without touching the network (bench / tests)."""

    def __init__(self, model_name="kresnik/wav2vec2-large-xlsr-korean", freeze=True, config=None):
        super().__init__()
        from transformers import Wav2Vec2Model
        if config is not None:
            config.output_hidden_states = True
            self.model = Wav2Vec2Model(config)
        else:
            self.model = Wav2Vec2Model.from_pretrained(model_name, output_hidden_states=True)
        self.output_dim = self.model.config.hidden_size
        if freeze:
            self.model.requires_grad_(False)

    def forward(self, x, attention_mask=None, host_lengths=None):
        # HF marks the conv feature extractor's output as requiring grad in train mode (a gradient-checkpointing
        # aid) unless freeze_feature_encoder() was called; the reference only sets requires_grad=False on the
        # parameters (main.py:26-31), so autograd back-propagates through seven frozen conv layers for nothing.
        # With every parameter frozen the flag changes no gradient that is ever used.
        fe = getattr(self.model, "feature_extractor", None)
        if fe is not None and getattr(fe, "_requires_grad", False) and not any(p.requires_grad for p in fe.parameters()):
            fe._requires_grad = False
        if fe is not None and not hasattr(fe, "_avctc_cached"):
            _install_feature_cache(fe)
        if attention_mask is not None:
            attention_mask = attention_mask.long()
        if self.sync_free and self._sync_free_supported():
            last, hidden_states = self._forward_sync_free(x, attention_mask, host_lengths)
        else:
            out = self.model(input_values=x, attention_mask=attention_mask, return_dict=True)
            last, hidden_states = out.last_hidden_state, out.hidden_states
        middle = torch.stack(hidden_states[6:10], dim=0).mean(dim=0)
        return last, middle

    # -------------------------------------------------------------------------------------- sync-free forward
    # Wav2Vec2Model.forward blocks the host on the GPU up to three times per call in train mode with an attention
    # mask: SpecAugment reads the utterance lengths back (`attention_mask.sum(-1).tolist()`), writes the mask
    # embedding through a boolean index (`nonzero`), and the SDPA mask builder asks `padding_mask.all()`.  Each one
    # drains the queue, so the host cannot enqueue the 24 (launch-bound) transformer layers while the GPU is still busy
    # with the convolutional front ends.  `_forward_sync_free` runs the SAME submodules in the SAME order with the same
    # random draws (numpy for SpecAugment, torch.rand([]) for LayerDrop, the CUDA generator for dropout) but takes the
    # lengths from the host copy of the mask and applies the masks with where/masked_fill.
    sync_free = True

    def _sync_free_supported(self):
        m = self.model
        cfg = m.config
        enc = m.encoder
        return (getattr(cfg, "_attn_implementation", None) == "sdpa" and getattr(m, "adapter", None) is None
                and not getattr(enc, "gradient_checkpointing", False)
                and type(enc).__name__ in ("Wav2Vec2Encoder", "Wav2Vec2EncoderStableLayerNorm"))

    def prefetch_features(self, x):
        """Enqueue the (frozen, cached) convolutional feature extractor for waveform tensor `x` now, so that later
        forward() calls on the same tensor find its output ready.  No-op when the extractor is trainable."""
        fe = self.model.feature_extractor
        if not hasattr(fe, "_avctc_cached"):
            if getattr(fe, "_requires_grad", False) and not any(p.requires_grad for p in fe.parameters()):
                fe._requires_grad = False
            _install_feature_cache(fe)
        fe(x)

    def begin_step(self):
        """Forget the cached feature-extractor output.  The cache exists to serve the SECOND call of a step (the reference
        runs the audio encoder once per speaker on the same waveform, trainer.py:94-95); a batch tensor that is kept
        resident and fed again in the next step must be encoded again, as it would be with any fresh batch."""
        st = getattr(getattr(self.model, "feature_extractor", None), "_avctc_cache_state", None)
        if st is not None:
            st["ref"] = None

    def _layer_segment(self, layer):
        seg = getattr(layer, "_avctc_graph_seg", None)
        if seg is None:
            from .graphed import GraphedSegment
            seg = GraphedSegment(lambda h, m: layer(h, attention_mask=m, output_attentions=False)[0],
                                 list(layer.parameters()), max_entries=4, modules=list(layer.modules()))
            object.__setattr__(layer, "_avctc_graph_seg", seg)
        return seg

    def _forward_sync_free(self, x, attention_mask, host_lengths):
        from transformers.models.wav2vec2.modeling_wav2vec2 import _compute_mask_indices
        m = self.model
        cfg = m.config
        extract = m.feature_extractor(x).transpose(1, 2)
        B, T = extract.shape[0], extract.shape[1]
        mask2d = None
        if attention_mask is not None:
            if host_lengths is None:                               # no host copy of the lengths: one read-back
                host_lengths = attention_mask.sum(-1).cpu()
            host_lengths = torch.as_tensor(host_lengths, dtype=torch.long).cpu()
            # upstream drops the attention mask when nothing is padded (`padding_mask.all()`, a GPU read-back, in
            # masking_utils); the host lengths answer the same question
            padded = bool((host_lengths < attention_mask.shape[1]).any())
            mask2d = m._get_feature_vector_attention_mask(T, attention_mask, add_adapter=False)
        hidden, extract = m.feature_projection(extract)
        # ---- SpecAugment (Wav2Vec2Model._mask_hidden_states) ----
        if getattr(cfg, "apply_spec_augment", True) and m.training:
            if cfg.mask_time_prob > 0:
                cpu_mask = None
                if attention_mask is not None:
                    lens = m._get_feat_extract_output_lengths(host_lengths)
                    cpu_mask = (torch.arange(T)[None, :] < lens.to(torch.long)[:, None])
                idx = _compute_mask_indices((B, T), mask_prob=cfg.mask_time_prob, mask_length=cfg.mask_time_length,
                                            attention_mask=cpu_mask, min_masks=cfg.mask_time_min_masks)
                idx = _to_device_async(torch.from_numpy(idx), hidden.device)
                hidden = torch.where(idx.unsqueeze(-1), m.masked_spec_embed.to(hidden.dtype), hidden)
            if cfg.mask_feature_prob > 0:
                idx = _compute_mask_indices((B, hidden.shape[2]), mask_prob=cfg.mask_feature_prob,
                                            mask_length=cfg.mask_feature_length, min_masks=cfg.mask_feature_min_masks)
                idx = _to_device_async(torch.from_numpy(idx), hidden.device)
                hidden = hidden.masked_fill(idx[:, None, :], 0)
        # ---- Wav2Vec2Encoder(.StableLayerNorm).forward ----
        enc = m.encoder
        stable = type(enc).__name__ == "Wav2Vec2EncoderStableLayerNorm"
        mask4d = None
        if mask2d is not None:
            hidden = hidden.masked_fill(~mask2d.unsqueeze(-1), 0)                # padded frames output 0
            if padded:
                mask4d = mask2d[:, None, None, :].expand(B, 1, T, T)             # SDPA: True = attend to that key
        pos = enc.pos_conv_embed(hidden)
        hidden = hidden + pos
        if not stable:
            hidden = enc.layer_norm(hidden)
        hidden = enc.dropout(hidden)
        all_hidden = ()
        for layer in enc.layers:
            all_hidden = all_hidden + (hidden,)
            draw = torch.rand([])                                                 # LayerDrop: host draw, as upstream
            skip = enc.training and bool(draw < cfg.layerdrop)
            if not skip:
                seg = self._layer_segment(layer)
                if seg.usable(hidden, mask4d):      # frozen layer, no gradient flows through it yet (layers 0-5 in
                    hidden = seg(hidden, mask4d)    # training, every frozen layer under no_grad): one graph launch
                else:
                    hidden = layer(hidden, attention_mask=mask4d, output_attentions=False)[0]
        if stable:
            hidden = enc.layer_norm(hidden)
        all_hidden = all_hidden + (hidden,)
        return hidden, all_hidden


def _to_device_async(t, device):
    """Small host tensor -> device without a stream synchronise (a pageable source makes the copy blocking)."""
    if device.type == "cuda":
        t = t.pin_memory()
    return t.to(device, non_blocking=True)


def _install_feature_cache(fe):
    """The trainer runs the audio encoder twice per step on the SAME waveform tensor (once per speaker mask,
    trainer.py:94-95).  The conv feature extractor is deterministic (no dropout) and frozen, so its output for an
    unchanged input tensor is reused instead of recomputed: identical values, one conv stack pass per step instead of
    two.  Installed as an instance-level forward wrapper, so module structure and state_dict keys do not change."""
    import weakref
    from .graphed import GraphedSegment
    inner = fe.forward
    state = {"ref": None, "key": None, "out": None}
    seg = GraphedSegment(inner, list(fe.parameters()), modules=list(fe.modules()))   # 7 x (conv, norm, GELU): one graph launch

    def cached_forward(input_values):
        frozen = not any(p.requires_grad for p in fe.parameters()) and not getattr(fe, "_requires_grad", False)
        if not frozen or torch.is_grad_enabled() and input_values.requires_grad:
            state["ref"] = None
            return inner(input_values)
        # identity of the live tensor OBJECT (a weak reference) + its version counter: a later batch that happens to be
        # allocated at the same address is a different object, and in-place edits bump the version
        key = (input_values._version, tuple(input_values.shape), input_values.dtype, torch.is_autocast_enabled(),
               fe.training)
        same = state["ref"] is not None and state["ref"]() is input_values and state["key"] == key
        if not same:
            with torch.no_grad():
                state["out"] = seg(input_values) if seg.usable(input_values) else inner(input_values)
            state["ref"], state["key"] = weakref.ref(input_values), key
        return state["out"]

    fe.forward = cached_forward
    fe._avctc_cached = True
    fe._avctc_cache_state = state


def install_frozen_cast_cache(root):
    """Under autocast every use of an fp32 weight launches a cast kernel; the autocast weight cache only covers
    parameters that require grad, so the FROZEN encoders (main.py:100-106: all of the visual encoder, all of wav2vec2
    but four layers) re-cast ~850 tensors per step, each a launch the host has to build.  For every Linear / Conv /
    PReLU under `root` whose own parameters are all frozen, keep the lower-precision copy of weight and bias and hand
    it to the module's forward; autocast then finds the dtype it wants and launches nothing.  The copy is the very
    rounding autocast applies, keyed on the parameter's version counter and storage so load_state_dict / in-place edits
    refresh it; a module whose parameters (again) require grad takes the normal path.  Parameters, state_dict and
    module structure are untouched (instance-level forward wrapper)."""
    kinds = (nn.Linear, nn.Conv1d, nn.Conv2d, nn.Conv3d, nn.PReLU)
    count = 0
    for mod in root.modules():
        if not isinstance(mod, kinds) or hasattr(mod, "_avctc_cast_cache") or hasattr(mod, "parametrizations"):
            continue
        _wrap_cast_cache(mod)
        count += 1
    return count


def _wrap_cast_cache(mod):
    inner = mod.forward
    cache = {}

    def forward(*args, **kwargs):
        params = mod._parameters
        w = params.get("weight")
        if w is None or w.dtype != torch.float32 or not torch.is_autocast_enabled(w.device.type):
            return inner(*args, **kwargs)
        b = params.get("bias")
        if w.requires_grad or (b is not None and b.requires_grad):
            return inner(*args, **kwargs)
        dt = torch.get_autocast_dtype(w.device.type)
        saved = {}
        for name, p in (("weight", w), ("bias", b)):
            if p is None or p.dtype != torch.float32:
                continue
            key = (p._version, p.data_ptr(), dt)
            hit = cache.get(name)
            if hit is None or hit[0] != key:
                hit = (key, p.detach().to(dt))
                cache[name] = hit
            saved[name] = p
            params[name] = hit[1]
        try:
            return inner(*args, **kwargs)
        finally:
            params.update(saved)

    mod.forward = forward
    mod._avctc_cast_cache = cache


def unfreeze_middle_layers(model):
    """main.py:26-31: only encoder.layers.6..9 of the wav2vec2 model train."""
    tags = tuple(f"encoder.layers.{i}." for i in range(6, 10))
    for name, p in model.named_parameters():
        p.requires_grad = any(t in name for t in tags)
