"""Producers that feed the hot path: VisualEncoder and AudioEncoder (SURVEY.md §8 row a15).

The third-party wav2vec2 stays HF/PyTorch except for its encoder layers that a gradient flows through: on CUDA under bf16
autocast those run on this library's kernels (csrc/wav2vec2_layer.cu) around torch's attention core, with dropout
identical to ATen's; the module path is the CPU path and the reference.  The frozen visual encoder's bf16-autocast forward on CUDA runs on this
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
                elif _w2v_native_applies(layer, hidden):
                    hidden = _w2v_native_layer(layer, hidden, mask4d)
                else:
                    hidden = layer(hidden, attention_mask=mask4d, output_attentions=False)[0]
        if stable:
            hidden = enc.layer_norm(hidden)
        all_hidden = all_hidden + (hidden,)
        return hidden, all_hidden


# ------------------------------------------------------------------------------------ native wav2vec2 layers
# The layers a gradient flows through (6-9 train, 10-23 carry the input gradient back to them) cannot be graphed; through
# HF's module code each layer-call costs ~100 dispatcher ops forward and 80-144 backward, and the host's enqueue of them
# bounded the train step.  On the native path a layer is two library calls per direction (csrc/wav2vec2_layer.cu) with
# torch's attention interface between them, called exactly as Wav2Vec2Attention.forward calls it (its dropout stream
# cannot be reproduced by our own kernel).  The module path stays the reference and the path for everything else.

def _w2v_native_applies(layer, hidden):
    """bf16-autocast CUDA forward of a Wav2Vec2EncoderLayerStableLayerNorm with sdpa attention, exact GELU, no adapter,
    fp32 parameters and dropout probabilities below 1, outside stream capture."""
    from transformers.models.wav2vec2.modeling_wav2vec2 import Wav2Vec2EncoderLayerStableLayerNorm
    if not (hidden.is_cuda and hidden.dtype == torch.bfloat16 and hidden.dim() == 3 and hidden.is_contiguous()
            and torch.is_autocast_enabled("cuda") and torch.get_autocast_dtype("cuda") == torch.bfloat16
            and not torch.cuda.is_current_stream_capturing()):
        return False
    if type(layer) is not Wav2Vec2EncoderLayerStableLayerNorm or layer.adapter_layer is not None:
        return False
    cfg = layer.attention.config
    if getattr(cfg, "_attn_implementation", None) != "sdpa" or cfg.hidden_act != "gelu":
        return False
    e, f = hidden.shape[-1], layer.feed_forward.intermediate_dense.out_features
    if e % 256 or e > 1024 or f % 8 or hidden.shape[0] * hidden.shape[1] == 0:
        return False
    ff = layer.feed_forward
    if any(not 0.0 <= d.p < 1.0 for d in (layer.dropout, ff.intermediate_dropout, ff.output_dropout)):
        return False
    return all(p.dtype == torch.float32 and p.is_cuda for p in layer.parameters())


_optimizer_steps = [0]
_optimizer_hook = []


def _optimizer_step_count():
    """torch.optim steps taken in this process since the first call.  Adam(fused=True) updates parameters in place without
    advancing their version counters, so a version key alone would keep serving the weights of before the step."""
    if not _optimizer_hook:
        from torch.optim.optimizer import register_optimizer_step_post_hook

        def bump(opt, args, kwargs):
            _optimizer_steps[0] += 1
        _optimizer_hook.append(register_optimizer_step_post_hook(bump))
    return _optimizer_steps[0]


def _w2v_params(layer):
    """bf16 weight copies the kernels read and the bf16-rounded biases autocast would add, made once per parameter
    version: frozen layers cast once, trainable ones once per optimizer step (shared by both calls of the step)."""
    a, ff = layer.attention, layer.feed_forward
    lins = (a.q_proj, a.k_proj, a.v_proj, a.out_proj, ff.intermediate_dense, ff.output_dense)
    params = [p for m in lins for p in (m.weight, m.bias)]
    steps = _optimizer_step_count() if any(p.requires_grad for p in params) else None
    key = (steps, tuple((p._version, p.data_ptr()) for p in params))
    hit = getattr(layer, "_avctc_w2v_cache", None)
    if hit is None or hit[0] != key:
        bf = torch.bfloat16
        with torch.no_grad():
            prm = {"wqkv": torch.cat([a.q_proj.weight, a.k_proj.weight, a.v_proj.weight]).to(bf),
                   "bqkv": torch.cat([a.q_proj.bias, a.k_proj.bias, a.v_proj.bias]).to(bf).float(),
                   "wo": a.out_proj.weight.to(bf), "bo": a.out_proj.bias.to(bf).float(),
                   "w1": ff.intermediate_dense.weight.to(bf), "b1": ff.intermediate_dense.bias.to(bf).float(),
                   "w2": ff.output_dense.weight.to(bf), "b2": ff.output_dense.bias.to(bf).float()}
        hit = (key, prm)
        object.__setattr__(layer, "_avctc_w2v_cache", hit)
    return hit[1]


class _W2VAttnIn(torch.autograd.Function):
    """q, k, v = projections of LayerNorm(x): avctc_w2v_attn_in_forward / _backward."""

    @staticmethod
    def forward(ctx, x, ln_w, ln_b, wq, bq, wk, bk, wv, bv, prm, eps):
        from . import _lib
        L = _lib.lib()
        b, t, e = x.shape
        m = b * t
        with _lib.device_guard(x.device):
            saved = torch.empty(L.avctc_w2v_workspace_bytes(m, e, 8, 0), dtype=torch.uint8, device=x.device)
            q, k, v = torch.empty_like(x), torch.empty_like(x), torch.empty_like(x)
            _lib.check(L.avctc_w2v_attn_in_forward(x.data_ptr(), m, e, ln_w.data_ptr(), ln_b.data_ptr(), eps,
                                                   prm["wqkv"].data_ptr(), prm["bqkv"].data_ptr(), q.data_ptr(),
                                                   k.data_ptr(), v.data_ptr(), saved.data_ptr(), saved.numel(),
                                                   _lib.stream_ptr(x.device)), "avctc_w2v_attn_in_forward")
        ctx.save_for_backward(x, ln_w, saved)
        ctx.prm = prm
        return q, k, v

    @staticmethod
    def backward(ctx, dq, dk, dv):
        from . import _lib
        L = _lib.lib()
        x, ln_w, saved = ctx.saved_tensors
        b, t, e = x.shape
        m, dev = b * t, x.device
        need = ctx.needs_input_grad
        wg = any(need[1:9])
        dq, dk, dv = (g.to(torch.bfloat16).contiguous() for g in (dq, dk, dv))
        with _lib.device_guard(dev):
            scratch = torch.empty(L.avctc_w2v_workspace_bytes(m, e, 8, 2), dtype=torch.uint8, device=dev)
            dx = torch.empty_like(x)
            g = [None] * 4
            if wg:
                g = [torch.empty((3 * e, e), device=dev), torch.empty(3 * e, device=dev), torch.empty(e, device=dev),
                     torch.empty(e, device=dev)]
            _lib.check(L.avctc_w2v_attn_in_backward(dq.data_ptr(), dk.data_ptr(), dv.data_ptr(), x.data_ptr(), m, e,
                                                    ln_w.data_ptr(), ctx.prm["wqkv"].data_ptr(), dx.data_ptr(),
                                                    *[a.data_ptr() if a is not None else None for a in g],
                                                    saved.data_ptr(), saved.numel(), scratch.data_ptr(), scratch.numel(),
                                                    _lib.stream_ptr(dev)), "avctc_w2v_attn_in_backward")
        if not wg:
            return dx, None, None, None, None, None, None, None, None, None, None
        gw, gb, glw, glb = g
        out = [glw, glb, gw[:e], gb[:e], gw[e:2 * e], gb[e:2 * e], gw[2 * e:], gb[2 * e:]]
        return (dx, *[o if n else None for o, n in zip(out, need[1:9])], None, None)


class _W2VAttnOutFFN(torch.autograd.Function):
    """out_proj, hidden dropout, residual, final LayerNorm, feed-forward with its two dropouts, residual:
    avctc_w2v_attn_out_ffn_forward / _backward.  The three dropouts take their generator offsets here, after the
    attention core took its own, in module order."""

    @staticmethod
    def forward(ctx, attn, x, wo, bo, ln_w, ln_b, w1, b1, w2, b2, prm, eps, probs):
        from . import _lib
        L = _lib.lib()
        b, t, e = x.shape
        m, f, dev = b * t, w1.shape[0], x.device
        with _lib.device_guard(dev):
            incr = L.avctc_w2v_dropout_increment(m, e, f, *probs, 1)
            _lib.check(0 if incr >= 0 else incr, "avctc_w2v_dropout_increment")
            seed = offset = 0
            if incr:
                gen = torch.cuda.default_generators[dev.index]
                seed, offset = gen.initial_seed(), gen.get_offset()
                gen.set_offset(offset + incr)
            saved = torch.empty(L.avctc_w2v_workspace_bytes(m, e, f, 1), dtype=torch.uint8, device=dev)
            y = torch.empty_like(x)
            _lib.check(L.avctc_w2v_attn_out_ffn_forward(attn.data_ptr(), x.data_ptr(), m, e, f, prm["wo"].data_ptr(),
                                                        prm["bo"].data_ptr(), ln_w.data_ptr(), ln_b.data_ptr(), eps,
                                                        prm["w1"].data_ptr(), prm["b1"].data_ptr(), prm["w2"].data_ptr(),
                                                        prm["b2"].data_ptr(), *probs, 1, seed, offset, y.data_ptr(),
                                                        saved.data_ptr(), saved.numel(), _lib.stream_ptr(dev)),
                       "avctc_w2v_attn_out_ffn_forward")
        wg = any(ctx.needs_input_grad[2:10])
        ctx.save_for_backward(attn if wg else None, ln_w, saved)
        ctx.prm, ctx.probs, ctx.seed, ctx.offset, ctx.dims = prm, probs, seed, offset, (b, t, e, f)
        return y

    @staticmethod
    def backward(ctx, dy):
        from . import _lib
        L = _lib.lib()
        attn, ln_w, saved = ctx.saved_tensors
        b, t, e, f = ctx.dims
        m, dev = b * t, ln_w.device
        need = ctx.needs_input_grad
        wg = any(need[2:10])
        dy = dy.to(torch.bfloat16).contiguous()
        prm = ctx.prm
        with _lib.device_guard(dev):
            scratch = torch.empty(L.avctc_w2v_workspace_bytes(m, e, f, 3), dtype=torch.uint8, device=dev)
            dattn, dx = torch.empty_like(dy), torch.empty_like(dy)
            g = [None] * 8
            if wg:
                g = [torch.empty((e, e), device=dev), torch.empty(e, device=dev), torch.empty(e, device=dev),
                     torch.empty(e, device=dev), torch.empty((f, e), device=dev), torch.empty(f, device=dev),
                     torch.empty((e, f), device=dev), torch.empty(e, device=dev)]
            _lib.check(L.avctc_w2v_attn_out_ffn_backward(
                dy.data_ptr(), attn.data_ptr() if attn is not None else dy.data_ptr(), m, e, f, prm["wo"].data_ptr(),
                ln_w.data_ptr(), prm["w1"].data_ptr(), prm["w2"].data_ptr(), *ctx.probs, 1, ctx.seed, ctx.offset,
                dattn.data_ptr(), dx.data_ptr(), *[a.data_ptr() if a is not None else None for a in g],
                saved.data_ptr(), saved.numel(), scratch.data_ptr(), scratch.numel(), _lib.stream_ptr(dev)),
                "avctc_w2v_attn_out_ffn_backward")
        return (dattn, dx, *[o if n else None for o, n in zip(g, need[2:10])], None, None, None)


def _w2v_native_layer(layer, hidden, mask4d):
    """Wav2Vec2EncoderLayerStableLayerNorm.forward(hidden, attention_mask=mask4d)[0] on the native path."""
    from transformers.modeling_utils import ALL_ATTENTION_FUNCTIONS
    from transformers.models.wav2vec2.modeling_wav2vec2 import eager_attention_forward
    a, ff = layer.attention, layer.feed_forward
    ln1, ln2 = layer.layer_norm, layer.final_layer_norm
    prm = _w2v_params(layer)
    b, t, _ = hidden.shape
    q, k, v = _W2VAttnIn.apply(hidden, ln1.weight, ln1.bias, a.q_proj.weight, a.q_proj.bias, a.k_proj.weight,
                               a.k_proj.bias, a.v_proj.weight, a.v_proj.bias, prm, ln1.eps)
    shape = (b, t, -1, a.head_dim)
    interface = ALL_ATTENTION_FUNCTIONS.get_interface(a.config._attn_implementation, eager_attention_forward)
    o, _ = interface(a, q.view(shape).transpose(1, 2), k.view(shape).transpose(1, 2), v.view(shape).transpose(1, 2),
                     mask4d, dropout=0.0 if not a.training else a.dropout, scaling=a.scaling, output_attentions=False)
    o = o.reshape(b, t, -1).contiguous()
    probs = tuple(float(d.p) if d.training else 0.0 for d in (layer.dropout, ff.intermediate_dropout, ff.output_dropout))
    return _W2VAttnOutFFN.apply(o, hidden, a.out_proj.weight, a.out_proj.bias, ln2.weight, ln2.bias,
                                ff.intermediate_dense.weight, ff.intermediate_dense.bias, ff.output_dense.weight,
                                ff.output_dense.bias, prm, ln2.eps, probs)


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
