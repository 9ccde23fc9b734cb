"""oracle/encoder_port.py — the reference's two encoders restated on stock torch / HF ops.  TEST INFRASTRUCTURE ONLY.

bench.py's `--impl reference` / `cpu_baseline` legs time the reference's train step on the host CPU.  The encoders are
the bulk of that step, and the reference arm must not run through the product's own `encoders.py` (which carries
scheduling changes: sync-free wav2vec2 forward, cast cache, channels-last), so this file restates
/root/reference/model/encoder.py with nothing but `torch.nn` modules and the UNMODIFIED `Wav2Vec2Model.forward`:

  VisualPort   encoder.py:57-75   Conv3d(1->64,(5,7,7),s(1,2,2)) + BN3d + PReLU + MaxPool3d, per-frame ResNet-18 trunk
               (BasicBlock x [2,2,2,2], PReLU, no stem, global average pool) -> [B,T,512]
  AudioPort    encoder.py:80-100  Wav2Vec2Model(output_hidden_states=True) -> (last_hidden_state, mean(hidden_states[6:10]))
  freeze policy main.py:26-31,100-106: visual encoder frozen, only wav2vec2 encoder.layers.6-9 train

Sub-module names follow the reference (`frontend3D`, `trunk.layerN.i.{conv1,bn1,relu,conv2,bn2,downsample}`, `model`) so
its state_dict loads.  Both ports were checked equal to the reference classes on CPU when written; that check needs the
reference's source, which is not part of this repository, so the suite does not carry it.  Random init only (no
checkpoint is reachable offline): wav2vec2 is built from the XLSR-53-large layout.
"""
from __future__ import annotations

import torch
import torch.nn as nn

_STAGES = ((64, 1), (128, 2), (256, 2), (512, 2))       # (width, stride of the first block) of trunk.layer1..4


class _Block(nn.Module):
    def __init__(self, cin, cout, stride):
        super().__init__()
        self.conv1 = nn.Conv2d(cin, cout, 3, stride, 1, bias=False)
        self.bn1 = nn.BatchNorm2d(cout)
        self.relu = nn.PReLU(cout)                       # ONE PReLU per block, used twice (encoder.py:11,18,22)
        self.conv2 = nn.Conv2d(cout, cout, 3, 1, 1, bias=False)
        self.bn2 = nn.BatchNorm2d(cout)
        self.downsample = None
        if stride != 1 or cin != cout:
            self.downsample = nn.Sequential(nn.Conv2d(cin, cout, 1, stride, bias=False), nn.BatchNorm2d(cout))

    def forward(self, x):
        y = self.bn2(self.conv2(self.relu(self.bn1(self.conv1(x)))))
        return self.relu(y + (x if self.downsample is None else self.downsample(x)))


class _Trunk(nn.Module):
    def __init__(self):
        super().__init__()
        cin = 64
        for i, (width, stride) in enumerate(_STAGES, start=1):
            self.add_module(f"layer{i}", nn.Sequential(_Block(cin, width, stride), _Block(width, width, 1)))
            cin = width
        self.avgpool = nn.AdaptiveAvgPool2d(1)

    def forward(self, x):
        for i in range(1, len(_STAGES) + 1):
            x = getattr(self, f"layer{i}")(x)
        return self.avgpool(x).flatten(1)


class VisualPort(nn.Module):
    def __init__(self):
        super().__init__()
        self.frontend3D = nn.Sequential(nn.Conv3d(1, 64, (5, 7, 7), (1, 2, 2), (2, 3, 3), bias=False), nn.BatchNorm3d(64),
                                        nn.PReLU(64), nn.MaxPool3d((1, 3, 3), (1, 2, 2), (0, 1, 1)))
        self.trunk = _Trunk()

    def forward(self, x):                                   # [B,1,T,H,W]
        b = x.shape[0]
        y = self.frontend3D(x)                              # [B,64,T,H',W']
        y = y.transpose(1, 2).reshape(-1, 64, y.shape[3], y.shape[4])
        return self.trunk(y).view(b, -1, 512)


def xlsr_large_config(**overrides):
    """XLSR-53-large layout of kresnik/wav2vec2-large-xlsr-korean (SURVEY.md §8c)."""
    from transformers import Wav2Vec2Config
    kw = dict(hidden_size=1024, num_hidden_layers=24, num_attention_heads=16, intermediate_size=4096,
              feat_extract_norm="layer", do_stable_layer_norm=True, conv_bias=True, num_conv_pos_embeddings=128,
              num_conv_pos_embedding_groups=16)
    kw.update(overrides)
    return Wav2Vec2Config(**kw)


class AudioPort(nn.Module):
    def __init__(self, config=None):
        super().__init__()
        from transformers import Wav2Vec2Model
        cfg = config if config is not None else xlsr_large_config()
        cfg.output_hidden_states = True
        self.model = Wav2Vec2Model(cfg)
        for name, p in self.model.named_parameters():       # main.py:26-31
            p.requires_grad = any(f"encoder.layers.{i}." in name for i in range(6, 10))

    def forward(self, x, attention_mask=None):
        out = self.model(input_values=x, attention_mask=None if attention_mask is None else attention_mask.long(),
                         return_dict=True)
        return out.last_hidden_state, torch.stack(out.hidden_states[6:10], 0).mean(0)
