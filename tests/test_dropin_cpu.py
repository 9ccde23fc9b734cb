"""CPU: the import-path shims under dropin/ expose the reference's module layout (main.py:8-11, model/trainer.py:7-8)
with the reference's signatures.  Run in a subprocess so the shim names (`model`, `contrastive`, `beam_search`) never
leak into this test process."""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

CODE = r'''
import inspect
from model.fusion_module import CrossAttentionFusion
from model.decoder import CTCDecoder
from model.trainer import MultimodalTrainer
from model.encoder import VisualEncoder, AudioEncoder
from contrastive import contrastive_loss_with_mask, TEMPERATURE, WEIGHT_POS_ALIGN, WEIGHT_NEG_SUPPRESS
from beam_search import simple_beam_search, fast_decode
sig = lambda f: str(inspect.signature(f))
assert sig(CrossAttentionFusion.__init__) == "(self, visual_dim, audio_dim, fused_dim, num_heads=4)"
assert sig(CrossAttentionFusion.forward) == "(self, visual_feat, audio_feat, mask=None)"
assert sig(CTCDecoder.__init__) == "(self, input_dim, vocab_size, blank_id=0)"
assert sig(CTCDecoder.forward) == "(self, x, target=None, input_lengths=None, target_lengths=None)"
assert sig(MultimodalTrainer.__init__) == ("(self, visual_encoder, audio_encoder, fusion_module, decoder1, tokenizer, "
                                           "learning_rate=0.0001, device='cuda', lambda_=0.1)")
assert sig(contrastive_loss_with_mask) == "(middle_feat, flat_mask, projection_layer=None)"
assert sig(simple_beam_search).startswith("(log_probs") and "beam_width=5" in sig(simple_beam_search) and "blank=0" in sig(simple_beam_search)
assert (TEMPERATURE, WEIGHT_POS_ALIGN, WEIGHT_NEG_SUPPRESS) == (0.07, 1.0, 0.3)
for m in ("train_epoch", "evaluate", "ctc_decode", "crop_or_pad_feat"):
    assert callable(getattr(MultimodalTrainer, m))
print("dropin ok")
'''


def test_dropin_shims_expose_reference_layout(tmp_path):
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([os.path.join(ROOT, "dropin"), ROOT]))
    r = subprocess.run([sys.executable, "-c", CODE], capture_output=True, text=True, env=env, cwd=tmp_path)
    assert r.returncode == 0, r.stderr[-2000:]
    assert "dropin ok" in r.stdout
