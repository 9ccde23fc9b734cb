"""multimodal-av-model_b200 — B200 (sm_100a) implementation of the AV-CTC hot path of
limeorange1102/multimodal-av-model behind the reference's own Python call surface.

Import name: ``multimodal_av_model_b200`` (alias shim at the repo root; the directory name carries a
hyphen).  Public names mirror the reference modules (SURVEY.md §8b):

    CrossAttentionFusion, CTCDecoder          model/fusion_module.py, model/decoder.py
    CTCLoss, ctc_loss                         nn.CTCLoss as used at model/trainer.py:25
    contrastive_loss_with_mask                contrastive.py
    simple_beam_search, fast_decode           beam_search.py  (+ beam_search_batch)
    MultimodalTrainer                         model/trainer.py
    forced_align, merge_tokens, TokenSpan     torchaudio.functional's CTC forced alignment, batched (align.py)
"""
from . import _lib
from .ctc import CTCLoss, ctc_loss

__all__ = ["CTCLoss", "ctc_loss"]


def _optional(module, names):
    import importlib
    m = importlib.import_module(f"{__name__}.{module}")
    for n in names:
        globals()[n] = getattr(m, n)
        __all__.append(n)


_optional("beam_search", ["simple_beam_search", "fast_decode", "beam_search_batch"])
_optional("fusion_module", ["CrossAttentionFusion"])
_optional("decoder", ["CTCDecoder"])
_optional("contrastive", ["contrastive_loss_with_mask"])
_optional("align", ["forced_align", "merge_tokens", "merge_tokens_batch", "TokenSpan"])
_optional("trainer", ["MultimodalTrainer"])
_optional("encoders", ["VisualEncoder", "AudioEncoder"])
