"""CPU: CTC forced alignment — the numpy oracle and merge_tokens against torchaudio's outputs stored in
tests/golden/align_cases.npz, and the fused-frame -> encoder-frame map trainer.align() uses."""
import numpy as np
import pytest
import torch

from conftest import load_cases
from oracle import align_oracle, np_oracle


def _pkg():
    import multimodal_av_model_b200 as pkg
    return pkg


CASES = load_cases("align_cases.npz")


@pytest.mark.parametrize("case", sorted(CASES))
def test_oracle_matches_torchaudio_fixture(case):
    c = CASES[case]
    paths, scores = align_oracle.ctc_forced_align(c["lp"], c["targets"], int(c["blank"]))
    assert np.array_equal(paths, c["paths"])
    assert np.array_equal(scores.view(np.uint32), c["scores"].view(np.uint32))


def test_fixture_covers_the_listed_cases():
    z = np.load(__import__("conftest").GOLDEN + "/align_cases.npz")
    names = set(str(n) for n in z["names"])
    assert {"random", "ties_int", "tight", "repeats", "blank3", "v800"} <= names
    assert str(z["torchaudio_version"]).startswith("2.")
    for c in CASES.values():
        tg = c["targets"]
        R = int((tg[1:] == tg[:-1]).sum())
        assert c["lp"].shape[0] >= len(tg) + R


@pytest.mark.parametrize("case", sorted(CASES))
def test_merge_tokens_matches_fixture_spans(case):
    pkg = _pkg()
    c = CASES[case]
    spans = pkg.merge_tokens(torch.from_numpy(c["paths"]), torch.from_numpy(c["scores"]), blank=int(c["blank"]))
    got = np.array([[s.token, s.start, s.end] for s in spans], dtype=np.int64).reshape(-1, 3)
    assert np.array_equal(got, c["spans"])
    assert [s.score for s in spans] == c["span_scores"].tolist()
    assert len(spans) == len(c["targets"])                          # one span per target token
    assert all(len(s) == s.end - s.start > 0 for s in spans)


def test_merge_tokens_batch_cuts_each_row_at_its_length():
    pkg = _pkg()
    from multimodal_av_model_b200.align import merge_tokens_batch
    paths = torch.tensor([[0, 5, 5, 0, 6, 0], [7, 7, 0, 8, 0, 9]])
    scores = torch.tensor([[-1., -2., -3., -4., -5., -6.], [-.5, -1.5, -2., -3., -4., -5.]])
    out = merge_tokens_batch(paths, scores, torch.tensor([6, 4]), blank=0)
    assert out[0] == pkg.merge_tokens(paths[0], scores[0], blank=0)
    assert [(s.token, s.start, s.end) for s in out[1]] == [(7, 0, 2), (8, 3, 4)]
    assert out[1][0].score == -1.0


def _masks(rng, B, t_enc):
    m = np.full((B, t_enc), 3, dtype=np.int64)
    for b in range(B):
        n = int(rng.integers(t_enc // 3, t_enc + 1))
        m[b, :n] = rng.choice([0, 1, 2], size=n, p=[0.3, 0.4, 0.3])
    return m


@pytest.mark.parametrize("t_v", [30, 150, 249, 400])
def test_fused_frame_map_matches_the_fusion_resample(t_v):
    """The encoder frame fused_frame_encoder_index gives each fused frame is the one select_pad_resample moves there:
    resample the encoder-frame INDEX as the mask is resampled (nearest) and compare."""
    from multimodal_av_model_b200.align import fused_frame_encoder_index, nearest_src_index
    rng = np.random.default_rng(t_v)
    B, t_enc = 6, 249
    m = _masks(rng, B, t_enc)
    enc = fused_frame_encoder_index(torch.from_numpy(m), t_v).numpy()
    speech = (m != 0) & (m != 3)
    Tp = int(speech.sum(1).max())
    assert np.array_equal(nearest_src_index(t_v, Tp).numpy(), np_oracle.nearest_src_index(t_v, Tp))
    _, m_rs = np_oracle.select_pad_resample(np.zeros((B, t_enc, 1)), m, t_v)
    # the mask is resampled with `nearest`: the fused frame's source rank is read off a rank-valued mask the same way
    ranks = np.zeros((B, Tp), dtype=np.int64)
    for b in range(B):
        fr = np.nonzero(speech[b])[0]
        ranks[b, :len(fr)] = fr + 1                                  # encoder frame + 1, 0 = padding
    want = (ranks[:, np_oracle.nearest_src_index(t_v, Tp)] if t_v != Tp else ranks) - 1
    assert np.array_equal(enc, want)
    # frames the fusion counts as input (resampled mask != 0) are exactly those with an encoder frame
    assert np.array_equal(enc >= 0, m_rs != 0)
    assert all(np.all(np.diff(e[e >= 0]) >= 0) for e in enc)


def test_forced_align_rejects_cpu_tensors():
    pkg = _pkg()
    lp = torch.randn(2, 10, 5).log_softmax(-1)
    with pytest.raises(RuntimeError, match="CUDA"):
        pkg.forced_align(lp, torch.ones(2, 3, dtype=torch.long))
