"""CPU: the LM-fused prefix beam search oracle (oracle/prefix_beam_lm_oracle.py) — the back-off walk on a hand-written
ARPA, the alpha = beta = 0 case against the plain search, every hypothesis of an unpruned search against the CTC loss
plus the LM's sentence probability — and the ARPA loaders' checks (oracle and ngram_lm.NgramLM)."""
import itertools
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import prefix_beam_lm_oracle as LO
from oracle import prefix_beam_oracle as O

# <s> a b c </s> <unk> are words; "zz" is not a model piece, so every n-gram with it is dropped
ARPA = """
\\data\\
ngram 1=7
ngram 2=6
ngram 3=3

\\1-grams:
-99\t<s>\t-0.5
-1.0\t</s>
-2.0\t<unk>
-0.7\ta\t-0.25
-0.9\tb\t-0.125
-1.25\tc
-0.3\tzz\t-0.1

\\2-grams:
-0.2\t<s> a\t-0.0625
-0.4\ta b\t-0.375
-0.6\tb </s>
-0.8\ta <unk>
-0.1\tzz a\t-0.2
-0.15\ta zz

\\3-grams:
-0.05\t<s> a b
-0.35\ta b c
-0.02\tzz a b

\\end\\
"""
VOCAB = ["_", "a", "b", "c", "d"]          # 0 = blank piece (absent from the LM), 4 = "d" (absent: <unk>)


def f32(x):
    return float(np.float32(x))


def _lm(text=ARPA, vocab=VOCAB):
    return LO.read_arpa(text, vocab)


def test_lm10_backoff_walk():
    lm = _lm()
    assert lm.order == 3
    # full hits at order 3
    assert lm.lm10("b", ("<s>", "a")) == f32(-0.05)
    assert lm.lm10("c", ("a", "b")) == f32(-0.35)
    # one back-off: (a b </s>) is absent -> bow(a b) + p(b </s>)
    assert lm.lm10("</s>", ("a", "b")) == 0.0 + f32(-0.375) + f32(-0.6)
    # two back-offs: (<s> a c) and (a c) are absent -> bow(<s> a) + bow(a) + p(c)
    assert lm.lm10("c", ("<s>", "a")) == (0.0 + f32(-0.0625)) + f32(-0.25) + f32(-1.25)
    # absent context: the 2-gram (c a) does not exist, so its bow is 0
    assert lm.lm10("a", ("c", "a")) == ((0.0 + 0.0) + f32(-0.25)) + f32(-0.7)
    # <unk>: the 2-gram (a <unk>) after the absent context (b a)
    assert lm.lm10("<unk>", ("b", "a")) == (0.0 + 0.0) + f32(-0.8)
    assert lm.word(4) == "<unk>" and lm.word(0) == "<unk>" and lm.word(2) == "b"
    # the context is truncated to order - 1 words
    assert lm.lm10("b", ("c", "c", "<s>", "a")) == f32(-0.05)
    # unigram with a bow-less context: (c) has no bow -> 0
    assert lm.lm10("b", ("c",)) == 0.0 + 0.0 + f32(-0.9)


def test_oov_ngrams_are_dropped_without_changing_queries():
    lm = _lm()
    assert not any("zz" in k for k in lm.probs)
    stripped = "\n".join(ln for ln in ARPA.splitlines() if "zz" not in ln).replace("ngram 1=7", "ngram 1=6")
    ref = _lm(stripped)
    words = ["<s>", "a", "b", "c", "</s>", "<unk>"]
    for n in range(0, 3):
        for h in itertools.product(words, repeat=n):
            for w in words[1:]:
                assert lm.lm10(w, ("<s>",) + h) == ref.lm10(w, ("<s>",) + h)
    assert lm.probs == ref.probs


@pytest.mark.parametrize("bad, match", [
    (ARPA.replace("-1.0\t</s>\n", ""), "lacks </s>"),
    (ARPA.replace("-2.0\t<unk>\n", ""), "lacks <unk>"),
    (ARPA.replace("-99\t<s>\t-0.5\n", ""), "lacks <s>"),
    (ARPA.replace("ngram 3=3", "ngram 3=3\nngram 6=1"), "order 6"),
    (ARPA.replace("\\end\\", "\\6-grams:\n-1\t<s> a b c a b\n\\end\\"), "order 6"),
    (ARPA.replace("-0.4\ta b", "nan\ta b"), "non-finite"),
    (ARPA.replace("-0.9\tb\t-0.125", "-0.9\tb\tinf"), "non-finite"),
    (ARPA.replace("-0.6\tb </s>", "-0.6\tb </s>\n-0.7\tb </s>"), "duplicate"),
])
def test_oracle_loader_rejects(bad, match):
    with pytest.raises(ValueError, match=match):
        _lm(bad)


def _pkg():
    import multimodal_av_model_b200 as pkg
    return pkg


def test_package_loader(tmp_path):
    pkg = _pkg()
    p = tmp_path / "lm.arpa"
    p.write_text(ARPA, encoding="utf-8")
    lm = pkg.NgramLM.from_arpa(str(p), VOCAB)
    assert lm.order == 3 and lm.counts == (6, 4, 2) and lm.vocab_size == 5
    for bad, match in [(ARPA.replace("-1.0\t</s>\n", ""), "lacks </s>"), (ARPA.replace("-2.0\t<unk>\n", ""), "<unk>"),
                       (ARPA.replace("-99\t<s>\t-0.5\n", ""), "<s>"),
                       (ARPA.replace("ngram 3=3", "ngram 3=3\nngram 6=1"), "order 6"),
                       (ARPA.replace("-0.4\ta b", "nan\ta b"), "non-finite"),
                       (ARPA.replace("-0.6\tb </s>", "-0.6\tb </s>\n-0.7\tb </s>"), "duplicate"),
                       (ARPA.replace("-0.02\tzz a b", "-0.02\tzz a b\n-0.03\tzz a b"), "duplicate")]:
        q = tmp_path / "bad.arpa"
        q.write_text(bad, encoding="utf-8")
        with pytest.raises(ValueError, match=match):
            pkg.NgramLM.from_arpa(str(q), VOCAB)
    with pytest.raises(ValueError, match="vocab"):
        pkg.NgramLM.from_arpa(str(p), [])
    with pytest.raises(ValueError, match="vocab"):
        pkg.NgramLM.from_arpa(str(p), [str(i) for i in range(1025)])


def test_search_checks_vocab_length_before_any_launch(tmp_path):
    pkg = _pkg()
    p = tmp_path / "lm.arpa"
    p.write_text(ARPA, encoding="utf-8")
    lm = pkg.NgramLM.from_arpa(str(p), VOCAB)
    with pytest.raises(RuntimeError, match="CUDA"):
        pkg.ctc_prefix_beam_search(torch.zeros(2, 3, 5), lm=lm)
    with pytest.raises(ValueError, match="pieces"):
        LO.prefix_beam_lm_search(np.zeros((3, 6), np.float32), 3, 2, 1, 0, _lm(), 0.5, 0.0)


def _rand_lp(seed, T, V, scale=2.0):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(T, V, generator=g, dtype=torch.float64) * scale).log_softmax(-1).float().numpy()


@pytest.mark.parametrize("blank", [0, 3])
def test_zero_weights_equal_the_plain_search(blank):
    lm = _lm()
    for seed in range(4):
        lp = _rand_lp(seed, 12, 5, scale=3.0)
        for B in (1, 3, 6):
            st, plain = O.prefix_beam_search(lp, 12, B, B, blank)
            st2, fused = LO.prefix_beam_lm_search(lp, 12, B, B, blank, lm, 0.0, 0.0)
            assert st == st2 == 0
            assert [(t, s) for t, s, _, _ in fused] == plain
            assert all(a == s and m == 0.0 for _, s, a, m in fused)


def _ctc_logprob(lp, toks, blank):
    lp64 = torch.from_numpy(lp).double()[:, None]
    tg = torch.tensor([list(toks)], dtype=torch.long) if toks else torch.zeros(1, 0, dtype=torch.long)
    return -F.ctc_loss(lp64, tg, torch.tensor([lp.shape[0]]), torch.tensor([len(toks)]), blank=blank,
                       reduction="none").item()


@pytest.mark.parametrize("alpha, beta", [(0.3, -0.5), (1.0, 1.5)])
def test_exhaustive_hypotheses_score_ctc_plus_lm(alpha, beta):
    """V = 3 (blank 0 + a, b), T = 3, B = 15: no prefix is pruned, so the hypotheses are the 9 feasible strings with
    acoustic = -ctc_loss and lm = alpha * ln P(l </s>) + beta * |l|, ranked by their sum."""
    vocab = ["_", "a", "b"]
    lm = _lm(vocab=vocab)
    lp = _rand_lp(17, 3, 3, scale=1.0)
    st, hyps = LO.prefix_beam_lm_search(lp, 3, 15, 15, 0, lm, alpha, beta, prune=False)
    assert st == 0 and len(hyps) == 9
    assert LO.prefix_beam_lm_search(lp, 3, 15, 15, 0, lm, alpha, beta) == (st, hyps)   # k = min(31, V) = V
    for toks, score, ac, lms in hyps:
        assert score == ac + lms
        assert abs(ac - _ctc_logprob(lp, toks, 0)) < 1e-12
        words = ["<s>"] + [lm.word(c) for c in toks]
        l10 = sum(lm.lm10(w, words[:i + 1]) for i, w in enumerate(words[1:] + ["</s>"]))
        assert abs(lms - (alpha * l10 * math.log(10.0) + beta * len(toks))) < 1e-12
    assert [h[1] for h in hyps] == sorted((h[1] for h in hyps), reverse=True)


def test_length_zero_and_failures():
    lm = _lm()
    lp = _rand_lp(1, 5, 5)
    st, hyps = LO.prefix_beam_lm_search(lp, 0, 3, 2, 0, lm, 0.5, 1.0)
    e = 0.5 * (lm.lm10("</s>", ("<s>",)) * LO.LN10)
    assert st == 0 and hyps == [((), 0.0 + e, 0.0, e)]
    assert LO.prefix_beam_lm_search(lp, 6, 3, 2, 0, lm, 0.5, 1.0) == (2, [])
    bad = lp.copy()
    bad[2, 1] = np.nan
    assert LO.prefix_beam_lm_search(bad, 5, 3, 2, 0, lm, 0.5, 1.0) == (1, [])
    for a, b in ((-0.1, 0.0), (math.inf, 0.0), (0.5, math.nan)):
        with pytest.raises(ValueError):
            LO.prefix_beam_lm_search(lp, 5, 3, 2, 0, lm, a, b)
