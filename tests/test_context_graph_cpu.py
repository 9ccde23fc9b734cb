"""CPU: contextual biasing (DESIGN.md §4.15) — the package's dense automaton tables (context_graph.ContextGraph) against
the oracle's dict automaton (oracle/context_graph_oracle.py), hand-computed phi / omega / delta, the builder's
rejections, the oracle's bias accounting, a never-hit context against the §4.13 / §4.14 searches, and an exhaustive
V = 3 search against the CTC loss and the rule applied to each hypothesis."""
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import context_graph_oracle as CO
from oracle import prefix_beam_lm_oracle as LO
from oracle import prefix_beam_oracle as O


def _pkg():
    import multimodal_av_model_b200 as pkg
    return pkg


def _bits(x):
    return np.float64(x).view(np.uint64)


def _random_phrases(seed, V, blank, n):
    """Random phrases over a small token set, with shared prefixes, suffixes of other phrases, duplicates with other
    weights and single-token phrases."""
    rng = np.random.default_rng(seed)
    toks = [c for c in rng.choice(V, size=min(V, 9), replace=False).tolist() if c != blank]
    out = []
    for _ in range(n):
        r = rng.random()
        w = float(rng.choice([0.5, 1.25, 2.0, 3.0, 0.1, 1.7]))
        if r < 0.25 and out:
            ids = list(out[rng.integers(len(out))][0])
            ids = ids[:rng.integers(1, len(ids) + 1)] + [int(rng.choice(toks))]      # shared prefix
        elif r < 0.45 and out:
            ids = list(out[rng.integers(len(out))][0])
            ids = ids[rng.integers(0, len(ids)):]                                     # suffix (or duplicate)
        elif r < 0.55:
            ids = [int(rng.choice(toks))]
        else:
            ids = [int(c) for c in rng.choice(toks, size=rng.integers(1, 7))]
        out.append((ids[:64], w))
    return out


@pytest.mark.parametrize("seed", range(6))
def test_dense_tables_equal_the_oracle_automaton(seed):
    pkg = _pkg()
    V, blank = 40, 3
    phrases = _random_phrases(seed, V, blank, 12 + 8 * seed)
    g = pkg.ContextGraph.from_phrases(phrases, V, blank)
    ac = CO.ContextAutomaton(phrases)
    assert g.num_nodes == ac.num_nodes
    alpha = sorted({c for ids, _ in phrases for c in ids})
    assert g.alphabet == len(alpha)
    assert g.token_sym.tolist() == [alpha.index(c) if c in alpha else -1 for c in range(V)]
    for v in range(g.num_nodes):
        assert _bits(g.node[v, 0]) == _bits(ac.phi[v]), v
        assert _bits(g.node[v, 1]) == _bits(ac.omega(v)), v
        for c in range(V):
            s = g.token_sym[c]
            assert (g.delta[v, s] if s >= 0 else 0) == ac.delta(v, c), (v, c)
    assert g.table_bytes == V * 4 + g.num_nodes * g.alphabet * 4 + g.num_nodes * 16


def test_hand_computed_ab_b_abc():
    """a = 1, b = 2, c = 3; weights ab 1.5, b 2.0, abc 0.5.  Nodes (BFS): 0 root, 1 a, 2 b, 3 ab, 4 abc.
    tau: a = max(1.5, 0.5), b = 2, ab = 1.5, abc = 0.5 -> phi: 1.5, 2, 3, 3.5.  fail: a -> 0, b -> 0, ab -> b,
    abc -> 0.  omega: a 0 (no phrase on its chain), b 2, ab 3 (ab itself ends a phrase before b), abc 3.5."""
    pkg = _pkg()
    phrases = [([1, 2], 1.5), ([2], 2.0), ([1, 2, 3], 0.5)]
    g = pkg.ContextGraph.from_phrases(phrases, 5, 0)
    assert g.token_sym.tolist() == [-1, 0, 1, 2, -1]
    assert g.node.tolist() == [[0.0, 0.0], [1.5, 0.0], [2.0, 2.0], [3.0, 3.0], [3.5, 3.5]]
    assert g.delta.tolist() == [[1, 2, 0], [1, 3, 0], [1, 2, 0], [1, 2, 4], [1, 2, 0]]
    ac = CO.ContextAutomaton(phrases)
    assert ac.fail == [0, 0, 0, 2, 0]
    # a: +1.5; b: (3 - 1.5) + 3 = 4.5; c: (3.5 - 3) + 3.5 = 4 -> G = 10, bias = 10 - 3.5 = 6.5 = ab (3) + abc (3.5)
    u, G = 0, 0.0
    for c, v, d in ((1, 1, 1.5), (2, 3, 4.5), (3, 4, 4.0)):
        u2, G2 = ac.step(u, G, c)
        assert u2 == v and G2 - G == d
        u, G = u2, G2
    assert CO.bias_of(ac, [1, 2, 3]) == 6.5
    assert CO.bias_of(ac, [1, 2]) == 3.0          # ab, not ab + b: omega credits the longest phrase ending here
    assert CO.bias_of(ac, [2]) == 2.0
    assert CO.bias_of(ac, [1]) == 0.0             # unfinished
    assert CO.bias_of(ac, [1, 4, 2]) == 2.0       # a broken by 4, then b


def test_builder_rejects_bad_input(monkeypatch):
    pkg = _pkg()
    from multimodal_av_model_b200 import context_graph as cg
    G = pkg.ContextGraph.from_phrases
    for phrases, match in [([[]], "tokens"), ([[1] * 65], "tokens"), ([[1, 9]], "outside"), ([[-1]], "outside"),
                           ([[1, 3]], "blank"), ([([1], float("nan"))], "finite"), ([([1], float("inf"))], "finite"),
                           ([([1], 0.0)], "> 0"), ([([1], -2.0)], "> 0"), ([], "empty")]:
        with pytest.raises(ValueError, match=match):
            G(phrases, 9, 3)
    with pytest.raises(ValueError, match="finite"):
        G([[1]], 9, 3, weight=float("inf"))
    assert G([[1] * 64], 9, 3).num_nodes == 65
    monkeypatch.setattr(cg, "MAX_TABLE_BYTES", 6 * 5 * 4)
    assert G([[1, 2, 4, 5, 6]], 9, 3).num_nodes == 6            # 6 nodes x 5 symbols: at the cap
    with pytest.raises(ValueError, match="bytes"):
        G([[1, 2, 4, 5, 6, 7]], 9, 3)
    monkeypatch.setattr(cg, "MAX_NODES", 4)
    with pytest.raises(ValueError, match="nodes"):
        G([[1, 2, 4, 5]], 9, 3)


def test_from_text_uses_the_tokenizer():
    pkg = _pkg()
    from multimodal_av_model_b200.synthetic import CharTokenizer
    tok = CharTokenizer(800)
    g = pkg.ContextGraph.from_text(["가나", "나다 가"], tok, weight=1.5)
    ref = pkg.ContextGraph.from_phrases([tok.encode("가나"), tok.encode("나다 가")], 800, 3, weight=1.5)
    assert g.vocab_size == 800 and g.blank == 3
    assert np.array_equal(g.delta, ref.delta) and np.array_equal(g.node, ref.node)
    with pytest.raises(TypeError):
        pkg.ContextGraph.from_text("가나", tok)


def _peaky(seq, V, blank, gap=True):
    """Log-probs that spell `seq`: each token one frame at ~0, a blank frame between tokens."""
    frames = []
    for c in seq:
        frames.append(c)
        if gap:
            frames.append(blank)
    lp = np.full((len(frames), V), -30.0, dtype=np.float32)
    for t, c in enumerate(frames):
        lp[t, c] = 0.0
    return torch.from_numpy(lp).log_softmax(-1).numpy()


def test_oracle_bias_accounting():
    V, blank = 8, 0
    phrases = [([1, 2, 3], 1.25), ([4, 5], 2.0)]
    ac = CO.ContextAutomaton(phrases)
    for seq, want in [([1, 2, 3], 3 * 1.25), ([6, 1, 2, 3, 7], 3 * 1.25), ([1, 2], 0.0), ([1, 2, 6, 3], 0.0),
                      ([4, 5, 6, 4, 5], 2 * 4.0), ([1, 2, 3, 4, 5], 3.75 + 4.0), ([4, 4, 5], 4.0)]:
        assert CO.bias_of(ac, seq) == want, seq
        st, hyps = CO.prefix_beam_bias_search(_peaky(seq, V, blank), 2 * len(seq), 3, 1, blank, ac)
        assert st == 0 and list(hyps[0][0]) == seq
        tokens, score, acoustic, lm, bias = hyps[0]
        assert bias == want and lm == 0.0 and score == (acoustic + 0.0) + bias


@pytest.mark.parametrize("blank", [0, 3])
def test_never_hit_context_reproduces_the_plain_and_lm_searches(blank):
    """Phrase tokens 14 and 15 sit far below every top-(2B+1) list: every bias is 0 and the search is §4.13 / §4.14."""
    V = 16
    vocab = ["_", "a", "b", "c"] + [f"x{i}" for i in range(V - 4)]
    arpa = LO.read_arpa(ARPA, vocab)
    phrases = [([14, 15], 2.0), ([15], 1.0)]
    for seed in range(4):
        g = torch.Generator().manual_seed(seed)
        lp = (torch.randn(14, V, generator=g, dtype=torch.float64) * 3.0)
        lp[:, 14:] -= 80.0
        lp = lp.log_softmax(-1).float().numpy()
        for B in (1, 3, 6):
            _, plain = O.prefix_beam_search(lp, 14, B, B, blank)
            st, biased = CO.prefix_beam_bias_search(lp, 14, B, B, blank, phrases)
            assert st == 0 and [t for t, *_ in biased] == [t for t, _ in plain]
            assert [_bits(a) for _, _, a, _, _ in biased] == [_bits(s) for _, s in plain]
            assert [_bits(s) for _, s, _, _, _ in biased] == [_bits(s) for _, s in plain]
            assert all(m == 0.0 and b == 0.0 for *_, m, b in biased)
            _, fused = LO.prefix_beam_lm_search(lp, 14, B, B, blank, arpa, 0.5, 0.25)
            st, both = CO.prefix_beam_bias_search(lp, 14, B, B, blank, phrases, lm=arpa, alpha=0.5, beta=0.25)
            assert [t for t, *_ in both] == [t for t, *_ in fused]
            for (_, s, a, m, b), (_, s2, a2, m2) in zip(both, fused):
                assert (_bits(s), _bits(a), _bits(m), b) == (_bits(s2), _bits(a2), _bits(m2), 0.0)


ARPA = """
\\data\\
ngram 1=6
ngram 2=3

\\1-grams:
-99\t<s>\t-0.5
-1.0\t</s>
-2.0\t<unk>
-0.7\ta\t-0.25
-0.9\tb\t-0.125
-1.25\tc

\\2-grams:
-0.2\t<s> a
-0.4\ta b
-0.6\tb </s>

\\end\\
"""


def _ctc_logprob(lp, toks, blank):
    lp64 = torch.from_numpy(lp).double()[:, None]
    tg = torch.tensor([list(toks)], dtype=torch.long) if toks else torch.zeros(1, 0, dtype=torch.long)
    return -F.ctc_loss(lp64, tg, torch.tensor([lp.shape[0]]), torch.tensor([len(toks)]), blank=blank,
                       reduction="none").item()


def test_exhaustive_hypotheses_score_ctc_plus_bias():
    """V = 3 (blank 0 + tokens 1, 2), T = 3, B = 15: nothing is pruned, so the hypotheses are the 9 feasible strings,
    each with acoustic = -ctc_loss and bias = the rule applied to its tokens, ranked by acoustic + bias."""
    phrases = [([1, 2], 1.5), ([2], 0.75), ([2, 2], 2.0), ([1, 1, 1], 0.5)]
    ac = CO.ContextAutomaton(phrases)
    g = torch.Generator().manual_seed(17)
    lp = torch.randn(3, 3, generator=g, dtype=torch.float64).log_softmax(-1).float().numpy()
    st, hyps = CO.prefix_beam_bias_search(lp, 3, 15, 15, 0, phrases, prune=False)
    assert st == 0 and len(hyps) == 9
    assert CO.prefix_beam_bias_search(lp, 3, 15, 15, 0, phrases) == (st, hyps)      # k = min(31, V) = V
    assert any(b > 0 for *_, b in hyps)
    for toks, score, acoustic, lm, bias in hyps:
        assert abs(acoustic - _ctc_logprob(lp, toks, 0)) < 1e-12
        assert lm == 0.0 and bias == CO.bias_of(ac, toks)
        assert score == (acoustic + 0.0) + bias
    assert [h[1] for h in hyps] == sorted((h[1] for h in hyps), reverse=True)


def test_length_zero_and_failures():
    lp = _peaky([1, 2], 5, 0)
    arpa = LO.read_arpa(ARPA, ["_", "a", "b", "c", "d"])
    assert CO.prefix_beam_bias_search(lp, 0, 3, 2, 0, [([1], 1.0)]) == (0, [((), 0.0, 0.0, 0.0, 0.0)])
    st, hyps = CO.prefix_beam_bias_search(lp, 0, 3, 2, 0, [([1], 1.0)], lm=arpa, alpha=0.5)
    e = 0.5 * (arpa.lm10("</s>", ("<s>",)) * LO.LN10)
    assert st == 0 and hyps == [((), (0.0 + e) + 0.0, 0.0, e, 0.0)]
    assert CO.prefix_beam_bias_search(lp, 5, 3, 2, 0, [([1], 1.0)]) == (2, [])
    bad = lp.copy()
    bad[1, 1] = np.nan
    assert CO.prefix_beam_bias_search(bad, 4, 3, 2, 0, [([1], 1.0)]) == (1, [])
    for phrases in ([([0], 1.0)], [([5], 1.0)]):
        with pytest.raises(ValueError):
            CO.prefix_beam_bias_search(lp, 4, 3, 2, 0, phrases)
    assert math.isfinite(CO.prefix_beam_bias_search(lp, 4, 3, 2, 0, [([1, 2], 1.0)])[1][0][4])


def test_search_checks_the_graph_before_any_launch():
    pkg = _pkg()
    g = pkg.ContextGraph.from_phrases([[1, 2]], 5, 0)
    with pytest.raises(RuntimeError, match="CUDA"):
        pkg.ctc_prefix_beam_search(torch.zeros(2, 3, 5), context=g)
