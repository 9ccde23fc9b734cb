"""CPU: the prefix beam search oracle (oracle/prefix_beam_oracle.py) — log_add against numpy, the 2B+1 pruning against
the unpruned search, every hypothesis against the CTC loss, repeats against blank-separated repeats — and the
workspace query of avctc_ctc_prefix_beam."""
import itertools
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import prefix_beam_oracle as O


def _rand_lp(seed, T, V, scale=2.0):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(T, V, generator=g, dtype=torch.float64) * scale).log_softmax(-1).float().numpy()


def test_log_add_matches_numpy():
    rng = np.random.default_rng(0)
    a = rng.uniform(-80, 10, 20000)
    b = a + np.concatenate([rng.uniform(-60, 60, 15000), rng.uniform(-800, 800, 5000)])
    ours = np.array([O.log_add(x, y) for x, y in zip(a, b)])
    ref = np.logaddexp(a, b)
    ulp = np.spacing(np.maximum(np.abs(a), np.abs(b)))
    assert (np.abs(ours - ref) <= 4 * ulp).all()
    # tiny results: relative accuracy where no cancellation happens
    assert O.log_add(0.0, -50.0) == pytest.approx(np.logaddexp(0.0, -50.0), rel=1e-15)
    assert O.log_add(-1e-3, -1e-3) == pytest.approx(np.logaddexp(-1e-3, -1e-3), rel=4e-16)


def test_log_add_infinities_and_large_gaps():
    inf = math.inf
    assert O.log_add(-inf, -inf) == -inf
    assert O.log_add(-inf, 2.5) == 2.5 and O.log_add(2.5, -inf) == 2.5
    assert O.log_add(inf, 1.0) == inf and O.log_add(1.0, inf) == inf and O.log_add(inf, inf) == inf
    assert O.log_add(0.0, -709.0) == 0.0 and O.log_add(-3.0, -1000.0) == -3.0
    assert O.log_add(-7.0, -7.0) == pytest.approx(-7.0 + math.log(2.0), abs=2e-15)
    assert O.log_add(1.0, 2.0) == O.log_add(2.0, 1.0)


@pytest.mark.parametrize("blank", ["first", "three", "last"])
def test_pruned_equals_unpruned(blank):
    for seed in range(4):
        T, V = 14, 40
        b = {"first": 0, "three": 3, "last": V - 1}[blank]
        lp = _rand_lp(seed, T, V, scale=3.0)
        for B in (1, 2, 4, 7):
            assert O.prefix_beam_search(lp, T, B, B, b) == O.prefix_beam_search(lp, T, B, B, b, prune=False), (seed, B)


def _ctc_logprob(lp, toks, blank):
    lp64 = torch.from_numpy(lp).double()[:, None]
    tg = torch.tensor([list(toks)], dtype=torch.long) if toks else torch.zeros(1, 0, dtype=torch.long)
    return -F.ctc_loss(lp64, tg, torch.tensor([lp.shape[0]]), torch.tensor([len(toks)]), blank=blank,
                       reduction="none").item()


def _feasible(T, labels):
    out = []
    for L in range(T + 1):
        for s in itertools.product(labels, repeat=L):
            if L + sum(1 for x, y in zip(s, s[1:]) if x == y) <= T:
                out.append(s)
    return out


@pytest.mark.parametrize("blank", [0, 1, 2])
def test_exhaustive_hypotheses_score_the_ctc_loss(blank):
    """V = 3, T = 3, B = 15: the beam never drops a prefix, so the hypotheses are exactly the 9 strings with finite CTC
    likelihood, each scoring -ctc_loss in fp64."""
    lp = _rand_lp(7 + blank, 3, 3, scale=1.0)
    st, hyps = O.prefix_beam_search(lp, 3, 15, 15, blank)
    assert st == 0
    labels = [c for c in range(3) if c != blank]
    assert sorted(h[0] for h in hyps) == sorted(_feasible(3, labels)) and len(hyps) == 9
    for toks, score in hyps:
        assert abs(score - _ctc_logprob(lp, toks, blank)) < 1e-12
    assert [h[1] for h in hyps] == sorted((h[1] for h in hyps), reverse=True)


def test_repeat_needs_a_blank_between():
    """'a a' over two frames is one 'a'; 'a _ a' is 'a a'.  Class 0 = blank, 1 = a, 2 = b; B = 15 keeps every prefix,
    so every score is the full CTC likelihood."""
    hi, lo = math.log(0.9), math.log(0.05)
    aa = np.array([[lo, hi, lo], [lo, hi, lo]], dtype=np.float32)
    st, hyps = O.prefix_beam_search(aa, 2, 15, 15, 0)
    assert st == 0 and hyps[0][0] == (1,)
    assert abs(hyps[0][1] - _ctc_logprob(aa, (1,), 0)) < 1e-12
    assert (1, 1) not in dict(hyps)        # two frames cannot hold a, blank, a
    a_a = np.array([[lo, hi, lo], [hi, lo, lo], [lo, hi, lo]], dtype=np.float32)
    st, hyps = O.prefix_beam_search(a_a, 3, 15, 15, 0)
    assert st == 0 and hyps[0][0] == (1, 1)
    for toks, score in hyps:
        assert abs(score - _ctc_logprob(a_a, toks, 0)) < 1e-12


def test_lengths_and_nan():
    lp = _rand_lp(1, 5, 6)
    assert O.prefix_beam_search(lp, 0, 3, 2, 0) == (0, [((), 0.0)])
    assert O.prefix_beam_search(lp, -1, 3, 2, 0) == (2, [])
    assert O.prefix_beam_search(lp, 6, 3, 2, 0) == (2, [])
    bad = lp.copy()
    bad[3, 4] = np.nan
    assert O.prefix_beam_search(bad, 5, 3, 2, 0) == (1, [])
    assert O.prefix_beam_search(bad, 3, 3, 2, 0)[0] == 0          # the NaN frame is past the length


def test_workspace_query():
    import multimodal_av_model_b200 as pkg
    if not __import__("os").path.exists(pkg._lib.LIB_PATH):
        import __graft_entry__
        __graft_entry__.build()
    lib = pkg._lib.lib()
    assert lib.avctc_ctc_prefix_beam_workspace_bytes(16, 150, 800, 5) > 0
    assert lib.avctc_ctc_prefix_beam_workspace_bytes(16, 150, 800, 15) > 0
    assert lib.avctc_ctc_prefix_beam_workspace_bytes(16, 150, 800, 16) == 0
    assert lib.avctc_ctc_prefix_beam_workspace_bytes(16, 150, 1025, 5) == 0
    assert lib.avctc_ctc_prefix_beam_workspace_bytes(16, 150, 1024, 5) > 0
    assert lib.avctc_ctc_prefix_beam_workspace_bytes(16, 150, 800, 0) == 0
    # the [N,T,2B+1] top-k lists dominate: values and classes, 4 bytes each
    ws = lib.avctc_ctc_prefix_beam_workspace_bytes(4096, 150, 800, 10)
    assert ws >= 2 * 4096 * 150 * 21 * 4


def test_argument_errors_raise_before_any_launch():
    import multimodal_av_model_b200 as pkg
    lp = torch.zeros(2, 3, 5)
    with pytest.raises(RuntimeError, match="CUDA"):
        pkg.ctc_prefix_beam_search(lp)
