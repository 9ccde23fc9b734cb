"""GPU: CTC prefix beam search with contextual biasing (csrc/ctc_prefix_beam.cu, context_graph.py) — tokens, lengths
and the bits of score, acoustic_score, lm_score and bias_score equal to the CPU oracle (oracle/context_graph_oracle.py)
on padded, tie-heavy, peaky, long and V = 801 batches, without an LM and with LM orders 1..4, with phrases taken from
the greedy paths and a 10 000-phrase graph; a never-hit context against the unbiased search; statuses, batch
independence, argument errors, the launch count, a recall check and trainer.transcribe(context=...)."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import context_graph_oracle as CO
from oracle import prefix_beam_lm_oracle as LO
from test_prefix_beam_lm_gpu import _write_arpa

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _pkg():
    import multimodal_av_model_b200 as pkg
    return pkg


def _bits(x):
    return np.float64(x).view(np.uint64)


def _rand_lp(seed, N, T, V, scale=3.0):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(N, T, V, generator=g) * scale).log_softmax(-1)


def _lengths(N, T, seed):
    ln = torch.from_numpy(np.random.default_rng(seed).integers(0, T + 1, size=N))
    ln[0], ln[1] = 0, T
    return ln


def _vocab(V):
    return [f"p{i}" for i in range(V)]


def _phrases(lp, blank, seed, n_random=20, weights=(1.0, 1.5, 2.0, 3.0)):
    """Stretches of the greedy paths (so that the search meets them), their one-token-longer variants, and random
    phrases, with random per-token weights."""
    rng = np.random.default_rng(seed)
    V = lp.shape[-1]
    out = []
    for row in lp.argmax(-1).tolist():
        toks = [c for i, c in enumerate(row) if c != blank and (i == 0 or c != row[i - 1])]
        for _ in range(3):
            if len(toks) >= 1:
                a = int(rng.integers(0, len(toks)))
                ids = toks[a:a + int(rng.integers(1, 5))]
                out.append((ids, float(rng.choice(weights))))
                if rng.random() < 0.3:
                    out.append((ids + [int(rng.integers(0, V))], float(rng.choice(weights))))
    for _ in range(n_random):
        out.append(([int(c) for c in rng.integers(0, V, size=int(rng.integers(1, 6)))], float(rng.choice(weights))))
    return [(ids, w) for ids, w in out if blank not in ids]


def _graphs(phrases, V, blank):
    return _pkg().ContextGraph.from_phrases(phrases, V, blank), CO.ContextAutomaton(phrases)


def _lms(tmp_path, V, order, seed, lp, blank):
    if order == 0:
        return None, None
    p = _write_arpa(tmp_path / "lm.arpa", _vocab(V), order, seed, lp=lp, blank=blank)
    return _pkg().NgramLM.from_arpa(str(p), _vocab(V)), LO.read_arpa(str(p), _vocab(V))


def _check(got, lp, lengths, B, nbest, blank, ac, olm, alpha, beta, rows=None):
    lp = lp.float().cpu().numpy()
    rows = range(lp.shape[0]) if rows is None else rows
    for i, n in enumerate(rows):
        st, ref = CO.prefix_beam_bias_search(lp[n], int(lengths[n]), B, nbest, blank, ac, lm=olm, alpha=alpha,
                                             beta=beta)
        assert st == 0
        assert [h.tokens for h in got[i]] == [list(r[0]) for r in ref], (n, B)
        for f, j in (("score", 1), ("acoustic_score", 2), ("lm_score", 3), ("bias_score", 4)):
            assert [_bits(getattr(h, f)) for h in got[i]] == [_bits(r[j]) for r in ref], (n, B, f)


@pytest.mark.parametrize("B, order", [(1, 0), (5, 0), (10, 0), (15, 0), (1, 1), (5, 2), (10, 3), (15, 4)])
def test_padded_batch_bit_exact(tmp_path, B, order):
    pkg = _pkg()
    N, T, V, blank = 16, 60, 800, 3
    lp = _rand_lp(B + 7 * order, N, T, V)
    ln = _lengths(N, T, B)
    g, ac = _graphs(_phrases(lp, blank, B + order), V, blank)
    lm, olm = _lms(tmp_path, V, order, B * 10 + order, lp, blank)
    got = pkg.ctc_prefix_beam_search(lp.to(DEV), ln.to(DEV), beam_width=B, nbest=B, blank=blank, lm=lm,
                                     lm_weight=0.5, token_bonus=0.5, context=g)
    assert all(type(h) is pkg.BiasedHypothesis for row in got for h in row)
    _check(got, lp, ln, B, B, blank, ac, olm, 0.5, 0.5)
    assert any(h.bias_score > 0 for row in got for h in row)
    assert len(got[0]) == 1 and got[0][0].tokens == [] and got[0][0].bias_score == 0.0
    if order == 0:
        assert all(h.lm_score == 0.0 for row in got for h in row)
    top = pkg.ctc_prefix_beam_search(lp.to(DEV), ln.to(DEV), beam_width=B, nbest=1, blank=blank, lm=lm,
                                     lm_weight=0.5, token_bonus=0.5, context=g)
    assert [h[:1] for h in got] == top


@pytest.mark.parametrize("quant, order", [(0.5, 0), (2.0, 3)])
def test_tie_heavy_input(tmp_path, quant, order):
    pkg = _pkg()
    N, T, V, blank, B = 16, 40, 40, 3, 6
    lp = torch.round(_rand_lp(11, N, T, V, scale=1.0) * quant) / quant
    ln = _lengths(N, T, 12)
    g, ac = _graphs(_phrases(lp, blank, 3, weights=(1.0, 2.0)), V, blank)
    lm, olm = _lms(tmp_path, V, order, 5, lp, blank)
    got = pkg.ctc_prefix_beam_search(lp.to(DEV), ln, beam_width=B, nbest=B, blank=blank, lm=lm, lm_weight=1.0,
                                     context=g)
    _check(got, lp, ln, B, B, blank, ac, olm, 1.0, 0.0)


@pytest.mark.parametrize("order", [0, 4])
def test_peaky_log_probs(tmp_path, order):
    pkg = _pkg()
    N, T, V, blank, B = 16, 100, 800, 3, 10
    g = torch.Generator().manual_seed(3)
    logits = torch.randn(N, T, V, generator=g)
    logits[:, :, blank] += 12.0
    burst = torch.rand(N, T, generator=g) < 0.15
    tok = torch.randint(0, V, (N, T), generator=g)
    logits[burst, tok[burst]] += 20.0
    lp = logits.log_softmax(-1)
    ln = _lengths(N, T, 4)
    cg, ac = _graphs(_phrases(lp, blank, 4), V, blank)
    lm, olm = _lms(tmp_path, V, order, 6, lp, blank)
    got = pkg.ctc_prefix_beam_search(lp.to(DEV), ln, beam_width=B, nbest=B, blank=blank, lm=lm, lm_weight=0.3,
                                     token_bonus=1.5, context=cg)
    _check(got, lp, ln, B, B, blank, ac, olm, 0.3, 1.5)


@pytest.mark.parametrize("order", [0, 2])
def test_vocab_801_blank_0(tmp_path, order):
    pkg = _pkg()
    N, T, V, B = 16, 60, 801, 10
    lp = _rand_lp(5, N, T, V)
    ln = _lengths(N, T, 5)
    g, ac = _graphs(_phrases(lp, 0, 5) + [([800], 2.5), ([800, 799], 1.0)], V, 0)
    lm, olm = _lms(tmp_path, V, order, 7, lp, 0)
    got = pkg.ctc_prefix_beam_search(lp.to(DEV), ln, beam_width=B, nbest=3, blank=0, lm=lm, lm_weight=1.0,
                                     token_bonus=-0.5, context=g)
    _check(got, lp, ln, B, 3, 0, ac, olm, 1.0, -0.5)


@pytest.mark.parametrize("order", [0, 3])
def test_long_utterances_trie_in_workspace(tmp_path, order):
    pkg = _pkg()
    N, T, V, B = 3, 1000, 801, 5
    lp = _rand_lp(6, N, T, V)
    ln = torch.tensor([1000, 731, 0])
    g, ac = _graphs(_phrases(lp, 3, 6), V, 3)
    lm, olm = _lms(tmp_path, V, order, 8, lp, 3)
    got = pkg.ctc_prefix_beam_search(lp.to(DEV), ln, beam_width=B, nbest=B, blank=3, lm=lm, lm_weight=0.3,
                                     context=g)
    _check(got, lp, ln, B, B, 3, ac, olm, 0.3, 0.0)


def test_ten_thousand_phrases(tmp_path):
    pkg = _pkg()
    N, T, V, B, blank = 8, 80, 800, 8, 3
    lp = _rand_lp(21, N, T, V)
    ln = _lengths(N, T, 21)
    rng = np.random.default_rng(21)
    phrases = _phrases(lp, blank, 21)
    phrases += [([int(c) for c in rng.integers(4, V, size=int(rng.integers(2, 13)))],
                 float(rng.choice([1.0, 2.0]))) for _ in range(10_000 - len(phrases))]
    g, ac = _graphs(phrases, V, blank)
    assert g.table_bytes > 126 * 2 ** 20                  # above the B200's L2
    for order in (0, 2):
        lm, olm = _lms(tmp_path, V, order, 9, lp, blank)
        got = pkg.ctc_prefix_beam_search(lp.to(DEV), ln, beam_width=B, nbest=4, blank=blank, lm=lm, lm_weight=0.5,
                                         context=g)
        _check(got, lp, ln, B, 4, blank, ac, olm, 0.5, 0.0)


@pytest.mark.parametrize("B, order", [(1, 0), (10, 0), (10, 3)])
def test_never_hit_context_equals_the_unbiased_search(tmp_path, B, order):
    pkg = _pkg()
    N, T, V, blank = 24, 80, 800, 3
    lp = _rand_lp(30 + B, N, T, V)
    lp[:, :, 790:] -= 60.0                                # never in a top-(2B+1) list
    lp = lp.log_softmax(-1).to(DEV)
    ln = _lengths(N, T, 31).to(DEV)
    g = pkg.ContextGraph.from_phrases([[790, 791], [795], ([799, 798, 797], 3.0)], V, blank)
    lm, _ = _lms(tmp_path, V, order, 9, lp.cpu(), blank)
    plain = pkg.ctc_prefix_beam_search(lp, ln, beam_width=B, nbest=B, blank=blank, lm=lm, lm_weight=0.5)
    biased = pkg.ctc_prefix_beam_search(lp, ln, beam_width=B, nbest=B, blank=blank, lm=lm, lm_weight=0.5, context=g)
    for p_row, b_row in zip(plain, biased):
        assert [h.tokens for h in p_row] == [h.tokens for h in b_row]
        acoustic = [h.score for h in p_row] if lm is None else [h.acoustic_score for h in p_row]
        assert [_bits(a) for a in acoustic] == [_bits(h.acoustic_score) for h in b_row]
        if lm is not None:
            assert [_bits(h.lm_score) for h in p_row] == [_bits(h.lm_score) for h in b_row]
        assert [_bits(h.score) for h in p_row] == [_bits(h.score) for h in b_row]
        assert all(h.bias_score == 0.0 for h in b_row)


def _raw(g, lp, ln, B, nbest, blank, lm=None, alpha=0.5, beta=0.0, null_ctx=False, **desc):
    pkg = _pkg()
    L = pkg._lib.lib()
    N, T, V = lp.shape
    ws_bytes = int(L.avctc_ctc_prefix_beam_workspace_bytes(N, T, V, B))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=DEV)
    tok = torch.full((N, nbest, T), -7, dtype=torch.int32, device=DEV)
    olen = torch.full((N, nbest), -7, dtype=torch.int32, device=DEV)
    osc = torch.zeros((4, N, nbest), dtype=torch.float64, device=DEV)
    st = torch.full((N,), -7, dtype=torch.int32, device=DEV)
    d = pkg._lib.ContextGraphDesc.from_buffer_copy(g.descriptor(lp.device))
    for k, v in desc.items():
        setattr(d, k, v)
    ld = pkg._lib.NgramLMDesc.from_buffer_copy(lm.descriptor(lp.device)) if lm is not None else None
    rc = L.avctc_ctc_prefix_beam_biased(lp.data_ptr(), lp.stride(0), lp.stride(1), N, T, V, ln.data_ptr(), B, nbest,
                                        blank, ctypes.addressof(ld) if ld is not None else None, alpha, beta,
                                        None if null_ctx else ctypes.addressof(d),
                                        tok.data_ptr(), olen.data_ptr(), osc[0].data_ptr(), osc[1].data_ptr(),
                                        osc[2].data_ptr(), osc[3].data_ptr(), st.data_ptr(), ws.data_ptr(), ws_bytes,
                                        pkg._lib.stream_ptr(lp.device))
    torch.cuda.synchronize()
    return rc, tok.cpu(), olen.cpu(), osc.cpu(), st.cpu()


def test_batch_independence_statuses_and_errors(tmp_path):
    pkg = _pkg()
    N, T, V, B, nbest = 6, 50, 100, 5, 3
    lp = _rand_lp(8, N, T, V)
    g, ac = _graphs(_phrases(lp, 3, 8), V, 3)
    lm, olm = _lms(tmp_path, V, 3, 10, lp, 3)
    lp[2, 17, 40] = float("nan")
    ln = torch.tensor([50, 40, 50, 51, -1, 10])
    lpd, lnd = lp.to(DEV), ln.to(DEV)
    for use_lm in (None, lm):
        rc, tok, olen, osc, st = _raw(g, lpd, lnd, B, nbest, 3, lm=use_lm, alpha=0.5, beta=0.2)
        assert rc == 0 and st.tolist() == [0, 0, 1, 2, 2, 0]
        for n in (2, 3, 4):
            assert (olen[n] == 0).all() and (osc[:, n] == -np.inf).all()
        good = [0, 1, 5]
        hyps = [[pkg.BiasedHypothesis(tok[n, i, :olen[n, i]].tolist(), *(float(osc[j, n, i]) for j in range(4)))
                 for i in range(nbest) if osc[0, n, i] > -np.inf] for n in good]
        _check(hyps, lp, ln, B, nbest, 3, ac, olm if use_lm is not None else None, 0.5, 0.2, rows=good)
    kw = dict(beam_width=B, nbest=nbest, blank=3, lm=lm, lm_weight=0.5, token_bonus=0.2, context=g)
    with pytest.raises(RuntimeError, match="utterance 2: .*NaN"):
        pkg.ctc_prefix_beam_search(lpd, lnd, **kw)
    with pytest.raises(RuntimeError, match="utterance 1: length 51 outside"):
        pkg.ctc_prefix_beam_search(lpd[[0, 3]], lnd[[0, 3]], **kw)
    sel = [5, 0, 1]
    for lm_ in (None, lm):
        kw["lm"] = lm_
        full = pkg.ctc_prefix_beam_search(lpd[sel], lnd[sel], **kw)
        for i, n in enumerate(sel):
            assert pkg.ctc_prefix_beam_search(lpd[n:n + 1], lnd[n:n + 1], **kw) == [full[i]]
    # C-level argument errors, before any launch
    for desc in ({"num_nodes": 0}, {"map_len": V - 1}, {"alphabet": 0}, {"alphabet": V + 1}, {"null_ctx": True}):
        rc, _, olen, _, st = _raw(g, lpd, lnd, B, nbest, 3, **desc)
        assert rc == -1 and (st == -7).all() and (olen == -7).all(), desc
    assert _raw(g, lpd, lnd, B, nbest, 3, lm=lm, alpha=-0.5)[0] == -1
    assert _raw(g, lpd, lnd, B, nbest, 3, lm=lm, beta=float("nan"))[0] == -1


def test_argument_errors_and_launch_count(tmp_path):
    pkg = _pkg()
    lp = _rand_lp(9, 4, 20, 30).to(DEV)
    g = pkg.ContextGraph.from_phrases([[1, 2], [5]], 30, 0)
    other_v = pkg.ContextGraph.from_phrases([[1, 2]], 31, 0)
    other_blank = pkg.ContextGraph.from_phrases([[1, 2]], 30, 3)
    bad = [({"context": other_v}, ValueError), ({"context": other_blank}, ValueError),
           ({"context": [[1, 2]]}, TypeError), ({"context": g, "beam_width": 16}, ValueError),
           ({"context": g, "blank": 30}, ValueError), ({"context": g, "lm": "x.arpa"}, TypeError)]
    for kw, exc in bad:
        before = pkg._lib.launch_count
        with pytest.raises(exc):
            pkg.ctc_prefix_beam_search(lp, **kw)
        assert pkg._lib.launch_count == before
    before = pkg._lib.launch_count
    pkg.ctc_prefix_beam_search(lp, beam_width=5, context=g)
    assert pkg._lib.launch_count - before == 2


def test_biasing_recovers_a_planted_phrase():
    """Each utterance says filler tokens around the phrase 5 6 7, but at the phrase's middle token the confusable
    token 16 scores slightly higher than 6: the unbiased search returns 5 16 7, the biased one the phrase, with a
    bias of exactly its sum of per-token weights (3 x 2.0)."""
    pkg = _pkg()
    rng = np.random.default_rng(0)
    V, blank, N = 20, 0, 12
    fillers = [1, 2, 3, 4, 8, 9, 10, 11, 12]
    refs, logits = [], []
    for _ in range(N):
        a = [int(c) for c in rng.choice(fillers, size=int(rng.integers(1, 5)))]
        b = [int(c) for c in rng.choice(fillers, size=int(rng.integers(1, 5)))]
        seq = a + [5, 6, 7] + b
        x = np.full((3 * len(seq), V), -8.0, dtype=np.float32)
        for i, c in enumerate(seq):
            for f in (3 * i, 3 * i + 1):
                x[f, c] = 4.0
                if c == 6 and i == len(a) + 1:
                    x[f, 16] = 4.0 + float(rng.uniform(0.2, 0.5))
            x[3 * i + 2, blank] = 5.0
        refs.append(seq)
        logits.append(x)
    T = max(len(x) for x in logits)
    lp = torch.full((N, T, V), -8.0)
    lp[:, :, blank] = 5.0
    for n, x in enumerate(logits):
        lp[n, :len(x)] = torch.from_numpy(x)
    lp = lp.log_softmax(-1)
    ln = torch.tensor([len(x) for x in logits])
    g = pkg.ContextGraph.from_phrases([[5, 6, 7]], V, blank, weight=2.0)
    plain = pkg.ctc_prefix_beam_search(lp.to(DEV), ln.to(DEV), beam_width=5, blank=blank)
    biased = pkg.ctc_prefix_beam_search(lp.to(DEV), ln.to(DEV), beam_width=5, blank=blank, context=g)
    for n, seq in enumerate(refs):
        conf = [16 if c == 6 else c for c in seq]
        assert plain[n][0].tokens == conf
        assert biased[n][0].tokens == seq and biased[n][0].bias_score == 6.0
    _check(biased, lp, ln, 5, 1, blank, CO.ContextAutomaton([([5, 6, 7], 2.0)]), None, 0.5, 0.0)


def _tiny_models(pkg):
    from multimodal_av_model_b200.encoders import unfreeze_middle_layers, xlsr_large_config
    cfg = xlsr_large_config(hidden_size=64, num_hidden_layers=10, num_attention_heads=4, intermediate_size=128,
                            conv_dim=(32,) * 7, num_conv_pos_embeddings=16, num_conv_pos_embedding_groups=4)
    torch.manual_seed(0)
    vis = pkg.VisualEncoder()
    for prm in vis.parameters():
        prm.requires_grad = False
    aud = pkg.AudioEncoder(freeze=True, config=cfg)
    unfreeze_middle_layers(aud.model)
    return vis, aud, pkg.CrossAttentionFusion(512, 64, 64), pkg.CTCDecoder(128, 800, blank_id=3)


def test_trainer_transcribe_with_context():
    pkg = _pkg()
    from multimodal_av_model_b200.synthetic import CharTokenizer, make_batch
    tok = CharTokenizer(800)
    tr = pkg.MultimodalTrainer(*_tiny_models(pkg), tok, device="cuda")
    batch = make_batch(pairs=2, seconds=2.0, t_v=60, seed=5, l_range=(4, 12))
    plain = tr.transcribe(batch, beam_width=5, nbest=3)
    chars = [ch for spk in plain for row in spk for t, _ in row[:1] for ch in t if 0xAC00 <= ord(ch) < 0xAC00 + 795]
    assert chars
    phrases = [chars[0], chars[-1] + chars[0]]
    biased = tr.transcribe(batch, beam_width=5, nbest=3, context=phrases)
    again = tr.transcribe(batch, beam_width=5, nbest=3, context=pkg.ContextGraph.from_text(phrases, tok))
    assert biased == again and len(biased) == 2
    for spk in biased:
        for row in spk:
            scores = [s for _, s in row]
            assert 1 <= len(row) <= 3 and all(type(s) is float and isinstance(t, str) for t, s in row)
            assert scores == sorted(scores, reverse=True)
    assert any(sb != sp for spk_p, spk_b in zip(plain, biased) for hp, hb in zip(spk_p, spk_b)
               for (_, sp), (_, sb) in zip(hp, hb))
