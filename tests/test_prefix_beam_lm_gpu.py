"""GPU: CTC prefix beam search with n-gram LM fusion (csrc/ctc_prefix_beam.cu, ngram_lm.py) — tokens, lengths and the
bits of score, acoustic_score and lm_score equal to the CPU oracle (oracle/prefix_beam_lm_oracle.py) on padded,
tie-heavy, peaky, long and V = 801 batches with LM orders 1..5; alpha = beta = 0 against the plain search; statuses,
argument errors, the launch count, a token-error-rate check and trainer.transcribe(lm=...)."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import prefix_beam_lm_oracle as LO

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


def _write_arpa(path, vocab, order, seed, lp=None, blank=3):
    """A random unnormalised token LM: 85 % of the pieces (the rest read as <unk>), and of each order a random subset
    of the n-grams along the greedy paths of `lp` plus random ones, so that hits, back-offs and absent contexts all
    occur.  Some n-grams use a word that is no model piece ("zz"): the loaders drop them."""
    rng = np.random.default_rng(seed)
    words = [w for w in vocab if rng.random() < 0.85] + ["zz"]
    grams = {1: {(w,) for w in words} | {("<s>",), ("</s>",), ("<unk>",)}}
    seqs = []
    if lp is not None:
        for row in lp.argmax(-1).tolist():
            toks = [c for i, c in enumerate(row) if c != blank and (i == 0 or c != row[i - 1])]
            seqs.append(["<s>"] + [vocab[c] if (vocab[c],) in grams[1] else "<unk>" for c in toks] + ["</s>"])
    for _ in range(40):
        seqs.append(["<s>"] + [words[i] for i in rng.integers(0, len(words), size=12)] + ["</s>"])
    for n in range(2, order + 1):
        g = set()
        for s in seqs:
            for i in range(len(s) - n + 1):
                if rng.random() < 0.6:
                    g.add(tuple(s[i:i + n]))
        grams[n] = g
    lines = ["\\data\\"] + [f"ngram {n}={len(grams[n])}" for n in range(1, order + 1)] + [""]
    for n in range(1, order + 1):
        lines.append(f"\\{n}-grams:")
        for ws in sorted(grams[n]):
            lp10 = -99.0 if ws == ("<s>",) else rng.uniform(-3.0, -0.05)
            s = f"{lp10:.6f}\t{' '.join(ws)}"
            if n < order and rng.random() < 0.7:
                s += f"\t{rng.uniform(-1.0, 0.3):.6f}"
            lines.append(s)
        lines.append("")
    lines.append("\\end\\")
    path.write_text("\n".join(lines) + "\n", encoding="utf-8")
    return path


def _lms(tmp_path, V, order, seed, lp=None, blank=3, name="lm.arpa"):
    p = _write_arpa(tmp_path / name, _vocab(V), order, seed, lp=lp, blank=blank)
    return _pkg().NgramLM.from_arpa(str(p), _vocab(V)), LO.read_arpa(str(p), _vocab(V))


def _check(got, lp, lengths, B, nbest, blank, olm, alpha, beta, rows=None):
    lp = lp.float().cpu().numpy()
    rows = range(lp.shape[0]) if rows is None else rows
    for i, n in enumerate(rows):
        st, ref = LO.prefix_beam_lm_search(lp[n], int(lengths[n]), B, nbest, blank, olm, alpha, beta)
        assert st == 0
        assert [h.tokens for h in got[i]] == [list(r[0]) for r in ref], (n, B)
        assert [_bits(h.score) for h in got[i]] == [_bits(r[1]) for r in ref], (n, B)
        assert [_bits(h.acoustic_score) for h in got[i]] == [_bits(r[2]) for r in ref], (n, B)
        assert [_bits(h.lm_score) for h in got[i]] == [_bits(r[3]) for r in ref], (n, B)


@pytest.mark.parametrize("B, order, alpha, beta", [(1, 1, 0.3, 0.0), (5, 2, 1.0, -0.5), (10, 3, 0.3, 1.5),
                                                   (15, 4, 1.0, 0.0), (15, 5, 0.3, -0.5), (5, 5, 1.0, 1.5)])
def test_padded_batch_bit_exact(tmp_path, B, order, alpha, beta):
    pkg = _pkg()
    N, T, V, blank = 16, 60, 800, 3
    lp = _rand_lp(B + order, N, T, V)
    ln = _lengths(N, T, B)
    lm, olm = _lms(tmp_path, V, order, B * 10 + order, lp=lp, blank=blank)
    assert lm.order == order and olm.order == order
    assert any(olm.word(c) == "<unk>" for c in range(V))
    got = pkg.ctc_prefix_beam_search(lp.to(DEV), ln.to(DEV), beam_width=B, nbest=B, blank=blank, lm=lm,
                                     lm_weight=alpha, token_bonus=beta)
    assert all(isinstance(h, pkg.LMHypothesis) for row in got for h in row)
    _check(got, lp, ln, B, B, blank, olm, alpha, beta)
    assert len(got[0]) == 1 and got[0][0].tokens == [] and got[0][0].acoustic_score == 0.0
    top = pkg.ctc_prefix_beam_search(lp.to(DEV), ln.to(DEV), beam_width=B, nbest=1, blank=blank, lm=lm,
                                     lm_weight=alpha, token_bonus=beta)
    assert [h[:1] for h in got] == top


@pytest.mark.parametrize("quant", [0.5, 2.0])
def test_tie_heavy_input(tmp_path, quant):
    pkg = _pkg()
    N, T, V, blank, B = 16, 40, 40, 3, 6
    lp = torch.round(_rand_lp(11, N, T, V, scale=1.0) * quant) / quant
    ln = _lengths(N, T, 12)
    lm, olm = _lms(tmp_path, V, 3, 5, lp=lp, blank=blank)
    got = pkg.ctc_prefix_beam_search(lp.to(DEV), ln, beam_width=B, nbest=B, blank=blank, lm=lm, lm_weight=1.0,
                                     token_bonus=0.0)
    _check(got, lp, ln, B, B, blank, olm, 1.0, 0.0)


def test_peaky_log_probs(tmp_path):
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
    lm, olm = _lms(tmp_path, V, 4, 6, lp=lp, blank=blank)
    got = pkg.ctc_prefix_beam_search(lp.to(DEV), ln, beam_width=B, nbest=B, blank=blank, lm=lm, lm_weight=0.3,
                                     token_bonus=1.5)
    _check(got, lp, ln, B, B, blank, olm, 0.3, 1.5)


def test_vocab_801_blank_0(tmp_path):
    pkg = _pkg()
    N, T, V, B = 16, 60, 801, 10
    lp = _rand_lp(5, N, T, V)
    ln = _lengths(N, T, 5)
    lm, olm = _lms(tmp_path, V, 3, 7, lp=lp, blank=0)
    got = pkg.ctc_prefix_beam_search(lp.to(DEV), ln, beam_width=B, nbest=3, blank=0, lm=lm, lm_weight=1.0,
                                     token_bonus=-0.5)
    _check(got, lp, ln, B, 3, 0, olm, 1.0, -0.5)


def test_long_utterances_trie_in_workspace(tmp_path):
    pkg = _pkg()
    N, T, V, B = 3, 1000, 801, 5
    lp = _rand_lp(6, N, T, V)
    ln = torch.tensor([1000, 731, 0])
    lm, olm = _lms(tmp_path, V, 4, 8, lp=lp, blank=3)
    got = pkg.ctc_prefix_beam_search(lp.to(DEV), ln, beam_width=B, nbest=B, blank=3, lm=lm, lm_weight=0.3,
                                     token_bonus=0.0)
    _check(got, lp, ln, B, B, 3, olm, 0.3, 0.0)


@pytest.mark.parametrize("B", [1, 10])
def test_zero_weights_equal_the_plain_search(tmp_path, B):
    pkg = _pkg()
    N, T, V, blank = 24, 80, 800, 3
    lp = _rand_lp(30 + B, N, T, V).to(DEV)
    ln = _lengths(N, T, 31).to(DEV)
    lm, _ = _lms(tmp_path, V, 3, 9, lp=lp.cpu(), blank=blank)
    plain = pkg.ctc_prefix_beam_search(lp, ln, beam_width=B, nbest=B, blank=blank)
    fused = pkg.ctc_prefix_beam_search(lp, ln, beam_width=B, nbest=B, blank=blank, lm=lm, lm_weight=0.0,
                                       token_bonus=0.0)
    for p_row, f_row in zip(plain, fused):
        assert [h.tokens for h in p_row] == [h.tokens for h in f_row]
        assert [_bits(h.score) for h in p_row] == [_bits(h.score) for h in f_row]
        assert [_bits(h.score) for h in p_row] == [_bits(h.acoustic_score) for h in f_row]
        assert all(h.lm_score == 0.0 for h in f_row)


def _raw(lm, lp, ln, B, nbest, blank, alpha, beta, order=None, map_len=None):
    pkg = _pkg()
    L = pkg._lib.lib()
    N, T, V = lp.shape
    ws_bytes = int(L.avctc_ctc_prefix_beam_workspace_bytes(N, T, V, B))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=DEV)
    tok = torch.full((N, nbest, T), -7, dtype=torch.int32, device=DEV)
    olen = torch.full((N, nbest), -7, dtype=torch.int32, device=DEV)
    osc = torch.zeros((3, N, nbest), dtype=torch.float64, device=DEV)
    st = torch.full((N,), -7, dtype=torch.int32, device=DEV)
    d = pkg._lib.NgramLMDesc.from_buffer_copy(lm.descriptor(lp.device))
    if order is not None:
        d.order = order
    if map_len is not None:
        d.map_len = map_len
    rc = L.avctc_ctc_prefix_beam_lm(lp.data_ptr(), lp.stride(0), lp.stride(1), N, T, V, ln.data_ptr(), B, nbest,
                                    blank, ctypes.addressof(d), alpha, beta, tok.data_ptr(), olen.data_ptr(),
                                    osc[0].data_ptr(), osc[1].data_ptr(), osc[2].data_ptr(), st.data_ptr(),
                                    ws.data_ptr(), ws_bytes, pkg._lib.stream_ptr(lp.device))
    torch.cuda.synchronize()
    return rc, tok.cpu(), olen.cpu(), osc.cpu(), st.cpu()


def test_batch_independence_statuses_and_errors(tmp_path):
    pkg = _pkg()
    N, T, V, B, nbest = 6, 50, 100, 5, 3
    lp = _rand_lp(8, N, T, V)
    lm, olm = _lms(tmp_path, V, 3, 10, lp=lp, blank=3)
    lp[2, 17, 40] = float("nan")
    ln = torch.tensor([50, 40, 50, 51, -1, 10])
    lpd, lnd = lp.to(DEV), ln.to(DEV)
    rc, tok, olen, osc, st = _raw(lm, lpd, lnd, B, nbest, 3, 0.5, 0.2)
    assert rc == 0 and st.tolist() == [0, 0, 1, 2, 2, 0]
    for n in (2, 3, 4):
        assert (olen[n] == 0).all() and (osc[:, n] == -np.inf).all()
    good = [0, 1, 5]
    hyps = [[pkg.LMHypothesis(tok[n, i, :olen[n, i]].tolist(), float(osc[0, n, i]), float(osc[1, n, i]),
                              float(osc[2, n, i])) for i in range(nbest) if osc[0, n, i] > -np.inf] for n in good]
    _check(hyps, lp, ln, B, nbest, 3, olm, 0.5, 0.2, rows=good)
    kw = dict(beam_width=B, nbest=nbest, blank=3, lm=lm, lm_weight=0.5, token_bonus=0.2)
    with pytest.raises(RuntimeError, match="utterance 2: .*NaN"):
        pkg.ctc_prefix_beam_search(lpd, lnd, **kw)
    with pytest.raises(RuntimeError, match="utterance 1: length 51 outside"):
        pkg.ctc_prefix_beam_search(lpd[[0, 3]], lnd[[0, 3]], **kw)
    # batch independence
    sel = [5, 0, 1]
    full = pkg.ctc_prefix_beam_search(lpd[sel], lnd[sel], **kw)
    for i, n in enumerate(sel):
        assert pkg.ctc_prefix_beam_search(lpd[n:n + 1], lnd[n:n + 1], **kw) == [full[i]]
    # C-level argument errors, before any launch
    for a, b, o, m in ((-0.5, 0.0, None, None), (float("inf"), 0.0, None, None), (0.5, float("nan"), None, None),
                       (0.5, 0.0, 0, None), (0.5, 0.0, 6, None), (0.5, 0.0, None, V - 1)):
        assert _raw(lm, lpd, lnd, B, nbest, 3, a, b, order=o, map_len=m)[0] == -1


def test_argument_errors_and_launch_count(tmp_path):
    pkg = _pkg()
    lp = _rand_lp(9, 4, 20, 30).to(DEV)
    lm, _ = _lms(tmp_path, 30, 2, 11)
    lm_other, _ = _lms(tmp_path, 31, 2, 11, name="other.arpa")
    bad = [({"lm": lm_other}, ValueError), ({"lm": lm, "lm_weight": -0.1}, ValueError),
           ({"lm": lm, "lm_weight": float("nan")}, ValueError), ({"lm": lm, "token_bonus": float("inf")}, ValueError),
           ({"lm": "lm.arpa"}, TypeError), ({"lm": lm, "beam_width": 16}, ValueError),
           ({"lm": lm, "blank": 30}, ValueError)]
    for kw, exc in bad:
        before = pkg._lib.launch_count
        with pytest.raises(exc):
            pkg.ctc_prefix_beam_search(lp, **kw)
        assert pkg._lib.launch_count == before
    before = pkg._lib.launch_count
    pkg.ctc_prefix_beam_search(lp, beam_width=5, lm=lm)
    assert pkg._lib.launch_count - before == 2


def _edit_distance(a, b):
    d = list(range(len(b) + 1))
    for i, x in enumerate(a, 1):
        prev, d[0] = d[0], i
        for j, y in enumerate(b, 1):
            prev, d[j] = d[j], min(d[j] + 1, d[j - 1] + 1, prev + (x != y))
    return d[-1]


def test_lm_lowers_token_error_rate(tmp_path):
    """Every position is acoustically ambiguous between the spoken token and a fixed confuser; a bigram LM whose
    counts follow the speaker's habits (token a is usually followed by succ[a]) recovers most of them."""
    pkg = _pkg()
    rng = np.random.default_rng(0)
    V, blank, N, L = 13, 0, 24, 20
    toks = list(range(1, 7))
    succ = {a: toks[a % 6] for a in toks}                    # 1->2->3->4->5->6->1
    conf = {a: a + 6 for a in toks}                          # confusers 7..12
    refs = []
    for _ in range(N):
        s = [int(rng.choice(toks))]
        while len(s) < L:
            s.append(succ[s[-1]] if rng.random() < 0.9 else int(rng.choice(toks)))
        refs.append(s)
    T = 3 * L
    logits = np.full((N, T, V), -8.0, dtype=np.float32)
    for n, s in enumerate(refs):
        for i, c in enumerate(s):
            for f in (3 * i, 3 * i + 1):
                noise = rng.normal(0.0, 0.6)
                logits[n, f, c] = 2.0 + noise
                logits[n, f, conf[c]] = 2.0 - noise
            logits[n, 3 * i + 2, blank] = 4.0
    lp = torch.from_numpy(logits).log_softmax(-1)
    vocab = [f"p{i}" for i in range(V)]
    lines = ["\\data\\", "ngram 1=%d" % (V + 2), "ngram 2=%d" % ((len(toks) + 1) * (V - 1)), "", "\\1-grams:",
             "-99\t<s>\t0", "-1\t</s>\t0", "-3\t<unk>\t0"]
    lines += [f"-1.5\tp{i}\t0" for i in range(1, V)] + [""]
    lines += ["\\2-grams:"]
    for a in ["<s>"] + [f"p{i}" for i in toks]:
        for b in range(1, V):
            p = 0.9 if (a != "<s>" and b == succ[int(a[1:])]) else 0.1 / (V - 2)
            lines.append(f"{np.log10(p):.6f}\t{a} p{b}")
    lines += ["", "\\end\\"]
    path = tmp_path / "bigram.arpa"
    path.write_text("\n".join(lines) + "\n", encoding="utf-8")
    lm = pkg.NgramLM.from_arpa(str(path), vocab)
    plain = pkg.ctc_prefix_beam_search(lp.to(DEV), beam_width=8, blank=blank)
    fused = pkg.ctc_prefix_beam_search(lp.to(DEV), beam_width=8, blank=blank, lm=lm, lm_weight=1.0)
    ter = lambda hyps: sum(_edit_distance(h[0].tokens, r) for h, r in zip(hyps, refs)) / (N * L)   # noqa: E731
    assert ter(fused) < ter(plain), (ter(fused), ter(plain))


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


def test_trainer_transcribe_with_lm(tmp_path):
    pkg = _pkg()
    from multimodal_av_model_b200.synthetic import CharTokenizer, make_batch
    tok = CharTokenizer(800)
    tr = pkg.MultimodalTrainer(*_tiny_models(pkg), tok, device="cuda")
    batch = make_batch(pairs=2, seconds=2.0, t_v=60, seed=5, l_range=(4, 12))
    p = _write_arpa(tmp_path / "lm.arpa", tok.id_to_token, 3, 12)
    lm = pkg.NgramLM.from_arpa(str(p), tok.id_to_token)
    plain = tr.transcribe(batch, beam_width=5, nbest=3)
    again = tr.transcribe(batch, beam_width=5, nbest=3, lm=None)
    zero = tr.transcribe(batch, beam_width=5, nbest=3, lm=lm, lm_weight=0.0, token_bonus=0.0)
    fused = tr.transcribe(batch, beam_width=5, nbest=3, lm=lm, lm_weight=1.0, token_bonus=0.5)
    assert len(fused) == 2
    for spk_p, spk_a, spk_z, spk_f in zip(plain, again, zero, fused):
        for hp, ha, hz, hf in zip(spk_p, spk_a, spk_z, spk_f):
            assert all(type(s) is float and isinstance(t, str) for t, s in hp)
            assert [t for t, _ in ha] == [t for t, _ in hp]
            assert [s for _, s in ha] == pytest.approx([s for _, s in hp], rel=1e-4)
            assert [s for _, s in hz] == pytest.approx([s for _, s in hp], rel=1e-4)
            scores = [s for _, s in hf]
            assert 1 <= len(hf) <= 3 and scores == sorted(scores, reverse=True)
    assert any(sf != sp for spk_p, spk_f in zip(plain, fused) for hp, hf in zip(spk_p, spk_f)
               for (_, sp), (_, sf) in zip(hp, hf))
