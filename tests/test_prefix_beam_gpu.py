"""GPU: CTC prefix beam search (csrc/ctc_prefix_beam.cu) — tokens, lengths and score bits equal to the CPU oracle
(oracle/prefix_beam_oracle.py) on padded, tie-heavy, peaky, long and small-vocabulary batches; per-utterance failures,
argument errors, the launch count and trainer.transcribe()."""
import numpy as np
import pytest
import torch

from oracle import prefix_beam_oracle as O

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


def _check(got, lp, lengths, B, nbest, blank, rows=None):
    """got[i] (hypotheses of utterance rows[i]) against the oracle: same tokens, same score bits."""
    lp = lp.float().cpu().numpy()
    rows = range(lp.shape[0]) if rows is None else rows
    for i, n in enumerate(rows):
        st, ref = O.prefix_beam_search(lp[n], int(lengths[n]), B, nbest, blank)
        assert st == 0
        assert [h.tokens for h in got[i]] == [list(t) for t, _ in ref], (n, B, nbest)
        assert [_bits(h.score) for h in got[i]] == [_bits(s) for _, s in ref], (n, B, nbest)


def _lengths(N, T, seed):
    ln = torch.from_numpy(np.random.default_rng(seed).integers(0, T + 1, size=N))
    ln[0], ln[1] = 0, T
    return ln


@pytest.mark.parametrize("B", [1, 5, 10, 15])
def test_padded_batch_bit_exact(B):
    pkg = _pkg()
    N, T, V, blank = 64, 150, 800, 3
    lp = _rand_lp(B, N, T, V)
    ln = _lengths(N, T, B)
    lpd = lp.to(DEV)
    full = pkg.ctc_prefix_beam_search(lpd, ln.to(DEV), beam_width=B, nbest=B, blank=blank)
    _check(full, lp, ln, B, B, blank)
    assert all(len(h) >= 1 for h in full)
    assert full[0] == [pkg.Hypothesis([], 0.0)]            # length 0: one empty hypothesis of score 0
    top = pkg.ctc_prefix_beam_search(lpd, ln.to(DEV), beam_width=B, nbest=1, blank=blank)
    assert [h[:1] for h in full] == top


@pytest.mark.parametrize("quant", [0.5, 2.0])
def test_tie_heavy_input(quant):
    """Log-probs on a coarse grid: many equal candidates, decided by the stable order alone."""
    pkg = _pkg()
    N, T, V, blank, B = 32, 60, 40, 3, 6
    lp = torch.round(_rand_lp(11, N, T, V, scale=1.0) * quant) / quant
    ln = _lengths(N, T, 12)
    got = pkg.ctc_prefix_beam_search(lp.to(DEV), ln, beam_width=B, nbest=B, blank=blank)
    _check(got, lp, ln, B, B, blank)


def test_peaky_long_blank_runs():
    """Like a trained head: blank near 1 on most frames, short bursts of one token."""
    pkg = _pkg()
    N, T, V, blank, B = 32, 150, 800, 3, 10
    g = torch.Generator().manual_seed(3)
    logits = torch.randn(N, T, V, generator=g)
    logits[:, :, blank] += 12.0
    burst = torch.rand(N, T, generator=g) < 0.15
    tok = torch.randint(0, V, (N, T), generator=g)
    logits[burst, tok[burst]] += 20.0
    lp = logits.log_softmax(-1)
    ln = _lengths(N, T, 4)
    got = pkg.ctc_prefix_beam_search(lp.to(DEV), ln, beam_width=B, nbest=B, blank=blank)
    _check(got, lp, ln, B, B, blank)


def test_vocab_801_blank_0():
    pkg = _pkg()
    N, T, V, B = 32, 150, 801, 10
    lp = _rand_lp(5, N, T, V)
    ln = _lengths(N, T, 5)
    _check(pkg.ctc_prefix_beam_search(lp.to(DEV), ln, beam_width=B, nbest=3, blank=0), lp, ln, B, 3, 0)


def test_long_utterances_trie_in_workspace():
    """T = 1000: 1 + T*B trie nodes do not fit shared memory and live in the workspace."""
    pkg = _pkg()
    N, T, V, B = 8, 1000, 801, 10
    lp = _rand_lp(6, N, T, V)
    ln = torch.tensor([1000, 999, 0, 500, 1000, 1, 731, 1000])
    _check(pkg.ctc_prefix_beam_search(lp.to(DEV), ln, beam_width=B, nbest=B, blank=3), lp, ln, B, B, 3)


@pytest.mark.parametrize("V", [3, 12, 20])
def test_vocab_smaller_than_2b_plus_1(V):
    pkg = _pkg()
    N, T, B = 16, 40, 10
    lp = _rand_lp(V, N, T, V, scale=1.5)
    ln = _lengths(N, T, V)
    _check(pkg.ctc_prefix_beam_search(lp.to(DEV), ln, beam_width=B, nbest=B, blank=1), lp, ln, B, B, 1)


def test_batch_independence_and_default_lengths():
    pkg = _pkg()
    N, T, V, B = 24, 80, 300, 5
    lp = _rand_lp(21, N, T, V).to(DEV)
    full = pkg.ctc_prefix_beam_search(lp, beam_width=B, nbest=2, blank=3)
    sel = [5, 0, 17]
    part = pkg.ctc_prefix_beam_search(lp[sel], beam_width=B, nbest=2, blank=3)
    assert part == [full[i] for i in sel]
    one = pkg.ctc_prefix_beam_search(lp[7:8].double(), torch.tensor([T]), beam_width=B, nbest=2, blank=3)
    assert one == [full[7]]
    _check(full[:4], lp[:4], [T] * 4, B, 2, 3)


def test_sampled_rows_of_a_large_batch():
    pkg = _pkg()
    N, T, V, B = 4096, 150, 800, 10
    lp = _rand_lp(40, N, T, V)
    ln = torch.from_numpy(np.random.default_rng(40).integers(100, T + 1, size=N))
    got = pkg.ctc_prefix_beam_search(lp.to(DEV), ln.to(DEV), beam_width=B, nbest=2, blank=3)
    rows = sorted(np.random.default_rng(41).choice(N, size=32, replace=False).tolist())
    _check([got[n] for n in rows], lp, ln, B, 2, 3, rows=rows)


def _raw(lp, ln, B, nbest, blank):
    pkg = _pkg()
    L = pkg._lib.lib()
    N, T, V = lp.shape
    ws_bytes = int(L.avctc_ctc_prefix_beam_workspace_bytes(N, T, V, B))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=DEV)
    tok = torch.full((N, nbest, T), -7, dtype=torch.int32, device=DEV)
    olen = torch.full((N, nbest), -7, dtype=torch.int32, device=DEV)
    osc = torch.zeros((N, nbest), dtype=torch.float64, device=DEV)
    st = torch.full((N,), -7, dtype=torch.int32, device=DEV)
    rc = L.avctc_ctc_prefix_beam(lp.data_ptr(), lp.stride(0), lp.stride(1), N, T, V, ln.data_ptr(), B, nbest, blank,
                                 tok.data_ptr(), olen.data_ptr(), osc.data_ptr(), st.data_ptr(), ws.data_ptr(), ws_bytes,
                                 pkg._lib.stream_ptr(lp.device))
    torch.cuda.synchronize()
    return rc, tok.cpu(), olen.cpu(), osc.cpu(), st.cpu()


def test_nan_row_and_bad_length_fail_only_their_utterance():
    pkg = _pkg()
    N, T, V, B, nbest = 6, 50, 100, 5, 3
    lp = _rand_lp(8, N, T, V)
    lp[2, 17, 40] = float("nan")
    ln = torch.tensor([50, 40, 50, 51, -1, 10])
    lpd, lnd = lp.to(DEV), ln.to(DEV)
    rc, tok, olen, osc, st = _raw(lpd, lnd, B, nbest, 3)
    assert rc == 0 and st.tolist() == [0, 0, 1, 2, 2, 0]
    for n in (2, 3, 4):
        assert (olen[n] == 0).all() and (osc[n] == -np.inf).all()
    good = [0, 1, 5]
    hyps = [[pkg.Hypothesis(tok[n, i, :olen[n, i]].tolist(), float(osc[n, i])) for i in range(nbest)
             if osc[n, i] > -np.inf] for n in good]
    _check(hyps, lp, ln, B, nbest, 3, rows=good)
    with pytest.raises(RuntimeError, match="utterance 2: .*NaN"):
        pkg.ctc_prefix_beam_search(lpd, lnd, beam_width=B, nbest=nbest, blank=3)
    with pytest.raises(RuntimeError, match="utterance 1: length 51 outside"):
        pkg.ctc_prefix_beam_search(lpd[[0, 3]], lnd[[0, 3]], beam_width=B, nbest=nbest, blank=3)


def test_argument_errors_and_launch_count():
    pkg = _pkg()
    lp = _rand_lp(9, 4, 20, 30).to(DEV)
    for kw in ({"beam_width": 0}, {"beam_width": 16}, {"beam_width": 5, "nbest": 6}, {"nbest": 0}, {"blank": 30},
               {"blank": -1}):
        before = pkg._lib.launch_count
        with pytest.raises(ValueError):
            pkg.ctc_prefix_beam_search(lp, **kw)
        assert pkg._lib.launch_count == before
    with pytest.raises(RuntimeError, match="not supported"):
        pkg.ctc_prefix_beam_search(torch.zeros(2, 5, 1025, device=DEV))
    with pytest.raises(RuntimeError, match="CUDA"):
        pkg.ctc_prefix_beam_search(lp.cpu())
    L = pkg._lib.lib()
    assert L.avctc_ctc_prefix_beam(lp.data_ptr(), 600, 30, 4, 20, 30, None, 5, 6, 0, None, None, None, None, None, 0,
                                   None) == -1
    before = pkg._lib.launch_count
    pkg.ctc_prefix_beam_search(lp, beam_width=5)
    assert pkg._lib.launch_count - before == 2


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


def test_trainer_transcribe_without_transcripts():
    pkg = _pkg()
    from multimodal_av_model_b200.synthetic import CharTokenizer, make_batch
    tr = pkg.MultimodalTrainer(*_tiny_models(pkg), CharTokenizer(800), device="cuda")
    batch = make_batch(pairs=3, seconds=2.0, t_v=60, seed=5, l_range=(4, 12))
    full = tr.transcribe(batch, beam_width=5, nbest=3)
    bare = {k: v for k, v in batch.items() if not k.startswith("text")}
    out = tr.transcribe(bare, beam_width=5, nbest=3)
    assert len(out) == 2 and all(len(spk) == 3 for spk in out)
    for spk, spk_full in zip(out, full):
        for hyps, hyps_full in zip(spk, spk_full):
            assert 1 <= len(hyps) <= 3 and len(hyps) == len(hyps_full)
            assert all(isinstance(text, str) for text, _ in hyps)
            scores = [s for _, s in hyps]
            assert scores == sorted(scores, reverse=True) and all(s <= 1e-9 for s in scores)
            assert scores == pytest.approx([s for _, s in hyps_full], rel=1e-4)   # transcripts play no part
    top = tr.transcribe(bare)                                  # default beam width, one hypothesis
    assert all(len(h) == 1 for spk in top for h in spk)
