"""GPU: batched CTC forced alignment (csrc/ctc_align.cu) — bit-exact with torchaudio's CPU forced_align through the
fixture and the numpy oracle, on padded batches, ties, bf16 input, the [T,B,V] view, bad input and trainer.align()."""
import numpy as np
import pytest
import torch

from conftest import load_cases
from oracle import align_oracle

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _pkg():
    import multimodal_av_model_b200 as pkg
    return pkg


def _bits(x):
    return np.asarray(x, dtype=np.float32).view(np.uint32)


def _check_rows(paths, scores, lp, tg, il, tl, blank):
    """Every row against the oracle on its own utterance (fp32 upcast of the input), padding = blank / 0."""
    paths, scores = paths.cpu().numpy(), scores.float().cpu().numpy()
    lp32 = lp.float().cpu().numpy()
    tg, il, tl = tg.cpu().numpy(), il.cpu().numpy(), tl.cpu().numpy()
    for n in range(paths.shape[0]):
        T = int(il[n])
        p, s = align_oracle.ctc_forced_align(lp32[n, :T], tg[n, :tl[n]], blank)
        assert np.array_equal(paths[n, :T], p), n
        assert np.array_equal(_bits(scores[n, :T]), _bits(s)), n
        assert (paths[n, T:] == blank).all() and (scores[n, T:] == 0).all()


def _batch(seed, N, T, V, Lmax, blank, lmin=1, rep=0.15, quant=0.0, slack=True):
    rng = np.random.default_rng(seed)
    g = torch.Generator().manual_seed(seed)
    z = torch.randn(N, T, V, generator=g)
    if quant:
        z = torch.round(z / quant) * quant
    lp = z.log_softmax(-1)
    if quant:
        lp = torch.round(lp * 4) / 4
    tl = rng.integers(lmin, Lmax + 1, size=N)
    ids = np.array([c for c in range(V) if c != blank])
    tg = np.zeros((N, Lmax), dtype=np.int64)
    il = np.zeros(N, dtype=np.int64)
    for n in range(N):
        row = rng.choice(ids, size=tl[n])
        for j in range(1, tl[n]):
            if rng.random() < rep:
                row[j] = row[j - 1]
        tg[n, :tl[n]] = row
        need = int(tl[n] + (row[1:] == row[:-1]).sum())
        il[n] = rng.integers(need, T + 1) if slack else need
    return lp, torch.from_numpy(tg), torch.from_numpy(il), torch.from_numpy(tl)


@pytest.mark.parametrize("case", sorted(load_cases("align_cases.npz")))
def test_fixture_bit_exact(case):
    pkg = _pkg()
    c = load_cases("align_cases.npz")[case]
    lp = torch.from_numpy(c["lp"]).to(DEV)[None]
    tg = torch.from_numpy(c["targets"]).to(DEV)[None]
    paths, scores = pkg.forced_align(lp, tg, blank=int(c["blank"]))
    assert paths.dtype == torch.int64 and scores.dtype == torch.float32 and paths.shape == (1, lp.shape[1])
    assert np.array_equal(paths[0].cpu().numpy(), c["paths"])
    assert np.array_equal(_bits(scores[0].cpu().numpy()), _bits(c["scores"]))


def test_fixture_cases_in_one_padded_batch():
    """All fixture cases of the smaller vocabularies padded into one batch (V = 40, T = max): same rows as alone."""
    pkg = _pkg()
    cases = [c for c in load_cases("align_cases.npz").values() if c["lp"].shape[1] <= 40]
    N, T, V = len(cases), max(c["lp"].shape[0] for c in cases), 40
    Lmax = max(len(c["targets"]) for c in cases)
    lp = torch.full((N, T, V), -1e4)                  # padding classes / frames never win
    tg = torch.zeros(N, Lmax, dtype=torch.long)
    for n, c in enumerate(cases):
        lp[n, :c["lp"].shape[0], :c["lp"].shape[1]] = torch.from_numpy(c["lp"])
        tg[n, :len(c["targets"])] = torch.from_numpy(c["targets"])
    blanks = {int(c["blank"]) for c in cases}
    for blank in blanks:
        sel = [n for n, c in enumerate(cases) if int(c["blank"]) == blank]
        il = torch.tensor([cases[n]["lp"].shape[0] for n in sel])
        tl = torch.tensor([len(cases[n]["targets"]) for n in sel])
        paths, scores = pkg.forced_align(lp[sel].to(DEV), tg[sel].to(DEV), il.to(DEV), tl.to(DEV), blank=blank)
        for i, n in enumerate(sel):
            Tn = int(il[i])
            assert np.array_equal(paths[i, :Tn].cpu().numpy(), cases[n]["paths"])
            assert np.array_equal(_bits(scores[i, :Tn].cpu().numpy()), _bits(cases[n]["scores"]))


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("blank", [0, 3])
def test_config2_padded_batch_against_oracle(dtype, blank):
    """N = 64, T = 1000, V = 801, L <= 80; bf16 input is compared with the oracle on its fp32 upcast."""
    pkg = _pkg()
    lp, tg, il, tl = _batch(10 + blank, 64, 1000, 801, 80, blank, lmin=10)
    lp = lp.to(dtype)
    paths, scores = pkg.forced_align(lp.to(DEV), tg.to(DEV), il.to(DEV), tl.to(DEV), blank=blank)
    assert scores.dtype == dtype
    _check_rows(paths, scores, lp, tg, il, tl, blank)


@pytest.mark.parametrize("quant", [1.0, 4.0])
def test_ties_and_tight_lengths(quant):
    """Quantized log-probs (many equal lattice scores) and T_b = L_b + R_b exactly: torchaudio's tie order."""
    pkg = _pkg()
    for slack, seed in ((True, 1), (False, 2)):
        lp, tg, il, tl = _batch(seed, 32, 150, 12, 58, 3, rep=0.4, quant=quant, slack=slack)
        paths, scores = pkg.forced_align(lp.to(DEV), tg.to(DEV), il.to(DEV), tl.to(DEV), blank=3)
        _check_rows(paths, scores, lp, tg, il, tl, 3)


def test_transposed_view_and_int32_targets():
    """The [T,B,V] tensor the CTC loss takes, aligned through its [B,T,V] transpose (stride_n = V, stride_t = B*V)."""
    pkg = _pkg()
    lp, tg, il, tl = _batch(5, 16, 150, 800, 58, 3, lmin=20)
    tbv = lp.transpose(0, 1).contiguous().to(DEV)
    view = tbv.transpose(0, 1)
    assert view.stride() == (800, 16 * 800, 1)
    paths, scores = pkg.forced_align(view, tg.to(DEV).int(), il.to(DEV), tl.to(DEV), blank=3)
    assert paths.dtype == torch.int32
    _check_rows(paths.long(), scores, lp, tg, il, tl, 3)


def test_batch_independence():
    pkg = _pkg()
    lp, tg, il, tl = _batch(7, 24, 300, 50, 40, 0)
    d = [x.to(DEV) for x in (lp, tg, il, tl)]
    paths, scores = pkg.forced_align(*d, blank=0)
    for n in (0, 5, 23):
        T = int(il[n])
        p1, s1 = pkg.forced_align(d[0][n:n + 1, :T], d[1][n:n + 1, :int(tl[n])], blank=0)
        assert torch.equal(p1[0], paths[n, :T]) and torch.equal(s1[0], scores[n, :T])


def test_empty_transcript_aligns_to_blank():
    pkg = _pkg()
    lp = torch.randn(3, 20, 9).log_softmax(-1).to(DEV)
    tg = torch.tensor([[4, 5], [0, 0], [6, 6]], device=DEV)
    il = torch.tensor([20, 11, 20], device=DEV)
    tl = torch.tensor([2, 0, 2], device=DEV)
    paths, scores = pkg.forced_align(lp, tg, il, tl, blank=3)
    assert (paths[1] == 3).all()
    assert torch.equal(scores[1, :11], lp[1, :11, 3]) and (scores[1, 11:] == 0).all()


def _raw_align(lp, tg, il, tl, blank, Lmax=None):
    """The C ABI directly: (return code, paths, scores, status)."""
    pkg = _pkg()
    N, T, V = lp.shape
    paths = torch.full((N, T), -7, dtype=torch.int32, device=DEV)
    scores = torch.full((N, T), 7.0, device=DEV)
    status = torch.full((N,), -7, dtype=torch.int32, device=DEV)
    rc = pkg._lib.lib().avctc_ctc_align(lp.data_ptr(), 0, lp.stride(0), lp.stride(1), N, T, V, tg.data_ptr(), tg.stride(0),
                                        il.data_ptr(), tl.data_ptr(), tg.shape[1] if Lmax is None else Lmax, blank,
                                        paths.data_ptr(), scores.data_ptr(), status.data_ptr(),
                                        pkg._lib.stream_ptr(lp.device))
    torch.cuda.synchronize()
    return rc, paths, scores, status


def test_invalid_utterances_set_only_their_own_status():
    pkg = _pkg()
    lp, tg, il, tl = _batch(3, 6, 40, 10, 8, 0, lmin=4)
    tg[1, 2] = 0                 # blank inside the transcript
    tg[2, 0] = 10                # label == V
    tg[3, 1] = -1                # negative label
    il[4] = int(tl[4]) - 1       # too short for its transcript
    tl[5] = 9                    # longer than the targets tensor
    d = [x.to(DEV) for x in (lp, tg, il, tl)]
    rc, paths, scores, status = _raw_align(*d, blank=0)
    assert rc == 0
    assert status.cpu().tolist() == [0, 1, 1, 1, 2, 3]
    assert (paths[1:] == 0).all() and (scores[1:] == 0).all()
    p0, s0 = pkg.forced_align(d[0][:1], d[1][:1], d[2][:1], d[3][:1], blank=0)
    assert torch.equal(paths[0].long(), p0[0]) and torch.equal(scores[0], s0[0])
    with pytest.raises(ValueError, match="utterance 1: targets Tensor shouldn't contain blank"):
        pkg.forced_align(*d, blank=0)
    for n, exc, msg in ((2, ValueError, "less than the CTC dimension"), (3, ValueError, "less than the CTC dimension"),
                        (4, RuntimeError, "targets length is too long for CTC"), (5, RuntimeError, "outside")):
        sel = [0, n]
        with pytest.raises(exc, match=f"utterance 1: .*{msg}"):
            pkg.forced_align(d[0][sel], d[1][sel], d[2][sel], d[3][sel], blank=0)


def test_longest_lattice_and_unsupported_shapes():
    """2L+1 = 511 is the largest lattice; 513 states, or more frames than shared memory holds back-pointers for, are
    AVCTC_ERR_UNSUPPORTED (-2)."""
    pkg = _pkg()
    lib = pkg._lib.lib()
    assert lib.avctc_ctc_align_supported(1000, 255) == 1 and lib.avctc_ctc_align_supported(1600, 255) == 1
    assert lib.avctc_ctc_align_supported(1000, 256) == 0 and lib.avctc_ctc_align_supported(4000, 10) == 0
    lp, tg, il, tl = _batch(4, 3, 600, 300, 255, 0, lmin=250, rep=0.0)
    tl[0] = 255
    tg[0] = torch.from_numpy(np.random.default_rng(0).permutation(np.arange(1, 300))[:255])
    il[0] = 600
    paths, scores = pkg.forced_align(lp.to(DEV), tg.to(DEV), il.to(DEV), tl.to(DEV), blank=0)
    _check_rows(paths, scores, lp, tg, il, tl, 0)
    d = [x.to(DEV) for x in (lp, tg, il, tl)]
    assert _raw_align(*d, blank=0, Lmax=256)[0] == -2
    big = torch.randn(1, 4000, 5, device=DEV).log_softmax(-1)
    one = torch.ones(1, 1, dtype=torch.long, device=DEV)
    assert _raw_align(big, one, torch.tensor([4000], device=DEV), torch.tensor([1], device=DEV), blank=0)[0] == -2
    with pytest.raises(RuntimeError, match="status -2"):
        pkg.forced_align(big, one)


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


def test_trainer_align_spans():
    pkg = _pkg()
    import torch.nn.functional as F
    from multimodal_av_model_b200.synthetic import CharTokenizer, make_batch
    tr = pkg.MultimodalTrainer(*_tiny_models(pkg), CharTokenizer(800), device="cuda")
    batch = make_batch(pairs=3, seconds=2.0, t_v=60, seed=5, l_range=(4, 12))
    out = tr.align(batch)
    assert len(out) == 2 and all(len(spk) == 3 for spk in out)
    for s in range(2):
        texts, lens = batch[f"text{s + 1}"], batch[f"text{s + 1}_lengths"]
        mask = batch[f"mask{s + 1}"]
        for b, spans in enumerate(out[s]):
            L = int(lens[b])
            assert [sp.token for sp in spans] == texts[b, :L].tolist()          # one span per target token
            assert all(sp.piece == tr.tokenizer.id_to_token[sp.token] for sp in spans)
            assert all(0 <= sp.start < sp.end for sp in spans)
            assert all(a.end <= b_.start for a, b_ in zip(spans, spans[1:]))   # ordered, disjoint
            secs = [x for sp in spans for x in (sp.start_sec, sp.end_sec)]
            assert all(x <= y for x, y in zip(secs, secs[1:]))
            # inside the speaker's speech frames (encoder frames at 20 ms: mask downsampled like the fusion sees it)
            t_enc = mask.shape[1]
            for k, st in zip((10, 3, 3, 3, 3, 2, 2), (5, 2, 2, 2, 2, 2, 2)):    # wav2vec2 feature-extractor frames
                t_enc = (t_enc - k) // st + 1
            ds = F.interpolate(mask.unsqueeze(1).float(), size=t_enc, mode="nearest").squeeze(1).long()[b]
            fr = torch.nonzero((ds != 0) & (ds != 3)).flatten()
            lo, hi = float(fr.min()) * 0.02, float(fr.max()) * 0.02 + 0.02
            assert lo - 1e-9 <= spans[0].start_sec and spans[-1].end_sec <= hi + 1e-9
