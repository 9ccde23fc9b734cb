"""CPU: the oracle (oracle/) against the fixtures produced by the reference itself (tests/golden/)."""
import numpy as np
import pytest

import oracle
from oracle import np_oracle
from conftest import load_cases

CTC = load_cases("ctc_cases.npz")
BEAM = load_cases("beam_cases.npz")
FUS = load_cases("fusion_cases.npz")
NCE = load_cases("infonce_cases.npz")


@pytest.mark.parametrize("name", sorted(CTC))
def test_ctc_oracle_matches_reference(name):
    c = CTC[name]
    lp = np.transpose(c["lp"], (1, 0, 2))  # fixture stores [B,T,V]; CTC sees the [T,B,V] view
    r = oracle.ctc_loss(lp, c["targets"], c["input_lengths"], c["target_lengths"], blank=int(c["blank"]),
                        reduction="mean", zero_infinity=bool(c["zero_infinity"]))
    # tight pin: the reference's CTCLoss run in float64 on the same inputs
    assert np.allclose(r["loss"], c["loss64"], rtol=1e-12, atol=1e-12)
    fin = np.isfinite(c["nll64"])
    assert np.array_equal(np.isfinite(r["nll"]), fin)
    assert np.allclose(r["nll"][fin], c["nll64"][fin], rtol=1e-12, atol=1e-12)
    g64 = np.transpose(c["grad64"], (1, 0, 2))
    scale = max(np.abs(g64).max(), 1e-30)
    assert np.abs(r["grad"] - g64).max() / scale < 1e-10
    # loose pin: the reference's float32 run (torch's own fp32 kernel drifts ~2.5e-4 at T=200)
    g32 = np.transpose(c["grad"], (1, 0, 2))
    assert np.allclose(r["loss"], c["loss"], rtol=2e-5, atol=2e-5)
    assert np.abs(r["grad"] - g32).max() / scale < 1e-3


def test_ctc_oracle_conventions():
    """SURVEY.md §4 item 3 edge cases, checked on the oracle itself."""
    rng = np.random.default_rng(0)
    T, B, V = 7, 2, 6
    z = rng.standard_normal((T, B, V))
    lp = z - np.log(np.exp(z).sum(-1, keepdims=True))
    tg = np.array([[1, 2], [4, 4]])
    # L = 0: nll = -sum_t lp[t, blank]
    r = oracle.ctc_loss(lp, tg, [T, T], [0, 0], blank=3, reduction="none")
    assert np.allclose(r["nll"], -lp[:, :, 3].sum(0))
    # repeated label needs T >= L + repeats
    r = oracle.ctc_loss(lp, tg, [T, 2], [2, 2], blank=3, reduction="none", zero_infinity=True)
    assert np.isinf(r["nll"][1]) and np.all(r["grad"][:, 1] == 0)
    # gradient rows sum to 0 (softmax-folded convention) and vanish beyond input_length
    r = oracle.ctc_loss(lp, tg, [5, T], [2, 2], blank=3, reduction="sum")
    assert np.abs(r["grad"][:5, 0].sum(-1)).max() < 1e-12
    assert np.all(r["grad"][5:, 0] == 0)
    # brute force over all alignments for a tiny case
    import itertools
    Tt, lab = 4, [1, 1]
    tot = 0.0
    for path in itertools.product(range(V), repeat=Tt):
        col, prev = [], None
        for c in path:
            if c != prev and c != 3:
                col.append(c)
            prev = c
        if col == lab:
            tot += np.exp(sum(lp[t, 0, c] for t, c in enumerate(path)))
    r = oracle.ctc_loss(lp[:Tt, :1], np.array([lab]), [Tt], [2], blank=3, reduction="none")
    assert np.allclose(r["nll"][0], -np.log(tot))


@pytest.mark.parametrize("name", sorted(k for k in BEAM if not k.startswith("topk")))
def test_beam_oracle_bit_exact(name):
    c = BEAM[name]
    ids = oracle.beam_search(c["lp"], int(c["beam"]), int(c["blank"]))
    assert ids == c["ids"].tolist()


@pytest.mark.parametrize("name", sorted(k for k in BEAM if k.startswith("topk")))
def test_topk_tie_order(name):
    c = BEAM[name]
    vals, idx = oracle.topk(c["row"], int(c["k"]))
    assert idx.tolist() == c["idx"].tolist()
    assert np.array_equal(vals, c["vals"])


def test_beam_equals_collapsed_first_topk():
    """SURVEY.md §8 a13 theorem: output == collapse(topk(row).indices[0] per frame)."""
    rng = np.random.default_rng(5)
    z = 3 * rng.standard_normal((30, 100)).astype(np.float32)
    lp = z - np.log(np.exp(z).sum(-1, keepdims=True))
    ids, scores, paths = oracle.beam_search(lp, 7, 3, debug=True)
    first = [int(oracle.topk(lp[t], 7)[1][0]) for t in range(30)]
    assert paths[0].tolist() == first
    assert np.all(np.diff(scores) <= 0)
    col, prev = [], None
    for c in first:
        if c != prev and c != 3:
            col.append(c)
        prev = c
    assert ids == col


def _params(c, prefix="param/"):
    return {k[len(prefix):]: v.astype(np.float64) for k, v in c.items() if k.startswith(prefix)}


@pytest.mark.parametrize("name", sorted(FUS))
def test_fusion_oracle_matches_reference(name):
    c = FUS[name]
    fused, il = np_oracle.fusion_forward(_params(c), c["visual"], c["audio"], c["mask"],
                                         num_heads=int(c["num_heads"]))
    assert il.tolist() == c["input_lengths"].tolist()
    assert np.abs(fused - c["fused"]).max() < 5e-6
    d = _params(c, "dec/")
    lp = np_oracle.ctc_head(fused, d["net.0.weight"], d["net.0.bias"])
    assert np.abs(lp - c["log_probs"]).max() < 1e-5


@pytest.mark.parametrize("name", sorted(NCE))
def test_infonce_oracle_matches_reference(name):
    c = NCE[name]
    w = c["w"].astype(np.float64) if "w" in c else None
    b = c["b"].astype(np.float64) if "b" in c else None
    loss, dmid, dw, db = np_oracle.contrastive_loss_with_mask(c["middle"], c["mask"].reshape(-1), w, b,
                                                              want_grad=True)
    assert np.allclose(loss, c["loss"], rtol=1e-5, atol=1e-6)
    assert np.abs(dmid - c["grad_middle"]).max() < 1e-6
    if w is not None:
        assert np.abs(dw - c["grad_w"]).max() < 1e-5
        assert np.abs(db - c["grad_b"]).max() < 1e-5


def test_interp_index_rules():
    torch = pytest.importorskip("torch")
    import torch.nn.functional as F
    for n_in, n_out in [(80000, 249), (249, 150), (200, 150), (17, 10), (5, 9), (149, 90), (3, 1)]:
        m = torch.arange(n_in).float()[None, None]
        ref = F.interpolate(m, size=n_out, mode="nearest")[0, 0].long().numpy()
        assert np.array_equal(np_oracle.nearest_src_index(n_out, n_in), ref)
        x = torch.randn(2, n_in, 3, dtype=torch.float64)
        ref = F.interpolate(x.permute(0, 2, 1), size=n_out, mode="linear", align_corners=True).permute(0, 2, 1)
        assert np.abs(np_oracle.linear_align_corners(x.numpy(), n_out) - ref.numpy()).max() < 1e-12


# ---------------------------------------------------------------- torch-CPU restatement (oracle/torch_port.py)
def test_torch_port_fusion_and_head_match_reference():
    import torch
    from oracle import torch_port as tp
    for name, c in FUS.items():
        dv, da = c["visual"].shape[-1], c["audio"].shape[-1]
        e = c["param/fusion_proj.weight"].shape[0]
        fus = tp.FusionPort(dv, da, e, num_heads=int(c["num_heads"]))
        fus.load_state_dict({k[6:]: torch.from_numpy(v) for k, v in c.items() if k.startswith("param/")})
        dec = tp.DecoderPort(2 * e, c["dec/net.0.weight"].shape[0], 3)
        dec.load_state_dict({k[4:]: torch.from_numpy(v) for k, v in c.items() if k.startswith("dec/")})
        vis = torch.from_numpy(c["visual"]).requires_grad_()
        aud = torch.from_numpy(c["audio"]).requires_grad_()
        fused, il = fus(vis, aud, torch.from_numpy(c["mask"]))
        lp = dec(fused)
        (lp * torch.from_numpy(c["r"])).sum().backward()
        assert il.tolist() == c["input_lengths"].tolist()
        assert torch.allclose(fused, torch.from_numpy(c["fused"]), atol=1e-6)
        assert torch.allclose(lp, torch.from_numpy(c["log_probs"]), atol=1e-5)
        assert torch.allclose(aud.grad, torch.from_numpy(c["grad_audio"]), atol=1e-5)
        assert torch.allclose(vis.grad, torch.from_numpy(c["grad_visual"]), atol=1e-5)
        for k, p in fus.named_parameters():
            g = c[f"grad/{k}"]
            if g.size == 0:
                assert p.grad is None           # cross_attn_visual is never used (SURVEY.md §3.3)
            else:
                assert torch.allclose(p.grad, torch.from_numpy(g), atol=2e-5), k


def test_torch_port_infonce_beam_and_step_match_reference():
    import torch
    from oracle import torch_port as tp
    for name, c in NCE.items():
        proj = None
        if "w" in c:
            proj = torch.nn.Linear(c["w"].shape[1], c["w"].shape[0])
            proj.load_state_dict({"weight": torch.from_numpy(c["w"]), "bias": torch.from_numpy(c["b"])})
        mid = torch.from_numpy(c["middle"]).requires_grad_()
        loss = tp.contrastive_loss_with_mask(mid, torch.from_numpy(c["mask"]).reshape(-1), proj)
        assert torch.allclose(loss, torch.from_numpy(c["loss"]), atol=1e-6)
        if loss.grad_fn is not None:
            loss.backward()
            assert torch.allclose(mid.grad, torch.from_numpy(c["grad_middle"]), atol=1e-6)
    for name, c in BEAM.items():
        if name.startswith("topk"):
            continue
        assert tp.simple_beam_search(torch.from_numpy(c["lp"]), int(c["beam"]), int(c["blank"])) == c["ids"].tolist()
    z = np.load(__import__("os").path.join(__import__("conftest").GOLDEN, "step_cases.npz"))
    p = {k[6:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("param/")}
    e = p["fusion_proj.weight"].shape[0]
    fus = tp.FusionPort(p["visual_proj.weight"].shape[1], p["audio_proj.weight"].shape[1], e)
    fus.load_state_dict(p)
    dec = tp.DecoderPort(2 * e, z["dec/net.0.weight"].shape[0], 3)
    dec.load_state_dict({k[4:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("dec/")})
    proj = torch.nn.Linear(z["proj/weight"].shape[1], z["proj/weight"].shape[0])
    proj.load_state_dict({"weight": torch.from_numpy(z["proj/weight"]), "bias": torch.from_numpy(z["proj/bias"])})
    feats = [dict(visual=torch.from_numpy(z[f"spk{s}/visual"]), audio=torch.from_numpy(z[f"spk{s}/audio"]),
                  middle=torch.from_numpy(z[f"spk{s}/middle"]), mask=torch.from_numpy(z[f"spk{s}/mask"]),
                  text=torch.from_numpy(z[f"spk{s}/text"]), text_len=torch.from_numpy(z[f"spk{s}/text_len"]))
             for s in (1, 2)]
    loss = tp.hot_path_losses(fus, dec, proj, feats, blank=3)
    loss.backward()
    assert torch.allclose(loss, torch.from_numpy(z["loss_total"]), atol=1e-6)
    for k, prm in fus.named_parameters():
        g = z[f"grad/{k}"]
        if g.size:
            assert torch.allclose(prm.grad, torch.from_numpy(g), atol=2e-5), k

