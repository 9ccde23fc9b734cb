"""oracle/gen_golden.py — produce tests/golden/*.npz by RUNNING THE REFERENCE ITSELF.

Run in the build container only (it needs /root/reference, which does not exist on the GPU box):

    python oracle/gen_golden.py            # rewrites tests/golden/*.npz

The reference (limeorange1102/multimodal-av-model) ships no tests or golden vectors (SURVEY.md §4),
so result parity is pinned by executing its own modules on seeded synthetic inputs under the
installed torch (version stored in every fixture):
  * beam_search.simple_beam_search                      (/root/reference/beam_search.py:2-42)
  * contrastive.contrastive_loss_with_mask              (/root/reference/contrastive.py:8-44)
  * model.fusion_module.CrossAttentionFusion            (/root/reference/model/fusion_module.py:5-67)
  * model.decoder.CTCDecoder                            (/root/reference/model/decoder.py:6-35)
  * nn.CTCLoss(blank=3, zero_infinity=True) as called at /root/reference/model/trainer.py:25,116-117
  * the loss combination of /root/reference/model/trainer.py:98-119 (from encoder features on)
Nothing from the reference is copied into this repository; only its outputs are stored.
"""
from __future__ import annotations

import os
import sys

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

REF = "/root/reference"
OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")


def _import_reference():
    if not os.path.isdir(REF):
        raise SystemExit("gen_golden.py needs /root/reference (build container only)")
    sys.path.insert(0, REF)
    import beam_search as ref_beam          # noqa: E402
    import contrastive as ref_con           # noqa: E402
    from model.fusion_module import CrossAttentionFusion as RefFusion   # noqa: E402
    from model.decoder import CTCDecoder as RefDecoder                  # noqa: E402
    return ref_beam, ref_con, RefFusion, RefDecoder


def _meta():
    return {"torch_version": np.array(torch.__version__), "generator": np.array("oracle/gen_golden.py")}


def make_targets(rng, B, Lmax, lens, V, blank, repeat_frac=0.1):
    tg = np.zeros((B, Lmax), dtype=np.int64)
    ids = np.array([c for c in range(V) if c != blank])
    for b in range(B):
        row = rng.choice(ids, size=lens[b])
        for j in range(1, lens[b]):
            if rng.random() < repeat_frac:
                row[j] = row[j - 1]
        tg[b, :lens[b]] = row
    return tg


def gen_ctc():
    rng = np.random.default_rng(11)
    cases = {}

    def run(name, T, B, V, blank, in_len, tg_len, zero_inf=True, repeat=0.1, dtype=torch.float32,
            scale=1.0, one_d=False):
        g = torch.Generator().manual_seed(len(cases) + 5)
        logits = torch.randn(B, T, V, generator=g, dtype=dtype) * scale
        # the reference feeds a transposed view of [B,T,V] (trainer.py:116)
        lp_btv = logits.log_softmax(-1).detach().requires_grad_()
        Lmax = max(max(tg_len), 1)
        tg = make_targets(rng, B, Lmax, tg_len, V, blank, repeat)
        il = torch.tensor(in_len, dtype=torch.long)
        tl = torch.tensor(tg_len, dtype=torch.long)
        crit = nn.CTCLoss(blank=blank, zero_infinity=zero_inf)
        tgt = torch.from_numpy(tg)
        if one_d:
            tgt = torch.cat([tgt[b, :tg_len[b]] for b in range(B)])
        loss = crit(lp_btv.transpose(0, 1), tgt, il, tl)
        loss.backward()
        nll = F.ctc_loss(lp_btv.detach().transpose(0, 1), tgt, il, tl, blank=blank, reduction="none")
        # same call on the float64 copy of the SAME inputs: the truth the 1e-4 tolerance is stated against
        # (torch's own fp32 kernel is ~2e-4 off it at T=200, see tests/test_oracle_golden.py)
        lp64 = lp_btv.detach().double().requires_grad_()
        loss64 = crit(lp64.transpose(0, 1), tgt, il, tl)
        loss64.backward()
        nll64 = F.ctc_loss(lp64.detach().transpose(0, 1), tgt, il, tl, blank=blank, reduction="none")
        cases[name] = dict(loss64=loss64.detach().numpy(), nll64=nll64.numpy(), grad64=lp64.grad.numpy(),
                           lp=lp_btv.detach().numpy(), targets=tg, input_lengths=il.numpy(),
                           target_lengths=tl.numpy(), blank=np.array(blank),
                           zero_infinity=np.array(zero_inf), loss=loss.detach().numpy(),
                           nll=nll.numpy(), grad=lp_btv.grad.numpy())

    # sizes keep the fixture file under 1 MB: the gradients of the full-vocabulary cases do not compress, so
    # those cases have few frames, and the long-label case has a small vocabulary (its point is L = 92)
    run("basic_v800_b3", T=12, B=2, V=800, blank=3, in_len=[12, 9], tg_len=[5, 1])
    run("blank0_v801", T=10, B=2, V=801, blank=0, in_len=[10, 9], tg_len=[4, 3])
    run("edges", T=12, B=6, V=20, blank=3, in_len=[12, 0, 5, 12, 3, 0], tg_len=[4, 2, 0, 0, 5, 0],
        repeat=0.5)
    run("repeats_tight", T=9, B=3, V=11, blank=3, in_len=[9, 9, 8], tg_len=[5, 4, 4], repeat=0.9)
    run("peaked", T=40, B=2, V=50, blank=3, in_len=[40, 33], tg_len=[12, 9], scale=8.0)
    run("fp64_truth", T=20, B=3, V=37, blank=3, in_len=[20, 18, 11], tg_len=[6, 7, 2], dtype=torch.float64)
    run("one_d_targets", T=16, B=3, V=30, blank=3, in_len=[16, 14, 16], tg_len=[5, 3, 6], one_d=True)
    run("long_labels", T=200, B=2, V=32, blank=3, in_len=[200, 190], tg_len=[92, 70])
    flat = {}
    for k, d in cases.items():
        for kk, vv in d.items():
            flat[f"{k}/{kk}"] = vv
    np.savez_compressed(os.path.join(OUT, "ctc_cases.npz"), **flat, **_meta())


def gen_beam(ref_beam):
    cases = {}
    rng = np.random.default_rng(3)

    def run(name, lp, beam, blank):
        ids = ref_beam.simple_beam_search(torch.from_numpy(lp), beam_width=beam, blank=blank)
        cases[name] = dict(lp=lp, beam=np.array(beam), blank=np.array(blank),
                           ids=np.array(ids, dtype=np.int64))

    def rand_lp(T, V, seed, scale=3.0):
        g = torch.Generator().manual_seed(seed)
        return (scale * torch.randn(T, V, generator=g)).log_softmax(-1).numpy()

    run("rand_b5", rand_lp(40, 800, 7), 5, 3)
    run("rand_b10", rand_lp(40, 800, 8), 10, 3)
    run("rand_b10_v801_blank0", rand_lp(32, 801, 9), 10, 0)
    run("rand_b1", rand_lp(12, 50, 10), 1, 3)
    # k*64 > V -> torch.topk uses nth_element + sort (TopKImpl.h:45,66-76)
    run("nth_element_path_b16", rand_lp(20, 800, 12), 16, 3)
    # tie stress: bf16-rounded values cast back to fp32
    lp = torch.from_numpy(rand_lp(40, 800, 13, scale=0.3)).bfloat16().float().numpy()
    run("ties_bf16_b10", lp, 10, 3)
    run("ties_bf16_b5", lp, 5, 3)
    # forced duplicate maxima, all-equal rows, -inf rows
    lp = rand_lp(30, 800, 14)
    for t in range(30):
        m = lp[t].max()
        pos = rng.choice(800, size=int(rng.integers(2, 13)), replace=False)
        lp[t, pos] = m
    lp[5, :] = np.float32(-6.68)
    lp[6, :] = -np.inf
    run("forced_ties_b10", lp, 10, 3)
    run("forced_ties_b5", lp, 5, 3)
    lpq = torch.from_numpy(rand_lp(25, 64, 15, scale=0.1)).bfloat16().float().numpy()
    run("ties_small_v64_b1", lpq, 1, 3)
    # collapse semantics: repeated tokens separated by blank must both survive (beam_search.py:37-40)
    lp = np.full((8, 10), -20.0, dtype=np.float32)
    for t, c in enumerate([4, 4, 3, 4, 5, 5, 3, 3]):
        lp[t, c] = -0.01
    run("collapse_rule", lp, 5, 3)
    flat = {}
    for k, d in cases.items():
        for kk, vv in d.items():
            flat[f"{k}/{kk}"] = vv
    # raw torch.topk tie cases (indices in torch's CPU order)
    tk = {}
    for i, (V, k) in enumerate([(800, 5), (800, 10), (801, 10), (800, 12), (800, 13), (800, 16), (64, 1), (64, 2)]):
        g = torch.Generator().manual_seed(100 + i)
        row = torch.randn(V, generator=g)
        pos = torch.randperm(V, generator=g)[:14]
        row[pos] = row.max()
        vals, idx = torch.topk(row, k)
        tk[f"topk{i}/row"] = row.numpy(); tk[f"topk{i}/k"] = np.array(k)
        tk[f"topk{i}/idx"] = idx.numpy(); tk[f"topk{i}/vals"] = vals.numpy()
        row2 = torch.zeros(V)
        vals, idx = torch.topk(row2, k)
        tk[f"topk_eq{i}/row"] = row2.numpy(); tk[f"topk_eq{i}/k"] = np.array(k)
        tk[f"topk_eq{i}/idx"] = idx.numpy(); tk[f"topk_eq{i}/vals"] = vals.numpy()
    np.savez_compressed(os.path.join(OUT, "beam_cases.npz"), **flat, **tk, **_meta())


def synth_mask(rng, B, T, pad_tail=True):
    """Mask in the style of dataset/multi_speaker_dataset.py:35-45 + collate pad 3 (collate_fn.py:40)."""
    m = np.full((B, T), 3, dtype=np.int64)
    for b in range(B):
        n = T - (int(rng.integers(0, T // 4)) if pad_tail and b > 0 else 0)
        n1 = int(rng.integers(n // 2, n + 1))
        n2 = int(rng.integers(n // 2, n + 1))
        if b % 2:
            n1 = n
        else:
            n2 = n
        both = min(n1, n2)
        row = np.zeros(n, dtype=np.int64)
        row[:both] = 1
        if n1 > n2:
            row[both:n1] = 2
        else:
            row[both:n2] = 0
        m[b, :n] = row
    return m


def gen_fusion(RefFusion, RefDecoder):
    torch.manual_seed(21)
    rng = np.random.default_rng(21)
    out = {}
    for name, (dv, da, e, h, B, Tv, Ta, V) in {
        "small": (32, 48, 32, 4, 3, 10, 17, 23),
        "equal_len": (16, 24, 16, 2, 2, 9, 9, 12),
    }.items():
        fus = RefFusion(dv, da, e, num_heads=h)
        dec = RefDecoder(2 * e, V, blank_id=3)
        vis = torch.randn(B, Tv, dv, requires_grad=True)
        aud = torch.randn(B, Ta, da, requires_grad=True)
        mask = synth_mask(rng, B, Ta)
        if name == "equal_len":
            mask[:] = 1
            mask[1, -2:] = 2
        fused, il = fus(vis, aud, mask=torch.from_numpy(mask))
        lp = dec(fused)
        r = torch.randn_like(lp)
        (lp * r).sum().backward()
        d = {f"{name}/param/{k}": v.detach().numpy() for k, v in fus.state_dict().items()}
        d.update({f"{name}/dec/{k}": v.detach().numpy() for k, v in dec.state_dict().items()})
        d.update({f"{name}/grad/{k}": (v.grad.numpy() if v.grad is not None else np.zeros(0, np.float32))
                  for k, v in fus.named_parameters()})
        d.update({f"{name}/dec_grad/{k}": v.grad.numpy() for k, v in dec.named_parameters()})
        d.update({f"{name}/visual": vis.detach().numpy(), f"{name}/audio": aud.detach().numpy(),
                  f"{name}/mask": mask, f"{name}/num_heads": np.array(h),
                  f"{name}/fused": fused.detach().numpy(), f"{name}/input_lengths": il.numpy(),
                  f"{name}/log_probs": lp.detach().numpy(), f"{name}/r": r.numpy(),
                  f"{name}/grad_visual": vis.grad.numpy(), f"{name}/grad_audio": aud.grad.numpy()})
        out.update(d)
    np.savez_compressed(os.path.join(OUT, "fusion_cases.npz"), **out, **_meta())


def gen_infonce(ref_con):
    torch.manual_seed(31)
    rng = np.random.default_rng(31)
    out = {}
    for name, (B, T, D, P, mode) in {
        "proj": (3, 21, 40, 16, "mixed"), "noproj": (2, 15, 24, 0, "mixed"),
        "no_strong": (2, 12, 24, 8, "no_strong"), "no_weak": (2, 12, 24, 8, "no_weak"),
    }.items():
        mid = torch.randn(B, T, D, requires_grad=True)
        mask = synth_mask(rng, B, T)
        if mode == "no_strong":
            mask[mask == 2] = 0
        if mode == "no_weak":
            mask[mask == 1] = 2
        proj = nn.Linear(D, P) if P else None
        loss = ref_con.contrastive_loss_with_mask(mid, torch.from_numpy(mask).reshape(-1), proj)
        if loss.grad_fn is not None:
            loss.backward()
        out.update({f"{name}/middle": mid.detach().numpy(), f"{name}/mask": mask,
                    f"{name}/loss": loss.detach().numpy(),
                    f"{name}/grad_middle": mid.grad.numpy() if mid.grad is not None else np.zeros_like(mid.detach().numpy())})
        if proj is not None:
            out.update({f"{name}/w": proj.weight.detach().numpy(), f"{name}/b": proj.bias.detach().numpy(),
                        f"{name}/grad_w": proj.weight.grad.numpy() if proj.weight.grad is not None else np.zeros_like(proj.weight.detach().numpy()),
                        f"{name}/grad_b": proj.bias.grad.numpy() if proj.bias.grad is not None else np.zeros_like(proj.bias.detach().numpy())})
    np.savez_compressed(os.path.join(OUT, "infonce_cases.npz"), **out, **_meta())


def gen_step(ref_con, RefFusion, RefDecoder):
    """Hot-path half of train_epoch (trainer.py:98-119) from synthetic ENCODER FEATURES on, fp32 CPU."""
    torch.manual_seed(41)
    rng = np.random.default_rng(41)
    B, Tv, Tenc, N, dv, da, e, V, P = 3, 12, 19, 6200, 24, 40, 16, 30, 8
    fus = RefFusion(dv, da, e, num_heads=4)
    dec = RefDecoder(2 * e, V, blank_id=3)
    proj = nn.Linear(da, P)
    crit = nn.CTCLoss(blank=3, zero_infinity=True)
    out = {}
    losses = []
    total = 0
    contrast = 0
    for spk in (1, 2):
        vis = torch.randn(B, Tv, dv)
        aud = torch.randn(B, Tenc, da)
        mid = torch.randn(B, Tenc, da)
        mask = synth_mask(rng, B, N)
        lens = [4, 3, 5]
        text = make_targets(rng, B, 5, lens, V, 3)
        mask_t = torch.from_numpy(mask)
        mask_ds = F.interpolate(mask_t.unsqueeze(1).float(), size=Tenc, mode="nearest").squeeze(1).long()
        c = ref_con.contrastive_loss_with_mask(mid, mask_ds.reshape(B * Tenc), projection_layer=proj)
        fused, il = fus(vis, aud, mask=mask_ds)
        lp = dec(fused)
        l = crit(lp.transpose(0, 1), torch.from_numpy(text), il, torch.tensor(lens))
        total = total + l
        contrast = contrast + c
        out.update({f"spk{spk}/visual": vis.numpy(), f"spk{spk}/audio": aud.numpy(),
                    f"spk{spk}/middle": mid.numpy(), f"spk{spk}/mask": mask, f"spk{spk}/text": text,
                    f"spk{spk}/text_len": np.array(lens), f"spk{spk}/mask_ds": mask_ds.numpy(),
                    f"spk{spk}/ctc": l.detach().numpy(), f"spk{spk}/contrast": c.detach().numpy(),
                    f"spk{spk}/input_lengths": il.numpy()})
    loss_total = total / 2 + 0.1 * contrast / 2      # trainer.py:119, lambda_=0.1
    loss_total.backward()
    out["loss_total"] = loss_total.detach().numpy()
    out.update({f"param/{k}": v.detach().numpy() for k, v in fus.state_dict().items()})
    out.update({f"dec/{k}": v.detach().numpy() for k, v in dec.state_dict().items()})
    out.update({"proj/weight": proj.weight.detach().numpy(), "proj/bias": proj.bias.detach().numpy()})
    out.update({f"grad/{k}": (v.grad.numpy() if v.grad is not None else np.zeros(0, np.float32))
                for k, v in fus.named_parameters()})
    out.update({f"dec_grad/{k}": v.grad.numpy() for k, v in dec.named_parameters()})
    np.savez_compressed(os.path.join(OUT, "step_cases.npz"), **out, **_meta())


def main():
    os.makedirs(OUT, exist_ok=True)
    ref_beam, ref_con, RefFusion, RefDecoder = _import_reference()
    gen_ctc()
    gen_beam(ref_beam)
    gen_fusion(RefFusion, RefDecoder)
    gen_infonce(ref_con)
    gen_step(ref_con, RefFusion, RefDecoder)
    for f in sorted(os.listdir(OUT)):
        print(f, os.path.getsize(os.path.join(OUT, f)))


if __name__ == "__main__":
    main()
