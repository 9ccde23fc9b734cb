"""oracle/align_oracle.py — CTC forced alignment: a numpy restatement of torchaudio's CPU forced_align, and the
generator of tests/golden/align_cases.npz.  TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).

    python oracle/align_oracle.py          # rewrites tests/golden/align_cases.npz (needs torchaudio, CPU only)

The fixture is torchaudio.functional.forced_align and merge_tokens run on the CPU, one utterance per case (torchaudio
version stored in it): random, tie-heavy (quantized log-probs), tight T = L+R, repeat-heavy, blank != 0 and V = 800.
ctc_forced_align below matches it bit for bit (tests/test_align_cpu.py).
"""
from __future__ import annotations

import os

import numpy as np

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden", "align_cases.npz")


def ctc_forced_align(log_probs, targets, blank=0):
    """torchaudio.functional.forced_align on CPU (torchaudio 2.11, libtorchaudio forced_align/cpu/compute.cpp) for
    ONE utterance: log_probs [T,V] (float32, or anything that upcasts to it exactly), targets [L] int.
    Returns (paths [T] int64, scores [T] float32 = log_probs[t, paths[t]]).  Viterbi over the [2L+1] CTC lattice
    in float32 with torchaudio's comparison order and frame window; vectorised over states per frame.
    L = 0 aligns every frame to blank (torchaudio cannot express it).  Raises ValueError for T < L + R."""
    lp = np.asarray(log_probs, dtype=np.float32)
    tg = np.asarray(targets, dtype=np.int64).reshape(-1)
    T, L = lp.shape[0], len(tg)
    if L == 0:
        paths = np.full(T, blank, dtype=np.int64)
        return paths, lp[np.arange(T), paths]
    S = 2 * L + 1
    R = int((tg[1:] == tg[:-1]).sum())
    if T < L + R:
        raise ValueError(f"T={T} < L+R={L + R}")
    lab = np.full(S, blank, dtype=np.int64)
    lab[1::2] = tg
    skip = np.zeros(S, dtype=bool)
    skip[3::2] = tg[1:] != tg[:-1]
    diff = np.zeros(L + 1, dtype=bool)              # diff[j] = tg[j] != tg[j-1]; out of range -> False
    diff[1:L] = tg[1:] != tg[:-1]
    ninf = np.float32(-np.inf)
    alpha = np.full(S, ninf, dtype=np.float32)
    start = 0 if T - (L + R) > 0 else 1
    end = 2
    alpha[start:end] = lp[0, lab[start:end]]
    bp = np.full((T, S), -1, dtype=np.int8)
    states = np.arange(S)
    for t in range(1, T):
        if T - t <= L + R:
            start += 2 if (start % 2 == 1 and diff[min(start // 2 + 1, L)]) else 1
        if t <= L + R:
            end += 2 if (end % 2 == 0 and end < 2 * L and diff[end // 2]) else 1
        x0 = alpha
        x1 = np.concatenate(([ninf], alpha[:-1]))
        x2 = np.where(skip, np.concatenate(([ninf, ninf], alpha[:-2])), ninf)
        c2 = (x2 > x1) & (x2 > x0)
        c1 = ~c2 & (x1 > x0) & (x1 > x2)
        pick = np.where(c2, x2, np.where(c1, x1, x0))
        win = (states >= start) & (states < end)
        alpha = np.where(win, pick + lp[t, lab], ninf).astype(np.float32)
        bp[t] = np.where(win, np.where(c2, 2, np.where(c1, 1, 0)), -1)
    s = S - 1 if alpha[S - 1] > alpha[S - 2] else S - 2
    paths = np.empty(T, dtype=np.int64)
    for t in range(T - 1, -1, -1):
        paths[t] = lab[s]
        s = min(s - int(bp[t, s]), S - 1)
    return paths, lp[np.arange(T), paths]


def _targets(rng, L, V, blank, repeat_frac):
    ids = np.array([c for c in range(V) if c != blank])
    row = rng.choice(ids, size=L)
    for j in range(1, L):
        if rng.random() < repeat_frac:
            row[j] = row[j - 1]
    return row.astype(np.int64)


def gen_align(path=OUT):
    """torchaudio.functional.forced_align (CPU) on one utterance per case, plus its merge_tokens spans."""
    import torch
    import torchaudio
    import torchaudio.functional as TAF
    rng = np.random.default_rng(23)
    # (name, T extra over L+R, L, V, blank, repeat fraction, quantization step of the logits (0 = none))
    specs = [("random", 60, 25, 30, 0, 0.1, 0), ("random_long", 150, 60, 12, 0, 0.1, 0),
             ("ties_half", 30, 20, 10, 0, 0.1, 0.5), ("ties_int", 20, 15, 6, 2, 0.2, 1.0),
             ("ties_flat", 10, 12, 5, 0, 0.2, 8.0), ("tight", 0, 30, 20, 0, 0.3, 0),
             ("tight_norep", 0, 25, 40, 1, 0.0, 0), ("tight_ties", 0, 18, 8, 0, 0.3, 1.0),
             ("slack1", 1, 20, 16, 0, 0.3, 0), ("repeats", 30, 30, 8, 0, 0.6, 0),
             ("blank3", 40, 20, 25, 3, 0.1, 0), ("blank_last", 40, 20, 25, 24, 0.1, 0),
             ("v800", 10, 10, 800, 3, 0.1, 0), ("one_label", 5, 1, 7, 0, 0.0, 0), ("one_frame", 0, 1, 7, 0, 0.0, 0)]
    out = {"names": np.array([s[0] for s in specs])}
    for i, (name, extra, L, V, blank, rep, q) in enumerate(specs):
        tg = _targets(rng, L, V, blank, rep)
        R = int((tg[1:] == tg[:-1]).sum())
        T = L + R + extra
        z = rng.standard_normal((T, V)).astype(np.float32)
        if q:
            z = np.round(z / q) * q
        lp = torch.from_numpy(z).log_softmax(-1)
        if q:
            lp = torch.round(lp * 4) / 4           # many exactly equal lattice scores
        paths, scores = TAF.forced_align(lp[None], torch.from_numpy(tg)[None], blank=blank)
        spans = TAF.merge_tokens(paths[0], scores[0], blank=blank)
        out[f"c{i}/lp"] = lp.numpy()
        out[f"c{i}/targets"] = tg
        out[f"c{i}/blank"] = np.array(blank)
        out[f"c{i}/paths"] = paths[0].numpy()
        out[f"c{i}/scores"] = scores[0].numpy()
        out[f"c{i}/spans"] = np.array([[sp.token, sp.start, sp.end] for sp in spans], dtype=np.int64).reshape(-1, 3)
        out[f"c{i}/span_scores"] = np.array([sp.score for sp in spans], dtype=np.float64)
    meta = {"torch_version": np.array(torch.__version__), "torchaudio_version": np.array(torchaudio.__version__),
            "generator": np.array("oracle/align_oracle.py"),
            "source": np.array("torchaudio.functional.forced_align / merge_tokens, CPU")}
    np.savez_compressed(path, **out, **meta)
    return path


if __name__ == "__main__":
    p = gen_align()
    print(p, os.path.getsize(p))
