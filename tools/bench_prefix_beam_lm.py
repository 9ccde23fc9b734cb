"""CTC prefix beam search with n-gram LM fusion (avctc_ctc_prefix_beam_lm) timed on the GPU next to the same search
without an LM (avctc_ctc_prefix_beam), on the shapes of tools/bench_prefix_beam.py.  Prints ONE JSON line.

    python tools/bench_prefix_beam_lm.py [--iters 20] [--out profiles/r07_bench_prefix_beam_lm.json]

LMs: seeded random ARPA files over the 800 model pieces, written to a temporary directory and loaded with
NgramLM.from_arpa: order 2 with 600k bigrams (most of the 800^2 possible ones; 32 MB of tables), and order 4 with
400k / 1.2M / 2.4M 2- / 3- / 4-grams (208 MB of tables, above the 126 MB L2).  Random n-grams make most lookups of a
decode miss and back off, the walk with the most probes.  Inputs are seeded log_softmax(3 * randn), blank 3,
lm_weight 0.5, token_bonus 1.0.  Times are CUDA-event device times of one call (both launches) with L2 overwritten
(256 MB write) before every iteration; the three variants are alternated within each iteration.  The oracle time is
per utterance on the host, with the order-4 LM.  The card's name and power limit are read in the same run.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench import l2_flusher                # noqa: E402
from bench_prefix_beam import SHAPES, card_info   # noqa: E402

V_LM = 800
ORDERS = {2: (600_000,), 4: (400_000, 1_200_000, 2_400_000)}


def write_arpa(path, order, counts, seed):
    """Seeded random token ARPA over pieces p0..p799: every piece, <s>, </s> and <unk> as 1-grams, then `counts`
    distinct random n-grams per order >= 2 (back-off weights on all but the highest order)."""
    rng = np.random.default_rng(seed)
    words = np.array(["<s>", "</s>", "<unk>"] + [f"p{i}" for i in range(V_LM)])
    nw = len(words)
    with open(path, "w", encoding="utf-8") as f:
        f.write("\\data\\\n" + "".join(f"ngram {n}={c}\n" for n, c in zip(range(1, order + 1),
                                                                       (nw,) + tuple(counts))) + "\n")
        f.write("\\1-grams:\n")
        for i, w in enumerate(words):
            f.write(f"{-99.0 if i == 0 else rng.uniform(-4, -1):.6f}\t{w}\t{rng.uniform(-1, 0):.6f}\n")
        for n, c in zip(range(2, order + 1), counts):
            f.write(f"\n\\{n}-grams:\n")
            ids = np.empty((0, n), dtype=np.int64)
            while len(ids) < c:                       # distinct n-grams: no word after </s>, no <s> inside
                cand = rng.integers(3, nw, size=(2 * c, n))
                cand[:, 0] = np.where(rng.random(2 * c) < 0.1, 0, cand[:, 0])
                cand[:, -1] = np.where(rng.random(2 * c) < 0.05, 1, cand[:, -1])
                ids = np.unique(np.concatenate([ids, cand]), axis=0)
            ids = ids[rng.permutation(len(ids))[:c]]
            lp = rng.uniform(-3, -0.1, size=c)
            bo = rng.uniform(-1, 0, size=c)
            text = [" ".join(words[r]) for r in ids]
            if n < order:
                f.write("".join(f"{a:.6f}\t{t}\t{b:.6f}\n" for a, t, b in zip(lp, text, bo)))
            else:
                f.write("".join(f"{a:.6f}\t{t}\n" for a, t in zip(lp, text)))
        f.write("\n\\end\\\n")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_prefix_beam_lm.py measures on a CUDA device; none found")
    import multimodal_av_model_b200 as pkg
    from multimodal_av_model_b200 import _lib
    from oracle import prefix_beam_lm_oracle as LO
    device = torch.device("cuda:0")
    flush = l2_flusher(device)
    L = _lib.lib()
    res = {"bench": "ctc_prefix_beam_lm", **card_info(), "cpu_cores": os.cpu_count(), "iters": args.iters,
           "timing": "CUDA events, L2 overwritten (256 MB) before every iteration, variants alternated; mean and min",
           "lm_weight": 0.5, "token_bonus": 1.0}
    vocab = [f"p{i}" for i in range(V_LM)]
    lms, olm = {}, None
    with tempfile.TemporaryDirectory() as tmp:
        for order, counts in ORDERS.items():
            path = os.path.join(tmp, f"o{order}.arpa")
            write_arpa(path, order, counts, seed=order)
            t0 = time.perf_counter()
            lms[order] = pkg.NgramLM.from_arpa(path, vocab)
            res[f"lm{order}"] = {"counts": list(lms[order].counts), "table_bytes": lms[order].table_bytes,
                                 "load_s": time.perf_counter() - t0}
            if order == 4:
                olm = LO.read_arpa(path, vocab)
    for name, N, T, V, B in SHAPES:
        lp = (torch.randn(N, T, V, generator=torch.Generator().manual_seed(N * 7 + T)) * 3.0).log_softmax(-1)
        lpd = lp.to(device)
        st = _lib.stream_ptr(device)
        ws_b = int(L.avctc_ctc_prefix_beam_workspace_bytes(N, T, V, B))
        ws = torch.empty(ws_b, dtype=torch.uint8, device=device)
        tok = torch.empty((N, B, T), dtype=torch.int32, device=device)
        olen = torch.empty((N, B), dtype=torch.int32, device=device)
        osc = torch.empty((3, N, B), dtype=torch.float64, device=device)
        ost = torch.empty((N,), dtype=torch.int32, device=device)

        def plain():
            _lib.check(L.avctc_ctc_prefix_beam(lpd.data_ptr(), lpd.stride(0), lpd.stride(1), N, T, V, None, B, B, 3,
                                               tok.data_ptr(), olen.data_ptr(), osc[0].data_ptr(), ost.data_ptr(),
                                               ws.data_ptr(), ws_b, st), "prefix_beam")

        def fused(desc):
            def run():
                _lib.check(L.avctc_ctc_prefix_beam_lm(
                    lpd.data_ptr(), lpd.stride(0), lpd.stride(1), N, T, V, None, B, B, 3, desc, 0.5, 1.0,
                    tok.data_ptr(), olen.data_ptr(), osc[0].data_ptr(), osc[1].data_ptr(), osc[2].data_ptr(),
                    ost.data_ptr(), ws.data_ptr(), ws_b, st), "prefix_beam_lm")
            return run

        variants = {"no_lm": plain}
        keep = []
        for order in ORDERS:
            lm = lms[order]
            d = _lib.NgramLMDesc.from_buffer_copy(lm.descriptor(device))
            if V != lm.vocab_size:              # the long shape's 801st class reads as <unk> (word id 2)
                d.map_len = V
                tw = torch.cat([torch.from_numpy(lm._token_word), torch.tensor([2] * (V - lm.vocab_size),
                                                                               dtype=torch.int32)]).to(device)
                keep.append(tw)
                d.token_word = tw.data_ptr()
            keep.append(d)
            variants[f"lm_order{order}"] = fused(ctypes.addressof(d))
        for fn in variants.values():
            for _ in range(3):
                fn()
        ts = {k: [] for k in variants}
        for _ in range(args.iters):
            for k, fn in variants.items():
                flush()
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record(); fn(); b.record()
                torch.cuda.synchronize(device)
                ts[k].append(a.elapsed_time(b))
        r = {"N": N, "T": T, "V": V, "beam": B, "blank": 3}
        for k, v in ts.items():
            r[f"{k}_ms"], r[f"{k}_min_ms"] = float(np.mean(v)), float(np.min(v))
        for order in ORDERS:
            r[f"lm_order{order}_over_no_lm"] = r[f"lm_order{order}_ms"] / r["no_lm_ms"]
        # sampled rows against the oracle (order-4 LM, the same 800 pieces), and its host time per utterance
        if V == V_LM:
            got = pkg.ctc_prefix_beam_search(lpd, beam_width=B, nbest=B, blank=3, lm=lms[4], lm_weight=0.5,
                                             token_bonus=1.0)
            lp_h = lp.numpy()
            rows = np.random.default_rng(0).choice(N, size=min(N, 4), replace=False).tolist()
            t0 = time.perf_counter()
            refs = [LO.prefix_beam_lm_search(lp_h[n], T, B, B, 3, olm, 0.5, 1.0)[1] for n in rows]
            r["oracle_cpu_ms_per_utterance"] = (time.perf_counter() - t0) * 1e3 / len(rows)
            r["oracle_rows_checked"] = len(rows)
            r["matches_oracle"] = all(
                [(h.tokens, h.score, h.acoustic_score, h.lm_score) for h in got[n]] ==
                [(list(t), s, a, m) for t, s, a, m in ref] for n, ref in zip(rows, refs))
        res[name] = r
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
