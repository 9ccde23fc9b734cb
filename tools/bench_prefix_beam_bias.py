"""CTC prefix beam search with contextual biasing (avctc_ctc_prefix_beam_biased) timed on the GPU next to the same
search without a context (avctc_ctc_prefix_beam / avctc_ctc_prefix_beam_lm), on the shapes of
tools/bench_prefix_beam.py.  Prints ONE JSON line.

    python tools/bench_prefix_beam_bias.py [--iters 20] [--out profiles/r08_bench_prefix_beam_bias.json]

Contexts: seeded random phrase lists over the model pieces 4..799, 2..12 tokens each, weight 2.0: 100 phrases (a
table of a few MB) and 10 000 phrases (about 60 000 nodes x ~800 symbols, a transition table above the 126 MB L2).
Each is timed without an LM and with the order-2 LM of tools/bench_prefix_beam_lm.py (600k bigrams), lm_weight 0.5,
token_bonus 1.0.  Inputs are seeded log_softmax(3 * randn), blank 3.  Times are CUDA-event device times of one call
(both launches) with L2 overwritten (256 MB write) before every iteration; the six variants are alternated within
each iteration.  Sampled rows of the 10 000-phrase + LM variant are checked against the oracle.  The card's name and
power limit are read in the same run.
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

from bench import l2_flusher                      # noqa: E402
from bench_prefix_beam import SHAPES, card_info   # noqa: E402
from bench_prefix_beam_lm import ORDERS, V_LM, write_arpa   # noqa: E402

CONTEXTS = (100, 10_000)


def random_phrases(n, seed):
    rng = np.random.default_rng(seed)
    return [[int(c) for c in rng.integers(4, V_LM, size=int(rng.integers(2, 13)))] for _ in range(n)]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_prefix_beam_bias.py measures on a CUDA device; none found")
    import multimodal_av_model_b200 as pkg
    from multimodal_av_model_b200 import _lib
    from oracle import context_graph_oracle as CO
    from oracle import prefix_beam_lm_oracle as LO
    device = torch.device("cuda:0")
    flush = l2_flusher(device)
    L = _lib.lib()
    res = {"bench": "ctc_prefix_beam_biased", **card_info(), "cpu_cores": os.cpu_count(), "iters": args.iters,
           "timing": "CUDA events, L2 overwritten (256 MB) before every iteration, variants alternated; mean and min",
           "lm_order": 2, "lm_weight": 0.5, "token_bonus": 1.0, "phrase_weight": 2.0}
    vocab = [f"p{i}" for i in range(V_LM)]
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "o2.arpa")
        write_arpa(path, 2, ORDERS[2], seed=2)
        lm = pkg.NgramLM.from_arpa(path, vocab)
        olm = LO.read_arpa(path, vocab)
    phrases = {n: random_phrases(n, seed=n) for n in CONTEXTS}
    graphs = {}
    for n in CONTEXTS:
        for V in sorted({s[3] for s in SHAPES}):
            t0 = time.perf_counter()
            graphs[n, V] = pkg.ContextGraph.from_phrases(phrases[n], V, 3)
            if V == V_LM:
                g = graphs[n, V]
                res[f"ctx{n}"] = {"phrases": n, "nodes": g.num_nodes, "alphabet": g.alphabet,
                                  "table_bytes": g.table_bytes, "build_s": time.perf_counter() - t0}
    oac = CO.ContextAutomaton([(p, 2.0) for p in phrases[CONTEXTS[-1]]])
    for name, N, T, V, B in SHAPES:
        lp = (torch.randn(N, T, V, generator=torch.Generator().manual_seed(N * 7 + T)) * 3.0).log_softmax(-1)
        lpd = lp.to(device)
        st = _lib.stream_ptr(device)
        ws_b = int(L.avctc_ctc_prefix_beam_workspace_bytes(N, T, V, B))
        ws = torch.empty(ws_b, dtype=torch.uint8, device=device)
        tok = torch.empty((N, B, T), dtype=torch.int32, device=device)
        olen = torch.empty((N, B), dtype=torch.int32, device=device)
        osc = torch.empty((4, N, B), dtype=torch.float64, device=device)
        ost = torch.empty((N,), dtype=torch.int32, device=device)
        keep = []
        d = _lib.NgramLMDesc.from_buffer_copy(lm.descriptor(device))
        if V != lm.vocab_size:              # the long shape's 801st class reads as <unk> (word id 2)
            d.map_len = V
            tw = torch.cat([torch.from_numpy(lm._token_word), torch.tensor([2] * (V - lm.vocab_size),
                                                                           dtype=torch.int32)]).to(device)
            keep.append(tw)
            d.token_word = tw.data_ptr()
        keep.append(d)
        lm_ptr = ctypes.addressof(d)

        def plain():
            _lib.check(L.avctc_ctc_prefix_beam(lpd.data_ptr(), lpd.stride(0), lpd.stride(1), N, T, V, None, B, B, 3,
                                               tok.data_ptr(), olen.data_ptr(), osc[0].data_ptr(), ost.data_ptr(),
                                               ws.data_ptr(), ws_b, st), "prefix_beam")

        def fused():
            _lib.check(L.avctc_ctc_prefix_beam_lm(
                lpd.data_ptr(), lpd.stride(0), lpd.stride(1), N, T, V, None, B, B, 3, lm_ptr, 0.5, 1.0,
                tok.data_ptr(), olen.data_ptr(), osc[0].data_ptr(), osc[1].data_ptr(), osc[2].data_ptr(),
                ost.data_ptr(), ws.data_ptr(), ws_b, st), "prefix_beam_lm")

        def biased(ctx_ptr, with_lm):
            def run():
                _lib.check(L.avctc_ctc_prefix_beam_biased(
                    lpd.data_ptr(), lpd.stride(0), lpd.stride(1), N, T, V, None, B, B, 3,
                    lm_ptr if with_lm else None, 0.5, 1.0, ctx_ptr, tok.data_ptr(), olen.data_ptr(),
                    osc[0].data_ptr(), osc[1].data_ptr(), osc[2].data_ptr(), osc[3].data_ptr(), ost.data_ptr(),
                    ws.data_ptr(), ws_b, st), "prefix_beam_biased")
            return run

        variants = {"no_context": plain, "no_context_lm2": fused}
        for n in CONTEXTS:
            ptr = ctypes.addressof(graphs[n, V].descriptor(device))
            variants[f"ctx{n}"] = biased(ptr, False)
            variants[f"ctx{n}_lm2"] = biased(ptr, True)
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
        for n in CONTEXTS:
            r[f"ctx{n}_over_no_context"] = r[f"ctx{n}_ms"] / r["no_context_ms"]
            r[f"ctx{n}_lm2_over_no_context_lm2"] = r[f"ctx{n}_lm2_ms"] / r["no_context_lm2_ms"]
        if V == V_LM:                       # sampled rows against the oracle (10 000 phrases + the order-2 LM)
            got = pkg.ctc_prefix_beam_search(lpd, beam_width=B, nbest=B, blank=3, lm=lm, lm_weight=0.5,
                                             token_bonus=1.0, context=graphs[CONTEXTS[-1], V])
            lp_h = lp.numpy()
            rows = np.random.default_rng(0).choice(N, size=min(N, 4), replace=False).tolist()
            refs = [CO.prefix_beam_bias_search(lp_h[n], T, B, B, 3, oac, lm=olm, alpha=0.5, beta=1.0)[1]
                    for n in rows]
            r["oracle_rows_checked"] = len(rows)
            r["matches_oracle"] = all(
                [(h.tokens, h.score, h.acoustic_score, h.lm_score, h.bias_score) for h in got[n]] ==
                [(list(t), s, a, m, b) for t, s, a, m, b in ref] for n, ref in zip(rows, refs))
            r["bias_hits"] = int(sum(h.bias_score != 0.0 for row in got for h in row))
        res[name] = r
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
