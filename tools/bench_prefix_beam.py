"""CTC prefix beam search (csrc/ctc_prefix_beam.cu) timed on the GPU, next to the reference-semantics beam decode
(avctc_beam_search) on the same inputs, torchaudio's cuda_ctc_decoder and the CPU oracle.  Prints ONE JSON line.

    python tools/bench_prefix_beam.py [--iters 20] [--out FILE]

Shapes: (16, 150, 800, B=5) = evaluate() of 8 pairs; (4096, 150, 800, B=10) = a large batch of short utterances;
(64, 1000, 801, B=10) = long utterances.  Inputs are seeded log_softmax(3 * randn) with blank 3.  Kernel times are
CUDA-event device times with L2 overwritten (256 MB write) before every iteration; api_ms is the host wall-clock of one
ctc_prefix_beam_search() call, which ends in its one read-back.  torchaudio's decoder only takes blank = 0 and skips
frames whose blank probability exceeds blank_skip_threshold, so it runs at blank = 0 on the same log-probs with
thresholds 1.0 and 0.95; its top-1 agreement with this search at blank = 0 is reported, not asserted.  The oracle time
is per utterance on the host.  The card's name and power limit are read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from bench import event_time, l2_flusher   # noqa: E402

SHAPES = [("eval", 16, 150, 800, 5), ("large_batch", 4096, 150, 800, 10), ("long", 64, 1000, 801, 10)]


def card_info():
    info = {"device": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit_and_max_sm_clock"] = q
    except Exception as e:  # noqa: BLE001
        info["power_limit_and_max_sm_clock"] = f"unavailable: {e}"
    return info


def _wall(fn, iters, flush, device):
    ts = []
    for _ in range(iters):
        flush()
        torch.cuda.synchronize(device)
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize(device)
        ts.append((time.perf_counter() - t0) * 1e3)
    return float(np.mean(ts))


def bench_shape(name, N, T, V, B, iters, flush, device):
    import multimodal_av_model_b200 as pkg
    from multimodal_av_model_b200 import _lib
    from oracle import prefix_beam_oracle as O
    L = _lib.lib()
    blank = 3
    g = torch.Generator().manual_seed(N * 7 + T)
    lp = (torch.randn(N, T, V, generator=g) * 3.0).log_softmax(-1).to(device)
    st = _lib.stream_ptr(lp.device)
    r = {"N": N, "T": T, "V": V, "beam": B, "blank": blank}

    ws_b = int(L.avctc_ctc_prefix_beam_workspace_bytes(N, T, V, B))
    ws = torch.empty(ws_b, dtype=torch.uint8, device=device)
    tok = torch.empty((N, B, T), dtype=torch.int32, device=device)
    olen = torch.empty((N, B), dtype=torch.int32, device=device)
    osc = torch.empty((N, B), dtype=torch.float64, device=device)
    ost = torch.empty((N,), dtype=torch.int32, device=device)

    def prefix():
        _lib.check(L.avctc_ctc_prefix_beam(lp.data_ptr(), lp.stride(0), lp.stride(1), N, T, V, None, B, B, blank,
                                           tok.data_ptr(), olen.data_ptr(), osc.data_ptr(), ost.data_ptr(),
                                           ws.data_ptr(), ws_b, st), "prefix_beam")

    bws_b = int(L.avctc_beam_workspace_bytes(N, T, V, B))
    bws = torch.empty(bws_b, dtype=torch.uint8, device=device)
    ids = torch.empty((N, T), dtype=torch.int32, device=device)
    ilen = torch.empty((N,), dtype=torch.int32, device=device)

    def reference_beam():
        _lib.check(L.avctc_beam_search(lp.data_ptr(), lp.stride(0), lp.stride(1), N, T, V, None, B, blank,
                                       ids.data_ptr(), ilen.data_ptr(), None, None, bws.data_ptr(), bws_b, st), "beam")

    r["prefix_beam_ms"], r["prefix_beam_min_ms"] = event_time(prefix, iters, 3, flush, device)
    r["beam_search_ms"], r["beam_search_min_ms"] = event_time(reference_beam, iters, 3, flush, device)
    r["prefix_over_beam_search"] = r["prefix_beam_ms"] / r["beam_search_ms"]
    r["api_ms"] = _wall(lambda: pkg.ctc_prefix_beam_search(lp, beam_width=B, nbest=1, blank=blank), 5, flush, device)

    # bit-exactness of sampled rows against the oracle, and its host time per utterance
    ours = pkg.ctc_prefix_beam_search(lp, beam_width=B, nbest=B, blank=blank)
    lp_h = lp.cpu().numpy()
    rows = np.random.default_rng(0).choice(N, size=min(N, 8), replace=False).tolist()
    t0 = time.perf_counter()
    refs = [O.prefix_beam_search(lp_h[n], T, B, B, blank)[1] for n in rows]
    r["oracle_cpu_ms_per_utterance"] = (time.perf_counter() - t0) * 1e3 / len(rows)
    r["oracle_rows_checked"] = len(rows)
    r["matches_oracle"] = all([(h.tokens, h.score) for h in ours[n]] == [(list(t), s) for t, s in ref]
                              for n, ref in zip(rows, refs))

    # torchaudio's CUDA prefix beam search (blank = 0 only)
    try:
        from torchaudio.models.decoder import cuda_ctc_decoder
        ours0 = pkg.ctc_prefix_beam_search(lp, beam_width=B, nbest=1, blank=0)
        lens32 = torch.full((N,), T, dtype=torch.int32, device=device)
        for thr in (1.0, 0.95):
            dec = cuda_ctc_decoder([str(i) for i in range(V)], nbest=1, beam_size=B, blank_skip_threshold=thr)
            out = dec(lp, lens32)
            key = f"cuda_ctc_decoder_skip{thr}"
            r[key + "_ms"] = _wall(lambda: dec(lp, lens32), iters, flush, device)
            agree = sum(1 for n in range(N) if out[n][0].tokens == (ours0[n][0].tokens if ours0[n] else None))
            r[key + "_top1_agreement"] = agree / N
    except Exception as e:  # noqa: BLE001
        r["cuda_ctc_decoder_error"] = f"{type(e).__name__}: {str(e).splitlines()[0][:200] if str(e) else ''}"
    return name, r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_prefix_beam.py measures on a CUDA device; none found")
    device = torch.device("cuda:0")
    flush = l2_flusher(device)
    res = {"bench": "ctc_prefix_beam", **card_info(), "cpu_cores": os.cpu_count(), "iters": args.iters,
           "timing": "CUDA events, L2 overwritten (256 MB) before every iteration; mean and min over iters"}
    for name, N, T, V, B in SHAPES:
        k, v = bench_shape(name, N, T, V, B, args.iters, flush, device)
        res[k] = v
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
