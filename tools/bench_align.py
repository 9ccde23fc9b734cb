"""Batched CTC forced alignment (csrc/ctc_align.cu) timed on the GPU, next to the forward-only CTC scan on the same
inputs and torchaudio's forced_align looped per utterance (CUDA and host CPU).  Prints ONE JSON line.

    python tools/bench_align.py [--iters 20] [--out FILE]

Shapes: (a) the evaluate() shape, N=16, T=150, V=800, L 20-58, blank 3; (b) BASELINE config 2, N=64, T=1000, V=801,
L 10-80, blank 0 (bench.ctc_case: the [T,B,V] tensor, aligned through its [B,T,V] transpose); each in fp32 and bf16.
Kernel times are CUDA-event device times with L2 overwritten (256 MB write) before every iteration, as bench.py does;
api_ms is the host wall-clock of one forced_align() call, which ends in its one status read-back.  The card's name and
power limit are read in the same run.
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

from bench import ctc_case, event_time, l2_flusher   # noqa: E402


def eval_case(device, dtype, N=16, T=150, V=800, blank=3, seed=150):
    g = torch.Generator().manual_seed(seed)
    lp = torch.randn(N, T, V, generator=g).log_softmax(-1).to(dtype).to(device)
    rng = np.random.default_rng(seed)
    tl = rng.integers(20, 59, size=N)
    Lm = int(tl.max())
    ids = np.array([c for c in range(V) if c != blank])
    tg = np.zeros((N, Lm), dtype=np.int64)
    il = np.zeros(N, dtype=np.int64)
    for n in range(N):
        row = rng.choice(ids, size=tl[n])
        tg[n, :tl[n]] = row
        il[n] = rng.integers(int(tl[n] + (row[1:] == row[:-1]).sum()), T + 1)
    t = lambda a: torch.from_numpy(a).to(device)
    return lp, t(tg), t(il), t(tl), Lm


def card_info():
    info = {"device": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit_and_max_sm_clock"] = q
    except Exception as e:  # noqa: BLE001
        info["power_limit_and_max_sm_clock"] = f"unavailable: {e}"
    return info


def bench_shape(name, lp_nbv, tg, il, tl, Lm, blank, iters, flush, device):
    """lp_nbv: [N,T,V] (possibly a strided view)."""
    import torchaudio.functional as TAF

    import multimodal_av_model_b200 as pkg
    from multimodal_av_model_b200 import _lib
    L = _lib.lib()
    N, T, V = lp_nbv.shape
    st = _lib.stream_ptr(lp_nbv.device)
    dt = _lib.dtype_enum(lp_nbv)
    paths = torch.empty((N, T), dtype=torch.int32, device=device)
    scores = torch.empty((N, T), dtype=lp_nbv.dtype, device=device)
    status = torch.empty((N,), dtype=torch.int32, device=device)
    nll = torch.empty(N, device=device)

    def align():
        _lib.check(L.avctc_ctc_align(lp_nbv.data_ptr(), dt, lp_nbv.stride(0), lp_nbv.stride(1), N, T, V, tg.data_ptr(),
                                     tg.stride(0), il.data_ptr(), tl.data_ptr(), Lm, blank, paths.data_ptr(),
                                     scores.data_ptr(), status.data_ptr(), st), "align")

    def scan():        # forward-only CTC: the same lattice chain with log-sum-exp (stride_t, stride_b of the [T,B,V] view)
        _lib.check(L.avctc_ctc_forward(lp_nbv.data_ptr(), dt, lp_nbv.stride(1), lp_nbv.stride(0), T, N, V, tg.data_ptr(),
                                       tg.stride(0), None, il.data_ptr(), tl.data_ptr(), Lm, blank, 0, nll.data_ptr(),
                                       None, 0, st), "ctc_forward")

    r = {"N": N, "T": T, "V": V, "Lmax": Lm, "blank": blank, "dtype": str(lp_nbv.dtype).replace("torch.", "")}
    r["align_ms"], r["align_min_ms"] = event_time(align, iters, 3, flush, device)
    r["ctc_forward_ms"], r["ctc_forward_min_ms"] = event_time(scan, iters, 3, flush, device)
    r["align_over_ctc_forward"] = r["align_ms"] / r["ctc_forward_ms"]
    torch.cuda.synchronize(device)
    ts = []
    for _ in range(5):
        flush()
        torch.cuda.synchronize(device)
        t0 = time.perf_counter()
        p_api, s_api = pkg.forced_align(lp_nbv, tg, il, tl, blank=blank)
        ts.append((time.perf_counter() - t0) * 1e3)
    r["api_ms"] = float(np.mean(ts))
    # torchaudio, one utterance per call (its forced_align takes no batch and no padding); results compared too
    ilh, tlh = il.cpu().tolist(), tl.cpu().tolist()
    lp_h = lp_nbv.float().cpu()
    tg_h = tg.cpu()
    per = [(lp_h[n:n + 1, :ilh[n]].contiguous(), tg_h[n:n + 1, :tlh[n]].contiguous()) for n in range(N)]
    p_cpu = [TAF.forced_align(a, b, blank=blank) for a, b in per]
    same = all(torch.equal(p_api[n, :ilh[n]].cpu(), p_cpu[n][0][0]) and
               torch.equal(s_api[n, :ilh[n]].float().cpu(), p_cpu[n][1][0]) for n in range(N))
    r["matches_torchaudio_cpu"] = bool(same)
    t0 = time.perf_counter()
    for a, b in per:
        TAF.forced_align(a, b, blank=blank)
    r["torchaudio_cpu_loop_ms"] = (time.perf_counter() - t0) * 1e3
    r["cpu_threads"] = torch.get_num_threads()
    try:
        per_d = [(a.to(device).to(lp_nbv.dtype), b.to(device)) for a, b in per]

        def ta_cuda():
            for a, b in per_d:
                TAF.forced_align(a, b, blank=blank)
        ta_cuda()
        torch.cuda.synchronize(device)
        t0 = time.perf_counter()
        for _ in range(3):
            ta_cuda()
        torch.cuda.synchronize(device)
        r["torchaudio_cuda_loop_ms"] = (time.perf_counter() - t0) * 1e3 / 3
    except Exception as e:  # noqa: BLE001
        r["torchaudio_cuda_loop_ms"] = None
        r["torchaudio_cuda_error"] = f"{type(e).__name__}: {str(e).splitlines()[0][:200]}"
    return name, r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_align.py measures on a CUDA device; none found")
    device = torch.device("cuda:0")
    flush = l2_flusher(device)
    res = {"bench": "ctc_forced_align", **card_info(), "cpu_cores": os.cpu_count(), "iters": args.iters,
           "timing": "CUDA events, L2 overwritten (256 MB) before every iteration; mean and min over iters"}
    for dtype in (torch.float32, torch.bfloat16):
        tag = "fp32" if dtype == torch.float32 else "bf16"
        lp, tg, il, tl, Lm = eval_case(device, dtype)
        k, v = bench_shape(f"eval_{tag}", lp, tg, il, tl, Lm, 3, args.iters, flush, device)
        res[k] = v
        lp, tg, il, tl, Lm = ctc_case(1000, device, dtype=dtype)
        k, v = bench_shape(f"config2_{tag}", lp.transpose(0, 1), tg, il, tl, Lm, 0, args.iters, flush, device)
        res[k] = v
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
