#!/usr/bin/env python
"""bench.py — the AV-CTC hot path on B200, next to the reference's CPU path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload train|ctc|beam|fusion|infonce]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

Headline (BASELINE.json metric "train utt/s at 1/2/4/8 B200; CTC loss GB/s; beam-search decode utt/s"):
  workload = BASELINE config 4: full AV-CTC + InfoNCE training step, 8 utterance pairs per GPU, 5 s of 16 kHz
  audio (T_enc 249) + 150 lip frames, 800-piece vocab (blank 3), random-init encoders, utterance-sharded data
  parallel.  "value" = utterances/s of the whole job with the batch resident in HBM; "e2e" = the same step fed
  from pinned host memory through MultimodalTrainer.train_step (H2D of the batch and a blocking D2H read of the loss
  inside the timed region, every step; e2e.epoch_* = the same steps through MultimodalTrainer.train_epoch).  The same JSON line carries the other two parts of the metric measured live:
  "ctc" (config 2, GB/s, the "roofline" object is this kernel pair), "beam" (config 5, utt/s), plus "fusion"
  (config 3, tensor-pipe fraction) and "hot_path" (the step from encoder features on).
  Every sub-benchmark carries, next to the sm_100a kernels, (1) the reference's arithmetic on the box's host cores
  ("cpu": torch CPU ops = what the reference executes, core count stated) and (2) the stock-torch CUDA formulation on
  the same B200 ("torch_cuda_ms": ATen/cuDNN/cuBLAS kernels, the library bar).  Rank 0 at N=1 only.
  --impl reference times the reference's train step on the host CPU: oracle/torch_port.py + oracle/encoder_port.py (the
  reference modules restated on stock torch/HF ops; /root/reference itself cannot travel to the GPU box), same config.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np
import torch

PAIRS_PER_GPU = 8          # main.py:88 batch_size=8 pairs -> 16 utterance streams per step per GPU
SECONDS = 5.0
T_V = 150
VOCAB, BLANK = 800, 3


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sustained=d["bf16_tflops_sustained"], src="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sustained=1400.0, src="fallback")


class ClockSampler:
    """nvidia-smi clocks/throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *a):
        if self.proc:
            time.sleep(0.15)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                pass

    def summary(self):
        sm, mx, reasons = [], 0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx = max(mx, float(r[1]))
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                continue
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons),
                "samples": len(sm)}


# ------------------------------------------------------------------------------------------------ GPU arm
class _NoEncoder(torch.nn.Module):
    def forward(self, *a, **k):
        raise RuntimeError("hot-path-only benchmark: the encoders are not built")


def build_models(device, seed=0, encoders=True):
    import multimodal_av_model_b200 as pkg
    from multimodal_av_model_b200.encoders import unfreeze_middle_layers, xlsr_large_config
    from multimodal_av_model_b200.synthetic import CharTokenizer
    torch.manual_seed(seed)
    np.random.seed(seed)        # wav2vec2's SpecAugment spans come from numpy's global generator: same args, same outputs
    if not encoders:
        fus = pkg.CrossAttentionFusion(512, 1024, 512)
        dec = pkg.CTCDecoder(1024, VOCAB, blank_id=BLANK)
        tr = pkg.MultimodalTrainer(_NoEncoder(), _NoEncoder(), fus, dec, CharTokenizer(VOCAB), device=device)
        tr.verbose = False
        fus.train(); dec.train()
        return tr
    vis = pkg.VisualEncoder(relu_type="prelu")
    for p in vis.parameters():                 # main.py:100-103
        p.requires_grad = False
    aud = pkg.AudioEncoder(freeze=True, config=xlsr_large_config())
    unfreeze_middle_layers(aud.model)          # main.py:105-106
    fus = pkg.CrossAttentionFusion(512, 1024, 512)
    dec = pkg.CTCDecoder(1024, VOCAB, blank_id=BLANK)
    tr = pkg.MultimodalTrainer(vis, aud, fus, dec, CharTokenizer(VOCAB), device=device)
    tr.verbose = False
    for m in (vis, aud, fus, dec):
        m.train()
    return tr


GC_LOG = {}      # label -> Python garbage collections inside a timed region (count per generation, milliseconds)


def timed_loop(fn, steps, warmup, device, world, label=None):
    import gc
    import torch.distributed as dist
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize(device)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize(device)
    stat = {"collections": [0, 0, 0], "ms": 0.0, "t0": 0.0}

    def on_gc(phase, info):
        if phase == "start":
            stat["t0"] = time.perf_counter()
        else:
            stat["collections"][info["generation"]] += 1
            stat["ms"] += (time.perf_counter() - stat["t0"]) * 1e3
    if label:
        gc.callbacks.append(on_gc)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        fn()
    b.record()
    torch.cuda.synchronize(device)
    if label:
        gc.callbacks.remove(on_gc)
        GC_LOG[label] = {"collections": stat["collections"], "ms": round(stat["ms"], 2)}
    if world > 1:
        dist.barrier()
    ms = torch.tensor([a.elapsed_time(b)], device=device)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    return float(ms.item())


def dump_outputs(path, tr, loss):
    """--dump-outputs: what the last timed train step produced, as the trainer reports it per step (train_epoch's log
    line), so that two builds can be compared output for output: the total loss train_step returned, its four terms and
    speaker 1's CTC log-probs [B, T, V], as <path>/{loss,ctc1,ctc2,contrastive1,contrastive2,log_probs}.npy in float32.
    The step's gradients and updated weights are not written: the gradient reductions add float partial sums with
    atomics, and where a gradient is only rounding noise (the attention key biases, whose exact gradient is zero) Adam
    turns that noise into whole learning-rate steps of either sign, so they differ from run to run by more than rounding.
    The loss terms and log-probs agree to rounding."""
    c1, c2, k1, k2 = tr._last_parts
    out = {"loss": loss, "ctc1": c1, "ctc2": c2, "contrastive1": k1, "contrastive2": k2,
           "log_probs": tr._last_log_probs}
    os.makedirs(path, exist_ok=True)
    for k, t in out.items():
        np.save(os.path.join(path, k + ".npy"), t.detach().float().cpu().numpy())


def bench_train(args, rank, local, world, device, hot_only=False):
    from multimodal_av_model_b200 import _lib
    from multimodal_av_model_b200.synthetic import make_batch
    tr = build_models(device, encoders=not hot_only)
    utt_per_step = 2 * PAIRS_PER_GPU * world
    out = {}
    if not hot_only:
        host = make_batch(pairs=PAIRS_PER_GPU, seconds=SECONDS, t_v=T_V, vocab=VOCAB, seed=1234 + rank, pin=True)
        dev_batch = {k: v.to(device) for k, v in host.items()}
        last = {}

        def step_resident():
            last["loss"] = tr.train_step(dev_batch)

        def step_e2e():
            return float(tr.train_step(host))          # H2D of the pinned batch + D2H read of the loss

        c0 = _lib.launch_count
        with ClockSampler(local) as cs:
            ms = timed_loop(step_resident, args.steps, args.warmup, device, world, label="value")
        launches = (_lib.launch_count - c0) // (args.steps + args.warmup)
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, tr, last["loss"])
        ms_e2e = timed_loop(step_e2e, args.steps, max(1, args.warmup // 2), device, world, label="e2e")
        # the same K steps through MultimodalTrainer.train_epoch (main.py:165): batch i+1 staged on a side stream while step i
        # runs, each step's loss sent to the pinned trainer.loss_log without blocking, one host sync at the end of the epoch
        epoch_batches = [host] * args.steps
        tr.train_epoch([host] * max(1, args.warmup // 2))
        ms_epoch = timed_loop(lambda: tr.train_epoch(epoch_batches), 1, 0, device, world, label="epoch")
        assert tr.last_epoch_steps == args.steps and tr.loss_log_count == args.steps
        h2d = int(sum(v.numel() * v.element_size() for k, v in host.items() if not k.endswith("_lengths") or k.startswith("text")))
        grad_params = sum(p.numel() for p in tr.parameters if p.requires_grad)
        out = dict(value=utt_per_step * args.steps / (ms / 1e3), ms_per_step=ms / args.steps,
                   e2e=dict(value=utt_per_step * args.steps / (ms_e2e / 1e3), unit="utt/s", h2d_bytes_per_step=h2d,
                            d2h_bytes_per_step=4, ms_per_step=ms_e2e / args.steps,
                            api="MultimodalTrainer.train_step(pinned host batch) + float(loss): H2D of the batch and a blocking "
                                "D2H read-back of the loss every step",
                            epoch_ms_per_step=ms_epoch / args.steps,
                            epoch_value=utt_per_step * args.steps / (ms_epoch / 1e3),
                            epoch_note="the same K steps through MultimodalTrainer.train_epoch: next batch staged on a side stream, "
                                       "per-step loss copied asynchronously into the pinned loss_log, one sync per epoch"),
                   gpu_launches=int(launches), clocks=cs.summary(), host_gc=dict(GC_LOG), allreduce_bytes_per_step=grad_params * 4 if world > 1 else 0)
        del dev_batch
    # hot path only (SURVEY.md §8d config 4, number A): from encoder features on, same trainer
    from multimodal_av_model_b200.synthetic import make_features
    f = make_features(pairs=PAIRS_PER_GPU, t_v=T_V, t_enc=249, seed=1234 + rank, dtype=torch.bfloat16)
    fd = {k: [t.to(device) for t in v] for k, v in f.items()}
    for k in ("audio", "middle"):
        fd[k] = [t.requires_grad_() for t in fd[k]]

    def hot_step():
        if tr._reducer is not None:
            tr._reducer.zero_grad()
        else:
            tr.optimizer.zero_grad(set_to_none=True)
        for k in ("audio", "middle"):
            for t in fd[k]:
                t.grad = None
        with torch.autocast("cuda", dtype=torch.bfloat16):
            total = tr.hot_path_loss(fd["visual"], fd["audio"], fd["middle"], fd["masks"], fd["texts"], fd["lens"])[0]
        total.backward()
        if tr._reducer is not None:
            tr._reducer.finish()
    ms_hot = timed_loop(hot_step, args.steps, args.warmup, device, world)
    out["hot_path"] = dict(value=utt_per_step * args.steps / (ms_hot / 1e3), unit="utt/s", ms_per_step=ms_hot / args.steps,
                           note="fusion+BiLSTM+CTC head+CTC+InfoNCE fwd+bwd from encoder features on (no encoders, no optimizer)")
    if world == 1 and not args.no_comparators:
        out["hot_path"].update(hot_path_comparators(tr, f, device, args))
    return out, tr



def hot_path_comparators(tr, f, device, args):
    """The same hot-path step (a) on the stock torch CUDA kernels of the same box — the reference's modules restated in
    oracle/torch_port.py moved to the GPU under bf16 autocast: cuBLAS projections, unfused MHA, cuDNN LSTM, ATen
    log_softmax / CTC / InfoNCE ops (SURVEY.md §2.1, the library kernels to beat) — and (b) on the host CPU in fp32."""
    from oracle import torch_port as tp
    res = {}
    torch.manual_seed(0)
    ref_f, ref_d, proj = tp.FusionPort(512, 1024, 512), tp.DecoderPort(1024, VOCAB, BLANK), torch.nn.Linear(1024, 128)
    ref_f.load_state_dict(tr.fusion_module.state_dict()); ref_d.load_state_dict(tr.decoder1.state_dict())

    def feats_on(dev, dtype):
        return [dict(visual=f["visual"][s].to(dev, dtype), audio=f["audio"][s].to(dev, dtype).requires_grad_(),
                     middle=f["middle"][s].to(dev, dtype).requires_grad_(), mask=f["masks"][s].to(dev),
                     text=f["texts"][s].to(dev), text_len=f["lens"][s].to(dev)) for s in range(2)]
    mods = [m.to(device) for m in (ref_f, ref_d, proj)]
    fg = feats_on(device, torch.bfloat16)

    def stock():
        for m in mods:
            m.zero_grad(set_to_none=True)
        with torch.autocast("cuda", dtype=torch.bfloat16):
            loss = tp.hot_path_losses(mods[0], mods[1], mods[2], fg, blank=BLANK)
        loss.backward()
    ms = timed_loop(stock, max(3, args.steps // 2), 3, device, 1) / max(3, args.steps // 2)
    res["torch_cuda_ms_per_step"] = ms
    res["torch_cuda_note"] = "oracle/torch_port modules on cuda, bf16 autocast: cuBLAS + unfused MHA + cuDNN LSTM + ATen CTC"
    mods = [m.to("cpu") for m in mods]
    fc = feats_on("cpu", torch.float32)
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)

    def cpu():
        for m in mods:
            m.zero_grad(set_to_none=True)
        tp.hot_path_losses(mods[0], mods[1], mods[2], fc, blank=BLANK).backward()
    cpu()
    t0 = time.perf_counter(); cpu(); dt = time.perf_counter() - t0
    res["cpu"] = {"ms_per_step": dt * 1e3, "value": 2 * PAIRS_PER_GPU / dt, "unit": "utt/s", "cores": threads, "kind": "port",
                  "sample": "1 step (after 1 warm-up) of the same 8-pair hot-path step, torch CPU ops fp32 (oracle/torch_port.py)"}
    return res


def cpu_time(fn, reps=2, warm=1):
    for _ in range(warm):
        fn()
    t0 = time.perf_counter()
    for _ in range(reps):
        fn()
    return (time.perf_counter() - t0) / reps * 1e3

def l2_flusher(device):
    buf = torch.empty(256 << 20, dtype=torch.uint8, device=device)
    return lambda: buf.zero_()


def event_time(fn, iters, warm, flush, device):
    for _ in range(warm):
        fn()
    ts = []
    for _ in range(iters):
        flush()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); fn(); b.record()
        torch.cuda.synchronize(device)
        ts.append(a.elapsed_time(b))
    return float(np.mean(ts)), float(np.min(ts))


def event_time_queued(fn, iters, warm, flush, device, hold_cycles=700000):
    """Device time of what fn enqueues, with the launch queue pre-filled: a spin kernel (~350 us) holds the GPU while the
    host enqueues fn's kernels, so the interval between the two events is the kernels' own back-to-back duration — what
    a GPU-bound training step (or a CUDA-graph replay) sees — not the host's enqueue latency."""
    for _ in range(warm):
        fn()
    ts = []
    for _ in range(iters):
        flush()
        torch.cuda._sleep(hold_cycles)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); fn(); b.record()
        torch.cuda.synchronize(device)
        ts.append(a.elapsed_time(b))
    return float(np.mean(ts)), float(np.min(ts))


def ctc_case(T, device, B=64, V=801, blank=0, dtype=torch.float32):
    g = torch.Generator().manual_seed(T)
    lp = torch.randn(T, B, V, generator=g).log_softmax(-1).to(dtype).to(device)
    rng = np.random.default_rng(T)
    hi = min(80, T // 2 - 1)
    tl = rng.integers(10, hi + 1, size=B)
    Lm = int(tl.max())
    il = rng.integers(max(2 * Lm + 1, T // 2), T + 1, size=B)
    ids = np.array([c for c in range(V) if c != blank])
    tg = np.zeros((B, Lm), dtype=np.int64)
    for b in range(B):
        row = rng.choice(ids, size=tl[b])
        for j in range(1, tl[b]):
            if rng.random() < 0.1:
                row[j] = row[j - 1]
        tg[b, :tl[b]] = row
    return lp, torch.from_numpy(tg).to(device), torch.from_numpy(il).to(device), torch.from_numpy(tl).to(device), Lm


def bench_ctc(device, iters=10, Ts=(250, 1000), comparators=True):
    """BASELINE config 2.  product_ms = pkg.ctc_loss(x, ...).backward() — the autograd route a trainer uses: the scan, the
    reduction and the gradient pass are enqueued back to back at forward time (ctc.py), backward() applies grad_out —
    as DEVICE time (launch queue pre-filled behind a spin kernel, event_time_queued); product_eager_ms = the same call
    timed from an idle GPU, i.e. including the host's Python/allocator/launch latency in front of the first kernel.
    abi_* = the same kernels through the C ABI with preallocated buffers (no allocator / autograd bookkeeping);
    scan_ms / grad_ms = each kernel pair alone.  Next to it: F.ctc_loss on the same GPU (ATen's sm_100 SIMT kernels) and
    on the host CPU (ATen LossCTC.cpp, what the reference runs at trainer.py:116-117 on a CPU box)."""
    import multimodal_av_model_b200 as pkg
    from multimodal_av_model_b200 import _lib
    L = _lib.lib()
    flush = l2_flusher(device)
    st = torch.cuda.current_stream(device).cuda_stream
    res = {}
    for T in Ts:
        lp, tg, il, tl, Lm = ctc_case(T, device)
        B, V = lp.shape[1], lp.shape[2]
        wsb = L.avctc_ctc_workspace_bytes(T, B, Lm)
        ws = torch.empty(wsb, dtype=torch.uint8, device=device)
        nll = torch.empty(B, device=device); go = torch.ones(1, device=device); grad = torch.empty_like(lp)
        loss = torch.empty(1, device=device)

        def fwd():
            _lib.check(L.avctc_ctc_forward(lp.data_ptr(), 0, lp.stride(0), lp.stride(1), T, B, V, tg.data_ptr(), tg.stride(0),
                                           None, il.data_ptr(), tl.data_ptr(), Lm, 0, 1, nll.data_ptr(), ws.data_ptr(), wsb, st), "fwd")
            _lib.check(L.avctc_ctc_reduce(nll.data_ptr(), tl.data_ptr(), B, 1, 1, loss.data_ptr(), st), "reduce")

        def bwd():
            _lib.check(L.avctc_ctc_backward(lp.data_ptr(), 0, lp.stride(0), lp.stride(1), T, B, V, tg.data_ptr(), tg.stride(0),
                                            None, il.data_ptr(), tl.data_ptr(), Lm, 0, 1, 1, nll.data_ptr(), go.data_ptr(), 0,
                                            grad.data_ptr(), ws.data_ptr(), wsb, st), "bwd")
        x = lp.clone().requires_grad_()

        def product():
            x.grad = None
            pkg.ctc_loss(x, tg, il, tl, blank=0, reduction="mean", zero_infinity=True).backward()
        t_prod_eager, _ = event_time(product, iters, 3, flush, device)
        t_prod, _ = event_time_queued(product, iters, 3, flush, device)
        t_all, t_min = event_time(lambda: (fwd(), bwd()), iters, 3, flush, device)
        t_f, _ = event_time(fwd, iters, 2, flush, device)
        t_b, _ = event_time(bwd, iters, 2, flush, device)
        alg = 2 * T * B * V * 4
        r = dict(product_ms=t_prod, product_eager_ms=t_prod_eager, gbs=alg / t_prod / 1e6, utt_per_s=B / t_prod * 1e3, abi_fwd_bwd_ms=t_all,
                 abi_gbs=alg / t_all / 1e6, scan_ms=t_f, grad_ms=t_b, grad_kernel_gbs=alg / t_b / 1e6, algorithmic_bytes=alg)
        if comparators:
            def torch_ref():
                x.grad = None
                torch.nn.functional.ctc_loss(x, tg, il, tl, blank=0, reduction="mean", zero_infinity=True).backward()
            t_torch, _ = event_time(torch_ref, max(3, iters // 2), 2, flush, device)
            r.update(torch_cuda_ms=t_torch, speedup_vs_torch_cuda=t_torch / t_prod)
            xc, tgc, ilc, tlc = lp.cpu().requires_grad_(), tg.cpu(), il.cpu(), tl.cpu()
            threads = os.cpu_count() or 1
            torch.set_num_threads(threads)

            def cpu_ref():
                xc.grad = None
                torch.nn.functional.ctc_loss(xc, tgc, ilc, tlc, blank=0, reduction="mean", zero_infinity=True).backward()
            t_cpu = cpu_time(cpu_ref, reps=3 if T <= 250 else 2)
            r["cpu"] = {"ms": t_cpu, "gbs": alg / t_cpu / 1e6, "utt_per_s": B / t_cpu * 1e3, "cores": threads, "kind": "port",
                        "sample": f"F.ctc_loss fwd+bwd on torch CPU (ATen LossCTC.cpp), the whole B={B} T={T} batch, fp32"}
        res[f"T{T}"] = r
    return res


def bench_beam(device, rank, world, iters=5, N=4096, T=150, beam=10, comparators=True):
    """BASELINE config 5: N utterances sharded contiguously over ranks, no collective.
    ms = the two decode kernels through the C ABI (log-probs resident in HBM, ids left on the device);
    e2e = beam_search_batch() from pinned host log-probs to Python token lists."""
    import multimodal_av_model_b200 as pkg
    from multimodal_av_model_b200 import _lib, ddp
    lo, hi = ddp.shard_range(N, rank, world)
    g = torch.Generator().manual_seed(7 + rank)
    n = hi - lo
    lp_host = (3 * torch.randn(n, T, VOCAB, generator=g)).log_softmax(-1).pin_memory()
    lp = lp_host.to(device)
    flush = l2_flusher(device)
    L = _lib.lib()
    st = torch.cuda.current_stream(device).cuda_stream
    wsb = int(L.avctc_beam_workspace_bytes(n, T, VOCAB, beam))
    ws = torch.empty(wsb, dtype=torch.uint8, device=device)
    out = torch.empty((n, T), dtype=torch.int32, device=device)
    ol = torch.empty(n, dtype=torch.int32, device=device)

    def kernels():
        _lib.check(L.avctc_beam_search(lp.data_ptr(), lp.stride(0), lp.stride(1), n, T, VOCAB, None, beam, BLANK,
                                       out.data_ptr(), ol.data_ptr(), None, None, ws.data_ptr(), wsb, st), "beam")
    t_k, _ = event_time(kernels, iters, 2, flush, device)
    ROUTES = {0: "unsupported", 1: "single kernel (one warp per utterance)", 2: "two-phase (top-k pass, then recurrence)",
              3: "fused top-k + recurrence kernel"}

    def route(m):           # asked from the library (avctc_beam_route): the rule lives in csrc/beam_search.cu
        return ROUTES[int(L.avctc_beam_route(m, T, VOCAB, beam))]
    sweep = {}
    if world == 1:          # what one rank decodes when the same 4096 utterances are sharded over 2 / 4 / 8 GPUs
        for m in (N // 2, N // 4, N // 8):
            def kernels_m(m=m):
                _lib.check(L.avctc_beam_search(lp.data_ptr(), lp.stride(0), lp.stride(1), m, T, VOCAB, None, beam, BLANK,
                                               out.data_ptr(), ol.data_ptr(), None, None, ws.data_ptr(), wsb, st), "beam")
            t_m, _ = event_time(kernels_m, iters, 2, flush, device)
            sweep[str(m)] = dict(ms=t_m, utt_per_s=m / t_m * 1e3, hbm_frac=m * T * VOCAB * 4 / t_m / 1e6 / measured_peaks()["hbm"],
                                 route=route(m))
    for _ in range(1):
        pkg.beam_search_batch(lp_host, beam_width=beam, blank=BLANK)       # host tensor: chunked copy || decode
    torch.cuda.synchronize(device)
    t0 = time.perf_counter()
    for _ in range(2):
        pkg.beam_search_batch(lp_host, beam_width=beam, blank=BLANK)
    t_e2e = (time.perf_counter() - t0) / 2 * 1e3
    out_d = dict(utterances=N, shard=n, beam=beam, ms=t_k, utt_per_s_shard=n / t_k * 1e3, e2e_ms=t_e2e,
                 e2e_utt_per_s_shard=n / t_e2e * 1e3, gbs=n * T * VOCAB * 4 / t_k / 1e6,
                 hbm_frac=n * T * VOCAB * 4 / t_k / 1e6 / measured_peaks()["hbm"],
                 algorithmic_bytes=n * T * VOCAB * 4, route=route(n), shard_sweep=sweep,
                 note="ms = decode kernels only (log-probs resident in HBM, ids left on the device) = what evaluate() pays, its "
                      "log-probs are device tensors; e2e = beam_search_batch() on pinned host log-probs: chunked H2D overlapped "
                      "with the decode kernels + D2H of ids + Python list construction (PCIe-bound)")
    if comparators and world == 1:
        # (1) the same search written with stock torch CUDA ops, batched over utterances: one torch.topk over all rows, then
        # T steps of [N, beam*beam] candidate scores -> torch.topk -> gather (float64 scores like the reference's Python floats)
        def torch_cuda_beam():
            vals, ids = torch.topk(lp, beam, dim=-1)                       # [n,T,beam]
            score = torch.zeros(n, 1, dtype=torch.float64, device=device)
            back = []
            for t in range(T):
                cand = (score[:, :, None] + vals[:, t, None, :].double()).reshape(n, -1)
                score, pick = torch.topk(cand, min(beam, cand.shape[1]), dim=-1)
                back.append(pick)
            return score, back, ids
        t_tc, _ = event_time(torch_cuda_beam, 2, 1, flush, device)
        out_d.update(torch_cuda_ms=t_tc, speedup_vs_torch_cuda=t_tc / t_k,
                     torch_cuda_note="batched stock-torch formulation (topk over all rows + T recurrence steps of topk/gather), "
                                     "no path reconstruction; the reference's own per-utterance Python loop is the cpu leg")
        # (2) the reference's simple_beam_search (beam_search.py:2-42) in a process pool over all host cores
        from oracle import torch_port as tp
        threads = os.cpu_count() or 1
        sample = min(n, max(64, 4 * threads))
        dt, _ = tp.beam_search_pool(lp_host[:sample], beam, BLANK, threads)
        out_d["cpu"] = {"utt_per_s": sample / dt, "ms_per_utt_per_core": dt * 1e3 * threads / sample, "cores": threads,
                        "kind": "port", "sample": f"simple_beam_search (Python loop + torch.topk per frame) on {sample} of the "
                                                  f"{N} utterances, {threads} worker processes x 1 thread"}
    return out_d


def bench_fusion(device, peaks, iters=10, comparators=True):
    """BASELINE config 3: projections + cross attention fwd/bwd, bf16, B=32, T_v=150, T_a=249."""
    import multimodal_av_model_b200 as pkg
    torch.manual_seed(0)
    fus = pkg.CrossAttentionFusion(512, 1024, 512).to(device)
    B, Tv, Ta = 32, 150, 249
    vis = torch.randn(B, Tv, 512, device=device, dtype=torch.bfloat16)
    aud = torch.randn(B, Ta, 1024, device=device, dtype=torch.bfloat16, requires_grad=True)
    mask = torch.zeros(B, Ta, dtype=torch.long, device=device)
    mask[:, :150] = 1; mask[:, 150:200] = 2
    for b in range(B):
        mask[b, Ta - (b % 7):] = 3
    flush = l2_flusher(device)
    r = torch.randn(B, Tv, 512, device=device, dtype=torch.bfloat16)      # bf16 in, bf16 out: what the BiLSTM hands back

    def fwd():
        with torch.no_grad():
            fus.fused_projection(vis, aud, mask)

    def fwd_bwd():
        fus.zero_grad(set_to_none=True); aud.grad = None
        f, _, _ = fus.fused_projection(vis, aud, mask)
        f.backward(r)
    t_f, _ = event_time(fwd, iters, 3, flush, device)
    t_fb, _ = event_time(fwd_bwd, iters, 3, flush, device)
    t_fq, _ = event_time_queued(fwd, iters, 2, flush, device)
    t_fbq, _ = event_time_queued(fwd_bwd, iters, 2, flush, device, hold_cycles=1400000)
    M = B * Tv
    flop_f = 2 * M * (512 * 512 * 4 + 1024 * 512 * 2) + 4 * B * Tv * Tv * 512
    out = dict(fwd_ms=t_f, fwd_bwd_ms=t_fb, fwd_tflops=flop_f / t_f / 1e9, fwd_bwd_tflops=3 * flop_f / t_fb / 1e9,
               tensor_frac_fwd=flop_f / t_f / 1e9 / peaks["tf_burst"], tensor_frac_fwd_bwd=3 * flop_f / t_fb / 1e9 / peaks["tf_burst"],
               queued_fwd_ms=t_fq, queued_fwd_bwd_ms=t_fbq, queued_tensor_frac_fwd=flop_f / t_fq / 1e9 / peaks["tf_burst"],
               queued_tensor_frac_fwd_bwd=3 * flop_f / t_fbq / 1e9 / peaks["tf_burst"],
               peak_tflops=peaks["tf_burst"], peak_src=peaks["src"] + " (burst cuBLAS bf16 peak: the path is timed alone)",
               note="fwd_ms / fwd_bwd_ms: eager calls through the Python op from an idle GPU (host prologue + one C-ABI call per "
                    "direction); queued_*: the same calls with the launch queue pre-filled behind a spin kernel = device time of "
                    "the kernel chain; graph_*: the same kernels replayed from a CUDA graph.  21.6 GFLOP fwd is ~13 us of tensor "
                    "work: the path is launch/latency bound at this size")
    # the same launches replayed from a CUDA graph: no host time, ~1 us between kernels (what a captured training step sees)
    try:
        side = torch.cuda.Stream(device=device)
        side.wait_stream(torch.cuda.current_stream(device))
        with torch.cuda.stream(side):
            for _ in range(3):
                fwd()
        torch.cuda.current_stream(device).wait_stream(side)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            fwd()
        t_g, _ = event_time(g.replay, iters, 3, flush, device)
        out.update(graph_fwd_ms=t_g, graph_tensor_frac_fwd=flop_f / t_g / 1e9 / peaks["tf_burst"])
        side.wait_stream(torch.cuda.current_stream(device))
        with torch.cuda.stream(side):
            for _ in range(3):
                fwd_bwd()
        torch.cuda.current_stream(device).wait_stream(side)
        g2 = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g2):
            fwd_bwd()
        t_g2, _ = event_time(g2.replay, iters, 3, flush, device)
        out.update(graph_fwd_bwd_ms=t_g2, graph_tensor_frac_fwd_bwd=3 * flop_f / t_g2 / 1e9 / peaks["tf_burst"])
    except Exception as e:          # capture is a measurement aid, never a requirement
        out.update(graph_fwd_ms=None, graph_error=str(e)[:120])
    if comparators:
        out.update(fusion_comparators(fus, vis, aud, mask, r, flush, device, iters, flop_f, peaks))
    return out


def fusion_comparators(fus, vis, aud, mask, r, flush, device, iters, flop_f, peaks):
    """Config 3 on (1) the stock torch CUDA kernels (nn.Linear / nn.MultiheadAttention = cuBLAS + ATen softmax, bf16
    autocast; the reference's formulation, fusion_module.py:40-63) and (2) the host CPU in fp32."""
    from oracle import torch_port as tp
    ref = tp.FusionPort(512, 1024, 512)
    ref.load_state_dict(fus.state_dict())
    ref.to(device)
    a2 = aud.detach().clone().requires_grad_()

    def t_fwd():
        with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
            ref.projection(vis, a2, mask)

    def t_fwd_bwd():
        ref.zero_grad(set_to_none=True); a2.grad = None
        with torch.autocast("cuda", dtype=torch.bfloat16):
            f, _ = ref.projection(vis, a2, mask)
        f.backward(r.to(f.dtype))
    tf, _ = event_time(t_fwd, iters, 3, flush, device)
    tfb, _ = event_time(t_fwd_bwd, iters, 3, flush, device)
    out = dict(torch_cuda_fwd_ms=tf, torch_cuda_fwd_bwd_ms=tfb, torch_cuda_tensor_frac_fwd_bwd=3 * flop_f / tfb / 1e9 / peaks["tf_burst"])
    ref.to("cpu")
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    vc, ac, mc, rc = vis.float().cpu(), aud.detach().float().cpu().requires_grad_(), mask.cpu(), r.float().cpu()

    def cpu():
        ref.zero_grad(set_to_none=True); ac.grad = None
        f, _ = ref.projection(vc, ac, mc)
        f.backward(rc)
    t_cpu = cpu_time(cpu, reps=2)
    out["cpu"] = {"fwd_bwd_ms": t_cpu, "tflops": 3 * flop_f / t_cpu / 1e9, "cores": threads, "kind": "port",
                  "sample": "FusionPort.projection fwd+bwd (nn.Linear + nn.MultiheadAttention on torch CPU ops, fp32), whole B=32 batch"}
    return out


def bench_lstm(device, iters=10):
    """temporal_model (2-layer BiLSTM 512->1024, fusion_module.py:21-27,64) fwd+bwd: the persistent sm_100a kernels against
    cuDNN (torch.nn.LSTM, fp32 weights under bf16 autocast) on the same GPU, at the hot-path shape (2B=16 sequences, T=150)
    and at config 3's batch (32)."""
    import multimodal_av_model_b200 as pkg
    from multimodal_av_model_b200.fusion_module import _BiLSTMFn
    flush = l2_flusher(device)
    torch.manual_seed(0)
    ref = torch.nn.LSTM(512, 512, num_layers=2, batch_first=True, bidirectional=True).to(device)
    res = {}
    for B in (16, 32):
        x = torch.randn(B, T_V, 512, device=device, dtype=torch.bfloat16, requires_grad=True)
        r = torch.randn(B, T_V, 1024, device=device, dtype=torch.bfloat16)

        def ours():
            ref.zero_grad(set_to_none=True); x.grad = None
            _BiLSTMFn.apply(x, *ref._flat_weights).backward(r)

        def ours_fwd():
            with torch.no_grad():
                _BiLSTMFn.apply(x, *ref._flat_weights)

        def cudnn():
            ref.zero_grad(set_to_none=True); x.grad = None
            with torch.autocast("cuda", dtype=torch.bfloat16):
                y, _ = ref(x)
            y.backward(r.to(y.dtype))
        t, _ = event_time(ours, iters, 3, flush, device)
        tf, _ = event_time(ours_fwd, iters, 3, flush, device)
        tc, _ = event_time(cudnn, max(3, iters // 2), 2, flush, device)
        res[f"B{B}"] = dict(fwd_ms=tf, fwd_bwd_ms=t, cudnn_fwd_bwd_ms=tc, speedup_vs_cudnn=tc / t,
                            us_per_step_fwd=tf * 1e3 / (2 * T_V))
    return res


def bench_infonce(device, peaks, iters=10):
    """SURVEY.md §8(d) 'InfoNCE (kernel 3)': contrastive_loss_with_mask fwd+bwd at config-4 sizes (8 x 249 rows of 1024
    features, Linear 1024->128 projection, sample-rate masks down-sampled to frame rate), bf16 features as under
    autocast.  HBM-bound on reading the feature rows once: algorithmic bytes = rows*1024*e + the projection weight.
    Beside it, the same loss written with stock torch CUDA ops (the reference's formulation, contrastive.py:13-44)."""
    import torch.nn.functional as F
    from multimodal_av_model_b200 import contrastive_loss_with_mask
    from multimodal_av_model_b200.synthetic import make_features
    f = make_features(pairs=PAIRS_PER_GPU, t_v=T_V, t_enc=249, seed=1234, dtype=torch.bfloat16)
    x = f["middle"][0].to(device).requires_grad_()
    mask = F.interpolate(f["masks"][0].to(device).unsqueeze(1).float(), size=249, mode="nearest").squeeze(1).long().reshape(-1)
    torch.manual_seed(0)
    proj = torch.nn.Linear(1024, 128).to(device)
    flush = l2_flusher(device)

    def ours():
        x.grad = None; proj.zero_grad(set_to_none=True)
        with torch.autocast("cuda", dtype=torch.bfloat16):
            contrastive_loss_with_mask(x, mask, projection_layer=proj).backward()

    def stock():
        x.grad = None; proj.zero_grad(set_to_none=True)
        with torch.autocast("cuda", dtype=torch.bfloat16):
            feat = x.reshape(-1, x.shape[-1]); keep = mask != 3
            z = F.normalize(proj(feat[keep]), dim=-1); m = mask[keep]
            loss = torch.zeros((), device=device, requires_grad=True)
            weak, strong, neg = z[m == 1], z[m == 2], z[m == 0]
            if len(weak) and len(strong):
                loss = loss + 1.0 * (-F.log_softmax(weak @ strong.T / 0.07, dim=-1)).mean()
            if len(weak) and len(neg):
                loss = loss + 0.3 * (-F.log_softmax(weak @ neg.T / 0.07, dim=-1)).mean()
            loss.backward()
    t, _ = event_time(ours, iters, 3, flush, device)
    t_q, _ = event_time_queued(ours, iters, 2, flush, device, hold_cycles=1400000)
    t_stock, _ = event_time(stock, iters, 3, flush, device)
    rows = x.shape[0] * x.shape[1]
    alg = rows * 1024 * 2 + 128 * 1024 * 4
    return dict(rows=rows, fwd_bwd_ms=t, queued_fwd_bwd_ms=t_q, torch_cuda_ms=t_stock, speedup_vs_torch_cuda=t_stock / t,
                algorithmic_bytes=alg, gbs=alg / t / 1e6, hbm_frac=alg / t / 1e6 / peaks["hbm"],
                note="fwd_bwd_ms: eager Python op from an idle GPU (projection GEMM + fused normalise/pair kernels, fwd+bwd); "
                     "queued_fwd_bwd_ms: the same call with the launch queue pre-filled = device time of its kernels; 4.6 MB of "
                     "input is ~1 us of HBM time, so the op is launch-latency bound at the reference's batch size; in the train "
                     "step both speakers' losses run on a side stream under the BiLSTM kernels")


# ------------------------------------------------------------------------------------------------ CPU arm
def cpu_train_sample(pairs, steps, warmup, threads, budget_s=300.0):
    """The reference's train step (trainer.py:62-125) on the host CPU: its modules restated on stock torch / HF ops
    (oracle/encoder_port.py: VisualEncoder + unmodified Wav2Vec2Model.forward; oracle/torch_port.py: fusion, CTC head,
    nn.CTCLoss, InfoNCE), fp32 (torch.cuda.amp autocast/GradScaler are no-ops on CPU), Adam with the reference's four
    parameter groups.  Nothing of the product package computes here; synthetic.make_batch only generates the inputs."""
    from oracle import encoder_port as ep
    from oracle import torch_port as tp
    from multimodal_av_model_b200.synthetic import make_batch
    torch.set_num_threads(threads)
    torch.manual_seed(0)
    vis = ep.VisualPort()
    for p in vis.parameters():                       # main.py:100-103
        p.requires_grad = False
    aud = ep.AudioPort()                             # main.py:105-106: only encoder.layers.6-9 train
    fus = tp.FusionPort(512, 1024, 512)
    dec = tp.DecoderPort(1024, VOCAB, BLANK)
    proj = torch.nn.Linear(1024, 128)
    opt = torch.optim.Adam([{"params": [p for p in aud.parameters() if p.requires_grad], "lr": 2e-5},
                            {"params": fus.parameters(), "lr": 1e-4}, {"params": dec.parameters(), "lr": 1e-4}])
    for m in (vis, aud, fus, dec):
        m.train()
    batch = make_batch(pairs=pairs, seconds=SECONDS, t_v=T_V, vocab=VOCAB, seed=1234)

    def step():
        opt.zero_grad()
        feats = []
        for s in ("1", "2"):
            lip = batch["lip" + s].permute(0, 2, 1, 3, 4).contiguous()
            v = vis(lip)
            a, mid = aud(batch["audio"], attention_mask=(batch["mask" + s] != 3))
            feats.append(dict(visual=v, audio=a, middle=mid, mask=batch["mask" + s], text=batch["text" + s],
                              text_len=batch["text" + s + "_lengths"]))
        loss = tp.hot_path_losses(fus, dec, proj, feats, blank=BLANK)
        loss.backward()
        opt.step()
        return float(loss.detach())
    # K timed steps after W warm-up steps as asked, unless that cannot end "within a few minutes" on this host: the first
    # step is timed and, if (W-1+K) more would exceed `budget_s`, warm-up stops there and K shrinks to what fits (>= 1).
    # The per-step workload (all `pairs`) is never reduced — the config stays the one the GPU arm runs.
    done_warm = 0
    if warmup > 0:
        t0 = time.perf_counter(); step(); est = time.perf_counter() - t0
        done_warm = 1
        if (warmup - 1 + steps) * est > budget_s:
            steps = max(1, min(steps, int(budget_s / est)))
        else:
            for _ in range(warmup - 1):
                step()
            done_warm = warmup
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = time.perf_counter() - t0
    return 2 * pairs * steps / dt, dt / steps, steps, done_warm


def train_config(world):
    """The workload BOTH arms run (BASELINE config 4) — the same dict on the `ours` and the `reference` line."""
    return {"workload": "config4: full AV-CTC + InfoNCE train step (encoders + fusion + BiLSTM + CTC head + CTC + InfoNCE + Adam)",
            "pairs_per_gpu": PAIRS_PER_GPU, "utterances_per_step": 2 * PAIRS_PER_GPU * world, "audio_s": SECONDS,
            "lip_frames": T_V, "t_enc": 249, "vocab": VOCAB, "blank": BLANK,
            "encoders": "random-init ResNet-18 front-end + wav2vec2-large (XLSR layout)",
            "parallelism": f"dp{world}, utterance-sharded",
            "l2": "per-step working set (1.3 GB of parameters + activations) exceeds the 126 MB L2; sub-benchmarks flush L2 "
                  "with a 256 MB write between iterations"}


def run_reference(args, rank):
    """--impl reference: the reference's CPU implementation of the SAME config (8 pairs per step), K timed steps after W
    warm-up steps exactly as asked, all host threads.  Under torchrun only rank 0 works."""
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    world = max(1, args.gpus)
    val, sec, steps, warm = cpu_train_sample(PAIRS_PER_GPU, args.steps, args.warmup, threads)
    line = {"impl": "reference", "metric": "train_utt_per_s", "value": val, "unit": "utt/s", "n_gpus": args.gpus,
            "steps": steps, "warmup": warm, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": train_config(world),
            "implementation": "reference train step on torch CPU ops, fp32: oracle/encoder_port.py (unmodified "
                              "Wav2Vec2Model.forward + ResNet-18 front end) + oracle/torch_port.py; one process, all host threads",
            "cpu_baseline": {"value": val, "unit": "utt/s", "cores": threads, "kind": "port",
                             "sample": f"{steps} step(s) after {warm} warm-up of {PAIRS_PER_GPU} pairs "
                                       f"(= {2 * PAIRS_PER_GPU} utterances) each: the full config-4 step, {sec:.1f} s/step"},
            "e2e": {"value": val, "unit": "utt/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


# ------------------------------------------------------------------------------------------------ main
_REAL_STDOUT = None


def _guard_stdout():
    """The driver reads ONE JSON line from stdout.  Libraries print there too (e.g. NCCL's version banner), so fd 1 is
    pointed at stderr for the whole run and the JSON line is written to the saved descriptor at the end."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    sys.stdout.flush()
    os.write(_REAL_STDOUT if _REAL_STDOUT is not None else 1, (json.dumps(line) + "\n").encode())


def source_hash(files=("ctc_loss.cu", "common.cuh")):
    """sha256 (first 16 hex) of the kernel sources a profile belongs to — profiles/*.json carry it, so a DRAM-traffic
    figure is only quoted while the kernels it was captured from are the ones being timed."""
    h = hashlib.sha256()
    for f in files:
        with open(os.path.join(ROOT, "multimodal-av-model_b200", "csrc", f), "rb") as fh:
            h.update(fh.read())
    return h.hexdigest()[:16]


def ctc_traffic():
    """(bytes per fwd+bwd launch pair, provenance) from profiles/ctc_traffic.json (written by
    `tools/ncu_summary.py traffic` from one `ncu --set full` capture of tools/run_ctc_once.py), or (None, why)."""
    path = os.path.join(ROOT, "profiles", "ctc_traffic.json")
    if not os.path.exists(path):
        return None, "no profiles/ctc_traffic.json"
    d = json.load(open(path))
    if d.get("source_hash") != source_hash():
        return None, f"profiles/ctc_traffic.json was captured from other kernel sources ({d.get('source_hash')}), not quoted"
    return d["traffic_bytes"], {"file": "profiles/ctc_traffic.json", "kernels": d.get("kernels"), "git_head": d.get("git_head")}


def main():
    _guard_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="train", choices=["train", "ctc", "beam", "fusion", "infonce", "lstm", "hot"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-comparators", action="store_true", help="skip the stock-torch CUDA / host CPU legs of the sub-benchmarks")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the loss terms and log-probs of the last timed train step "
                                                           "to DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload != "train"):
        ap.error("--dump-outputs needs --impl ours --workload train")
    rank = int(os.environ.get("RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    args.warmup = max(args.warmup, 3)
    from multimodal_av_model_b200 import ddp
    rank, local, world = ddp.init_distributed()
    device = torch.device("cuda", local)
    torch.cuda.set_device(device)
    peaks = measured_peaks()
    comparators = (world == 1) and not args.no_comparators
    line = {"metric": "train_utt_per_s", "unit": "utt/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": train_config(world),
            "implementation": "PyTorch encoders + sm_100a fusion/BiLSTM/CTC head/CTC/InfoNCE kernels, bf16 autocast"}
    wl = args.workload
    if wl in ("train", "hot"):
        out, tr = bench_train(args, rank, local, world, device, hot_only=(wl == "hot"))
        line.update(out)
        del tr
        torch.cuda.empty_cache()
    ctc = bench_ctc(device, comparators=comparators) if wl in ("train", "ctc") else None
    beam = bench_beam(device, rank, world, comparators=comparators) if wl in ("train", "beam") else None
    fusion = bench_fusion(device, peaks, comparators=comparators) if wl in ("train", "fusion") else None
    if wl in ("train", "lstm"):
        line["lstm"] = bench_lstm(device)
    if wl in ("train", "infonce"):
        line["infonce"] = bench_infonce(device, peaks)
    if beam is not None:
        import torch.distributed as dist
        t = torch.tensor([beam["ms"], beam["e2e_ms"]], device=device)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        beam["utt_per_s"] = beam["utterances"] / float(t[0]) * 1e3
        beam["e2e_utt_per_s"] = beam["utterances"] / float(t[1]) * 1e3
        line["beam"] = beam
    if ctc is not None:
        line["ctc"] = ctc
        top = ctc["T1000"]
        traffic, prov = ctc_traffic()
        line["roofline"] = {"bound": "hbm", "kernel": "ctc_scan_ws_kernel + ctc_grad_lin_kernel (CTC fwd+bwd, config 2: B=64 T=1000 V=801 fp32)",
                            "achieved": top["gbs"], "peak": peaks["hbm"], "unit": "GB/s", "frac": top["gbs"] / peaks["hbm"],
                            "peak_src": peaks["src"] + " (burst copy bandwidth, MEASURED_PEAKS.json: the kernel pair is timed alone)",
                            "traffic": traffic, "traffic_src": prov,
                            "algorithmic_bytes": top["algorithmic_bytes"],
                            "frac_T250": ctc["T250"]["gbs"] / peaks["hbm"] if "T250" in ctc else None,
                            "abi_frac": top["abi_gbs"] / peaks["hbm"], "grad_kernel_frac": top["grad_kernel_gbs"] / peaks["hbm"],
                            "note": "achieved = 2*T*B*V*4 bytes / device time of pkg.ctc_loss(x, ...).backward() (one pair of CUDA events "
                                    "around the autograd call, launch queue pre-filled behind a spin kernel so that host enqueue "
                                    "latency is not counted; ctc.T1000.product_eager_ms is the same call from an idle GPU: scan + reduce + gradient pass enqueued back to back at forward time, "
                                    "backward applies grad_out); the scan is a 1000-step dependent recurrence over 128 CTAs "
                                    "(latency-bound), the gradient pass streams and starts on each utterance as soon as its alpha/beta "
                                    "rows are complete, so the total is below scan_ms + grad_ms (each timed alone); abi_frac = the same "
                                    "kernels through the C ABI with preallocated buffers; traffic = dram__bytes_read+write of both "
                                    "kernels from the ncu --set full capture named in traffic_src (null when the kernel sources changed)"}
    if fusion is not None:
        line["fusion"] = fusion
    if wl not in ("train",):
        line["metric"] = {"ctc": "ctc_fwd_bwd_gbs", "beam": "beam_decode_utt_per_s", "fusion": "fusion_tensor_frac",
                          "infonce": "infonce_fwd_bwd_gbs", "lstm": "bilstm_fwd_bwd_ms", "hot": "hot_path_utt_per_s"}[wl]
        line["unit"] = {"ctc": "GB/s", "beam": "utt/s", "fusion": "fraction of bf16 tensor peak", "infonce": "GB/s", "lstm": "ms",
                        "hot": "utt/s"}[wl]
        line["config"] = {"workload": {"ctc": "config2: CTC fwd+bwd micro-benchmark B=64 T=250/1000 V=801 L in [10,80] fp32",
                                       "beam": "config5: beam-10 decode of 4096 x [150,800] log-prob utterances",
                                       "fusion": "config3: fusion projections + cross attention fwd/bwd bf16 B=32 T_v=150 T_a=249",
                                       "infonce": "config4 sizes: InfoNCE fwd+bwd on 8 x 249 rows of 1024 bf16 features",
                                       "lstm": "2-layer BiLSTM 512->1024 fwd+bwd, T=150, B=16/32, bf16",
                                       "hot": "config4 from encoder features on (fusion+BiLSTM+head+CTC+InfoNCE fwd+bwd), 8 pairs"}[wl],
                          "l2": "256 MB write between timed iterations flushes L2"}
        line["dtype"] = {"ctc": "f32", "beam": "f32 values, f64 scores", "fusion": "bf16", "infonce": "bf16 in, f32 math",
                         "lstm": "bf16", "hot": "bf16"}[wl]
        line["value"] = {"ctc": lambda: ctc["T1000"]["gbs"], "beam": lambda: beam["utt_per_s"], "fusion": lambda: fusion["tensor_frac_fwd_bwd"],
                         "infonce": lambda: line["infonce"]["gbs"], "lstm": lambda: line["lstm"]["B16"]["fwd_bwd_ms"],
                         "hot": lambda: line["hot_path"]["value"]}[wl]()
        if wl == "lstm":
            line["higher_is_better"] = False
    if rank == 0 and world == 1 and wl == "train" and not args.no_cpu_baseline:
        threads = os.cpu_count() or 1
        v, sec, _, _ = cpu_train_sample(PAIRS_PER_GPU, 1, 1, threads)
        line["cpu_baseline"] = {"value": v, "unit": "utt/s", "cores": threads, "kind": "port",
                                "sample": f"1 step (after 1 warm-up) of the same {PAIRS_PER_GPU} pairs (= {2 * PAIRS_PER_GPU} utterances): "
                                          "the full config-4 step on torch CPU ops, fp32 (oracle/encoder_port.py + "
                                          f"oracle/torch_port.py), {sec:.1f} s/step"}
    if rank == 0:
        emit(line)
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
