"""Where the audio encoder's and the backward's time goes in the config-4 train step, host against device (B200).

    python tools/profile_audio.py --out DIR [--steps N] [--calls N] [--module-only]

Writes DIR/audio_step_segments.txt, DIR/audio_layer_call.txt and DIR/audio_gemm.txt; every file starts with the card's
name, power limit and max SM clock (nvidia-smi):
  1. one train step (bench.py's models and batch) split into segments (visual encoder x2, audio encoder x2, hot path
     forward, backward, optimizer).  For each segment: the device time, as the sum of its kernels in a torch.profiler
     run of its own (a kernel belongs to the segment whose host window issued it), and the host enqueue time, from a
     host clock around the segment's calls with no synchronise inside, in a run without the profiler.  A segment whose
     host time is at or above its device time is host-bound.
  2. one gradient-carrying wav2vec2 layer-call at the config-4 shape ([8, 249, 1024] bf16, ragged boolean mask, train
     mode, bf16 autocast), forward plus backward, trainable and frozen, on the module path and on the native path:
     device time (sum of kernels, profiler run), host time (enqueue of forward + backward, no synchronise inside),
     wall time per call (CUDA events over --calls calls) and kernels per call.
  3. this library's tcgen05 GEMM against cuBLAS (torch.matmul) at the layer's shapes, M = 1992: forward, input
     gradient and weight gradient of the q|k|v, out, FFN1 and FFN2 projections (CUDA events, bf16 in, bf16 out for
     forward / input gradient, fp32 out for the weight gradient; single launch, no split-K).
--module-only takes the module path in 1 (the measurement before the native layers; the parent commit's profile).
"""
from __future__ import annotations

import argparse
import collections
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        return r.stdout.strip().splitlines()[0]
    except Exception as e:                       # the numbers below still stand; say why the card is not named
        return f"nvidia-smi unavailable ({e})"


def kernels_by_window(prof, windows):
    """Sum the device time of the kernels each host window [t0, t1) (profiler clock, us) issued."""
    dev = collections.defaultdict(float)
    count = collections.defaultdict(int)
    for e in prof.events():
        if e.device_type != torch.autograd.DeviceType.CPU or not e.kernels:
            continue
        t = e.time_range.start
        label = next((lab for lab, t0, t1 in windows if t0 <= t < t1), "unattributed")
        for k in e.kernels:
            dev[label] += k.duration
            count[label] += 1
    return dev, count


class Segments:
    """Wraps the step's entry points.  Host-clock mode records (label, t0, t1) per call; with annotate = True each call
    runs inside record_function("seg:<label>") so that a profiler run sees the windows on its own clock."""

    def __init__(self, tr):
        self.windows, self.annotate, self.saved = [], False, []
        self._wrap(tr.visual_encoder, "forward", "visual encoder")
        self._wrap(tr.audio_encoder, "forward", "audio encoder")
        self._wrap(tr, "hot_path_loss", "hot path forward")
        self._wrap(tr.optimizer, "step", "optimizer")
        self._wrap(torch.Tensor, "backward", "backward")

    def _wrap(self, obj, attr, label):
        inner = getattr(obj, attr)
        seg = self

        def f(*a, **k):
            if seg.annotate:
                with torch.profiler.record_function("seg:" + label):
                    return inner(*a, **k)
            t0 = time.perf_counter()
            out = inner(*a, **k)
            seg.windows.append((label, t0, time.perf_counter()))
            return out
        setattr(obj, attr, f)
        self.saved.append((obj, attr, inner))

    def restore(self):
        for obj, attr, inner in reversed(self.saved):
            setattr(obj, attr, inner)


SEGMENTS = ("visual encoder", "audio encoder", "hot path forward", "backward", "optimizer")


def step_segments(dev, steps, module_only):
    import bench
    from multimodal_av_model_b200 import encoders
    from multimodal_av_model_b200.synthetic import make_batch
    from torch.profiler import ProfilerActivity, profile
    if module_only:
        encoders._w2v_native_applies = lambda layer, hidden: False
    tr = bench.build_models(dev)
    host = make_batch(pairs=bench.PAIRS_PER_GPU, seconds=bench.SECONDS, t_v=bench.T_V, vocab=bench.VOCAB, seed=1234,
                      pin=True)
    batch = {k: v.to(dev) for k, v in host.items()}
    seg = Segments(tr)
    try:
        for _ in range(3):
            tr.train_step(batch)
        torch.cuda.synchronize()
        seg.windows.clear()                          # host enqueue, no profiler
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(steps):
            tr.train_step(batch)
        b.record()
        torch.cuda.synchronize()
        step_ms = a.elapsed_time(b) / steps
        host, calls = collections.defaultdict(float), collections.defaultdict(int)
        for lab, t0, t1 in seg.windows:
            host[lab] += (t1 - t0) * 1e3
            calls[lab] += 1
        seg.annotate = True                          # device time: a profiler run of its own
        with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
            for _ in range(steps):
                tr.train_step(batch)
            torch.cuda.synchronize()
    finally:
        seg.restore()
    windows = [(e.name[4:], e.time_range.start, e.time_range.end) for e in prof.events() if e.name.startswith("seg:")]
    devt, kcount = kernels_by_window(prof, windows)
    lines = [f"{'segment':<18} {'device ms':>10} {'host ms':>9} {'kernels':>8} {'calls':>6}  bound"]
    for lab in SEGMENTS:
        d, h = devt[lab] / 1e3 / steps, host[lab] / steps
        lines.append(f"{lab:<18} {d:10.3f} {h:9.3f} {kcount[lab] / steps:8.0f} {calls[lab] / steps:6.1f}  "
                     f"{'host' if h >= d else 'device'}")
    if devt.get("unattributed"):
        lines.append(f"{'outside segments':<18} {devt['unattributed'] / 1e3 / steps:10.3f}")
    lines.append(f"{'step (events)':<18} {step_ms:10.3f}   ({steps} steps after 3 warm-up, 8 pairs, resident batch, "
                 f"{'module path' if module_only else 'native wav2vec2 layers'})")
    return "\n".join(lines)


def layer_call(dev, calls):
    from transformers.models.wav2vec2.modeling_wav2vec2 import Wav2Vec2EncoderLayerStableLayerNorm
    from multimodal_av_model_b200 import encoders
    from multimodal_av_model_b200.encoders import xlsr_large_config
    from torch.profiler import ProfilerActivity, profile
    cfg = xlsr_large_config()
    cfg._attn_implementation = "sdpa"
    torch.manual_seed(0)
    layer = Wav2Vec2EncoderLayerStableLayerNorm(cfg).to(dev).train()
    encoders.install_frozen_cast_cache(layer)       # as the trainer does for the frozen encoders
    B, T = 8, 249
    lens = torch.tensor([249, 240, 231, 249, 200, 190, 248, 160])
    m = torch.arange(T)[None, :] < lens[:, None]
    mask4d = m.to(dev)[:, None, None, :].expand(B, 1, T, T)
    x0 = torch.randn(B, T, 1024, device=dev).to(torch.bfloat16)
    g = torch.randn(B, T, 1024, device=dev).to(torch.bfloat16)

    def run(native):
        x = x0.detach().requires_grad_()
        with torch.autocast("cuda", dtype=torch.bfloat16):
            y = encoders._w2v_native_layer(layer, x, mask4d) if native else \
                layer(x, attention_mask=mask4d, output_attentions=False)[0]
        y.backward(g)
        layer.zero_grad(set_to_none=True)

    lines = [f"{'variant':<10} {'path':<7} {'device ms':>10} {'host ms':>8} {'wall ms':>8} {'kernels':>8}"]
    for trainable in (True, False):
        layer.requires_grad_(trainable)
        for native in (False, True):
            for _ in range(3):
                run(native)
            torch.cuda.synchronize()
            h = 0.0
            for _ in range(calls):
                t0 = time.perf_counter()
                run(native)
                h += time.perf_counter() - t0
                torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(calls):
                run(native)
            b.record()
            torch.cuda.synchronize()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                run(native)
                torch.cuda.synchronize()
            kern = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA
                    and not e.name.startswith(("Memcpy", "Memset"))]
            dev_ms = sum(e.time_range.elapsed_us() for e in kern) / 1e3
            lines.append(f"{'trainable' if trainable else 'frozen':<10} {'native' if native else 'module':<7} "
                         f"{dev_ms:10.3f} {h / calls * 1e3:8.3f} {a.elapsed_time(b) / calls:8.3f} {len(kern):8d}")
    return "\n".join(lines)


def gemm_table(dev, iters=50):
    from multimodal_av_model_b200.gemm import gemm, operand
    M = 1992
    shapes = [("q|k|v", 3 * 1024, 1024), ("out", 1024, 1024), ("FFN1", 4096, 1024), ("FFN2", 1024, 4096)]

    def t(fn):
        for _ in range(3):
            fn()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(iters):
            fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / iters * 1e3

    lines = [f"{'proj':<6} {'pass':<6} {'N':>5} {'K':>5} {'avctc us':>9} {'cuBLAS us':>10} {'avctc TFLOP/s':>14}"]
    for name, N, K in shapes:
        x = torch.randn(M, K, device=dev).to(torch.bfloat16)
        w = torch.randn(N, K, device=dev).to(torch.bfloat16)
        dy = torch.randn(M, N, device=dev).to(torch.bfloat16)
        y = torch.empty(M, N, device=dev, dtype=torch.bfloat16)
        dx = torch.empty(M, K, device=dev, dtype=torch.bfloat16)
        gw = torch.empty(N, K, device=dev, dtype=torch.float32)
        runs = {"fwd": (lambda: gemm(operand(x), operand(w), M, N, K, y), lambda: torch.matmul(x, w.t())),
                "dgrad": (lambda: gemm(operand(dy), operand(w, "mn"), M, K, N, dx), lambda: torch.matmul(dy, w)),
                "wgrad": (lambda: gemm(operand(dy, "mn"), operand(x, "mn"), N, K, M, gw),
                          lambda: torch.matmul(dy.t(), x))}
        for p, (ours, ref) in runs.items():
            a, r = t(ours), t(ref)
            lines.append(f"{name:<6} {p:<6} {N:5d} {K:5d} {a:9.1f} {r:10.1f} {2 * M * N * K / a / 1e6:14.0f}")
    return "\n".join(lines)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--module-only", action="store_true")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("profile_audio: needs a CUDA device")
    os.makedirs(args.out, exist_ok=True)
    dev = torch.device("cuda", 0)
    head = f"card: {card()}  (name, power limit, max SM clock)\ntorch {torch.__version__}\n"
    outs = []
    if not args.module_only:
        outs.append(("audio_layer_call.txt", "one wav2vec2 layer-call [8,249,1024] bf16, ragged mask, train mode, "
                     f"forward + backward ({args.calls} calls after 3 warm-up):\n", lambda: layer_call(dev, args.calls)))
        outs.append(("audio_gemm.txt", "tcgen05 GEMM against cuBLAS, M = 1992 (CUDA events, 50 launches):\n",
                     lambda: gemm_table(dev)))
    outs.append(("audio_step_segments.txt", "config-4 train step, device (profiler) and host (enqueue) time per "
                 "segment:\n", lambda: step_segments(dev, args.steps, args.module_only)))
    for fname, title, fn in outs:
        text = head + title + fn() + "\n"
        print(text, flush=True)
        open(os.path.join(args.out, fname), "w").write(text)
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
