"""Where the visual encoder's time goes, and its share of the config-4 train step (B200).

    python tools/profile_visual.py --out DIR [--calls N] [--steps N]

Writes DIR/visual_timing.txt, DIR/visual_kernels.txt and DIR/step_segments.txt:
  1. card name, power limit and max SM clock (nvidia-smi), printed next to every number;
  2. one VisualEncoder call at the config-4 shape [8,1,150,96,96] fp32, train mode, frozen, bf16 autocast: the eager
     `_forward_impl` and the graphed `forward`, CUDA events over --calls calls after warm-up;
  3. the kernels of one eager call (torch.profiler, a run of its own) grouped as front-end taps / front-end conv /
     BN statistics / BN apply / PReLU / add / pooling / trunk convs;
  4. one train step (bench.py's models and batch) split into segments by CUDA events on the main stream: visual x2,
     audio encoder x2, hot path forward, backward, optimizer.  The step is GPU bound, so the host runs ahead and the
     event gaps are device time.
"""
from __future__ import annotations

import argparse
import collections
import os
import re
import subprocess
import sys

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


def event_ms(fn, calls, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(calls):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / calls


def make_visual(dev):
    import multimodal_av_model_b200 as pkg
    from multimodal_av_model_b200.encoders import install_frozen_cast_cache
    torch.manual_seed(0)
    vis = pkg.VisualEncoder(relu_type="prelu").to(dev).train()
    for p in vis.parameters():
        p.requires_grad = False
    install_frozen_cast_cache(vis)               # as MultimodalTrainer does
    return vis


GROUPS = ("front-end taps", "front-end conv", "BN statistics", "BN apply", "PReLU", "add", "pooling", "trunk convs",
          "other")


def classify(name, seen_bn):
    n = name.lower()
    if re.match(r"(void )?vis_", n):             # this library's kernels (csrc/visual_encoder.cu)
        if "frontend_conv" in n:
            return "front-end conv"
        if "stats" in n or "finalize" in n:
            return "BN statistics"
        if "pool" in n:
            return "pooling"
        return "BN apply"
    if "at::native" in n or "at::" in n:
        if "batch_norm" in n:
            return "BN statistics" if re.search(r"collect|welford|stat|reduce", n) and "transform" not in n else "BN apply"
        if "prelu" in n:
            return "PReLU"
        if "max_pool" in n or "avg_pool" in n or "adaptive" in n or "mean" in n or "reduce" in n:
            return "pooling"
        if "add" in n:
            return "add"
        return "front-end taps" if not seen_bn else "other"
    return "front-end conv" if not seen_bn else "trunk convs"


def kernel_table(vis, x):
    from torch.profiler import ProfilerActivity, profile
    with torch.autocast("cuda", dtype=torch.bfloat16):
        for _ in range(3):
            vis._forward_impl(x)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            vis._forward_impl(x)
            torch.cuda.synchronize()
    kern = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA
            and not e.name.startswith(("Memcpy", "Memset"))]
    kern.sort(key=lambda e: e.time_range.start)
    groups = collections.OrderedDict((g, [0.0, 0]) for g in GROUPS)
    per_name = collections.OrderedDict()
    seen_bn = False
    for e in kern:
        g = classify(e.name, seen_bn)
        seen_bn = seen_bn or g in ("BN statistics", "BN apply")
        us = e.time_range.elapsed_us()
        groups[g][0] += us
        groups[g][1] += 1
        k = (g, e.name[:110])
        per_name.setdefault(k, [0.0, 0])
        per_name[k][0] += us
        per_name[k][1] += 1
    total = sum(v[0] for v in groups.values())
    lines = [f"{'group':<16} {'ms':>8} {'share':>6} {'kernels':>8}"]
    for g, (us, n) in groups.items():
        if n:
            lines.append(f"{g:<16} {us / 1e3:8.3f} {us / total:6.1%} {n:8d}")
    lines.append(f"{'sum of kernels':<16} {total / 1e3:8.3f}        {sum(v[1] for v in groups.values()):8d}")
    lines.append("")
    lines.append(f"{'group':<16} {'ms':>8} {'n':>4}  kernel")
    for (g, name), (us, n) in sorted(per_name.items(), key=lambda kv: -kv[1][0]):
        lines.append(f"{g:<16} {us / 1e3:8.3f} {n:4d}  {name}")
    return "\n".join(lines)


def step_segments(dev, steps):
    import bench
    from multimodal_av_model_b200.synthetic import make_batch
    tr = bench.build_models(dev)
    host = make_batch(pairs=bench.PAIRS_PER_GPU, seconds=bench.SECONDS, t_v=bench.T_V, vocab=bench.VOCAB, seed=1234,
                      pin=True)
    batch = {k: v.to(dev) for k, v in host.items()}
    marks = []

    def mark(label):
        ev = torch.cuda.Event(enable_timing=True)
        ev.record()
        marks.append((label, ev))

    def wrap(obj, attr, label):
        inner = getattr(obj, attr)

        def f(*a, **k):
            mark("start")
            out = inner(*a, **k)
            mark(label)
            return out
        setattr(obj, attr, f)
        return inner

    v_fwd = wrap(tr.visual_encoder, "forward", "visual encoder")
    a_fwd = wrap(tr.audio_encoder, "forward", "audio encoder")
    h_fwd = wrap(tr, "hot_path_loss", "hot path forward")
    o_step = wrap(tr.optimizer, "step", "optimizer")
    backward = torch.Tensor.backward

    def bwd(self, *a, **k):
        mark("start")
        out = backward(self, *a, **k)
        mark("backward")
        return out
    torch.Tensor.backward = bwd
    try:
        for _ in range(3):
            tr.train_step(batch)
        torch.cuda.synchronize()
        marks.clear()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(steps):
            tr.train_step(batch)
        b.record()
        torch.cuda.synchronize()
    finally:
        torch.Tensor.backward = backward
        tr.visual_encoder.forward, tr.audio_encoder.forward, tr.hot_path_loss, tr.optimizer.step = (
            v_fwd, a_fwd, h_fwd, o_step)
    step_ms = a.elapsed_time(b) / steps
    seg = collections.OrderedDict()
    prev = None
    for label, ev in marks:
        if label != "start" and prev is not None:
            seg.setdefault(label, [0.0, 0])
            seg[label][0] += prev.elapsed_time(ev)
            seg[label][1] += 1
        prev = ev
    lines = [f"{'segment':<18} {'ms/step':>8} {'calls/step':>10}"]
    covered = 0.0
    for label, (ms, n) in seg.items():
        lines.append(f"{label:<18} {ms / steps:8.3f} {n / steps:10.1f}")
        covered += ms / steps
    lines.append(f"{'rest (gaps)':<18} {step_ms - covered:8.3f}")
    lines.append(f"{'step':<18} {step_ms:8.3f}   ({steps} steps after 3 warm-up, 8 pairs, resident batch)")
    return "\n".join(lines)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--steps", type=int, default=10)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("profile_visual: needs a CUDA device")
    os.makedirs(args.out, exist_ok=True)
    dev = torch.device("cuda", 0)
    head = f"card: {card()}  (name, power limit, max SM clock)\ntorch {torch.__version__}\n"

    vis = make_visual(dev)
    x = torch.rand(8, 1, 150, 96, 96, device=dev)

    def eager():
        with torch.autocast("cuda", dtype=torch.bfloat16):
            return vis._forward_impl(x)

    def graphed():
        with torch.autocast("cuda", dtype=torch.bfloat16):
            return vis(x)
    t_eager = event_ms(eager, args.calls)
    t_graph = event_ms(graphed, args.calls)
    timing = (head + f"VisualEncoder [8,1,150,96,96] fp32 in, train mode, frozen, bf16 autocast, CUDA events over "
              f"{args.calls} calls after 3 warm-up:\n  eager _forward_impl {t_eager:8.3f} ms/call\n"
              f"  graphed forward     {t_graph:8.3f} ms/call\n")
    print(timing, flush=True)
    open(os.path.join(args.out, "visual_timing.txt"), "w").write(timing)

    table = head + "kernels of one eager VisualEncoder call (torch.profiler, separate run), [8,1,150,96,96]:\n" + \
        kernel_table(vis, x) + "\n"
    print(table, flush=True)
    open(os.path.join(args.out, "visual_kernels.txt"), "w").write(table)
    del vis, x
    torch.cuda.empty_cache()

    seg = head + "config-4 train step split by CUDA events on the main stream:\n" + step_segments(dev, args.steps) + "\n"
    print(seg, flush=True)
    open(os.path.join(args.out, "step_segments.txt"), "w").write(seg)


if __name__ == "__main__":
    main()
