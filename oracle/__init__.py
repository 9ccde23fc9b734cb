"""oracle/ — CPU restatement of the reference's AV-CTC hot path.  TEST INFRASTRUCTURE ONLY.

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` / ``--impl reference``
legs may import this package, and only as the checker or the timed CPU baseline.  Nothing in
``multimodal-av-model_b200/`` imports it; the product fails loudly when its CUDA library is missing.

Parity status: the reference (/root/reference) has no tests or golden vectors of its own
(SURVEY.md §4, §8c).  The oracle is pinned instead against outputs of the reference's own Python
modules executed in the build container by ``oracle/gen_golden.py`` (fixtures committed under
``tests/golden/`` with the torch version recorded).  There is nothing to compile under
``oracle/_ref``: the reference is pure Python and cannot travel to the GPU box.

Layers:
  * ``ctc_oracle.c`` / ``beam_oracle.cpp``  plain C/C++ (float64 CTC alpha-beta; libstdc++ top-k tie order
    + literal beam search) -> ``oracle/_build/liboracle.so``, called through ctypes below.
  * ``np_oracle.py``   numpy float64 restatement of fusion_module / decoder / contrastive arithmetic.
  * ``torch_port.py``  restatement of the same modules on torch CPU ops (what the reference really
    executes); used for gradients at larger sizes and as the timed CPU baseline.
  * ``w2v_oracle.py``  float64 forward and backward of the two wav2vec2 layer halves csrc/wav2vec2_layer.cu runs,
    written out without autograd, with optional bf16 rounding at the module path's points.
  * ``fusion_oracle.py``  float64 forward and backward of the fusion-path kernels (resample, softmax, column sums,
    log-softmax, attention, GEMM), with optional bf16 rounding where the attention kernel materialises bf16.
"""
from __future__ import annotations

import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "_build", "liboracle.so")
_lib = None


def build(force: bool = False) -> str:
    """Compile the C/C++ oracle with gcc/g++ (recipe: oracle/Makefile)."""
    srcs = [os.path.join(_HERE, f) for f in ("ctc_oracle.c", "beam_oracle.cpp", "Makefile")]
    stale = (not os.path.exists(_LIB_PATH)) or any(
        os.path.getmtime(s) > os.path.getmtime(_LIB_PATH) for s in srcs)
    if force or stale:
        subprocess.run(["make", "-C", _HERE, "-s"], check=True)
    return _LIB_PATH


def lib() -> ctypes.CDLL:
    global _lib
    if _lib is None:
        build()
        L = ctypes.CDLL(_LIB_PATH)
        c_i64p = ctypes.POINTER(ctypes.c_int64)
        c_dp = ctypes.POINTER(ctypes.c_double)
        c_fp = ctypes.POINTER(ctypes.c_float)
        c_ip = ctypes.POINTER(ctypes.c_int)
        L.ctc_oracle.restype = ctypes.c_int
        L.ctc_oracle.argtypes = [c_dp, ctypes.c_int64, ctypes.c_int64, ctypes.c_int, ctypes.c_int,
                                 ctypes.c_int, c_i64p, ctypes.c_int64, c_i64p, c_i64p, ctypes.c_int,
                                 ctypes.c_int, ctypes.c_int, ctypes.c_double, c_dp, c_dp, c_dp]
        L.topk_oracle.restype = ctypes.c_int
        L.topk_oracle.argtypes = [c_fp, ctypes.c_int, ctypes.c_int, c_fp, c_i64p]
        L.beam_oracle.restype = ctypes.c_int
        L.beam_oracle.argtypes = [c_fp, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                  c_i64p, c_ip, c_dp, c_i64p, c_ip]
        L.beam_oracle_batch.restype = ctypes.c_int
        L.beam_oracle_batch.argtypes = [c_fp, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                        ctypes.c_int, c_i64p, c_ip]
        _lib = L
    return _lib


def _p(a, ct):
    return a.ctypes.data_as(ctypes.POINTER(ct))


_RED = {"none": 0, "mean": 1, "sum": 2}


def ctc_loss(log_probs, targets, input_lengths, target_lengths, blank=0, reduction="mean",
             zero_infinity=False, grad_out=1.0, want_grad=True):
    """float64 CTC.  log_probs: array-like [T,B,V]; targets [B,Lmax] int.  Returns dict with
    nll[B], loss (scalar for mean/sum, None for 'none'), grad[T,B,V] (d loss / d log_probs in
    torch's softmax-folded convention; for 'none' the gradient of sum_b nll_b * grad_out)."""
    lp = np.ascontiguousarray(np.asarray(log_probs, dtype=np.float64))
    T, B, V = lp.shape
    tg = np.ascontiguousarray(np.asarray(targets, dtype=np.int64))
    if tg.ndim == 1:  # concatenated targets -> padded 2-D
        tl_ = np.asarray(target_lengths, dtype=np.int64)
        out = np.zeros((B, max(int(tl_.max()) if B else 0, 1)), dtype=np.int64)
        o = 0
        for b in range(B):
            out[b, :tl_[b]] = tg[o:o + tl_[b]]
            o += int(tl_[b])
        tg = out
    il = np.ascontiguousarray(np.asarray(input_lengths, dtype=np.int64))
    tl = np.ascontiguousarray(np.asarray(target_lengths, dtype=np.int64))
    nll = np.zeros(B, dtype=np.float64)
    loss = np.zeros(1, dtype=np.float64)
    grad = np.zeros((T, B, V), dtype=np.float64) if want_grad else None
    rc = lib().ctc_oracle(_p(lp, ctypes.c_double), B * V, V, T, B, V, _p(tg, ctypes.c_int64),
                          tg.shape[1] if tg.ndim == 2 else 0, _p(il, ctypes.c_int64),
                          _p(tl, ctypes.c_int64), int(blank), _RED[reduction], int(zero_infinity),
                          float(grad_out), _p(nll, ctypes.c_double), _p(loss, ctypes.c_double),
                          _p(grad, ctypes.c_double) if want_grad else None)
    if rc != 0:
        raise ValueError("ctc_oracle: bad lengths")
    return {"nll": nll, "loss": None if reduction == "none" else float(loss[0]), "grad": grad}


def topk(row, k):
    """torch.topk(row, k) on CPU incl. its tie order.  row: float32 [V]."""
    r = np.ascontiguousarray(np.asarray(row, dtype=np.float32))
    vals = np.zeros(k, dtype=np.float32)
    idx = np.zeros(k, dtype=np.int64)
    rc = lib().topk_oracle(_p(r, ctypes.c_float), r.shape[0], int(k), _p(vals, ctypes.c_float),
                           _p(idx, ctypes.c_int64))
    if rc != 0:
        raise ValueError("topk_oracle: bad k")
    return vals, idx


def beam_search(log_probs, beam_width=5, blank=0, debug=False):
    """simple_beam_search(log_probs[T,V]) -> list[int] (optionally also final beams)."""
    lp = np.ascontiguousarray(np.asarray(log_probs, dtype=np.float32))
    T, V = lp.shape
    out = np.zeros(max(T, 1), dtype=np.int64)
    n = ctypes.c_int(0)
    if debug:
        sc = np.zeros(beam_width, dtype=np.float64)
        paths = np.zeros((beam_width, max(T, 1)), dtype=np.int64)
        nf = ctypes.c_int(0)
        rc = lib().beam_oracle(_p(lp, ctypes.c_float), T, V, int(beam_width), int(blank),
                               _p(out, ctypes.c_int64), ctypes.byref(n), _p(sc, ctypes.c_double),
                               _p(paths, ctypes.c_int64), ctypes.byref(nf))
        if rc != 0:
            raise ValueError("beam_oracle: bad beam width")
        return out[:n.value].tolist(), sc[:nf.value], paths[:nf.value, :T]
    rc = lib().beam_oracle(_p(lp, ctypes.c_float), T, V, int(beam_width), int(blank),
                           _p(out, ctypes.c_int64), ctypes.byref(n), None, None, None)
    if rc != 0:
        raise ValueError("beam_oracle: bad beam width")
    return out[:n.value].tolist()


def beam_search_batch(log_probs, beam_width=5, blank=0):
    """[N,T,V] float32 -> list of N token lists."""
    lp = np.ascontiguousarray(np.asarray(log_probs, dtype=np.float32))
    N, T, V = lp.shape
    out = np.zeros((N, max(T, 1)), dtype=np.int64)
    n = np.zeros(N, dtype=np.int32)
    rc = lib().beam_oracle_batch(_p(lp, ctypes.c_float), N, T, V, int(beam_width), int(blank),
                                 _p(out, ctypes.c_int64), _p(n, ctypes.c_int))
    if rc != 0:
        raise ValueError("beam_oracle: bad beam width")
    return [out[i, :n[i]].tolist() for i in range(N)]
