"""CPU restatement of the CTC prefix beam search that csrc/ctc_prefix_beam.cu runs (DESIGN.md §4.13).  Test
infrastructure only: the package never imports it.

    log_add(a, b)                                              log(exp(a) + exp(b)), bit-reproducible (see below)
    prefix_beam_search(lp[T,V], length, B, nbest, blank, prune=True) -> (status, [(tokens, score), ...])

The search, for one utterance, in fp64 natural logs (tot(s) = log_add(pb(s), pnb(s))):
  * start: the beam is [()] with pb = 0, pnb = -inf;
  * per frame t < length: K_t = torch.topk(lp[t], min(2B+1, V)) on the CPU, in its order (prune=False: all V classes);
    K_t[0] NaN fails the utterance (status 1).  Walking the beam in rank order, each entry s contributes first its stay
    candidate (pb' = tot(s) + lp[t,blank]; pnb' = pnb(s) + lp[t,last(s)], -inf for (); if s[:-1] is in the beam as p,
    pnb' = log_add(pnb', ext(p, last(s))), with ext(p, c) = (c == last(p) ? pb(p) : tot(p)) + lp[t,c]), then one
    candidate s+c per c of K_t in order with c != blank and s+c not in the beam (pb' = -inf, pnb' = ext(s, c));
  * candidates whose tot' is -inf (or NaN) are dropped, the rest stably sorted by tot' descending, the first B kept;
  * the result is the first min(nbest, |beam|) entries with their tot; length 0 gives [((), 0.0)]; a length outside
    [0, T] fails with status 2.

log_add is one fixed sequence of IEEE fp64 operations (no library transcendental, no fused multiply-add), so that the
CUDA kernel, which evaluates the same sequence with __dadd_rn / __dmul_rn / __ddiv_rn, gets the same bits:
  a >= b after a swap; b = -inf -> a; d = b - a < -708 (or NaN) -> a;
  exp(d) = 2^k * P(r): k = floor(d * (1/ln2) + 0.5), r = (d - k*ln2_hi) - k*ln2_lo, P = Taylor series to r^13 (Horner);
  log1p(e) = 2 s Q(s^2): s = e / (2 + e), Q = sum_{n<=16} z^n / (2n+1) (Horner);  result a + (s * Q) * 2.
"""
from __future__ import annotations

import math

import numpy as np
import torch

NEG_INF = float("-inf")
CUTOFF = -708.0                       # exp(d) below ~2^-1021: 2^k stays a normal number, and the term is below 1 ulp
INV_LN2 = float.fromhex("0x1.71547652b82fep+0")
LN2_HI = float.fromhex("0x1.62e42fee00000p-1")     # fdlibm's split of ln 2: k * LN2_HI is exact for |k| < 2^20
LN2_LO = float.fromhex("0x1.a39ef35793c76p-33")
EXP_C = [float.fromhex(h) for h in (             # 1/n!, n = 0..13
    "0x1.0000000000000p+0", "0x1.0000000000000p+0", "0x1.0000000000000p-1", "0x1.5555555555555p-3",
    "0x1.5555555555555p-5", "0x1.1111111111111p-7", "0x1.6c16c16c16c17p-10", "0x1.a01a01a01a01ap-13",
    "0x1.a01a01a01a01ap-16", "0x1.71de3a556c734p-19", "0x1.27e4fb7789f5cp-22", "0x1.ae64567f544e4p-26",
    "0x1.1eed8eff8d898p-29", "0x1.6124613a86d09p-33")]
LOG_C = [float.fromhex(h) for h in (             # 1/(2n+1), n = 0..16
    "0x1.0000000000000p+0", "0x1.5555555555555p-2", "0x1.999999999999ap-3", "0x1.2492492492492p-3",
    "0x1.c71c71c71c71cp-4", "0x1.745d1745d1746p-4", "0x1.3b13b13b13b14p-4", "0x1.1111111111111p-4",
    "0x1.e1e1e1e1e1e1ep-5", "0x1.af286bca1af28p-5", "0x1.8618618618618p-5", "0x1.642c8590b2164p-5",
    "0x1.47ae147ae147bp-5", "0x1.2f684bda12f68p-5", "0x1.1a7b9611a7b96p-5", "0x1.0842108421084p-5",
    "0x1.f07c1f07c1f08p-6")]


def log_add(a: float, b: float) -> float:
    if b > a:
        a, b = b, a
    if b == NEG_INF:
        return a
    d = b - a
    if not d >= CUTOFF:
        return a
    k = float(math.floor(d * INV_LN2 + 0.5))
    r = (d - k * LN2_HI) - k * LN2_LO
    p = EXP_C[13]
    for c in EXP_C[12::-1]:
        p = p * r + c
    e = math.ldexp(p, int(k))
    s = e / (2.0 + e)
    z = s * s
    q = LOG_C[16]
    for c in LOG_C[15::-1]:
        q = q * z + c
    return a + (s * q) * 2.0


def _topk_lists(lp: np.ndarray, k: int):
    """torch.topk on the CPU, row by row in its own order (ties included): ([T,k] float values, [T,k] int classes)."""
    v, i = torch.topk(torch.from_numpy(np.ascontiguousarray(lp, dtype=np.float32)), k, dim=-1)
    return v.double().tolist(), i.tolist()


def prefix_beam_search(lp, length, B: int, nbest: int, blank: int, prune: bool = True):
    """lp: [T,V] float32 log-probs of one utterance.  Returns (status, hyps): status 0 with hyps = [(tokens tuple,
    score float)], or status 1 (NaN row) / 2 (length outside [0, T]) with hyps = []."""
    lp = np.asarray(lp, dtype=np.float32)
    T, V = lp.shape
    if not 1 <= B or not 1 <= nbest <= B or not 0 <= blank < V:
        raise ValueError("bad B / nbest / blank")
    length = int(length)
    if length < 0 or length > T:
        return 2, []
    if length == 0:
        return 0, [((), 0.0)]
    k = min(2 * B + 1, V) if prune else V
    kv, ki = _topk_lists(lp[:length], k)
    rows = lp[:length].astype(np.float64)
    # beam: list of (prefix, pb, pnb, tot) in rank order
    beam = [((), 0.0, NEG_INF, 0.0)]
    for t in range(length):
        vals, idx = kv[t], ki[t]
        if vals[0] != vals[0]:
            return 1, []
        row = rows[t]
        lpb = float(row[blank])
        where = {e[0]: e for e in beam}
        cands = []
        for s, pb, pnb, tot in beam:
            if s:
                c = s[-1]
                lpc = float(row[c])
                spnb = pnb + lpc
                p = where.get(s[:-1])
                if p is not None:
                    ext = ((p[1] if (p[0] and p[0][-1] == c) else p[3])) + lpc
                    spnb = log_add(spnb, ext)
            else:
                spnb = NEG_INF
            spb = tot + lpb
            cands.append((log_add(spb, spnb), s, spb, spnb))
            last = s[-1] if s else -1
            for v, c in zip(vals, idx):
                if c == blank:
                    continue
                sc = s + (c,)
                if sc in where:
                    continue
                e = (pb if c == last else tot) + v
                cands.append((e, sc, NEG_INF, e))
        kept = [x for x in cands if x[0] > NEG_INF]
        kept.sort(key=lambda x: -x[0])          # stable: earlier candidates win ties
        beam = [(s, pb, pnb, tot) for tot, s, pb, pnb in kept[:B]]
    return 0, [(s, tot) for s, _, _, tot in beam[:nbest]]
