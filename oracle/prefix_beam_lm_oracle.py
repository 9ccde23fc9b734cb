"""CPU restatement of the CTC prefix beam search with token n-gram shallow fusion that csrc/ctc_prefix_beam.cu runs
(DESIGN.md §4.14).  Test infrastructure only: the package never imports it, and it shares no code with the package's
ARPA loader (multimodal-av-model_b200/ngram_lm.py).

    read_arpa(text_or_path, vocab) -> ArpaLM                 token-level back-off n-gram, order 1..5
    ArpaLM.lm10(word, history) -> float                       log10 P(word | history), back-off walk of §4.14
    prefix_beam_lm_search(lp[T,V], length, B, nbest, blank, lm, alpha, beta, prune=True)
        -> (status, [(tokens, score, acoustic_score, lm_score), ...])

The search is prefix_beam_oracle.prefix_beam_search (§4.13) with one change: each prefix s carries an LM score L(s)
(L(()) = 0; an extension s+c adds delta = alpha * (lm10(c | <s> s) * LN10) + beta; a stay keeps L), and candidates are
ranked by key = tot' + L'.  Candidates whose tot' is -inf are dropped, the rest stably sorted by key descending and the
first B kept.  After the last frame every entry gets E = alpha * (lm10(</s> | <s> s) * LN10) and the beam is stably
re-sorted by tot + (L + E); a hypothesis reports acoustic = tot, lm = L + E, score = acoustic + lm.
"""
from __future__ import annotations

import math
import os

import numpy as np

from .prefix_beam_oracle import NEG_INF, _topk_lists, log_add

LN10 = float.fromhex("0x1.26bb1bbb55516p+1")
MARKERS = ("<s>", "</s>", "<unk>")
MAX_ORDER = 5


def _f32(text: str) -> float:
    """An ARPA value as KenLM stores it: parsed as a double, rounded to fp32, widened back exactly."""
    v = float(text)
    if not math.isfinite(v):
        raise ValueError(f"non-finite ARPA value {text!r}")
    return float(np.float32(v))


class ArpaLM:
    """probs[(w1, ..., wn)] = (log10 p, log10 bow) for every n-gram whose words are all model pieces or markers."""

    def __init__(self, order, probs, vocab):
        self.order = order
        self.probs = probs
        self.vocab = list(vocab)

    def word(self, token: int) -> str:
        w = self.vocab[token]
        return w if (w,) in self.probs else "<unk>"

    def lm10(self, word: str, history) -> float:
        """history: the words before `word`, <s> first.  acc = 0; for the context suffixes h from longest (order - 1
        words at most) to shortest: (h, word) in the table -> acc + logp, done; else acc += bow(h) (0 if h is absent);
        the empty suffix is the unigram of word (present: the caller maps absent pieces to <unk>)."""
        h = tuple(history)[len(history) - min(len(history), self.order - 1):]
        acc = 0.0
        for m in range(len(h), -1, -1):
            suf = h[len(h) - m:]
            hit = self.probs.get(suf + (word,))
            if hit is not None:
                return acc + hit[0]
            acc = acc + self.probs.get(suf, (0.0, 0.0))[1]
        raise AssertionError("unreachable: the unigram ends the walk")


def read_arpa(src, vocab) -> ArpaLM:
    text = open(src, encoding="utf-8").read() if os.path.exists(str(src)) else str(src)
    keep = set(vocab) | set(MARKERS)
    probs = {}
    seen = set()
    counts = {}
    section = 0
    order = 0
    for raw in text.splitlines():
        line = raw.strip()
        if not line:
            continue
        if line == "\\data\\":
            section = -1
            continue
        if line == "\\end\\":
            break
        if line.startswith("\\") and line.endswith("-grams:"):
            section = int(line[1:line.index("-")])
            if section > MAX_ORDER:
                raise ValueError(f"order {section} > {MAX_ORDER}")
            order = max(order, section)
            continue
        if section == -1:
            if line.startswith("ngram "):
                n, c = line[6:].split("=")
                if int(n) > MAX_ORDER:
                    raise ValueError(f"order {int(n)} > {MAX_ORDER}")
                counts[int(n)] = int(c)
            continue
        if section < 1:
            continue
        f = line.split()
        if len(f) not in (section + 1, section + 2):
            raise ValueError(f"bad {section}-gram line {raw!r}")
        words = tuple(f[1:section + 1])
        logp = _f32(f[0])
        bow = _f32(f[section + 1]) if len(f) == section + 2 else 0.0
        if words in seen:
            raise ValueError(f"duplicate n-gram {words}")
        seen.add(words)
        if all(w in keep for w in words):        # no query can reach an n-gram with another word
            probs[words] = (logp, bow)
    for m in MARKERS:
        if (m,) not in probs:
            raise ValueError(f"the ARPA file lacks {m}")
    order = max([order] + list(counts))
    if not 1 <= order <= MAX_ORDER:
        raise ValueError(f"order {order} outside 1..{MAX_ORDER}")
    return ArpaLM(order, probs, vocab)


def _delta(lm: ArpaLM, word, hist, alpha, beta):
    return alpha * (lm.lm10(word, hist) * LN10) + beta


def prefix_beam_lm_search(lp, length, B: int, nbest: int, blank: int, lm: ArpaLM, alpha: float, beta: float,
                          prune: bool = True):
    """lp: [T,V] float32 log-probs of one utterance.  Returns (status, hyps): status 0 with hyps = [(tokens tuple,
    score, acoustic_score, lm_score)], or status 1 (NaN row) / 2 (length outside [0, T]) with hyps = []."""
    lp = np.asarray(lp, dtype=np.float32)
    T, V = lp.shape
    if not 1 <= B or not 1 <= nbest <= B or not 0 <= blank < V:
        raise ValueError("bad B / nbest / blank")
    if len(lm.vocab) != V:
        raise ValueError(f"the LM's vocabulary has {len(lm.vocab)} pieces, log_probs {V} classes")
    if not (math.isfinite(alpha) and alpha >= 0.0 and math.isfinite(beta)):
        raise ValueError("bad alpha / beta")
    length = int(length)
    if length < 0 or length > T:
        return 2, []
    hist = lambda s: ("<s>",) + tuple(lm.word(c) for c in s)   # noqa: E731
    # beam: list of (prefix, pb, pnb, tot, L) in rank order
    beam = [((), 0.0, NEG_INF, 0.0, 0.0)]
    if length:
        k = min(2 * B + 1, V) if prune else V
        kv, ki = _topk_lists(lp[:length], k)
        rows = lp[:length].astype(np.float64)
    for t in range(length):
        vals, idx = kv[t], ki[t]
        if vals[0] != vals[0]:
            return 1, []
        row = rows[t]
        lpb = float(row[blank])
        where = {e[0]: e for e in beam}
        cands = []                               # (key, tot', prefix, pb', pnb', L')
        for s, pb, pnb, tot, L in beam:
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
            stot = log_add(spb, spnb)
            cands.append((stot + L, stot, s, spb, spnb, L))
            last = s[-1] if s else -1
            h = hist(s)
            for v, c in zip(vals, idx):
                if c == blank:
                    continue
                sc = s + (c,)
                if sc in where:
                    continue
                e = (pb if c == last else tot) + v
                Lc = L + _delta(lm, lm.word(c), h, alpha, beta)
                cands.append((e + Lc, e, sc, NEG_INF, e, Lc))
        kept = [x for x in cands if x[1] > NEG_INF]
        kept.sort(key=lambda x: -x[0])          # stable: earlier candidates win ties
        beam = [(s, pb, pnb, tot, L) for _, tot, s, pb, pnb, L in kept[:B]]
    fin = []
    for s, _, _, tot, L in beam:
        lm_score = L + alpha * (lm.lm10("</s>", hist(s)) * LN10)
        fin.append((tot + lm_score, s, tot, lm_score))
    fin.sort(key=lambda x: -x[0])
    return 0, [(s, score, tot, lms) for score, s, tot, lms in fin[:nbest]]
