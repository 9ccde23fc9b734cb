"""CPU restatement of the contextually biased CTC prefix beam search that csrc/ctc_prefix_beam.cu runs (DESIGN.md
§4.15), with or without the token n-gram LM of §4.14.  Test infrastructure only: the package never imports it, and it
shares no code with the package's graph builder (multimodal-av-model_b200/context_graph.py): the automaton here is
dicts, and its transition walks fail links at query time instead of reading a dense table.

    ContextAutomaton(phrases)                         phrases: [(token ids, weight)], weight a float > 0
    ContextAutomaton.delta(u, c) -> node              the Aho-Corasick transition
    ContextAutomaton.phi[v], .omega(v), .fail[v]      depth potential, completion credit, fail link
    bias_of(automaton, tokens) -> float               the rule applied directly to one token sequence
    prefix_beam_bias_search(lp[T,V], length, B, nbest, blank, phrases, lm=None, alpha=0.5, beta=0.0, prune=True)
        -> (status, [(tokens, score, acoustic_score, lm_score, bias_score), ...])

The automaton: node 0 is the root; trie nodes are numbered in BFS order, within a level by parent number, then token
id.  tau(v) = max weight of the phrases through v; phi(root) = 0, phi(v) = phi(parent) + tau(v); fail(v) = the longest
proper suffix of v's path that is a trie node; delta(u, c) = child(u, c) if present, else delta(fail(u), c), and the
root when the root has no such child; omega(v) = phi(e) for the first e on v, fail(v), fail(fail(v)), ... that ends a
phrase, 0 if none does.

The search is prefix_beam_lm_oracle.prefix_beam_lm_search (§4.14; §4.13 without an LM) with each prefix s also
carrying a node u(s) and a bias score G(s) (root and 0 for ()).  A stay keeps both; an extension s+c (the repeat
extension included) moves to v = delta(u, c) and adds (phi(v) - phi(u)) + omega(v) to G.  Candidates are ranked by
key = (tot' + L') + G' with an LM, tot' + G' without; those with tot' = -inf are dropped, the rest stably sorted by key
descending and the first B kept.  After the last frame: bias = G - phi(u), lm = L + E (0 without an LM), score =
(acoustic + lm) + bias, and the beam is stably re-sorted by score.
"""
from __future__ import annotations

import math

import numpy as np

from .prefix_beam_lm_oracle import LN10, ArpaLM
from .prefix_beam_oracle import NEG_INF, _topk_lists, log_add


class ContextAutomaton:
    def __init__(self, phrases):
        phrases = [(tuple(int(c) for c in ids), float(w)) for ids, w in phrases]
        if not phrases:
            raise ValueError("no phrases")
        for ids, w in phrases:
            if not ids or not (math.isfinite(w) and w > 0.0):
                raise ValueError(f"bad phrase {ids} / weight {w}")
        # every prefix of every phrase is a trie node; tau = max weight of the phrases it starts
        tau = {}
        for ids, w in phrases:
            for i in range(1, len(ids) + 1):
                tau[ids[:i]] = max(tau.get(ids[:i], 0.0), w)
        ends = {ids for ids, _ in phrases}
        # BFS numbering: level by level, sorted by (parent's number, token)
        self.paths = [()]
        num = {(): 0}
        depth = max(len(ids) for ids, _ in phrases)
        for d in range(1, depth + 1):
            level = sorted((p for p in tau if len(p) == d), key=lambda p: (num[p[:-1]], p[-1]))
            for p in level:
                num[p] = len(self.paths)
                self.paths.append(p)
        n = len(self.paths)
        self.children = [dict() for _ in range(n)]
        self.phi = [0.0] * n
        self.end = [False] * n
        for v in range(1, n):
            p = self.paths[v]
            u = num[p[:-1]]
            self.children[u][p[-1]] = v
            self.phi[v] = self.phi[u] + tau[p]
            self.end[v] = p in ends
        self.fail = [0] * n
        for v in range(1, n):                       # BFS order: fail(parent) is known
            p = self.paths[v]
            u = num[p[:-1]]
            self.fail[v] = 0 if u == 0 else self.delta(self.fail[u], p[-1])

    @property
    def num_nodes(self) -> int:
        return len(self.paths)

    def delta(self, u: int, c: int) -> int:
        while True:
            v = self.children[u].get(c)
            if v is not None:
                return v
            if u == 0:
                return 0
            u = self.fail[u]

    def omega(self, v: int) -> float:
        while v != 0:
            if self.end[v]:
                return self.phi[v]
            v = self.fail[v]
        return 0.0

    def step(self, u: int, G: float, c: int):
        """One extension by token c from node u with bias score G: (v, G')."""
        v = self.delta(u, c)
        return v, G + ((self.phi[v] - self.phi[u]) + self.omega(v))


def bias_of(ac: ContextAutomaton, tokens) -> float:
    """The final bias of a hypothesis: G - phi(u) after stepping through its tokens from the root."""
    u, G = 0, 0.0
    for c in tokens:
        u, G = ac.step(u, G, int(c))
    return G - ac.phi[u]


def prefix_beam_bias_search(lp, length, B: int, nbest: int, blank: int, phrases, lm: ArpaLM = None,
                            alpha: float = 0.5, beta: float = 0.0, prune: bool = True):
    """lp: [T,V] float32 log-probs of one utterance; phrases: [(ids, weight)] or a ContextAutomaton.  Returns (status,
    hyps): status 0 with hyps = [(tokens tuple, score, acoustic_score, lm_score, bias_score)], or status 1 (NaN row) /
    2 (length outside [0, T]) with hyps = []."""
    lp = np.asarray(lp, dtype=np.float32)
    T, V = lp.shape
    if not 1 <= B or not 1 <= nbest <= B or not 0 <= blank < V:
        raise ValueError("bad B / nbest / blank")
    ac = phrases if isinstance(phrases, ContextAutomaton) else ContextAutomaton(phrases)
    if any(not 0 <= c < V or c == blank for p in ac.paths for c in p):
        raise ValueError("a phrase token is the blank or outside [0, V)")
    if lm is not None:
        if len(lm.vocab) != V:
            raise ValueError(f"the LM's vocabulary has {len(lm.vocab)} pieces, log_probs {V} classes")
        if not (math.isfinite(alpha) and alpha >= 0.0 and math.isfinite(beta)):
            raise ValueError("bad alpha / beta")
    length = int(length)
    if length < 0 or length > T:
        return 2, []
    hist = lambda s: ("<s>",) + tuple(lm.word(c) for c in s)   # noqa: E731
    # beam: list of (prefix, pb, pnb, tot, L, u, G) in rank order
    beam = [((), 0.0, NEG_INF, 0.0, 0.0, 0, 0.0)]
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
        cands = []                               # (key, tot', prefix, pb', pnb', L', u', G')
        for s, pb, pnb, tot, L, u, G in beam:
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
            cands.append((((stot + L) if lm is not None else stot) + G, stot, s, spb, spnb, L, u, G))
            last = s[-1] if s else -1
            h = hist(s) if lm is not None else None
            for v, c in zip(vals, idx):
                if c == blank:
                    continue
                sc = s + (c,)
                if sc in where:
                    continue
                e = (pb if c == last else tot) + v
                if lm is not None:
                    Lc = L + (alpha * (lm.lm10(lm.word(c), h) * LN10) + beta)
                    key = e + Lc
                else:
                    Lc = 0.0
                    key = e
                uc, Gc = ac.step(u, G, c)
                cands.append((key + Gc, e, sc, NEG_INF, e, Lc, uc, Gc))
        kept = [x for x in cands if x[1] > NEG_INF]
        kept.sort(key=lambda x: -x[0])          # stable: earlier candidates win ties
        beam = [(s, pb, pnb, tot, L, u, G) for _, tot, s, pb, pnb, L, u, G in kept[:B]]
    fin = []
    for s, _, _, tot, L, u, G in beam:
        lm_score = L + alpha * (lm.lm10("</s>", hist(s)) * LN10) if lm is not None else 0.0
        bias = G - ac.phi[u]
        fin.append(((tot + lm_score) + bias, s, tot, lm_score, bias))
    fin.sort(key=lambda x: -x[0])
    return 0, [(s, score, tot, lms, bias) for score, s, tot, lms, bias in fin[:nbest]]
