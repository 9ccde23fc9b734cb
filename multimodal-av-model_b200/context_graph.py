"""Contextual biasing for the CTC prefix beam search: a phrase list as an Aho-Corasick automaton (DESIGN.md §4.15).

    ctx = ContextGraph.from_phrases([[17, 42, 9], ([5, 6], 3.0)], vocab_size=V, blank=3, weight=2.0)
    ctx = ContextGraph.from_text(["홍길동", "서울역"], tokenizer, weight=2.0)
    ctc_prefix_beam_search(log_probs, ..., context=ctx)  -> BiasedHypothesis entries (bias_score per hypothesis)

Each phrase is a sequence of 1..64 model token ids (no blank) with a per-token weight w > 0 in nats.  A hypothesis
that contains a phrase earns the sum of its per-token weights once per occurrence; a partial match earns credit while
it is being spelled (so the phrase survives the beam) and loses it again if it breaks off or never completes.

The automaton is built on the host with numpy and uploaded once per device, in the layout include/avctc_b200.h
documents for avctc_context_graph:
  * nodes in BFS order (root 0; within a level by parent number, then token id);
  * tau(v) = max weight of the phrases through v, phi(v) = phi(parent) + tau(v), omega(v) = phi of the first node on
    v's fail chain that ends a phrase (0 if none);
  * token_sym[V]: the context-alphabet symbol of a token (the distinct phrase tokens in ascending id order), -1 for a
    token of no phrase; delta[num_nodes, A]: the dense transition table (a token of no phrase returns to the root).
"""
from __future__ import annotations

import math
from typing import Dict, List, Sequence, Tuple

import numpy as np
import torch

from . import _lib

MAX_PHRASE_TOKENS = 64
MAX_NODES = 1 << 24
MAX_TABLE_BYTES = 1 << 30


def _entry(p, weight) -> Tuple[List[int], float]:
    """A phrase given as token ids, or as an (ids, weight) pair."""
    if isinstance(p, tuple) and len(p) == 2 and not isinstance(p[0], (int, np.integer)):
        ids, w = p
    else:
        ids, w = p, weight
    if isinstance(ids, str):
        raise TypeError("a phrase is a sequence of token ids; use ContextGraph.from_text for text")
    return [int(c) for c in ids], w


class ContextGraph:
    """A phrase list ready for ctc_prefix_beam_search(..., context=...)."""

    def __init__(self, vocab_size: int, blank: int, token_sym: np.ndarray, delta: np.ndarray, node: np.ndarray,
                 num_phrases: int):
        self.vocab_size = vocab_size
        self.blank = blank
        self.token_sym = token_sym            # int32 [V]
        self.delta = delta                    # int32 [num_nodes, A]
        self.node = node                      # float64 [num_nodes, 2]: phi, omega
        self.num_phrases = num_phrases
        self._dev: Dict[int, tuple] = {}

    @property
    def num_nodes(self) -> int:
        return self.node.shape[0]

    @property
    def alphabet(self) -> int:
        return self.delta.shape[1]

    @property
    def table_bytes(self) -> int:
        """Device bytes of the tables (token map, transition table, node values)."""
        return self.token_sym.nbytes + self.delta.nbytes + self.node.nbytes

    @classmethod
    def from_text(cls, texts: Sequence[str], tokenizer, weight: float = 2.0) -> "ContextGraph":
        """Phrases as text, encoded with tokenizer.encode; V and blank come from tokenizer.vocab_size / blank_id."""
        if isinstance(texts, str):
            raise TypeError("texts must be a sequence of phrases, not one string")
        return cls.from_phrases([tokenizer.encode(t) for t in texts], int(tokenizer.vocab_size),
                                int(tokenizer.blank_id), weight=weight)

    @classmethod
    def from_phrases(cls, phrases, vocab_size: int, blank: int, weight: float = 2.0) -> "ContextGraph":
        """phrases: token-id sequences, or (ids, weight) pairs; `weight` applies to bare sequences."""
        V, blank = int(vocab_size), int(blank)
        if not 1 <= V <= 1024:
            raise ValueError(f"vocab_size must be in [1, 1024], got {V}")
        if not 0 <= blank < V:
            raise ValueError(f"blank must be in [0, {V}), got {blank}")
        entries = [_entry(p, weight) for p in phrases]
        if not entries:
            raise ValueError("the phrase list is empty")
        for i, (ids, w) in enumerate(entries):
            if not 1 <= len(ids) <= MAX_PHRASE_TOKENS:
                raise ValueError(f"phrase {i} has {len(ids)} tokens; 1..{MAX_PHRASE_TOKENS} allowed")
            for c in ids:
                if not 0 <= c < V:
                    raise ValueError(f"phrase {i}: token {c} outside [0, {V})")
                if c == blank:
                    raise ValueError(f"phrase {i}: token {c} is the blank")
            if isinstance(w, bool) or not isinstance(w, (int, float, np.floating, np.integer)):
                raise ValueError(f"phrase {i}: weight {w!r} is not a number")
            if not (math.isfinite(float(w)) and float(w) > 0.0):
                raise ValueError(f"phrase {i}: weight {w} must be finite and > 0")
        # trie with temporary ids: children[u][c] = child, tau = max weight through the node, end = ends a phrase
        children: List[Dict[int, int]] = [{}]
        tau = [0.0]
        end = [False]
        for ids, w in entries:
            u = 0
            for c in ids:
                v = children[u].get(c)
                if v is None:
                    v = children[u][c] = len(children)
                    children.append({})
                    tau.append(float(w))
                    end.append(False)
                else:
                    tau[v] = max(tau[v], float(w))
                u = v
            end[u] = True
            if len(children) > MAX_NODES:
                raise ValueError(f"the phrases need more than {MAX_NODES} automaton nodes")
        return cls._build(V, blank, children, tau, end, len(entries))

    @classmethod
    def _build(cls, V, blank, children, tau, end, num_phrases) -> "ContextGraph":
        # BFS numbering: parents in their order, children by token id; each depth is a contiguous range
        old_of, par, tok, depth = [0], [-1], [-1], [0]
        i = 0
        while i < len(old_of):
            kids = children[old_of[i]]
            for c in sorted(kids):
                old_of.append(kids[c])
                par.append(i)
                tok.append(c)
                depth.append(depth[i] + 1)
            i += 1
        n = len(old_of)
        old_of = np.array(old_of, dtype=np.int64)
        par = np.array(par, dtype=np.int64)
        tau_n = np.array(tau, dtype=np.float64)[old_of]
        end_n = np.array(end, dtype=bool)[old_of]
        tok = np.array(tok[1:], dtype=np.int64)              # token of the edge into node 1..n-1
        alpha_tokens = np.unique(tok)
        A = len(alpha_tokens)
        if n * A * 4 > MAX_TABLE_BYTES:
            raise ValueError(f"the transition table needs {n * A * 4} bytes; at most {MAX_TABLE_BYTES} allowed")
        token_sym = np.full(V, -1, dtype=np.int32)
        token_sym[alpha_tokens] = np.arange(A, dtype=np.int32)
        sym = np.concatenate([[-1], token_sym[tok]]).astype(np.int64)     # sym[v]: symbol of the edge into v
        bounds = np.searchsorted(np.array(depth), np.arange(depth[-1] + 2))   # bounds[d] = first node of depth d
        phi = np.zeros(n, dtype=np.float64)
        omega = np.zeros(n, dtype=np.float64)
        fail = np.zeros(n, dtype=np.int64)
        delta = np.zeros((n, A), dtype=np.int32)
        c = np.arange(bounds[1], bounds[2])
        delta[0, sym[c]] = c                                 # the root's row: its children, else the root
        for d in range(1, len(bounds) - 1):
            # depth d: every row it reads (parents' fails, fails) is at a smaller depth and complete
            v = np.arange(bounds[d], bounds[d + 1])
            pv = par[v]
            phi[v] = phi[pv] + tau_n[v]                      # one fp64 add per level
            fail[v] = 0 if d == 1 else delta[fail[pv], sym[v]]
            omega[v] = np.where(end_n[v], phi[v], omega[fail[v]])
            delta[v] = delta[fail[v]]
            c = np.arange(bounds[d + 1], bounds[d + 2]) if d + 2 < len(bounds) else np.arange(0)
            delta[par[c], sym[c]] = c                        # a node's own children override its fail's row
        node = np.ascontiguousarray(np.stack([phi, omega], axis=1))
        return cls(V, blank, token_sym, delta, node, num_phrases)

    def descriptor(self, device) -> _lib.ContextGraphDesc:
        """The avctc_context_graph of this graph's tables on `device`, uploaded on first use and kept."""
        idx = device.index if device.index is not None else torch.cuda.current_device()
        hit = self._dev.get(idx)
        if hit is None:
            dev = torch.device("cuda", idx)
            bufs = [torch.from_numpy(self.token_sym).to(dev), torch.from_numpy(self.delta).to(dev),
                    torch.from_numpy(self.node).to(dev)]
            d = _lib.ContextGraphDesc()
            d.num_nodes, d.alphabet, d.map_len = self.num_nodes, self.alphabet, self.vocab_size
            d.token_sym, d.delta, d.node = bufs[0].data_ptr(), bufs[1].data_ptr(), bufs[2].data_ptr()
            hit = self._dev[idx] = (d, bufs)
        return hit[0]
