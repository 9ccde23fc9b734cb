"""Token-level back-off n-gram language model for shallow fusion in the CTC prefix beam search (DESIGN.md §4.14).

    lm = NgramLM.from_arpa(path, vocab)      vocab[i] = the piece of model token i, e.g. tokenizer.id_to_token
    lm.order, lm.counts                       order (1..5) and the n-grams kept per order
    ctc_prefix_beam_search(log_probs, ..., lm=lm, lm_weight=0.5, token_bonus=0.0)

The ARPA file's words are the model's pieces plus <s>, </s> and <unk> (a token LM: pieces as space-separated words,
estimated e.g. with KenLM's `lmplz`; see INTEGRATION.md).  Model token i is looked up as the word vocab[i], or as <unk>
when the LM lacks it.  Values are parsed as Python floats and rounded to fp32, as KenLM stores them.  N-grams with a
word that is neither a model piece nor a marker are dropped: no query can reach them.  The tables are built on the
host with numpy and uploaded once per device; the layout is the one include/avctc_b200.h documents for
avctc_ngram_lm (dense unigrams, one open-addressing hash table per order >= 2).
"""
from __future__ import annotations

import math
from typing import Dict, List, Sequence, Tuple

import numpy as np
import torch

from . import _lib

MAX_ORDER = 5
MAX_VOCAB = 1024
BOS, EOS, UNK = 0, 1, 2              # LM word ids of the markers; pieces follow
_BITS = 11
_EMPTY = np.uint64(0xFFFF_FFFF_FFFF_FFFF)
_HASH_MUL = np.uint64(0x9E3779B97F4A7C15)


def _parse_arpa(path: str) -> Tuple[int, List[List[Tuple[List[str], float, float]]]]:
    """-> (order, grams[n-1] = [(words, log10 p, log10 bow)]), every value a finite double (rounded to fp32 when the
    tables are built)."""
    declared = 0
    grams: List[list] = [[] for _ in range(MAX_ORDER)]
    section = 0
    with open(path, encoding="utf-8") as f:
        for raw in f:
            line = raw.strip()
            if not line:
                continue
            if line == "\\data\\":
                section = -1
            elif line == "\\end\\":
                break
            elif line.startswith("\\") and line.endswith("-grams:"):
                section = int(line[1:line.index("-")])
                if not 1 <= section <= MAX_ORDER:
                    raise ValueError(f"{path}: {section}-grams: order must be 1..{MAX_ORDER}")
            elif section == -1:
                if line.startswith("ngram "):
                    n = int(line[6:].split("=")[0])
                    if not 1 <= n <= MAX_ORDER:
                        raise ValueError(f"{path}: order {n} outside 1..{MAX_ORDER}")
                    declared = max(declared, n)
            elif section >= 1:
                fl = line.split()
                if len(fl) not in (section + 1, section + 2):
                    raise ValueError(f"{path}: bad {section}-gram line {line!r}")
                logp = float(fl[0])
                bow = float(fl[section + 1]) if len(fl) == section + 2 else 0.0
                if not (math.isfinite(logp) and math.isfinite(bow)):
                    raise ValueError(f"{path}: non-finite value in {line!r}")
                grams[section - 1].append((fl[1:section + 1], logp, bow))
    order = max([declared] + [n + 1 for n in range(MAX_ORDER) if grams[n]])
    if order < 1:
        raise ValueError(f"{path}: no n-grams")
    return order, grams[:order]


def _hash_table(keys: np.ndarray, vals: np.ndarray) -> np.ndarray:
    """Open addressing with linear probing, at most half full: [capacity, 2] uint64 rows (key, logp | bow << 32)."""
    cap = 2
    while cap < 2 * len(keys):
        cap *= 2
    mask = np.uint64(cap - 1)
    tab = np.zeros((cap, 2), dtype=np.uint64)
    tab[:, 0] = _EMPTY
    h = keys * _HASH_MUL
    slot = (h ^ (h >> np.uint64(29))) & mask
    pending = np.arange(len(keys))
    while len(pending):
        s = slot[pending]
        free = pending[tab[s, 0] == _EMPTY]
        _, first = np.unique(slot[free], return_index=True)      # one key per free slot per round
        win = free[first]
        tab[slot[win], 0] = keys[win]
        tab[slot[win], 1] = vals[win]
        taken = np.zeros(len(keys), dtype=bool)
        taken[win] = True
        pending = pending[~taken[pending]]
        slot[pending] = (slot[pending] + np.uint64(1)) & mask
    return tab


def _pack_vals(logp: np.ndarray, bow: np.ndarray) -> np.ndarray:
    lo = logp.astype(np.float32).view(np.uint32).astype(np.uint64)
    hi = bow.astype(np.float32).view(np.uint32).astype(np.uint64)
    return lo | (hi << np.uint64(32))


class NgramLM:
    """A token-level back-off n-gram LM, ready for ctc_prefix_beam_search(..., lm=...)."""

    def __init__(self, order: int, counts: Tuple[int, ...], vocab_size: int, num_words: int,
                 token_word: np.ndarray, unigram: np.ndarray, tables: List[np.ndarray]):
        self.order = order
        self.counts = counts              # n-grams kept per order, 1-grams first
        self.vocab_size = vocab_size
        self.num_words = num_words
        self._token_word = token_word
        self._unigram = unigram
        self._tables = tables
        self._dev: Dict[int, tuple] = {}

    @property
    def table_bytes(self) -> int:
        """Device bytes of the tables (token map, unigrams, hash tables)."""
        return self._token_word.nbytes + self._unigram.nbytes + sum(t.nbytes for t in self._tables)

    @classmethod
    def from_arpa(cls, path: str, vocab: Sequence[str]) -> "NgramLM":
        vocab = list(vocab)
        if not 1 <= len(vocab) <= MAX_VOCAB:
            raise ValueError(f"vocab must list 1..{MAX_VOCAB} pieces (id -> piece), got {len(vocab)}")
        order, grams = _parse_arpa(path)
        arpa_words = {w[0]: i for i, (w, _, _) in enumerate(grams[0])}
        if len(arpa_words) != len(grams[0]):
            raise ValueError(f"{path}: duplicate 1-gram")
        for m in ("<s>", "</s>", "<unk>"):
            if m not in arpa_words:
                raise ValueError(f"{path}: the LM lacks {m}")
        # LM word ids: the markers, then the distinct pieces the LM has, in vocab order
        word_id = {"<s>": BOS, "</s>": EOS, "<unk>": UNK}
        for p in vocab:
            if p in arpa_words and p not in word_id:
                word_id[p] = len(word_id)
        num_words = len(word_id)
        token_word = np.array([word_id.get(p, UNK) for p in vocab], dtype=np.int32)
        # dev_of[ARPA word index] = LM word id, -1 for a word no query can reach (the last entry stands for every
        # word that has no 1-gram)
        n_uni = len(grams[0])
        dev_of = np.full(n_uni + 1, -1, dtype=np.int64)
        for w, i in arpa_words.items():
            dev_of[i] = word_id.get(w, -1)
        all_words = dict(arpa_words)
        unigram = np.zeros((num_words, 2), dtype=np.float32)
        counts = []
        tables = []
        for n, g in enumerate(grams, start=1):
            ids = np.array([[all_words.setdefault(w, len(all_words)) for w in words] for words, _, _ in g],
                           dtype=np.int64).reshape(len(g), n)
            if n > 1 and len(np.unique(ids, axis=0)) != len(ids):
                raise ValueError(f"{path}: duplicate {n}-gram")
            logp = np.array([x[1] for x in g], dtype=np.float64)
            bow = np.array([x[2] for x in g], dtype=np.float64)
            dev = dev_of[np.minimum(ids, n_uni)]
            keep = (dev >= 0).all(axis=1)
            dev, logp, bow = dev[keep], logp[keep], bow[keep]
            counts.append(int(keep.sum()))
            if n == 1:
                unigram[dev[:, 0], 0] = logp
                unigram[dev[:, 0], 1] = bow
                continue
            keys = np.zeros(len(dev), dtype=np.uint64)
            for j in range(n):
                keys = (keys << np.uint64(_BITS)) | dev[:, j].astype(np.uint64)
            tables.append(_hash_table(keys, _pack_vals(logp, bow)))
        return cls(order, tuple(counts), len(vocab), num_words, token_word, unigram, tables)

    def descriptor(self, device) -> _lib.NgramLMDesc:
        """The avctc_ngram_lm of this LM's tables on `device`, uploaded on first use and kept."""
        idx = device.index if device.index is not None else torch.cuda.current_device()
        hit = self._dev.get(idx)
        if hit is None:
            dev = torch.device("cuda", idx)
            bufs = [torch.from_numpy(self._token_word).to(dev), torch.from_numpy(self._unigram).to(dev)]
            bufs += [torch.from_numpy(t.view(np.int64)).to(dev) for t in self._tables]
            d = _lib.NgramLMDesc()
            d.order, d.num_words, d.bos, d.eos, d.map_len = self.order, self.num_words, BOS, EOS, self.vocab_size
            d.token_word, d.unigram = bufs[0].data_ptr(), bufs[1].data_ptr()
            for j, (t, b) in enumerate(zip(self._tables, bufs[2:])):
                d.table[j] = b.data_ptr()
                d.capacity[j] = t.shape[0]
            hit = self._dev[idx] = (d, bufs)
        return hit[0]
