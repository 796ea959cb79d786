"""Reference for lexicons (INTEGRATION.md section 9), built on the unchanged oracle like charset_ref.py.

``Trie`` restates the automaton over the tokenizer table; ``walk`` is the greedy choice along it with float64 ``p``;
``lexicon_forward`` is the oracle's ``PARSeq.forward`` (fixed 26-step schedule, one refinement) with a per-crop state in
every AR choice.  The refinement context is the walked AR tokens; the ids are a second walk over the returned logits.
"""
from __future__ import annotations

import numpy as np
import torch

N_CLASSES = 95
L = 26
DONE = -1


def byte_classes(itos: str, eos_id: int) -> dict:
    """character -> the classes (1..94, not eos_id) that print it, in class order."""
    out: dict = {}
    for c in range(1, N_CLASSES):
        if c != eos_id:
            out.setdefault(itos[c], []).append(c)
    return out


class Trie:
    """allow: bool [S, 95]; succ[s]: class -> successor state (DONE after class 0).  State 0 is the root."""

    def __init__(self, allow, succ):
        self.allow = np.asarray(allow, bool)
        self.succ = succ

    @property
    def n_states(self) -> int:
        return len(self.succ)


def make_trie(words, itos: str, eos_id: int, mask=None) -> Trie:
    """The trie over the distinct words (those whose every character `mask` (bool [95]) allows, when given)."""
    bc = byte_classes(itos, eos_id)
    if mask is not None:
        words = [w for w in words if all(any(mask[c] for c in bc[ch]) for ch in w)]
    kids, ends = [{}], [False]
    for w in sorted(set(words)):
        s = 0
        for ch in w:
            if ch not in kids[s]:
                kids[s][ch] = len(kids)
                kids.append({})
                ends.append(False)
            s = kids[s][ch]
        ends[s] = True
    allow = np.zeros((len(kids), N_CLASSES), bool)
    succ = []
    for s in range(len(kids)):
        m = {}
        if ends[s]:
            m[0] = DONE
        for ch, t in kids[s].items():
            for c in bc[ch]:
                m[c] = t
        for c in m:
            allow[s, c] = True
        succ.append(m)
    return Trie(allow, succ)


def one_state(mask) -> Trie:
    """One state allowing `mask` (bool [95]): class 0 to DONE, every other allowed class back to the state."""
    mask = np.asarray(mask, bool)
    return Trie(mask[None].copy(), [{c: (DONE if c == 0 else 0) for c in np.flatnonzero(mask)}])


def choose(row, allow) -> int:
    """The first maximum over the allowed classes; the lowest allowed class when none compares (all NaN or -inf)."""
    best, bi = -np.inf, None
    for c in np.flatnonzero(allow):
        if row[c] > best:
            best, bi = row[c], int(c)
    return int(np.flatnonzero(allow)[0]) if bi is None else bi


def step(trie: Trie, s: int, row):
    """-> (class, next state, allowed classes) of one greedy choice in state s (DONE allows every class)."""
    allow = np.ones(N_CLASSES, bool) if s == DONE else trie.allow[s]
    c = choose(row, allow)
    return c, (DONE if s == DONE else trie.succ[s][c]), allow


def walk(logits, trie: Trie):
    """logits [26, 95] -> (ids int32 [26], p float64 [26]): the walk from the root; p renormalised over each position's
    allowed classes, 1 / sum_{c allowed} exp(l[c] - l[id]) (NaN where an allowed logit is NaN or all are -inf)."""
    ids = np.zeros(len(logits), np.int32)
    p = np.zeros(len(logits), np.float64)
    s = 0
    for t, row in enumerate(np.asarray(logits)):
        c, s_next, allow = step(trie, s, row)
        l64 = np.asarray(row, np.float64)[allow]
        best = max((v for v in l64 if not np.isnan(v)), default=-np.inf)
        with np.errstate(invalid="ignore", over="ignore"):
            p[t] = 1.0 / np.exp(l64 - best).sum()
        ids[t] = c
        s = s_next
    return ids, p


def text_of(ids, itos: str, eos_id: int) -> str:
    """The text decode_ids gives: the characters before the first class 0, class eos_id dropped."""
    out = []
    for c in ids:
        if c == 0:
            break
        if c != eos_id:
            out.append(itos[int(c)])
    return "".join(out)


@torch.no_grad()
def lexicon_forward(parseq, images, tries, forced_tokens: torch.Tensor | None = None, taps: dict | None = None):
    """The oracle's PARSeq.forward with each crop b's AR choices walking tries[b].  taps (optional dict) receives
    ar_logits (N, 26, 95) and ar_tokens (N, 26) like the oracle's taps.  -> the refinement logits (N, 26, 95)."""
    bs = images.shape[0]
    num_steps = parseq.max_label_length + 1
    memory = parseq.encode(images)
    pos_queries = parseq.pos_queries[:, :num_steps].expand(bs, -1, -1)
    query_mask = torch.triu(torch.full((num_steps, num_steps), float("-inf")), 1)
    tgt_in = torch.full((bs, num_steps), parseq.pad_id, dtype=torch.long)
    tgt_in[:, 0] = parseq.bos_id
    state = [0] * bs
    logits = []
    for i in range(num_steps):
        j = i + 1
        tgt_out = parseq.decode(tgt_in[:, :j], memory, tgt_query=pos_queries[:, i:j], tgt_query_mask=query_mask[i:j, :j])
        p_i = parseq.head(tgt_out)
        logits.append(p_i)
        if j < num_steps:
            if forced_tokens is None:
                for b in range(bs):
                    c, state[b], _ = step(tries[b], state[b], p_i[b, 0].numpy())
                    tgt_in[b, j] = c
            else:
                tgt_in[:, j] = forced_tokens[:, i]
    logits = torch.cat(logits, dim=1)
    if taps is not None:
        taps["ar_logits"] = logits
        taps["ar_tokens"] = tgt_in.clone()
    query_mask[torch.triu(torch.ones(num_steps, num_steps, dtype=torch.bool), 2)] = 0
    tgt_padding_mask = (tgt_in == parseq.eos_id).int().cumsum(-1) > 0
    tgt_out = parseq.decode(tgt_in, memory, tgt_padding_mask, tgt_query=pos_queries,
                            tgt_query_mask=query_mask[:, : tgt_in.shape[1]])
    return parseq.head(tgt_out)
