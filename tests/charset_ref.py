"""Reference for character filters (INTEGRATION.md section 7), built on the unchanged oracle.

``class_mask_ref`` restates the class-mask rule over the tokenizer table.  ``masked_forward`` is the oracle's
``PARSeq.forward`` (fixed 26-step schedule, one refinement) with constrained greedy decoding: the AR feedback and the
refinement context are ``logits.masked_fill(~mask, -inf).argmax(-1)``, the returned logits stay unmasked.  With an
all-true mask it runs exactly the oracle's operations.  ``masked_pmax`` is the renormalised probability in float64.
"""
from __future__ import annotations

import numpy as np
import torch

N_CLASSES = 95


def class_mask_ref(itos: str, eos_id: int, allow: str | None = None, block: str | None = None) -> np.ndarray:
    """bool [95]: classes 0 and eos_id always; class c otherwise iff (allow is None or itos[c] in allow) and
    (block is None or itos[c] not in block)."""
    out = np.zeros(N_CLASSES, bool)
    for c in range(N_CLASSES):
        ch = itos[c]
        out[c] = c in (0, eos_id) or ((allow is None or ch in allow) and (block is None or ch not in block))
    return out


def mask_words(mask: np.ndarray) -> np.ndarray:
    """bool [..., 95] -> the uint32 [..., 4] device format (bit c & 31 of word c >> 5)."""
    m = np.asarray(mask, bool)
    bits = np.zeros(m.shape[:-1] + (128,), bool)
    bits[..., :N_CLASSES] = m
    w = bits.reshape(m.shape[:-1] + (4, 32)).astype(np.uint64) << np.arange(32, dtype=np.uint64)
    return w.sum(-1).astype(np.uint32)


def words_to_bool(words: np.ndarray) -> np.ndarray:
    """uint32 [..., 4] -> bool [..., 95]."""
    w = np.asarray(words, np.uint32)
    bits = (w[..., :, None] >> np.arange(32, dtype=np.uint32)) & 1
    return bits.reshape(w.shape[:-1] + (128,))[..., :N_CLASSES].astype(bool)


def masked_argmax(logits, mask: np.ndarray) -> np.ndarray:
    """First-max argmax over the allowed classes: logits [..., 95], mask bool broadcastable to it."""
    return np.where(mask, logits, -np.inf).argmax(-1)


def masked_pmax(logits, mask: np.ndarray) -> np.ndarray:
    """1 / sum_{c allowed} exp(l[c] - max_{c allowed} l[c]) in float64."""
    l64 = np.where(mask, np.asarray(logits, np.float64), -np.inf)
    return 1.0 / np.exp(l64 - l64.max(-1, keepdims=True)).sum(-1)


@torch.no_grad()
def masked_forward(parseq, images, class_mask: torch.Tensor | None = None, forced_tokens: torch.Tensor | None = None,
                   taps: dict | None = None):
    """The oracle's PARSeq.forward with class_mask (N, 95) bool applied to every greedy choice.  taps (optional dict)
    receives ar_logits (N, 26, 95) and ar_tokens (N, 26) like the oracle's taps."""
    bs = images.shape[0]
    num_steps = parseq.max_label_length + 1
    memory = parseq.encode(images)

    def pick(lg):
        return lg.argmax(-1) if class_mask is None else lg.masked_fill(~class_mask[:, None, :], float("-inf")).argmax(-1)

    pos_queries = parseq.pos_queries[:, :num_steps].expand(bs, -1, -1)
    query_mask = torch.triu(torch.full((num_steps, num_steps), float("-inf")), 1)
    tgt_in = torch.full((bs, num_steps), parseq.pad_id, dtype=torch.long)
    tgt_in[:, 0] = parseq.bos_id
    logits = []
    for i in range(num_steps):
        j = i + 1
        tgt_out = parseq.decode(tgt_in[:, :j], memory, tgt_query=pos_queries[:, i:j], tgt_query_mask=query_mask[i:j, :j])
        p_i = parseq.head(tgt_out)
        logits.append(p_i)
        if j < num_steps:
            tgt_in[:, j] = pick(p_i)[:, 0] if forced_tokens is None else forced_tokens[:, i]
    logits = torch.cat(logits, dim=1)
    if taps is not None:
        taps["ar_logits"] = logits
        taps["ar_tokens"] = tgt_in.clone()
    query_mask[torch.triu(torch.ones(num_steps, num_steps, dtype=torch.bool), 2)] = 0
    bos = torch.full((bs, 1), parseq.bos_id, dtype=torch.long)
    tgt_in = torch.cat([bos, pick(logits[:, :-1])], dim=1)
    if forced_tokens is not None:
        tgt_in = torch.cat([bos, forced_tokens], dim=1)
    tgt_padding_mask = (tgt_in == parseq.eos_id).int().cumsum(-1) > 0
    tgt_out = parseq.decode(tgt_in, memory, tgt_padding_mask, tgt_query=pos_queries,
                            tgt_query_mask=query_mask[:, : tgt_in.shape[1]])
    return parseq.head(tgt_out)
