"""Float64 restatement of PARSeq's attention operations, the reference the attention kernels are tested against.

Plain torch, no kernel code.  The mask rules are the oracle's (oracle/models.py, PARSeq.forward): the AR step p sees
the context keys 0..p (``query_mask = triu(-inf, 1)``); the refinement pass sees every key except p + 1 (the cloze
mask) and nothing from the first EOS on (``(tgt_in == eos).cumsum(-1) > 0``).  tests/test_attention_ref_cpu.py checks
these functions against the oracle's own modules, so a mistake here cannot hide the same mistake in a kernel.

Each function returns a ``Ref``: the output, and per output element the quantities the kernel error bound of
tests/test_attention_gpu.py is built from (all float64, same shape as ``out``):
  A      sum_j P_j |V_j|, over the allowed keys j (P: the reference probabilities)
  qk     scale * max_j sum_i |q_i k_ji| over the allowed keys j (the largest score magnitude an fp32 dot can reach)
  span   max_j (s_max - s_j) over the allowed keys j, scaled scores (the largest argument an exp() receives)
"""
from __future__ import annotations

from typing import NamedTuple

import torch

ENC_SCALE = 64 ** -0.5    # timm Attention: head_dim ** -0.5, head dim 64
DEC_SCALE = 32 ** -0.5    # nn.MultiheadAttention: head dim 32 (PARSeq-base 384 / 12, PARSeq-tiny 192 / 6)
MEM_KEYS = 128            # encoder tokens = decoder memory rows per crop


class Ref(NamedTuple):
    out: torch.Tensor
    A: torch.Tensor
    qk: torch.Tensor
    span: torch.Tensor


def attend(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, scale: float, allowed: torch.Tensor | None = None) -> Ref:
    """softmax(scale * q k^T, masked to `allowed`) v in float64.  q [..., Q, d], k / v [..., K, d], allowed bool
    broadcastable to [..., Q, K] (None: every key)."""
    q, k, v = q.double(), k.double(), v.double()
    s = (q @ k.transpose(-1, -2)) * scale
    qk = (q.abs() @ k.abs().transpose(-1, -2)) * scale
    if allowed is not None:
        allowed = allowed.expand_as(s)
        s = s.masked_fill(~allowed, float("-inf"))
        qk = qk.masked_fill(~allowed, 0.0)
    p = torch.softmax(s, dim=-1)
    smax = s.amax(dim=-1, keepdim=True)
    gap = smax - s
    if allowed is not None:
        gap = gap.masked_fill(~allowed, 0.0)
    d = v.shape[-1]
    out = p @ v
    return Ref(out, p @ v.abs(), qk.amax(dim=-1, keepdim=True).expand(*out.shape[:-1], d),
               gap.amax(dim=-1, keepdim=True).expand(*out.shape[:-1], d))


def _merge_heads(r: Ref, shape) -> Ref:
    """[n, heads, Q, dh] -> [n * Q, heads * dh] (the kernels' row-major output)."""
    return Ref(*(t.permute(0, 2, 1, 3).reshape(shape) for t in r))


def enc_attention(qkv: torch.Tensor, heads: int) -> Ref:
    """timm Attention without its projections: qkv [crops*128][3D] (q | k | v, head-major inside each, head dim 64)
    -> [crops*128][D]."""
    rows, D3 = qkv.shape
    D = D3 // 3
    n = rows // MEM_KEYS
    x = qkv.double().reshape(n, MEM_KEYS, 3, heads, D // heads).permute(2, 0, 3, 1, 4)
    return _merge_heads(attend(x[0], x[1], x[2], ENC_SCALE), (rows, D))


def first_eos(tokens: torch.Tensor, eos_id: int) -> torch.Tensor:
    """Index of the first EOS among tokens[:, 1:] per crop (L when there is none)."""
    L = tokens.shape[1]
    e = tokens[:, 1:] == eos_id
    return torch.where(e.any(dim=1), e.int().argmax(dim=1) + 1, torch.full_like(tokens[:, 0], L))


def self_allowed(tokens: torch.Tensor, p0: int, np_: int, refine: bool, eos_id: int) -> torch.Tensor:
    """bool [n, np, L]: may query position p0 + i of crop c attend to key j?"""
    n, L = tokens.shape
    j = torch.arange(L, device=tokens.device)[None, None, :]
    p = torch.arange(p0, p0 + np_, device=tokens.device)[None, :, None]
    if not refine:
        return (j <= p).expand(n, np_, L)
    return (j != p + 1) & (j < first_eos(tokens, eos_id)[:, None, None])


def dec_self_attention(q_table: torch.Tensor, kv_table: torch.Tensor, tokens: torch.Tensor, p0: int, np_: int,
                       refine: bool, eos_id: int, heads: int, q_bf16: bool = False) -> Ref:
    """nn.MultiheadAttention core of the query stream over the content stream: query p = q_table[p] (fp32 [L][D], already
    projected; rounded to bf16 first when q_bf16), key / value j of crop c = row (j, tokens[c][j]) of kv_table
    ([L][n_tok][2D], K | V).  -> [n * np][D], crop-major."""
    n, L = tokens.shape
    D = q_table.shape[1]
    dh = D // heads
    kv = kv_table.double()[torch.arange(L, device=tokens.device)[None, :], tokens.long()]   # [n, L, 2D]
    k = kv[..., :D].reshape(n, L, heads, dh).transpose(1, 2)
    v = kv[..., D:].reshape(n, L, heads, dh).transpose(1, 2)
    q = q_table[p0:p0 + np_]
    q = (q.bfloat16() if q_bf16 else q).double().reshape(1, np_, heads, dh).transpose(1, 2)
    allowed = self_allowed(tokens, p0, np_, refine, eos_id)[:, None]
    return _merge_heads(attend(q, k, v, DEC_SCALE, allowed), (n * np_, D))


def dec_cross_attention(q: torch.Tensor, mem_kv: torch.Tensor, heads: int) -> Ref:
    """Cross attention over all 128 memory rows, no mask: q [n][np][D], mem_kv [n][128][2D] (K | V) -> [n * np][D]."""
    n, np_, D = q.shape
    dh = D // heads
    m = mem_kv.double()
    k = m[..., :D].reshape(n, MEM_KEYS, heads, dh).transpose(1, 2)
    v = m[..., D:].reshape(n, MEM_KEYS, heads, dh).transpose(1, 2)
    qh = q.double().reshape(n, np_, heads, dh).transpose(1, 2)
    return _merge_heads(attend(qh, k, v, DEC_SCALE), (n * np_, D))
