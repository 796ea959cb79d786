"""tests/attn_ref.py against the oracle's own attention modules and masks, in float64.

The encoder reference must reproduce timm's Attention (oracle/models.py) between its qkv and proj layers; the decoder
references must reproduce nn.MultiheadAttention between its in_proj and out_proj, with the masks built exactly as
PARSeq.forward builds them.  The kernel tests trust attn_ref only because of this file."""
import pytest
import torch

import attn_ref as R
from oracle.models import Attention, DecoderLayer

VARIANTS = [(384, 6, 12), (192, 3, 6)]   # (D, encoder heads, decoder heads): PARSeq-base, PARSeq-tiny
EOS, BOS, N_TOK = 0, 95, 97               # the oracle's ids


def _close(a, b):
    err = float((a - b).abs().max())
    assert err <= 1e-10 * max(1.0, float(b.abs().max())), err


@pytest.mark.parametrize("D,enc_heads,dec_heads", VARIANTS)
def test_encoder_reference_matches_timm_attention(D, enc_heads, dec_heads):
    torch.manual_seed(0)
    m = Attention(D, enc_heads).double().eval()
    x = torch.randn(3, R.MEM_KEYS, D, dtype=torch.float64)
    with torch.no_grad():
        want = m(x)
        qkv = m.qkv(x).reshape(-1, 3 * D)
        got = m.proj(R.enc_attention(qkv, enc_heads).out.reshape(3, R.MEM_KEYS, D))
    _close(got, want)


def _mha(D, heads):
    torch.manual_seed(1)
    return DecoderLayer(D, heads, 4 * D).double().eval()


def _proj(mha, x, part):
    D = mha.embed_dim
    w, b = mha.in_proj_weight[part * D:(part + 1) * D], mha.in_proj_bias[part * D:(part + 1) * D]
    return x @ w.t() + b


def _tokens(L):
    """One crop per refinement case: first EOS among tokens[1..] at 1, 2, 13, L - 1, none, and EOS at 5 and 9."""
    g = torch.Generator().manual_seed(2)
    t = torch.randint(1, 95, (6, L), generator=g)
    t[:, 0] = BOS
    for c, e in enumerate([1, 2, 13, L - 1]):
        t[c, e] = EOS
    t[5, 5] = EOS
    t[5, 9] = EOS
    return t


@pytest.mark.parametrize("D,enc_heads,dec_heads", VARIANTS)
@pytest.mark.parametrize("refine", [False, True])
def test_self_attention_reference_matches_oracle(D, enc_heads, dec_heads, refine):
    L = 26
    layer = _mha(D, dec_heads)
    mha = layer.self_attn
    g = torch.Generator().manual_seed(3)
    q_in = torch.randn(L, D, generator=g, dtype=torch.float64)             # query stream input by position
    c_in = torch.randn(L, N_TOK, D, generator=g, dtype=torch.float64)      # content stream input by (position, token)
    tokens = _tokens(L)
    n = tokens.shape[0]
    with torch.no_grad():
        q_table = _proj(mha, q_in, 0)
        kv_table = torch.cat([_proj(mha, c_in, 1), _proj(mha, c_in, 2)], dim=-1)
        content = c_in[torch.arange(L)[None, :], tokens]                   # [n, L, D]
        # the oracle's masks (PARSeq.forward)
        query_mask = torch.triu(torch.full((L, L), float("-inf"), dtype=torch.float64), 1)
        if refine:
            query_mask[torch.triu(torch.ones(L, L, dtype=torch.bool), 2)] = 0
            pad = (tokens == EOS).int().cumsum(-1) > 0
            want = mha(q_in.expand(n, L, D), content, content, attn_mask=query_mask, key_padding_mask=pad,
                       need_weights=False)[0]
            got = R.dec_self_attention(q_table, kv_table, tokens, 0, L, True, EOS, dec_heads).out
            _close(mha.out_proj(got).reshape(n, L, D), want)
        else:
            for i in [0, 1, 2, 3, 15, 24, 25]:
                j = i + 1
                want = mha(q_in[i:j].expand(n, 1, D), content[:, :j], content[:, :j], attn_mask=query_mask[i:j, :j],
                           need_weights=False)[0]
                got = R.dec_self_attention(q_table, kv_table, tokens, i, 1, False, EOS, dec_heads).out
                _close(mha.out_proj(got).reshape(n, 1, D), want)


@pytest.mark.parametrize("D,enc_heads,dec_heads", VARIANTS)
def test_cross_attention_reference_matches_oracle(D, enc_heads, dec_heads):
    mha = _mha(D, dec_heads).cross_attn
    g = torch.Generator().manual_seed(4)
    n, np_ = 3, 26
    x = torch.randn(n, np_, D, generator=g, dtype=torch.float64)
    memory = torch.randn(n, R.MEM_KEYS, D, generator=g, dtype=torch.float64)
    with torch.no_grad():
        want = mha(x, memory, memory, need_weights=False)[0]
        mem_kv = torch.cat([_proj(mha, memory, 1), _proj(mha, memory, 2)], dim=-1)
        got = R.dec_cross_attention(_proj(mha, x, 0), mem_kv, dec_heads).out
        _close(mha.out_proj(got).reshape(n, np_, D), want)


def test_refinement_mask_rule():
    """The mask restated on small cases by hand: cloze key p + 1, and nothing from the first EOS of tokens[1..] on."""
    t = torch.tensor([[BOS, 7, EOS, 8, EOS], [BOS, 7, 8, 9, 10], [EOS, 7, 8, EOS, 9]])
    a = R.self_allowed(t, 0, 5, True, EOS)
    assert a[0].tolist() == [[True, False, False, False, False], [True, True, False, False, False],
                             [True, True, False, False, False], [True, True, False, False, False],
                             [True, True, False, False, False]]
    assert a[1, 2].tolist() == [True, True, True, False, True]
    assert a[1, 4].tolist() == [True, True, True, True, True]
    assert a[2, 0].tolist() == [True, False, True, False, False]   # tokens[0] is never an EOS key for the rule
    assert R.self_allowed(t, 2, 1, False, EOS)[:, 0].tolist() == [[True, True, True, False, False]] * 3
