"""Every attention kernel against the float64 reference of tests/attn_ref.py, through the launchers the engine calls.

Kernels: k_attn_enc<true/false>, k_dec_score_table, k_dec_self_attn_ar<12/6>, k_dec_self_attn, k_dec_attn_refine<32, true>
and <128, false>, k_dec_cross_attn<384/192>.

Error bound, per output element, from the reference's own data (attn_ref.Ref: A = sum_j P_j |V_j|, qk = scale *
max_j sum_i |q_i k_ji|, span = the largest scaled score gap to the row maximum, all over the allowed keys):

    |out - ref| <= 2^-8 |ref| + (1 + 2^-8) (p_bf16 + 2 n_keys 2^-24 + 2 ds) A
    ds = qk (K 2^-24 [+ 2^-8 where the kernel rounds q to bf16]) + (2 + 1.2 span) 2^-23

  2^-8 |ref|          bf16 rounding of the output; (1 + 2^-8) because it rounds the kernel's value, not the reference
  p_bf16 = 2^-8       P rounded to bf16 for the tensor-core P V (k_attn_enc, k_dec_attn_refine); 0 where P stays fp32
  2 n_keys 2^-24      fp32 accumulation of the exponentials' sum and of P V over n_keys terms
  2 ds                a score error ds moves the output by at most 2 ds A to first order: fp32 accumulation of the
                      K-term dot products (K = 64 encoder, 32 decoder), q's bf16 rounding, and the exp evaluation
                      (__expf / ex2.approx: within 2 + 1.2 |x| ulp for an argument x)

Inputs are where the kernels go wrong: flat, random-init-like and peaked scores (a hot key of scaled score +-40, so
some rows are near one-hot and others have keys far enough below the maximum to flush), exact two-way ties, the maximum
at key 0 and at the last key, V spanning 1e-3..1e2 with a head-dependent sign balance and one all-zero head.  Every head
gets its own statistics, so reading a neighbour's head is a large error.  Masked self-attention keys are poisoned: a
key behind the first EOS, or behind the AR position, scores +40 above the rest with V = +-1e4; the cloze key p + 1 of
query p scores +40 above the rest.  Output rows a launch must not write carry a NaN canary."""
import math

import pytest
import torch

import attn_ref as R

pytestmark = pytest.mark.gpu

EOS, POISON, BOS, N_TOK = 0, 1, 95, 97   # decoder token ids: POISON is any token a kernel must never attend to
HOT = 40.0                               # scaled score of a hot / poisoned key


def _ptr(t):
    return None if t is None else t.data_ptr()


def _call(rc, what):
    from tuatara_b200._native import check

    check(rc, what)
    torch.cuda.synchronize()


def _bound(ref, k_dot, n_keys, q_bf16=False, p_bf16=False):
    ds = ref.qk * (k_dot * 2.0 ** -24 + (2.0 ** -8 if q_bf16 else 0.0)) + (2.0 + 1.2 * ref.span) * 2.0 ** -23
    # (1 + 2^-8): the output rounding acts on the kernel's fp32 value, which carries the other errors
    return 2.0 ** -8 * ref.out.abs() + (1 + 2.0 ** -8) * ((2.0 ** -8 if p_bf16 else 0.0) + 2 * n_keys * 2.0 ** -24 + 2 * ds) * ref.A


def _assert_within(out, ref, bound, what):
    """out (any float dtype) vs ref.out elementwise against `bound`; prints the worst err / bound."""
    out = out.double()
    assert torch.isfinite(out).all(), f"{what}: non-finite output (an unwritten row, or a NaN from the kernel)"
    err = (out - ref.out).abs()
    bad = err > bound
    zero = bound == 0
    ratio = float((err[~zero] / bound[~zero]).max()) if (~zero).any() else 0.0
    print(f"{what}: worst err/bound {ratio:.3g}")
    if bad.any():
        r, c = bad.nonzero()[0].tolist()
        raise AssertionError(f"{what}: {int(bad.sum())}/{bad.numel()} elements out of bound (worst err/bound {ratio:.3g}); "
                             f"first at row {r} col {c}: out {float(out[r, c]):.6g} ref {float(ref.out[r, c]):.6g} "
                             f"bound {float(bound[r, c]):.3g}")
    return ratio


def _canary(rows, D):
    return torch.full((rows, D), float("nan"), dtype=torch.bfloat16, device="cuda")


def _assert_canary(t, what):
    assert torch.isnan(t.float()).all(), f"{what}: a row the launch must not write was written"


# ------------------------------------------------------------------------------------------------ input generators
def _v(g, G, heads, nk, dh):
    """V [G = n * heads][nk][dh]: magnitudes 1e-3..1e2, sign balance set by the head, the last head all zero."""
    h = torch.arange(G, device="cuda") % heads
    mag = 10.0 ** (torch.rand(G, nk, dh, device="cuda", generator=g) * 5 - 3)
    pos = (h + 1).double() / (heads + 1)
    sign = torch.where(torch.rand(G, nk, dh, device="cuda", generator=g) < pos[:, None, None].float(), 1.0, -1.0)
    v = mag * sign
    v[h == heads - 1] = 0
    return v


def _qk(g, n, heads, nq, nk, dh):
    """q [n*heads][nq][dh], k [n*heads][nk][dh] in a score regime chosen per (crop, head): flat, random-init-like,
    peaked (hot key at 0 or the last key), an exact two-way tie of hot keys, and a hot key 4x as strong (rows with
    keys far below the maximum).  Scaled scores: scale * q.k with scale * sqrt(dh) = 1."""
    G = n * heads
    crop = torch.arange(G, device="cuda") // heads
    regime = (torch.arange(G, device="cuda") % heads + crop) % 5
    sig = torch.tensor([0.05, 1.0, 1.0, 1.0, 1.0], device="cuda")[regime]
    lam = torch.tensor([0.0, 0.0, HOT, HOT, 4 * HOT], device="cuda")[regime]
    q = torch.randn(G, nq, dh, device="cuda", generator=g) * sig[:, None, None]
    k = torch.randn(G, nk, dh, device="cuda", generator=g) * sig[:, None, None]
    u = torch.randn(G, dh, device="cuda", generator=g)
    hot = (lam * math.sqrt(dh))[:, None] * u / u.norm(dim=1, keepdim=True)   # scale * q.hot ~ N(0, lam^2)
    t1 = torch.where(crop % 2 == 0, 0, nk - 1)
    t1 = torch.where(regime == 4, crop % nk, t1)
    t2 = torch.where(regime == 3, nk - 1 - t1 - (crop % 7), t1).clamp(0, nk - 1)
    idx = torch.arange(G, device="cuda")
    has = lam > 0
    k[idx[has], t1[has]] = hot[has]
    k[idx[has], t2[has]] = hot[has]
    return q, k


def _regimes_reached(ref, what):
    """The inputs must really contain near one-hot rows and rows with flushed keys (span beyond exp's fp32 range)."""
    assert float(ref.span.max()) > 104, f"{what}: no row with keys below the fp32 exp range"
    assert float((ref.span >= 30).double().mean()) > 0.1, f"{what}: too few peaked rows"
    assert float((ref.span < 1).double().mean()) > 0.05, f"{what}: too few flat rows"


# ------------------------------------------------------------------------------------------------------ encoder
@pytest.mark.parametrize("D,heads", [(384, 6), (192, 3)])
@pytest.mark.parametrize("onepass", [1, 0])
@pytest.mark.parametrize("crops", [1, 7, 300, 2000])
def test_attn_enc(native_lib, D, heads, onepass, crops):
    g = torch.Generator(device="cuda").manual_seed(crops * 10 + heads)
    q, k = _qk(g, crops, heads, R.MEM_KEYS, R.MEM_KEYS, 64)
    v = _v(g, crops * heads, heads, R.MEM_KEYS, 64)
    # timm layout: [crop][token][q|k|v][head][64]
    qkv = torch.stack([t.reshape(crops, heads, R.MEM_KEYS, 64).transpose(1, 2) for t in (q, k, v)], dim=2)
    qkv = qkv.reshape(crops * R.MEM_KEYS, 3 * D).to(torch.bfloat16).contiguous()
    out = _canary((crops + 1) * R.MEM_KEYS, D)
    _call(native_lib.tt_attn_enc_dev(_ptr(qkv), _ptr(out), crops, D, heads, onepass, None), "tt_attn_enc_dev")
    what = f"k_attn_enc<{bool(onepass)}> D{D} crops{crops}"
    rows = crops * R.MEM_KEYS
    _assert_canary(out[rows:], what)
    worst = 0.0
    for c0 in range(0, crops, 250):
        c1 = min(crops, c0 + 250)
        ref = R.enc_attention(qkv[c0 * R.MEM_KEYS:c1 * R.MEM_KEYS], heads)
        if crops >= 7 and c0 == 0:
            _regimes_reached(ref, what)
        bound = _bound(ref, 64, R.MEM_KEYS, p_bf16=True)
        worst = max(worst, _assert_within(out[c0 * R.MEM_KEYS:c1 * R.MEM_KEYS], ref, bound, f"{what} crops {c0}..{c1}"))
    print(f"{what}: worst err/bound over all crops {worst:.3g}")


# ------------------------------------------------------------------------------------------- decoder self attention
def _dec_tables(g, L, D, heads):
    """q_table fp32 [L][D] and kv_table bf16 [L][N_TOK][2D] with per-head statistics, the cloze key and the poison.
    Head dims: 0..30 carry the cloze term (query p has +15 on dim p, key (j, normal token) +15 on dim j - 1, so query p
    scores +225 / sqrt(32) ~ +40 on key p + 1 and nothing extra elsewhere); dim 31 the poison (every query +15, the
    EOS and POISON rows +15)."""
    dh = 32
    sig_q = torch.tensor([0.1, 0.5, 1.0, 2.0], device="cuda").repeat(heads)[:heads]
    sig_k = torch.tensor([1.0, 0.5, 0.25, 0.1], device="cuda").repeat(heads)[:heads]
    big = math.sqrt(HOT / R.DEC_SCALE)   # ~15: big * big * scale = HOT
    q = torch.randn(L, heads, dh, device="cuda", generator=g) * sig_q[None, :, None]
    p = torch.arange(min(L, 31), device="cuda")
    q[p, :, p] += big
    q[:, :, 31] += big
    k = torch.randn(L, N_TOK, heads, dh, device="cuda", generator=g) * sig_k[None, None, :, None]
    j = torch.arange(1, L, device="cuda")
    k[j, 2:, :, (j - 1).clamp(max=30)] += big
    k[:, [EOS, POISON], :, 31] += big
    v = _v(g, heads, heads, L * N_TOK, dh).reshape(heads, L, N_TOK, dh).permute(1, 2, 0, 3).contiguous()
    v[:, [EOS, POISON]] = torch.where(torch.rand(L, 2, heads, dh, device="cuda", generator=g) < 0.5, 1e4, -1e4)
    q_table = q.reshape(L, D).float().contiguous()
    kv_table = torch.cat([k.reshape(L, N_TOK, D), v.reshape(L, N_TOK, D)], dim=-1).to(torch.bfloat16).contiguous()
    return q_table, kv_table


def _ar_tokens(g, n, L, p):
    """Context tokens 0..p ordinary (BOS first), every later position POISON (an AR step must not read it)."""
    t = torch.randint(2, N_TOK, (n, L), device="cuda", generator=g, dtype=torch.int32)
    t[:, 0] = BOS
    t[:, p + 1:] = POISON
    return t.contiguous()


def _refine_tokens(g, n, L):
    """Crop c cycles through: first EOS at 1, 2, 13, 25 (L - 1 when shorter), L - 1, no EOS, and EOS at 5, 9 and 20 with
    ordinary tokens between.  After a lone EOS the rest is POISON."""
    t = torch.randint(2, N_TOK, (n, L), device="cuda", generator=g, dtype=torch.int32)
    t[:, 0] = BOS
    for c in range(n):
        kind = c % 7
        if kind < 5:
            e = [1, 2, 13, 25, L - 1][kind]
            e = min(e, L - 1)
            t[c, e] = EOS
            t[c, e + 1:] = POISON
        elif kind == 6:
            for e in (5, 9, 20):
                if e < L:
                    t[c, e] = EOS
    return t.contiguous()


def _active_cases(n):
    """(name, active list or None, n_act): identity, a permutation, a sparse subset, nothing live."""
    perm = torch.randperm(n, generator=torch.Generator().manual_seed(n))
    sparse = torch.arange(1, n, 3)
    return [("identity", None, n), ("permutation", perm, n), ("sparse", sparse, len(sparse)), ("empty", perm, 0)]


def _score_table(native_lib, q_table, kv_table, L, D, heads):
    sc = torch.full((L, L, N_TOK, heads), float("nan"), device="cuda")
    _call(native_lib.tt_dec_score_table_dev(_ptr(q_table), _ptr(kv_table), L, N_TOK, D, heads, _ptr(sc), None),
           "tt_dec_score_table_dev")
    return sc


@pytest.mark.parametrize("D,heads", [(384, 12), (192, 6)])
def test_dec_score_table(native_lib, D, heads):
    L = 26
    q_table, kv_table = _dec_tables(torch.Generator(device="cuda").manual_seed(heads), L, D, heads)
    sc = _score_table(native_lib, q_table, kv_table, L, D, heads)
    q = q_table.double().reshape(L, 1, 1, heads, 32)
    k = kv_table[..., :D].double().reshape(1, L, N_TOK, heads, 32)
    ref = (q * k).sum(-1) * R.DEC_SCALE
    bound = (q.abs() * k.abs()).sum(-1) * R.DEC_SCALE * 33 * 2.0 ** -24   # 32-term fp32 dot, then the scale multiply
    err = (sc.double() - ref).abs()
    print(f"k_dec_score_table D{D}: worst err/bound {float((err / bound).max()):.3g}")
    assert (err <= bound).all()


def _run_self(native_lib, n, D, heads, L, p0, np_, refine, q_table, sc, kv_table, tokens, active=None, n_act=None,
              extra=8):
    rows = n * np_
    out = _canary(rows + extra, D)
    act = None if active is None else active.to(device="cuda", dtype=torch.int32)
    na = None if n_act is None else torch.tensor([n_act], device="cuda", dtype=torch.int32)
    _call(native_lib.tt_dec_self_attn_dev(n, D, heads, L, p0, np_, refine, _ptr(act), _ptr(na), _ptr(q_table),
                                                      _ptr(sc), _ptr(kv_table), _ptr(tokens), EOS, N_TOK, _ptr(out), None),
           "tt_dec_self_attn_dev")
    return out


@pytest.mark.parametrize("D,heads", [(384, 12), (192, 6)])
def test_dec_self_attn_ar(native_lib, D, heads):
    """k_dec_self_attn_ar<heads> at the AR steps p (the j0 += 4 tail included), under every kind of early-exit list."""
    L, n = 26, 300
    g = torch.Generator(device="cuda").manual_seed(100 + heads)
    q_table, kv_table = _dec_tables(g, L, D, heads)
    sc = _score_table(native_lib, q_table, kv_table, L, D, heads)
    for p in [0, 1, 2, 3, 15, 24, 25]:
        tokens = _ar_tokens(g, n, L, p)
        ref = R.dec_self_attention(q_table, kv_table, tokens, p, 1, False, EOS, heads)
        bound = _bound(ref, 32, p + 1)
        for name, active, n_act in _active_cases(n):
            what = f"k_dec_self_attn_ar<{heads}> p{p} {name}"
            out = _run_self(native_lib, n, D, heads, L, p, 1, 0, q_table, sc, kv_table, tokens,
                            active, None if active is None else n_act)
            crops = torch.arange(n) if active is None else active[:n_act]
            _assert_canary(out[n_act:], what)
            if n_act:
                c = crops.cuda()
                _assert_within(out[:n_act], R.Ref(*(t[c] for t in ref)), bound[c], what)


@pytest.mark.parametrize("D,heads", [(384, 12), (192, 6)])
def test_dec_self_attn_ar_bits_match_direct(native_lib, D, heads):
    """The score table path and k_dec_self_attn (no table) sum in the same order: identical bits at every AR step."""
    L, n = 26, 300
    g = torch.Generator(device="cuda").manual_seed(200 + heads)
    q_table, kv_table = _dec_tables(g, L, D, heads)
    sc = _score_table(native_lib, q_table, kv_table, L, D, heads)
    perm = torch.randperm(n, generator=torch.Generator().manual_seed(3))
    for p in range(L):
        tokens = _ar_tokens(g, n, L, p)
        direct = _run_self(native_lib, n, D, heads, L, p, 1, 0, q_table, None, kv_table, tokens)
        table = _run_self(native_lib, n, D, heads, L, p, 1, 0, q_table, sc, kv_table, tokens)
        assert torch.equal(direct[:n].view(torch.int16), table[:n].view(torch.int16)), f"step {p}: bits differ"
        listed = _run_self(native_lib, n, D, heads, L, p, 1, 0, q_table, sc, kv_table, tokens, perm, n)
        assert torch.equal(direct[perm.cuda()].view(torch.int16), listed[:n].view(torch.int16)), f"step {p} listed"


@pytest.mark.parametrize("D,heads,L,p0,np_", [
    (384, 12, 26, 0, 26),   # k_dec_attn_refine<32, true>: the product's refinement pass
    (384, 12, 17, 0, 17),
    (384, 12, 32, 0, 32),
    (192, 6, 26, 0, 26),    # k_dec_self_attn: PARSeq-tiny's refinement pass
    (192, 6, 32, 0, 32),
    (384, 12, 26, 3, 5),    # k_dec_self_attn with 12 heads (a partial refinement pass)
])
def test_dec_self_attn_refine(native_lib, D, heads, L, p0, np_):
    n = 70
    g = torch.Generator(device="cuda").manual_seed(300 + L + np_ + heads)
    q_table, kv_table = _dec_tables(g, L, D, heads)
    tokens = _refine_tokens(g, n, L)
    mma = D == 384 and p0 == 0 and np_ == L
    what = f"{'k_dec_attn_refine<32,true>' if mma else 'k_dec_self_attn'} D{D} L{L} p{p0}+{np_}"
    out = _run_self(native_lib, n, D, heads, L, p0, np_, 1, q_table, None, kv_table, tokens)
    _assert_canary(out[n * np_:], what)
    ref = R.dec_self_attention(q_table, kv_table, tokens, p0, np_, True, EOS, heads, q_bf16=mma)
    _assert_within(out[:n * np_], ref, _bound(ref, 32, L, q_bf16=mma, p_bf16=mma), what)


# ------------------------------------------------------------------------------------------ decoder cross attention
def _cross_inputs(g, n, np_, D, heads):
    q, k = _qk(g, n, heads, np_, R.MEM_KEYS, 32)
    v = _v(g, n * heads, heads, R.MEM_KEYS, 32)
    q = q.reshape(n, heads, np_, 32).transpose(1, 2).reshape(n, np_, D).to(torch.bfloat16).contiguous()
    kv = torch.cat([t.reshape(n, heads, R.MEM_KEYS, 32).transpose(1, 2).reshape(n, R.MEM_KEYS, D) for t in (k, v)], dim=-1)
    return q, kv.to(torch.bfloat16).contiguous()


def _run_cross(native_lib, n, D, heads, np_, q, mem_kv, active=None, n_act=None, extra=8):
    out = _canary(n * np_ + extra, D)
    act = None if active is None else active.to(device="cuda", dtype=torch.int32)
    na = None if n_act is None else torch.tensor([n_act], device="cuda", dtype=torch.int32)
    _call(native_lib.tt_dec_cross_attn_dev(n, D, heads, 26, 0, np_, _ptr(act), _ptr(na), _ptr(q), _ptr(mem_kv),
                                                       _ptr(out), None), "tt_dec_cross_attn_dev")
    return out


@pytest.mark.parametrize("D,heads", [(384, 12), (192, 6)])
@pytest.mark.parametrize("n", [300, 3000])
def test_dec_cross_attn_ar(native_lib, D, heads, n):
    """k_dec_cross_attn<D> for one AR step: q / out rows by slot, memory by crop.  3000 crops with 2999 live make the
    bounded grid's blocks walk several slots each."""
    g = torch.Generator(device="cuda").manual_seed(400 + n + heads)
    q, mem_kv = _cross_inputs(g, n, 1, D, heads)
    cases = _active_cases(n) if n == 300 else [("2999 of 3000", torch.randperm(n, generator=torch.Generator().manual_seed(9)), n - 1)]
    for name, active, n_act in cases:
        what = f"k_dec_cross_attn<{D}> n{n} {name}"
        crops = torch.arange(n) if active is None else active[:n_act]
        c = crops.cuda()
        # the query of slot s is row s: give slot s crop active[s]'s query so the reference is that crop's attention
        qs = torch.zeros_like(q)
        qs[:n_act] = q[c]
        out = _run_cross(native_lib, n, D, heads, 1, qs, mem_kv, active, None if active is None else n_act)
        _assert_canary(out[n_act:], what)
        if n_act:
            ref = R.dec_cross_attention(qs[:n_act], mem_kv[c], heads)
            if n == 3000:
                _regimes_reached(ref, what)
            _assert_within(out[:n_act], ref, _bound(ref, 32, R.MEM_KEYS), what)


@pytest.mark.parametrize("D,heads,np_", [(384, 12, 2), (384, 12, 17), (384, 12, 26), (384, 12, 32), (192, 6, 26)])
def test_dec_cross_attn_refine(native_lib, D, heads, np_):
    """The refinement pass's cross attention: k_dec_attn_refine<128, false> (PARSeq-base, partial m-tiles at 2 / 17 / 26)
    and k_dec_cross_attn<192> over np positions (PARSeq-tiny)."""
    n = 150
    g = torch.Generator(device="cuda").manual_seed(500 + np_ + heads)
    q, mem_kv = _cross_inputs(g, n, np_, D, heads)
    mma = D == 384
    what = f"{'k_dec_attn_refine<128,false>' if mma else 'k_dec_cross_attn<192>'} np{np_}"
    out = _run_cross(native_lib, n, D, heads, np_, q, mem_kv)
    _assert_canary(out[n * np_:], what)
    ref = R.dec_cross_attention(q, mem_kv, heads)
    _regimes_reached(ref, what)
    _assert_within(out[:n * np_], ref, _bound(ref, 32, R.MEM_KEYS, p_bf16=mma), what)
