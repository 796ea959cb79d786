"""k_enc_qkv_attn (enc_qkv_attn.cu): the LayerNorm-folded qkv projection and the encoder self attention in one kernel.

Its output must be bit for bit the two-launch path it replaces on the same inputs: the qkv GEMM with the LayerNorm
consumer epilogue (tt_linear_ln_dev) followed by k_attn_enc<true> (tt_attn_enc_dev).  The kernel issues the projection's
k-steps in the GEMM's order, applies the same epilogue arithmetic and calls the same softmax code, so any difference is a
bug.  The output must also stay within the float64 bound of tests/attn_ref.py on that bf16 qkv.  The weights put the
heads in the score regimes test_attention_gpu.py checks for: flat, random-init-like and peaked rows, some with keys
flushed below the fp32 exp range.  Rows past the last crop carry a NaN canary the launch must leave alone."""
import math

import pytest
import torch

import attn_ref as R
from test_attention_gpu import _assert_canary, _assert_within, _bound, _canary, _regimes_reached

pytestmark = pytest.mark.gpu

# scaled score std per head (q and k rows scaled by its square root): flat, random-init-like, peaked, peaked with keys
# far below the maximum
SCORE_STD = {6: [0.01, 1.0, 10.0, 40.0, 0.01, 4.0], 3: [0.01, 10.0, 40.0]}


def _check(rc, what):
    from tuatara_b200._native import check

    check(rc, what)
    torch.cuda.synchronize()


def _inputs(crops, D, heads, parts, seed):
    """hi = bf16(x) [crops*128][D], stats [rows][parts][2] of x, folded weights Wf [3D][D] and c0, c1 [3D]."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    M = crops * 128
    x = torch.randn(M, D, device="cuda", generator=g) * 1.5 + 0.3
    gamma = 1.0 + 0.2 * (torch.rand(D, device="cuda", generator=g) - 0.5)
    beta = 0.05 * torch.randn(D, device="cuda", generator=g)
    W = torch.randn(3 * D, D, device="cuda", generator=g) / math.sqrt(D)
    s = torch.tensor(SCORE_STD[heads], device="cuda").sqrt().repeat_interleave(64)
    W[:D] *= s[:, None]
    W[D:2 * D] *= s[:, None]
    b = 0.02 * torch.randn(3 * D, device="cuda", generator=g)
    Wf = (W * gamma[None, :]).to(torch.bfloat16)
    c1 = Wf.double().sum(1).float()
    c0 = (b.double() + W.double() @ beta.double()).float()
    xs = x.reshape(M, parts, D // parts)
    stats = torch.stack([xs.sum(2), (xs * xs).sum(2)], dim=2)
    return x.to(torch.bfloat16).contiguous(), stats.contiguous(), Wf.contiguous(), c0.contiguous(), c1.contiguous()


def _run(native_lib, crops, D, heads, parts, seed):
    xh, stats, Wf, c0, c1 = _inputs(crops, D, heads, parts, seed)
    rows = crops * 128
    qkv = torch.empty(rows, 3 * D, dtype=torch.bfloat16, device="cuda")
    _check(native_lib.tt_linear_ln_dev(xh.data_ptr(), rows, D, Wf.data_ptr(), c0.data_ptr(), c1.data_ptr(), 3 * D, stats.data_ptr(),
                                       parts, 1e-6, qkv.data_ptr(), None), "tt_linear_ln_dev")
    ref = _canary(rows + 128, D)
    _check(native_lib.tt_attn_enc_dev(qkv.data_ptr(), ref.data_ptr(), crops, D, heads, 1, None), "tt_attn_enc_dev")
    out = _canary(rows + 128, D)
    _check(native_lib.tt_enc_qkv_attn_dev(xh.data_ptr(), stats.data_ptr(), parts, Wf.data_ptr(), c0.data_ptr(), c1.data_ptr(),
                                          out.data_ptr(), crops, D, heads, 1e-6, None), "tt_enc_qkv_attn_dev")
    what = f"k_enc_qkv_attn D{D} crops{crops} parts{parts}"
    _assert_canary(out[rows:], what)
    same = out[:rows].view(torch.int16) == ref[:rows].view(torch.int16)
    if not bool(same.all()):
        r, c = (~same).nonzero()[0].tolist()
        raise AssertionError(f"{what}: {int((~same).sum())}/{same.numel()} elements differ from the two-launch path; first at "
                             f"row {r} col {c}: {float(out[r, c])} vs {float(ref[r, c])}")
    return qkv, out, what


@pytest.mark.parametrize("D,heads", [(384, 6), (192, 3)])
@pytest.mark.parametrize("crops", [1, 7, 149, 300, 2400])
def test_enc_qkv_attn_matches_two_launches(native_lib, D, heads, crops):
    qkv, out, what = _run(native_lib, crops, D, heads, 2, seed=crops * 10 + heads)
    worst = 0.0
    for c0 in range(0, crops, 250):
        c1 = min(crops, c0 + 250)
        ref = R.enc_attention(qkv[c0 * R.MEM_KEYS:c1 * R.MEM_KEYS], heads)
        if crops >= 7 and c0 == 0:
            _regimes_reached(ref, what)
        bound = _bound(ref, 64, R.MEM_KEYS, p_bf16=True)
        worst = max(worst, _assert_within(out[c0 * R.MEM_KEYS:c1 * R.MEM_KEYS], ref, bound, f"{what} crops {c0}..{c1}"))
    print(f"{what}: worst err/bound over all crops {worst:.3g}")


@pytest.mark.parametrize("D,heads", [(384, 6), (192, 3)])
@pytest.mark.parametrize("parts", [1, 3, 4])
def test_enc_qkv_attn_layernorm_partials(native_lib, D, heads, parts):
    """every partial count a residual GEMM can leave (the patch embedding's included): the producer has <= 4 N tiles"""
    _run(native_lib, 149, D, heads, parts, seed=parts)
