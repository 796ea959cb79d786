#!/usr/bin/env python
"""Kernel time of one PARSeq-base encoder block's LN1 + qkv + attention: the two-launch pair (LayerNorm-consumer qkv GEMM,
then k_attn_enc<true>) against k_enc_qkv_attn, at 2400 and 9600 crops, arms alternating, CUDA events around `--iters`
launches per sample.  The inputs (hi 0.24 / 0.94 GB) exceed the 126 MB L2.  Reports the median microseconds per block
and each arm's share of the two rooflines: tensor (the qkv projection's FLOPs plus the attention's 4 x 128 x 128 x 64
per crop-head, over 2250 TFLOP/s dense BF16) and HBM (the bytes each arm must move at 7.7 TB/s: the pair writes and
reads qkv, the fused kernel does not), both data-sheet figures for a 1000 W card.  Also checks the outputs are identical.

    python tools/qkv_attn_bench.py [--crops 2400 9600] [--iters 20] [--samples 7] [--out FILE.json]
"""
import argparse
import json
import statistics
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

PEAK_TF, PEAK_BW = 2250e12, 7.7e12


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True, timeout=30).stdout.strip()
    return [s.strip() for s in out.split(",")]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--crops", type=int, nargs="+", default=[2400, 9600])
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--samples", type=int, default=7)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()

    import torch

    from tuatara_b200 import _native

    lib = _native.lib()
    check = _native.check
    D, heads, parts = 384, 6, 2
    g = torch.Generator(device="cuda").manual_seed(0)
    Wf = (torch.randn(3 * D, D, device="cuda", generator=g) / D ** 0.5).to(torch.bfloat16)
    c0 = torch.randn(3 * D, device="cuda", generator=g) * 0.02
    c1 = Wf.float().sum(1).contiguous()
    res = {"gpu": gpu_info(), "D": D, "iters": a.iters, "samples": a.samples, "sizes": []}
    for crops in a.crops:
        M = crops * 128
        x = torch.randn(M, D, device="cuda", generator=g) * 1.5 + 0.3
        hi = x.to(torch.bfloat16)
        xs = x.reshape(M, parts, D // parts)
        stats = torch.stack([xs.sum(2), (xs * xs).sum(2)], dim=2).contiguous()
        del x, xs
        qkv = torch.empty(M, 3 * D, dtype=torch.bfloat16, device="cuda")
        att_a = torch.empty(M, D, dtype=torch.bfloat16, device="cuda")
        att_b = torch.empty_like(att_a)

        def pair():
            check(lib.tt_linear_ln_dev(hi.data_ptr(), M, D, Wf.data_ptr(), c0.data_ptr(), c1.data_ptr(), 3 * D, stats.data_ptr(), parts,
                                       1e-6, qkv.data_ptr(), None), "tt_linear_ln_dev")
            check(lib.tt_attn_enc_dev(qkv.data_ptr(), att_a.data_ptr(), crops, D, heads, 1, None), "tt_attn_enc_dev")

        def fused():
            check(lib.tt_enc_qkv_attn_dev(hi.data_ptr(), stats.data_ptr(), parts, Wf.data_ptr(), c0.data_ptr(), c1.data_ptr(),
                                          att_b.data_ptr(), crops, D, heads, 1e-6, None), "tt_enc_qkv_attn_dev")

        arms = {"two_launch": pair, "fused": fused}
        for f in arms.values():   # warm-up: module load, tensor maps, smem attributes
            f()
        torch.cuda.synchronize()
        identical = bool(torch.equal(att_a.view(torch.int16), att_b.view(torch.int16)))
        times = {k: [] for k in arms}
        for _ in range(a.samples):
            for k, f in arms.items():
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(a.iters):
                    f()
                e1.record()
                torch.cuda.synchronize()
                times[k].append(e0.elapsed_time(e1) * 1e3 / a.iters)
        flops = 2.0 * M * D * 3 * D + 4.0 * crops * heads * 128 * 128 * 64
        bytes_ = {"two_launch": M * D * 2 + M * parts * 8 + M * 3 * D * 2 * 2 + M * D * 2, "fused": M * D * 2 + M * parts * 8 + M * D * 2}
        row = {"crops": crops, "identical": identical}
        for k in arms:
            us = statistics.median(times[k])
            row[k] = {"us_median": round(us, 1), "us_min": round(min(times[k]), 1), "us_max": round(max(times[k]), 1),
                      "tensor_roofline_frac": round(flops / PEAK_TF / (us * 1e-6), 3),
                      "hbm_roofline_frac": round(bytes_[k] / PEAK_BW / (us * 1e-6), 3), "hbm_bytes": bytes_[k]}
        row["speedup"] = round(row["two_launch"]["us_median"] / row["fused"]["us_median"], 3)
        res["sizes"].append(row)
        print(json.dumps(row), flush=True)
        del hi, stats, qkv, att_a, att_b
        torch.cuda.empty_cache()
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(json.dumps(res, indent=1) + "\n")
    print(json.dumps(res))


if __name__ == "__main__":
    main()
