#!/usr/bin/env python
"""Cost of per-word scores (tt_ocr_options.with_scores) on BASELINE's 512-page step: synthetic 1280 x 1280 pages with
their score-map overrides resident in HBM, built the way bench.py builds its headline step, through tt_ocr_pages_ex with
with_scores = 0 and 1.  The two arms alternate step by step on one engine (three execution slots, 32-page recognition
batches).  Reports pages/s, device-to-host bytes per step and kernel launches per step for each arm, and checks that
text and bbox are identical between the arms.

    python tools/scores_bench.py [--pages 512] [--steps 4] [--warmup 1] [--out FILE.json]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import time
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

WORDS = 300


def gpu_info():
    """Card name and power limit (read only)."""
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = [s.strip() for s in out.split(",")]
        return name, power
    except Exception:  # noqa: BLE001 - the numbers are still reported, without the card's name
        return "unknown", "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pages", type=int, default=512)
    ap.add_argument("--steps", type=int, default=4, help="timed steps per arm")
    ap.add_argument("--warmup", type=int, default=1, help="untimed steps per arm")
    ap.add_argument("--out", help="also write the JSON result here")
    args = ap.parse_args()

    import torch

    if not torch.cuda.is_available():
        raise SystemExit("scores_bench.py: no CUDA device (the library has no CPU fallback)")
    import tuatara_b200 as tb
    from tuatara_b200 import _native, synth, weights

    lib = tb.lib()
    tmp = tempfile.TemporaryDirectory(prefix="tuatara_scores_bench_")
    wdir = weights.export_random(Path(tmp.name) / "weights_seed0", seed=0)
    cfg = tb.default_config()
    cfg.max_batch_pages = 32
    cfg.slots_per_gpu = 3
    eng = tb.Engine(wdir, devices=[0], cfg=cfg)
    n = args.pages
    with ThreadPoolExecutor(min(16, os.cpu_count() or 4)) as ex:
        pages_np = list(ex.map(synth.synth_page, range(n)))
        maps_np = list(ex.map(synth.synth_score_maps, range(n)))
    pages = [torch.from_numpy(p).cuda() for p in pages_np]
    maps = [torch.from_numpy(m).cuda() for m in maps_np]
    arr = (_native.tt_image * n)(*[_native.tt_image(t.data_ptr(), t.shape[0], t.shape[1], 3, t.shape[1] * 3) for t in pages])
    ptrs = (C.c_void_p * n)(*[m.data_ptr() for m in maps])
    opts = {s: _native.tt_ocr_options(1, 1, ptrs, 0, s) for s in (0, 1)}

    def step(scores, keep=False):
        res = C.POINTER(_native.tt_result)()
        tb.check(lib.tt_ocr_pages_ex(eng._h, arr, n, C.byref(opts[scores]), C.byref(res)), "tt_ocr_pages_ex")
        r = res.contents
        items = sum(r.pages[i].n_items for i in range(r.n_pages))
        out = None
        if keep:
            out = [[(r.pages[p].items[i].text, tuple(r.pages[p].items[i].bbox)) for i in range(r.pages[p].n_items)]
                   for p in range(r.n_pages)]
        lib.tt_result_free(res)
        assert items == n * WORDS, items
        return out

    for _ in range(args.warmup):
        for s in (0, 1):
            step(s)
    acc = {s: dict(sec=0.0, d2h=0, launches=0) for s in (0, 1)}
    for _ in range(args.steps):
        for s in (0, 1):
            torch.cuda.synchronize()
            h0, d0 = C.c_ulonglong(), C.c_ulonglong()
            lib.tt_io_bytes(C.byref(h0), C.byref(d0))
            l0 = tb.launch_count()
            t0 = time.perf_counter()
            step(s)
            torch.cuda.synchronize()   # tt_ocr_pages_ex returns after its last device sync; this closes the window
            acc[s]["sec"] += time.perf_counter() - t0
            h1, d1 = C.c_ulonglong(), C.c_ulonglong()
            lib.tt_io_bytes(C.byref(h1), C.byref(d1))
            acc[s]["d2h"] += d1.value - d0.value
            acc[s]["launches"] += tb.launch_count() - l0
    same = step(0, keep=True) == step(1, keep=True)
    eng.close()
    name, power = gpu_info()
    arms = {f"with_scores_{s}": dict(pages_per_s=n * args.steps / a["sec"], ms_per_step=a["sec"] / args.steps * 1e3,
                                     d2h_bytes_per_step=a["d2h"] / args.steps, launches_per_step=a["launches"] / args.steps)
            for s, a in acc.items()}
    a0, a1 = arms["with_scores_0"], arms["with_scores_1"]
    line = dict(
        workload=f"{n} synthetic 1280x1280 pages per step, 300 words each, pages + score-map overrides resident in HBM, "
                 "one engine on one GPU (3 slots, 32-page recognition batches), arms alternating step by step",
        gpu=name, power_limit=power, steps_per_arm=args.steps, warmup_per_arm=args.warmup, **arms,
        cost_pct=(a0["pages_per_s"] / a1["pages_per_s"] - 1.0) * 100.0,
        extra_d2h_bytes_per_crop=(a1["d2h_bytes_per_step"] - a0["d2h_bytes_per_step"]) / (n * WORDS),
        text_and_bbox_identical=same)
    print(json.dumps(line), flush=True)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(json.dumps(line, indent=1) + "\n")
    if not same:
        raise SystemExit("text / bbox differ between the arms")


if __name__ == "__main__":
    main()
