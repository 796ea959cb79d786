#!/usr/bin/env python
"""Cost of character filters (tt_ocr_pages_filtered) on BASELINE's 512-page step: synthetic 1280 x 1280 pages with
their score-map overrides resident in HBM, built the way bench.py builds its headline step.  Three arms alternate step
by step on one engine (three execution slots, 32-page recognition batches):
  none   tt_ocr_pages_ex, no filter
  all    an allowlist of every printable character: a mask that allows every class, so the tokens are those of `none`
         and the difference is the pure cost of the masked kernels and the 16-byte-per-crop mask upload
  digits an allowlist of the ten digits (for information: it changes the decoded lengths, so the AR early exit's work)
Reports pages/s per arm with the spread over its steps, host-to-device bytes and kernel launches per step, and checks
that `all` returns exactly the items of `none`.

    python tools/charset_bench.py [--pages 512] [--steps 6] [--warmup 1] [--out FILE.json]
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

WORDS = 300
PRINTABLE = "".join(chr(c) for c in range(32, 127))
ARMS = {"none": None, "all": PRINTABLE, "digits": "0123456789"}


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
    ap.add_argument("--steps", type=int, default=6, help="timed steps per arm")
    ap.add_argument("--warmup", type=int, default=1, help="untimed steps per arm")
    ap.add_argument("--out", help="also write the JSON result here")
    args = ap.parse_args()

    import torch

    if not torch.cuda.is_available():
        raise SystemExit("charset_bench.py: no CUDA device (the library has no CPU fallback)")
    import tuatara_b200 as tb
    from tuatara_b200 import _native, synth, weights

    lib = tb.lib()
    tmp = tempfile.TemporaryDirectory(prefix="tuatara_charset_bench_")
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
    opt = _native.tt_ocr_options(1, 1, ptrs, 0, 0)
    filters = {k: None if a is None else _native.tt_char_filter(a.encode(), None) for k, a in ARMS.items()}

    def step(arm, keep=False):
        res = C.POINTER(_native.tt_result)()
        f = filters[arm]
        if f is None:
            tb.check(lib.tt_ocr_pages_ex(eng._h, arr, n, C.byref(opt), C.byref(res)), "tt_ocr_pages_ex")
        else:
            tb.check(lib.tt_ocr_pages_filtered(eng._h, arr, n, C.byref(opt), C.byref(f), 1, C.byref(res)),
                     "tt_ocr_pages_filtered")
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
        for arm in ARMS:
            step(arm)
    acc = {arm: dict(rates=[], h2d=0, launches=0) for arm in ARMS}
    for _ in range(args.steps):
        for arm in ARMS:
            torch.cuda.synchronize()
            h0, d0 = C.c_ulonglong(), C.c_ulonglong()
            lib.tt_io_bytes(C.byref(h0), C.byref(d0))
            l0 = tb.launch_count()
            t0 = time.perf_counter()
            step(arm)
            torch.cuda.synchronize()   # tt_ocr_pages_* return after their last device sync; this closes the window
            acc[arm]["rates"].append(n / (time.perf_counter() - t0))
            h1, d1 = C.c_ulonglong(), C.c_ulonglong()
            lib.tt_io_bytes(C.byref(h1), C.byref(d1))
            acc[arm]["h2d"] += h1.value - h0.value
            acc[arm]["launches"] += tb.launch_count() - l0
    plain, every = step("none", keep=True), step("all", keep=True)
    same = plain == every
    digits = step("digits", keep=True)
    digits_ok = all(set(t.decode("latin-1")) <= set("0123456789") for page in digits for t, _ in page)
    eng.close()
    name, power = gpu_info()
    arms = {}
    for arm, a in acc.items():
        r = a["rates"]
        arms[arm] = dict(pages_per_s_median=statistics.median(r), pages_per_s_min=min(r), pages_per_s_max=max(r),
                         pages_per_s_steps=r, h2d_bytes_per_step=a["h2d"] / args.steps,
                         launches_per_step=a["launches"] / args.steps)
    a0, a1 = arms["none"], arms["all"]
    line = dict(
        workload=f"{n} synthetic 1280x1280 pages per step, 300 words each, pages + score-map overrides resident in HBM, "
                 "one engine on one GPU (3 slots, 32-page recognition batches), arms alternating step by step",
        gpu=name, power_limit=power, steps_per_arm=args.steps, warmup_per_arm=args.warmup, arms=arms,
        all_vs_none_cost_pct=(a0["pages_per_s_median"] / a1["pages_per_s_median"] - 1.0) * 100.0,
        none_spread_pct=(a0["pages_per_s_max"] / a0["pages_per_s_min"] - 1.0) * 100.0,
        all_spread_pct=(a1["pages_per_s_max"] / a1["pages_per_s_min"] - 1.0) * 100.0,
        extra_h2d_bytes_per_crop=(a1["h2d_bytes_per_step"] - a0["h2d_bytes_per_step"]) / (n * WORDS),
        all_items_identical_to_none=same, digits_text_only_digits=digits_ok)
    print(json.dumps(line), flush=True)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(json.dumps(line, indent=1) + "\n")
    if not same or not digits_ok:
        raise SystemExit("the all-allowing arm differs from no filter, or the digits arm produced another character")


if __name__ == "__main__":
    main()
