#!/usr/bin/env python
"""Cost of the contrast re-read (tt_ocr_pages_contrast) on BASELINE's 512-page step: synthetic 1280 x 1280 pages with
their score-map overrides resident in HBM, built the way bench.py builds its headline step.  Four arms alternate step by
step on one engine (three execution slots, 32-page recognition batches):
  off     tt_ocr_pages_ex, today's call
  fixed   contrast_ths = 1e-30: every per-word pass and the count read-back run, and only words whose conf is below
          1e-30 (none with trained weights; the fraction is reported) are read again: the fixed cost
  easy    EasyOCR's defaults (contrast_ths 0.1, adjust_contrast 0.5) on the bench pages
  worst   contrast_ths = 2 on the bench pages squeezed into a 48-level band: every word below the threshold, every crop
          low contrast, so every word is read twice
Reports pages/s per arm with the spread over its steps, launches and host<->device bytes per word, and, from one one-slot
step per arm with stage events (run apart from the timed steps), the contrast and parseq stage times and the fraction of
words re-read.  The card's name, power limit and max SM clock are read in the same run.

    python tools/contrast_bench.py [--pages 512] [--steps 5] [--warmup 1] [--out FILE.json]
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
ARMS = {"off": None, "fixed": (1e-30, 0.5), "easy": (0.1, 0.5), "worst": (2.0, 0.5)}
STAGES = ("contrast_stats", "contrast_apply", "contrast_select", "parseq_encoder", "parseq_decoder")


def gpu_info():
    """Card name, power limit and max SM clock (read only)."""
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = [s.strip() for s in out.split(",")]
        return name, power, clock
    except Exception:  # noqa: BLE001 - the numbers are still reported, without the card's name
        return "unknown", "unknown", "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pages", type=int, default=512)
    ap.add_argument("--steps", type=int, default=5, help="timed steps per arm")
    ap.add_argument("--warmup", type=int, default=1, help="untimed steps per arm")
    ap.add_argument("--out", help="also write the JSON result here")
    args = ap.parse_args()

    import torch

    if not torch.cuda.is_available():
        raise SystemExit("contrast_bench.py: no CUDA device (the library has no CPU fallback)")
    import tuatara_b200 as tb
    from tuatara_b200 import _native, synth, weights

    lib = tb.lib()
    tmp = tempfile.TemporaryDirectory(prefix="tuatara_contrast_bench_")
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
    faded = [(104 + (t.to(torch.int32) * 48) // 255).to(torch.uint8).contiguous() for t in pages]   # 104..152
    maps = [torch.from_numpy(m).cuda() for m in maps_np]

    def images(ts):
        return (_native.tt_image * n)(*[_native.tt_image(t.data_ptr(), t.shape[0], t.shape[1], 3, t.shape[1] * 3) for t in ts])

    arr = {"plain": images(pages), "faded": images(faded)}
    ptrs = (C.c_void_p * n)(*[m.data_ptr() for m in maps])
    opt = _native.tt_ocr_options(1, 1, ptrs, 0, 0)

    def step(arm, keep=False):
        res = C.POINTER(_native.tt_result)()
        a = arr["faded" if arm == "worst" else "plain"]
        if ARMS[arm] is None:
            tb.check(lib.tt_ocr_pages_ex(eng._h, a, n, C.byref(opt), C.byref(res)), "tt_ocr_pages_ex")
        else:
            ths, adj = ARMS[arm]
            tb.check(lib.tt_ocr_pages_contrast(eng._h, a, n, C.byref(opt), None, 0, None, 0, None, 0, ths, adj, C.byref(res)),
                     "tt_ocr_pages_contrast")
        r = res.contents
        items = sum(r.pages[i].n_items for i in range(r.n_pages))
        out = None
        if keep:
            out = [[(r.pages[p].items[i].text, tuple(r.pages[p].items[i].bbox)) for i in range(r.pages[p].n_items)]
                   for p in range(r.n_pages)]
        lib.tt_result_free(res)
        assert items == n * WORDS, items
        return out

    def stages(arm):
        """Stage times (ms) of one step on one slot, from the library's stage events, and the words read again."""
        lib.tt_engine_set_slots(eng._h, 1)
        lib.tt_profile_enable(1)
        lib.tt_profile_stages(None, 0)
        try:
            step(arm)
            torch.cuda.synchronize()
            buf = C.create_string_buffer(1 << 16)
            lib.tt_profile_stages(buf, len(buf))
        finally:
            lib.tt_profile_enable(0)
            lib.tt_profile_collect(None, None, None)   # drop the per-launch records the profile also kept
            lib.tt_engine_set_slots(eng._h, 3)
        out, reread = {}, 0.0
        for row in buf.value.decode().splitlines():
            f = row.split(",")
            if len(f) == 5 and f[0] in STAGES:
                out[f[0] + "_ms"] = float(f[2])
                if f[0] == "contrast_apply":   # the stage's bytes are 128 * 96 * 4 per word read again
                    reread = float(f[4]) / (128 * 96 * 4)
        return out, reread / (n * WORDS)

    for _ in range(args.warmup):
        for arm in ARMS:
            step(arm)
    acc = {arm: dict(rates=[], h2d=0, d2h=0, launches=0) for arm in ARMS}
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
            acc[arm]["d2h"] += d1.value - d0.value
            acc[arm]["launches"] += tb.launch_count() - l0
    kept = {arm: step(arm, keep=True) for arm in ("off", "fixed", "easy")}
    fixed_same = kept["fixed"] == kept["off"]
    boxes_same = all([[b for _, b in p] for p in kept[arm]] == [[b for _, b in p] for p in kept["off"]] for arm in kept)
    stage_ms = {arm: stages(arm) for arm in ARMS}
    eng.close()
    name, power, clock = gpu_info()
    arms = {}
    for arm, a in acc.items():
        r = a["rates"]
        arms[arm] = dict(pages_per_s_median=statistics.median(r), pages_per_s_min=min(r), pages_per_s_max=max(r),
                         pages_per_s_steps=r, spread_pct=(max(r) / min(r) - 1.0) * 100.0,
                         launches_per_step=a["launches"] / args.steps,
                         launches_per_word=a["launches"] / args.steps / (n * WORDS),
                         h2d_bytes_per_word=a["h2d"] / args.steps / (n * WORDS),
                         d2h_bytes_per_word=a["d2h"] / args.steps / (n * WORDS),
                         words_reread_fraction=stage_ms[arm][1], one_slot_stage_ms=stage_ms[arm][0],
                         contrast_ths=None if ARMS[arm] is None else ARMS[arm][0],
                         adjust_contrast=None if ARMS[arm] is None else ARMS[arm][1],
                         pages="squeezed to 104..152" if arm == "worst" else "as synthesised")
    line = dict(
        workload=f"{n} synthetic 1280x1280 pages per step, 300 words each, pages + score-map overrides resident in HBM, "
                 "one engine on one GPU (3 slots, 32-page recognition batches), arms alternating step by step",
        gpu=name, power_limit=power, max_sm_clock=clock, steps_per_arm=args.steps, warmup_per_arm=args.warmup, arms=arms,
        fixed_items_identical_to_off=fixed_same, boxes_identical_in_off_fixed_easy=boxes_same)
    print(json.dumps(line), flush=True)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(json.dumps(line, indent=1) + "\n")
    if (arms["fixed"]["words_reread_fraction"] == 0 and not fixed_same) or not boxes_same:
        raise SystemExit("the fixed-cost arm read no word again but differs from the off arm, or an arm moved a box")


if __name__ == "__main__":
    main()
