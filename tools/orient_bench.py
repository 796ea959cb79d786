#!/usr/bin/env python
"""Cost of rotation candidates (tt_ocr_pages_oriented) on BASELINE's 512-page step: synthetic 1280 x 1280 pages with
their score-map overrides resident in HBM, built the way bench.py builds its headline step.  Four arms alternate step
by step on one engine (three execution slots, 32-page recognition batches):
  plain  tt_ocr_pages_ex, today's call
  none   tt_ocr_pages_oriented with no rotation: must be the plain call (same items, launches and bytes)
  r180   rotation_info = [180]: two candidates per word
  r3     rotation_info = [90, 180, 270]: four candidates per word
Reports pages/s per arm with the spread over its steps, launches and host<->device bytes per step and per word, and the
crop_resize / orient_select / parseq stage times of one one-slot step per arm (stage events, run apart from the timed
steps).  Recognition work grows with 1 + |rotation_info|; the cost in pages/s is what this measures.

    python tools/orient_bench.py [--pages 512] [--steps 5] [--warmup 1] [--out FILE.json]
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
ARMS = {"plain": None, "none": [], "r180": [180], "r3": [90, 180, 270]}


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
    ap.add_argument("--steps", type=int, default=5, help="timed steps per arm")
    ap.add_argument("--warmup", type=int, default=1, help="untimed steps per arm")
    ap.add_argument("--out", help="also write the JSON result here")
    args = ap.parse_args()

    import torch

    if not torch.cuda.is_available():
        raise SystemExit("orient_bench.py: no CUDA device (the library has no CPU fallback)")
    import tuatara_b200 as tb
    from tuatara_b200 import _native, synth, weights

    lib = tb.lib()
    tmp = tempfile.TemporaryDirectory(prefix="tuatara_orient_bench_")
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
    rots = {k: None if a is None else (C.c_int * max(len(a), 1))(*a) for k, a in ARMS.items()}

    def step(arm, keep=False):
        res = C.POINTER(_native.tt_result)()
        if rots[arm] is None:
            tb.check(lib.tt_ocr_pages_ex(eng._h, arr, n, C.byref(opt), C.byref(res)), "tt_ocr_pages_ex")
        else:
            tb.check(lib.tt_ocr_pages_oriented(eng._h, arr, n, C.byref(opt), None, 0, rots[arm], len(ARMS[arm]),
                                               C.byref(res)), "tt_ocr_pages_oriented")
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
        """Stage times (ms) of one step on one slot, from the library's stage events."""
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
        out = {}
        for row in buf.value.decode().splitlines():
            f = row.split(",")
            if len(f) == 5 and f[0] in ("crop_resize", "orient_select", "parseq_encoder", "parseq_decoder"):
                out[f[0] + "_ms"] = float(f[2])
        return out

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
    kept = {arm: step(arm, keep=True) for arm in ARMS}
    same = kept["none"] == kept["plain"]
    boxes_same = all([[b for _, b in p] for p in kept[arm]] == [[b for _, b in p] for p in kept["plain"]] for arm in ARMS)
    stage_ms = {arm: stages(arm) for arm in ARMS}
    eng.close()
    name, power = gpu_info()
    arms = {}
    for arm, a in acc.items():
        r = a["rates"]
        arms[arm] = dict(pages_per_s_median=statistics.median(r), pages_per_s_min=min(r), pages_per_s_max=max(r),
                         pages_per_s_steps=r, spread_pct=(max(r) / min(r) - 1.0) * 100.0,
                         launches_per_step=a["launches"] / args.steps,
                         h2d_bytes_per_word=a["h2d"] / args.steps / (n * WORDS),
                         d2h_bytes_per_word=a["d2h"] / args.steps / (n * WORDS),
                         one_slot_stage_ms=stage_ms[arm])
    line = dict(
        workload=f"{n} synthetic 1280x1280 pages per step, 300 words each, pages + score-map overrides resident in HBM, "
                 "one engine on one GPU (3 slots, 32-page recognition batches), arms alternating step by step",
        gpu=name, power_limit=power, steps_per_arm=args.steps, warmup_per_arm=args.warmup, arms=arms,
        none_items_identical_to_plain=same, boxes_identical_in_every_arm=boxes_same)
    print(json.dumps(line), flush=True)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(json.dumps(line, indent=1) + "\n")
    if not same or not boxes_same:
        raise SystemExit("the no-rotation arm differs from the plain call, or an arm moved a box")


if __name__ == "__main__":
    main()
