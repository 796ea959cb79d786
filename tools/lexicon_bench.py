#!/usr/bin/env python
"""Cost of lexicons (tt_ocr_pages_lexicon) on BASELINE's 512-page step: synthetic 1280 x 1280 pages with their
score-map overrides resident in HBM, built the way bench.py builds its headline step.  Four arms alternate step by step
on one engine (three execution slots, 32-page recognition batches):
  none   tt_ocr_pages_ex, no lexicon
  null   a lexicon request whose entries are all NULL: one-state automata, so the items must be those of `none` (checked)
         and the difference is the pure cost of the state path (dependent state loads, the table and 4-byte roots)
  1k     1 000 seeded pseudo-words for every page
  100k   100 000 seeded pseudo-words for every page
Reports pages/s per arm with the spread over its steps, host-to-device bytes and launches per step, the table bytes, the
host time to build each lexicon and to fold it into a request, the parseq_decoder stage time of one one-slot step per arm
(stage events, run apart from the timed steps), and the card's name and power limit read in the same run.

    python tools/lexicon_bench.py [--pages 512] [--steps 6] [--warmup 1] [--out FILE.json]
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

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

WORDS = 300
ARMS = ("none", "null", "1k", "100k")
ALPHABET = "abcdefghijklmnopqrstuvwxyzABCDEFGHIJKLMNOPQRSTUVWXYZ0123456789-"


def pseudo_words(n, seed):
    """n distinct seeded pseudo-words of 2..12 characters (nothing is downloaded)."""
    rng = np.random.default_rng(seed)
    out = set()
    while len(out) < n:
        out.add("".join(rng.choice(list(ALPHABET), int(rng.integers(2, 13)))))
    return sorted(out)


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
        raise SystemExit("lexicon_bench.py: no CUDA device (the library has no CPU fallback)")
    import tuatara_b200 as tb
    from tuatara_b200 import _native, synth, weights

    lib = tb.lib()
    tmp = tempfile.TemporaryDirectory(prefix="tuatara_lexicon_bench_")
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
    words = {"1k": pseudo_words(1000, 1), "100k": pseudo_words(100000, 2)}
    lexicons, build_ms, info = {}, {}, {}
    for k, w in words.items():
        t0 = time.perf_counter()
        lexicons[k] = tb.Lexicon(w)
        build_ms[k] = (time.perf_counter() - t0) * 1e3
        info[k] = dict(zip(("words", "states"), lexicons[k].info()))
    handles = {"null": (C.c_void_p * 1)(None)}
    handles.update({k: (C.c_void_p * 1)(lexicons[k]._h.value) for k in words})

    def step(arm, keep=False):
        res = C.POINTER(_native.tt_result)()
        if arm == "none":
            tb.check(lib.tt_ocr_pages_ex(eng._h, arr, n, C.byref(opt), C.byref(res)), "tt_ocr_pages_ex")
        else:
            tb.check(lib.tt_ocr_pages_lexicon(eng._h, arr, n, C.byref(opt), None, 0, None, 0, handles[arm], 1, C.byref(res)),
                     "tt_ocr_pages_lexicon")
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
            if f[0] in ("parseq_encoder", "parseq_decoder", "lexicon_table"):
                out[f[0]] = float(f[2])
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
    stage_ms = {arm: stages(arm) for arm in ARMS}
    plain, null = step("none", keep=True), step("null", keep=True)
    same = plain == null
    in_lexicon = {}
    for k in words:
        ws = set(w.encode() for w in words[k])
        in_lexicon[k] = all(t in ws for page in step(k, keep=True) for t, _ in page)
    # host time of make_request's fold for the 100k lexicon: a request of zero pages builds nothing, so time one page
    # with detect_only (detection is the same in every arm)
    one = (_native.tt_image * 1)(arr[0])
    opt1 = _native.tt_ocr_options(1, 1, (C.c_void_p * 1)(ptrs[0]), 1, 0)
    fold_ms = {}
    for arm in ARMS[1:]:
        t = []
        for _ in range(5):
            res = C.POINTER(_native.tt_result)()
            t0 = time.perf_counter()
            tb.check(lib.tt_ocr_pages_lexicon(eng._h, one, 1, C.byref(opt1), None, 0, None, 0, handles[arm], 1, C.byref(res)),
                     "tt_ocr_pages_lexicon")
            t.append((time.perf_counter() - t0) * 1e3)
            lib.tt_result_free(res)
        fold_ms[arm] = statistics.median(t)
    eng.close()
    name, power = gpu_info()
    arms = {}
    for arm, a in acc.items():
        r = a["rates"]
        arms[arm] = dict(pages_per_s_median=statistics.median(r), pages_per_s_min=min(r), pages_per_s_max=max(r),
                         pages_per_s_steps=r, h2d_bytes_per_step=a["h2d"] / args.steps,
                         launches_per_step=a["launches"] / args.steps, one_slot_stage_ms=stage_ms[arm],
                         detect_only_page_ms=fold_ms.get(arm))
    a0, a1 = arms["none"], arms["null"]
    line = dict(
        workload=f"{n} synthetic 1280x1280 pages per step, 300 words each, pages + score-map overrides resident in HBM, "
                 "one engine on one GPU (3 slots, 32-page recognition batches), arms alternating step by step",
        gpu=name, power_limit=power, steps_per_arm=args.steps, warmup_per_arm=args.warmup, arms=arms,
        # the request's table: the done state (95 successors) and the trie, 5 words per state, one successor per trie
        # edge and per word end (ALPHABET has no backslash, the one character with two classes)
        lexicons={k: dict(info[k], create_ms=build_ms[k],
                          table_bytes=4 * (5 * (info[k]["states"] + 1) + 95 + info[k]["states"] - 1 + info[k]["words"]))
                  for k in words},
        null_vs_none_cost_pct=(a0["pages_per_s_median"] / a1["pages_per_s_median"] - 1.0) * 100.0,
        none_spread_pct=(a0["pages_per_s_max"] / a0["pages_per_s_min"] - 1.0) * 100.0,
        null_spread_pct=(a1["pages_per_s_max"] / a1["pages_per_s_min"] - 1.0) * 100.0,
        extra_h2d_bytes_per_step={k: arms[k]["h2d_bytes_per_step"] - a0["h2d_bytes_per_step"] for k in ARMS[1:]},
        one_slot_decoder_ms_minus_none={k: stage_ms[k]["parseq_decoder"] - stage_ms["none"]["parseq_decoder"]
                                        for k in ARMS[1:]},
        null_items_identical_to_none=same, items_in_their_lexicon=in_lexicon)
    print(json.dumps(line), flush=True)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(json.dumps(line, indent=1) + "\n")
    if not same or not all(in_lexicon.values()):
        raise SystemExit("the all-NULL arm differs from no lexicon, or an item is not a word of its lexicon")


if __name__ == "__main__":
    main()
