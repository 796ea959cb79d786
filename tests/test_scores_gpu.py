"""Per-word scores on the GPU: the fused refinement head (k_argmax_conf) against its own logits and the oracle, the
detection score against the oracle's maxVal, and the scored entry points against the unscored ones."""
import ctypes as C
import sys
from pathlib import Path

import cv2
import numpy as np
import pytest
import torch

import tuatara_b200 as tb
from oracle import imagemaps
from oracle import tuatara_ref as R
from scores_ref import image_to_data_scored
from tuatara_b200 import _native, synth

pytestmark = pytest.mark.gpu

FIXTURES = ["resume_example", "funsd_0001129658", "funsd_91372360", "table_english", "rotated_text"]
TEXT_THRESHOLD = float(np.float32(0.7))
FLT_MIN = float(np.finfo(np.float32).tiny)


def _fixtures():
    return np.load(Path(__file__).parent / "golden" / "fixture_images.npz")


def _crops(n, seed):
    """Seeded 32x128 crops: a third cut from the fixture pages, a third from a synthetic page, the rest noise; the
    first two blank (black, white)."""
    rng = np.random.default_rng(seed)
    fx = _fixtures()
    srcs = [fx[f"{k}.img"] for k in FIXTURES] + [synth.synth_page(seed)]
    out = []
    for i in range(2 * n // 3):
        img = srcs[i % len(srcs)] if i < n // 3 else srcs[-1]
        h, w = img.shape[:2]
        cw, ch = int(rng.integers(20, min(200, w))), int(rng.integers(10, min(60, h)))
        x, y = int(rng.integers(0, w - cw)), int(rng.integers(0, h - ch))
        out.append(cv2.resize(img[y:y + ch, x:x + cw], (128, 32)))
    out += list(rng.integers(0, 256, (n - len(out), 32, 128, 3), dtype=np.uint8))
    crops = np.ascontiguousarray(np.stack(out))
    crops[0] = 0
    crops[1] = 255
    return crops


def _softmax_max64(logits):
    l64 = logits.astype(np.float64)
    return 1.0 / np.exp(l64 - l64.max(-1, keepdims=True)).sum(-1)


def _end(ids):
    """End position of each row: the first id 0, else the last position."""
    z = ids == 0
    return np.where(z.any(-1), z.argmax(-1), ids.shape[-1] - 1)


def test_parseq_scores_match_own_logits(engine):
    crops = _crops(300, seed=31)
    logits, ids0 = engine.parseq_forward(crops)
    ids1, p1 = engine.parseq_forward_scores(crops)
    ids2, p2 = engine.parseq_forward_scores(crops)
    assert np.array_equal(ids1, ids0)
    assert p1.tobytes() == p2.tobytes() and np.array_equal(ids2, ids1)
    want = _softmax_max64(logits)
    err = np.abs(p1 - want)
    print("pmax vs float64 softmax of the logits: max abs", float(err.max()), "max rel", float((err / want).max()))
    assert (err <= 1e-6 + 1e-5 * want).all()
    # a request over kMaxCropsPerPass (32768 crops per PARSeq pass): the same crops in two smaller calls
    big = np.concatenate([crops] * 110)[:32768 + 200]
    big[300:] = np.random.default_rng(32).integers(0, 256, big[300:].shape, dtype=np.uint8)
    ib, pb = engine.parseq_forward_scores(big)
    h = 16484
    ia, pa = engine.parseq_forward_scores(big[:h])
    ic, pc = engine.parseq_forward_scores(big[h:])
    i2, p2 = np.concatenate([ia, ic]), np.concatenate([pa, pc])
    assert np.array_equal(ib, i2)
    d = np.abs(np.log(pb.astype(np.float64)) - np.log(p2.astype(np.float64)))
    print("32968 crops in one call vs two: max |d log p|", float(d.max()))
    assert float(d.max()) <= 5e-4
    assert np.array_equal(ib[:300], ids1)


def test_confidence_against_the_oracle(engine, oracle_models):
    """log p = l_max - logsumexp(l) is 2-Lipschitz in the max norm of the logits, so for crops whose ids equal the
    oracle's the per-position bound holds whatever the bf16 error of the logits is."""
    _, parseq = oracle_models
    crops = _crops(48, seed=33)
    logits, _ = engine.parseq_forward(crops)
    ids, p = engine.parseq_forward_scores(crops)
    x = torch.from_numpy(crops).permute(0, 3, 1, 2).float().div(255.0)
    with torch.no_grad():
        ref = parseq(x).numpy()
    ref_ids = ref.argmax(-1)
    p_ref = _softmax_max64(ref)
    e = _end(ids)
    checked = 0
    for i in range(len(crops)):
        t = np.arange(e[i] + 1)
        if not np.array_equal(ids[i, t], ref_ids[i, t]):
            continue
        bound = 2.0 * np.abs(logits[i, t].astype(np.float64) - ref[i, t]).max(-1) + 1e-5
        d = np.abs(np.log(p[i, t].astype(np.float64)) - np.log(p_ref[i, t]))
        assert (d <= bound).all(), (i, d, bound)
        checked += 1
    print("crops with the oracle's ids", checked, "of", len(crops), "; median p", float(np.median(p)))
    assert checked >= len(crops) // 2
    assert float(np.median(p)) > 1.0 / 95


def _pages():
    """Two synthetic pages with override maps (300 boxes each) and the five fixture pages with their golden maps."""
    fx = _fixtures()
    pages = [synth.synth_page(i) for i in range(2)] + [np.ascontiguousarray(fx[f"{k}.img"]) for k in FIXTURES]
    maps = [synth.synth_score_maps(i) for i in range(2)] + [imagemaps.maps_f32(fx[f"{k}.maps_u8"]) for k in FIXTURES]
    return pages, [np.ascontiguousarray(m) for m in maps]


def _oracle(page, maps):
    """The oracle's boxes and scores for an overridden page (no network runs: both are replaced)."""
    st = R.Stages()
    craft = lambda x: (torch.zeros(1, x.shape[2] // 2, x.shape[3] // 2, 2), None)  # noqa: E731  (overridden)
    parseq = lambda x: torch.zeros(x.shape[0], 26, 95)  # noqa: E731
    out = image_to_data_scored(page.copy(), craft, parseq, score_override=(maps[..., 0], maps[..., 1]), stages=st)
    return out, st


def test_detection_score_matches_oracle(engine):
    pages, maps = _pages()
    got = engine.ocr_pages(pages, score_override=maps, scores=True)
    total = 0
    for k in range(len(pages)):
        ref, _ = _oracle(pages[k], maps[k])
        assert [g["bbox"] for g in got[k]] == [r["bbox"] for r in ref]
        for g, r in zip(got[k], ref):
            assert np.float32(g["det_score"]).tobytes() == np.float32(r["det_score"]).tobytes()
            assert g["det_score"] >= TEXT_THRESHOLD
        total += len(ref)
    assert len(got[0]) == len(got[1]) == 300 and total > 600


def test_scores_leave_items_unchanged(engine):
    pages, maps = _pages()
    plain = engine.ocr_pages(pages, score_override=maps)
    scored = engine.ocr_pages(pages, score_override=maps, scores=True)
    compared = 0
    for k in range(len(pages)):
        assert [dict(text=s["text"], bbox=s["bbox"]) for s in scored[k]] == plain[k]
        for s in scored[k]:
            assert len(s["char_conf"]) == len(s["text"])
            assert s["conf"] is not None
            if s["char_conf"]:
                assert s["conf"] <= min(s["char_conf"])
        # the stage-level head on the crops of the same boxes (a different batch: the batch-invariance bound)
        _, st = _oracle(pages[k], maps[k])
        crops = tb.crop_resize(pages[k], st.crop_rects)
        ids, p = engine.parseq_forward_scores(crops)
        texts, conf, char_conf = tb.decode_scores(ids, p)
        e = _end(ids)
        for i, s in enumerate(scored[k]):
            if s["text"] != texts[i]:
                continue
            d = np.abs(np.log(np.asarray(s["char_conf"], np.float64)) - np.log(char_conf[i].astype(np.float64)))
            assert (d <= 5e-4).all(), (k, i, d)
            log_conf = float(np.log(p[i, :e[i] + 1].astype(np.float64)).sum())
            tol = 5e-4 * (e[i] + 1) + 1e-6
            if s["conf"] >= FLT_MIN:
                assert abs(np.log(s["conf"]) - log_conf) <= tol, (k, i, s["conf"], log_conf)
            else:   # the product fell below the normal range of float32
                assert log_conf <= np.log(FLT_MIN) + tol, (k, i, s["conf"], log_conf)
            compared += 1
        assert compared >= 0.95 * sum(len(s) for s in scored[:k + 1]), (k, compared)


def test_detect_only_with_scores(engine):
    pages, maps = _pages()
    got = engine.ocr_pages(pages[:3], score_override=maps[:3], detect_only=True, scores=True)
    boxes = engine.ocr_pages(pages[:3], score_override=maps[:3], detect_only=True)
    for k in range(3):
        assert [dict(text=g["text"], bbox=g["bbox"]) for g in got[k]] == boxes[k] and len(got[k]) > 0
        ref, _ = _oracle(pages[k], maps[k])
        for g, r in zip(got[k], ref):
            assert g["conf"] is None and g["char_conf"] == [] and g["text"] == ""
            assert g["det_score"] == r["det_score"] and g["det_score"] >= TEXT_THRESHOLD
    # the C ABI: conf -1, and tt_item_scores refuses a result made without with_scores
    lib = tb.lib()
    arr = (_native.tt_image * 1)(_native.image_struct(pages[2]))
    m = maps[2]
    ptrs = (C.c_void_p * 1)(m.ctypes.data)
    for with_scores in (1, 0):
        opt = _native.tt_ocr_options(0, 0, ptrs, 1, with_scores)
        res = C.POINTER(_native.tt_result)()
        tb.check(lib.tt_ocr_pages_ex(engine._h, arr, 1, C.byref(opt), C.byref(res)), "tt_ocr_pages_ex")
        try:
            conf, det, cc, n = C.c_float(), C.c_float(), C.POINTER(C.c_float)(), C.c_int()
            rc = lib.tt_item_scores(res, 0, 0, C.byref(conf), C.byref(det), C.byref(cc), C.byref(n))
            if with_scores:
                assert rc == 0 and conf.value == -1.0 and n.value == 0 and not cc and det.value >= TEXT_THRESHOLD
                assert lib.tt_item_scores(res, 0, res.contents.pages[0].n_items, None, None, None, None) != 0
                assert lib.tt_item_scores(res, 1, 0, None, None, None, None) != 0
            else:
                assert rc != 0 and b"with_scores" in lib.tt_last_error()
        finally:
            lib.tt_result_free(res)


def test_empty_page_with_scores(engine):
    blank = np.full((320, 512, 3), 255, np.uint8)
    zero_maps = np.zeros((160, 256, 2), np.float32)
    assert engine.ocr_pages([blank], score_override=[zero_maps], scores=True) == [[]]
    assert engine.ocr_pages([blank], score_override=[zero_maps], detect_only=True, scores=True) == [[]]
    assert engine.ocr_pages([], scores=True) == []
    page = np.ascontiguousarray(synth.synth_page(0)[:320, :384])
    maps = np.ascontiguousarray(synth.synth_score_maps(0)[:160, :192])
    got = engine.ocr_pages([blank, page], score_override=[zero_maps, maps], scores=True)
    assert got[0] == [] and len(got[1]) > 0 and all(g["conf"] is not None for g in got[1])


def test_pytuatara_scored_against_engine(engine, weights_dir, native_lib):
    sys.path.insert(0, str(_native.LIB_PATH.parent))
    import pytuatara

    fx = _fixtures()
    pages = [np.ascontiguousarray(fx["resume_example.img"])] + \
        [np.ascontiguousarray(synth.synth_page(s)[:h, :w]) for s, (h, w) in ((0, (607, 763)), (2, (754, 1000)))]
    n_items = 0
    for page in pages:
        got = pytuatara.image_to_data_scored(image=page.copy(), weights_dir=weights_dir, outputs_dir="outputs")
        assert all(set(g) == {"text", "bbox", "conf", "det_score", "char_conf"} for g in got)
        assert got == engine.ocr_pages([page], scores=True)[0]
        assert got == tb.image_to_data_scored(page, weights_dir, "outputs")
        plain = pytuatara.image_to_data(image=page.copy(), weights_dir=weights_dir, outputs_dir="outputs")
        assert [dict(text=g["text"], bbox=g["bbox"]) for g in got] == plain
        n_items += len(got)
    batch = pytuatara.images_to_data_scored(images=pages, weights_dir=weights_dir, outputs_dir="outputs")
    assert [[dict(text=g["text"], bbox=g["bbox"]) for g in p] for p in batch] == \
        [pytuatara.image_to_data(image=p, weights_dir=weights_dir, outputs_dir="outputs") for p in pages]
    assert n_items > 0
