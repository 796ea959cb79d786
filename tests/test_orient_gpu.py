"""Rotation candidates on the GPU: the rotated crops bit for bit against cv2, the rectified candidates against
cv2.warpPerspective, k_orient_select against the host rule, and tt_ocr_pages_oriented end to end against a host
recomputation of every candidate, the unrotated path and the oracle."""
import ctypes as C
import math
import sys

import cv2
import numpy as np
import pytest
import torch

import tuatara_b200 as tb
from oracle import tuatara_ref as R
from orient_ref import candidate_crop, candidate_set, conf_of, image_to_data_oriented, select
from test_charset_gpu import _io
from test_scores_gpu import _fixtures, _oracle, _pages
from tuatara_b200 import _native, synth

pytestmark = pytest.mark.gpu

ANGLES = (0, 90, 180, 270)


def _random_rects(rng, H, W, n):
    """Clamped rects of every kind: w or h = 1, empty, on the border, wider or taller than 4096 pixels."""
    out = []
    for i in range(n):
        k = i % 8
        if k == 0:
            w, h = 1, int(rng.integers(1, 80))
        elif k == 1:
            w, h = int(rng.integers(1, 300)), 1
        elif k == 2:
            w, h = (0, int(rng.integers(0, 30))) if i % 16 < 8 else (int(rng.integers(0, 30)), 0)
        elif k == 3 and W > 4097:
            w, h = int(rng.integers(4097, W + 1)), int(rng.integers(1, 60))
        elif k == 4 and H > 4097:
            w, h = int(rng.integers(1, 60)), int(rng.integers(4097, H + 1))
        else:
            w, h = int(rng.integers(1, min(400, W))), int(rng.integers(1, min(200, H)))
        x, y = int(rng.integers(0, W - w + 1)), int(rng.integers(0, H - h + 1))
        if k == 6:   # on the border
            x, y = (W - w, y) if i % 2 else (x, H - h)
        out.append((x, y, w, h))
    return out


def _big_page(seed):
    rng = np.random.default_rng(seed)
    page = rng.integers(0, 256, (4500, 4700, 3), dtype=np.uint8)
    page[:1280, :1280] = synth.synth_page(seed)
    return np.ascontiguousarray(page)


def _check_rotated_crops(page, rects):
    plain = tb.crop_resize(page, rects)
    for a in ANGLES:
        got = tb.crop_resize(page, rects, [a] * len(rects))
        want = np.stack([candidate_crop(page, r, a) for r in rects])
        bad = [i for i in range(len(rects)) if got[i].tobytes() != want[i].tobytes()]
        assert not bad, (a, len(bad), [rects[i] for i in bad[:5]])
        if a == 0:
            assert got.tobytes() == plain.tobytes()
    mixed = [ANGLES[i % 4] for i in range(len(rects))]
    got = tb.crop_resize(page, rects, mixed)
    assert all(np.array_equal(got[i], candidate_crop(page, r, a)) for i, (r, a) in enumerate(zip(rects, mixed)))


def test_rotated_crops_bit_exact_vs_cv2(native_lib):
    pages, maps = _pages()
    total = 0
    for k in range(2, len(pages)):   # the fixture pages and the rects the path crops there
        _, st = _oracle(pages[k], maps[k])
        _check_rotated_crops(pages[k], st.crop_rects)
        total += len(st.crop_rects)
    page = _big_page(5)
    rects = _random_rects(np.random.default_rng(6), *page.shape[:2], 200)
    _check_rotated_crops(page, rects)
    print("fixture rects", total, "random rects", len(rects))
    assert total > 100


def test_rotated_crops_equivariance(native_lib):
    page = np.ascontiguousarray(synth.synth_page(3)[:900, :1100])
    H, W = page.shape[:2]
    rects = _random_rects(np.random.default_rng(7), H, W, 400)
    rects = [r for r in rects if r[2] <= W and r[3] <= H]
    flip = np.ascontiguousarray(page[::-1, ::-1])
    turn = np.ascontiguousarray(np.rot90(page))   # 90 degrees counter-clockwise
    r180 = [(W - x - w, H - y - h, w, h) for x, y, w, h in rects]
    r90 = [(y, W - x - w, h, w) for x, y, w, h in rects]
    for a in ANGLES:
        n = len(rects)
        base = tb.crop_resize(page, rects, [(a + 180) % 360] * n)
        assert tb.crop_resize(flip, r180, [a] * n).tobytes() == base.tobytes(), a
        base = tb.crop_resize(page, rects, [(a + 90) % 360] * n)
        assert tb.crop_resize(turn, r90, [a] * n).tobytes() == base.tobytes(), a


def test_rectified_candidates_vs_cv2(native_lib):
    pages, maps = _pages()
    same = total = worst = 0
    closer = checked = 0
    for k in (0, 2, 3, 6):
        _, st = _oracle(pages[k], maps[k])
        for a in ANGLES:
            quads = np.stack([np.roll(tb.rect_to_quad(b), -(a // 90), 0) for b in st.boxes])
            got = tb.crop_warp(pages[k], quads)
            want = np.stack([R.rectified_crop(pages[k], q) for q in quads])
            d = np.abs(got.astype(int) - want.astype(int))
            same += int((d == 0).sum())
            total += d.size
            worst = max(worst, int(d.max()))
    # direction: an axis-aligned box's rectified candidate a looks like the rectify = 0 candidate a, not a + 180 (on a
    # smooth random page: no flat region where the two are equal, and the half-pixel offset of the warp barely shows)
    rng = np.random.default_rng(8)
    page = cv2.resize(rng.integers(0, 256, (48, 48, 3), dtype=np.uint8), (1280, 1280), interpolation=cv2.INTER_CUBIC)
    for _ in range(60):
        w, h = int(rng.integers(40, 300)), int(rng.integers(12, 60))
        x, y = int(rng.integers(0, 1280 - w)), int(rng.integers(0, 1280 - h))
        rect = ((x + w / 2.0, y + h / 2.0), (float(w), float(h)), 0.0)
        roi = tb.rect_bounding(rect)
        for a in ANGLES:
            warp = tb.crop_warp(page, np.roll(tb.rect_to_quad(rect), -(a // 90), 0)[None])[0].astype(int)
            near = np.abs(warp - candidate_crop(page, roi, a).astype(int)).mean()
            far = np.abs(warp - candidate_crop(page, roi, (a + 180) % 360).astype(int)).mean()
            closer += near < far
            checked += 1
    print(f"rectified candidates: {same / total:.6f} of pixels identical, worst {worst}; direction {closer}/{checked}")
    assert same / total >= 0.9999 and worst <= 8
    assert closer == checked


def _select_dev(ids, p, angles, with_p=True):
    n = ids.shape[0] // len(angles)
    di, dp = torch.from_numpy(ids).cuda(), torch.from_numpy(p).cuda()
    oi = torch.empty((n, 26), dtype=torch.int32, device="cuda")
    op = torch.empty((n, 26), dtype=torch.float32, device="cuda") if with_p else None
    oa = torch.empty(n, dtype=torch.int32, device="cuda")
    a = (C.c_int * len(angles))(*angles)
    tb.check(tb.lib().tt_orient_select_dev(di.data_ptr(), dp.data_ptr(), n, a, len(angles), oi.data_ptr(),
                                            op.data_ptr() if with_p else None, oa.data_ptr(), None), "tt_orient_select_dev")
    torch.cuda.synchronize()
    return oi.cpu().numpy(), None if op is None else op.cpu().numpy(), oa.cpu().numpy()


@pytest.mark.parametrize("rotation_info", [[180], [90, 270], [90, 180, 270]])
def test_orient_select_matches_the_host_rule(native_lib, rotation_info):
    angles = candidate_set(rotation_info)
    Rn, n = len(angles), 3000
    rng = np.random.default_rng(len(angles))
    ids = rng.integers(1, 95, (n * Rn, 26)).astype(np.int32)
    ids[rng.random(ids.shape) < 0.08] = 0
    ids[rng.random(ids.shape) < 0.05] = 88
    p = rng.uniform(0.3, 1.0, (n * Rn, 26)).astype(np.float32)
    v = ids.reshape(n, Rn, 26)
    q = p.reshape(n, Rn, 26)
    for w in range(n):
        kind = w % 10
        if kind == 0:                              # exact tie with candidate 0
            v[w, -1], q[w, -1] = v[w, 0], q[w, 0]
        elif kind == 1:                            # every candidate equal
            v[w, :], q[w, :] = v[w, 0], q[w, 0]
        elif kind == 2:                            # NaN in candidate 0 and in a later one
            q[w, 0, 0] = np.nan
            q[w, -1, 1] = np.nan
        elif kind == 3:                            # products that underflow to 0: 0 ties
            q[w, :, :] = 1e-30
            v[w, :, :] = 7
        elif kind == 4:                            # id 0 at position 0
            v[w, :, 0] = 0
        elif kind == 5:                            # no end class
            v[w, :][v[w, :] == 0] = 5
        elif kind == 6:                            # the same conf reached with different ids
            v[w, 1:] = np.where(v[w, 0] == 0, 0, 9)
            q[w, 1:] = q[w, 0]
    oi, op, oa = _select_dev(ids, p, angles)
    confs = np.array([[conf_of(v[w, r], q[w, r]) for r in range(Rn)] for w in range(n)])
    for w in range(n):
        b = select(confs[w])
        assert oa[w] == angles[b], (w, confs[w], oa[w])
        assert np.array_equal(oi[w], v[w, b]) and op[w].tobytes() == q[w, b].tobytes()
    oi2, op2, oa2 = _select_dev(ids, p, angles, with_p=False)
    assert np.array_equal(oi2, oi) and np.array_equal(oa2, oa) and op2 is None
    print("angles chosen:", {a: int((oa == a).sum()) for a in angles}, "zero-conf words", int((confs.max(1) == 0).sum()))


def _engine(weights_dir, rectify):
    cfg = tb.default_config()
    cfg.rectify = rectify
    cfg.slots_per_gpu = 1
    return tb.Engine(weights_dir, cfg=cfg)


def _host_oriented(engine, page, maps, rotation_info, rectify, mask):
    """Every candidate of every word of one page through the stage entry points, decoded and chosen on the host."""
    _, st = _oracle(page, maps)
    cands = candidate_set(rotation_info)
    crops = []
    for rect, box in zip(st.crop_rects, st.boxes):
        if rectify:
            crops.append(tb.crop_warp(page, np.stack([np.roll(tb.rect_to_quad(box), -(a // 90), 0) for a in cands])))
        else:
            crops.append(tb.crop_resize(page, [rect] * len(cands), cands))
    crops = np.concatenate(crops)
    masks = None if mask is None else np.tile(mask, (len(crops), 1))
    ids, p = engine.parseq_forward_scores(crops, class_masks=masks)
    texts, conf, cc = tb.decode_scores(ids, p)
    out = []
    for w in range(len(st.crop_rects)):
        k = [w * len(cands) + r for r in range(len(cands))]
        b = select([conf[i] for i in k])
        i = k[b]
        out.append(dict(text=texts[i], conf=float(conf[i]), char_conf=[float(v) for v in cc[i]], angle=cands[b]))
    return out


@pytest.mark.parametrize("rectify", [0, 1])
def test_whole_path_equals_host_recomputation(native_lib, weights_dir, rectify):
    eng = _engine(weights_dir, rectify)
    pages, maps = _pages()
    filters = [None, ("0123456789", None), None, (None, "aeiou"), None, ("ABCDEFGHIJKLMNOPQRSTUVWXYZ", None), None]
    rotation_info = [90, 180, 270]
    words = moved = 0
    try:
        for k in range(len(pages)):
            f = filters[k]
            kw = {} if f is None else dict(allowlist=f[0], blocklist=f[1])
            mask = None if f is None else tb.char_filter_mask(*f)
            want = _host_oriented(eng, pages[k], maps[k], rotation_info, rectify, mask)
            for scores in (False, True):
                got = eng.ocr_pages([pages[k]], score_override=[maps[k]], scores=scores, rotation_info=rotation_info,
                                    **kw)[0]
                assert len(got) == len(want)
                for g, w in zip(got, want):
                    assert g["text"] == w["text"] and g["angle"] == w["angle"], (k, g, w)
                    if scores:
                        assert np.float32(g["conf"]).tobytes() == np.float32(w["conf"]).tobytes()
                        assert np.array_equal(np.float32(g["char_conf"]), np.float32(w["char_conf"]))
            words += len(want)
            moved += sum(w["angle"] != 0 for w in want)
        # filters on some pages of one request: each page as if it ran alone
        allow = [f[0] if f else None for f in filters]
        block = [f[1] if f else None for f in filters]
        batch = eng.ocr_pages(pages, score_override=maps, scores=True, rotation_info=rotation_info, allowlist=allow,
                              blocklist=block)
        for k in range(len(pages)):
            alone = eng.ocr_pages([pages[k]], score_override=[maps[k]], scores=True, rotation_info=rotation_info,
                                  allowlist=allow[k], blocklist=block[k])[0]
            assert batch[k] == alone, k
    finally:
        eng.close()
    print(f"rectify={rectify}: {words} words, {moved} read at another angle than 0")
    assert words > 600 and moved > 0


def test_nothing_else_moves(engine):
    pages, maps = _pages()
    lib = tb.lib()
    lib.tt_engine_set_slots(engine._h, 1)   # one slot: the recognition batches, so the launches, are deterministic
    try:
        for scores in (False, True):
            c0, (h0, d0) = tb.launch_count(), _io()
            plain = engine.ocr_pages(pages, score_override=maps, scores=scores)
            c1, (h1, d1) = tb.launch_count(), _io()
            empty = engine.ocr_pages(pages, score_override=maps, scores=scores, rotation_info=[])
            c2, (h2, d2) = tb.launch_count(), _io()
            assert c2 - c1 == c1 - c0 and h2 - h1 == h1 - h0 and d2 - d1 == d1 - d0
            assert [[{k: v for k, v in it.items() if k != "angle"} for it in p] for p in empty] == plain
            assert all(it["angle"] == 0 for p in empty for it in p)
            # n_rotations == 0 through the C ABI: the plain result, no angle block
            arr = (_native.tt_image * len(pages))(*[_native.image_struct(p) for p in pages])
            ptrs = (C.c_void_p * len(pages))(*[tb.ptr(m) for m in maps])
            opt = _native.tt_ocr_options(0, 0, ptrs, 0, int(scores))
            res = C.POINTER(_native.tt_result)()
            c3, (h3, d3) = tb.launch_count(), _io()
            tb.check(lib.tt_ocr_pages_oriented(engine._h, arr, len(pages), C.byref(opt), None, 0, None, 0, C.byref(res)),
                     "tt_ocr_pages_oriented")
            c4, (h4, d4) = tb.launch_count(), _io()
            try:
                assert c4 - c3 == c1 - c0 and h4 - h3 == h1 - h0 and d4 - d3 == d1 - d0
                assert [[res.contents.pages[p].items[i].text.decode("latin-1") for i in range(res.contents.pages[p].n_items)]
                        for p in range(len(pages))] == [[it["text"] for it in p] for p in plain]
                a = C.c_int()
                assert lib.tt_item_angle(res, 0, 0, C.byref(a)) != 0
                assert b"without rotation" in lib.tt_last_error()
            finally:
                lib.tt_result_free(res)
            # with rotations: boxes, det_score and order unchanged; D2H per word = the plain D2H + 4 bytes
            for rot in ([180], [90, 180, 270]):
                _, (h5, d5) = tb.launch_count(), _io()
                got = engine.ocr_pages(pages, score_override=maps, scores=scores, rotation_info=rot)
                _, (h6, d6) = tb.launch_count(), _io()
                words = sum(len(p) for p in got)
                assert [[it["bbox"] for it in p] for p in got] == [[it["bbox"] for it in p] for p in plain]
                if scores:
                    assert [[it["det_score"] for it in p] for p in got] == [[it["det_score"] for it in p] for p in plain]
                assert (d6 - d5) - (d1 - d0) == 4 * words, (rot, scores, d6 - d5, d1 - d0, words)
                assert all(it["angle"] in candidate_set(rot) for p in got for it in p)
                print(f"scores={scores} rotation_info={rot}: H2D {(h6 - h5) / words:.1f} vs {(h1 - h0) / words:.1f} "
                      f"bytes per word, D2H {(d6 - d5) / words:.1f} vs {(d1 - d0) / words:.1f}")
    finally:
        lib.tt_engine_set_slots(engine._h, 0)


def test_pass_boundary(native_lib, weights_dir):
    """R = 3 candidates and more than 32 768 candidate crops in one recognition batch: whole words per pass."""
    cfg = tb.default_config()
    cfg.max_batch_pages = 64
    cfg.slots_per_gpu = 1
    eng = tb.Engine(weights_dir, cfg=cfg)
    try:
        n = 37
        pages = [synth.synth_page(i) for i in range(n)]
        maps = [synth.synth_score_maps(i) for i in range(n)]
        rot = [90, 270]
        big = eng.ocr_pages(pages, score_override=maps, scores=True, rotation_info=rot)
        assert 3 * sum(len(p) for p in big) > 32768
        small = []
        for i in range(0, n, 8):
            small += eng.ocr_pages(pages[i:i + 8], score_override=maps[i:i + 8], scores=True, rotation_info=rot)
    finally:
        eng.close()
    words = [(a, b) for pa, pb in zip(big, small) for a, b in zip(pa, pb)]
    same_text = sum(a["text"] == b["text"] for a, b in words)
    same_angle = sum(a["angle"] == b["angle"] for a, b in words)
    print(f"{len(words)} words: text equal {same_text}, angle equal {same_angle}")
    assert [[it["bbox"] for it in p] for p in big] == [[it["bbox"] for it in p] for p in small]
    assert same_text == len(words) and same_angle == len(words)


def test_detect_only_with_rotations(engine):
    pages, maps = _pages()
    boxes = engine.ocr_pages(pages[:3], score_override=maps[:3], detect_only=True)
    got = engine.ocr_pages(pages[:3], score_override=maps[:3], detect_only=True, rotation_info=[90, 180])
    assert [[{k: v for k, v in it.items() if k != "angle"} for it in p] for p in got] == boxes
    assert all(it["angle"] == -1 for p in got for it in p) and sum(len(p) for p in got) > 0
    got = engine.ocr_pages(pages[:3], score_override=maps[:3], detect_only=True, scores=True, rotation_info=[180])
    assert all(it["angle"] == -1 and it["conf"] is None for p in got for it in p)


def test_against_the_oracle(engine, oracle_models):
    """Strings against the oracle's oriented path; the angle wherever the oracle's margin between its best and second
    candidate exceeds the 2-Lipschitz bound of log conf in the logits' error (test_scores_gpu's bound)."""
    _, parseq = oracle_models
    fx = _fixtures()
    from oracle import imagemaps

    rot = [90, 180, 270]
    same = total = angle_checked = 0
    for key in ("funsd_91372360", "table_english", "rotated_text"):   # the oracle's PARSeq runs on the CPU
        page = np.ascontiguousarray(fx[f"{key}.img"])
        maps = np.ascontiguousarray(imagemaps.maps_f32(fx[f"{key}.maps_u8"]))
        craft = lambda x: (torch.zeros(1, x.shape[2] // 2, x.shape[3] // 2, 2), None)  # noqa: E731  (overridden)
        with torch.no_grad():
            ref = image_to_data_oriented(page.copy(), craft, parseq, rot, score_override=(maps[..., 0], maps[..., 1]))
        got = engine.ocr_pages([page], score_override=[maps], scores=True, rotation_info=rot)[0]
        assert [g["bbox"] for g in got] == [r["bbox"] for r in ref]
        _, st = _oracle(page, maps)
        cands = candidate_set(rot)
        crops = np.stack([candidate_crop(page, r, a) for r in st.crop_rects for a in cands])
        logits, ids = engine.parseq_forward(crops)
        for w, (g, r) in enumerate(zip(got, ref)):
            total += 1
            same += g["text"] == r["text"]
            logc, bound = [], []
            for c in range(len(cands)):
                lr = r["logits"][c].astype(np.float64)
                le = logits[w * len(cands) + c].astype(np.float64)
                z = np.flatnonzero(lr.argmax(-1) == 0)
                e = int(z[0]) if len(z) else 25
                t = np.arange(e + 1)
                pr = 1.0 / np.exp(lr - lr.max(-1, keepdims=True)).sum(-1)
                logc.append(float(np.log(pr[t]).sum()))
                ok = np.array_equal(ids[w * len(cands) + c, t], lr.argmax(-1)[t])
                bound.append(float(2.0 * np.abs(le[t] - lr[t]).max(-1).sum()) if ok else math.inf)
            b0 = int(np.argmax(logc))   # the engine must pick it when it beats every other candidate by both bounds
            if all(logc[b0] - logc[c] > bound[b0] + bound[c] + 1e-6 for c in range(len(cands)) if c != b0):
                angle_checked += 1
                assert g["angle"] == cands[b0], (key, w, logc, bound)
    print(f"oracle: {same}/{total} strings equal, angle checked for {angle_checked} words")
    assert same >= 0.8 * total and total > 100


def test_bindings_against_engine(engine, weights_dir, native_lib):
    sys.path.insert(0, str(_native.LIB_PATH.parent))
    import pytuatara

    fx = _fixtures()
    pages = [np.ascontiguousarray(fx["resume_example.img"])] + \
        [np.ascontiguousarray(synth.synth_page(s)[:h, :w]) for s, (h, w) in ((0, (607, 763)), (2, (754, 1000)))]
    for rot, kw in (([180], {}), ([90, 180, 270], dict(allowlist="0123456789")), ([], {})):
        for page in pages:
            want_s = engine.ocr_pages([page], scores=True, rotation_info=rot, **kw)[0]
            want = [dict(text=s["text"], bbox=s["bbox"], angle=s["angle"]) for s in want_s]
            assert engine.ocr_pages([page], rotation_info=rot, **kw)[0] == want
            assert pytuatara.image_to_data(page.copy(), weights_dir, "outputs", rotation_info=rot, **kw) == want
            assert tb.image_to_data(page, weights_dir, "outputs", rotation_info=rot, **kw) == want
            assert pytuatara.image_to_data_scored(page.copy(), weights_dir, "outputs", rotation_info=rot, **kw) == want_s
            assert tb.image_to_data_scored(page, weights_dir, "outputs", rotation_info=rot, **kw) == want_s
        want = engine.ocr_pages(pages, rotation_info=rot, **kw)
        assert pytuatara.images_to_data(pages, weights_dir, "outputs", rotation_info=rot, **kw) == want
        assert tb.images_to_data(pages, weights_dir, "outputs", rotation_info=rot, **kw) == want
        want_s = engine.ocr_pages(pages, scores=True, rotation_info=rot, **kw)
        assert pytuatara.images_to_data_scored(pages, weights_dir, "outputs", rotation_info=rot, **kw) == want_s
        assert tb.images_to_data_scored(pages, weights_dir, "outputs", rotation_info=rot, **kw) == want_s
    # an invalid angle: the error names it (ctypes) / the soft failure (pytuatara)
    with pytest.raises(tb.TuataraError, match="45"):
        engine.ocr_pages(pages[:1], rotation_info=[45])
    assert pytuatara.image_to_data(pages[0].copy(), weights_dir, "outputs", rotation_info=[45]) == []
