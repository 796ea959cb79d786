"""The contrast re-read on the GPU: the stretch bit for bit against the EasyOCR-derived reference, k_contrast_select
against the host rule, contrast_ths = 0 against the path without it, and tt_ocr_pages_contrast end to end against a host
recomputation from the first read, the reference stretch and the stage entry points; the pass boundary, detect_only,
the oracle and the bindings."""
import sys

import numpy as np
import pytest
import torch

import tuatara_b200 as tb
from contrast_ref import adjust_crop, image_to_data_contrast, keep_second, reread_words
from orient_ref import conf_of
from test_charset_gpu import _io
from test_contrast_cpu import _edge_crops
from test_scores_gpu import _fixtures, _oracle, _pages
from tuatara_b200 import _native, synth

pytestmark = pytest.mark.gpu

LEXICON_WORDS = ["TOTAL", "INVOICE", "Date", "2024", "Name", "Address", "No.", "amount", "A1", "x"]


def _faded(page):
    """The page squeezed into the band 100..140: every crop of it has low contrast."""
    return np.ascontiguousarray((100 + page.astype(np.int32) * 40 // 255).astype(np.uint8))


def _band_crops():
    """Grey crops with chosen percentiles: 411 pixels at lo (410 at lo and one at lo + 1 for a half-integer low), the
    rest at hi.  contrast = (hi - lo) / (hi + lo): 20 / 60 is exactly 0.5, 20 / 61 just above, 20 / 59 just below."""
    out = []
    for lo, hi, half in ((20, 60, False), (20, 61, False), (20, 59, False), (20, 60, True), (3, 4, False), (0, 9, True),
                         (250, 255, True), (0, 255, False), (100, 100, False)):
        g = np.full(4096, hi, np.uint8)
        g[:411] = lo
        if half:
            g[410] = lo + 1
        np.random.default_rng(lo * 1000 + hi).shuffle(g)
        out.append(np.repeat(g.reshape(32, 128, 1), 3, axis=2))
    return out


def _check_stretch(crops, adjust):
    got, flags = tb.contrast_adjust(crops, adjust)
    n = 0
    for i, c in enumerate(crops):
        want, s = adjust_crop(c, adjust)
        assert bool(flags[i]) == s, (i, adjust)
        assert got[i].tobytes() == want.tobytes(), (i, adjust, int((got[i] != want).sum()))
        n += s
    return n


def test_stretch_bit_exact(native_lib):
    pages, maps = _pages()
    crops = []
    for k in (2, 3, 5):   # fixture pages and their faded versions, cut where the path cuts them
        _, st = _oracle(pages[k], maps[k])
        crops += list(tb.crop_resize(pages[k], st.crop_rects[:150]))
        crops += list(tb.crop_resize(_faded(pages[k]), st.crop_rects[:150]))
    crops += _band_crops() + _edge_crops(np.random.default_rng(3))
    crops += list(np.random.default_rng(4).integers(0, 256, (200, 32, 128, 3), dtype=np.uint8))
    crops = np.ascontiguousarray(np.stack(crops))
    stretched = {a: _check_stretch(crops, a) for a in (0.5, 0.1, 1.0, 0.3)}
    band = np.stack(_band_crops())
    _, flags = tb.contrast_adjust(band, 0.5)
    assert flags[:3].tolist() == [False, False, True]   # exactly at 0.5, just above, just below
    # adjust_contrast at a crop's own contrast (in float) and the next floats around it
    for c, x in ((band[2], 39.0 / 79.0), (band[0], 0.5), (band[4], 1.0 / 10.0)):
        x = np.float32(x)
        for a in (np.nextafter(x, np.float32(0)), x, np.nextafter(x, np.float32(1))):
            _check_stretch(c[None], float(min(a, np.float32(1))))
    print(f"{len(crops)} crops, stretched per adjust_contrast: {stretched}")
    assert stretched[0.5] > 300 and stretched[1.0] > stretched[0.1]


def _select_dev(ids, p, lst, ids2, p2):
    d = [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in (ids, p, lst, ids2, p2)]
    tb.check(tb.lib().tt_contrast_select_dev(d[0].data_ptr(), d[1].data_ptr(), d[2].data_ptr(), len(lst), d[3].data_ptr(),
                                             d[4].data_ptr(), None), "tt_contrast_select_dev")
    torch.cuda.synchronize()
    return d[0].cpu().numpy(), d[1].cpu().numpy()


def test_select_matches_the_host_rule(native_lib):
    rng = np.random.default_rng(11)
    n, m = 4000, 2500
    ids = rng.integers(1, 95, (n, 26)).astype(np.int32)
    ids[rng.random(ids.shape) < 0.08] = 0
    p = rng.uniform(0.3, 1.0, (n, 26)).astype(np.float32)
    lst = np.sort(rng.choice(n, m, replace=False)).astype(np.int32)
    ids2 = rng.integers(1, 95, (m, 26)).astype(np.int32)
    ids2[rng.random(ids2.shape) < 0.08] = 0
    p2 = rng.uniform(0.3, 1.0, (m, 26)).astype(np.float32)
    for i, w in enumerate(lst):
        kind = i % 8
        if kind == 0:                              # exact tie
            ids2[i], p2[i] = ids[w], p[w]
        elif kind == 1:                            # the same conf with different ids
            ids2[i] = np.where(ids[w] == 0, 0, 9)
            p2[i] = p[w]
        elif kind == 2:                            # NaN in the first read
            p[w, 0] = np.nan
        elif kind == 3:                            # NaN in the second read
            p2[i, 0] = np.nan
        elif kind == 4:                            # both underflow to 0
            p[w], p2[i] = 1e-30, 1e-30
            ids[w], ids2[i] = 7, 7
        elif kind == 5:                            # no end class in either
            ids[w][ids[w] == 0] = 5
            ids2[i][ids2[i] == 0] = 5
    oi, op = _select_dev(ids, p, lst, ids2, p2)
    replaced = 0
    listed = set(lst.tolist())
    for w in range(n):
        if w not in listed:
            assert np.array_equal(oi[w], ids[w]) and op[w].tobytes() == p[w].tobytes()
    for i, w in enumerate(lst):
        second = keep_second(conf_of(ids[w], p[w]), conf_of(ids2[i], p2[i]))
        want_i, want_p = (ids2[i], p2[i]) if second else (ids[w], p[w])
        assert np.array_equal(oi[w], want_i) and op[w].tobytes() == want_p.tobytes(), (i, w)
        replaced += second
    print(f"{replaced} of {m} listed words replaced")
    assert 0 < replaced < m


def test_off_means_off(engine):
    pages, maps = _pages()
    lib = tb.lib()
    lib.tt_engine_set_slots(engine._h, 1)   # one slot: the recognition batches, so the launches, are deterministic
    lex = tb.Lexicon(LEXICON_WORDS)
    try:
        for scores in (False, True):
            for kw in ({}, dict(rotation_info=[90, 180, 270]), dict(lexicon=lex, allowlist="0123456789ATOL")):
                c0, (h0, d0) = tb.launch_count(), _io()
                want = engine.ocr_pages(pages, score_override=maps, scores=scores, **kw)
                c1, (h1, d1) = tb.launch_count(), _io()
                # adjust_contrast given: tt_ocr_pages_contrast with contrast_ths = 0
                got = engine.ocr_pages(pages, score_override=maps, scores=scores, contrast_ths=0.0, adjust_contrast=0.7, **kw)
                c2, (h2, d2) = tb.launch_count(), _io()
                assert got == want, (scores, kw.keys())
                assert c2 - c1 == c1 - c0 and h2 - h1 == h1 - h0 and d2 - d1 == d1 - d0, (scores, kw.keys())
    finally:
        lib.tt_engine_set_slots(engine._h, 0)


def _engine(weights_dir, rectify, **cfg_kw):
    cfg = tb.default_config()
    cfg.rectify = rectify
    cfg.slots_per_gpu = 1
    for k, v in cfg_kw.items():
        setattr(cfg, k, v)
    return tb.Engine(weights_dir, cfg=cfg)


def _host_contrast(eng, page, maps, rectify, kw, ths, adjust=0.5):
    """Every word from the first read (the path without the re-read), the reference stretch of its crop and the stage
    entry points, chosen on the host; -> (want items, the first read, indices of the words read again)."""
    first = eng.ocr_pages([page], score_override=[maps], scores=True, **kw)[0]
    _, st = _oracle(page, maps)
    crops = []
    for item, rect, box in zip(first, st.crop_rects, st.boxes):
        a = item.get("angle", 0)
        if rectify:
            crops.append(tb.crop_warp(page, np.roll(tb.rect_to_quad(box), -(a // 90), 0)[None])[0])
        else:
            crops.append(tb.crop_resize(page, [rect], [a])[0])
    crops = np.stack(crops)
    idx, adj = reread_words([it["conf"] for it in first], crops, ths, adjust)
    got_adj, flags = tb.contrast_adjust(crops, adjust)   # the stage entry point agrees on the crops the path cuts
    assert got_adj[idx].tobytes() == adj.tobytes()
    want = [dict(it) for it in first]
    if idx:
        if kw.get("lexicon") is not None:
            _, ids, p = eng.parseq_forward_lexicon(adj, kw["lexicon"])
        else:
            masks = None
            if kw.get("allowlist") is not None or kw.get("blocklist") is not None:
                masks = np.tile(tb.char_filter_mask(kw.get("allowlist"), kw.get("blocklist")), (len(adj), 1))
            ids, p = eng.parseq_forward_scores(adj, class_masks=masks)
        texts, conf, cc = tb.decode_scores(ids, p)
        for k, i in enumerate(idx):
            if keep_second(want[i]["conf"], conf[k]):
                want[i].update(text=texts[k], conf=float(conf[k]), char_conf=[float(v) for v in cc[k]])
    return want, first, idx


@pytest.mark.parametrize("rectify", [0, 1])
def test_whole_path_equals_host_recomputation(native_lib, weights_dir, rectify):
    eng = _engine(weights_dir, rectify)
    pages, maps = _pages()
    lex = tb.Lexicon(LEXICON_WORDS)
    cases = [(_faded(pages[0]), maps[0]), (_faded(pages[3]), maps[3]), (pages[2], maps[2]), (pages[1], maps[1])]
    configs = [{}, dict(allowlist="0123456789"), dict(lexicon=lex), dict(rotation_info=[90, 180, 270]),
               dict(rotation_info=[90, 180, 270], blocklist="aeiou"), dict(rotation_info=[90, 180, 270], lexicon=lex)]
    words = reread = won = 0
    try:
        for ci, (page, m) in enumerate(cases):
            for kw in configs:
                want, first, idx = _host_contrast(eng, page, m, rectify, kw, 2.0)
                for scores in (False, True):
                    got = eng.ocr_pages([page], score_override=[m], scores=scores, contrast_ths=2.0, **kw)[0]
                    assert len(got) == len(want)
                    for g, w, f in zip(got, want, first):
                        assert g["text"] == w["text"] and g["bbox"] == f["bbox"], (ci, kw.keys(), g, w)
                        assert g.get("angle") == f.get("angle")
                        if scores:
                            assert np.float32(g["conf"]).tobytes() == np.float32(w["conf"]).tobytes()
                            assert np.array_equal(np.float32(g["char_conf"]), np.float32(w["char_conf"]))
                            assert g["det_score"] == f["det_score"]
                words += len(want)
                reread += len(idx)
                won += sum(w["text"] != f["text"] or w["conf"] != f["conf"] for w, f in zip(want, first))
                if ci < 2:   # the faded pages: every crop is low contrast
                    assert len(idx) == len(want)
    finally:
        eng.close()
    print(f"rectify={rectify}: {words} words, {reread} read again, {won} took the second read")
    assert reread > 1000 and won > 0


def test_pass_boundary(native_lib, weights_dir):
    """R = 3 candidates, more than 32 768 candidate crops in one recognition batch, every word read again."""
    eng = _engine(weights_dir, 0, max_batch_pages=64)
    try:
        n = 37
        pages = [_faded(synth.synth_page(i)) for i in range(n)]
        maps = [synth.synth_score_maps(i) for i in range(n)]
        kw = dict(scores=True, rotation_info=[90, 270], contrast_ths=2.0)
        big = eng.ocr_pages(pages, score_override=maps, **kw)
        assert 3 * sum(len(p) for p in big) > 32768
        small = []
        for i in range(0, n, 8):
            small += eng.ocr_pages(pages[i:i + 8], score_override=maps[i:i + 8], **kw)
    finally:
        eng.close()
    assert big == small


def test_detect_only_unchanged(engine):
    pages, maps = _pages()
    boxes = engine.ocr_pages(pages[:3], score_override=maps[:3], detect_only=True)
    assert engine.ocr_pages(pages[:3], score_override=maps[:3], detect_only=True, contrast_ths=2.0) == boxes
    got = engine.ocr_pages(pages[:3], score_override=maps[:3], detect_only=True, scores=True, contrast_ths=0.1)
    assert all(it["conf"] is None for p in got for it in p) and sum(len(p) for p in got) > 0


def test_against_the_oracle(engine, oracle_models):
    _, parseq = oracle_models
    fx = _fixtures()
    from oracle import imagemaps

    same = total = reread = 0
    for key in ("funsd_91372360", "table_english"):   # the oracle's PARSeq runs on the CPU
        page = _faded(fx[f"{key}.img"])
        maps = np.ascontiguousarray(imagemaps.maps_f32(fx[f"{key}.maps_u8"]))
        craft = lambda x: (torch.zeros(1, x.shape[2] // 2, x.shape[3] // 2, 2), None)  # noqa: E731  (overridden)
        with torch.no_grad():
            ref = image_to_data_contrast(page.copy(), craft, parseq, 2.0, score_override=(maps[..., 0], maps[..., 1]))
        got = engine.ocr_pages([page], score_override=[maps], contrast_ths=2.0)[0]
        assert [g["bbox"] for g in got] == [r["bbox"] for r in ref]
        total += len(ref)
        same += sum(g["text"] == r["text"] for g, r in zip(got, ref))
        reread += sum(r["reread"] for r in ref)
    print(f"oracle: {same}/{total} strings equal, {reread} read again")
    assert same >= 0.8 * total and total > 50 and reread == total


def test_bindings_against_engine(engine, weights_dir, native_lib):
    sys.path.insert(0, str(_native.LIB_PATH.parent))
    import pytuatara

    fx = _fixtures()
    pages = [_faded(fx["resume_example.img"]), np.ascontiguousarray(synth.synth_page(0)[:607, :763]),
             _faded(synth.synth_page(2)[:754, :1000])]
    for kw in (dict(contrast_ths=2.0), dict(contrast_ths=0.1, adjust_contrast=0.8, rotation_info=[180]),
               dict(contrast_ths=2.0, allowlist="0123456789")):
        for page in pages:
            want_s = engine.ocr_pages([page], scores=True, **kw)[0]
            want = [{k: v for k, v in s.items() if k in ("text", "bbox", "angle")} for s in want_s]
            assert engine.ocr_pages([page], **kw)[0] == want
            assert pytuatara.image_to_data(page.copy(), weights_dir, "outputs", **kw) == want
            assert tb.image_to_data(page, weights_dir, "outputs", **kw) == want
            assert pytuatara.image_to_data_scored(page.copy(), weights_dir, "outputs", **kw) == want_s
            assert tb.image_to_data_scored(page, weights_dir, "outputs", **kw) == want_s
        want = engine.ocr_pages(pages, **kw)
        assert pytuatara.images_to_data(pages, weights_dir, "outputs", **kw) == want
        assert tb.images_to_data(pages, weights_dir, "outputs", **kw) == want
        want_s = engine.ocr_pages(pages, scores=True, **kw)
        assert pytuatara.images_to_data_scored(pages, weights_dir, "outputs", **kw) == want_s
        assert tb.images_to_data_scored(pages, weights_dir, "outputs", **kw) == want_s
    # an invalid value: the error names it (ctypes) / the soft failure (pytuatara)
    with pytest.raises(tb.TuataraError, match="contrast_ths is -1"):
        engine.ocr_pages(pages[:1], contrast_ths=-1.0)
    with pytest.raises(tb.TuataraError, match="adjust_contrast is 0"):
        engine.ocr_pages(pages[:1], contrast_ths=0.1, adjust_contrast=0.0)
    assert pytuatara.image_to_data(pages[0].copy(), weights_dir, "outputs", contrast_ths=float("nan")) == []
