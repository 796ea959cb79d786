"""Character filters on the GPU: the masked greedy decode (fused and unfused AR step, refinement head) against its own
logits and the oracle, bit-identity of a filter that allows every class, and the filtered entry points end to end."""
import ctypes as C
import string
import sys

import numpy as np
import pytest
import torch

import tuatara_b200 as tb
from charset_ref import masked_argmax, masked_forward, masked_pmax, words_to_bool
from test_scores_gpu import _crops, _fixtures, _pages
from tuatara_b200 import _native, synth

pytestmark = pytest.mark.gpu

PRINTABLE = "".join(chr(c) for c in range(32, 127))
DIGITS = string.digits
FILTERS = [(None, None), (DIGITS, None), (string.ascii_uppercase, None), ("", None), (None, string.ascii_lowercase),
           (string.ascii_letters, "aeiouAEIOU")]


def _masks(n, seed):
    """Per-crop class masks drawn from FILTERS: uint32 [n, 4] and bool [n, 95]."""
    pick = np.random.default_rng(seed).integers(0, len(FILTERS), n)
    table = np.stack([tb.char_filter_mask(a, b) for a, b in FILTERS])
    w = np.ascontiguousarray(table[pick])
    return w, words_to_bool(w)


def _forward_masked(engine, crops, masks, forced=None):
    """tt_parseq_forward_masked with every output: (logits [n, 26, 95], ids [n, 26], pmax [n, 26])."""
    x = np.ascontiguousarray(crops, np.uint8)
    n = len(x)
    logits = np.empty((n, 26, 95), np.float32)
    ids = np.empty((n, 26), np.int32)
    p = np.empty((n, 26), np.float32)
    ft = None if forced is None else np.ascontiguousarray(forced, np.int32)
    m = np.ascontiguousarray(masks, np.uint32)
    tb.check(tb.lib().tt_parseq_forward_masked(engine._h, tb.ptr(x), n, tb.ptr(ft), tb.ptr(m), tb.ptr(logits), tb.ptr(ids),
                                               tb.ptr(p)), "tt_parseq_forward_masked")
    return logits, ids, p


def _io():
    h2d, d2h = C.c_ulonglong(), C.c_ulonglong()
    tb.lib().tt_io_bytes(C.byref(h2d), C.byref(d2h))
    return h2d.value, d2h.value


def _obeys(text, allow, block):
    return all((allow is None or ch in allow) and (block is None or ch not in block) for ch in text)


@pytest.mark.parametrize("fused", ["1", "0"])
@pytest.mark.parametrize("n", [300, 600])   # 600: two half-batches on two streams (fused path)
def test_all_allowing_mask_is_bit_identical(engine, monkeypatch, fused, n):
    monkeypatch.setenv("TT_DEC_FUSED", fused)
    crops = _crops(n, seed=41)
    ones = np.tile(tb.char_filter_mask(PRINTABLE), (n, 1))
    assert np.array_equal(ones[0], tb.char_filter_mask())
    l0, i0 = engine.parseq_forward(crops)
    l1, i1 = engine.parseq_forward(crops, class_masks=ones)
    assert l1.tobytes() == l0.tobytes() and i1.tobytes() == i0.tobytes()
    j0, p0 = engine.parseq_forward_scores(crops)
    j1, p1 = engine.parseq_forward_scores(crops, class_masks=ones)
    assert j1.tobytes() == j0.tobytes() and p1.tobytes() == p0.tobytes()
    assert np.array_equal(j0, i0)


def test_all_allowing_filter_end_to_end(engine):
    """Same items and scores, the same launches, 16 more bytes per crop host to device and nothing more back."""
    pages, maps = _pages()
    lib = tb.lib()
    lib.tt_engine_set_slots(engine._h, 1)   # one slot: the recognition batches, so the launches, are deterministic
    try:
        c0, (h0, d0) = tb.launch_count(), _io()
        plain = engine.ocr_pages(pages, score_override=maps, scores=True)
        c1, (h1, d1) = tb.launch_count(), _io()
        filt = engine.ocr_pages(pages, score_override=maps, scores=True, allowlist=PRINTABLE)
        c2, (h2, d2) = tb.launch_count(), _io()
    finally:
        lib.tt_engine_set_slots(engine._h, 0)
    assert filt == plain
    crops = sum(len(p) for p in plain)
    assert crops > 600
    assert c2 - c1 == c1 - c0
    assert d2 - d1 == d1 - d0
    assert (h2 - h1) - (h1 - h0) == 16 * crops


@pytest.mark.parametrize("fused", ["1", "0"])
def test_refinement_head_under_teacher_forcing(engine, monkeypatch, fused):
    monkeypatch.setenv("TT_DEC_FUSED", fused)
    n = 300
    crops = _crops(n, seed=43)
    _, free_ids = engine.parseq_forward(crops)
    forced = np.ascontiguousarray(free_ids[:, :25])
    w, mb = _masks(n, seed=44)
    l0, _ = engine.parseq_forward(crops, forced)
    l1, i1, p1 = _forward_masked(engine, crops, w, forced)
    assert l1.tobytes() == l0.tobytes()
    assert np.array_equal(i1, masked_argmax(l1, mb[:, None, :]))
    assert all(mb[i][i1[i]].all() for i in range(n))
    want = masked_pmax(l1, mb[:, None, :])
    err = np.abs(p1 - want)
    print("masked pmax vs float64: max abs", float(err.max()))
    assert (err <= 1e-6 + 1e-5 * want).all()
    # the AR logits under forcing do not depend on the masks either
    monkeypatch.setenv("TT_PARSEQ_AR_LOGITS", "1")
    a0, _ = engine.parseq_forward(crops, forced)
    a1, _, _ = _forward_masked(engine, crops, w, forced)
    assert a1.tobytes() == a0.tobytes()


def _ar_self_consistency(engine, monkeypatch, crops, w, mb, refinement_logits=True):
    """Free masked run vs a re-run forced with the host's masked argmax of the free run's AR logits: the AR logits up
    to each crop's end step, the ids and p are byte-identical, so every token the device fed back was the masked argmax."""
    monkeypatch.setenv("TT_PARSEQ_AR_LOGITS", "1")
    ar, ids, p = _forward_masked(engine, crops, w)
    fed = masked_argmax(ar, mb[:, None, :])                       # [n, 26]: the token each step should feed back
    z = fed == 0
    end = np.where(z.any(-1), z.argmax(-1), 25)
    forced = np.ascontiguousarray(fed[:, :25]).astype(np.int32)
    forced[np.arange(25)[None, :] > end[:, None]] = 0             # after the end: any value
    ar_f, ids_f, p_f = _forward_masked(engine, crops, w, forced)
    bad = [i for i in range(len(crops)) if ar_f[i, :end[i] + 1].tobytes() != ar[i, :end[i] + 1].tobytes()]
    assert not bad, (len(bad), bad[:10])
    assert ids_f.tobytes() == ids.tobytes() and p_f.tobytes() == p.tobytes()
    assert all(mb[i][ids[i]].all() for i in range(len(crops)))
    if refinement_logits:
        monkeypatch.setenv("TT_PARSEQ_AR_LOGITS", "0")
        lr, _, _ = _forward_masked(engine, crops, w)
        lr_f, _, _ = _forward_masked(engine, crops, w, forced)
        assert lr_f.tobytes() == lr.tobytes()
    return end


@pytest.mark.parametrize("fused", ["1", "0"])
@pytest.mark.parametrize("n", [300, 600])
def test_ar_feedback_is_the_masked_argmax(engine, monkeypatch, fused, n):
    monkeypatch.setenv("TT_DEC_FUSED", fused)
    crops = _crops(n, seed=45)
    w, mb = _masks(n, seed=46)
    end = _ar_self_consistency(engine, monkeypatch, crops, w, mb)
    print("end steps: median", float(np.median(end)), "crops ending before the last step", int((end < 25).sum()))


def test_ar_feedback_across_the_pass_boundary(engine, monkeypatch):
    """A request over kMaxCropsPerPass (32 768 crops per PARSeq pass): the second pass reads its own crops' masks."""
    crops = _crops(300, seed=47)
    big = np.concatenate([crops] * 110)[:32768 + 200]
    big[300:] = np.random.default_rng(48).integers(0, 256, big[300:].shape, dtype=np.uint8)
    w, mb = _masks(len(big), seed=49)
    _ar_self_consistency(engine, monkeypatch, big, w, mb, refinement_logits=False)


def test_filters_end_to_end(engine):
    pages, maps = _pages()
    plain = engine.ocr_pages(pages, score_override=maps, scores=True)
    changed = nonempty = 0
    for allow, block in [(DIGITS, None), (None, string.ascii_lowercase), (string.ascii_uppercase + DIGITS, "O0")]:
        got = engine.ocr_pages(pages, score_override=maps, scores=True, allowlist=allow, blocklist=block)
        for g_page, p_page in zip(got, plain):
            assert [g["bbox"] for g in g_page] == [p["bbox"] for p in p_page]
            assert [g["det_score"] for g in g_page] == [p["det_score"] for p in p_page]
            for g, p in zip(g_page, p_page):
                assert _obeys(g["text"], allow, block), (allow, block, g["text"])
                assert len(g["char_conf"]) == len(g["text"]) and g["conf"] is not None
                nonempty += bool(g["text"])
                changed += g["text"] != p["text"]
        print(allow, block, "non-empty texts so far:", nonempty, "changed:", changed)
    # the seeded random-init model often prefers the end class once its letters are forbidden: a digits-only word is
    # then empty, which obeys the filter; the other filters keep text to check
    assert nonempty > 100 and changed > 0
    # a filter per page, None entries included: each page as if it ran alone with its own filter
    allow = [DIGITS, None, string.ascii_uppercase, None, "", None, "abcdefg"]
    block = [None, string.ascii_lowercase, None, None, None, None, "b"]
    batch = engine.ocr_pages(pages, score_override=maps, allowlist=allow, blocklist=block)
    for k in range(len(pages)):
        alone = engine.ocr_pages([pages[k]], score_override=[maps[k]], allowlist=allow[k], blocklist=block[k])[0]
        assert batch[k] == alone, k
        assert all(_obeys(it["text"], allow[k], block[k]) for it in batch[k])
        if allow[k] is None and block[k] is None:
            assert batch[k] == [dict(text=p["text"], bbox=p["bbox"]) for p in plain[k]], k
    assert all(it["text"] == "" for it in batch[4]) and len(batch[4]) > 0
    # detect_only ignores a filter
    boxes = engine.ocr_pages(pages[:3], score_override=maps[:3], detect_only=True)
    assert engine.ocr_pages(pages[:3], score_override=maps[:3], detect_only=True, allowlist=DIGITS) == boxes


def test_masked_decode_against_the_oracle(engine, oracle_models):
    _, parseq = oracle_models
    crops = _crops(48, seed=33)
    nonempty = 0
    x = torch.from_numpy(crops).permute(0, 3, 1, 2).float().div(255.0)
    for allow, block in [(DIGITS, None), (None, string.ascii_lowercase)]:
        m = tb.char_filter_mask(allow, block)
        mb = words_to_bool(m)
        w = np.tile(m, (len(crops), 1))
        mt = torch.from_numpy(np.tile(mb, (len(crops), 1)))
        _, ids = engine.parseq_forward(crops, class_masks=w)
        taps = {}
        ref = masked_forward(parseq, x, mt, taps=taps).numpy()
        got_s, ref_s = tb.decode_ids(ids), tb.decode_ids(masked_argmax(ref, mb).astype(np.int32))
        same = sum(a == b for a, b in zip(got_s, ref_s))
        print(allow, block, "free-running strings equal to the masked oracle:", same, "of", len(crops))
        assert same >= 0.8 * len(crops)
        assert all(_obeys(s, allow, block) for s in got_s)
        nonempty += sum(bool(s) for s in got_s)
        # teacher forced with the oracle's masked AR tokens: the refinement ids wherever the oracle's margin is clear
        forced = taps["ar_tokens"][:, 1:].numpy().astype(np.int32)
        _, ids_f = engine.parseq_forward(crops, forced, class_masks=w)
        ref_f = masked_forward(parseq, x, mt, forced_tokens=torch.from_numpy(forced).long()).numpy()
        top2 = np.sort(np.where(mb, ref_f, -np.inf), -1)[..., -2:]
        clear = (top2[..., 1] - top2[..., 0]) > 0.5
        want = masked_argmax(ref_f, mb)
        print("positions with a clear margin:", int(clear.sum()), "of", clear.size)
        assert clear.sum() > clear.size // 2
        assert np.array_equal(ids_f[clear], want[clear])
    print("non-empty filtered strings:", nonempty)
    assert nonempty > 0


def test_filtered_bindings_against_engine(engine, weights_dir, native_lib):
    sys.path.insert(0, str(_native.LIB_PATH.parent))
    import pytuatara

    fx = _fixtures()
    pages = [np.ascontiguousarray(fx["resume_example.img"])] + \
        [np.ascontiguousarray(synth.synth_page(s)[:h, :w]) for s, (h, w) in ((0, (607, 763)), (2, (754, 1000)))]
    for allow, block in [(DIGITS, None), (None, "aeiou"), (string.ascii_uppercase, "XYZ")]:
        kw = dict(allowlist=allow, blocklist=block)
        for page in pages:
            want = engine.ocr_pages([page], **kw)[0]
            assert pytuatara.image_to_data(page.copy(), weights_dir, "outputs", **kw) == want
            assert tb.image_to_data(page, weights_dir, "outputs", **kw) == want
            want_s = engine.ocr_pages([page], scores=True, **kw)[0]
            assert pytuatara.image_to_data_scored(page.copy(), weights_dir, "outputs", **kw) == want_s
            assert tb.image_to_data_scored(page, weights_dir, "outputs", **kw) == want_s
            assert [dict(text=s["text"], bbox=s["bbox"]) for s in want_s] == want
        want = engine.ocr_pages(pages, **kw)
        assert pytuatara.images_to_data(pages, weights_dir, "outputs", **kw) == want
        assert tb.images_to_data(pages, weights_dir, "outputs", **kw) == want
    allow, block = [DIGITS, None, "ABCDEFabcdef"], ["5", "aeiou", None]
    want = engine.ocr_pages(pages, allowlist=allow, blocklist=block)
    assert pytuatara.images_to_data(pages, weights_dir, "outputs", allowlist=allow, blocklist=block) == want
    assert tb.images_to_data(pages, weights_dir, "outputs", allowlist=allow, blocklist=block) == want
    want_s = engine.ocr_pages(pages, scores=True, allowlist=allow, blocklist=block)
    assert pytuatara.images_to_data_scored(pages, weights_dir, "outputs", allowlist=allow, blocklist=block) == want_s
    assert tb.images_to_data_scored(pages, weights_dir, "outputs", allowlist=allow, blocklist=block) == want_s
    assert sum(len(p) for p in want) > 0
    # n_filters outside {0, 1, n_pages}, and NULL filters with n_filters > 0, fail with a message
    lib = tb.lib()
    arr = (_native.tt_image * 2)(*[_native.image_struct(p) for p in pages[:2]])
    f = (_native.tt_char_filter * 3)(*[_native.tt_char_filter(b"0", None)] * 3)
    res = C.POINTER(_native.tt_result)()
    assert lib.tt_ocr_pages_filtered(engine._h, arr, 2, None, f, 3, C.byref(res)) != 0
    assert b"n_filters" in lib.tt_last_error()
    assert lib.tt_ocr_pages_filtered(engine._h, arr, 2, None, None, 2, C.byref(res)) != 0
    assert b"filters is NULL" in lib.tt_last_error()
    assert lib.tt_ocr_pages_filtered(engine._h, arr, 2, None, f, 2, C.byref(res)) == 0
    try:
        assert res.contents.n_pages == 2
    finally:
        lib.tt_result_free(res)
