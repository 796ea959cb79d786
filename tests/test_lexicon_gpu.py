"""Lexicons on the GPU: k_lexicon_walk against the reference walk, bit-identity of one-state automata, the refinement
walk under teacher forcing, the AR feedback as the walked choice, the lexicon entry points end to end, the oracle and the
bindings."""
import ctypes as C
import string
import sys

import numpy as np
import pytest
import torch

import tuatara_b200 as tb
from charset_ref import words_to_bool
from lexicon_ref import lexicon_forward, make_trie, step, text_of, walk
from test_charset_gpu import _io
from test_scores_gpu import _crops, _fixtures, _pages
from tuatara_b200 import _native, synth

pytestmark = pytest.mark.gpu

TABLE = None


def _table():
    global TABLE
    if TABLE is None:
        TABLE = tb.tokenizer_table()
    return TABLE[0], TABLE[1]


def _words(n, seed, alphabet=string.ascii_letters + string.digits + "-\\'", lo=1, hi=12):
    rng = np.random.default_rng(seed)
    a = list(alphabet)
    return ["".join(rng.choice(a, int(rng.integers(lo, hi + 1)))) for _ in range(n)]


def _walk_dev(lex, logits):
    x = torch.from_numpy(np.ascontiguousarray(logits, np.float32)).cuda()
    n = x.shape[0]
    ids = torch.empty((n, 26), dtype=torch.int32, device="cuda")
    p = torch.empty((n, 26), dtype=torch.float32, device="cuda")
    tb.check(tb.lib().tt_lexicon_walk_dev(lex._h, x.data_ptr(), n, ids.data_ptr(), p.data_ptr(), None), "tt_lexicon_walk_dev")
    torch.cuda.synchronize()
    return ids.cpu().numpy(), p.cpu().numpy()


def _check_walk(lex, trie, logits):
    ids, p = _walk_dev(lex, logits)
    for i in range(len(logits)):
        want_ids, want_p = walk(logits[i], trie)
        assert np.array_equal(ids[i], want_ids), (i, ids[i], want_ids)
        nan = np.isnan(want_p)
        assert np.array_equal(np.isnan(p[i]), nan), i
        err = np.abs(p[i][~nan] - want_p[~nan])
        assert (err <= 1e-6 + 1e-5 * want_p[~nan]).all(), (i, float(err.max()))
    return ids


def test_walk_kernel_against_the_reference():
    itos, eos = _table()
    rng = np.random.default_rng(3)
    cases = [
        (["a", "ab", "abc"], None),                       # prefix words
        (["x" * 25, "y" * 25, "xy"], None),               # 25-byte words
        (["a\\b", "\\", "\\\\", "b\\"], None),            # backslash, printed by classes 69 and 87
        (_words(500, 4), None),
        (_words(500, 5), tb.char_filter_mask(string.ascii_lowercase + string.digits)),   # folded lexicon
    ]
    for words, mask in cases:
        kept = words if mask is None else [w for w in words if all(ch in string.ascii_lowercase + string.digits for ch in w)]
        lex = tb.Lexicon(kept)
        trie = make_trie(kept, itos, eos, None if mask is None else words_to_bool(mask))
        logits = rng.normal(0, 3, (64, 26, 95)).astype(np.float32)
        logits[:8] = np.round(logits[:8])                  # ties
        logits[8:12] = np.float32(np.nan)                  # all NaN
        logits[12:16] = -np.inf                            # all -inf
        logits[16:20, :, [69, 87]] += 20.0                 # favour backslash ...
        logits[20:24, :, 87] += 1.0                        # ... either class
        logits[24:28, 3:, 0] += 30.0                       # early ends
        logits[28:32, ::2, :] = np.float32(np.nan)         # NaN rows between finite ones
        ids = _check_walk(lex, trie, logits)
        for row in ids:
            t = text_of(row, itos, eos)
            assert t in set(kept) or 0 not in row, t


def test_one_state_automata_are_bit_identical(engine, monkeypatch):
    """All-NULL lexicon requests equal tt_ocr_pages_ex (and a filter-only page tt_ocr_pages_filtered): items, scores and
    angles; fused and unfused; with one slot 4 more bytes per crop host to device plus the table."""
    pages, maps = _pages()
    lib = tb.lib()
    for fused in ("1", "0"):
        monkeypatch.setenv("TT_DEC_FUSED", fused)
        lib.tt_engine_set_slots(engine._h, 1)
        try:
            h0 = _io()[0]
            plain = engine.ocr_pages(pages, score_override=maps, scores=True)
            h1 = _io()[0]
            null = engine.ocr_pages(pages, score_override=maps, scores=True, lexicon=[None] * len(pages))
            h2 = _io()[0]
        finally:
            lib.tt_engine_set_slots(engine._h, 0)
        assert null == plain
        crops = sum(len(p) for p in plain)
        table = 4 * (5 * 2 + 95 + 95)   # done state + one state allowing the 95 classes
        assert (h2 - h1) - (h1 - h0) == table + 4 * crops
        rot = engine.ocr_pages(pages, score_override=maps, scores=True, rotation_info=[180])
        assert engine.ocr_pages(pages, score_override=maps, scores=True, rotation_info=[180], lexicon=[None] * len(pages)) == rot
        allow = [string.digits, None, string.ascii_uppercase, None, None, "abc", None]
        filt = engine.ocr_pages(pages, score_override=maps, scores=True, allowlist=allow)
        assert engine.ocr_pages(pages, score_override=maps, scores=True, allowlist=allow, lexicon=[None] * len(pages)) == filt


def test_refinement_under_teacher_forcing(engine, monkeypatch):
    itos, eos = _table()
    n = 300
    crops = _crops(n, seed=51)
    words = _words(2000, 52)
    lex = tb.Lexicon(words)
    trie = make_trie(words, itos, eos)
    _, free = engine.parseq_forward(crops)
    forced = np.ascontiguousarray(free[:, :25])
    for fused in ("1", "0"):
        monkeypatch.setenv("TT_DEC_FUSED", fused)
        l0, _ = engine.parseq_forward(crops, forced)
        l1, ids, p = engine.parseq_forward_lexicon(crops, lex, forced)
        assert l1.tobytes() == l0.tobytes()
        for i in range(n):
            want_ids, want_p = walk(l1[i], trie)
            assert np.array_equal(ids[i], want_ids), i
            assert (np.abs(p[i] - want_p) <= 1e-6 + 1e-5 * want_p).all(), i
            assert text_of(ids[i], itos, eos) in set(words)
        monkeypatch.setenv("TT_PARSEQ_AR_LOGITS", "1")
        a0, _ = engine.parseq_forward(crops, forced)
        a1, _, _ = engine.parseq_forward_lexicon(crops, lex, forced)
        assert a1.tobytes() == a0.tobytes()
        monkeypatch.setenv("TT_PARSEQ_AR_LOGITS", "0")


def _ar_self_consistency(engine, monkeypatch, crops, lex, trie, words):
    """Free lexicon run vs a re-run forced with the host's walk of the free run's AR logits: the AR logits up to each
    crop's end step are byte-identical, so every token the device fed back was the walked choice; the refinement ids of
    the free run spell a word."""
    itos, eos = _table()
    monkeypatch.setenv("TT_PARSEQ_AR_LOGITS", "1")
    ar, ids, p = engine.parseq_forward_lexicon(crops, lex)
    n = len(crops)
    fed = np.zeros((n, 25), np.int32)
    end = np.full(n, 25)
    for i in range(n):
        s = 0
        for t in range(25):
            c, s, _ = step(trie, s, ar[i, t])
            fed[i, t] = c
            if c == 0:
                end[i] = t
                break
    ar_f, _, _ = engine.parseq_forward_lexicon(crops, lex, fed)
    bad = [i for i in range(n) if ar_f[i, :end[i] + 1].tobytes() != ar[i, :end[i] + 1].tobytes()]
    assert not bad, (len(bad), bad[:10])
    monkeypatch.setenv("TT_PARSEQ_AR_LOGITS", "0")
    ws = set(words)
    assert all(text_of(ids[i], itos, eos) in ws for i in range(n))
    return end


@pytest.mark.parametrize("fused", ["1", "0"])
@pytest.mark.parametrize("n", [300, 600])   # 600: two half-batches on two streams (fused path)
def test_ar_feedback_is_the_walked_choice(engine, monkeypatch, fused, n):
    itos, eos = _table()
    monkeypatch.setenv("TT_DEC_FUSED", fused)
    words = _words(3000, 53 + n)
    end = _ar_self_consistency(engine, monkeypatch, _crops(n, seed=54), tb.Lexicon(words), make_trie(words, itos, eos),
                               words)
    print("end steps: median", float(np.median(end)), "ending before the last step", int((end < 25).sum()))


def test_lexicon_across_the_pass_boundary(engine, weights_dir):
    """One recognition batch of more than 32 768 crops (two PARSeq passes), per-page lexicons: the second pass reads its
    own crops' roots, so the results equal those of batches that stay within one pass."""
    pages, maps = _pages()
    k = 120   # 300 words per synthetic page
    big_p, big_m = [pages[i % 2] for i in range(k)], [maps[i % 2] for i in range(k)]
    lexs = [tb.Lexicon(_words(200, 60 + i)) for i in range(3)]
    per = [lexs[i % 3] if i % 4 else None for i in range(k)]
    cfg = tb.default_config()
    cfg.max_batch_pages = 128
    cfg.slots_per_gpu = 1
    eng = tb.Engine(weights_dir, cfg=cfg)
    try:
        out = eng.ocr_pages(big_p, score_override=big_m, scores=True, lexicon=per)
    finally:
        eng.close()
    assert sum(len(p) for p in out) > 32768
    assert out == engine.ocr_pages(big_p, score_override=big_m, scores=True, lexicon=per)
    plain = engine.ocr_pages(big_p[:1], score_override=big_m[:1], scores=True)[0]
    assert all(out[i] == plain for i in range(0, k, 4))   # the NULL entries (all of them page 0): the plain results


def test_lexicon_end_to_end(native_lib, weights_dir, engine):
    pages, maps = _pages()
    words = _words(1000, 70) + ["a", "I", "the"]
    lex = tb.Lexicon(words)
    ws = set(words)
    for rectify in (0, 1):
        cfg = tb.default_config()
        cfg.rectify = rectify
        eng = engine if rectify == 0 else tb.Engine(weights_dir, cfg=cfg)
        for scores in (False, True):
            for rot in (None, [90, 180, 270]):
                plain = eng.ocr_pages(pages, score_override=maps, scores=scores, rotation_info=rot)
                got = eng.ocr_pages(pages, score_override=maps, scores=scores, rotation_info=rot, lexicon=lex)
                for g_page, p_page in zip(got, plain):
                    assert [g["bbox"] for g in g_page] == [p["bbox"] for p in p_page]
                    for g, p in zip(g_page, p_page):
                        assert g["text"] in ws, g["text"]
                        if scores:
                            assert g["det_score"] == p["det_score"] and len(g["char_conf"]) == len(g["text"])
                print(f"rectify={rectify} scores={scores} rot={rot}: {sum(len(p) for p in got)} items in the lexicon")
        if rectify:
            eng.close()
    # a filter folds into the lexicon: every word is from the folded list
    folded = engine.ocr_pages(pages, score_override=maps, allowlist=string.ascii_lowercase, lexicon=lex)
    low = {w for w in ws if all(ch in string.ascii_lowercase for ch in w)}
    assert all(it["text"] in low for p in folded for it in p)
    # per-page lexicons in one batch equal each page alone; detect_only ignores the lexicon
    other = tb.Lexicon(_words(50, 71, alphabet=string.digits))
    per = [lex, None, other, lex, None, other, lex]
    batch = engine.ocr_pages(pages, score_override=maps, scores=True, lexicon=per)
    for k in range(len(pages)):
        assert batch[k] == engine.ocr_pages([pages[k]], score_override=[maps[k]], scores=True, lexicon=[per[k]])[0], k
    boxes = engine.ocr_pages(pages[:3], score_override=maps[:3], detect_only=True)
    assert engine.ocr_pages(pages[:3], score_override=maps[:3], detect_only=True, lexicon=lex) == boxes


def test_lexicon_decode_against_the_oracle(engine, oracle_models):
    _, parseq = oracle_models
    itos, eos = _table()
    crops = _crops(48, seed=33)
    x = torch.from_numpy(crops).permute(0, 3, 1, 2).float().div(255.0)
    words = _words(3000, 80)
    lex, trie = tb.Lexicon(words), make_trie(words, itos, eos)
    _, ids, _ = engine.parseq_forward_lexicon(crops, lex)
    taps = {}
    ref = lexicon_forward(parseq, x, [trie] * len(crops), taps=taps).numpy()
    got_s = [text_of(r, itos, eos) for r in ids]
    ref_s = [text_of(walk(r, trie)[0], itos, eos) for r in ref]
    same = sum(a == b for a, b in zip(got_s, ref_s))
    print("free-running strings equal to the oracle's lexicon decode:", same, "of", len(crops))
    assert same >= 0.8 * len(crops)
    forced = taps["ar_tokens"][:, 1:].numpy().astype(np.int32)
    _, ids_f, _ = engine.parseq_forward_lexicon(crops, lex, forced)
    ref_f = lexicon_forward(parseq, x, [trie] * len(crops), forced_tokens=torch.from_numpy(forced).long()).numpy()
    want = np.stack([walk(r, trie)[0] for r in ref_f])
    # positions with a clear margin among the classes the walk allows there, up to the first disagreement
    clear = np.zeros(want.shape, bool)
    for i in range(len(crops)):
        s = 0
        for t in range(26):
            allow = np.ones(95, bool) if s < 0 else trie.allow[s]
            top2 = np.sort(ref_f[i, t][allow])[-2:]
            clear[i, t] = len(top2) < 2 or top2[1] - top2[0] > 0.5
            if ids_f[i, t] != want[i, t]:
                break
            _, s, _ = step(trie, s, ref_f[i, t])
    print("positions with a clear margin:", int(clear.sum()), "of", clear.size)
    assert clear.sum() > clear.size // 2
    assert np.array_equal(ids_f[clear], want[clear])


def test_lexicon_bindings_against_engine(engine, weights_dir, native_lib):
    sys.path.insert(0, str(_native.LIB_PATH.parent))
    import pytuatara

    fx = _fixtures()
    pages = [np.ascontiguousarray(fx["resume_example.img"])] + \
        [np.ascontiguousarray(synth.synth_page(s)[:h, :w]) for s, (h, w) in ((0, (607, 763)), (2, (754, 1000)))]
    words = _words(500, 90) + ["a", "I"]
    lex = tb.Lexicon(words)
    for form in (lex, words, tuple(words)):
        for page in pages[:2]:
            want = engine.ocr_pages([page], lexicon=lex)[0]
            assert pytuatara.image_to_data(page.copy(), weights_dir, "outputs", lexicon=form) == want
            assert tb.image_to_data(page, weights_dir, "outputs", lexicon=form) == want
            want_s = engine.ocr_pages([page], scores=True, lexicon=lex)[0]
            assert pytuatara.image_to_data_scored(page.copy(), weights_dir, "outputs", lexicon=form) == want_s
            assert tb.image_to_data_scored(page, weights_dir, "outputs", lexicon=form) == want_s
    per = [lex, None, words[:50]]
    want = engine.ocr_pages(pages, lexicon=[lex, None, tb.Lexicon(words[:50])])
    assert pytuatara.images_to_data(pages, weights_dir, "outputs", lexicon=per) == want
    assert tb.images_to_data(pages, weights_dir, "outputs", lexicon=per) == want
    want_s = engine.ocr_pages(pages, scores=True, lexicon=lex)
    assert pytuatara.images_to_data_scored(pages, weights_dir, "outputs", lexicon=words) == want_s
    assert tb.images_to_data_scored(pages, weights_dir, "outputs", lexicon=lex) == want_s
    assert sum(len(p) for p in want) > 0
    res = C.POINTER(_native.tt_result)()
    arr = (_native.tt_image * 2)(*[_native.image_struct(p) for p in pages[:2]])
    h = (C.c_void_p * 1)(lex._h.value)
    assert tb.lib().tt_ocr_pages_lexicon(engine._h, arr, 2, None, None, 0, None, 0, h, 1, C.byref(res)) == 0
    try:
        assert res.contents.n_pages == 2
    finally:
        tb.lib().tt_result_free(res)
