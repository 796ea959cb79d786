"""Lexicons without a GPU: word validation, the trie's size against the reference, the argument checks of
tt_ocr_pages_lexicon, unchanged struct layouts, the header at C++14 without OpenCV, the keywords of both Python
packages and self-checks of the reference walk."""
import ctypes as C
import inspect
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

from charset_ref import class_mask_ref, masked_argmax, masked_pmax
from lexicon_ref import make_trie, one_state, text_of, walk

ROOT = Path(__file__).resolve().parents[1]


@pytest.fixture(scope="module")
def tb(native_lib):
    import tuatara_b200

    return tuatara_b200


def _create(tb, words):
    arr = (C.c_char_p * max(len(words), 1))(*words)
    h = C.c_void_p()
    rc = tb.lib().tt_lexicon_create(arr, len(words), C.byref(h))
    return rc, h, tb.lib().tt_last_error().decode()


@pytest.mark.parametrize("words, index, what", [
    ([b""], 0, "0 bytes long"),
    ([b"ok", b"x" * 26], 1, "26 bytes long"),
    ([b"a", b"b]"], 1, "0x5d (']')"),
    ([b"~"], 0, "0x7e ('~')"),
    ([b"ab", b"c", b"a\tb"], 2, "byte 0x09"),
    ([b"caf\xc3\xa9"], 0, "byte 0xc3"),
])
def test_create_rejects_invalid_words(tb, words, index, what):
    rc, h, err = _create(tb, words)
    assert rc != 0 and not h.value
    assert f"word {index}" in err and what in err, err


def test_create_rejects_empty_lists(tb):
    h = C.c_void_p()
    assert tb.lib().tt_lexicon_create(None, 3, C.byref(h)) != 0
    assert b"words is NULL" in tb.lib().tt_last_error()
    arr = (C.c_char_p * 1)(b"a")
    assert tb.lib().tt_lexicon_create(arr, 0, C.byref(h)) != 0
    assert b"n_words is 0" in tb.lib().tt_last_error()


def test_info_counts_distinct_words_and_trie_states(tb):
    itos, eos, _, _ = tb.tokenizer_table()
    rng = np.random.default_rng(0)
    letters = "abcXYZ019\\'-"
    words = ["a", "ab", "abc", "abc", "x" * 25, "\\", "a\\b", "0-9"] + \
        ["".join(rng.choice(list(letters), int(rng.integers(1, 8)))) for _ in range(300)]
    lex = tb.Lexicon(words)
    ref = make_trie(words, itos, eos)
    assert lex.info() == (len(set(words)), ref.n_states)
    # both backslash classes lead to one child
    bs = [c for c in range(1, 95) if itos[c] == "\\"]
    assert bs == [69, 87] and ref.allow[0, 69] and ref.allow[0, 87] and ref.succ[0][69] == ref.succ[0][87]
    assert not ref.allow[:, 88].any()


def test_lexicon_arguments_fail_before_the_engine(tb):
    """Every argument error of tt_ocr_pages_lexicon is reported with e == NULL: nothing reaches the engine."""
    from tuatara_b200 import _native

    lib = tb.lib()
    img = np.zeros((32, 32, 3), np.uint8)
    arr = (_native.tt_image * 2)(*[_native.image_struct(img)] * 2)
    res = C.POINTER(_native.tt_result)()
    lex = tb.Lexicon(["123", "4567"])
    h = (C.c_void_p * 3)(lex._h.value, lex._h.value, None)
    assert lib.tt_ocr_pages_lexicon(None, arr, 2, None, None, 0, None, 0, h, 3, C.byref(res)) != 0
    assert b"n_lexicons must be 0, 1 or n_pages (2), got 3" in lib.tt_last_error()
    assert lib.tt_ocr_pages_lexicon(None, arr, 2, None, None, 0, None, 0, None, 1, C.byref(res)) != 0
    assert b"lexicons is NULL but n_lexicons is 1" in lib.tt_last_error()
    f = (_native.tt_char_filter * 2)(_native.tt_char_filter(None, None), _native.tt_char_filter(b"abc", None))
    assert lib.tt_ocr_pages_lexicon(None, arr, 2, None, f, 2, None, 0, h, 2, C.byref(res)) != 0
    assert b"page 1" in lib.tt_last_error() and b"none of its lexicon's 2 words" in lib.tt_last_error()
    # the other checks keep their order and messages
    bad = (C.c_int * 1)(45)
    assert lib.tt_ocr_pages_lexicon(None, arr, 2, None, None, 0, bad, 1, h, 1, C.byref(res)) != 0
    assert b"rotation_info holds 45" in lib.tt_last_error()
    assert lib.tt_ocr_pages_lexicon(None, arr, 2, None, f, 3, None, 0, h, 1, C.byref(res)) != 0
    assert b"n_filters" in lib.tt_last_error()
    # valid arguments reach the engine check
    f2 = (_native.tt_char_filter * 1)(_native.tt_char_filter(b"0123456789", None))
    assert lib.tt_ocr_pages_lexicon(None, arr, 2, None, f2, 1, None, 0, h, 2, C.byref(res)) != 0
    assert b"null argument" in lib.tt_last_error()


def test_struct_layouts_unchanged(tb):
    from tuatara_b200 import _native

    assert C.sizeof(_native.tt_item) == 24 and C.sizeof(_native.tt_result) == 16
    assert C.sizeof(_native.tt_ocr_options) == 24 and C.sizeof(_native.tt_char_filter) == 16
    assert C.sizeof(_native.tt_config) == 36


def test_header_compiles_at_cpp14_without_opencv(tmp_path):
    src = tmp_path / "t.cpp"
    src.write_text('#include "tuatara.h"\n'
                   "int main() {\n"
                   '  tuatara::Lexicon lex(std::vector<std::string>{"INV-001", "INV-002"});\n'
                   "  tuatara::Lexicon moved(std::move(lex));\n"
                   "  tuatara::ImageView v;\n"
                   '  auto a = image_to_data(v, "w", "o", moved);\n'
                   '  auto b = tuatara::image_to_data_scored_batch({v}, "w", "o", std::vector<const tuatara::Lexicon*>{&moved, nullptr});\n'
                   '  auto c = tuatara::image_to_data_oriented(v, "w", "o", {180}, moved);\n'
                   "  return static_cast<int>(a.size() + b.size() + c.size()) + (moved.ok() ? 0 : 1) + static_cast<int>(moved.error().size());\n"
                   "}\n")
    r = subprocess.run(["g++", "-std=c++14", "-Wall", "-Werror", "-fsyntax-only", "-I", str(ROOT / "include"), str(src)],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr


def test_keywords(tb):
    sys.path.insert(0, str(Path(tb._native.LIB_PATH).parent))
    import pytuatara

    for fn in (tb.image_to_data, tb.images_to_data, tb.image_to_data_scored, tb.images_to_data_scored,
               tb.Engine.ocr_pages):
        assert inspect.signature(fn).parameters["lexicon"].kind == inspect.Parameter.KEYWORD_ONLY
    for name in ("image_to_data", "images_to_data", "image_to_data_scored", "images_to_data_scored"):
        assert "*, allowlist" in getattr(pytuatara, name).__doc__ and "lexicon" in getattr(pytuatara, name).__doc__
    img = np.zeros((8, 8, 3), np.uint8)
    with pytest.raises(TypeError):
        pytuatara.image_to_data(img, "w", "o", None, None, None, ["a"])   # keyword only
    # the accepted forms, normalised without a GPU
    lex = tb.Lexicon(["a"])
    assert tb._lexicon_arg(None, 2, strict=True) is None
    assert tb._lexicon_arg(lex, 2, strict=True) == [lex]
    one = tb._lexicon_arg(("ab", "cd"), 2, strict=True)
    assert len(one) == 1 and one[0].info() == (2, 5)
    assert tb._lexicon_arg([lex, None], 2, strict=True) == [lex, None]
    per = tb._lexicon_arg([None, ["x", "y"]], 2, strict=False)
    assert per[0] is None and per[1].info() == (2, 3)
    with pytest.raises(TypeError):
        tb._lexicon_arg([None, ["x", "y"]], 2, strict=True)      # Engine.ocr_pages: Lexicon or None per page
    with pytest.raises(TypeError):
        tb._lexicon_arg(["x", lex], 2, strict=True)              # a mix
    with pytest.raises(TypeError):
        tb._lexicon_arg("abc", 1, strict=False)
    with pytest.raises(ValueError):
        tb._lexicon_arg([lex, None, None], 2, strict=True)
    # the module functions hand Engine.ocr_pages one Lexicon for every page, or the per-page list
    assert tb._engine_lexicon(lex, 3) is lex and tb._engine_lexicon(["a", "b"], 3).info() == (2, 3)
    assert tb._engine_lexicon([None], 1) == [None] and tb._engine_lexicon([lex, None, lex], 3) == [lex, None, lex]
    for form in (lex, ["a"], [None, ["x"], lex]):
        tb._lexicon_arg(tb._engine_lexicon(form, 3), 3, strict=True)
    with pytest.raises(tb.TuataraError, match="word 1"):
        tb.Lexicon(["ok", "no~"])


def test_reference_walks_spell_words(tb):
    itos, eos, _, _ = tb.tokenizer_table()
    rng = np.random.default_rng(1)
    words = ["a", "ab", "abc", "x" * 25, "a\\b", "Q7", "7Q"]
    trie = make_trie(words, itos, eos)
    for _ in range(200):
        logits = rng.normal(0, 3, (26, 95)).astype(np.float32)
        ids, p = walk(logits, trie)
        assert text_of(ids, itos, eos) in words
        assert np.all((p > 0) & (p <= 1))
    # a one-state trie is the masked argmax and the renormalised probability
    for allow, block in [(None, None), ("0123456789", None), (None, "aeiou")]:
        mask = class_mask_ref(itos, eos, allow, block)
        logits = rng.normal(0, 3, (26, 95)).astype(np.float32)
        logits[5, 0] = 50.0   # the word ends at position 5 at the latest: the done state allows every class after it
        ids, p = walk(logits, one_state(mask))
        want = masked_argmax(logits, mask)
        e = int(np.flatnonzero(want == 0)[0]) + 1
        assert np.array_equal(ids[:e], want[:e])
        assert np.allclose(p[:e], masked_pmax(logits, mask)[:e], rtol=1e-12)
        assert np.array_equal(ids[e:], logits[e:].argmax(-1))
