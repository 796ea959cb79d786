"""The contrast re-read without a GPU: the reference against EasyOCR and against its own table form, the device's grey
formula against cv2 over every BGR triple, the argument checks of the new entry points, the exported symbols, the
header at C++14 without OpenCV and the keywords of both Python packages."""
import ctypes as C
import inspect
import math
import re
import subprocess
import sys
from pathlib import Path

import cv2
import numpy as np
import pytest

from contrast_ref import (GREY_COEF, GREY_SHIFT, adjust_contrast_grey, adjust_crop, contrast_grey, contrast_params,
                          grey_formula, keep_second, reread_words, stretch_table)

ROOT = Path(__file__).resolve().parents[1]


@pytest.fixture(scope="module")
def tb(native_lib):
    import tuatara_b200

    return tuatara_b200


def _edge_crops(rng):
    """Crops of every kind the stretch meets: constant, all black (high + low < 10), saturated, narrow bands with
    half-integer percentiles, and random ones."""
    out = [np.zeros((32, 128, 3), np.uint8), np.full((32, 128, 3), 255, np.uint8), np.full((32, 128, 3), 3, np.uint8),
           np.full((32, 128, 3), 128, np.uint8)]
    for i in range(300):
        lo = int(rng.integers(0, 256))
        hi = int(rng.integers(lo, min(256, lo + (3 if i % 3 == 0 else 256))))
        c = rng.integers(lo, hi + 1, (32, 128, 3), dtype=np.uint8)
        if i % 5 == 0:
            c[..., 1:] = c[..., :1]   # grey page
        if i % 7 == 0:
            c[:, :10] = 255           # saturated strip
        out.append(c)
    return out


def test_reference_is_easyocr_on_grey_pages():
    rng = np.random.default_rng(0)
    stretched = 0
    for c in _edge_crops(rng):
        g = c[..., 0].copy()
        page = np.repeat(g[..., None], 3, axis=2)
        for target in (0.5, 0.1, 1.0):
            got, s = adjust_crop(page, target)
            target = float(np.float32(target))   # the engine takes adjust_contrast as a float
            want = adjust_contrast_grey(g, target)
            assert np.array_equal(got[..., 0], want) and np.array_equal(got[..., 1], want) and np.array_equal(got[..., 2], want)
            assert s == (contrast_grey(g)[0] < target)
            stretched += s
    assert stretched > 100


def test_table_form_equals_elementwise_form():
    rng = np.random.default_rng(1)
    crops = _edge_crops(rng) + list(rng.integers(0, 256, (3000, 32, 128, 3), dtype=np.uint8) // rng.integers(1, 40, (3000, 1, 1, 1)).astype(np.uint8))
    n = halves = 0
    for c in crops:
        g = cv2.cvtColor(c, cv2.COLOR_BGR2GRAY)
        contrast, high, low = contrast_grey(g)
        if contrast >= 0.5:
            continue
        n += 1
        halves += high != math.floor(high) or low != math.floor(low)
        assert np.array_equal(stretch_table(low, high)[g], adjust_contrast_grey(g, 0.5))
        # the percentiles as the device takes them from the sorted values
        s = np.sort(g.ravel()).astype(np.float64)
        assert low == s[410] - (s[410] - s[409]) * 0.5 and high == s[3686] - (s[3686] - s[3685]) * 0.5
    assert n > 1000 and halves > 10, (n, halves)


def test_device_grey_formula_is_cv2_for_every_triple():
    src = (ROOT / "tuatara_b200" / "csrc" / "contrast.cu").read_text()
    m = re.search(r"\(b \* (\d+) \+ g \* (\d+) \+ r \* (\d+) \+ \(1 << (\d+)\)\) >> (\d+)", src)
    assert m, "the grey expression of k_contrast_stats"
    assert tuple(int(v) for v in m.groups()) == (*GREY_COEF, GREY_SHIFT - 1, GREY_SHIFT)
    v = np.arange(1 << 24, dtype=np.uint32)
    img = np.stack([(v >> 16) & 255, (v >> 8) & 255, v & 255], -1).astype(np.uint8).reshape(4096, 4096, 3)
    assert np.array_equal(grey_formula(img), cv2.cvtColor(img, cv2.COLOR_BGR2GRAY))


def test_selection_and_reread_rules():
    assert keep_second(0.2, 0.3) and not keep_second(0.3, 0.3) and not keep_second(0.3, 0.2)
    assert not keep_second(float("nan"), 0.9) and not keep_second(0.5, float("nan"))
    assert not keep_second(0.0, 0.0) and keep_second(0.0, 1e-30)
    low = np.full((32, 128, 3), 100, np.uint8)
    low[:, ::2] = 104
    high = np.zeros((32, 128, 3), np.uint8)
    high[:, ::2] = 250
    assert contrast_params(low, 0.5)[0] and not contrast_params(high, 0.5)[0]
    idx, crops = reread_words([0.05, 0.05, 0.5, float("nan")], [low, high, low, low], 0.1, 0.5)
    assert idx == [0] and crops.shape == (1, 32, 128, 3) and not np.array_equal(crops[0], low)


def _contrast(lib, arr, n, ths, adj, res, lex=None, n_lex=0):
    return lib.tt_ocr_pages_contrast(None, arr, n, None, None, 0, None, 0, lex, n_lex, ths, adj, C.byref(res))


def test_contrast_arguments_fail_before_the_engine(tb):
    """Every argument error of tt_ocr_pages_contrast is reported with e == NULL: nothing reaches the engine."""
    from tuatara_b200 import _native

    lib = tb.lib()
    img = np.zeros((32, 32, 3), np.uint8)
    arr = (_native.tt_image * 1)(_native.image_struct(img))
    res = C.POINTER(_native.tt_result)()
    for ths, word in ((float("nan"), b"contrast_ths is nan"), (float("inf"), b"contrast_ths is inf"),
                      (float("-inf"), b"contrast_ths is -inf"), (-0.5, b"contrast_ths is -0.5"), (-1e-3, b"-0.001")):
        assert _contrast(lib, arr, 1, ths, 0.5, res) != 0
        assert word in lib.tt_last_error(), (ths, lib.tt_last_error())
    for adj, word in ((0.0, b"adjust_contrast is 0;"), (-0.5, b"adjust_contrast is -0.5"), (1.5, b"adjust_contrast is 1.5"),
                      (float("nan"), b"adjust_contrast is nan"), (float("inf"), b"adjust_contrast is inf")):
        assert _contrast(lib, arr, 1, 0.1, adj, res) != 0
        assert word in lib.tt_last_error(), (adj, lib.tt_last_error())
        assert _contrast(lib, arr, 1, 0.0, adj, res) != 0   # checked with the re-read off too
        assert word in lib.tt_last_error()
    # after the lexicons: a lexicon error comes first, and the names are the new entry point's
    assert _contrast(lib, arr, 1, float("nan"), 0.5, res, None, 1) != 0
    assert b"tt_ocr_pages_contrast: lexicons is NULL but n_lexicons is 1" in lib.tt_last_error()
    lex = tb.Lexicon(["ab"])
    h = (C.c_void_p * 1)(lex._h.value)
    assert _contrast(lib, arr, 1, -1.0, 0.5, res, h, 1) != 0
    assert b"tt_ocr_pages_contrast: contrast_ths is -1" in lib.tt_last_error()
    # valid values, the edges included, reach the engine check
    for ths, adj in ((0.0, 0.5), (2.0, 1.0), (1e-30, 1e-6), (0.1, 0.5)):
        assert _contrast(lib, arr, 1, ths, adj, res) != 0
        assert b"null argument" in lib.tt_last_error(), (ths, adj)
    out = np.zeros((1, 32, 128, 3), np.uint8)
    for adj in (0.0, 1.01, float("nan")):
        assert lib.tt_contrast_adjust(tb.ptr(out), 1, adj, tb.ptr(out), None) != 0
        assert b"adjust_contrast is" in lib.tt_last_error()
    with pytest.raises(ValueError):
        tb.contrast_adjust(np.zeros((2, 32, 127, 3), np.uint8))
    assert lib.tt_contrast_select_dev(None, None, None, 1, None, None, None) != 0
    assert b"tt_contrast_select_dev" in lib.tt_last_error()


def test_symbols_exported(tb):
    out = subprocess.run(["nm", "-D", "--defined-only", str(tb._native.LIB_PATH)], capture_output=True, text=True,
                         check=True).stdout
    for name in ("tt_ocr_pages_contrast", "tt_contrast_adjust", "tt_contrast_select_dev"):
        assert re.search(rf"\bT {name}$", out, re.M), name


def test_header_compiles_at_cpp14_without_opencv(tb, tmp_path):
    src = tmp_path / "t.cpp"
    src.write_text('#include "tuatara.h"\n'
                   "int main() {\n"
                   "  tuatara::ImageView v;\n"
                   "  tuatara::Contrast easy;\n"
                   "  tuatara::Contrast strong{2.f, 1.f};\n"
                   '  auto a = image_to_data(v, "", "o", easy);\n'
                   '  auto b = tuatara::image_to_data_batch({v, v}, "", "o", strong);\n'
                   '  auto c = tuatara::image_to_data_scored(v, "", "o", easy);\n'
                   '  auto d = tuatara::image_to_data_scored_batch({v}, "", "o", easy);\n'
                   '  auto e = tuatara::image_to_data_oriented(v, "", "o", {180}, easy);\n'
                   '  auto f = tuatara::image_to_data_oriented_batch({v}, "w", "", {90, 270}, strong);\n'
                   "  return static_cast<int>(a.size() + b.size() + c.size() + d.size() + e.size() + f.size()) +\n"
                   "         (easy.contrast_ths == 0.1f && easy.adjust_contrast == 0.5f ? 0 : 1);\n"
                   "}\n")
    exe = tmp_path / "t"
    subprocess.run(["g++", "-std=c++14", "-Wall", "-Werror", f"-I{ROOT / 'include'}", str(src), "-o", str(exe),
                    f"-L{tb._native.LIB_PATH.parent}", "-ltuatara_b200", f"-Wl,-rpath,{tb._native.LIB_PATH.parent}"],
                   check=True)
    r = subprocess.run([str(exe)], capture_output=True, text=True)
    assert r.returncode == 0
    assert r.stderr.count("Please provide a value for weights_dir") == 5
    assert r.stderr.count("Please provide a value for outputs_dir") == 1


def test_keywords(tb):
    sys.path.insert(0, str(Path(tb._native.LIB_PATH).parent))
    import pytuatara

    for fn in (tb.image_to_data, tb.images_to_data, tb.image_to_data_scored, tb.images_to_data_scored,
               tb.Engine.ocr_pages):
        params = inspect.signature(fn).parameters
        assert params["contrast_ths"].kind == inspect.Parameter.KEYWORD_ONLY and params["contrast_ths"].default == 0.0
        assert params["adjust_contrast"].kind == inspect.Parameter.KEYWORD_ONLY and params["adjust_contrast"].default == 0.5
    img = np.zeros((8, 8, 3), np.uint8)
    for name in ("image_to_data", "images_to_data", "image_to_data_scored", "images_to_data_scored"):
        doc = getattr(pytuatara, name).__doc__
        assert re.search(r"\*,.*contrast_ths: [^=]+ = 0\.0, adjust_contrast: [^=]+ = 0\.5\)", doc), doc
    for fn in (pytuatara.image_to_data, pytuatara.image_to_data_scored, tb.image_to_data, tb.image_to_data_scored):
        assert fn(img, "", "o", contrast_ths=0.1) == []
        assert fn(img, "w", "", contrast_ths=0.1, adjust_contrast=0.3) == []
    for fn in (pytuatara.images_to_data, pytuatara.images_to_data_scored):
        assert fn([img, img], "", "o", contrast_ths=2.0) == []
    with pytest.raises(TypeError):
        pytuatara.image_to_data(img, "w", "o", None, None, None, None, 0.1)   # keyword only
    assert "contrast_adjust" in tb.__all__
