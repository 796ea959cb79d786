"""Rotation candidates without a GPU: the reference's candidates and choice rule, the argument checks of the new entry
points, unchanged struct layouts, the header at C++14 without OpenCV and the pytuatara keyword."""
import ctypes as C
import subprocess
import sys
from pathlib import Path

import cv2
import numpy as np
import pytest

from orient_ref import candidate_crop, candidate_quad, candidate_set, conf_of, rotate, select

ROOT = Path(__file__).resolve().parents[1]


def test_candidate_set_and_directions():
    assert candidate_set([]) == [0]
    assert candidate_set([270, 90]) == [0, 90, 270]
    assert candidate_set((180, 90, 270)) == [0, 90, 180, 270]
    img = np.arange(2 * 3 * 3, dtype=np.uint8).reshape(2, 3, 3)
    # counter-clockwise: the top-right pixel comes to the top-left at 90, the bottom-left at 270
    assert np.array_equal(rotate(img, 90)[0, 0], img[0, 2])
    assert np.array_equal(rotate(img, 270)[0, 0], img[1, 0])
    assert np.array_equal(rotate(img, 180), img[::-1, ::-1])
    assert np.array_equal(rotate(rotate(img, 90), 270), img)
    assert rotate(img, 90).shape == (3, 2, 3)


def test_candidate_crops_and_quads():
    rng = np.random.default_rng(0)
    page = rng.integers(0, 256, (60, 90, 3), dtype=np.uint8)
    r = (5, 7, 40, 12)
    c0 = candidate_crop(page, r, 0)
    assert np.array_equal(c0, cv2.resize(page[7:19, 5:45], (128, 32)))
    # the rotation comes before the resize: the ROI's height becomes the 128 columns
    c90 = candidate_crop(page, r, 90)
    assert np.array_equal(c90, cv2.resize(cv2.rotate(page[7:19, 5:45], cv2.ROTATE_90_COUNTERCLOCKWISE), (128, 32)))
    assert not candidate_crop(page, (3, 3, 0, 5), 90).any()
    rect = ((40.0, 20.0), (30.0, 10.0), 0.0)
    from oracle import tuatara_ref as R

    q = R.rect_to_quad(rect)
    assert np.array_equal(candidate_quad(rect, 0), q)
    assert np.array_equal(candidate_quad(rect, 90), q[[1, 2, 3, 0]])
    assert np.array_equal(candidate_quad(rect, 180), q[[2, 3, 0, 1]])
    assert np.array_equal(candidate_quad(rect, 270), q[[3, 0, 1, 2]])


def test_selection_rule():
    ids = np.full(26, 5, np.int32)
    p = np.full(26, 0.9, np.float32)
    p64 = float(p[0])   # multiplied in double, rounded once
    ids[3] = 0
    assert conf_of(ids, p) == float(np.float32(p64 * p64 * p64 * p64))   # the end position is a factor
    ids[0] = 0
    assert conf_of(ids, p) == float(p[0])
    prod = 1.0
    for _ in range(26):
        prod *= p64
    assert conf_of(np.full(26, 7, np.int32), p) == float(np.float32(prod))   # no end class: every position
    assert conf_of(np.full(26, 7, np.int32), np.ones(26, np.float32)) == 1.0
    assert select([0.5, 0.5, 0.5]) == 0                         # ties stay with the earlier candidate
    assert select([0.5, 0.6, 0.6]) == 1
    assert select([0.0, 0.0]) == 0                              # 0 wins a tie
    assert select([float("nan"), 0.9]) == 0                     # NaN: no comparison succeeds
    assert select([0.2, float("nan"), 0.3]) == 2
    assert select([0.2, 0.1, 0.25, 0.24]) == 2


def test_struct_layouts_unchanged(native_lib, tmp_path):
    from tuatara_b200 import _native

    assert C.sizeof(_native.tt_ocr_options) == 24 and C.sizeof(_native.tt_item) == 24
    assert C.sizeof(_native.tt_config) == 36 and C.sizeof(_native.tt_result) == 16
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "tuatara_c.h"\n'
                   "int main(void) {\n"
                   '  printf("%zu %zu %zu %zu %zu %zu\\n", sizeof(tt_ocr_options), sizeof(tt_item), sizeof(tt_page_result),\n'
                   "         sizeof(tt_result), sizeof(tt_config), offsetof(tt_ocr_options, with_scores));\n  return 0;\n}\n")
    exe = tmp_path / "layout"
    subprocess.run(["gcc", f"-I{ROOT / 'include'}", str(src), "-o", str(exe)], check=True)
    out = subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()
    assert [int(v) for v in out] == [24, 24, 16, 16, 36, 20]


def test_oriented_call_checks_its_angles(native_lib):
    """Checked before any device work, so no engine is needed to see the messages."""
    import tuatara_b200 as tb
    from tuatara_b200 import _native

    lib = tb.lib()
    res = C.POINTER(_native.tt_result)()
    for bad, word in (([45], b"45"), ([0], b" 0"), ([90, 360], b"360"), ([180, 180], b"180 twice"), ([-90], b"-90"),
                      ([90, 270, 90], b"90 twice")):
        a = (C.c_int * len(bad))(*bad)
        assert lib.tt_ocr_pages_oriented(None, None, 1, None, None, 0, a, len(bad), C.byref(res)) != 0
        msg = lib.tt_last_error()
        assert word in msg and b"rotation_info" in msg, msg
    assert lib.tt_ocr_pages_oriented(None, None, 1, None, None, 0, None, 2, C.byref(res)) != 0
    assert b"NULL" in lib.tt_last_error()
    assert lib.tt_ocr_pages_oriented(None, None, 1, None, None, 0, None, -1, C.byref(res)) != 0
    a = (C.c_int * 1)(90)
    f = (_native.tt_char_filter * 3)(*[_native.tt_char_filter(b"0", None)] * 3)
    assert lib.tt_ocr_pages_oriented(None, None, 2, None, f, 3, a, 1, C.byref(res)) != 0
    assert b"n_filters" in lib.tt_last_error()
    # n_rotations == 0 is tt_ocr_pages_filtered: its checks
    assert lib.tt_ocr_pages_oriented(None, None, 2, None, None, 0, None, 0, C.byref(res)) != 0
    assert b"null argument" in lib.tt_last_error()
    assert lib.tt_item_angle(None, 0, 0, None) != 0
    assert lib.tt_orient_select_dev(None, None, 1, None, 0, None, None, None, None) != 0
    assert b"n_candidates" in lib.tt_last_error()
    with pytest.raises(TypeError):
        tb._rotations(90)
    with pytest.raises(TypeError):
        tb._rotations(["90"])
    with pytest.raises(TypeError):
        tb._rotations("90")
    assert list(tb._rotations(range(90, 360, 90))) == [90, 180, 270]
    with pytest.raises(ValueError, match="angles"):
        tb.crop_resize(np.zeros((4, 4, 3), np.uint8), [[0, 0, 2, 2]], angles=[0, 90])


def test_oriented_header_compiles_without_opencv(native_lib, tmp_path):
    src = tmp_path / "oriented.cpp"
    src.write_text('#include "tuatara.h"\n'
                   "int main() {\n"
                   "  tuatara::ImageView v;\n"
                   "  tuatara::CharFilter digits{\"0123456789\"};\n"
                   "  std::vector<tuatara::ScoredItem> a = tuatara::image_to_data_oriented(v, \"\", \"out\", {180});\n"
                   "  std::vector<tuatara::ScoredItem> b = tuatara::image_to_data_oriented(v, \"w\", \"\", {90, 270}, digits);\n"
                   "  std::vector<std::vector<tuatara::ScoredItem>> c =\n"
                   "      tuatara::image_to_data_oriented_batch({v, v}, \"\", \"out\", {90, 180, 270});\n"
                   "  std::vector<std::vector<tuatara::ScoredItem>> d =\n"
                   "      tuatara::image_to_data_oriented_batch({v}, \"\", \"out\", {180}, {digits});\n"
                   "  tuatara::ScoredItem s;\n"
                   "  return static_cast<int>(a.size() + b.size() + c.size() + d.size()) + s.angle;\n}\n")
    from tuatara_b200 import _native

    exe = tmp_path / "oriented"
    subprocess.run(["g++", "-std=c++14", "-Wall", "-Werror", f"-I{ROOT / 'include'}", str(src), "-o", str(exe),
                    f"-L{_native.LIB_PATH.parent}", "-ltuatara_b200", f"-Wl,-rpath,{_native.LIB_PATH.parent}"], check=True)
    r = subprocess.run([str(exe)], capture_output=True, text=True)
    assert r.returncode == 0
    assert r.stderr.count("Please provide a value for weights_dir") == 3
    assert r.stderr.count("Please provide a value for outputs_dir") == 1


def test_pytuatara_rotation_keyword(native_lib):
    from tuatara_b200 import _native

    sys.path.insert(0, str(_native.LIB_PATH.parent))
    import pytuatara

    import tuatara_b200 as tb

    img = np.zeros((4, 4, 3), np.uint8)
    for fn in (pytuatara.image_to_data, pytuatara.image_to_data_scored):
        assert "rotation_info" in fn.__doc__
        assert fn(img, "", "o", rotation_info=[180]) == []
        assert fn(img, "w", "", rotation_info=[90, 270], allowlist="0") == []
        with pytest.raises(TypeError):
            fn(img, "w", "o", rotation_info=90)
        with pytest.raises(TypeError):
            fn(img, "w", "o", rotation_info=["90"])
        with pytest.raises(TypeError):
            fn(img, "w", "o", None, None, [90])   # keyword only
    for fn in (pytuatara.images_to_data, pytuatara.images_to_data_scored):
        assert "rotation_info" in fn.__doc__
        assert fn([img, img], "", "o", rotation_info=(90, 180)) == []
    for fn in (tb.image_to_data, tb.image_to_data_scored):
        assert fn(img, "", "o", rotation_info=[180]) == []
