"""Character filters without a GPU: the class-mask rule against a restatement over the tokenizer table, the C ABI's
struct and argument checks, the C++ header without OpenCV, the pytuatara keywords and the masked reference decode."""
import ctypes as C
import string
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

from charset_ref import class_mask_ref, mask_words, masked_argmax, masked_forward, words_to_bool

ROOT = Path(__file__).resolve().parents[1]
PRINTABLE = "".join(chr(c) for c in range(32, 127))


def test_char_filter_mask_rule(native_lib):
    import tuatara_b200 as tb

    itos, eos, _, _ = tb.tokenizer_table()
    assert eos == 88
    cases = [(None, None), ("0123456789", None), (string.ascii_uppercase, None), ("", None), ("", ""),
             (None, string.ascii_lowercase), (None, string.punctuation), ("\\", None), ("~] éü", None),
             (None, "~] "), (string.ascii_letters + string.digits, "aeiouAEIOU0"), (PRINTABLE, None), ("abc", "abc"),
             ("'\"`", "`")]
    for allow, block in cases:
        got = tb.char_filter_mask(allow, block)
        want = class_mask_ref(itos, eos, allow, block)
        assert got.dtype == np.uint32 and got.shape == (4,)
        assert np.array_equal(got, mask_words(want)), (allow, block, got, mask_words(want))
        assert np.array_equal(words_to_bool(got), want)
        assert got[3] == 0
        assert want[0] and want[88], (allow, block)
    full = tb.char_filter_mask()
    assert np.array_equal(words_to_bool(full), np.ones(95, bool))
    # every printable character allows every class: the same mask as no filter
    assert np.array_equal(tb.char_filter_mask(PRINTABLE), full)
    # '\' is printed by two classes
    bs = words_to_bool(tb.char_filter_mask("\\"))
    assert sorted(np.flatnonzero(bs)) == [0, 69, 87, 88]
    assert np.array_equal(words_to_bool(tb.char_filter_mask(None, "\\")), ~bs | np.isin(np.arange(95), [0, 88]))
    # characters no class prints are ignored
    assert np.array_equal(tb.char_filter_mask("~] é"), tb.char_filter_mask(""))
    assert np.array_equal(tb.char_filter_mask(None, "~] é"), full)
    assert sorted(np.flatnonzero(words_to_bool(tb.char_filter_mask("")))) == [0, 88]
    # allow and block together: block wins
    ab = words_to_bool(tb.char_filter_mask("0123456789abc", "2b"))
    assert "".join(itos[c] for c in np.flatnonzero(ab) if c not in (0, 88)) == "013456789ac"
    # 93 printing classes, 92 distinct characters
    printing = [c for c in range(1, 95) if c != 88]
    assert len(printing) == 93 and len({itos[c] for c in printing}) == 92
    assert tb.lib().tt_char_filter_mask(None, tb.ptr(np.zeros(4, np.uint32))) != 0


def test_char_filter_struct_layout(native_lib, tmp_path):
    from tuatara_b200 import _native

    assert C.sizeof(_native.tt_char_filter) == 16
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "tuatara_c.h"\n'
                   "int main(void) {\n"
                   '  printf("%zu %zu %zu %zu\\n", sizeof(tt_char_filter), offsetof(tt_char_filter, block),\n'
                   "         sizeof(tt_ocr_options), sizeof(tt_item));\n  return 0;\n}\n")
    exe = tmp_path / "layout"
    subprocess.run(["gcc", f"-I{ROOT / 'include'}", str(src), "-o", str(exe)], check=True)
    out = subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()
    assert [int(v) for v in out] == [16, 8, 24, 24]


def test_filtered_call_checks_its_filter_count(native_lib):
    """n_filters must be 0, 1 or n_pages, and filters may only be NULL with n_filters == 0 (checked before any device
    work, so no engine is needed to see the messages)."""
    import tuatara_b200 as tb
    from tuatara_b200 import _native

    lib = tb.lib()
    res = C.POINTER(_native.tt_result)()
    f = (_native.tt_char_filter * 3)(*[_native.tt_char_filter(b"0123", None)] * 3)
    for n_filters in (2, 3, -1):
        assert lib.tt_ocr_pages_filtered(None, None, 4, None, f, n_filters, C.byref(res)) != 0
        assert b"n_filters" in lib.tt_last_error()
    assert lib.tt_ocr_pages_filtered(None, None, 2, None, None, 1, C.byref(res)) != 0
    assert b"filters is NULL" in lib.tt_last_error()
    assert lib.tt_ocr_pages_filtered(None, None, 2, None, None, 0, C.byref(res)) != 0   # no filter: tt_ocr_pages_ex's checks
    assert b"null argument" in lib.tt_last_error()


def test_filtered_header_compiles_without_opencv(native_lib, tmp_path):
    src = tmp_path / "filtered.cpp"
    src.write_text('#include "tuatara.h"\n'
                   "int main() {\n"
                   "  tuatara::ImageView v;\n"
                   "  tuatara::CharFilter digits{\"0123456789\"};\n"
                   "  tuatara::CharFilter f;\n"
                   "  f.block = \"abc\";\n"
                   "  std::vector<OutputItem> a = image_to_data(v, \"\", \"out\", digits);\n"
                   "  std::vector<std::vector<OutputItem>> b = tuatara::image_to_data_batch({v, v}, \"w\", \"\", {digits, f});\n"
                   "  std::vector<tuatara::ScoredItem> c = tuatara::image_to_data_scored(v, \"\", \"out\", f);\n"
                   "  std::vector<std::vector<tuatara::ScoredItem>> d = tuatara::image_to_data_scored_batch({v}, \"\", \"out\", {f});\n"
                   "  return static_cast<int>(a.size() + b.size() + c.size() + d.size());\n}\n")
    from tuatara_b200 import _native

    exe = tmp_path / "filtered"
    subprocess.run(["g++", "-std=c++14", "-Wall", "-Werror", f"-I{ROOT / 'include'}", str(src), "-o", str(exe),
                    f"-L{_native.LIB_PATH.parent}", "-ltuatara_b200", f"-Wl,-rpath,{_native.LIB_PATH.parent}"], check=True)
    r = subprocess.run([str(exe)], capture_output=True, text=True)
    assert r.returncode == 0
    assert r.stderr.count("Please provide a value for weights_dir") == 3
    assert r.stderr.count("Please provide a value for outputs_dir") == 1


def test_pytuatara_filter_keywords(native_lib):
    from tuatara_b200 import _native

    sys.path.insert(0, str(_native.LIB_PATH.parent))
    import pytuatara

    import tuatara_b200 as tb

    img = np.zeros((4, 4, 3), np.uint8)
    for fn in (pytuatara.image_to_data, pytuatara.image_to_data_scored):
        assert "allowlist" in fn.__doc__ and "blocklist" in fn.__doc__
        assert fn(img, "", "o", allowlist="0123") == []
        assert fn(img, "w", "", blocklist="abc") == []
        assert fn(img, "", "o", allowlist=None, blocklist=None) == []
        with pytest.raises(RuntimeError, match="Input array should have 3 dimensions"):
            fn(np.zeros((4, 4), np.uint8), "w", "o", allowlist="0")
        with pytest.raises(RuntimeError, match="Input array should have 3 channels"):
            fn(np.zeros((4, 4, 4), np.uint8), "w", "o", allowlist="0")
        with pytest.raises(TypeError):
            fn(img, "w", "o", "0123")            # keyword only
        with pytest.raises(TypeError):
            fn(img, "", "o", allowlist=["0"])   # one page: a str or None
    for fn in (pytuatara.images_to_data, pytuatara.images_to_data_scored):
        assert "allowlist" in fn.__doc__ and "blocklist" in fn.__doc__
        assert fn([img, img], "", "o", allowlist="0") == []
        assert fn([img, img], "", "o", allowlist=["0", None], blocklist="a") == []
        with pytest.raises(ValueError, match="one entry per page"):
            fn([img, img], "", "o", allowlist=["0"])
        with pytest.raises(ValueError, match="one entry per page"):
            fn([img], "", "o", blocklist=["a", "b"])
        with pytest.raises(TypeError):
            fn([img], "", "o", allowlist=[3])
    # the ctypes twins
    assert tb.image_to_data(img, "", "o", allowlist="0") == []
    assert tb.image_to_data_scored(img, "w", "", blocklist="0") == []
    with pytest.raises(RuntimeError, match="Input array should have 3 dimensions"):
        tb.image_to_data(np.zeros((4, 4), np.uint8), "w", "o", allowlist="0")
    with pytest.raises(ValueError, match="one entry per page"):
        tb._filters(["0"], None, 2)
    with pytest.raises(TypeError):
        tb._filters(None, [b"a"], 1)
    assert tb._filters(None, None, 3) is None
    assert len(tb._filters("0", None, 3)) == 1 and len(tb._filters(["0", None, "1"], "a", 3)) == 3


def _oracle_tiny():
    from oracle.models import make_parseq

    return make_parseq("tiny", 0)


def _images(n, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.rand((n, 3, 32, 128), generator=g)


def test_masked_reference_decode(native_lib):
    import tuatara_b200 as tb

    itos, eos, _, _ = tb.tokenizer_table()
    parseq = _oracle_tiny()
    x = _images(6, 0)
    # all-true mask: the oracle's own forward
    taps_ref, taps = {}, {}
    ref = parseq(x, taps=taps_ref)
    got = masked_forward(parseq, x, torch.ones(6, 95, dtype=torch.bool), taps=taps)
    assert torch.equal(got, ref)
    assert torch.equal(taps["ar_logits"], taps_ref["ar_logits"]) and torch.equal(taps["ar_tokens"], taps_ref["ar_tokens"])
    # digits (and one crop with nothing but the two silent classes): every AR token and refinement id is allowed
    masks = np.stack([class_mask_ref(itos, eos, "0123456789")] * 5 + [class_mask_ref(itos, eos, "")])
    m = torch.from_numpy(masks)
    taps = {}
    out = masked_forward(parseq, x, m, taps=taps)
    ar_tok = taps["ar_tokens"][:, 1:].numpy()
    ref_ids = masked_argmax(out.numpy(), masks[:, None, :])
    for i in range(6):
        assert masks[i][ar_tok[i]].all(), i
        assert masks[i][ref_ids[i]].all(), i
    # the AR feedback and the refinement context are the masked argmax of the AR logits
    ar = taps["ar_logits"].numpy()
    assert np.array_equal(ar_tok, masked_argmax(ar[:, :-1], masks[:, None, :]))
    forced = torch.from_numpy(masked_argmax(ar[:, :-1], masks[:, None, :])).long()
    assert torch.equal(masked_forward(parseq, x, m, forced_tokens=forced), out)
    # the returned logits are not masked, and masking changes the decode
    assert np.isfinite(out.numpy()).all()
    assert not np.array_equal(ar_tok, taps_ref["ar_tokens"][:, 1:].numpy())

