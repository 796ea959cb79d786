"""Per-word scores without a GPU: the C ABI stays layout compatible, the host decoder follows the definitions
(INTEGRATION.md, "Confidence and detection scores"), the oracle's opt-in scores follow the same definitions, and the
scored C++ / pytuatara entry points keep the soft failures of image_to_data."""
import ctypes as C
import math
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parents[1]
EOS_ID = 88  # tokenizer eos_id: dropped from the text, kept in conf


def _restated(ids, p):
    """The definitions, restated: e = first position of id 0 (else the last); conf = prod(p[0..e]) in double rounded
    once to float32; char_conf = p[t] of the positions that produce a character: before the first id 0 (all of them
    when there is none) and id != 88."""
    zero = np.flatnonzero(ids == 0)
    e = int(zero[0]) if len(zero) else len(ids) - 1
    conf = np.float32(math.prod(float(x) for x in p[:e + 1]))
    stop = int(zero[0]) if len(zero) else len(ids)
    char_conf = np.array([p[t] for t in range(stop) if ids[t] != EOS_ID], np.float32)
    return e, conf, char_conf


def test_result_struct_layouts_unchanged(native_lib, tmp_path):
    from tuatara_b200 import _native

    assert C.sizeof(_native.tt_item) == 24
    assert C.sizeof(_native.tt_page_result) == 16
    assert C.sizeof(_native.tt_result) == 16
    assert C.sizeof(_native.tt_ocr_options) == 24
    assert _native.tt_ocr_options.detect_only.offset == 16
    assert _native.tt_ocr_options.with_scores.offset == 20
    # the header itself, as a C compiler lays it out
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "tuatara_c.h"\n'
                   "int main(void) {\n"
                   '  printf("%zu %zu %zu %zu %zu %zu %zu\\n", sizeof(tt_item), sizeof(tt_page_result), sizeof(tt_result),\n'
                   "         sizeof(tt_ocr_options), offsetof(tt_ocr_options, detect_only), offsetof(tt_ocr_options, with_scores),\n"
                   "         offsetof(tt_ocr_options, score_override));\n  return 0;\n}\n")
    exe = tmp_path / "layout"
    subprocess.run(["gcc", f"-I{ROOT / 'include'}", str(src), "-o", str(exe)], check=True)
    out = subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()
    assert [int(v) for v in out] == [24, 16, 16, 24, 16, 20, 8]


def test_decode_scores_definition(native_lib):
    import tuatara_b200 as tb

    rng = np.random.default_rng(0)
    n, L = 400, 26
    ids = rng.integers(0, 95, (n, L)).astype(np.int32)
    p = rng.uniform(0.01, 1.0, (n, L)).astype(np.float32)
    ids[0, 0] = 0                                  # end at position 0: empty text, conf == p[0]
    ids[1][ids[1] == 0] = 5                        # no end: 26 factors
    ids[2, :12] = [7, EOS_ID, 9, EOS_ID, 11, 12, EOS_ID, 13, 0, 14, 0, EOS_ID]   # id 88 before the end
    ids[3, :6] = [20, 21, 22, 0, 23, 24]           # ids after the end are ignored
    ids[4] = EOS_ID                                # only id 88: empty text, 26 factors
    p[5] = 1e-3                                    # underflows: 26 factors of 1e-3 is below the smallest float32
    ids[5][ids[5] == 0] = 1
    texts, conf, char_conf = tb.decode_scores(ids, p)
    assert texts == tb.decode_ids(ids)
    for i in range(n):
        e, want_conf, want_cc = _restated(ids[i], p[i])
        assert conf[i].tobytes() == want_conf.tobytes(), (i, conf[i], want_conf)
        assert len(char_conf[i]) == len(texts[i])
        assert np.array_equal(char_conf[i], want_cc), i
    assert texts[0] == "" and conf[0] == p[0, 0]
    assert conf[1].tobytes() == np.float32(math.prod(float(x) for x in p[1])).tobytes()
    assert texts[2] == tb.tokenizer_table()[0][7] + tb.tokenizer_table()[0][9] + tb.tokenizer_table()[0][11] + \
        tb.tokenizer_table()[0][12] + tb.tokenizer_table()[0][13]
    assert np.array_equal(char_conf[2], p[2, [0, 2, 4, 5, 7]])
    assert conf[2].tobytes() == np.float32(math.prod(float(x) for x in p[2, :9])).tobytes()   # both 88s inside
    assert conf[3].tobytes() == np.float32(math.prod(float(x) for x in p[3, :4])).tobytes()
    assert texts[4] == "" and len(char_conf[4]) == 0
    assert conf[5] == 0.0
    # the rest of each char_conf row is zero
    out = np.zeros((n, 64), np.uint8)
    cc = np.full((n, L), np.nan, np.float32)
    tb.check(tb.lib().tt_decode_scores(tb.ptr(ids), tb.ptr(p), n, L, tb.ptr(out), 64, None, tb.ptr(cc)), "tt_decode_scores")
    for i in range(n):
        assert (cc[i, len(texts[i]):] == 0).all()


def test_oracle_scores_definition(oracle_models):
    """The reference scores (scores_ref.py, from the oracle's run) on hand-built logits: the same definitions, p computed
    here in float64; det_score is the oracle's maxVal of the component."""
    import torch

    from oracle import tuatara_ref as R
    from scores_ref import image_to_data_scored
    from tuatara_b200 import synth

    craft, _ = oracle_models
    page = np.ascontiguousarray(synth.synth_page(0)[:320, :384])
    maps = np.ascontiguousarray(synth.synth_score_maps(0)[:160, :192])
    rng = np.random.default_rng(1)
    logits = rng.standard_normal((64, 26, 95)).astype(np.float32)
    seqs = {0: [0], 1: [3] * 26, 2: [7, EOS_ID, 9, EOS_ID, 0], 3: [20, 21, 0, 22, 23, 24]}
    for i, seq in seqs.items():
        for t, c in enumerate(seq):
            logits[i, t, c] += 8.0
    logits[1, :, 0] -= 20.0
    fed = []

    def parseq(x):   # run_parseq feeds 4 crops at a time
        k = sum(len(f) for f in fed)
        fed.append(x)
        return torch.from_numpy(logits[k:k + x.shape[0]])

    override = (maps[..., 0], maps[..., 1])
    plain = R.image_to_data(page.copy(), craft, lambda x: torch.zeros(x.shape[0], 26, 95), score_override=override)
    fed.clear()
    st = R.Stages()
    got = image_to_data_scored(page.copy(), craft, parseq, score_override=override, stages=st)
    n = len(got)
    assert n >= 4 and n == len(plain) and [g["bbox"] for g in got] == [p["bbox"] for p in plain]
    l64 = logits[:n].astype(np.float64)
    p = 1.0 / np.exp(l64 - l64.max(-1, keepdims=True)).sum(-1)
    ids = l64.argmax(-1)
    for i, item in enumerate(got):
        assert set(item) == {"text", "bbox", "conf", "det_score", "char_conf"}
        e, _, _ = _restated(ids[i], p[i])
        assert math.isclose(item["conf"], math.prod(p[i, :e + 1]), rel_tol=1e-5, abs_tol=1e-37)
        stop = e if ids[i, e] == 0 else e + 1
        want_cc = [p[i, t] for t in range(stop) if ids[i, t] != EOS_ID]
        assert len(item["char_conf"]) == len(item["text"]) == len(want_cc)
        assert np.allclose(item["char_conf"], want_cc, rtol=1e-5, atol=0)
        assert item["det_score"] >= np.float32(0.7) and np.float32(item["det_score"]) == item["det_score"]
        dbg = st.det_debug
        assert item["det_score"] == np.float32(dbg.text_norm[dbg.labels == dbg.mapper[i]].max())
    assert got[0]["text"] == "" and math.isclose(got[0]["conf"], p[0, 0], rel_tol=1e-5)
    assert len(got[1]["text"]) == 26 and math.isclose(got[1]["conf"], math.prod(p[1]), rel_tol=1e-5, abs_tol=1e-37)
    assert len(got[2]["text"]) == 2 and math.isclose(got[2]["conf"], math.prod(p[2, :5]), rel_tol=1e-5)
    assert len(got[3]["text"]) == 2 and math.isclose(got[3]["conf"], math.prod(p[3, :3]), rel_tol=1e-5)


def test_scored_header_compiles_without_opencv(native_lib, tmp_path):
    src = tmp_path / "scored.cpp"
    src.write_text('#include "tuatara.h"\n'
                   "int main() {\n"
                   "  tuatara::ImageView v;\n"
                   "  std::vector<tuatara::ScoredItem> r = tuatara::image_to_data_scored(v, \"\", \"out\");\n"
                   "  std::vector<std::vector<tuatara::ScoredItem>> b = tuatara::image_to_data_scored_batch({v}, \"\", \"out\");\n"
                   "  float c = r.empty() ? 0.f : r[0].confidence + r[0].detection_score + r[0].char_confidence.size();\n"
                   "  return static_cast<int>(r.size() + b.size() + c);\n}\n")
    from tuatara_b200 import _native

    exe = tmp_path / "scored"
    subprocess.run(["g++", "-std=c++14", f"-I{ROOT / 'include'}", str(src), "-o", str(exe), f"-L{_native.LIB_PATH.parent}",
                    "-ltuatara_b200", f"-Wl,-rpath,{_native.LIB_PATH.parent}"], check=True)
    r = subprocess.run([str(exe)], capture_output=True, text=True)
    assert r.returncode == 0 and "Please provide a value for weights_dir" in r.stderr


def test_pytuatara_scored_signature(native_lib):
    from tuatara_b200 import _native

    sys.path.insert(0, str(_native.LIB_PATH.parent))
    import pytuatara

    import tuatara_b200 as tb

    for fn in (pytuatara.image_to_data_scored, pytuatara.images_to_data_scored):
        doc = fn.__doc__
        assert "weights_dir" in doc and "outputs_dir" in doc
    assert "image" in pytuatara.image_to_data_scored.__doc__ and "images" in pytuatara.images_to_data_scored.__doc__
    with pytest.raises(RuntimeError, match="Input array should have 3 dimensions"):
        pytuatara.image_to_data_scored(image=np.zeros((4, 4), np.uint8), weights_dir="w", outputs_dir="o")
    with pytest.raises(RuntimeError, match="Input array should have 3 channels"):
        pytuatara.image_to_data_scored(image=np.zeros((4, 4, 4), np.uint8), weights_dir="w", outputs_dir="o")
    assert pytuatara.image_to_data_scored(np.zeros((4, 4, 3), np.uint8), "", "o") == []
    assert pytuatara.image_to_data_scored(np.zeros((4, 4, 3), np.uint8), "w", "") == []
    assert pytuatara.images_to_data_scored([np.zeros((4, 4, 3), np.uint8)], "", "o") == []
    # the ctypes twin
    assert tb.image_to_data_scored(np.zeros((4, 4, 3), np.uint8), "", "o") == []
    with pytest.raises(RuntimeError, match="Input array should have 3 dimensions"):
        tb.image_to_data_scored(np.zeros((4, 4), np.uint8), "w", "o")
