"""The C-ABI library loads and exports every symbol include/tuatara_c.h declares; the C++ header
compiles without OpenCV; pytuatara keeps the reference's module/function/keyword names.  No compute
calls that need a GPU."""
import os
import re
import subprocess
import sys
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parents[1]


def _declared():
    txt = (ROOT / "include" / "tuatara_c.h").read_text()
    return sorted(set(re.findall(r"TT_API[^;]*?\b(tt_\w+)\s*\(", txt)))


def test_every_declared_symbol_is_exported(native_lib):
    from tuatara_b200 import _native

    names = _declared()
    assert len(names) >= 25
    out = subprocess.run(["nm", "-D", "--defined-only", str(_native.LIB_PATH)], capture_output=True, text=True, check=True).stdout
    exported = set(re.findall(r" T (tt_\w+)", out))
    assert set(names) <= exported, sorted(set(names) - exported)
    assert set(names) == set(_native.SIGNATURES), "ctypes table out of sync with the header"
    for n in names:
        getattr(native_lib, n)


def test_no_gpu_fails_loudly(native_lib, tmp_path):
    """Without a CUDA device the product path must refuse, not fall back to anything.  The engine is created in a
    child process that sees no device, so the refusal is checked on GPU machines too."""
    code = ("import sys\nimport tuatara_b200 as tb\n"
            "try:\n    tb.Engine(sys.argv[1])\n"
            "except tb.TuataraError as e:\n    print(e)\n    raise SystemExit(0)\n"
            "raise SystemExit('tt_engine_create succeeded without a device')\n")
    r = subprocess.run([sys.executable, "-c", code, str(tmp_path)], cwd=ROOT, capture_output=True, text=True,
                       env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert r.returncode == 0, r.stdout + r.stderr
    assert re.search("no CUDA device|cannot open|CUDA", r.stdout), r.stdout


def test_product_never_imports_oracle():
    """oracle/ is test infrastructure: no product file may import, include, link or execute it."""
    for p in (ROOT / "tuatara_b200").rglob("*.py"):
        for line in p.read_text().splitlines():
            code = line.split("#", 1)[0]
            if re.match(r"\s*(from|import)\s", code) or "subprocess" in code or "open(" in code:
                assert "oracle" not in code, (p, line)
    srcs = list((ROOT / "tuatara_b200" / "csrc").iterdir()) + list((ROOT / "include").iterdir()) + \
        list((ROOT / "tuatara_b200" / "bindings").iterdir())
    for p in srcs:
        for line in p.read_text().splitlines():
            if line.lstrip().startswith("#include") or "dlopen" in line or "fopen" in line:
                assert "oracle" not in line, (p, line)


def test_cpp_header_compiles_without_opencv(native_lib, tmp_path):
    src = tmp_path / "caller.cpp"
    src.write_text('#include "tuatara.h"\n'
                   "int main(int argc, char** argv) {\n"
                   "  tuatara::ImageView v; std::vector<OutputItem> r = image_to_data(v, \"\", \"out\");\n"
                   "  return static_cast<int>(r.size());\n}\n")
    from tuatara_b200 import _native

    exe = tmp_path / "caller"
    subprocess.run(["g++", "-std=c++14", f"-I{ROOT / 'include'}", str(src), "-o", str(exe), f"-L{_native.LIB_PATH.parent}",
                    "-ltuatara_b200", f"-Wl,-rpath,{_native.LIB_PATH.parent}"], check=True)
    r = subprocess.run([str(exe)], capture_output=True, text=True)
    assert r.returncode == 0 and "Please provide a value for weights_dir" in r.stderr  # tuatara.cpp:315-318


def test_pytuatara_module_signature(native_lib):
    from tuatara_b200 import _native

    sys.path.insert(0, str(_native.LIB_PATH.parent))
    import numpy as np
    import pytuatara

    doc = pytuatara.image_to_data.__doc__
    assert "image" in doc and "weights_dir" in doc and "outputs_dir" in doc  # bindings/python.cpp:57
    with pytest.raises(RuntimeError, match="Input array should have 3 dimensions"):  # python.cpp:15-17
        pytuatara.image_to_data(image=np.zeros((4, 4), np.uint8), weights_dir="w", outputs_dir="o")
    assert pytuatara.image_to_data(np.zeros((4, 4, 3), np.uint8), "", "o") == []
