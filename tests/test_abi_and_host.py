"""CPU-side checks of the drop-in boundary: the C-ABI library loads and exports every symbol the
header declares, refuses to run without a GPU (no fallback), and the host mirror keeps the
reference's Python surface (linemodLevelup/pybind11.cpp:7-35)."""
import ctypes
import importlib
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    text = open(os.path.join(ROOT, "include", "linemod_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(lm_[a-z_0-9]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    lib = importlib.import_module("6dpose_b200._lib")
    L = lib.load()
    names = declared_symbols()
    assert len(names) >= 20
    for n in names:
        assert hasattr(L, n), "liblinemod_b200.so does not export %s" % n
    assert sorted(lib.SYMBOLS) == names, "6dpose_b200/_lib.py SYMBOLS out of date with the header"


def test_no_cpu_fallback_without_a_device():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    lib = importlib.import_module("6dpose_b200._lib")
    with pytest.raises(lib.LinemodLibraryError) as e:
        lib.NativeDetector([4, 8])
    assert "no CPU fallback" in str(e.value)


def test_product_path_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "6dpose_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".cpp", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle", src, re.M), f
                assert "lm_oracle" not in src and "liblm_ref" not in src, f
    shim = open(os.path.join(ROOT, "linemodLevelup_pybind", "__init__.py")).read()
    assert "oracle" not in shim


def test_python_surface_matches_the_reference_binding():
    mod = importlib.import_module("linemodLevelup_pybind")
    for cls in ("Detector", "Match", "poseRefine"):
        assert hasattr(mod, cls)
    m = mod.Match()
    for attr in ("x", "y", "similarity", "class_id", "template_id"):
        assert hasattr(m, attr)
    d0, d1, d2 = mod.Detector(), mod.Detector([4, 8]), mod.Detector(150, [4, 8])
    assert (d0.num_features, d0.T_at_level) == (63, [5, 8])      # LL.cpp:1663-1672
    assert (d1.num_features, d1.T_at_level) == (63, [4, 8])      # LL.cpp:1674-1682
    assert (d2.num_features, d2.T_at_level) == (150, [4, 8])     # LL.cpp:1684-1692
    for name in ("addTemplate", "writeClasses", "readClasses", "match", "getTemplates"):
        assert callable(getattr(d2, name))
    with pytest.raises(TypeError):
        d2.getTemplates("x", 0)                                   # unregistered return type in the reference
    with pytest.raises(TypeError):
        d2.match([np.zeros((8, 8, 3), np.uint8), np.zeros((8, 8), np.uint16)], 75, [])  # masks default not convertible
    p = mod.poseRefine()
    assert p.getResidual() == -1 and p.getR() is None and p.getT() is None   # LL.h:10, empty Mat -> None


def test_bank_yaml_round_trip(tmp_path, synth):
    bk = importlib.import_module("6dpose_b200.bank")
    bank = synth.synth_bank(5, num_features=16, levels=2, seed=2, class_ids=("03_template",))
    fmt = str(tmp_path / "%s.yaml")
    bank.write_class("03_template", fmt % "03_template", 2)
    again = bk.TemplateBank()
    assert again.read_class(fmt % "03_template", 2) == "03_template"
    a, b = bank.pack(["03_template"], 4), again.pack(["03_template"], 4)
    for k in a:
        assert np.array_equal(a[k], b[k])
    # OpenCV itself can parse what we write (same dialect as the reference's FileStorage output)
    import cv2
    fs = cv2.FileStorage(fmt % "03_template", cv2.FILE_STORAGE_READ)
    assert fs.getNode("class_id").string() == "03_template"
    assert int(fs.getNode("pyramid_levels").real()) == 2
    tps = fs.getNode("template_pyramids")
    assert tps.size() == 5
    f0 = tps.at(0).getNode("templates").at(0).getNode("features").at(0)
    assert [int(f0.at(i).real()) for i in range(3)] == bank.classes["03_template"][0][0].features[0].tolist()
    with pytest.raises(RuntimeError):
        again.read_class(fmt % "03_template", 2)      # class already loaded, LL.cpp:2059
    with pytest.raises(RuntimeError):
        bk.TemplateBank().read_class(fmt % "03_template", 3)  # pyramid_levels mismatch, LL.cpp:2052


def test_reads_the_reference_fixture_banks(tmp_path):
    from test_bank_packed import write_reference_yaml
    bk = importlib.import_module("6dpose_b200.bank")
    b = bk.TemplateBank()
    b.read_class(write_reference_yaml("127", str(tmp_path / "127.yaml")), 2)
    tps = b.classes["06_template"]
    assert len(tps) == 89 and len(tps[0]) == 4
    assert tps[0][0].features.shape == (127, 3) and tps[0][2].features.shape == (63, 3)
    assert (tps[0][0].width, tps[0][0].height) == (37, 72)
    assert tps[0][0].features[0].tolist() == [3, 12, 0]
    old = bk.TemplateBank()
    old.read_class(os.path.join(ROOT, "tests", "golden", "writeClasses_06_template.yaml.gz"), 2)   # older dialect, float depth: key
    assert old.num_templates() == 1


def test_finish_orders_shuffled_records_and_validates_boxes():
    """lm_finish = (work, seq) ordering (counting sort inside the library) + the reference's std::sort /
    std::unique: any permutation of the same records gives the same matches; lm_set_boxes checks its input.
    Host-only handle: no GPU involved."""
    lib = importlib.import_module("6dpose_b200._lib")
    synth = importlib.import_module("6dpose_b200.synth")
    bank = synth.synth_bank(30, num_features=63, seed=9, class_ids=("01_template", "02_template"))
    packed = bank.pack(bank.class_ids(), 4)
    nat = lib.NativeDetector([4, 8], device=-1)
    nat.load_bank(packed, 4)
    nat.select(None, 0, 1)
    rng = np.random.RandomState(3)
    n = 4000
    rec = np.zeros(n, lib.RECORD_DTYPE)
    rec["work"] = rng.randint(0, 60, n)
    rec["seq"] = rng.permutation(n)          # unique (work, seq) pairs
    rec["x"] = rng.randint(0, 40, n) * 4
    rec["y"] = rng.randint(0, 30, n) * 4
    rec["similarity"] = (rng.randint(750, 1000, n) / 10.0).astype(np.float32)  # many ties
    want = nat.finish(rec[np.lexsort((rec["seq"], rec["work"]))])
    for _ in range(3):
        got = nat.finish(rec[rng.permutation(n)])
        assert got.tobytes() == want.tobytes()
    assert len(want) <= n and np.all(np.diff(want["similarity"]) <= 0)
    bad = rec.copy()
    bad["work"][5] = 60                       # outside the selection
    with pytest.raises(RuntimeError):
        nat.finish(bad)
    G = packed["tmeta"].shape[0]
    nat.set_boxes(np.full((G, 2), 50, np.int32))
    nat.set_boxes(None)
    with pytest.raises(RuntimeError):
        nat.set_boxes(np.full((G + 1, 2), 50, np.int32))
    with pytest.raises(RuntimeError):
        nat.set_boxes(np.full((G, 2), 40000, np.int32))
    with pytest.raises(lib.LinemodLibraryError):   # GPU stages refuse on a host-only handle
        nat.enqueue_post(0.5, 3)
