"""Packed bank files (SURVEY.md section 8f-4): lossless against the YAML dialect of the reference
(LL.cpp:2093-2146), integrity-checked, and usable through Detector.readClasses / writeClasses."""
import hashlib
import importlib
import os
import time

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
bk = importlib.import_module("6dpose_b200.bank")
synth = importlib.import_module("6dpose_b200.synth")
pkg = importlib.import_module("6dpose_b200")


def bank_from_golden(name, class_id="06_template"):
    g = np.load(os.path.join(HERE, "golden", name))
    b = bk.TemplateBank()
    tm = g["tmeta"].copy()
    b.classes[class_id] = bk.PackedPyramids(tm, g["feats"], tm.shape[1] // 2)
    return b


def write_reference_yaml(name, path):
    """Writes the reference's bank file test/case1/<name>/06_template.yaml (name: 127 or allScales) byte for byte from the
    golden bank, adding the per-template `depth:` lines the bank arrays do not hold; checked against the file's SHA-256
    (tests/golden/make_golden.py)."""
    g = np.load(os.path.join(HERE, "golden", "reference_yaml.npz"))
    if name == "allScales":
        from oracle import golden
        packed, _ = golden.allscales_full_bank()
        b = bk.TemplateBank()
        b.classes["06_template"] = bk.PackedPyramids(packed["tmeta"], packed["feats"], 2)
    else:
        b = bank_from_golden("bank_%s.npz" % name)
    b.write_class("06_template", path, 2)
    if name + "_depth" in g.files:
        depth = iter(g[name + "_depth"].ravel().tolist())
        lines = []
        for ln in open(path).read().split("\n"):
            lines.append(ln)
            if ln.startswith("            pyramid_level: "):
                lines.append("            depth: %d" % next(depth))
        with open(path, "w") as fh:
            fh.write("\n".join(lines))
    assert hashlib.sha256(open(path, "rb").read()).hexdigest() == str(g[name + "_sha256"]), name
    return path


def same_pack(a, b):
    return all(np.array_equal(a[k], b[k]) for k in ("class_begin", "tmeta", "feats"))


def test_round_trip_yaml_packed_yaml(tmp_path):
    bank = synth.synth_bank(40, num_features=63, seed=3, class_ids=("01_template", "02_template"))
    ids = bank.class_ids()
    want = bank.pack(ids, 4)
    back = bk.TemplateBank()
    for cid in ids:
        bank.write_packed(cid, str(tmp_path / (cid + ".lmb")), 2)
        assert back.read_packed(str(tmp_path / (cid + ".lmb")), 2) == cid
    assert same_pack(back.pack(ids, 4), want)
    # Template objects materialise on demand and write back as the same YAML
    t = back.classes[ids[0]][3][1]
    u = bank.classes[ids[0]][3][1]
    assert (t.width, t.height, t.pyramid_level) == (u.width, u.height, u.pyramid_level)
    assert np.array_equal(t.features, u.features)
    back.write_class(ids[1], str(tmp_path / "b.yaml"), 2)
    bank.write_class(ids[1], str(tmp_path / "a.yaml"), 2)
    assert open(str(tmp_path / "a.yaml")).read() == open(str(tmp_path / "b.yaml")).read()


def test_reference_fixture_bank_survives_packing(tmp_path):
    """Golden subset (every 7th template) of the reference's committed allScales bank."""
    b = bank_from_golden("bank_allScales.npz")
    want = b.pack(["06_template"], 4)
    assert want["tmeta"].shape[0] == 427
    p = str(tmp_path / "06_template.lmb")
    b.write_packed("06_template", p, 2)
    r = bk.TemplateBank()
    r.read_packed(p, 2)
    assert same_pack(r.pack(["06_template"], 4), want)


def test_full_reference_bank_yaml_vs_packed(tmp_path):
    """The reference's own 2989-template YAML: parse, pack, reload -- identical, much smaller and faster."""
    REF_BANK = write_reference_yaml("allScales", str(tmp_path / "allScales.yaml"))
    t0 = time.perf_counter()
    y = bk.TemplateBank()
    y.read_class(REF_BANK, 2)
    t_yaml = time.perf_counter() - t0
    want = y.pack(["06_template"], 4)
    assert want["tmeta"].shape[0] == 2989
    p = str(tmp_path / "06_template.lmb")
    y.write_packed("06_template", p, 2)
    t0 = time.perf_counter()
    r = bk.TemplateBank()
    r.read_packed(p, 2)
    got = r.pack(["06_template"], 4)
    t_packed = time.perf_counter() - t0
    assert same_pack(got, want)
    assert t_packed < t_yaml
    assert os.path.getsize(p) * 4 < os.path.getsize(REF_BANK)
    print("yaml %.2f s (%d MB)  packed %.4f s (%.1f MB)" % (t_yaml, os.path.getsize(REF_BANK) >> 20, t_packed,
                                                          os.path.getsize(p) / 2 ** 20))


def test_errors_mirror_read_class(tmp_path):
    bank = synth.synth_bank(6, num_features=63, seed=4, class_ids=("01_template",))
    p = str(tmp_path / "c.lmb")
    bank.write_packed("01_template", p, 2)
    with pytest.raises(RuntimeError, match="pyramid_levels"):   # LL.cpp:2052
        bk.TemplateBank().read_packed(p, 3)
    b = bk.TemplateBank()
    b.read_packed(p, 2)
    with pytest.raises(RuntimeError, match="already loaded"):   # LL.cpp:2059
        b.read_packed(p, 2)
    blob = bytearray(open(p, "rb").read())
    blob[len(blob) // 2] ^= 0x10
    open(p, "wb").write(bytes(blob))
    with pytest.raises(RuntimeError, match="checksum"):
        bk.TemplateBank().read_packed(p, 2)
    open(p, "wb").write(bytes(blob[:-16]))
    with pytest.raises(RuntimeError):
        bk.TemplateBank().read_packed(p, 2)
    open(p, "wb").write(b"%YAML:1.0\n---\n")
    with pytest.raises(RuntimeError, match="not a packed"):
        bk.TemplateBank().read_packed(p, 2)
    with pytest.raises(RuntimeError, match="cannot open"):
        bk.TemplateBank().read_packed(str(tmp_path / "missing.lmb"), 2)


def test_detector_surface_and_cache(tmp_path, monkeypatch):
    bank = synth.synth_bank(12, num_features=63, seed=5, class_ids=("01_template", "02_template"))
    det = pkg.Detector(63, [4, 8])
    det.bank = bank
    det.writeClasses(str(tmp_path / "%s.yaml"))
    det.writeClasses(str(tmp_path / "%s.lmb"))
    want = bank.pack(bank.class_ids(), 4)
    d2 = pkg.Detector(63, [4, 8])
    d2.readClasses(["01_template", "02_template"], str(tmp_path / "%s.lmb"))
    assert same_pack(d2.bank.pack(d2.bank.class_ids(), 4), want)
    # YAML through the packed sibling cache
    monkeypatch.setenv("LINEMOD_B200_BANK_CACHE", "1")
    d3 = pkg.Detector(63, [4, 8])
    d3.readClasses(["01_template"], str(tmp_path / "%s.yaml"))
    side = str(tmp_path / "01_template.yaml.lmb")
    assert os.path.exists(side)
    d4 = pkg.Detector(63, [4, 8])
    d4.readClasses(["01_template"], str(tmp_path / "%s.yaml"))     # served by the cache
    assert isinstance(d4.bank.classes["01_template"], bk.PackedPyramids)
    assert same_pack(d4.bank.pack(["01_template"], 4), d3.bank.pack(["01_template"], 4))
    # a YAML newer than its cache wins
    b2 = synth.synth_bank(3, num_features=63, seed=6, class_ids=("01_template",))
    b2.write_class("01_template", str(tmp_path / "01_template.yaml"), 2)
    os.utime(str(tmp_path / "01_template.yaml"), (time.time() + 5, time.time() + 5))
    d5 = pkg.Detector(63, [4, 8])
    d5.readClasses(["01_template"], str(tmp_path / "%s.yaml"))
    assert d5.numTemplates() == 3
    # addTemplate on a packed class unpacks it first
    d4.bank.classes["01_template"] = list(d4.bank.classes["01_template"])
    assert len(d4.bank.classes["01_template"]) == d3.numTemplates("01_template")
