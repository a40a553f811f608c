#!/usr/bin/env python
"""Regenerates tests/golden/*.npz from the reference's own fixtures (needs the reference checkout named by
LM_REFERENCE_ROOT and oracle/_ref built from it: `make -C oracle ref REF=$LM_REFERENCE_ROOT/linemodLevelup`).

Inputs : linemodLevelup/test/case1/0000_{rgb,dep}.png (+ _half), banks 63/, 127/, allScales/
         (reference: linemodLevelup/test.cpp:90-128, 174-181 -- the invocations the reference's own
         test driver makes: Detector(127,{5,8}) + thr 75, Detector() + allScales + thr 80).
Stored : the quantized label pyramids produced by 6dpose_b200/frontend.py (so the GPU box needs no
         reference checkout), the packed template banks, and the expected match lists computed by the
         REFERENCE'S OWN CODE (oracle/_ref = linemodLevelup.cpp compiled unmodified).
"""
import gzip
import hashlib
import importlib
import os
import re
import sys

import cv2
import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
REF = os.path.join(os.environ.get("LM_REFERENCE_ROOT", ""), "linemodLevelup")
CASE = os.path.join(REF, "test", "case1", "")
OUT = os.path.dirname(os.path.abspath(__file__))


def main():
    fe = importlib.import_module("6dpose_b200.frontend")
    bk = importlib.import_module("6dpose_b200.bank")
    from oracle import oracle, ref
    assert ref.build(), "oracle/_ref could not be built (is /root/reference mounted?)"

    frames = {}
    for tag, suffix in (("full", ""), ("half", "_half")):
        rgb = cv2.imread(CASE + "0000_rgb%s.png" % suffix)  # BGR, as cv::imread in test.cpp:90
        dep = cv2.imread(CASE + "0000_dep%s.png" % suffix, cv2.IMREAD_UNCHANGED)
        q = fe.quantize_pyramid([rgb, dep], 2)
        frames[tag] = q
    np.savez_compressed(os.path.join(OUT, "frames_case1.npz"),
                        **{"%s_l%d_m%d" % (tag, l, m): frames[tag][l][m] for tag in frames for l in range(2) for m in range(2)})

    cases = []
    for bank_name, limit, T, thresholds in (("127", None, [5, 8], (75.0, 60.0)), ("63", None, [5, 8], (75.0, 60.0)),
                                           ("allScales", 7, [5, 8], (75.0, 65.0))):
        b = bk.TemplateBank()
        b.read_class(CASE + bank_name + "/06_template.yaml", 2)
        if limit:  # every limit-th template of the 2989 (all radii 600..1800 mm stay represented)
            b.classes["06_template"] = b.classes["06_template"][::limit]
        packed = b.pack(b.class_ids(), 4)
        np.savez_compressed(os.path.join(OUT, "bank_%s.npz" % bank_name), class_begin=packed["class_begin"],
                            tmeta=packed["tmeta"], feats=packed["feats"].astype(np.int16), T=np.asarray(T, np.int32))
        for tag in frames:
            for thr in thresholds:
                want = ref.match(frames[tag], T, packed, thr)
                again = oracle.match(frames[tag], T, packed, thr)
                assert np.array_equal(want, again), "restatement and reference disagree"
                key = "%s_%s_%g" % (bank_name, tag, thr)
                cases.append((key, want))
                print(key, len(want), want[:2])
    np.savez_compressed(os.path.join(OUT, "expected_case1.npz"), **{k: v for k, v in cases})


def make_allscales_full():
    """bank_allScales_full_{a,b}.npz / expected_allScales_full.npz: the reference's own large-bank invocation
    (linemodLevelup/test.cpp:174-181: Detector() -> T = {5, 8}, 63 features, readClasses(allScales), match at 80) on
    the fixture frame with ALL 2989 templates, plus threshold 75 (the drivers' value, linemod_and_levelup_test.py:324;
    61 912 coarse candidates) and the half-occluded frame at 80.  Expected lists by oracle/_ref (the reference's code)."""
    fe = importlib.import_module("6dpose_b200.frontend")
    bk = importlib.import_module("6dpose_b200.bank")
    from oracle import oracle, ref
    assert ref.build()
    b = bk.TemplateBank()
    b.read_class(CASE + "allScales/06_template.yaml", 2)
    packed = b.pack(b.class_ids(), 4)
    T = [5, 8]
    save_allscales_full_bank(packed, T)
    out = {}
    for tag, suffix, thresholds in (("full", "", (80.0, 75.0)), ("half", "_half", (80.0,))):
        rgb = cv2.imread(CASE + "0000_rgb%s.png" % suffix)
        dep = cv2.imread(CASE + "0000_dep%s.png" % suffix, cv2.IMREAD_UNCHANGED)
        q = fe.quantize_pyramid([rgb, dep], 2)
        for thr in thresholds:
            want, st = ref.match(q, T, packed, thr), None
            again, st = oracle.match(q, T, packed, thr, want_stats=True)
            assert np.array_equal(want, again), "restatement and reference disagree"
            out["%s_%g" % (tag, thr)] = want
            out["%s_%g_stats" % (tag, thr)] = np.asarray([int(st["coarse_candidates"]), int(st["coarse_byte_adds"]),
                                                           int(st["refine_byte_adds"])], np.int64)
            print("allScales full", tag, thr, len(want), want[:2], {k: int(v) for k, v in st.items()})
    np.savez_compressed(os.path.join(OUT, "expected_allScales_full.npz"), **out)


def save_allscales_full_bank(packed, T):
    """bank_allScales_full_{a,b}.npz: the packed bank, its features split at a template boundary so that each file stays
    under 1 MB; read back with oracle.golden.allscales_full_bank()."""
    assert packed["feats"].max() < 256 and packed["feats"].min() >= 0
    tm = packed["tmeta"].astype(np.int32)
    cut = int(tm[len(tm) // 2, 0, 2])
    feats = packed["feats"].astype(np.uint8)
    np.savez_compressed(os.path.join(OUT, "bank_allScales_full_a.npz"), class_begin=packed["class_begin"], tmeta=tm,
                        feats=feats[:cut], T=np.asarray(T, np.int32))
    np.savez_compressed(os.path.join(OUT, "bank_allScales_full_b.npz"), feats=feats[cut:])


def make_reference_tables():
    """reference_tables.npz: the reference's normal quantization table (linemodLevelup/normal_lut.i) and the similarity
    table of the compiled reference (oracle/_ref), the one SIMILARITY_LUT line linemodLevelup.cpp leaves active."""
    from oracle import ref
    body = open(os.path.join(REF, "normal_lut.i")).read()
    body = body[body.index("{"):]
    normal = np.array([int(x) for x in re.findall(r"\d+", body)], np.uint8)[:8000].reshape(20, 20, 20)
    lines = open(os.path.join(REF, "linemodLevelup.cpp")).read().split("\n")
    active = [ln for ln in lines if ln.startswith("CV_DECL_ALIGNED(16) static const unsigned char SIMILARITY_LUT")]
    assert len(active) == 1
    sim = ref.similarity_lut()
    assert sim.tolist() == [int(v) for v in re.search(r"\{(.*)\}", active[0]).group(1).split(",")]
    np.savez_compressed(os.path.join(OUT, "reference_tables.npz"), normal_lut=normal, similarity_lut=sim)


def make_synth_expected():
    """expected_synth.npz: the compiled reference's match lists on the synthetic cases of tests/test_golden_and_ref.py,
    and whether it rejects that module's malformed bank."""
    from oracle import oracle, ref
    sys.path.insert(0, os.path.dirname(OUT))
    tg = importlib.import_module("test_golden_and_ref")
    synth = importlib.import_module("6dpose_b200.synth")
    out = {}
    for case in tg.SYNTH_CASES:
        q, packed = tg.synth_case(synth, *case)
        want = ref.match(q, case[0], packed, case[-1])
        assert len(want) > 0 and np.array_equal(want, oracle.match(q, case[0], packed, case[-1]))
        out[tg.synth_key(*case)] = want
    q, T, packed = tg.malformed_case(synth)
    try:
        ref.match(q, T, packed, 80.0)
        out["malformed_bank_raises"] = np.bool_(False)
    except RuntimeError:
        out["malformed_bank_raises"] = np.bool_(True)
    np.savez_compressed(os.path.join(OUT, "expected_synth.npz"), **out)


def make_yaml_fixtures():
    """reference_yaml.npz: the SHA-256 of the reference's bank files 127/ and allScales/06_template.yaml, which
    tests/test_bank_packed.py rewrites byte for byte from bank_127.npz / bank_allScales_full_{a,b}.npz plus the
    per-template `depth:` values of allScales (the bank arrays do not hold them).  writeClasses_06_template.yaml.gz:
    the reference's recorded writeClasses output (an older dialect with a float depth: key), as it is."""
    out = {}
    for name in ("127", "allScales"):
        blob = open(CASE + name + "/06_template.yaml", "rb").read()
        out[name + "_sha256"] = np.str_(hashlib.sha256(blob).hexdigest())
        depth = re.findall(rb"^ *depth: (.*)$", blob, re.M)
        if depth:
            assert all(d == b"%d" % int(d) for d in depth)
            out[name + "_depth"] = np.asarray([int(d) for d in depth], np.int32).reshape(-1, 4)
    np.savez_compressed(os.path.join(OUT, "reference_yaml.npz"), **out)
    with open(os.path.join(OUT, "writeClasses_06_template.yaml.gz"), "wb") as fh:
        fh.write(gzip.compress(open(CASE + "writeClasses/06_template.yaml", "rb").read(), 9, mtime=0))


if __name__ == "__main__":
    main()
    make_allscales_full()
    make_reference_tables()
    make_synth_expected()
    make_yaml_fixtures()


def make_train_golden():
    """train_case1.npz: the reference's training fixture (test.cpp:36-51 train_test: train_{rgb,dep,mask}.png
    -> Detector().addTemplate -> writeClasses/06_template.yaml, the reference's own recorded output)."""
    bk = importlib.import_module("6dpose_b200.bank")
    rgb = cv2.imread(CASE + "train_rgb.png")
    dep = cv2.imread(CASE + "train_dep.png", cv2.IMREAD_UNCHANGED)
    mask = cv2.cvtColor(cv2.imread(CASE + "train_mask.png"), cv2.COLOR_RGB2GRAY)
    ref = bk.TemplateBank()
    ref.read_class(CASE + "writeClasses/06_template.yaml", 2)
    p = ref.pack(["06_template"], 4)
    np.savez_compressed(os.path.join(OUT, "train_case1.npz"), rgb=rgb, dep=dep, mask=mask, tmeta=p["tmeta"],
                        feats=p["feats"].astype(np.int16))


if __name__ == "__main__":
    make_train_golden()
    # frame_crop_case1.npz: a 400x320 window of the reference's fixture frame around the object (raw RGB-D,
    # for the GPU front-end test)
    rgb = cv2.imread(CASE + "0000_rgb.png")
    dep = cv2.imread(CASE + "0000_dep.png", cv2.IMREAD_UNCHANGED)
    np.savez_compressed(os.path.join(OUT, "frame_crop_case1.npz"), rgb=rgb[40:360, 200:600].copy(), dep=dep[40:360, 200:600].copy())
