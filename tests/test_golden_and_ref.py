"""Pinning of the oracle against the committed golden vectors that the reference's own linemodLevelup.cpp, compiled
unmodified (oracle/_ref), produced on the reference's fixture frame and template banks and on synthetic cases
(tests/golden/make_golden.py)."""
import importlib
import os

import numpy as np
import pytest

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load_golden():
    fr = np.load(os.path.join(GOLD, "frames_case1.npz"))
    frames = {tag: [[fr["%s_l%d_m%d" % (tag, l, m)] for m in range(2)] for l in range(2)] for tag in ("full", "half")}
    banks = {}
    for name in ("127", "63", "allScales"):
        b = np.load(os.path.join(GOLD, "bank_%s.npz" % name))
        banks[name] = (dict(class_begin=b["class_begin"], tmeta=b["tmeta"], feats=b["feats"].astype(np.int32)), b["T"].tolist())
    exp = np.load(os.path.join(GOLD, "expected_case1.npz"))
    cases = []
    for key in exp.files:
        bank, tag, thr = key.split("_")
        cases.append((bank, tag, float(thr), exp[key]))
    return frames, banks, cases


def test_oracle_reproduces_the_reference_golden_vectors(oracle):
    frames, banks, cases = load_golden()
    assert len(cases) == 12
    nonempty = 0
    for bank, tag, thr, want in cases:
        packed, T = banks[bank]
        got = oracle.match(frames[tag], T, packed, thr)
        assert np.array_equal(got, want), (bank, tag, thr)
        nonempty += len(want) > 0
    assert nonempty >= 9


def load_allscales_full():
    """The reference's own large-bank invocation (linemodLevelup/test.cpp:174-181): Detector() = 63 features, T = {5, 8},
    ALL 2989 templates of test/case1/allScales, threshold 80; plus threshold 75 (61 912 coarse candidates)."""
    from oracle import golden
    packed, T = golden.allscales_full_bank()
    exp = np.load(os.path.join(GOLD, "expected_allScales_full.npz"))
    cases = [(k.split("_")[0], float(k.split("_")[1]), exp[k], exp[k + "_stats"]) for k in exp.files if not k.endswith("_stats")]
    return packed, T, cases


def test_oracle_reproduces_the_full_allscales_golden_vectors(oracle):
    frames, _, _ = load_golden()
    packed, T, cases = load_allscales_full()
    assert int(packed["class_begin"][-1]) == 2989 and len(cases) == 3
    for tag, thr, want, stats in cases:
        got, st = oracle.match(frames[tag], T, packed, thr, want_stats=True)
        assert np.array_equal(got, want), (tag, thr)
        assert [int(st["coarse_candidates"]), int(st["coarse_byte_adds"]), int(st["refine_byte_adds"])] == stats.tolist()
    full75 = [c for c in cases if c[0] == "full" and c[1] == 75.0][0]
    assert len(full75[2]) == 157 and int(full75[3][0]) == 61912   # BASELINE.md section 2's candidate count


def test_golden_top_match_sits_on_the_ground_truth_box():
    # GT box of the object in the fixture frame: [331, 130, 65, 64] (linemodLevelup/test.cpp:86)
    _, _, cases = load_golden()
    top = [c for c in cases if c[0] == "127" and c[1] == "full" and c[2] == 75.0][0][3][0]
    assert abs(int(top["x"]) - 331) <= 4 and abs(int(top["y"]) - 130) <= 4


# synthetic cases on which the compiled reference (oracle/_ref) recorded its results in expected_synth.npz
SYNTH_CASES = [
    ([4, 8], 640, 480, 150, 70, 75.0), ([5, 8], 640, 480, 127, 50, 70.0), ([5, 8], 640, 480, 63, 50, 70.0),
    ([8], 320, 240, 40, 35, 60.0), ([2, 4, 8], 640, 512, 96, 35, 70.0), ([4, 8], 320, 256, 32, 3, -1.0),
]


def synth_case(synth, T, W, H, nf, n, thr):
    bank = synth.synth_bank(n, num_features=nf, levels=len(T), seed=21, class_ids=("01_template", "02_template"))
    q, _ = synth.synth_frame(W, H, levels=len(T), seed=9, bank=bank, plant=6, T=T)
    return q, bank.pack(bank.class_ids(), 2 * len(T))


def synth_key(T, W, H, nf, n, thr):
    return "T%s_%dx%d_f%d_n%d_thr%g" % ("-".join(str(t) for t in T), W, H, nf, n, thr)


def malformed_case(synth):
    """A bank whose level-1 colour template lost features: the reference's CV_Assert fires on it."""
    T = [4, 8]
    bank = synth.synth_bank(4, num_features=150, levels=2, seed=8)
    bank.classes["01_template"][2][2].features = bank.classes["01_template"][2][2].features[:10]
    q, _ = synth.synth_frame(320, 256, levels=2, seed=6)
    return q, T, bank.pack(bank.class_ids(), 4)


@pytest.mark.parametrize("T,W,H,nf,n,thr", SYNTH_CASES)
def test_oracle_equals_compiled_reference(oracle, synth, T, W, H, nf, n, thr):
    q, packed = synth_case(synth, T, W, H, nf, n, thr)
    want = np.load(os.path.join(GOLD, "expected_synth.npz"))[synth_key(T, W, H, nf, n, thr)]
    a = oracle.match(q, T, packed, thr)
    assert len(want) > 0 and np.array_equal(a, want)


def test_similarity_lut_equals_the_compiled_reference_table(oracle):
    assert np.array_equal(oracle.similarity_lut(), np.load(os.path.join(GOLD, "reference_tables.npz"))["similarity_lut"])


def test_reference_assertion_matches_oracle_error(oracle, synth):
    q, T, packed = malformed_case(synth)
    assert bool(np.load(os.path.join(GOLD, "expected_synth.npz"))["malformed_bank_raises"])   # the compiled reference raised
    with pytest.raises(RuntimeError):
        oracle.match(q, T, packed, 80.0)


@pytest.mark.gpu
def test_cuda_path_reproduces_the_reference_golden_vectors():
    lib = importlib.import_module("6dpose_b200._lib")
    frames, banks, cases = load_golden()
    for bank, tag, thr, want in cases:
        packed, T = banks[bank]
        nat = lib.NativeDetector(T)
        nat.load_bank(packed, 4)
        got = nat.match_quantized(frames[tag], thr)
        assert len(got) == len(want), (bank, tag, thr)
        for k in ("x", "y", "template_id", "similarity"):
            assert np.array_equal(got[k], want[k]), (bank, tag, thr, k)
        assert np.array_equal(got["class_index"], want["class_idx"])


@pytest.mark.gpu
def test_cuda_path_reproduces_the_full_allscales_golden_vectors():
    """All 2989 templates of the reference's allScales bank on its fixture frame, thresholds 80 (test.cpp:174-181) and
    75: match lists bit-identical to the compiled reference, candidate / algorithmic byte counters equal."""
    lib = importlib.import_module("6dpose_b200._lib")
    frames, _, _ = load_golden()
    packed, T, cases = load_allscales_full()
    nat = lib.NativeDetector(T)
    nat.load_bank(packed, 4)
    for tag, thr, want, stats in cases:
        got = nat.match_quantized(frames[tag], thr)
        assert len(got) == len(want), (tag, thr)
        for k in ("x", "y", "template_id", "similarity"):
            assert np.array_equal(got[k], want[k]), (tag, thr, k)
        c = nat.counters()
        assert [c["coarse_candidates"], c["scan_bytes"], c["refine_bytes"]] == stats.tolist(), (tag, thr)
