"""Detector.addTemplates (template extraction on the GPU, lm_extract_templates) against the host trainer
(training.add_template, which tests/test_training.py pins to the reference's own recorded output): the same ids,
and the same templates feature for feature, on views built from committed data only."""
import importlib
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
H, W = 480, 640


@pytest.fixture(scope="module")
def train_case():
    return np.load(os.path.join(GOLD, "train_case1.npz"))


def _synth_ramp():
    """A sawtooth colour ramp (strong, consistently oriented gradients everywhere) over a depth plane."""
    yy, xx = np.mgrid[0:H, 0:W]
    saw = (np.abs((xx + yy) % 64 - 32) * 8).clip(0, 255).astype(np.uint8)
    return np.stack([saw, saw // 2, 255 - saw], 2), (800 + 0.5 * xx).astype(np.uint16)


@pytest.fixture(scope="module")
def views(train_case):
    """About 48 seeded views: sources and masks, and a name per view."""
    synth = importlib.import_module("6dpose_b200.synth")
    rng = np.random.default_rng(2024)
    out = []
    for i, (rgb, dep, mk) in enumerate(synth.warp_views(train_case["rgb"], train_case["dep"], train_case["mask"], 30, seed=5)):
        if i in (3, 17):
            mk = None                                        # no mask
        elif i in (5, 21):
            mk = mk.copy()
            mk[:, : W // 2][mk[:, : W // 2] > 0] = 1          # mixed nonzero values 1 and 255
        elif i == 9:
            mk = np.zeros((0, 0), np.uint8)                 # empty = no mask
        out.append(("warp%d" % i, rgb, dep, mk))
    icp = np.load(os.path.join(GOLD, "icp_case1.npz"))
    model = icp["model"]
    for i, (rgb, dep, mk) in enumerate(synth.warp_views(synth.synth_rgbd(W, H, seed=31)[0], model, (model > 0).astype(np.uint8) * 255, 6,
                                                         seed=6)):
        out.append(("icp%d" % i, rgb, dep, mk))
    yy, xx = np.mgrid[0:H, 0:W]
    for i in range(8):
        rgb, dep = synth.synth_rgbd(W, H, seed=100 + i)
        cx, cy, a, b = rng.uniform(200, 440), rng.uniform(150, 330), rng.uniform(40, 120), rng.uniform(40, 120)
        if i % 2:
            mk = ((((xx - cx) / a) ** 2 + ((yy - cy) / b) ** 2) < 1).astype(np.uint8) * 255     # ellipse
        else:
            mk = np.zeros((H, W), np.uint8)
            mk[int(cy - b): int(cy + b), int(cx - a): int(cx + a)] = 255                  # rectangle
        out.append(("synth%d" % i, rgb, dep, mk))
    flat = np.full((H, W, 3), 90, np.uint8)                   # no gradient: colour fails at level 0
    out.append(("flat", flat, train_case["dep"], train_case["mask"]))
    ramp, plane = _synth_ramp()
    small = np.zeros((H, W), np.uint8)
    small[200:210, 300:340] = 255                            # normals fail at level 1 only (Detector())
    out.append(("small", ramp, plane, small))
    out.append(("ramp", ramp, plane, (((xx - 320) ** 2 + (yy - 240) ** 2) < 90 ** 2).astype(np.uint8) * 255))
    return out


def _host(pkg, det_args, views, class_id="obj"):
    det = pkg.Detector(*det_args)
    ids = [det.addTemplate([rgb, dep], class_id, mk) for _, rgb, dep, mk in views]
    return det, ids


def _gpu(pkg, det_args, views, class_id="obj"):
    det = pkg.Detector(*det_args)
    ids = det.addTemplates([[rgb, dep] for _, rgb, dep, _ in views], class_id, [mk for _, _, _, mk in views])
    return det, ids


def _same_bank(a, b, slots):
    ca, cb = a.bank.class_ids(), b.bank.class_ids()
    assert ca == cb
    pa, pb = a.bank.pack(ca, slots), b.bank.pack(cb, slots)
    for k in ("class_begin", "tmeta", "feats"):
        assert np.array_equal(pa[k], pb[k]), k


def test_known_answer_reference_training_fixture(pkg, train_case):
    det = pkg.Detector()
    assert det.addTemplates([[train_case["rgb"], train_case["dep"]]], "06_template", [train_case["mask"]]) == [0]
    got = det.bank.pack(["06_template"], 4)
    assert np.array_equal(got["tmeta"], train_case["tmeta"])
    assert np.array_equal(got["feats"], train_case["feats"].astype(np.int32))


@pytest.mark.parametrize("det_args", [(), (150, [4, 8]), (63, [2, 4, 8])], ids=["default", "nf150", "three_levels"])
def test_parity_with_the_host_trainer(pkg, views, det_args):
    host, want = _host(pkg, det_args, views)
    gpu, got = _gpu(pkg, det_args, views)
    names = [v[0] for v in views]
    assert got == want, [(n, g, w) for n, g, w in zip(names, got, want) if g != w]
    _same_bank(host, gpu, 2 * host.pyramid_levels)
    ok = [n for n, i in zip(names, got) if i >= 0]
    assert len(ok) >= 30 and "flat" not in ok
    if det_args == ():
        assert "small" not in ok and "ramp" in ok


def test_normals_fail_only_at_level_one(pkg, views):
    """The `small` view passes colour at both levels and normals at level 0 (so its failure is the level-1 normals)."""
    training = importlib.import_module("6dpose_b200.training")
    fe = importlib.import_module("6dpose_b200.frontend")
    _, rgb, dep, mk = [v for v in views if v[0] == "small"][0]
    got = []
    for m in range(2):
        pyr = fe.ColorPyramid(rgb, mk, 10.0, 63, 55.0) if m == 0 else fe.NormalPyramid(dep, mk, 2000, 50, 63, 2)
        for l in range(2):
            if l:
                pyr.pyrDown()
            got.append((training.extract_color_template if m == 0 else training.extract_normal_template)(pyr) is not None)
    assert got == [True, True, True, False]


def test_bank_semantics(pkg, views, tmp_path):
    mix = [v for v in views if v[0] in ("warp0", "flat", "warp1", "small", "synth1", "warp2")]
    # a class that already holds templates: ids continue; another class is left alone
    host, _ = _host(pkg, (), mix[:2])
    gpu, _ = _gpu(pkg, (), mix[:2])
    _host_ids = [host.addTemplate([r, d], "obj", m) for _, r, d, m in mix[2:]]
    _host_ids += [host.addTemplate([r, d], "other", m) for _, r, d, m in mix[:1]]
    gpu_ids = gpu.addTemplates([[r, d] for _, r, d, _ in mix[2:]], "obj", [m for _, _, _, m in mix[2:]])
    gpu_ids += gpu.addTemplates([[r, d] for _, r, d, _ in mix[:1]], "other", [m for _, _, _, m in mix[:1]])
    assert gpu_ids == _host_ids and gpu_ids[0] == 2 and -1 in gpu_ids
    _same_bank(host, gpu, 4)
    # writeClasses / readClasses round trip of a GPU-trained bank
    fmt = str(tmp_path / "%s.yaml")
    gpu.writeClasses(fmt)
    again = pkg.Detector()
    again.readClasses(gpu.classIds(), fmt)
    _same_bank(gpu, again, 4)
    # a class read from a packed .lmb file is unpacked to a list first
    gpu.writeClasses(str(tmp_path / "%s.lmb"))
    a, b = pkg.Detector(), pkg.Detector()
    a.readClasses(["obj"], str(tmp_path / "%s.lmb"))
    b.readClasses(["obj"], str(tmp_path / "%s.lmb"))
    ids_a = [a.addTemplate([r, d], "obj", m) for _, r, d, m in mix]
    ids_b = b.addTemplates([[r, d] for _, r, d, _ in mix], "obj", [m for _, _, _, m in mix])
    assert ids_a == ids_b and isinstance(b.bank.classes["obj"], list)
    _same_bank(a, b, 4)
    # an all-failing batch: no ids, the class exists anyway (LL.cpp:1947)
    c = pkg.Detector()
    flat = [v for v in views if v[0] == "flat"][0]
    assert c.addTemplates([[flat[1], flat[2]]] * 3, "09_template", [flat[3]] * 3) == [-1, -1, -1]
    assert c.numTemplates("09_template") == 0 and "09_template" in c.classIds()
    # no views: nothing to do, no class created (as an empty loop of addTemplate)
    empty = pkg.Detector()
    assert empty.addTemplates([], "x", []) == [] and "x" not in empty.classIds()


def test_errors(pkg, train_case):
    rgb, dep, mk = train_case["rgb"], train_case["dep"], train_case["mask"]
    det = pkg.Detector()
    with pytest.raises(TypeError):
        det.addTemplates([[rgb.astype(np.float32), dep]], "e", [mk])
    with pytest.raises(TypeError):
        det.addTemplates([[rgb, dep.astype(np.int32)]], "e", [mk])
    with pytest.raises(TypeError):
        det.addTemplates([[rgb, dep]], "e", [np.dstack([mk, mk, mk])])
    with pytest.raises(RuntimeError):
        det.addTemplates([[rgb, dep, dep]], "e", [mk])
    with pytest.raises(RuntimeError):
        det.addTemplates([[rgb, dep]], "e", [mk[:100]])
    with pytest.raises(RuntimeError, match="one size"):
        det.addTemplates([[rgb, dep], [rgb[:240, :320], dep[:240, :320]]], "e", [None, None])
    three = pkg.Detector(63, [2, 4, 8])
    with pytest.raises(RuntimeError, match="multiples of 2"):
        three.addTemplates([[rgb[:474], dep[:474]]], "e", [None])
    assert "e" not in det.classIds() and "e" not in three.classIds()
