"""Acceptance run of the reference's own driver, linemod_and_levelup_test.py (north_star: "runs unchanged against the
new backend"; the calls it makes: Detector(150, [4, 8]) :19, readClasses :283, match(..., 75, ids, masks=[]) :324,
poseRefine().process(...) / getR / getT :363-368).

The script lives in the reference checkout, which is mounted in the build container only and must not be copied, so the
acceptance run is split in two halves that meet in a committed call trace (tests/golden/driver_trace.npz):

  * here (no GPU, reference checkout present): tools/run_reference_driver.py executes the UNMODIFIED script against
    `linemodLevelup_pybind` with the C-ABI handles replaced by oracle-backed stand-ins (test infrastructure: the CPU
    restatement + oracle/icp_oracle.py).  This checks the Python surface the script drives -- constructor, readClasses,
    match with its keyword, Match attributes, poseRefine surface, dtypes -- and that the recorded trace still equals the
    committed one;
  * on the GPU box: the recorded calls (same arrays, same arguments, same order) are replayed through the real module
    (CUDA backend) and must return the recorded match list bit-exactly and the recorded poses within 1e-4 (ICP parity
    is UNPINNED: the expected poses come from the ICP oracle, see oracle/icp_oracle.py).

`python tests/test_reference_driver.py --record` regenerates the trace."""
import importlib
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden", "driver_trace.npz")
sys.path.insert(0, os.path.join(ROOT, "tools"))
REF = importlib.import_module("run_reference_driver").REF   # the checkout the harness runs the script from
TOL = 1e-4


class OracleDetector:
    """Stand-in for _lib.NativeDetector backed by the CPU oracle (surface test only)."""

    def __init__(self, T, device=0):
        self.T = [int(t) for t in T]
        self.packed = None

    def load_bank(self, packed, slots):
        self.packed = packed
        self.class_sel = None

    def select(self, class_indices=None, shard_index=0, shard_count=1, layout=0):
        assert (shard_index, shard_count) == (0, 1)
        self.class_sel = None if class_indices is None else list(class_indices)

    def match_quantized(self, quantized, threshold):
        from oracle import oracle
        lib = importlib.import_module("6dpose_b200._lib")
        p = self.packed
        if self.class_sel is not None:  # the oracle matches every class of the dict it is given, in order
            cb, tm = p["class_begin"], p["tmeta"]
            parts = [tm[cb[c]:cb[c + 1]] for c in self.class_sel]
            sub = dict(class_begin=np.cumsum([0] + [len(x) for x in parts]).astype(np.int32),
                       tmeta=np.ascontiguousarray(np.concatenate(parts)), feats=p["feats"])
            w = oracle.match(quantized, self.T, sub, threshold)
            cls = np.asarray(self.class_sel, np.int32)[w["class_idx"]]
        else:
            w = oracle.match(quantized, self.T, p, threshold)
            cls = w["class_idx"]
        out = np.zeros(len(w), lib.MATCH_DTYPE)
        for k in ("x", "y", "similarity", "template_id"):
            out[k] = w[k]
        out["class_index"] = cls
        return out


class OracleIcp:
    """Stand-in for _lib.NativeIcp backed by oracle/icp_oracle.py."""

    def __init__(self, device=0):
        pass

    def process_batch(self, scene_depth, model_depths, sceneK, modelKs, Rs, ts, detect_xy, max_iterations=30):
        from oracle import icp_oracle
        n = len(model_depths)
        Ro, to, res = np.full((n, 3, 3), np.nan), np.full((n, 3), np.nan), np.zeros(n, np.float32)
        for i in range(n):
            r = icp_oracle.pose_refine(scene_depth, model_depths[i], sceneK, modelKs[i], Rs[i], np.asarray(ts[i]).reshape(3),
                                       int(detect_xy[i][0]), int(detect_xy[i][1]), max_iter=max_iterations)
            res[i] = r["residual"]
            if r["R"] is not None:
                Ro[i], to[i] = r["R"], r["t"].reshape(3)
        return Ro, to, res


def run_script_with_oracle_backends():
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    lib = importlib.import_module("6dpose_b200._lib")
    pr = importlib.import_module("6dpose_b200.pose_refine")
    harness = importlib.import_module("run_reference_driver")
    saved = (lib.NativeDetector, lib.NativeIcp, dict(pr._icp), os.environ.get("LINEMOD_B200_FRONTEND"), list(sys.argv))
    lib.NativeDetector, lib.NativeIcp = OracleDetector, OracleIcp
    pr._icp.clear()
    os.environ["LINEMOD_B200_FRONTEND"] = "cv2"  # the host front-end (frontend.py); the GPU one is tested in test_gpu_frontend.py
    sys.argv = ["linemod_and_levelup_test.py"]
    try:
        return harness.main(trace={})
    finally:
        lib.NativeDetector, lib.NativeIcp = saved[0], saved[1]
        pr._icp.clear()
        pr._icp.update(saved[2])
        if saved[3] is None:
            os.environ.pop("LINEMOD_B200_FRONTEND", None)
        else:
            os.environ["LINEMOD_B200_FRONTEND"] = saved[3]
        sys.argv = saved[4]
        for name in ("params", "params.dataset_params", "pysixd", "pysixd.inout", "pysixd.renderer", "pysixd.view_sampler", "pysixd.misc"):
            sys.modules.pop(name, None)


def trace_arrays(trace):
    lib = importlib.import_module("6dpose_b200._lib")
    assert len(trace["match_calls"]) == 1
    mc = trace["match_calls"][0]
    m = np.zeros(len(mc["matches"]), lib.MATCH_DTYPE)
    for i, x in enumerate(mc["matches"]):
        assert x.class_id == "06_template"
        m[i] = (x.x, x.y, x.similarity, 0, x.template_id)
    out = dict(rgb=mc["sources"][0], depth=mc["sources"][1], render=trace["render"], threshold=np.float64(mc["threshold"]),
               T=np.asarray(mc["T"], np.int32), num_features=np.int32(mc["num_features"]), matches=m,
               n_refine=np.int32(len(trace["refine_calls"])))
    for i, rc in enumerate(trace["refine_calls"]):
        a = rc["args"]
        out.update({"rf%d_modelDepth" % i: a[1], "rf%d_sceneK" % i: a[2], "rf%d_modelK" % i: a[3], "rf%d_modelR" % i: a[4],
                    "rf%d_modelT" % i: a[5], "rf%d_xy" % i: np.asarray([int(a[6]), int(a[7])], np.int32),
                    "rf%d_R" % i: rc["R"], "rf%d_t" % i: rc["t"], "rf%d_residual" % i: np.float64(rc["residual"])})
        assert np.array_equal(a[0], mc["sources"][1])  # the scene depth handed to poseRefine is the frame's
    return out


@pytest.mark.skipif(not os.path.isdir(os.path.join(REF, "linemodLevelup")), reason="reference checkout not found")
def test_unmodified_driver_runs_against_the_module_surface(oracle):
    trace = run_script_with_oracle_backends()
    mc = trace["match_calls"][0]
    # what the script hands the module (SURVEY 8b): RGB u8 HxWx3, depth u16 mm, threshold 75, one class id, masks=[]
    assert mc["sources"][0].dtype == np.uint8 and mc["sources"][0].shape == (480, 640, 3)
    assert mc["sources"][1].dtype == np.uint16 and mc["sources"][1].shape == (480, 640)
    assert (mc["threshold"], mc["class_ids"], mc["masks"], mc["T"], mc["num_features"]) == (75, ["06_template"], [], [4, 8], 150)
    assert len(mc["matches"]) > 10 and len(trace["refine_calls"]) == 3   # top5 = 3 survivors of the NMS
    for rc in trace["refine_calls"]:
        assert [a.dtype for a in rc["args"][:6]] == [np.uint16, np.uint16, np.float32, np.float32, np.float32, np.float32]
        assert rc["R"].shape == (3, 3) and rc["R"].dtype == np.float64 and rc["t"].shape == (3, 1) and 0 <= rc["residual"] <= 1
    got = trace_arrays(trace)
    gold = np.load(GOLD)
    assert sorted(gold.files) == sorted(got.keys())
    for k in gold.files:
        if k.startswith("rf") and k[-2:] in ("_R", "_t"):
            assert np.allclose(got[k], gold[k], rtol=0, atol=1e-9), k
        else:
            assert np.array_equal(got[k], gold[k]), k
    # one of the three poses the script refines sits on the ground-truth box of the fixture frame, [331, 130, 65, 64]
    # (linemodLevelup/test.cpp:86)
    assert any(abs(int(rc["args"][6]) - 331) <= 6 and abs(int(rc["args"][7]) - 130) <= 6 for rc in trace["refine_calls"])


@pytest.mark.gpu
def test_recorded_driver_calls_through_the_cuda_backend(tmp_path):
    """Replays the script's calls, in its order and with its arguments, through the real module."""
    gold = np.load(GOLD)
    bk = importlib.import_module("6dpose_b200.bank")
    mod = importlib.import_module("linemodLevelup_pybind")
    from oracle import golden
    packed, _ = golden.allscales_full_bank()   # the bank the recorded run read
    bank = bk.TemplateBank()
    bank.classes["06_template"] = bk.PackedPyramids(packed["tmeta"], packed["feats"], 2)   # one class: feat_begin is class-local
    bank.write_packed("06_template", str(tmp_path / "06_template.lmb"), 2)
    for frontend in ("gpu", "cv2"):
        detector = mod.Detector(int(gold["num_features"]), gold["T"].tolist())      # :19
        detector.frontend = frontend
        detector.readClasses(["06_template"], str(tmp_path / "%s.lmb"))            # :283
        matches = detector.match([gold["rgb"], gold["depth"]], float(gold["threshold"]), ["06_template"], masks=[])   # :324
        want = gold["matches"]
        assert len(matches) == len(want) > 0
        for m, w in zip(matches, want):
            assert (m.x, m.y, m.template_id, m.class_id) == (int(w["x"]), int(w["y"]), int(w["template_id"]), "06_template")
            assert np.float32(m.similarity) == w["similarity"]
    for i in range(int(gold["n_refine"])):                                          # :363-368
        p = mod.poseRefine()
        x, y = [int(v) for v in gold["rf%d_xy" % i]]
        p.process(gold["depth"], gold["rf%d_modelDepth" % i], gold["rf%d_sceneK" % i], gold["rf%d_modelK" % i],
                  gold["rf%d_modelR" % i], gold["rf%d_modelT" % i], x, y)
        R, t = p.getR(), p.getT()
        assert R.shape == (3, 3) and t.shape == (3, 1)
        assert np.linalg.norm(R - gold["rf%d_R" % i]) / np.linalg.norm(gold["rf%d_R" % i]) <= TOL
        assert np.linalg.norm(t - gold["rf%d_t" % i]) / np.linalg.norm(gold["rf%d_t" % i]) <= TOL
        assert abs(p.getResidual() - float(gold["rf%d_residual" % i])) <= 1e-6


if __name__ == "__main__" and "--record" in sys.argv:
    sys.path.insert(0, ROOT)
    from oracle import oracle as _o
    _o.build()
    np.savez_compressed(GOLD, **trace_arrays(run_script_with_oracle_backends()))
    print("wrote", GOLD, os.path.getsize(GOLD), "bytes")
