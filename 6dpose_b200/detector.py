"""Host-side mirror of the reference's Python surface (linemodLevelup/pybind11.cpp:7-35).

`Detector`, `Match` and `poseRefine` keep the reference's names, argument order, keyword names and
error behaviour; underneath, `Detector.match` calls the C-ABI library (CUDA, sm_100a) through
ctypes.  The quantization front-end runs on the GPU (or cv2, `Detector.frontend`); addTemplate extracts on the
host (cv2, as the reference does) and addTemplates extracts many views at once on the GPU.
"""
import os

import numpy as np

from . import _lib, frontend
from .bank import TemplateBank


class Match:
    """linemodLevelup::Match (pybind11.cpp:16-22): default-constructible, read/write attributes."""
    __slots__ = ("x", "y", "similarity", "class_id", "template_id")

    def __init__(self, x=0, y=0, similarity=0.0, class_id="", template_id=0):
        # the reference binds only the default constructor; the arguments are this module's fast path
        self.x = x
        self.y = y
        self.similarity = similarity
        self.class_id = class_id
        self.template_id = template_id

    def __repr__(self):
        return "Match(x=%d, y=%d, similarity=%.4f, class_id=%r, template_id=%d)" % (
            self.x, self.y, self.similarity, self.class_id, self.template_id)


def _default_device():
    for key in ("LINEMOD_B200_DEVICE", "LOCAL_RANK"):
        v = os.environ.get(key)
        if v is not None and v != "":
            return int(v)
    return 0


class Detector:
    """linemodLevelup::Detector as bound at pybind11.cpp:25-34.

    Detector()                      -> 63 features, T = [5, 8]          (LL.cpp:1663-1672)
    Detector(T)                     -> 63 features, T as given          (LL.cpp:1674-1682)
    Detector(num_features, T)       -> ColorGradient(10, nf, 55), DepthNormal(2000, 50, nf, 2)  (LL.cpp:1684-1692)
    """

    def __init__(self, *args):
        if len(args) == 0:
            nf, T = 63, [5, 8]
        elif len(args) == 1:
            nf, T = 63, list(args[0])
        elif len(args) == 2:
            nf, T = int(args[0]), list(args[1])
        else:
            raise TypeError("Detector(): incompatible constructor arguments")
        if not all(isinstance(t, (int, np.integer)) for t in T):
            raise TypeError("Detector(): T must be a list of ints")
        self.num_features = nf
        self.T_at_level = [int(t) for t in T]
        self.pyramid_levels = len(self.T_at_level)
        self.bank = TemplateBank()
        self._native = None
        self._bank_dirty = True
        self._class_order = []
        self._selection = None
        self._peers = None  # (rank, world) once dist.connect_peers has wired the fused exchange
        self.device = _default_device()
        self.shard = (0, 1)  # (index, count): template shard matched by this process (multi-GPU)
        self.shard_layout = _lib.SHARD_CONTIGUOUS
        # quantization front-end used by match(): "gpu" (CUDA, lm_match_images) or "cv2" (host, frontend.py);
        # both produce the same label images (tests/test_gpu_frontend.py)
        self.frontend = os.environ.get("LINEMOD_B200_FRONTEND", "gpu")

    # ---- template IO ----------------------------------------------------------------------
    def readClasses(self, class_ids, format):
        """Detector::readClasses, LL.cpp:2124-2134 (format is a printf pattern with one %s).

        Beyond the reference: a pattern ending in ".lmb" names packed bank files (bank.py), and with
        LINEMOD_B200_BANK_CACHE=1 a YAML is read through a packed sibling `<file>.lmb` (built on first use)."""
        for cid in class_ids:
            self.bank.read_any(format % cid, self.pyramid_levels)
        self._bank_dirty = True

    def writeClasses(self, format):
        """Detector::writeClasses, LL.cpp:2136-2146 (".lmb" pattern: packed bank files)."""
        from .bank import PACKED_SUFFIX
        for cid in self.bank.class_ids():
            if (format % cid).endswith(PACKED_SUFFIX):
                self.bank.write_packed(cid, format % cid, self.pyramid_levels)
            else:
                self.bank.write_class(cid, format % cid, self.pyramid_levels)

    def addTemplate(self, sources, class_id, object_mask):
        """Detector::addTemplate, LL.cpp:1943-1975: returns the template id, or -1 on failure."""
        from . import training
        tid = training.add_template(self, sources, class_id, object_mask)
        if tid >= 0:
            self._bank_dirty = True
        return tid

    def addTemplates(self, sources_list, class_id, object_masks):
        """Beyond the reference: addTemplate for many views of one size, extracted on the GPU in one call
        (lm_extract_templates).  Returns list[int] of template ids (-1 where extraction fails), and leaves the bank,
        feature for feature, as [addTemplate(s, class_id, m) for s, m in zip(sources_list, object_masks)] would.
        object_masks entries may be None or empty (no mask).  The image size must be a multiple of
        2^(pyramid_levels - 1); addTemplate serves other sizes."""
        from . import training
        if self._native is None:
            self._native = _lib.NativeDetector(self.T_at_level, self.device)
            self._bank_dirty = True
        ids = training.add_templates(self, self._native, list(sources_list), class_id, list(object_masks))
        if any(i >= 0 for i in ids):
            self._bank_dirty = True
        return ids

    def getTemplates(self, class_id, template_id):
        # The reference returns std::vector<Template>, a type pybind11.cpp never registers: calling it
        # from Python raises TypeError.  Kept for surface parity.
        raise TypeError("Unable to convert function return value to a Python type! (Template is not bound)")

    def numTemplates(self, class_id=None):
        return self.bank.num_templates(class_id)

    def classIds(self):
        return self.bank.class_ids()

    # ---- matching -------------------------------------------------------------------------
    def _ensure_native(self):
        if self._native is None:
            self._native = _lib.NativeDetector(self.T_at_level, self.device)
            self._bank_dirty = True
        if self._bank_dirty:
            self._class_order = self.bank.class_ids()  # std::map iteration order
            packed = self.bank.pack(self._class_order, self.pyramid_levels * 2)
            self._native.load_bank(packed, self.pyramid_levels * 2)
            self._bank_dirty = False
            self._selection = None
        return self._native

    def _select(self, class_ids):
        nat = self._ensure_native()
        if not class_ids:
            sel = None  # all classes, map order (LL.cpp:1753-1759)
        else:
            index = {c: i for i, c in enumerate(self._class_order)}
            sel = [index[c] for c in class_ids if c in index]  # unknown ids are skipped (LL.cpp:1765-1767)
        key = (None if sel is None else tuple(sel), self.shard, self.shard_layout)
        if key != self._selection:
            nat.select(sel, self.shard[0], self.shard[1], self.shard_layout)
            self._selection = key
        return nat

    def _whole_bank_only(self, what):
        # a detector left holding ONE template shard (dist.py) would silently return that shard's matches only
        if self.shard[1] > 1 and self._peers is None:
            raise RuntimeError("%s on a detector that holds template shard %d of %d without a connected peer exchange: "
                               "use dist.match_quantized_sharded, or reset detector.shard = (0, 1)" % (what, self.shard[0], self.shard[1]))

    def quantize(self, sources, masks=None):
        """The host front-end: list over levels of [color_labels, normal_labels] (u8)."""
        return frontend.quantize_pyramid(sources, self.pyramid_levels, masks, self.num_features)

    def match(self, sources, threshold, class_ids, masks=None):
        """Detector::match (LL.cpp:1702-1777) -> list[Match], sorted, duplicates pruned.

        As in the reference binding the declared default for `masks` is not convertible; every caller
        passes masks=[] (linemod_and_levelup_test.py:324)."""
        if masks is None:
            raise TypeError("match(): incompatible function arguments (masks must be a list; pass masks=[])")
        if len(sources) != 2:
            raise RuntimeError("sources.size() == modalities.size()")  # CV_Assert LL.cpp:1707
        sources = [self._as_source(s, i) for i, s in enumerate(sources)]
        self._whole_bank_only("match()")
        if self.frontend == "gpu" and self.shard[1] == 1:
            nat = self._select(list(class_ids))
            return self._to_matches(nat.match_images(sources[0], sources[1], list(masks), float(threshold)))
        quantized = self.quantize(sources, list(masks))
        return self.match_quantized(quantized, threshold, class_ids)

    def match_quantized(self, quantized, threshold, class_ids=()):
        """Same as match() but starting from quantized label images (the accelerated path proper)."""
        self._whole_bank_only("match_quantized()")
        nat = self._select(list(class_ids))
        out = nat.match_quantized(quantized, float(threshold))
        return self._to_matches(out)

    # ---- post-match stage (SURVEY.md 8f-3; the reference's drivers do this on the host) ----
    def setBoxes(self, sizes):
        """Box size (width, height) per template for the NMS: dict class_id -> array [n_templates, 2], as the
        drivers' template-info files give it (linemod_and_levelup_test.py:248-249, 337-338).  None = the
        templates' own width/height."""
        nat = self._ensure_native()
        if sizes is None:
            nat.set_boxes(None)
            return
        rows = []
        for cid in self._class_order:
            wh = np.asarray(sizes[cid], np.int32).reshape(-1, 2)
            if wh.shape[0] != self.bank.num_templates(cid):
                raise ValueError("class %s: %d box sizes for %d templates" % (cid, wh.shape[0], self.bank.num_templates(cid)))
            rows.append(wh)
        nat.set_boxes(np.concatenate(rows, 0))

    def match_top(self, quantized, threshold, class_ids=(), iou_threshold=0.5, top_k=3):
        """match + nms(dets, iou_threshold)[:top_k] of the reference's drivers (linemod_and_levelup_test.py:
        34-61, 325-350) in one call; the NMS runs on the GPU and only the survivors are copied back.
        Returns (list[Match] best first, number of raw matches before sort/unique)."""
        self._whole_bank_only("match_top()")
        nat = self._select(list(class_ids))
        out, nrec = nat.match_top(quantized, float(threshold), float(iou_threshold), int(top_k))
        return self._to_matches(out), nrec

    def _to_matches(self, out):
        # column-wise conversion + map(): building ~1400 objects field by field from numpy scalars costs 10x the
        # GPU match itself
        names = self._class_order
        return list(map(Match, out["x"].tolist(), out["y"].tolist(), out["similarity"].tolist(),
                        [names[c] for c in out["class_index"].tolist()], out["template_id"].tolist()))

    @staticmethod
    def _as_source(a, i):
        a = np.asarray(a)
        if i == 0:
            if a.dtype != np.uint8 or a.ndim != 3 or a.shape[2] != 3:
                raise TypeError("sources[0] must be a uint8 HxWx3 colour image")
        else:
            if a.dtype != np.uint16 or a.ndim != 2:
                raise TypeError("sources[1] must be a uint16 HxW depth image (mm)")
        return np.ascontiguousarray(a)
