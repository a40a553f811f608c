"""Template extraction (host, cv2 + numpy): Detector::addTemplate and what it calls.

Training is not on the accelerated path (SURVEY.md section 8 row f2); it exists so that the
reference's `mode = 'train' / 'render_train'` drivers (linemod_and_levelup_test.py:94-300) run against
this backend and produce banks the GPU matcher consumes.  Restates (reference:
linemodLevelup/linemodLevelup.cpp, "LL.cpp"):

  select_scattered_features   <- QuantizedPyramid::selectScatteredFeatures   LL.cpp:279-318
  extract_color_template      <- ColorGradientPyramid::extractTemplate      LL.cpp:589-643
  extract_normal_template     <- DepthNormalPyramid::extractTemplate        LL.cpp:888-966
  crop_templates              <- cropTemplates                              LL.cpp:234-277
  add_template                <- Detector::addTemplate                      LL.cpp:1943-1975

add_templates is the batched GPU path (lm_extract_templates, csrc/lm_train.cuh): the same templates, feature for
feature, for many views in one call.
"""
import math

import cv2
import numpy as np

from . import frontend
from .bank import Template

_LABEL_OF = {1 << i: i for i in range(8)}


def select_scattered_features(cands, num_features, distance):
    """cands: list of (x, y, label, score) already sorted; returns (features list, enough?)."""
    feats = []
    distance = np.float32(distance)
    distance_sq = np.float32(distance * distance)
    n = len(cands)
    i = 0
    xs = np.zeros(num_features, np.int64)
    ys = np.zeros(num_features, np.int64)
    k = 0
    while k < num_features:
        cx, cy = cands[i][0], cands[i][1]
        if k == 0:
            keep = True
        else:
            d = (cx - xs[:k]) ** 2 + (cy - ys[:k]) ** 2
            keep = bool(np.all(d >= distance_sq))
        if keep:
            feats.append((cx, cy, cands[i][2]))
            xs[k], ys[k] = cx, cy
            k += 1
        i += 1
        if i == n:
            i = 0
            distance = np.float32(distance - np.float32(1.0))
            distance_sq = np.float32(distance * distance)
    return feats, len(feats) == num_features


def _stable_by_score(cands):
    # Candidate::operator< sorts high scores first; std::stable_sort keeps ties in scan order
    return sorted(cands, key=lambda c: -c[3])


def extract_color_template(pyr):
    """ColorGradientPyramid::extractTemplate (LL.cpp:589-643).  Returns Template or None."""
    mask = pyr.mask
    local_mask = None
    if mask is not None:
        eroded = cv2.erode(mask, None, iterations=1, borderType=cv2.BORDER_REPLICATE)
        local_mask = cv2.subtract(mask, eroded)
    thr_sq = np.float32(pyr.strong_threshold) * np.float32(pyr.strong_threshold)
    ok = (pyr.angle > 0) & (pyr.magnitude > thr_sq)
    if local_mask is not None:
        ok &= local_mask != 0
    rs, cs = np.nonzero(ok)  # row-major scan order
    if rs.size < pyr.num_features:
        return None
    labels = np.log2(pyr.angle[rs, cs]).astype(np.int64)
    scores = pyr.magnitude[rs, cs]
    cands = _stable_by_score(list(zip(cs.tolist(), rs.tolist(), labels.tolist(), scores.tolist())))
    distance = float(len(cands) // pyr.num_features + 1)
    feats, enough = select_scattered_features(cands, pyr.num_features, distance)
    if not enough:
        return None
    return Template(-1, -1, pyr.pyramid_level, np.asarray(feats, np.int32).reshape(-1, 3))


def extract_normal_template(pyr):
    """DepthNormalPyramid::extractTemplate (LL.cpp:888-966)."""
    normal = pyr.normal
    mask = pyr.mask
    local_mask = None
    if mask is not None:
        local_mask = cv2.erode(mask, None, iterations=2, borderType=cv2.BORDER_REPLICATE)
    distances = []
    temp = np.zeros(normal.shape, np.uint8)
    for i in range(8):
        if local_mask is None:
            temp[:] = 1 << i
        else:
            temp[local_mask != 0] = 1 << i
        temp = cv2.bitwise_and(temp, normal)
        distances.append(cv2.distanceTransform(temp, cv2.DIST_C, 3))
    ok = (normal != 0) & (normal != 255)
    if local_mask is not None:
        ok &= local_mask != 0
    rs, cs = np.nonzero(ok)
    cands = []
    label_counts = [0] * 8
    for r, c in zip(rs.tolist(), cs.tolist()):
        q = int(normal[r, c])
        if q not in _LABEL_OF:
            raise RuntimeError("Invalid value of quantized parameter")  # getLabel, LL.cpp:176-192
        label = _LABEL_OF[q]
        score = float(distances[label][r, c])
        if score >= pyr.extract_threshold:
            cands.append([c, r, label, score])
            label_counts[label] += 1
    if len(cands) < pyr.num_features:
        return None
    for cd in cands:
        cd[3] = float(np.float32(cd[3]) / np.float32(label_counts[cd[2]]))
    cands = _stable_by_score([tuple(c) for c in cands])
    area = float(normal.size) if local_mask is None else float(cv2.countNonZero(local_mask))
    distance = np.float32(math.sqrt(np.float32(area))) / np.float32(math.sqrt(np.float32(pyr.num_features))) + np.float32(1.5)
    feats, _ = select_scattered_features(cands, pyr.num_features, distance)  # return value ignored in the reference
    return Template(-1, -1, pyr.pyramid_level, np.asarray(feats, np.int32).reshape(-1, 3))


def crop_templates(templates):
    """cropTemplates (LL.cpp:234-277): common box over all levels/modalities, even origin."""
    min_x = min_y = 2 ** 31 - 1
    max_x = max_y = -2 ** 31
    for t in templates:
        if t.features.shape[0] == 0:
            continue
        x = t.features[:, 0].astype(np.int64) << t.pyramid_level
        y = t.features[:, 1].astype(np.int64) << t.pyramid_level
        min_x, max_x = min(min_x, int(x.min())), max(max_x, int(x.max()))
        min_y, max_y = min(min_y, int(y.min())), max(max_y, int(y.max()))
    if min_x % 2 == 1:
        min_x -= 1
    if min_y % 2 == 1:
        min_y -= 1
    for t in templates:
        t.width = (max_x - min_x) >> t.pyramid_level
        t.height = (max_y - min_y) >> t.pyramid_level
        t.features = t.features.copy()
        t.features[:, 0] -= min_x >> t.pyramid_level
        t.features[:, 1] -= min_y >> t.pyramid_level
    return min_x, min_y, max_x - min_x, max_y - min_y


def _check_mask(object_mask):
    if object_mask is None or not np.asarray(object_mask).size:
        return None
    mask = np.ascontiguousarray(object_mask)
    if mask.ndim == 3:
        raise TypeError("object_mask must be single channel")
    if mask.dtype != np.uint8:
        raise TypeError("object_mask must be uint8 (255 = object)")
    return mask


def class_templates(detector, class_id):
    """class_templates[class_id] (LL.cpp:1947): created even when every extraction fails.  A class loaded from a
    packed bank file is unpacked to a list before it grows."""
    pyramids = detector.bank.classes.setdefault(class_id, [])
    if not isinstance(pyramids, list):
        pyramids = detector.bank.classes[class_id] = list(pyramids)
    return pyramids


def append_template(pyramids, tp, cropped=False):
    """The end of Detector::addTemplate (LL.cpp:1962-1974): cropTemplates, then the pyramid gets the next id."""
    if not cropped:
        crop_templates(tp)
    pyramids.append(tp)
    return len(pyramids) - 1


def add_template(detector, sources, class_id, object_mask):
    """Detector::addTemplate (LL.cpp:1943-1975): template id, or -1 when extraction fails."""
    if len(sources) != 2:
        raise RuntimeError("sources.size() == modalities.size()")
    src = [detector._as_source(s, i) for i, s in enumerate(sources)]
    mask = _check_mask(object_mask)
    pyramids = class_templates(detector, class_id)
    L = detector.pyramid_levels
    nf = detector.num_features
    tp = [None] * (2 * L)
    for m in range(2):
        if m == 0:
            pyr = frontend.ColorPyramid(src[0], mask, 10.0, nf, 55.0)
        else:
            pyr = frontend.NormalPyramid(src[1], mask, 2000, 50, nf, 2)
        for l in range(L):
            if l > 0:
                pyr.pyrDown()
            t = extract_color_template(pyr) if m == 0 else extract_normal_template(pyr)
            if t is None:
                return -1
            tp[l * 2 + m] = t
    return append_template(pyramids, tp)


def add_templates(detector, native, sources_list, class_id, object_masks):
    """add_template over many views of one size, extracted on the GPU in one call (lm_extract_templates; cropTemplates
    runs inside the library).  Same ids and bank as calling add_template per view in order.  Every input is checked
    before the bank changes: a bad view raises and adds nothing."""
    if len(object_masks) != len(sources_list):
        raise RuntimeError("%d object masks for %d views" % (len(object_masks), len(sources_list)))
    rgbs, deps, masks = [], [], []
    for sources, object_mask in zip(sources_list, object_masks):
        if len(sources) != 2:
            raise RuntimeError("sources.size() == modalities.size()")
        rgb, dep = detector._as_source(sources[0], 0), detector._as_source(sources[1], 1)
        mask = _check_mask(object_mask)
        shape = rgbs[0].shape[:2] if rgbs else rgb.shape[:2]
        if rgb.shape[:2] != shape or dep.shape != shape:
            raise RuntimeError("all views of one addTemplates call must have one size: %r, then rgb %r / depth %r"
                               % (shape, rgb.shape[:2], dep.shape))
        if mask is not None and mask.shape != shape:
            raise RuntimeError("mask.size() == source.size(): mask %r for images %r" % (mask.shape, shape))
        rgbs.append(rgb)
        deps.append(dep)
        masks.append(mask)
    if not rgbs:
        return []
    ok, tmeta, feats = native.extract_templates(detector.num_features, rgbs, deps, masks)
    pyramids = class_templates(detector, class_id)
    ids = []
    for v in range(len(rgbs)):
        if not ok[v]:
            ids.append(-1)
            continue
        tp = [Template(w, h, s_ // 2, feats[v, b:b + n].copy()) for s_, (w, h, b, n) in enumerate(tmeta[v].tolist())]
        ids.append(append_template(pyramids, tp, cropped=True))
    return ids
