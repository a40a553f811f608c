"""Synthetic template banks and quantized frames (SURVEY.md section 8d).

No datasets or renderer exist offline, so the benchmark workloads are generated:
  * banks shaped like the reference's rendered banks: `views` base shapes x `variants` in-plane/scale
    variants each (3115 = 89 x 35), `num_features` per modality at level 0 and half of that per level
    above (LL.cpp:560, 860), colour features on the outline, depth-normal features in the interior,
    crop invariants of cropTemplates (LL.cpp:234-277) enforced;
  * frames generated directly as quantized one-hot label images with the fixture frame's statistics
    (P(nonzero) = 0.485 colour / 0.91 normals), spatially coherent, with K templates planted so that
    known (template_id, x, y, 100 %) answers exist.
"""
import numpy as np

from .bank import Template, TemplateBank


def _outline_points(rng, w, h, n):
    t = rng.uniform(0, 2 * np.pi, n)
    rx, ry = w / 2.0, h / 2.0
    x = np.clip(np.rint(rx + rx * np.cos(t) * rng.uniform(0.9, 1.0, n)), 0, w)
    y = np.clip(np.rint(ry + ry * np.sin(t) * rng.uniform(0.9, 1.0, n)), 0, h)
    return x.astype(np.int32), y.astype(np.int32)


def _interior_points(rng, w, h, n):
    t = rng.uniform(0, 2 * np.pi, n)
    r = np.sqrt(rng.uniform(0, 0.8, n))
    x = np.clip(np.rint(w / 2.0 + w / 2.0 * r * np.cos(t)), 0, w)
    y = np.clip(np.rint(h / 2.0 + h / 2.0 * r * np.sin(t)), 0, h)
    return x.astype(np.int32), y.astype(np.int32)


def _pin_extents(x, y, w, h):
    """cropTemplates leaves min x = min y = 0 and max x = width, max y = height at level 0."""
    x[0], y[1] = 0, 0
    x[2], y[3] = w, h
    return x, y


def synth_bank(n_templates, num_features=150, levels=2, seed=1234, class_ids=("01_template",), variants=35,
               size_range=((20, 126), (24, 142))):
    """TemplateBank with n_templates per class.  Template k = base shape k // variants, jittered."""
    rng = np.random.default_rng(seed)
    bank = TemplateBank()
    for cid in class_ids:
        tps = []
        base = None
        for k in range(n_templates):
            if k % variants == 0 or base is None:
                w = int(rng.integers(size_range[0][0] // 2, size_range[0][1] // 2 + 1)) * 2
                h = int(rng.integers(size_range[1][0] // 2, size_range[1][1] // 2 + 1)) * 2
                base = dict(w=w, h=h, lv=[])
                for l in range(levels):
                    nf = max(num_features >> l, 4)
                    wl, hl = w >> l, h >> l
                    cx, cy = _outline_points(rng, wl, hl, nf)
                    dx, dy = _interior_points(rng, wl, hl, nf)
                    # orientation follows the outline tangent; normals vary smoothly over the interior
                    cl = (np.floor((np.arctan2(cy - hl / 2.0, cx - wl / 2.0) + np.pi) / np.pi * 8) % 8).astype(np.int32)
                    dl = ((dx * 3 // max(wl, 1)) + 3 * (dy * 3 // max(hl, 1))).astype(np.int32) % 8
                    base["lv"].append((cx, cy, cl, dx, dy, dl))
            tp = []
            w, h = base["w"], base["h"]
            for l in range(levels):
                wl, hl = w >> l, h >> l
                cx, cy, cl, dx, dy, dl = [a.copy() for a in base["lv"][l]]
                if k % variants:
                    # in-plane/scale variant: jitter a third of the features by one pixel, relabel a few
                    for xs, ys, ls in ((cx, cy, cl), (dx, dy, dl)):
                        n = xs.shape[0]
                        pick = rng.random(n) < 0.33
                        xs[pick] = np.clip(xs[pick] + rng.integers(-1, 2, pick.sum()), 0, wl)
                        ys[pick] = np.clip(ys[pick] + rng.integers(-1, 2, pick.sum()), 0, hl)
                        rel = rng.random(n) < 0.1
                        ls[rel] = (ls[rel] + rng.integers(1, 8, rel.sum())) % 8
                if l == 0:
                    cx, cy = _pin_extents(cx, cy, wl, hl)
                tp.append(Template(wl, hl, l, np.stack([cx, cy, cl], 1)))
                tp.append(Template(wl, hl, l, np.stack([dx, dy, dl], 1)))
            tps.append(tp)
        bank.classes[cid] = tps
    return bank


def _block_field(rng, H, W, block, hi):
    bh, bw = (H + block - 1) // block + 1, (W + block - 1) // block + 1
    lab = rng.integers(0, hi, (bh, bw))
    oy, ox = rng.integers(0, block, 2)
    return np.kron(lab, np.ones((block, block), np.int64))[oy:oy + H, ox:ox + W]


def _coherent_labels(rng, H, W, p_nonzero, label_block, salt, mask_block):
    """One-hot label image: piecewise-constant labels (label_block px regions) with `salt` random
    relabels, switched on in mask_block px cells with probability p_nonzero.  The parameters used
    by synth_frame reproduce the spread-mask bit-count histogram of the reference's fixture frame
    (test/case1/0000_*) to within a few percent per bin, so candidate rates are realistic."""
    img = _block_field(rng, H, W, label_block, 8)
    s = rng.random((H, W)) < salt
    img = np.where(s, rng.integers(0, 8, (H, W)), img)
    on = _block_field(rng, H, W, mask_block, 1000) < int(p_nonzero * 1000)
    return np.where(on, 1 << img, 0).astype(np.uint8)


def synth_frame(W=640, H=480, levels=2, seed=42, bank=None, plant=8, T=(4, 8)):
    """Quantized pyramid [[colour, normals] per level] + list of planted (class_id, template_id, x, y).

    Level l+1 is the nearest-neighbour decimation of level l (what DepthNormalPyramid::pyrDown does,
    LL.cpp:865-868).  Planted templates are written at every level so both the coarse scan and the
    refinement see a 100 % match."""
    rng = np.random.default_rng(seed)
    q = [[_coherent_labels(rng, H, W, 0.485, 16, 0.04, 2), _coherent_labels(rng, H, W, 0.91, 48, 0.02, 16)]]
    for l in range(1, levels):
        q.append([np.ascontiguousarray(a[::2, ::2]) for a in q[-1]])
    planted = []
    if bank is not None and plant > 0:
        cids = bank.class_ids()
        border = 8 * T[0]
        for k in range(plant):
            cid = cids[k % len(cids)]
            tps = bank.classes[cid]
            tid = int(rng.integers(0, len(tps)))
            tp = tps[tid]
            w, h = tp[0].width, tp[0].height
            step = 2 ** (levels - 1) * T[-1]  # keep the plant on the coarse sampling grid
            xmax, ymax = W - w - border - step, H - h - border - step
            if xmax <= border or ymax <= border:
                continue
            x = int(rng.integers(border, xmax) // step * step)
            y = int(rng.integers(border, ymax) // step * step)
            for l in range(levels):
                for m in range(2):
                    t = tp[l * 2 + m]
                    fx = (x >> l) + t.features[:, 0]
                    fy = (y >> l) + t.features[:, 1]
                    q[l][m][fy, fx] = (1 << t.features[:, 2]).astype(np.uint8)
            planted.append((cid, tid, x, y))
    return q, planted


def synth_rgbd(W=640, H=480, seed=7):
    """Structured raw RGB-D frame (u8 HxWx3, u16 HxW mm): smooth colour blobs with edges and noise; depth
    planes, bumps, sensor holes and a far background -- exercises every branch of the quantization
    front-end (used by the front-end tests and the front-end timing in bench.py)."""
    import cv2
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:H, 0:W].astype(np.float32)
    rgb = np.zeros((H, W, 3), np.float32)
    depth = np.full((H, W), 1200.0, np.float32) + 0.2 * xx + 0.1 * yy
    for _ in range(12):
        cx, cy, r = rng.uniform(0, W), rng.uniform(0, H), rng.uniform(15, 80)
        m = ((xx - cx) ** 2 + (yy - cy) ** 2) < r * r
        rgb[m] = rng.uniform(0, 255, 3)
        depth[m] = rng.uniform(500, 1900) + 40 * np.sqrt(np.clip(1 - ((xx[m] - cx) ** 2 + (yy[m] - cy) ** 2) / (r * r), 0, 1))
    rgb += rng.normal(0, 6, rgb.shape)
    rgb = cv2.GaussianBlur(np.clip(rgb, 0, 255).astype(np.uint8), (3, 3), 0)
    depth += rng.normal(0, 1.5, depth.shape)
    depth[rng.random((H, W)) < 0.03] = 0   # sensor holes
    depth[:, : W // 10] = 2600              # beyond the distance threshold
    return rgb, np.clip(depth, 0, 65535).astype(np.uint16)


def warp_views(rgb, depth, mask, n, seed=0, max_angle=30.0, scale=(0.8, 1.2), max_shift=40):
    """n training views from one (rgb, depth, mask) view under seeded in-plane rotation, scale and shift about the
    mask's centre: rgb interpolated linearly, depth and mask nearest (no renderer is needed to grow a bank for
    extraction tests and timings).  Returns a list of (rgb, depth, mask)."""
    import cv2
    rng = np.random.default_rng(seed)
    H, W = depth.shape
    ys, xs = np.nonzero(mask)
    cx, cy = (float(xs.mean()), float(ys.mean())) if xs.size else (W / 2.0, H / 2.0)
    out = []
    for _ in range(n):
        M = cv2.getRotationMatrix2D((cx, cy), float(rng.uniform(-max_angle, max_angle)), float(rng.uniform(*scale)))
        M[:, 2] += rng.uniform(-max_shift, max_shift, 2)
        out.append((cv2.warpAffine(rgb, M, (W, H), flags=cv2.INTER_LINEAR),
                    cv2.warpAffine(depth, M, (W, H), flags=cv2.INTER_NEAREST),
                    cv2.warpAffine(mask, M, (W, H), flags=cv2.INTER_NEAREST)))
    return out
