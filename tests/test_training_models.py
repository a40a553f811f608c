"""numpy models of the template-extraction kernels (6dpose_b200/csrc/lm_train.cuh), checked against what they
replace: cv2.distanceTransform / cv2.erode as training.py calls them, and training.select_scattered_features.
CPU only; the kernels themselves are pinned to the host trainer in tests/test_gpu_training.py."""
import importlib

import cv2
import numpy as np
import pytest

INF = 0x3FFFFFFF  # TR_INF


def coldist_model(nfg):
    """k_tr_coldist: per pixel of label c, the distance along its column to the nearest pixel that is not c
    (beyond the image: INF); 0 for pixels without a label."""
    H, W = nfg.shape
    g = np.zeros((H, W), np.int64)
    for x in range(W):
        run, prev = 0, 0
        for y in range(H):
            c = nfg[y, x]
            run = 0 if not c else (INF if y == 0 else ((min(run + 1, INF) if run < INF else INF) if prev == c else 1))
            g[y, x] = run
            prev = c
        run, prev = 0, 0
        for y in range(H - 1, -1, -1):
            c = nfg[y, x]
            run = 0 if not c else (INF if y == H - 1 else ((min(run + 1, INF) if run < INF else INF) if prev == c else 1))
            if c:
                g[y, x] = min(g[y, x], run)
            prev = c
    return g


def rowdist_model(nfg, g):
    """k_tr_normcand's row pass: min over x' of max(|x - x'|, col(x')), scanned outwards with the kernel's early stop;
    float32, FLT_MAX where no pixel is not c."""
    H, W = nfg.shape
    out = np.zeros((H, W), np.float32)
    for y in range(H):
        for x in range(W):
            c = nfg[y, x]
            if not c:
                continue
            best = int(g[y, x])
            d = 1
            while d < best:
                lin, rin = x - d >= 0, x + d < W
                if not lin and not rin:
                    break
                if lin:
                    best = min(best, max(d, int(g[y, x - d])) if nfg[y, x - d] == c else d)
                if rin:
                    best = min(best, max(d, int(g[y, x + d])) if nfg[y, x + d] == c else d)
                d += 1
            out[y, x] = np.float32(3.4028235e38) if best >= INF else np.float32(best)
    return out


def _labels(rng, H, W, block, p_zero):
    lab = (1 << rng.integers(0, 8, ((H + block - 1) // block, (W + block - 1) // block))).astype(np.uint8)
    lab = np.kron(lab, np.ones((block, block), np.uint8))[:H, :W]
    lab[rng.random((H, W)) < p_zero] = 0
    return lab


@pytest.mark.parametrize("seed,H,W,block,p_zero", [(1, 24, 32, 4, 0.05), (2, 17, 23, 6, 0.0), (3, 30, 20, 10, 0.02),
                                                   (4, 16, 16, 3, 0.3)])
def test_separable_chessboard_distance_equals_cv2(seed, H, W, block, p_zero):
    """Regions touch the border (beyond the image counts as far away) and some labels cover a whole row / column."""
    rng = np.random.default_rng(seed)
    nfg = _labels(rng, H, W, block, p_zero)
    got = rowdist_model(nfg, coldist_model(nfg))
    for i in range(8):
        temp = (nfg == (1 << i)).astype(np.uint8) * (1 << i)
        want = cv2.distanceTransform(temp, cv2.DIST_C, 3)
        sel = nfg == (1 << i)
        assert np.array_equal(got[sel], want[sel]), (i, got[sel][:8], want[sel][:8])


@pytest.mark.parametrize("shape", [(12, 9), (1, 7), (5, 1)])
def test_no_zero_pixel_gives_flt_max(shape):
    nfg = np.full(shape, 4, np.uint8)
    got = rowdist_model(nfg, coldist_model(nfg))
    want = cv2.distanceTransform(nfg, cv2.DIST_C, 3)
    assert np.array_equal(got, want) and float(want.max()) == float(np.finfo(np.float32).max)


def border_model(mask):
    """k_tr_prep, colour: mask - erode(mask, 3x3) is nonzero iff mask > min of the clamped 3x3 neighbourhood."""
    H, W = mask.shape
    ys, xs = np.clip(np.arange(H)[:, None] + np.arange(-1, 2)[None], 0, H - 1), np.clip(np.arange(W)[:, None] + np.arange(-1, 2)[None], 0, W - 1)
    m3 = np.full(mask.shape, 255, np.int32)
    for dy in range(3):
        for dx in range(3):
            m3 = np.minimum(m3, mask[ys[:, dy]][:, xs[:, dx]])
    return mask > m3


def erode5_model(mask):
    """k_tr_prep, normals: erode(mask, 3x3, 2 iterations, BORDER_REPLICATE) = min over the clamped 5x5 neighbourhood."""
    H, W = mask.shape
    out = np.full(mask.shape, 255, np.uint8)
    for dy in range(-2, 3):
        for dx in range(-2, 3):
            ys = np.clip(np.arange(H) + dy, 0, H - 1)
            xs = np.clip(np.arange(W) + dx, 0, W - 1)
            out = np.minimum(out, mask[ys][:, xs])
    return out


@pytest.mark.parametrize("seed", [0, 1, 2, 3])
def test_mask_models_equal_cv2_on_non_binary_masks(seed):
    rng = np.random.default_rng(seed)
    H, W = 40 + seed, 52 - seed
    mask = np.kron(rng.choice(np.array([0, 1, 7, 128, 255], np.uint8), (H // 4 + 1, W // 4 + 1)), np.ones((4, 4), np.uint8))[:H, :W]
    mask[rng.random((H, W)) < 0.05] = rng.integers(0, 256, 1, dtype=np.uint8)[0]
    eroded = cv2.erode(mask, None, iterations=1, borderType=cv2.BORDER_REPLICATE)
    assert np.array_equal(border_model(mask), cv2.subtract(mask, eroded) != 0)
    assert np.array_equal(erode5_model(mask), cv2.erode(mask, None, iterations=2, borderType=cv2.BORDER_REPLICATE))


def select_warp_model(cands, num_features, distance):
    """k_tr_select: 32 candidates tested at once against the kept set; the first that passes is kept and only the
    lanes after it are re-tested against it; a pass that keeps nothing skips to the first distance at which the
    farthest candidate passes.  Returns (features, number of windows processed)."""
    f32 = np.float32
    need = lambda d: int(np.ceil(f32(d * d)))
    n = len(cands)
    dist = f32(distance)
    kept, feats = [], []
    i, windows, kept_any, far = 0, 0, False, -1
    while len(kept) < num_features:
        win = cands[i:i + min(32, n - i)]
        windows += 1
        md = [min([(c[0] - kx) ** 2 + (c[1] - ky) ** 2 for kx, ky in kept], default=2 ** 31 - 1) for c in win]
        live = [m >= need(dist) for m in md]
        j = 0
        while j < len(win) and len(kept) < num_features:
            if not live[j]:
                j += 1
                continue
            c = win[j]
            kept.append((c[0], c[1]))
            feats.append((c[0], c[1], c[2]))
            kept_any = True
            for t in range(j + 1, len(win)):
                md[t] = min(md[t], (win[t][0] - c[0]) ** 2 + (win[t][1] - c[1]) ** 2)
                live[t] = live[t] and md[t] >= need(dist)
            md[j] = 0
            j += 1
        far = max([far] + md)
        i += len(win)
        if i == n:
            i = 0
            dist = f32(dist - f32(1.0))
            if not kept_any:
                while need(dist) > far:
                    dist = f32(dist - f32(1.0))
            kept_any, far = False, -1
    return feats, windows


@pytest.mark.parametrize("seed,n,nf,colour", [(0, 300, 63, True), (1, 1000, 31, False), (2, 64, 63, True), (3, 200, 150, False),
                                              (4, 3000, 63, True)])
def test_warp_selection_equals_select_scattered_features(seed, n, nf, colour):
    training = importlib.import_module("6dpose_b200.training")
    rng = np.random.default_rng(seed)
    H, W = 60, 80
    idx = np.sort(rng.choice(H * W, n, replace=False))
    ys, xs = idx // W, idx % W
    if colour:
        scores = rng.integers(3026, 20000, n).astype(np.float64)
        distance = float(n // nf + 1)
    else:
        scores = (rng.integers(1, 6, n).astype(np.float32) / np.float32(7)).astype(np.float64)
        distance = np.float32(np.sqrt(np.float32(H * W))) / np.float32(np.sqrt(np.float32(nf))) + np.float32(1.5)
    cands = training._stable_by_score(list(zip(xs.tolist(), ys.tolist(), rng.integers(0, 8, n).tolist(), scores.tolist())))
    want, enough = training.select_scattered_features(cands, nf, distance)
    got, windows = select_warp_model(cands, nf, distance)
    assert enough and got == want
    assert windows < (n + 31) // 32 * 64   # several passes, but not one per distance step
