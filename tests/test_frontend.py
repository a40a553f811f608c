"""The shared cv2 quantization front-end (6dpose_b200/frontend.py): tables against the reference's
(tests/golden/reference_tables.npz), filters against naive per-pixel restatements."""
import importlib
import os

import numpy as np
import pytest

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.fixture(scope="module")
def fe():
    return importlib.import_module("6dpose_b200.frontend")


def test_normal_lut_equals_reference_table(fe):
    assert np.array_equal(fe.normal_lut(), np.load(os.path.join(GOLD, "reference_tables.npz"))["normal_lut"])


def naive_hysteresis(mag, angle, thr):
    rows, cols = angle.shape
    q = np.clip(np.rint(angle * np.float32(16.0 / 360.0)), 0, 255).astype(np.uint8)
    q[0, :] = 0; q[-1, :] = 0; q[:, 0] = 0; q[:, -1] = 0
    q[1:-1, 1:-1] &= 7
    out = np.zeros_like(q)
    for r in range(1, rows - 1):
        for c in range(1, cols - 1):
            if mag[r, c] > thr:
                hist = [0] * 8
                for v in q[r - 1:r + 2, c - 1:c + 2].ravel():
                    hist[v] += 1
                best, idx = 0, -1
                for i in range(8):
                    if best < hist[i]:
                        idx, best = i, hist[i]
                if best >= 5:
                    out[r, c] = 1 << idx
    return out


def test_hysteresis_against_naive_loops(fe):
    rng = np.random.default_rng(0)
    angle = (rng.integers(0, 8, (24, 32)) * 45 + rng.uniform(-5, 5, (24, 32))).astype(np.float32) % 360
    angle = np.kron(angle[::4, ::4], np.ones((4, 4), np.float32))  # coherent patches so that votes pass
    mag = rng.uniform(0, 200, (24, 32)).astype(np.float32)
    assert np.array_equal(fe._hysteresis(mag, angle, np.float32(100.0)), naive_hysteresis(mag, angle, 100.0))


def naive_normals(depth, dist_thr=2000, diff_thr=50):
    H, W = depth.shape
    lut = importlib.import_module("6dpose_b200.frontend").normal_lut()
    out = np.zeros((H, W), np.uint8)
    r = 5
    for y in range(r, H - r - 1):
        for x in range(r, W - r - 1):
            d = int(depth[y, x])
            if d >= dist_thr:
                continue
            A = [0, 0, 0, 0]; b = [0, 0]
            for j in (-r, 0, r):
                for i in (-r, 0, r):
                    if i == 0 and j == 0:
                        continue
                    delta = int(depth[y + j, x + i]) - d
                    f = 1 if abs(delta) < diff_thr else 0
                    A[0] += f * i * i; A[1] += f * i * j; A[3] += f * j * j
                    b[0] += f * i * delta; b[1] += f * j * delta
            det = A[0] * A[3] - A[1] * A[1]
            ddx = A[3] * b[0] - A[1] * b[1]
            ddy = -A[1] * b[0] + A[0] * b[1]
            nx, ny, nz = np.float32(1150 * ddx), np.float32(1150 * ddy), np.float32(-det * d)
            s = np.sqrt(nx * nx + ny * ny + nz * nz, dtype=np.float32)
            if s > 0:
                inv = np.float32(1.0) / s
                v1 = int(nx * inv * np.float32(10) + np.float32(10))
                v2 = int(ny * inv * np.float32(10) + np.float32(10))
                v3 = min(int(nz * inv * np.float32(20) + np.float32(20)), 19)
                out[y, x] = lut[v3, v2, v1]
    import cv2
    return cv2.medianBlur(out, 5)


def test_depth_normals_against_naive_loops(fe):
    rng = np.random.default_rng(1)
    yy, xx = np.mgrid[0:40, 0:48]
    depth = (800 + 3 * xx + 2 * yy + rng.integers(0, 3, (40, 48))).astype(np.uint16)
    depth[10:20, 10:20] = 0      # sensor shadow
    depth[25:30, 30:40] = 2500   # beyond the distance threshold
    assert np.array_equal(fe.quantize_depth(depth), naive_normals(depth))


def test_pyramid_shapes_and_one_hot_labels(fe):
    rng = np.random.default_rng(2)
    rgb = rng.integers(0, 255, (96, 128, 3), dtype=np.uint8)
    depth = rng.integers(500, 1500, (96, 128)).astype(np.uint16)
    mask = np.zeros((96, 128), np.uint8)
    mask[20:80, 30:100] = 255
    q = fe.quantize_pyramid([rgb, depth], 2, [mask, mask])
    assert [a.shape for a in q[0]] == [(96, 128)] * 2 and [a.shape for a in q[1]] == [(48, 64)] * 2
    for lvl in q:
        for a in lvl:
            nz = a[a > 0]
            assert np.all((nz & (nz - 1)) == 0)          # one-hot
    assert q[0][0][:20].max() == 0 and q[0][1][:, :30].max() == 0   # outside the mask
    with pytest.raises(RuntimeError):
        fe.quantize_pyramid([rgb], 2)
    with pytest.raises(TypeError):
        fe.quantize_color(depth)
