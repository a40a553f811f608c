"""CPU tests of the oracle (oracle/lm_oracle.cpp): against an independent numpy restatement of the
same reference functions on small cases, against the reference's own tables (tests/golden/reference_tables.npz),
and against the committed golden fixtures."""
import os

import numpy as np
import pytest

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


# ---- a second, deliberately naive restatement (numpy + Python loops), small cases only ----------
def np_spread(q, T):
    H, W = q.shape
    out = np.zeros_like(q)
    for dy in range(T):
        for dx in range(T):
            out[:H - dy, :W - dx] |= q[dy:, dx:]
    return out


def np_response(sp):
    out = np.zeros((8,) + sp.shape, np.uint8)
    for o in range(8):
        hit = (sp >> o) & 1
        nb = ((sp >> ((o + 1) % 8)) | (sp >> ((o + 7) % 8))) & 1
        out[o] = np.where(hit == 1, 4, nb)
    return out


def np_linear_memories(q, T):
    r = np_response(np_spread(q, T))
    H, W = q.shape
    lm = np.zeros((8, T * T, (H // T) * (W // T)), np.uint8)
    for o in range(8):
        for gy in range(T):
            for gx in range(T):
                lm[o, gy * T + gx] = r[o][gy::T, gx::T].ravel()
    return lm


def np_match(quantized, T, bank, class_ids, threshold):
    """Detector::match after quantization, LL.cpp:1721-1776, written with flat numpy arrays."""
    L = len(T)
    lms = [[np_linear_memories(quantized[l][m], T[l]) for m in range(2)] for l in range(L)]
    flat = [[[lms[l][m][o].ravel() for o in range(8)] for m in range(2)] for l in range(L)]
    out = []
    for ci, cid in enumerate(class_ids):
        for tid, tp in enumerate(bank.classes[cid]):
            l = L - 1
            Tl = T[l]
            rows, cols = quantized[l][0].shape
            Wd, Hd = cols // Tl, rows // Tl
            total = np.zeros(Wd * Hd, np.int64)
            nf = 0
            for m in range(2):
                t = tp[l * 2 + m]
                nf += len(t.features)
                P = (Hd - ((t.height - 1) // Tl + 1)) * Wd + (Wd - ((t.width - 1) // Tl + 1)) + 1
                for x, y, lab in t.features.tolist():
                    if x >= cols or y >= rows or P <= 0:
                        continue
                    base = ((y % Tl) * Tl + x % Tl) * (Wd * Hd) + (y // Tl) * Wd + x // Tl
                    total[:P] += flat[l][m][lab][base:base + P]
            cands = []
            off = Tl // 2 + (Tl % 2 - 1)
            for j in range(Wd * Hd):
                score = np.float32(np.float32(total[j]) * np.float32(100.0)) / np.float32(4 * nf)
                if score > np.float32(threshold):
                    cands.append([(j % Wd) * Tl + off, (j // Wd) * Tl + off, score])
            for l in range(L - 2, -1, -1):
                Tl = T[l]
                rows, cols = quantized[l][0].shape
                Wd = cols // Tl
                plane = Wd * (rows // Tl)
                border = 8 * Tl
                off = Tl // 2 + (Tl % 2 - 1)
                max_x = cols - tp[l * 2].width - border
                max_y = rows - tp[l * 2].height - border
                keep = []
                for c in cands:
                    x = min(max(c[0] * 2 + 1, border), max_x)
                    y = min(max(c[1] * 2 + 1, border), max_y)
                    cx, cy = int(x / Tl) - 8, int(y / Tl) - 8  # truncation toward zero
                    patch = np.zeros((16, 16), np.int64)
                    nf2 = 0
                    for m in range(2):
                        t = tp[l * 2 + m]
                        nf2 += len(t.features)
                        for fx, fy, lab in t.features.tolist():
                            fx += cx * Tl
                            fy += cy * Tl
                            if fx < 0 or fy < 0 or fx >= cols or fy >= rows:
                                continue
                            base = ((fy % Tl) * Tl + fx % Tl) * plane + (fy // Tl) * Wd + fx // Tl
                            for r in range(16):
                                patch[r] += flat[l][m][lab][base + r * Wd: base + r * Wd + 16]
                    best, br, bc = np.float32(0), -1, -1
                    for r in range(16):
                        for cc in range(16):
                            s = np.float32(np.float32(patch[r, cc]) * np.float32(100.0)) / np.float32(4 * nf2)
                            if s > best:
                                best, br, bc = s, r, cc
                    c[0] = (int(x / Tl) - 8 + bc) * Tl + off
                    c[1] = (int(y / Tl) - 8 + br) * Tl + off
                    c[2] = best
                    if not (best < np.float32(threshold)):
                        keep.append(c)
                cands = keep
            out += [(c[0], c[1], np.float32(c[2]), ci, tid) for c in cands]
    return out


def test_similarity_lut_rule_matches_reference_table(oracle):
    lut = oracle.similarity_lut()
    assert set(np.unique(lut)) == {0, 1, 4}
    assert lut.tolist() == np.load(os.path.join(GOLD, "reference_tables.npz"))["similarity_lut"].tolist()


@pytest.mark.parametrize("T,H,W", [(4, 32, 48), (5, 40, 80), (8, 64, 64), (2, 16, 32)])
def test_linear_memories_against_numpy(oracle, T, H, W):
    rng = np.random.default_rng(T)
    q = np.where(rng.random((H, W)) < 0.5, 1 << rng.integers(0, 8, (H, W)), 0).astype(np.uint8)
    assert np.array_equal(oracle.spread(q, T), np_spread(q, T))
    assert np.array_equal(oracle.response_maps(np_spread(q, T)), np_response(np_spread(q, T)))
    assert np.array_equal(oracle.linear_memories(q, T), np_linear_memories(q, T))


def test_linear_memories_size_assertions(oracle):
    q = np.zeros((30, 40), np.uint8)
    with pytest.raises(RuntimeError):
        oracle.linear_memories(q, 4)  # rows % T


@pytest.mark.parametrize("T,W,H,nf,thr", [([4, 8], 256, 192, 24, 55.0), ([5, 8], 240, 160, 20, 50.0),
                                          ([8], 128, 128, 12, 50.0), ([2, 4], 160, 128, 16, 60.0)])
def test_match_against_numpy(oracle, synth, T, W, H, nf, thr):
    bank = synth.synth_bank(4, num_features=nf, levels=len(T), seed=13, variants=2,
                            size_range=((16, 40), (16, 40)))
    q, planted = synth.synth_frame(W, H, levels=len(T), seed=17, bank=bank, plant=2, T=T)
    cids = bank.class_ids()
    got = oracle.match(q, T, bank.pack(cids, 2 * len(T)), thr)
    raw = np_match(q, T, bank, cids, thr)
    # the numpy restatement stops before std::sort/std::unique: compare as sets after the same dedupe rule
    assert len(raw) >= len(got) > 0
    want = {(x, y, float(s), c) for x, y, s, c, t in raw}
    have = {(int(r["x"]), int(r["y"]), float(r["similarity"]), int(r["class_idx"])) for r in got}
    assert have == want
    # sorted by similarity descending, template_id ascending among equal similarities (LL.h:236-242)
    sims = got["similarity"]
    assert np.all(sims[:-1] >= sims[1:])
    eq = sims[:-1] == sims[1:]
    assert np.all(got["template_id"][:-1][eq] <= got["template_id"][1:][eq])
    # every record the oracle returns exists, with its template id, in the naive restatement
    full = {(x, y, float(s), c, t) for x, y, s, c, t in raw}
    for r in got:
        assert (int(r["x"]), int(r["y"]), float(r["similarity"]), int(r["class_idx"]), int(r["template_id"])) in full


def test_threads_do_not_change_the_result(oracle, synth):
    T = [4, 8]
    bank = synth.synth_bank(40, num_features=64, seed=3)
    q, _ = synth.synth_frame(320, 256, seed=4, bank=bank, plant=3, T=T)
    packed = bank.pack(bank.class_ids(), 4)
    a = oracle.match(q, T, packed, 70.0, n_threads=1)
    b = oracle.match(q, T, packed, 70.0, n_threads=4)
    assert len(a) > 0 and np.array_equal(a, b)


def test_planted_templates_are_found(oracle, synth):
    T = [4, 8]
    bank = synth.synth_bank(70, num_features=150, seed=7)
    q, planted = synth.synth_frame(640, 480, seed=11, bank=bank, plant=4, T=T)
    got = oracle.match(q, T, bank.pack(bank.class_ids(), 4), 90.0)
    found = {(int(r["template_id"]), int(r["x"]), int(r["y"])) for r in got}
    for cid, tid, x, y in planted:
        # refined location = plant + sampling offset (T/2 + T%2 - 1 = 1 at T=4)
        assert (tid, x + 1, y + 1) in found, (tid, x, y)
