"""GPU parity tests proper: the CUDA path (through the C-ABI) against the CPU oracle, bit-exact.

Bar (BASELINE.json north_star): template ids, (x, y) and integer similarity scores bit-exact; the
float similarity is the same two IEEE operations, compared with ==."""
import importlib

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _native(T, bank):
    lib = importlib.import_module("6dpose_b200._lib")
    nat = lib.NativeDetector(T)
    packed = bank.pack(bank.class_ids(), len(T) * 2)
    nat.load_bank(packed, len(T) * 2)
    return nat, packed


def _assert_same(got, want):
    assert len(got) == len(want), (len(got), len(want))
    for k in ("x", "y", "template_id"):
        assert np.array_equal(got[k], want[k]), k
    assert np.array_equal(got["class_index"], want["class_idx"])
    assert np.array_equal(got["similarity"], want["similarity"])  # exact float equality


@pytest.mark.parametrize("T,W,H,nf", [([4, 8], 640, 480, 150), ([5, 8], 640, 480, 127), ([4, 8], 320, 256, 63),
                                     ([8], 320, 240, 40), ([2, 4, 8], 640, 512, 96)])
def test_linear_memories_bit_exact(synth, oracle, T, W, H, nf):
    bank = synth.synth_bank(8, num_features=nf, levels=len(T), seed=3)
    q, _ = synth.synth_frame(W, H, levels=len(T), seed=5, bank=bank, plant=2, T=T)
    nat, _ = _native(T, bank)
    nat.upload_quantized(q)
    nat.run(80.0)
    for l, t in enumerate(T):
        for m in range(2):
            want = oracle.linear_memories(q[l][m], t)
            got = nat.linear_memories(l, m, want.shape)
            assert np.array_equal(got, want), (l, m)


@pytest.mark.parametrize("T,W,H,nf,n,thr", [
    ([4, 8], 640, 480, 150, 140, 75.0),
    ([4, 8], 640, 480, 150, 140, 90.0),
    ([5, 8], 640, 480, 127, 70, 75.0),   # T not a power of two, 16-bit at L0 / 8-bit at L1 in the reference
    ([5, 8], 640, 480, 63, 70, 70.0),    # the reference's 8-bit (_64) path at both levels
    ([4, 8], 320, 256, 40, 35, 60.0),
    ([8], 320, 240, 40, 35, 60.0),       # single level: no refinement
    ([2, 4, 8], 640, 512, 96, 35, 70.0), # three levels
    ([4, 8], 640, 480, 300, 35, 75.0),   # 300 features at the lowest level: byte-wise coarse kernel
    ([4, 8], 800, 480, 150, 35, 75.0),   # 47 position words, bit-planes still fit shared memory
    ([4, 8], 960, 640, 150, 35, 75.0),   # 75 position words (3 rounds), bit-planes read from global memory
    ([4, 8], 1280, 960, 150, 20, 80.0),  # BASELINE config 5 frame size: 150 words (5 rounds)
])
def test_match_bit_exact_synthetic(synth, oracle, T, W, H, nf, n, thr):
    bank = synth.synth_bank(n, num_features=nf, levels=len(T), seed=21, class_ids=("01_template", "02_template"))
    q, planted = synth.synth_frame(W, H, levels=len(T), seed=9, bank=bank, plant=6, T=T)
    nat, packed = _native(T, bank)
    got = nat.match_quantized(q, thr)
    want = oracle.match(q, T, packed, thr)
    assert len(want) > 0
    _assert_same(got, want)
    c = nat.counters()
    _, st = oracle.match(q, T, packed, thr, want_stats=True)
    assert c["coarse_candidates"] == int(st["coarse_candidates"])
    assert c["scan_bytes"] == int(st["coarse_byte_adds"])
    assert c["refine_bytes"] == int(st["refine_byte_adds"])


def test_bench_workload_3115_templates_bit_exact(synth, oracle):
    """The workload the headline numbers are quoted on (bench.py, BASELINE.json configs[1]): 3115 templates (89 views x
    35 variants), 150 features per modality at level 0, T = [4, 8], 640x480 frames of bench.py's ring (seeds 1000 + i),
    threshold 75 -- and 90 for the candidate-rate sweep.  Match lists and the candidate / algorithmic-byte counters equal
    the oracle's."""
    import os
    T = [4, 8]
    bank = synth.synth_bank(3115, num_features=150, levels=2, seed=1234, variants=35)
    nat, packed = _native(T, bank)
    threads = os.cpu_count() or 1
    for seed, thr in ((1000, 75.0), (1001, 75.0), (1175, 75.0), (1002, 90.0)):
        q, planted = synth.synth_frame(640, 480, levels=2, seed=seed, bank=bank, plant=8, T=T)
        got = nat.match_quantized(q, thr)
        want, st = oracle.match(q, T, packed, thr, n_threads=threads, want_stats=True)
        assert len(want) >= len(planted) > 0
        _assert_same(got, want)
        c = nat.counters()
        assert c["templates"] == 3115
        assert c["coarse_candidates"] == int(st["coarse_candidates"])
        assert c["scan_bytes"] == int(st["coarse_byte_adds"])
        assert c["refine_bytes"] == int(st["refine_byte_adds"])


def test_match_mixed_kernels_and_ragged_templates(synth, oracle):
    """Templates whose modalities have different sizes / feature counts (never produced by
    cropTemplates, but legal input): unequal template_positions per modality, empty modality,
    a template larger than the frame, out-of-image features.  Exercises the byte-wise coarse kernel
    next to the bit-sliced one in the same call."""
    T = [4, 8]
    bank = synth.synth_bank(24, num_features=150, levels=2, seed=77)
    tps = bank.classes["01_template"]
    tps[1][3].width += 16            # L1 depth template wider than L1 colour template -> different P
    tps[2][3].features = tps[2][3].features[:0]   # empty L1 depth modality
    tps[3][2].width = 400; tps[3][2].height = 300; tps[3][3].width = 400; tps[3][3].height = 300  # P <= 0
    tps[4][2].features[0, 0] = 330   # x beyond the 320-wide L1 image: skipped (LL.cpp:1330)
    tps[5][0].features[3, 1] = 479   # L0 feature pushed out of the image by the patch offset
    q, _ = synth.synth_frame(640, 480, levels=2, seed=4, bank=bank, plant=5, T=T)
    nat, packed = _native(T, bank)
    for thr in (60.0, 75.0):
        got = nat.match_quantized(q, thr)
        want, st = oracle.match(q, T, packed, thr, want_stats=True)
        _assert_same(got, want)
        c = nat.counters()
        assert c["coarse_candidates"] == int(st["coarse_candidates"])
        assert c["scan_bytes"] == int(st["coarse_byte_adds"])
        assert c["refine_bytes"] == int(st["refine_byte_adds"])


def test_negative_threshold_passes_every_cell(synth, oracle):
    """threshold < 0: every sampled cell is a candidate, including the wrapped / zero ones beyond
    template_positions (LL.cpp:1836-1852 scans all Hd x Wd cells)."""
    T = [4, 8]
    bank = synth.synth_bank(3, num_features=32, levels=2, seed=5)
    q, _ = synth.synth_frame(320, 256, levels=2, seed=6, bank=bank, plant=1, T=T)
    nat, packed = _native(T, bank)
    got = nat.match_quantized(q, -1.0)
    want, st = oracle.match(q, T, packed, -1.0, want_stats=True)
    assert int(st["coarse_candidates"]) == 3 * (320 // 2 // 8) * (256 // 2 // 8)
    _assert_same(got, want)


def test_reference_assertion_is_an_error(synth, oracle):
    """First modality < 64 features but a later one > 63: the reference asserts in similarity_64
    (LL.cpp:1457); the oracle reports it and the C-ABI refuses the selection (RuntimeError)."""
    T = [4, 8]
    bank = synth.synth_bank(4, num_features=150, levels=2, seed=8)
    tps = bank.classes["01_template"]
    tps[2][2].features = tps[2][2].features[:10]
    q, _ = synth.synth_frame(320, 256, levels=2, seed=6)
    packed = bank.pack(bank.class_ids(), 4)
    with pytest.raises(RuntimeError):
        oracle.match(q, T, packed, 80.0)
    lib = importlib.import_module("6dpose_b200._lib")
    nat = lib.NativeDetector(T)
    with pytest.raises(RuntimeError):
        nat.load_bank(packed, 4)


@pytest.mark.parametrize("T,W,H,nf,n,thr", [
    ([4, 8], 320, 2080, 150, 140, 75.0),  # 16-bit path
    ([5, 8], 320, 2640, 63, 70, 70.0),    # the reference's 8-bit (_64) path
])
def test_two_levels_without_filter_bit_exact(synth, oracle, T, W, H, nf, n, thr):
    """Two pyramid levels on a frame whose first refined level is more than 512 cells high: the filter's descriptors
    cannot address it, so the byte-wise k_refine<false> refines every coarse candidate unfiltered."""
    bank = synth.synth_bank(n, num_features=nf, levels=2, seed=21, class_ids=("01_template", "02_template"))
    q, _ = synth.synth_frame(W, H, levels=2, seed=9, bank=bank, plant=6, T=T)
    nat, packed = _native(T, bank)
    got = nat.match_quantized(q, thr)
    want, st = oracle.match(q, T, packed, thr, want_stats=True)
    assert len(want) > 0
    _assert_same(got, want)
    c = nat.counters()
    assert c["coarse_candidates"] == int(st["coarse_candidates"])
    assert c["refine_bytes"] == int(st["refine_byte_adds"])
    assert c["filter_bytes_read"] == 0


def test_unsafe_templates_take_the_byte_path_next_to_the_bit_sliced_one(synth, oracle):
    """A bank in which some templates are not eligible for the bit-sliced refinement (a feature outside the template box:
    "unsafe") next to eligible ones: the filter hands the former to the byte-wise kernel (second survivor list), the
    two exact kernels append to the same result block."""
    T = [4, 8]
    bank = synth.synth_bank(60, num_features=150, levels=2, seed=33)
    tps = bank.classes["01_template"]
    for k in range(0, 60, 3):
        tps[k][0].features[5, 0] = tps[k][0].width + 6   # beyond the box: template k is "unsafe"
    q, _ = synth.synth_frame(640, 480, levels=2, seed=12, bank=bank, plant=6, T=T)
    nat, packed = _native(T, bank)
    for thr in (70.0, 75.0):
        got = nat.match_quantized(q, thr)
        want, st = oracle.match(q, T, packed, thr, want_stats=True)
        assert len(want) > 0
        _assert_same(got, want)
        assert nat.counters()["refine_bytes"] == int(st["refine_byte_adds"])
