"""Pins the CPU oracle (oracle/cvs_oracle.c) against every known answer the reference holds for the hot
path (SURVEY.md section 8c).  CPU only."""
import json
import os

import numpy as np
import pytest

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")


def test_k2_mean_filter_report_matrices(oracle):
    # REPORT/report.tex:2351-2378: 3x3 mean filter, zero padded, on matrices A and B
    A = np.array([[120, 131, 112], [112, 101, 82], [44, 106, 65]], dtype=np.uint8)
    B = np.array([[120, 139, 90], [99, 126, 106], [46, 75, 88]], dtype=np.uint8)
    A_out = np.array([[51, 73, 47], [68, 96, 66], [40, 56, 39]], dtype=np.uint8)
    B_out = np.array([[53, 75, 51], [67, 98, 69], [38, 60, 43]], dtype=np.uint8)
    k = oracle.mean_kernel(3)
    for m, want in ((A, A_out), (B, B_out)):
        img = np.repeat(m.reshape(3, 3, 1), 3, axis=2)  # same matrix in the three channels
        got = oracle.noise_filter(img, 3, 3, 3, k).reshape(3, 3, 3)
        for ch in range(3):
            assert np.array_equal(got[:, :, ch], want)
    # report.tex:2365, :2380: 5 bytes exceed T=20 between A and B, none after filtering
    assert oracle.count_difference(A, B, 20) == 5
    assert oracle.count_difference(A_out, B_out, 20) == 0


def test_k2_channel_interleaving(oracle):
    # tests/noise_filter_benchmark/v1.cu:122 keeps matrix B in channel 2 of a 3x3x3 image: the other
    # channels must not leak into it
    rng = np.random.default_rng(1)
    B = np.array([[120, 139, 90], [99, 126, 106], [46, 75, 88]], dtype=np.uint8)
    img = rng.integers(0, 256, size=(3, 3, 3), dtype=np.uint8)
    img[:, :, 2] = B
    got = oracle.noise_filter(img, 3, 3, 3, oracle.mean_kernel(3)).reshape(3, 3, 3)
    assert np.array_equal(got[:, :, 2], [[53, 75, 51], [67, 98, 69], [38, 60, 43]])


def test_k4_histogram_example(oracle):
    # REPORT/report.tex:3141-3187: 3x3 gray matrix -> counts 0:2, 10:1, 130:1, 255:5
    gray = np.array([0, 0, 10, 130, 255, 255, 255, 255, 255], dtype=np.uint8)
    h = oracle.histogram1(gray)
    want = np.zeros(256, dtype=np.int32)
    want[0], want[10], want[130], want[255] = 2, 1, 1, 5
    assert np.array_equal(h, want)
    assert np.array_equal(oracle.histogram3(np.repeat(gray, 3)), want)


def test_k6_red_byte_of_changed_index(oracle):
    # REPORT/report.tex:2234: red = i + (2 - i % 3)
    for i in range(30):
        out = oracle.red_overlap_from_xs(np.zeros(33, dtype=np.uint8), np.array([i], dtype=np.int32))
        assert out[i + (2 - i % 3)] == 255 and out.sum() == 255


def test_k5_structural_constants():
    # REPORT/report.tex:1440, :762
    N = 3 * 1920 * 1080
    assert 1024 * 6075 == N and -(-6075 // 32) == 190


def test_twomax_quirk(oracle):
    # server.cpp:108-127: sec_max is set to the NEW max, so index_sec_max is the previous running arg-max
    h = np.zeros(256, dtype=np.int32)
    h[100], h[200] = 10, 5
    # running arg-max: ties (>=) move forward through the zero bins up to 99, then 100; afterwards 0-count
    # bins never satisfy >= 10.  imax=100, isec=99 -> 99
    assert oracle.threshold_twomax(h, 0, 255) == (100 + 99) // 2
    assert oracle.threshold_twomax(h, 50, 200) == 99
    h2 = np.zeros(256, dtype=np.int32)
    h2[0] = 7  # arg-max at bin 0: isec stays -1 -> (0 + -1)/2 == 0 in C
    assert oracle.threshold_twomax(h2, 0, 255) == 0
    assert oracle.threshold_twomax(h2, 50, 200) == 50
    h3 = np.full(256, 3, dtype=np.int32)  # all ties: imax=255, isec=254
    assert oracle.threshold_twomax(h3, 50, 200) == 200


def test_a1_semantics_edges(oracle):
    # tests/cuda_streaming/test.cu:560-576
    prev = np.array([100, 100, 100, 100, 255, 0, 50], dtype=np.uint8)
    cur = np.array([120, 121, 80, 79, 0, 255, 50], dtype=np.uint8)
    pos, xs, diff, ref, _ = oracle.diff_compact(cur, prev, 20)
    assert pos == 4
    assert xs.tolist() == [1, 3, 4, 5]
    assert diff.tolist() == [21, (79 - 100) & 255, 1, 255]
    assert ref.tolist() == [100, 121, 100, 79, 0, 255, 50]
    # client round trip (client/opencv.cpp:64-66) reproduces the new reference exactly
    assert np.array_equal(oracle.client_apply(prev, xs, diff), ref)


def test_heat_pixel_endpoints(oracle):
    # tests/heat_map_benchmark/cpu.cu:19-27: d=0 -> blue, d=255 -> green, d>=510 -> red
    assert oracle.heat_pixel(0) == (0, 0, 255)
    r, g, b = oracle.heat_pixel(255)
    assert g == 255 and r == 0 and b in (0, 1)
    assert oracle.heat_pixel(510)[0] == 255


def test_k1_fixture_changed_bytes(oracle):
    # REPORT/report.tex:2594: 369,350 changed bytes (5.93 %) between f1.jpg and f2.jpg (committed byte for byte as
    # tests/golden/k1_f1.jpg, k1_f2.jpg)
    cv2 = pytest.importorskip("cv2")
    a = cv2.imread(os.path.join(GOLDEN, "k1_f1.jpg"))
    b = cv2.imread(os.path.join(GOLDEN, "k1_f2.jpg"))
    assert a.shape == (1080, 1920, 3)
    assert oracle.count_difference(a, b, 20) == 369350
    pos, xs, diff, ref, _ = oracle.diff_compact(b, a, 20)
    assert pos == 369350
    assert np.all(np.diff(xs) > 0)
    assert np.array_equal(oracle.client_apply(a, xs, diff), ref)


def test_k1_committed_fixture_copies(oracle):
    # the same pair as committed fixtures (tests/golden/k1_f1.jpg, k1_f2.jpg: byte copies of the reference's
    # tests/noise_filter_benchmark/f1.jpg and f2.jpg, whose SHA-256 digests are pinned below)
    cv2 = pytest.importorskip("cv2")
    import hashlib
    for name, digest in (("k1_f1.jpg", "809f5ef0d3b6a54f663c2c61989b31232a2262180ceaa6fdf8cdde65e0c1df49"),
                         ("k1_f2.jpg", "4a2b18dde169e7859cec82626416eee48a50de520674790e08c426e9c5f25dea")):
        with open(os.path.join(GOLDEN, name), "rb") as x:
            assert hashlib.sha256(x.read()).hexdigest() == digest, name
    with open(os.path.join(GOLDEN, "k1_f1_f2.json")) as f:
        g = json.load(f)
    a = cv2.imread(os.path.join(GOLDEN, "k1_f1.jpg"))
    b = cv2.imread(os.path.join(GOLDEN, "k1_f2.jpg"))
    sha = lambda x: hashlib.sha256(np.ascontiguousarray(x).tobytes()).hexdigest()
    assert sha(a) == g["sha256_f1"] and sha(b) == g["sha256_f2"]
    pos, xs, diff, ref, _ = oracle.diff_compact(b, a, 20)
    assert pos == 369350 == oracle.count_difference(a, b, 20)
    assert sha(xs) == g["sha256_xs"] and sha(diff) == g["sha256_diff"] and sha(ref) == g["sha256_new_reference"]


def test_golden_k1_record():
    # the K1 facts as recorded by tests/golden/make_golden.py in the build container (travels to the GPU box)
    with open(os.path.join(GOLDEN, "k1_f1_f2.json")) as f:
        g = json.load(f)
    assert g["changed_bytes"] == 369350 and g["total_bytes"] == 6220800


def test_a1_matches_an_independent_numpy_restatement(oracle):
    # second, independent statement of tests/cuda_streaming/test.cu:560-576 (vectorised numpy) on random frames,
    # including the wrap cases of the uint8 difference and several thresholds
    rng = np.random.default_rng(7)
    for n, thr in ((1, 20), (97, 20), (4096, 0), (4096, 20), (4099, 127), (5000, 200), (333, 255), (333, -1)):
        prev = rng.integers(0, 256, size=n, dtype=np.uint8)
        cur = rng.integers(0, 256, size=n, dtype=np.uint8)
        near = rng.random(n) < 0.5  # half the bytes close to the reference so both branches are exercised
        cur = np.where(near, np.clip(prev.astype(int) + rng.integers(-25, 26, size=n), 0, 255), cur).astype(np.uint8)
        df = cur.astype(np.int32) - prev.astype(np.int32)
        changed = (df < -thr) | (df > thr)
        pos, xs, diff, ref, after = oracle.diff_compact(cur, prev, thr)
        assert pos == int(changed.sum())
        assert np.array_equal(xs, np.flatnonzero(changed).astype(np.int32))
        assert np.array_equal(diff, (df[changed] & 0xFF).astype(np.uint8))
        assert np.array_equal(ref, np.where(changed, cur, prev))
        # the payload overwrites the head of the frame buffer, the tail keeps the input (kernels.cu:522)
        assert np.array_equal(after[pos:], cur[pos:]) and np.array_equal(after[:pos], diff)
        assert np.array_equal(oracle.client_apply(prev, xs, diff), ref)


def test_filters_match_independent_numpy_restatements(oracle):
    rng = np.random.default_rng(11)
    w, h = 37, 23
    a = rng.integers(0, 256, size=(h, w, 3), dtype=np.uint8)
    b = rng.integers(0, 256, size=(h, w, 3), dtype=np.uint8)
    # gray average / weighted (server.cpp:96-101, grayscale-weighted/cpu.cu:38-42)
    assert np.array_equal(oracle.gray_avg1(a, w, h), (a.astype(int).sum(axis=2) // 3).astype(np.uint8).reshape(-1))
    wg = (0.114 * a[:, :, 0].astype(np.float64) + 0.587 * a[:, :, 1].astype(np.float64)) + 0.299 * a[:, :, 2].astype(np.float64)
    assert np.array_equal(oracle.gray_weighted1(a, w, h), wg.astype(np.uint8).reshape(-1))
    # red map (heat_map_red_benchmark/cpu.cu:38-55)
    ch = (np.abs(a.astype(int) - b.astype(int)) > 20).any(axis=2)
    red = np.zeros((h, w, 3), dtype=np.uint8)
    red[:, :, 2] = np.where(ch, 255, 0)
    assert np.array_equal(oracle.red_map(a, b, w, h, 20), red.reshape(-1))
    # heat map (heat_map_benchmark/cpu.cu:19-27,54-66)
    d = np.abs(a.astype(int) - b.astype(int)).sum(axis=2)
    x = (d / 510.0).astype(np.float32).astype(np.float64)
    r = np.minimum(np.maximum(np.sin(np.pi * x - np.pi / 2.0) * 255.0, 0.0), 255.0).astype(int)
    g = np.minimum(np.maximum(np.sin(np.pi * x) * 255.0, 0.0), 255.0).astype(int)
    bl = np.minimum(np.maximum(np.sin(np.pi * x + np.pi / 2.0) * 255.0, 0.0), 255.0).astype(int)
    heat = np.stack([bl, g, r], axis=2).astype(np.uint8)
    assert np.array_equal(oracle.heat_map(a, b, w, h), heat.reshape(-1))
