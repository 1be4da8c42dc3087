"""The anchor-scan restatement (oracle/scan_oracle.c) against the reference's own golden strings
(src/lib/extractor/test/ScannerTest.cpp), against cv2 for the OpenCV arithmetic it restates, and against the results of the
reference's ScanState / Anchor classes compiled unmodified (stored in tests/golden/ref_outputs.json)."""
import ctypes as C

import cv2
import numpy as np
import pytest

import oracle_lib as ol
from scan_oracle_lib import ScanOracle, anchor_str, join

SO = ScanOracle()
GOLD = ol.manifest()["scan_goldens"]


def _scanner(sample):
    rgb = ol.load_sample(sample)
    t, bin_, _ = SO.preprocess(rgb)
    assert t >= 0
    return SO.scanner(bin_)


@pytest.mark.parametrize("ksize,shape", [(3, (211, 317)), (5, (96, 333)), (7, (80, 81)), (9, (130, 64)), (3, (5, 4))])
def test_gaussian_blur_is_cv2s(ksize, shape):
    rng = np.random.default_rng(ksize)
    for img in (rng.integers(0, 256, shape, dtype=np.uint8), (rng.integers(0, 2, shape) * 255).astype(np.uint8)):
        out = np.zeros_like(img)
        assert SO.lib.cbo_scan_gaussian_blur(ol._ptr(img), shape[1], shape[0], ksize, ol._ptr(out)) == 0
        assert np.array_equal(out, cv2.GaussianBlur(img, (ksize, ksize), 0))


def test_otsu_is_cv2s():
    rng = np.random.default_rng(2)
    imgs = [np.clip(rng.normal(rng.integers(40, 200), rng.integers(5, 80), (64, 64)), 0, 255).astype(np.uint8) for _ in range(40)]
    imgs += [np.zeros((8, 8), np.uint8), np.full((8, 8), 255, np.uint8), rng.integers(0, 2, (32, 32)).astype(np.uint8) * 255]
    imgs += [cv2.cvtColor(ol.load_sample(s), cv2.COLOR_RGB2GRAY) for s in ("6bit/4_30_f0_627.jpg", "b/ex2434.jpg")]
    for img in imgs:
        img = np.ascontiguousarray(img)
        t, _ = cv2.threshold(img, 0, 255, cv2.THRESH_BINARY | cv2.THRESH_OTSU)
        assert SO.lib.cbo_scan_otsu(ol._ptr(img), img.size) == int(t)


@pytest.mark.parametrize("sample", ["6bit/4_30_f0_627.jpg", "6bit/4_30_f1_360.jpg", "6bit/4color_ecc30_fountain_0.png"])
def test_preprocess_is_the_reference_pipeline_in_cv2(sample):
    # Scanner::preprocess_image(img, fast=true), Scanner.h:146-166
    rgb = ol.load_sample(sample)
    t, bin_, blurred = SO.preprocess(rgb)
    gray = cv2.cvtColor(rgb, cv2.COLOR_RGB2GRAY)
    unit = SO.lib.cbo_scan_blur_size(rgb.shape[1], rgb.shape[0])
    assert unit == 3
    bl = cv2.GaussianBlur(gray, (unit, unit), 0)
    tt, want = cv2.threshold(bl, 0, 255, cv2.THRESH_BINARY | cv2.THRESH_OTSU)
    assert np.array_equal(blurred, bl) and t == int(tt) and np.array_equal(bin_, want)


def test_blur_size_rule():
    # max(nextPowerOfTwoPlusOne(unsigned(min(cols, rows) * 0.002)), 3), Scanner.h:93-103, :155-157
    for (w, h), k in {(1280, 960): 3, (1499, 2000): 3, (1500, 1500): 5, (2499, 4000): 5, (2704, 3052): 9, (4499, 4499): 9, (4500, 6000): 17}.items():
        assert SO.lib.cbo_scan_blur_size(w, h) == k
    big = np.zeros((4500, 4500, 3), np.uint8)
    assert SO.scan(big)[0] is None                      # kernels beyond 9 taps are not restated: reported, not guessed


def test_scanner_piecemeal_golden():
    # ScannerTest/testPiecemealScan, ScannerTest.cpp:16-52
    g = GOLD[0]
    s = _scanner(g["sample"])
    c1 = SO.t1(s)
    for want in g["t1_contains"]:
        assert want in join(c1)
    c2 = [p for c in c1 for p in SO.t2(s, c)]
    for want in g["t2_contains"]:
        assert want in join(c2)
    c3 = [p for c in c2 for p in SO.t3(s, c)]
    for want in g["t3_contains"]:
        assert want in join(c3)
    c4 = [p for c in c3 for p in SO.t4(s, c, True)]
    cands, _ = SO.filter(SO.deduplicate(s, c4))
    assert join(cands) == g["piecemeal_filtered"]


@pytest.mark.parametrize("g", GOLD, ids=lambda g: g["sample"])
def test_scan_goldens(g):
    # ScannerTest/testBottomRightCorner(.2 .3 .4), testExampleScan(.2 .3): ScannerTest.cpp:54-176
    rgb = ol.load_sample(g["sample"])
    if "primary" in g:
        s = _scanner(g["sample"])
        cands, cutoff = SO.primary(s)
        assert cutoff == g["cutoff"] and join(cands) == g["primary"]
        four, ok = SO.bottom_right(s, cands, cutoff)
        assert ok and join(four) == g["scan"]
    anchors, _ = SO.scan(rgb)
    assert join(anchors) == g["scan"]


def test_sort_top_to_bottom_goldens():
    for g in ol.manifest()["sort_goldens"]:
        assert join(SO.sort_top_to_bottom([tuple(a) for a in g["in"]])) == g["out"], g["source"]


def scanstate_patterns(run):
    """extractor/ScanState.h through scan_horizontal on one-row images: run(kind, row) -> the patterns found, as (x0, x1, 0, 0)"""
    rng = np.random.default_rng(9)
    out = []
    for trial in range(300):
        n = int(rng.integers(1, 400))
        # runs with lengths around the 1:1:4:1:1 (and 1:2:2 ...) ratios, so that patterns do occur
        unit = int(rng.integers(1, 12))
        runs = []
        while sum(runs) < n:
            runs.append(max(1, int(unit * rng.choice([1, 1, 1, 2, 4, 4, 3]) + rng.integers(-1, 2))))
        row = np.concatenate([np.full(r, (i + trial) % 2, np.uint8) for i, r in enumerate(runs)])[:n]
        for kind in (114, 122):
            out.append([tuple(int(v) for v in p) for p in run(kind, row)])
    return out


def restated_scanstate(kind, row):
    s = SO.scanner((row * 255).reshape(1, row.size))
    return SO.t1(s, kind=kind, skip=1, y=0, yend=1)


def anchor_ops(op):
    """extractor/Anchor.h: is_mergeable / merge / size drive dedup and filter_candidates.  op(a, b) -> (a and b deduplicated,
    a as the reference prints it, filter_candidates' cutoff on three copies of a)"""
    rng = np.random.default_rng(10)
    out = []
    for trial in range(500):
        ax, ay = int(rng.integers(0, 1200)), int(rng.integers(0, 1200))
        a = (ax, ax + int(rng.integers(1, 80)), ay, ay + int(rng.integers(0, 80)))
        b = (ax + int(rng.integers(-40, 40)), ax + int(rng.integers(1, 90)), ay + int(rng.integers(-40, 40)), ay + int(rng.integers(0, 90)))
        merged, text, cutoff = op(a, b)
        out.append(([tuple(int(v) for v in x) for x in merged], text, int(cutoff)))
    return out


def restated_anchor_op(a, b):
    s = SO.scanner(np.zeros((4, 960), np.uint8))          # merge_cutoff = 960 / 30 = 32
    return SO.deduplicate(s, [a, b]), anchor_str(a), SO.filter([a, a, a])[1]


def test_scan_state_machine_is_the_references():
    # extractor/ScanState.h compiled unmodified (oracle/_ref; tests/golden/make_ref_goldens.py) against the restatement
    got = scanstate_patterns(restated_scanstate)
    assert sum(len(p) for p in got) > 200
    assert ol.digest(got) == ol.ref_outputs()["scanstate_patterns"]


def test_anchor_arithmetic_is_the_references():
    # extractor/Anchor.h compiled unmodified (oracle/_ref; tests/golden/make_ref_goldens.py) against the restatement
    assert ol.digest(anchor_ops(restated_anchor_op)) == ol.ref_outputs()["anchor_ops"]


def test_upscaled_picture_uses_the_nine_tap_blur_and_still_scans():
    rgb = ol.load_sample("6bit/4_30_f0_627.jpg")
    big = cv2.resize(rgb, None, fx=3, fy=3, interpolation=cv2.INTER_LINEAR)      # 2880 x 3840: unit = 9
    assert SO.lib.cbo_scan_blur_size(big.shape[1], big.shape[0]) == 9
    t, bin_, blurred = SO.preprocess(big)
    bl = cv2.GaussianBlur(cv2.cvtColor(big, cv2.COLOR_RGB2GRAY), (9, 9), 0)
    tt, want = cv2.threshold(bl, 0, 255, cv2.THRESH_BINARY | cv2.THRESH_OTSU)
    assert np.array_equal(blurred, bl) and t == int(tt) and np.array_equal(bin_, want)
    anchors, cutoff = SO.scan(big)
    assert len(anchors) == 4
    # the same four anchors as at the original size, three times as far out (within the scan's granularity)
    small = SO.scan(rgb)[0]
    for a, b in zip(anchors, small):
        assert abs((a[0] + a[1]) // 2 - 3 * ((b[0] + b[1]) // 2)) <= 6 and abs((a[2] + a[3]) // 2 - 3 * ((b[2] + b[3]) // 2)) <= 6


def test_adaptive_scanner_variant():
    # Scanner(img, fast=false): ScannerTest/testExampleScan.Adaptive (ScannerTest.cpp:178-189) and cv2's adaptiveThreshold on the blurred picture
    g = GOLD[0]
    rgb = ol.load_sample(g["sample"])
    h, w = rgb.shape[:2]
    bin_ = np.zeros((h, w), np.uint8)
    SO.lib.cbo_scan_preprocess_adaptive.argtypes = [C.POINTER(C.c_uint8), C.c_int, C.c_int, C.POINTER(C.c_uint8)]
    assert SO.lib.cbo_scan_preprocess_adaptive(ol._ptr(rgb), w, h, ol._ptr(bin_)) == 0
    bl = cv2.GaussianBlur(cv2.cvtColor(rgb, cv2.COLOR_RGB2GRAY), (3, 3), 0)
    want = cv2.adaptiveThreshold(bl, 255, cv2.ADAPTIVE_THRESH_MEAN_C, cv2.THRESH_BINARY, 65, -10)      # unit: 960 * 0.05 = 48 -> 65
    assert np.array_equal(bin_, want)
    from scan_oracle_lib import Anchor
    out = (Anchor * 4)(); cutoff = C.c_uint(0)
    SO.lib.cbo_scan2.argtypes = [C.POINTER(C.c_uint8), C.c_int, C.c_int, C.c_int, C.POINTER(Anchor), C.POINTER(C.c_uint)]
    n = SO.lib.cbo_scan2(ol._ptr(rgb), w, h, 0, out, C.byref(cutoff))
    assert n == 4 and join([out[i].tup() for i in range(4)]) == g["scan_adaptive"]


def _average_hash(rgb):
    # image_hash::average_hash (image_hash/average_hash.h:19-40): gray, cv::resize to 8 x 8, threshold = Cell::mean_grayscale (floor of the mean)
    g = cv2.resize(cv2.cvtColor(rgb, cv2.COLOR_RGB2GRAY), (8, 8))
    thr = int(g.astype(np.uint32).sum()) // 64
    v = 0
    for b in (g > thr).reshape(-1):
        v = (v << 1) | int(b)
    return v


@pytest.mark.parametrize("sample,want", [("6bit/4_30_f2_734.jpg", 0xc7f8205e686bc02), ("6bit/4_30_f0_627.jpg", 0x29c64eaca3356394)])
def test_extractor_goldens(sample, want, tmp_path):
    """ExtractorTest/testExtract, testExtractMid (extractor/test/ExtractorTest.cpp:13-50): ExtractorPlus::extract =
    Scanner::scan -> Corners -> Deskewer, written as JPEG, read back, average_hash.  Scan by the restatement, the two OpenCV calls of
    Deskewer::deskew by cv2: the reference's golden hashes come out.  (testExtractUpscale's 2.9 MB picture is not stored here; the
    9-tap blur it exercises is checked by test_upscaled_picture_uses_the_nine_tap_blur_and_still_scans.)"""
    rgb = ol.load_sample(sample)
    anchors, _ = SO.scan(rgb)
    assert len(anchors) == 4
    src = np.array(SO.corners(anchors), np.float32).reshape(4, 2)
    dst = np.array([[30, 30], [994, 30], [30, 994], [994, 994]], np.float32)            # Deskewer.h:27-32, padding 0
    out = cv2.warpPerspective(rgb, cv2.getPerspectiveTransform(src, dst), (1024, 1024), flags=cv2.INTER_LINEAR)
    p = str(tmp_path / "ex.jpg")
    cv2.imwrite(p, cv2.cvtColor(out, cv2.COLOR_RGB2BGR))
    back = np.ascontiguousarray(cv2.cvtColor(cv2.imread(p), cv2.COLOR_BGR2RGB))
    assert _average_hash(back) == want
