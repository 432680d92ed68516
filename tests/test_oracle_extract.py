"""Oracle self-consistency: the independent restatement (oracle/orb_port_extract.cpp) against the
reference's own ORBextractor.cc compiled verbatim (oracle/_ref), and against cv2 4.13 run the way
ORBextractor.cc:789-829 runs it (one cv::FAST call per cell).  Where the verbatim build is absent, the results it gave are taken
from tests/golden/reference.json (tests/reference_golden.py)."""
import math

import numpy as np
import pytest

from orb_slam2_b200 import synth
from tests.reference_golden import ref  # noqa: F401  (fixture)


def _live(O, fn):
    """fn on the verbatim reference build where it is built, else None (the stored results stand in)."""
    return fn if O.have_ref() else None

SHAPES = [(synth.KITTI, 2000), (synth.TUM, 1000), (synth.EUROC, 1200)]


@pytest.mark.parametrize("shape,nf", SHAPES)
@pytest.mark.parametrize("seed", [1, 2])
def test_port_equals_verbatim_reference(oracle, shape, nf, seed, ref):
    w, h = shape
    img = synth.mono_frame(seed, 0, 0, w, h)
    O, P = oracle, oracle.PortExtractor(nf)
    names = ("scale", "inv_scale", "sigma2", "inv_sigma2", "per_level", "umax")
    ref.expect([getattr(P, n) for n in names], _live(O, lambda: [getattr(O.RefExtractor(nf), n) for n in names]))

    def run(E):
        k, d = E(img)
        return k, d, [E.level(l) for l in range(8)]
    kp, dp, lp = run(P)
    assert len(kp) >= nf
    ref.expect((kp, dp, lp), _live(O, lambda: run(O.RefExtractor(nf))))    # all 7 KeyPoint fields, same order; descriptors; pyramid


@pytest.mark.parametrize("nf", [500, 2000, 4000])
def test_port_equals_reference_white_noise(oracle, nf, ref):
    img = synth.white_noise(11, 640, 360)
    ref.expect(oracle.PortExtractor(nf)(img), _live(oracle, lambda: oracle.RefExtractor(nf)(img)))


def test_reference_call_is_repeatable(oracle, ref):
    """The monotonic allocator makes the address-ordered quadtree tie-break deterministic: a second call on the same image, after
    another image, gives the first call's result (for the reference build and the restatement alike)."""
    img = synth.mono_frame(4, 0, 0, *synth.KITTI)
    other = synth.white_noise(1, 400, 300)

    def twice(E):
        k1, d1 = E(img)
        E(other)
        k2, d2 = E(img)
        assert np.array_equal(k1, k2) and np.array_equal(d1, d2)
        return k1, d1
    ref.expect(twice(oracle.PortExtractor(2000)), _live(oracle, lambda: twice(oracle.RefExtractor(2000))))


def test_edge_cases(oracle, ref):
    O, P = oracle, oracle.PortExtractor(1000)
    R = O.RefExtractor(1000) if O.have_ref() else None
    blank = np.full((240, 320), 128, np.uint8)
    k, d = P(blank)
    assert len(k) == 0 and d.shape == (0, 32)
    ref.expect((k, d), _live(O, lambda: R(blank)))
    one = blank.copy()
    one[100:140, 150:200] = 220            # a single bright rectangle: 4 corners per level
    kp, dp = P(one)
    assert len(kp) > 0
    ref.expect((kp, dp), _live(O, lambda: R(one)))
    weak = blank.copy()
    weak[60:120, 70:150] = 140             # contrast 12: only reachable through the minThFAST=7 fallback
    kp, dp = P(weak)
    assert len(kp) > 0 and kp["response"].max() < 20
    ref.expect((kp, dp), _live(O, lambda: R(weak)))
    plateau = blank.copy()
    plateau[::2, ::2] = 200                # dense equal-score ties: strict NMS keeps none of a tie pair
    ref.expect(P(plateau), _live(O, lambda: R(plateau)))


def _cells_cv2(level_img, ini_th=20, min_th=7):
    """ORBextractor.cc:765-829 with the real cv2.FAST, one call per cell."""
    cv2 = pytest.importorskip("cv2")
    H, W = level_img.shape
    minB, maxBX, maxBY = 16, W - 16, H - 16
    width, height = float(maxBX - minB), float(maxBY - minB)
    nCols, nRows = int(width / 30), int(height / 30)
    wCell, hCell = math.ceil(width / nCols), math.ceil(height / nRows)
    det = {t: cv2.FastFeatureDetector_create(threshold=t, nonmaxSuppression=True) for t in (ini_th, min_th)}
    out = []
    for i in range(nRows):
        iniY = minB + i * hCell
        maxY = iniY + hCell + 6
        if iniY >= maxBY - 3:
            continue
        maxY = min(maxY, maxBY)
        for j in range(nCols):
            iniX = minB + j * wCell
            maxX = iniX + wCell + 6
            if iniX >= maxBX - 6:
                continue
            maxX = min(maxX, maxBX)
            sub = np.ascontiguousarray(level_img[iniY:maxY, iniX:maxX])
            k = det[ini_th].detect(sub, None)
            if len(k) == 0:
                k = det[min_th].detect(sub, None)
            for kp in k:
                out.append((int(kp.pt[0]) + iniX, int(kp.pt[1]) + iniY, int(kp.response)))
    return out


@pytest.mark.parametrize("shape", [synth.KITTI, synth.TUM, (179, 134), (719, 217)])
def test_whole_level_candidates_equal_per_cell_cv2(oracle, shape):
    w, h = shape
    for img in (synth.mono_frame(6, 0, 0, w, h), synth.white_noise(2, w, h),
                (synth.mono_frame(7, 0, 0, w, h) // 8 + 100).astype(np.uint8)):   # low contrast: fallback cells
        P = oracle.PortExtractor(1000)
        P(img)
        got = [tuple(r) for r in P.candidates(0).tolist()]
        want = _cells_cv2(img)
        assert got == want


@pytest.mark.parametrize("N", [5, 60, 434, 869])
def test_quadtree_port_equals_reference(oracle, N, ref):
    rng = np.random.default_rng(N)
    R = oracle.RefExtractor(2000) if oracle.have_ref() else None
    for width, height in [(1210, 343), (608, 448), (147, 102), (315, 73)]:
        for n in (1, 2, 7, 300, 5000):
            n = min(n, (width - 6) * (height - 6) // 4)
            flat = rng.choice((width - 6) * (height - 6), size=n, replace=False)
            xs, ys = 3 + flat % (width - 6), 3 + flat // (width - 6)
            sc = rng.integers(7, 60, n)           # few distinct responses: exercises first-wins ties
            order = np.lexsort((xs, ys))
            xys = np.stack([xs[order], ys[order], sc[order]], 1).astype(np.int32)
            got = oracle.port_distribute(xys, width, height, N)
            ref.expect(got, _live(oracle, lambda: R.distribute(xys.astype(np.float32), width, height, N).astype(np.int32)))
