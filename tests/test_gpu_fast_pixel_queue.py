"""FAST candidate parity at the edges of fast_kernel's per-pixel scoring: the cheap reject queues single pixels, the exact
score runs on pixel pairs, and the minThFAST fallback (pass B) rescans cells whose iniThFAST corners were all suppressed.
Every level's candidate set (x, y, score) must equal the oracle port's."""
import numpy as np
import pytest

from orb_slam2_b200 import synth

pytestmark = pytest.mark.gpu

# FAST ring, radius 3, in circular order
RX = [0, 1, 2, 3, 3, 3, 2, 1, 0, -1, -2, -3, -3, -3, -2, -1]
RY = [3, 3, 2, 1, 0, -1, -2, -3, -3, -3, -2, -1, 0, 1, 2, 3]
THRESHOLDS = [(20, 7), (12, 7), (7, 20), (140, 7)]


def cand_set(c):
    return sorted(map(tuple, c.tolist()))


def check_levels(G, P, img, nlevels=8):
    G(img)
    P(img)
    for l in range(nlevels):
        assert cand_set(G.debug_candidates(l)) == cand_set(P.candidates(l)), f"FAST candidates level {l}"


def ring_probes(w, h, ini, mn):
    """Isolated centre pixels whose ring differences sit at t - 1, t, t + 1 for both thresholds, and at the saturated
    0/255 extremes, on arcs of 8, 9, 12 and 16 ring pixels of either polarity.  Probes run up to the right image border."""
    img = np.full((h, w), 128, np.uint8)
    used = np.zeros((h, w), bool)
    diffs = sorted({d for t in (ini, mn) for d in (t - 1, t, t + 1) if 0 < d <= 255})
    cases = []
    for d in diffs:
        lo = (255 - d) // 2
        for arc in (8, 9, 12, 16):
            cases += [(lo, lo + d, arc), (lo + d, lo, arc)]        # bright and dark arcs
    for arc in (8, 9, 16):
        cases += [(0, 255, arc), (255, 0, arc)]
    xs = list(range(22, w - 21, 9)) + [w - 21, w - 20]      # the last columns clip the tile's last word
    ys = range(22, h - 21, 9)
    i = 0
    for y in ys:
        for x in xs:
            if x > w - 20 or used[y - 4:y + 5, x - 4:x + 5].any():
                continue
            centre, ring, arc = cases[i % len(cases)]
            first = (7 * i) % 16
            img[y - 3:y + 4, x - 3:x + 4] = centre               # the ring pixels off the arc differ by 0
            used[y - 3:y + 4, x - 3:x + 4] = True
            for k in range(arc):
                img[y + RY[(first + k) % 16], x + RX[(first + k) % 16]] = ring
            i += 1
    return img


@pytest.mark.parametrize("ini,mn", THRESHOLDS)
@pytest.mark.parametrize("w", [640, 643])
def test_ring_differences_at_threshold(ini, mn, w):
    from oracle import oracle_lib as O
    from orb_slam2_b200.extractor import ORBextractor
    img = ring_probes(w, 360, ini, mn)
    check_levels(ORBextractor(1000, 1.2, 8, ini, mn), O.PortExtractor(1000, 1.2, 8, ini, mn), img)


@pytest.mark.parametrize("ini,mn", THRESHOLDS)
def test_white_noise_fills_the_pixel_queue(ini, mn):
    """Nearly every pixel survives the reject: each warp's queue segment runs many 64-pixel rounds."""
    from oracle import oracle_lib as O
    from orb_slam2_b200.extractor import ORBextractor
    img = synth.white_noise(32, *synth.KITTI)
    check_levels(ORBextractor(2000, 1.2, 8, ini, mn), O.PortExtractor(2000, 1.2, 8, ini, mn), img)


def test_plateau_cell_falls_back_with_pass_a_pixels():
    """A cell whose only iniThFAST corners are an equal-score pair (strict NMS drops both) falls back to minThFAST.  The
    pixel 8 rows below passes the iniThFAST reject (8 ring pixels at +30) but scores 9: it is scored in pass A and is
    the cell's only minThFAST candidate, so pass B must take it from pass A's pixels."""
    from oracle import oracle_lib as O
    from orb_slam2_b200.extractor import ORBextractor
    bg = 100
    img = np.full((300, 400), bg, np.uint8)
    img[50, 60] = img[50, 61] = 250
    cx, cy = 60, 58
    for k in range(16):
        img[cy + RY[k], cx + RX[k]] = bg + (30 if k < 8 else 10)
    G, P = ORBextractor(1000, 1.2, 8, 20, 7), O.PortExtractor(1000, 1.2, 8, 20, 7)
    check_levels(G, P, img)
    assert (cx, cy, 9) in cand_set(G.debug_candidates(0))


@pytest.mark.parametrize("w", [1241, 1242, 1243])
def test_right_border_tiles(w):
    """Domain widths that are not a multiple of 4 pixels: the last word of the right-most tiles is partly outside."""
    from oracle import oracle_lib as O
    from orb_slam2_b200.extractor import ORBextractor
    img = synth.mono_frame(33, 0, 0, w, 375)
    img[:, w - 40:] = ring_probes(w, 375, 20, 7)[:, w - 40:]
    check_levels(ORBextractor(2000), O.PortExtractor(2000), img)


def test_batch_of_64_equals_single_images():
    from orb_slam2_b200.extractor import ORBextractor
    imgs = [synth.mono_frame(90 + i, 0, 0, *synth.KITTI) for i in range(60)]
    imgs += [synth.white_noise(91, *synth.KITTI), ring_probes(1242, 375, 20, 7),
             np.full((375, 1242), 77, np.uint8), synth.mono_frame(99, 0, 0, *synth.KITTI)[:, ::-1].copy()]
    G = ORBextractor(2000)
    G.extract_batch(imgs)
    batched = [[cand_set(G.debug_candidates(l, i)) for l in range(8)] for i in range(len(imgs))]
    S = ORBextractor(2000)
    for i, im in enumerate(imgs):
        S(im)
        for l in range(8):
            assert cand_set(S.debug_candidates(l)) == batched[i][l], f"image {i} level {l}"
