"""GPU parity tests proper: the CUDA path through the C ABI vs the oracle (same seeded inputs),
the committed golden vectors produced by the reference itself, and size-independent properties.
Bar: bit-exact for every integer/byte field (octave, response, 256-bit descriptor, counts, order) and —
because the float pipeline is replicated op for op — bit-exact for x, y, angle too (the stated
tolerance in BASELINE.json is 1e-4 px/rad; the tests assert equality and report the max deviation)."""
import glob
import os

import numpy as np
import pytest

from orb_slam2_b200 import synth
from tests.reference_golden import ref  # noqa: F401  (fixture)

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.fixture(scope="module")
def X():
    from orb_slam2_b200.extractor import ORBextractor
    return ORBextractor


def assert_kps_equal(kg, dg, kp, dp):
    assert len(kg) == len(kp), (len(kg), len(kp))
    for f in ("octave", "response", "size", "class_id"):
        assert np.array_equal(kg[f], kp[f]), f
    assert np.array_equal(dg, dp), f"{int((dg != dp).any(axis=1).sum())} descriptors differ"
    for f in ("x", "y", "angle"):
        dev = np.abs(kg[f].astype(np.float64) - kp[f].astype(np.float64)).max() if len(kg) else 0.0
        assert dev <= 1e-4, (f, dev)        # north_star tolerance
        assert np.array_equal(kg[f], kp[f]), (f, dev)   # and in fact bit-identical


@pytest.mark.parametrize("path", sorted(glob.glob(os.path.join(GOLD, "extract_*.npz"))), ids=os.path.basename)
def test_matches_reference_golden_vectors(X, path):
    g = np.load(path)
    w, h, nf, ini, mn, seed = g["meta"].tolist()
    img = synth.mono_frame(seed, 0, 0, w, h)
    kg, dg = X(nf, 1.2, 8, ini, mn)(img)
    assert_kps_equal(kg, dg, g["keypoints"], g["descriptors"])


@pytest.mark.parametrize("shape,nf", [(synth.KITTI, 2000), (synth.TUM, 1000), (synth.EUROC, 1200), ((1241, 376), 2000)])
@pytest.mark.parametrize("seed", [11, 12])
def test_matches_oracle_all_stages(X, oracle, shape, nf, seed):
    w, h = shape
    img = synth.mono_frame(seed, 0, 0, w, h)
    G, P = X(nf), oracle.PortExtractor(nf)
    kg, dg = G(img)
    kp, dp = P(img)
    assert np.array_equal(G.GetScaleFactors(), P.scale) and np.array_equal(G.mnFeaturesPerLevel, P.per_level)
    assert np.array_equal(G.GetInverseScaleSigmaSquares(), P.inv_sigma2)
    for l in range(8):
        assert np.array_equal(G.pyramid(l), P.level(l)), f"pyramid level {l}"
        cg, cp = G.debug_candidates(l), P.candidates(l)
        assert sorted(map(tuple, cg.tolist())) == sorted(map(tuple, cp.tolist())), f"FAST candidates level {l}"
        sel = G.debug_selected(l)
        m = kp["octave"] == l
        assert len(sel) == int(m.sum()), f"quadtree count level {l}"
        assert np.array_equal(sel[:, 2], kp["response"][m].astype(np.int32)), f"quadtree order level {l}"
        if P.blurred(l) is not None:
            assert np.array_equal(G.debug_blurred(l), P.blurred(l)), f"blur level {l}"
    assert_kps_equal(kg, dg, kp, dp)


def test_matches_verbatim_reference_build(X, oracle, ref):
    """Against the reference's ORBextractor.cc compiled verbatim (oracle/_ref) where it is built, and always against what that
    build gave on this frame (tests/golden/reference.json)."""
    img = synth.mono_frame(21, 0, 0, *synth.KITTI)
    kg, dg = X(2000)(img)
    if oracle.have_ref():
        kr, dr = oracle.RefExtractor(2000)(img)
        assert_kps_equal(kg, dg, kr, dr)
    ref.expect((kg, dg))


@pytest.mark.parametrize("nf", [300, 1000, 4000])
def test_white_noise_stress(X, oracle, nf):
    """~10x the corner density of a natural frame: tens of thousands of candidates per level."""
    img = synth.white_noise(31, 640, 360)
    kg, dg = X(nf)(img)
    kp, dp = oracle.PortExtractor(nf)(img)
    assert_kps_equal(kg, dg, kp, dp)


def test_edge_cases(X, oracle):
    G, P = X(1000), oracle.PortExtractor(1000)
    blank = np.full((240, 320), 128, np.uint8)
    k, d = G(blank)
    assert len(k) == 0 and d.shape == (0, 32)              # zero keypoints -> descriptors released (:1064)
    k, d = G(np.zeros((0, 0), np.uint8))
    assert len(k) == 0                                      # empty image -> silent return (:1046)
    one = blank.copy(); one[100:140, 150:200] = 220
    assert_kps_equal(*G(one), *P(one))
    weak = blank.copy(); weak[60:120, 70:150] = 140         # only reachable through the minThFAST fallback
    kg, dg = G(weak)
    assert len(kg) > 0 and kg["response"].max() < 20
    assert_kps_equal(kg, dg, *P(weak))
    plateau = blank.copy(); plateau[::2, ::2] = 200         # equal-score plateaus: strict NMS
    assert_kps_equal(*G(plateau), *P(plateau))
    sat = synth.mono_frame(41, 0, 0, 400, 300).astype(np.int32) * 3 - 150
    sat = np.clip(sat, 0, 255).astype(np.uint8)             # saturated blacks/whites
    assert_kps_equal(*G(sat), *P(sat))
    # keypoints at the [19, W-20] extremes: bright dots exactly on the detection-domain border
    ext = blank.copy()
    for (x, y) in [(19, 19), (300, 19), (19, 220), (300, 220), (160, 19), (19, 120)]:
        ext[y - 1:y + 2, x - 1:x + 2] = 255
    assert_kps_equal(*G(ext), *P(ext))


def test_thresholds_and_levels_variants(X, oracle):
    img = synth.mono_frame(51, 0, 0, 752, 480)
    for (nf, sf, nl, ini, mn) in [(1200, 1.2, 8, 12, 7), (800, 1.5, 4, 20, 7), (1500, 1.1, 12, 30, 10), (500, 1.2, 8, 7, 20)]:
        kg, dg = X(nf, sf, nl, ini, mn)(img)
        kp, dp = oracle.PortExtractor(nf, sf, nl, ini, mn)(img)
        assert_kps_equal(kg, dg, kp, dp)


@pytest.mark.parametrize("sf,nl", [(2.0, 3), (2.5, 3), (3.1, 2), (1.05, 6)])
def test_pyramid_scale_factor_extremes(X, oracle, sf, nl):
    """Scale factors above ~2 leave the 12-byte source window of the table-driven resize kernel and take the
    generic one; 1.05 packs the window tightly.  Every level and the final keypoints must still match."""
    img = synth.mono_frame(52, 0, 0, 1000, 700)
    G, P = X(600, sf, nl, 20, 7), oracle.PortExtractor(600, sf, nl, 20, 7)
    kg, dg = G(img)
    kp, dp = P(img)
    for l in range(nl):
        assert np.array_equal(G.pyramid(l), P.level(l)), f"pyramid level {l}"
        if P.blurred(l) is not None:
            assert np.array_equal(G.debug_blurred(l), P.blurred(l)), f"blur level {l}"
    assert_kps_equal(kg, dg, kp, dp)


def test_batch_equals_single_and_handles_reshape(X, oracle):
    G = X(1000)
    imgs = [synth.mono_frame(60 + i, 0, 0, 640, 480) for i in range(5)]
    singles = [X(1000)(im) for im in imgs]
    batch = G.extract_batch(imgs)
    for (ks, ds), (kb, db) in zip(singles, batch):
        assert np.array_equal(ks, kb) and np.array_equal(ds, db)
    # same handle, new shape, then back (workspace re-geometry), plus a strided (non-contiguous rows) view
    other = synth.mono_frame(70, 0, 0, 500, 300)
    assert_kps_equal(*G(other), *oracle.PortExtractor(1000)(other))
    wide = np.zeros((480, 700), np.uint8); wide[:, :640] = imgs[0]
    kv, dv = G(wide[:, :640])
    assert np.array_equal(kv, singles[0][0]) and np.array_equal(dv, singles[0][1])
    k2, d2 = G(imgs[1])
    assert np.array_equal(k2, singles[1][0])                # repeatable after other work on the handle


def test_unsupported_shapes_are_errors_not_garbage(X):
    from orb_slam2_b200._lib import BorbError
    with pytest.raises(BorbError):
        X(1000)(np.zeros((100, 100), np.uint8))             # level 7 would have no FAST cell (reference: div by zero)
    with pytest.raises(BorbError):
        X(1000)(np.zeros((200, 5000), np.uint8))            # wider than BORB_MAX_DIM


def test_full_size_properties(X):
    """Size-independent checks at BASELINE's full KITTI size, batch 16."""
    G = X(2000)
    imgs = [synth.mono_frame(80, 0, i, *synth.KITTI) for i in range(16)]
    res = G.extract_batch(imgs)
    again = G.extract_batch(imgs)
    quota = G.mnFeaturesPerLevel
    scale = G.GetScaleFactors()
    for (k, d), (k2, d2) in zip(res, again):
        assert np.array_equal(k, k2) and np.array_equal(d, d2)           # idempotent
        assert np.all(np.diff(k["octave"]) >= 0)                         # levels concatenated 0..7
        for l in range(8):
            n = int((k["octave"] == l).sum())
            assert quota[l] <= n <= quota[l] + 3                         # never trimmed, <= quota+3 (SURVEY a4)
            m = k["octave"] == l
            lx, ly = k["x"][m] / scale[l], k["y"][m] / scale[l]
            lw, lh = np.rint(np.float32(1242) / scale[l]), np.rint(np.float32(375) / scale[l])
            assert lx.min() >= 18.99 and ly.min() >= 18.99 and lx.max() <= lw - 19.99 and ly.max() <= lh - 19.99
        assert np.all((k["angle"] >= 0) & (k["angle"] < 360)) and np.all(k["class_id"] == -1)
        assert np.all(k["response"] >= 7)
        # no two keypoints of one level share a pixel
        key = k["octave"].astype(np.int64) * (1 << 40) + np.rint(k["x"] * 64).astype(np.int64) * (1 << 20) + np.rint(k["y"] * 64).astype(np.int64)
        assert len(np.unique(key)) == len(k)
    # flipping the image left-right changes the keypoints (sanity: results depend on the input)
    kf, _ = G(imgs[0][:, ::-1].copy())
    assert not np.array_equal(kf["x"][:50], res[0][0]["x"][:50])


@pytest.mark.parametrize("channels,rgb", [(3, True), (3, False), (4, True), (4, False)])
def test_colour_input_is_converted_like_cvtcolor(X, channels, rgb):
    """Tracking::GrabImage* call cv::cvtColor(RGB2GRAY/BGR2GRAY/RGBA2GRAY/BGRA2GRAY) first (src/Tracking.cc:172-197);
    the conversion is fused into the upload.  Level 0 must equal cv2's gray image, the keypoints those of the gray path."""
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(8)
    gray = synth.mono_frame(71, 0, 0, 640, 480)
    col = np.stack([np.clip(gray.astype(np.int32) + rng.integers(-40, 41, gray.shape), 0, 255).astype(np.uint8) for _ in range(channels)], 2)
    code = {(3, True): cv2.COLOR_RGB2GRAY, (3, False): cv2.COLOR_BGR2GRAY, (4, True): cv2.COLOR_RGBA2GRAY, (4, False): cv2.COLOR_BGRA2GRAY}[(channels, rgb)]
    want = cv2.cvtColor(col, code)
    G = X(1000)
    G.set_input_format(channels, rgb)
    kc, dc = G(col)
    assert np.array_equal(G.pyramid(0), want)
    kg, dg = X(1000)(want)
    assert_kps_equal(kc, dc, kg, dg)
    # batch of scattered colour frames, and a strided view
    outs = G.extract_batch([col, col[:, ::-1].copy()])
    assert np.array_equal(outs[0][0], kc) and np.array_equal(outs[0][1], dc)
    wide = np.zeros((480, 700, channels), np.uint8); wide[:, :640] = col
    kv, dv = G(wide[:, :640])
    assert np.array_equal(kv, kc) and np.array_equal(dv, dc)
    # back to gray on the same handle
    kb, db = G(want)
    assert_kps_equal(kb, db, kg, dg)
