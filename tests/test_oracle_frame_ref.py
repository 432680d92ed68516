"""CPU: pins the restatements of Frame::ComputeStereoMatches (oracle/orb_port_stereo.cpp), of the feature grid and of
Frame::isInFrustum (oracle/orb_port_match.cpp) — and through them the CUDA kernels — to the REFERENCE SOURCE:
/root/reference/src/Frame.cc compiled verbatim against the reference's real include/Frame.h (oracle/_ref/libframeref.so,
oracle/Makefile target `ref`, oracle/frameref_wrap.cpp, oracle/frameshim/pre.hpp).  Where that build is absent, the results it
gave are taken from tests/golden/reference.json (tests/reference_golden.py)."""
import numpy as np
import pytest

from orb_slam2_b200 import synth
from tests import match_fixtures as mf
from tests.reference_golden import ref  # noqa: F401  (fixture)


@pytest.fixture(scope="module")
def O(oracle):
    return oracle


def _live(O, fn):
    """fn on the reference-side library where it is built, else None (the stored results stand in)."""
    return fn if O.have_frameref() else None


@pytest.mark.parametrize("shape,nf,bf,fx,seed", [((640, 360), 1000, 386.1448, 718.856, 1), ((752, 480), 1200, 47.9, 435.2, 2),
                                                 (synth.KITTI, 2000, 386.1448, 718.856, 3)])
def test_compute_stereo_matches_equals_reference_source(O, shape, nf, bf, fx, seed, ref):
    w, h = shape
    L, R, _ = synth.stereo_pair(seed, 0, 0, w, h)
    E1, E2 = O.PortExtractor(nf), O.PortExtractor(nf)
    kl, dl = E1(L)
    kr, dr = E2(R)
    pl, pr = [E1.level(i) for i in range(8)], [E2.level(i) for i in range(8)]
    ur_p, dp_p, _ = O.port_stereo(kl, dl, kr, dr, pl, pr, E1.scale, E1.inv_scale, bf, fx)
    assert (ur_p >= 0).sum() > 0.3 * len(kl)
    ref.expect((ur_p, dp_p), _live(O, lambda: O.ref_stereo(kl, dl, kr, dr, pl, pr, E1.scale, E1.inv_scale, bf, fx)))


def test_stereo_degenerate_inputs(O, ref):
    """Unrelated left / right images (few, poor matches: the median cull and the rejection branches dominate)."""
    L = synth.mono_frame(5, 0, 0, 640, 360)
    R = synth.mono_frame(6, 0, 0, 640, 360)
    E1, E2 = O.PortExtractor(800), O.PortExtractor(800)
    kl, dl = E1(L)
    kr, dr = E2(R)
    pl, pr = [E1.level(i) for i in range(8)], [E2.level(i) for i in range(8)]
    ur_p, dp_p, _ = O.port_stereo(kl, dl, kr, dr, pl, pr, E1.scale, E1.inv_scale, 386.1448, 718.856)
    ref.expect((ur_p, dp_p), _live(O, lambda: O.ref_stereo(kl, dl, kr, dr, pl, pr, E1.scale, E1.inv_scale, 386.1448, 718.856)))


def test_feature_grid_equals_reference_source(O, ref):
    v = mf.two_views(O, 7)
    k = v["kl"]
    rng = np.random.default_rng(1)
    for bounds in [(0.0, 0.0, 640.0, 480.0), (-12.5, -7.25, 652.0, 491.5)]:
        queries = []
        for _ in range(150):
            x, y, r = rng.uniform(-30, 670), rng.uniform(-30, 510), rng.uniform(2, 80)
            queries.append((x, y, r, int(rng.integers(-1, 7)), int(rng.integers(-1, 8))))
        ref.expect([O.port_features_in_area(k, bounds, *q) for q in queries],                 # same features in the same order
                   _live(O, lambda: [O.ref_features_in_area(k, bounds, *q) for q in queries]))


@pytest.mark.parametrize("seed", [7, 8])
@pytest.mark.parametrize("limit", [0.5, 0.8])
def test_is_in_frustum_equals_reference_source(O, seed, limit, ref):
    v = mf.two_views(O, seed)
    F, P, Tcw, _, K = mf.world_points_case(v, seed + 70)
    fields = ("count", "in_view", "proj_x", "proj_y", "proj_xr", "level", "view_cos")
    Ow = ref.value(_live(O, lambda: O.ref_is_in_frustum(F, P, Tcw, K, 40.0, limit)["Ow"]))   # mOw as Frame::UpdatePoseMatrices computes it
    port = O.port_is_in_frustum(F, P, Tcw, Ow, K, 40.0, limit)
    assert port["count"] > 100
    ref.expect({f: port[f] for f in fields}, _live(O, lambda: {f: v for f, v in O.ref_is_in_frustum(F, P, Tcw, K, 40.0, limit).items() if f in fields}))


TUM1_K = (517.306408, 516.469215, 318.643040, 255.313989)
TUM1_DIST = (0.262383, -0.953104, -0.005358, 0.002628, 1.163314)


def _synthetic_depth(seed, w=640, h=480):
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:h, 0:w]
    raw = (5000.0 * (1.5 + 0.8 * np.sin(xx / 90.0) * np.cos(yy / 70.0))).astype(np.uint16)
    raw[rng.random((h, w)) < 0.15] = 0                       # holes of the depth sensor
    return raw


@pytest.mark.parametrize("dist", [TUM1_DIST, TUM1_DIST[:4], (0.0, 0.0, 0.0, 0.0), (-0.28, 0.07, 0.0002, 0.00002)])
def test_rgbd_leg_port_equals_reference_and_cv2(oracle, dist, ref):
    """UndistortKeyPoints + ComputeStereoFromRGBD + ComputeImageBounds (src/Frame.cc:404-464, :643-664): the restatement equals the
    verbatim Frame.cc (whose cv::undistortPoints stand-in is itself pinned here against cv2 4.13) bit for bit."""
    import cv2
    from orb_slam2_b200 import synth
    E = oracle.PortExtractor(1000)
    keys, _ = E(synth.mono_frame(5, 0, 0, 640, 480))
    depth = oracle.port_depth_to_float(_synthetic_depth(3), 1.0 / 5000.0)
    assert np.array_equal(depth, _synthetic_depth(3).astype(np.float32) * np.float32(1.0 / 5000.0))
    K4 = np.array(TUM1_K, np.float32); D = np.array(dist, np.float32)
    p = oracle.port_rgbd_frame(keys, K4, D, 40.0, depth)
    ref.expect(p, _live(oracle, lambda: oracle.ref_rgbd_frame(keys, K4, D, 40.0, depth)))
    assert p["count"] > 500
    # cv2 pin of the un-vendored primitive
    Km = np.array([[K4[0], 0, K4[2]], [0, K4[1], K4[3]], [0, 0, 1]], np.float32)
    pts = np.stack([keys["x"], keys["y"]], 1).astype(np.float32).reshape(-1, 1, 2)
    if D[0] != 0:
        und = cv2.undistortPoints(pts, Km, D.reshape(-1, 1), None, Km).reshape(-1, 2)
        assert np.array_equal(und[:, 0], p["keys_un"]["x"]) and np.array_equal(und[:, 1], p["keys_un"]["y"])
        assert np.abs(und - pts.reshape(-1, 2)).max() > 0.5
        corners = cv2.undistortPoints(np.array([[[0, 0]], [[640, 0]], [[0, 480]], [[640, 480]]], np.float32), Km, D.reshape(-1, 1), None, Km).reshape(4, 2)
        want = [min(corners[0, 0], corners[2, 0]), min(corners[0, 1], corners[1, 1]), max(corners[1, 0], corners[3, 0]), max(corners[2, 1], corners[3, 1])]
        assert np.array_equal(p["bounds"], np.array(want, np.float32))
    else:
        assert np.array_equal(p["keys_un"], keys) and np.array_equal(p["bounds"], np.array([0, 0, 640, 480], np.float32))
    # depth association semantics: truncating (v, u) lookup on the DISTORTED keypoint, uRight from the undistorted x
    i = int(np.nonzero(p["depth"] > 0)[0][0])
    assert p["depth"][i] == depth[int(keys["y"][i]), int(keys["x"][i])]
    assert p["u_right"][i] == np.float32(p["keys_un"]["x"][i] - np.float32(40.0) / p["depth"][i])
    assert np.all(p["u_right"][p["depth"] < 0] == -1)
