"""CPU: pins the matcher restatements of oracle/orb_port_match.cpp — and through them the CUDA kernels, which the gpu-marked
tests compare with those restatements bit for bit — to the REFERENCE SOURCE: /root/reference/src/ORBmatcher.cc compiled
verbatim (oracle/_ref/libmatchref.so; oracle/Makefile target `ref`, oracle/matchref_wrap.cpp) against plain-data stand-ins of
Frame / KeyFrame / MapPoint.  Every Search* / Fuse method of include/ORBmatcher.h is covered.  What the stand-ins restate
rather than compile (the 64x48 grid query, PredictScale, cv::Mat 3x3 arithmetic) is listed in oracle/matchshim/ORBmatcher.h.
Where that build is absent, the results it gave are taken from tests/golden/reference.json (tests/reference_golden.py)."""
import numpy as np
import pytest

from tests import match_fixtures as mf
from tests.reference_golden import ref  # noqa: F401  (fixture)


@pytest.fixture(scope="module")
def O(oracle):
    return oracle


def _live(O, fn):
    """fn on the reference-side library where it is built, else None (the stored results stand in)."""
    return fn if O.have_matchref() else None


@pytest.fixture(scope="module")
def views(oracle):
    return {s: mf.two_views(oracle, s) for s in (7, 8)}


def test_descriptor_distance(O, views, ref):
    d = views[7]["dl"]
    rng = np.random.default_rng(0)
    pairs = [(d[rng.integers(0, len(d))], d[rng.integers(0, len(d))]) for _ in range(200)]
    ref.expect([int(np.unpackbits(a ^ b).sum()) for a, b in pairs], _live(O, lambda: [O.ref_descriptor_distance(a, b) for a, b in pairs]))


@pytest.mark.parametrize("seed", [7, 8])
@pytest.mark.parametrize("th,ratio", [(1.0, 0.8), (3.0, 0.8), (5.0, 0.9)])
def test_search_by_projection_local_map(O, views, seed, th, ratio, ref):
    F, mps = mf.projection_case(views[seed], seed + 10, n_mp=400)
    n_p, m_p = O.port_search_by_projection(F, mps, th, ratio)
    assert n_p > 30
    ref.expect((n_p, O.owner_from_matches(F, mps, m_p)), _live(O, lambda: O.ref_search_by_projection(F, mps, th, ratio)))


@pytest.mark.parametrize("seed", [7, 8])
@pytest.mark.parametrize("mono,mb", [(True, 0.08), (False, 0.08), (False, 100.0)])
@pytest.mark.parametrize("th,ori", [(7.0, True), (15.0, True), (15.0, False)])
def test_search_by_projection_last_frame(O, views, seed, mono, mb, th, ori, ref):
    Cur, Last, Tcw, K = mf.last_frame_case(views[seed], seed + 20)
    # a last-frame pose that puts the camera motion along +z (forward), -z (backward) or makes it irrelevant (mono / huge mb)
    for dz in (0.5, -0.5):
        TcwLast = np.array(Tcw, np.float32).copy(); TcwLast[2, 3] += np.float32(dz)
        fw, bw = ref.value(_live(O, lambda: O.ref_forward_backward(Tcw, TcwLast, mb, mono)))
        n_p, s_p = O.port_search_by_projection_last(Cur, Last, Tcw, K, 40.0, th, fw, bw, ori)
        assert n_p > 10
        ref.expect((n_p, O.owner_from_state(Cur.occupied, s_p)),
                   _live(O, lambda: O.ref_search_by_projection_last(Cur, Last, Tcw, TcwLast, K, 40.0, mb, th, mono, ori)))
    assert (fw, bw) != (False, False) or mono or mb > 1


@pytest.mark.parametrize("seed", [7, 8])
@pytest.mark.parametrize("th,orb_dist,ori", [(10.0, 100, True), (3.0, 64, True), (10.0, 100, False), (25.0, 50, True)])
def test_search_by_projection_keyframe(O, views, seed, th, orb_dist, ori, ref):
    Cur, P, Tcw, _, K = mf.world_points_case(views[seed], seed + 30)
    Ow = ref.value(_live(O, lambda: O.ref_camera_center(Tcw)))        # -Rcw.t()*tcw as the reference evaluates it (:1478)
    n_p, s_p = O.port_search_by_projection_kf(Cur, P, Tcw, Ow, K, th, orb_dist, ori)
    assert n_p > 20
    ref.expect((n_p, O.owner_from_state(Cur.occupied, s_p)), _live(O, lambda: O.ref_search_by_projection_kf(Cur, P, Tcw, K, th, orb_dist, ori)))


@pytest.mark.parametrize("seed", [7, 8])
@pytest.mark.parametrize("th,scale", [(3, 1.0), (10, 1.0), (25, 1.7), (10, 0.6)])
def test_search_by_projection_sim3(O, views, seed, th, scale, ref):
    KF, P, Tcw, _, K = mf.world_points_case(views[seed], seed + 40)
    Scw = (np.float32(scale) * np.asarray(Tcw, np.float32)).astype(np.float32)     # [s*R | s*t]
    T, Ow = ref.value(_live(O, lambda: O.ref_decompose_scw(Scw)))    # :298-303 evaluated by the reference-side arithmetic
    n_p, s_p = O.port_search_by_projection_sim3(KF, P, T, Ow, K, th)
    assert n_p > 20
    ref.expect((n_p, O.owner_from_state(KF.occupied, s_p)), _live(O, lambda: O.ref_search_by_projection_sim3(KF, P, Scw, K, th)))


@pytest.mark.parametrize("seed", [7, 8])
@pytest.mark.parametrize("ratio,ori", [(0.7, True), (0.9, True), (0.75, False)])
def test_search_by_bow_both(O, views, seed, ratio, ori, ref):
    voc = O.PortVocabulary.random(10, 4, 5)
    kf1, kf2 = mf.keyframe_views(views[seed], voc, seed + 1)
    n_p, m_p = O.port_search_by_bow(kf1, kf2, ratio, ori)
    assert n_p > 20
    ref.expect((n_p, m_p), _live(O, lambda: O.ref_search_by_bow(kf1, kf2, ratio, ori)))
    n_p, m_p = O.port_search_by_bow_kf(kf1, kf2, ratio, ori)
    assert n_p > 10
    ref.expect((n_p, m_p), _live(O, lambda: O.ref_search_by_bow_kf(kf1, kf2, ratio, ori)))


@pytest.mark.parametrize("seed", [7, 8])
@pytest.mark.parametrize("only_stereo,ori", [(False, True), (True, True), (False, False)])
def test_search_for_triangulation(O, views, seed, only_stereo, ori, ref):
    voc = O.PortVocabulary.random(10, 4, 5)
    kf1, kf2 = mf.keyframe_views(views[seed], voc, seed + 2, mp_frac=0.4)
    F12 = mf.rectified_F12(seed)
    K2 = (525.0, 525.0, 319.5, 239.5)
    Ow1 = np.array([0.3, -0.05, -2.0], np.float32)                    # camera 1 behind camera 2: the epipole falls inside the image
    T2w = np.eye(4, dtype=np.float32)[:3]
    ex, ey = ref.value(_live(O, lambda: O.ref_epipole(Ow1, T2w, K2)))   # :663-670 evaluated by the reference-side arithmetic
    pairs_p = O.port_search_for_triangulation(kf1, kf2, F12, (ex, ey), only_stereo, ori)
    assert len(pairs_p) > 5
    ref.expect(pairs_p, _live(O, lambda: O.ref_search_for_triangulation(kf1, kf2, F12, Ow1, T2w, K2, only_stereo, ori)))


@pytest.mark.parametrize("seed", [7, 8])
@pytest.mark.parametrize("window,ratio,ori", [(100, 0.9, True), (30, 0.9, True), (100, 0.7, False)])
def test_search_for_initialization(O, views, seed, window, ratio, ori, ref):
    from orb_slam2_b200.matcher import FrameView
    v = views[seed]
    b = (0.0, 0.0, float(v["w"]), float(v["h"]))
    F1, F2 = FrameView(v["kl"], v["dl"], v["scale"], b), FrameView(v["kr"], v["dr"], v["scale"], b)
    prev = np.stack([v["kl"]["x"], v["kl"]["y"]], 1).astype(np.float32)
    n_p, m_p, p_p = O.port_search_for_initialization(F1, F2, prev, window, ratio, ori)
    assert n_p > 5
    ref.expect((n_p, m_p, p_p), _live(O, lambda: O.ref_search_for_initialization(F1, F2, prev, window, ratio, ori)))


@pytest.mark.parametrize("seed", [7, 8])
@pytest.mark.parametrize("th", [7.5, 3.0, 15.0])
def test_search_by_sim3(O, views, seed, th, ref):
    KF1, KF2, P1, P2, T1w, T2w, _, _, K = mf.sim3_case(views[seed], seed + 60)
    s12 = np.float32(1.03)
    a = 0.004
    R12 = np.array([[np.cos(a), -np.sin(a), 0], [np.sin(a), np.cos(a), 0], [0, 0, 1]], np.float32)
    t12 = np.array([0.4, 0.01, -0.02], np.float32)
    S12, S21 = ref.value(_live(O, lambda: O.ref_sim3_mats(s12, R12, t12)))   # :1119-1122 evaluated by the reference-side arithmetic
    n_p, m_p = O.port_search_by_sim3(KF1, KF2, P1, P2, T1w, T2w, S12, S21, K, th)
    assert n_p > 20
    ref.expect((n_p, m_p), _live(O, lambda: O.ref_search_by_sim3(KF1, KF2, P1, P2, T1w, T2w, s12, R12, t12, K, th)))


@pytest.mark.parametrize("seed", [7, 8])
@pytest.mark.parametrize("th", [3.0, 6.0])
def test_fuse_both(O, views, seed, th, ref):
    KF, P, Tcw, _, K, bf = mf.fuse_case(views[seed], seed + 50)
    Ow = ref.value(_live(O, lambda: O.ref_camera_center(Tcw)))
    n_p, b_p = O.port_fuse(KF, P, Tcw, Ow, K, bf, th, False)
    assert n_p > 20
    ref.expect((n_p, b_p), _live(O, lambda: O.ref_fuse(KF, P, Tcw, Ow, K, bf, th, False)))
    Scw = (np.float32(1.4) * np.asarray(Tcw, np.float32)).astype(np.float32)
    T, Ow2 = ref.value(_live(O, lambda: O.ref_decompose_scw(Scw)))
    n_p, b_p = O.port_fuse(KF, P, T, Ow2, K, bf, th, True)
    assert n_p > 20
    ref.expect((n_p, b_p), _live(O, lambda: O.ref_fuse(KF, P, Scw, Ow2, K, bf, th, True)))
