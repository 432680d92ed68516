"""CPU: the oracle (restatement AND verbatim reference build) reproduces the committed golden vectors.  Where the verbatim build
is absent, what it gave is taken from tests/golden/reference.json (tests/reference_golden.py)."""
import glob
import os

import numpy as np
import pytest

from orb_slam2_b200 import synth
from tests.reference_golden import ref  # noqa: F401  (fixture)

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def golden_extract_cases():
    return sorted(glob.glob(os.path.join(GOLD, "extract_*.npz")))


@pytest.mark.parametrize("path", golden_extract_cases(), ids=os.path.basename)
def test_port_reproduces_golden(oracle, path):
    g = np.load(path)
    w, h, nf, ini, mn, seed = g["meta"].tolist()
    img = synth.mono_frame(seed, 0, 0, w, h)
    k, d = oracle.PortExtractor(nf, 1.2, 8, ini, mn)(img)
    assert np.array_equal(k, g["keypoints"]) and np.array_equal(d, g["descriptors"])


@pytest.mark.parametrize("path", golden_extract_cases()[:2], ids=os.path.basename)
def test_verbatim_reference_reproduces_golden(oracle, path, ref):
    g = np.load(path)
    w, h, nf, ini, mn, seed = g["meta"].tolist()
    img = synth.mono_frame(seed, 0, 0, w, h)
    ref.expect((g["keypoints"], g["descriptors"]), (lambda: oracle.RefExtractor(nf, 1.2, 8, ini, mn)(img)) if oracle.have_ref() else None)


def test_stereo_restatement_reproduces_golden(oracle):
    g = np.load(os.path.join(GOLD, "stereo_kitti_2000.npz"))
    w, h, nf, seed = g["meta"].tolist()
    bf, fx = g["cam"].tolist()
    L, R, disp = synth.stereo_pair(seed, 0, 0, w, h)
    EL, ER = oracle.PortExtractor(nf), oracle.PortExtractor(nf)
    kl, dl = EL(L)
    kr, dr = ER(R)
    assert np.array_equal(kl, g["kl"]) and np.array_equal(kr, g["kr"])
    ur, dp, _ = oracle.port_stereo(kl, dl, kr, dr, [EL.level(i) for i in range(8)], [ER.level(i) for i in range(8)],
                                   EL.scale, EL.inv_scale, bf, fx)
    assert np.array_equal(ur, g["u_right"]) and np.array_equal(dp, g["depth"])
    # sanity of the restatement itself: recovered disparities follow the synthetic ground truth
    m = ur >= 0
    assert m.sum() > 800
    truth = disp[np.clip(kl["y"][m].astype(int), 0, h - 1), np.clip(np.rint(ur[m]).astype(int), 0, w - 1)]
    assert np.median(np.abs((kl["x"][m] - ur[m]) - truth)) < 1.0
    assert np.all(dp[m] > 0) and np.all(dp[~m] == -1) and np.all(ur[~m] == -1)


def test_stereo_golden_equals_verbatim_frame_cc(oracle, ref):
    """The stereo golden vectors were generated with the restatement; the reference's own Frame.cc, compiled verbatim
    (oracle/_ref/libframeref.so), produces exactly the same numbers on the same inputs."""
    g = np.load(os.path.join(GOLD, "stereo_kitti_2000.npz"))
    w, h, nf, seed = g["meta"].tolist()
    bf, fx = g["cam"].tolist()
    L, R, _ = synth.stereo_pair(seed, 0, 0, w, h)
    EL, ER = oracle.PortExtractor(nf), oracle.PortExtractor(nf)
    kl, dl = EL(L)
    kr, dr = ER(R)
    live = lambda: oracle.ref_stereo(kl, dl, kr, dr, [EL.level(i) for i in range(8)], [ER.level(i) for i in range(8)], EL.scale, EL.inv_scale, bf, fx)
    ref.expect((g["u_right"], g["depth"]), live if oracle.have_frameref() else None)


# ---- matcher golden vectors: outputs of the verbatim-compiled src/ORBmatcher.cc (tests/golden/make_golden_match.py)
from tests.golden_match_cases import CASES, flatten          # noqa: E402


@pytest.mark.parametrize("name", sorted(CASES))
def test_matcher_restatement_reproduces_golden(oracle, name):
    g = np.load(os.path.join(GOLD, "match_ref.npz"))
    build, port, _gpu = CASES[name]
    assert np.array_equal(flatten(port(oracle, build(oracle))), g[name])


def test_gpu_side_of_the_golden_cases_binds_to_the_product_api(oracle):
    """The `gpu` half of every golden case (run on the B200 by tests/test_gpu_match.py) is exercised here without a GPU: a
    stand-in ORBmatcher checks each call against the real method's signature (inspect.signature(...).bind) and answers with the
    restatement, so a mistake in the call plumbing cannot hide until the GPU run."""
    import inspect
    from orb_slam2_b200 import matcher as RealM

    class FakeMatcher:
        def __init__(self, nnratio=0.6, checkOri=True, device=0):
            inspect.signature(RealM.ORBmatcher.__init__).bind(self, nnratio, checkOri)
            self.r, self.o = nnratio, checkOri

        def _bind(self, meth, *a, **k):
            inspect.signature(getattr(RealM.ORBmatcher, meth)).bind(self, *a, **k)

        def SearchByProjection(self, *a, **k):
            self._bind("SearchByProjection", *a, **k); F, mps, th = a
            return oracle.port_search_by_projection(F, mps, th, self.r)

        def SearchByProjectionLast(self, *a, **k):
            self._bind("SearchByProjectionLast", *a, **k); Cur, Last, Tcw, K, bf, th, fw, bw = a
            return oracle.port_search_by_projection_last(Cur, Last, Tcw, K, bf, th, fw, bw, self.o)

        def SearchByProjectionKF(self, *a, **k):
            self._bind("SearchByProjectionKF", *a, **k); Cur, P, Tcw, Ow, K, th, od = a
            return oracle.port_search_by_projection_kf(Cur, P, Tcw, Ow, K, th, od, self.o)

        def SearchByProjectionSim3(self, *a, **k):
            self._bind("SearchByProjectionSim3", *a, **k); KF, P, Tcw, Ow, K, th = a
            return oracle.port_search_by_projection_sim3(KF, P, Tcw, Ow, K, th)

        def SearchByBoW(self, *a, **k):
            self._bind("SearchByBoW", *a, **k)
            return oracle.port_search_by_bow(a[0], a[1], self.r, self.o)

        def SearchByBoW_KF(self, *a, **k):
            self._bind("SearchByBoW_KF", *a, **k)
            return oracle.port_search_by_bow_kf(a[0], a[1], self.r, self.o)

        def SearchForTriangulation(self, *a, **k):
            self._bind("SearchForTriangulation", *a, **k); kf1, kf2, F12, epi = a
            return oracle.port_search_for_triangulation(kf1, kf2, F12, epi, False, self.o)

        def SearchForInitialization(self, *a, **k):
            self._bind("SearchForInitialization", *a, **k); F1, F2, prev, win = a
            return oracle.port_search_for_initialization(F1, F2, prev, win, self.r, self.o)

        def SearchBySim3(self, *a, **k):
            self._bind("SearchBySim3", *a, **k)
            return oracle.port_search_by_sim3(*a)

        def Fuse(self, *a, **k):
            self._bind("Fuse", *a, **k); KF, P, Tcw, Ow, K, bf, th = a
            return oracle.port_fuse(KF, P, Tcw, Ow, K, bf, th, k.get("Scw", False))

    class FakeM:
        ORBmatcher = FakeMatcher

    g = np.load(os.path.join(GOLD, "match_ref.npz"))
    for name, (build, _port, gpu) in CASES.items():
        assert np.array_equal(flatten(gpu(FakeM, build(oracle))), g[name]), name
