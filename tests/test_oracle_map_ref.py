"""CPU: pins MapPoint::PredictScale (both overloads), the *DistanceInvariance getters and ComputeDistinctiveDescriptors of the
restatements to the REFERENCE SOURCE: /root/reference/src/MapPoint.cc compiled verbatim against the reference's real
include/MapPoint.h (oracle/_ref/libmapref.so, oracle/mapref_wrap.cpp, oracle/mapshim/pre.hpp).  Where that build is absent, the
results it gave are taken from tests/golden/reference.json (tests/reference_golden.py)."""
import ctypes as C

import numpy as np
import pytest

from tests import match_fixtures as mf
from tests.reference_golden import ref  # noqa: F401  (fixture)


@pytest.fixture(scope="module")
def O(oracle):
    return oracle


def _live(O, fn):
    """fn on the reference-side library where it is built, else None (the stored results stand in)."""
    return fn if O.have_mapref() else None


def _logf(x):
    libm = C.CDLL("libm.so.6"); libm.logf.restype = C.c_float; libm.logf.argtypes = [C.c_float]
    return float(libm.logf(float(np.float32(x))))


@pytest.mark.parametrize("sf,nl", [(1.2, 8), (1.5, 4), (1.1, 12), (2.0, 3)])
def test_predict_scale_equals_reference_source(O, sf, nl, ref):
    rng = np.random.default_rng(int(sf * 10) + nl)
    logs = _logf(sf)
    n = 200000
    maxd = rng.uniform(0.5, 60.0, n).astype(np.float32)
    # distances spread over the whole pyramid and beyond, plus exact level boundaries (ratio = sf^k) where ceil() is touchy
    dist = (maxd / np.float32(sf) ** rng.uniform(-2.0, nl + 2.0, n)).astype(np.float32)
    k = rng.integers(0, nl, n // 10)
    dist[: n // 10] = (maxd[: n // 10] / (np.float32(sf) ** k.astype(np.float32))).astype(np.float32)
    port = O.port_predict_scale(maxd, dist, logs, nl)
    ref.expect(port, _live(O, lambda: O.ref_predict_scale(maxd, dist, logs, nl, use_frame=False)))     # PredictScale(dist, KeyFrame*)
    ref.expect(port, _live(O, lambda: O.ref_predict_scale(maxd, dist, logs, nl, use_frame=True)))      # PredictScale(dist, Frame*)
    assert set(np.unique(port).tolist()) == set(range(nl))


def test_distance_invariance_getters(O, ref):
    rng = np.random.default_rng(1)
    mx = rng.uniform(0.1, 100, 10000).astype(np.float32); mn = rng.uniform(0.01, 50, 10000).astype(np.float32)
    ref.expect((np.float32(1.2) * mx, np.float32(0.8) * mn), _live(O, lambda: O.ref_distance_invariance(mx, mn)))


def test_distinctive_descriptor_equals_reference_source(O, ref):
    d = mf.two_views(O, 7)["dl"]
    rng = np.random.default_rng(5)
    for n in [1, 2, 3, 4, 5, 8, 13, 33, 64, 100, 257]:
        base = d[rng.integers(0, len(d))]
        g = np.repeat(base[None], n, 0).copy()
        for i in range(n):
            for bit in rng.integers(0, 256, rng.integers(0, 12)):
                g[i, bit >> 3] ^= np.uint8(1 << (bit & 7))
        idx = O.port_distinctive_descriptor(g)
        assert idx >= 0, n
        ref.expect(g[idx], _live(O, lambda: O.ref_distinctive_descriptor(g)))
    g = d[rng.integers(0, len(d), 40)]
    ref.expect(g[O.port_distinctive_descriptor(g)], _live(O, lambda: O.ref_distinctive_descriptor(g)))
    # bad keyframes are left out (:263-267): equivalent to restating on the remaining descriptors
    bad = (rng.random(40) < 0.3).astype(np.uint8)
    keep = g[bad == 0]
    ref.expect(keep[O.port_distinctive_descriptor(keep)], _live(O, lambda: O.ref_distinctive_descriptor(g, bad)))
    assert O.port_distinctive_descriptor(g[:0]) == -1
    ref.expect(None, _live(O, lambda: O.ref_distinctive_descriptor(g[:0])))
