"""GPU: the C++ adapters — the reference-side binding of the drop-in boundary — EXECUTED, not just compiled.

oracle/libadaptmatch.so = integration/ORBmatcher_borb.cc (the product's drop-in replacement of src/ORBmatcher.cc, i.e.
include/borb_matcher_adapters.hpp instantiated for every ORBmatcher method) compiled against the oracle's plain-data
Frame / KeyFrame / MapPoint stand-ins and wrapped by the SAME C wrappers (oracle/matchref_wrap.cpp) that drive the verbatim
src/ORBmatcher.cc in libmatchref.so.  Swapping the library under oracle_lib.ref_* therefore sends every call of
tests/test_oracle_match_ref.py — all eleven Search* / Fuse methods + DescriptorDistance, several parameter sets each — through
ORBmatcher -> adapter -> C ABI -> CUDA kernels -> write-back, and the results must equal the restatements that the CPU suite pins
to the reference source.  Plus: the golden vectors recorded from the verbatim reference, and the ORBextractor / stereo adapter as
a compiled C++ program."""
import os
import subprocess
import textwrap

import numpy as np
import pytest

from tests import match_fixtures as mf
from tests import test_oracle_match_ref as T
from tests.reference_golden import Reference, ref  # noqa: F401  (fixture of the re-collected tests)

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ADAPT_SO = os.path.join(ROOT, "oracle", "libadaptmatch.so")


@pytest.fixture(scope="module", params=["host_view", "resident_frame"])
def O(oracle, request):
    """host_view: the adapters pass the Frame's host arrays with every call; resident_frame: the wrapper binds a device-resident
    copy of every Frame it builds (borb::adapt::make_resident -> borb_frame_create), so the same fixtures exercise
    borb_frame_view::resident through the adapters (BORB_ADAPT_RESIDENT is read by oracle/matchref_wrap.cpp per call)."""
    assert os.path.exists(ADAPT_SO), "build() did not build oracle/libadaptmatch.so"
    saved = oracle.MATCHREF_SO
    oracle.MATCHREF_SO = ADAPT_SO                     # every oracle.ref_* matcher call now runs the ADAPTERS on the GPU
    if request.param == "resident_frame":
        os.environ["BORB_ADAPT_RESIDENT"] = "1"
    yield oracle
    os.environ.pop("BORB_ADAPT_RESIDENT", None)
    oracle.MATCHREF_SO = saved


@pytest.fixture(scope="module")
def views(oracle):
    return {s: mf.two_views(oracle, s) for s in (7, 8)}


# the reference-pinning tests, re-collected here against the adapter library
test_descriptor_distance = T.test_descriptor_distance
test_search_by_projection_local_map = T.test_search_by_projection_local_map
test_search_by_projection_last_frame = T.test_search_by_projection_last_frame
test_search_by_projection_keyframe = T.test_search_by_projection_keyframe
test_search_by_projection_sim3 = T.test_search_by_projection_sim3
test_search_by_bow_both = T.test_search_by_bow_both
test_search_for_triangulation = T.test_search_for_triangulation
test_search_for_initialization = T.test_search_for_initialization
test_search_by_sim3 = T.test_search_by_sim3
test_fuse_both = T.test_fuse_both


def test_adapters_reproduce_the_reference_golden_vectors(O):
    """tests/golden/match_ref.npz = outputs of the verbatim src/ORBmatcher.cc; the adapter library, driven through the same
    wrappers, must agree with them (the check make_golden_match.py applied to the reference when it recorded the file)."""
    from tests.golden.make_golden_match import check_against_reference
    from tests.golden_match_cases import CASES, flatten
    g = np.load(os.path.join(ROOT, "tests", "golden", "match_ref.npz"))
    direct = 0
    for name, (build, port, _gpu) in CASES.items():
        c = build(O)
        res = port(O, c)
        assert np.array_equal(flatten(res), g[name]), name          # the restatement reproduces the golden file ...
        direct += bool(check_against_reference(name, c, res))       # ... and the adapters, converted to its convention, equal it
    assert direct >= 9


EXTRACTOR_PROG = textwrap.dedent(r'''
    #include <opencv2/core/core.hpp>
    #include "borb_adapters.hpp"
    #include <cstdio>
    #include <cstdlib>
    // argv: in.bin out.bin ; in.bin = int w, int h, then left image, right image (u8)
    int main(int argc, char** argv) {
        try {
            FILE* f = std::fopen(argv[1], "rb");
            int w, h; if (std::fread(&w, 4, 1, f) != 1 || std::fread(&h, 4, 1, f) != 1) return 2;
            cv::Mat L(h, w, CV_8UC1), R(h, w, CV_8UC1);
            if (std::fread(L.data, 1, (size_t)w * h, f) != (size_t)w * h || std::fread(R.data, 1, (size_t)w * h, f) != (size_t)w * h) return 2;
            std::fclose(f);
            ORB_SLAM2::ORBextractor EL(1000, 1.2f, 8, 20, 7), ER(1000, 1.2f, 8, 20, 7);
            std::vector<cv::KeyPoint> kl, kr; cv::Mat dl, dr;
            EL(L, cv::Mat(), kl, dl); ER(R, cv::Mat(), kr, dr);
            std::vector<float> ur, dp;
            borb::ComputeStereoMatches(EL, ER, 386.1448f, 386.1448f / 718.856f, (int)kl.size(), ur, dp);
            EL.SyncPyramid();
            FILE* o = std::fopen(argv[2], "wb");
            int n = (int)kl.size(), m = (int)kr.size(), lv = EL.GetLevels();
            std::fwrite(&n, 4, 1, o); std::fwrite(&m, 4, 1, o);
            std::fwrite(kl.data(), sizeof(cv::KeyPoint), n, o); std::fwrite(kr.data(), sizeof(cv::KeyPoint), m, o);
            for (int i = 0; i < n; i++) std::fwrite(dl.ptr(i), 1, 32, o);
            for (int i = 0; i < m; i++) std::fwrite(dr.ptr(i), 1, 32, o);
            std::fwrite(ur.data(), 4, n, o); std::fwrite(dp.data(), 4, n, o);
            const cv::Mat& p3 = EL.mvImagePyramid[3];
            int pw = p3.cols, ph = p3.rows; std::fwrite(&pw, 4, 1, o); std::fwrite(&ph, 4, 1, o);
            for (int y = 0; y < ph; y++) std::fwrite(p3.ptr(y), 1, pw, o);
            std::fwrite(&lv, 4, 1, o);
            std::fclose(o);
        } catch (const std::exception& e) { std::printf("error: %s\n", e.what()); return 3; }
        return 0;
    }
''')


def test_extractor_and_stereo_adapter_program(oracle, tmp_path):
    """include/borb_adapters.hpp (ORB_SLAM2::ORBextractor with the reference's signature, SyncPyramid, borb::ComputeStereoMatches)
    compiled into a C++ program, run on the GPU, outputs equal to the oracle bit for bit."""
    from orb_slam2_b200 import synth
    from orb_slam2_b200._lib import KP_DTYPE
    so = os.path.join(ROOT, "orb_slam2_b200", "libborb.so")
    src = tmp_path / "ext_adapter.cpp"; src.write_text(EXTRACTOR_PROG)
    exe = tmp_path / "ext_adapter"
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-I", os.path.join(ROOT, "include"), "-I", os.path.join(ROOT, "oracle", "cvshim"), str(src), "-o", str(exe),
                           so, f"-Wl,-rpath,{os.path.dirname(so)}"])
    L, R, _ = synth.stereo_pair(11, 0, 0, 640, 360)
    with open(tmp_path / "in.bin", "wb") as f:
        f.write(np.array([640, 360], np.int32).tobytes()); f.write(L.tobytes()); f.write(R.tobytes())
    r = subprocess.run([str(exe), str(tmp_path / "in.bin"), str(tmp_path / "out.bin")], capture_output=True, text=True)
    assert r.returncode == 0, (r.returncode, r.stdout, r.stderr)
    raw = open(tmp_path / "out.bin", "rb").read()
    n, m = np.frombuffer(raw, np.int32, 2)
    o = 8
    kl = np.frombuffer(raw, KP_DTYPE, n, o); o += 28 * n
    kr = np.frombuffer(raw, KP_DTYPE, m, o); o += 28 * m
    dl = np.frombuffer(raw, np.uint8, 32 * n, o).reshape(n, 32); o += 32 * n
    dr = np.frombuffer(raw, np.uint8, 32 * m, o).reshape(m, 32); o += 32 * m
    ur = np.frombuffer(raw, np.float32, n, o); o += 4 * n
    dp = np.frombuffer(raw, np.float32, n, o); o += 4 * n
    pw, ph = np.frombuffer(raw, np.int32, 2, o); o += 8
    p3 = np.frombuffer(raw, np.uint8, pw * ph, o).reshape(ph, pw)
    E1, E2 = oracle.PortExtractor(1000), oracle.PortExtractor(1000)
    kl_o, dl_o = E1(L); kr_o, dr_o = E2(R)
    ur_o, dp_o, _ = oracle.port_stereo(kl_o, dl_o, kr_o, dr_o, [E1.level(i) for i in range(8)], [E2.level(i) for i in range(8)], E1.scale, E1.inv_scale, 386.1448, 718.856)
    assert np.array_equal(kl, kl_o) and np.array_equal(kr, kr_o) and np.array_equal(dl, dl_o) and np.array_equal(dr, dr_o)
    assert np.array_equal(ur, ur_o) and np.array_equal(dp, dp_o) and (ur >= 0).sum() > 200
    assert np.array_equal(p3, E1.level(3))                              # mvImagePyramid through SyncPyramid


# ---------------------------------------------------------------------------------------------------------------------------
# KeyFrameDatabase: integration/KeyFrameDatabase_borb.cc (the drop-in replacement of src/KeyFrameDatabase.cc) behind the real
# include/KeyFrameDatabase.h, wrapped by the same oracle/dbowref_wrap.cpp as the verbatim build
ADAPT_DBOW_SO = os.path.join(ROOT, "oracle", "libadaptdbow.so")


@pytest.fixture(scope="module")
def world(oracle, tmp_path_factory):
    """tests/test_oracle_dbow_ref.py's fixture with oracle.DBOWREF_SO pointing at the ADAPTER library: every
    KeyFrameDatabase::add / DetectLoopCandidates / DetectRelocalizationCandidates call of those tests now runs
    adapter -> borb_kfdb_add / borb_kfdb_query (GPU) -> the adapter's host part."""
    assert os.path.exists(ADAPT_DBOW_SO), "build() did not build oracle/libadaptdbow.so"
    saved = oracle.DBOWREF_SO
    oracle.DBOWREF_SO = ADAPT_DBOW_SO
    pv = oracle.PortVocabulary.random(10, 3, 5)
    path = tmp_path_factory.mktemp("voc") / "voc.txt"
    pv.save_text(str(path))
    path.write_text(path.read_text().rstrip("\n"))
    rv = oracle.RefVocabulary(path)                     # CDLL(ADAPT_DBOW_SO): its database entry points are the product's adapter
    yield dict(O=oracle, pv=pv, rv=rv, v=mf.two_views(oracle, 7))
    oracle.DBOWREF_SO = saved


from tests import test_oracle_dbow_ref as TD      # noqa: E402

test_keyframe_database_adapter_equals_reference_source = TD.test_keyframe_database_equals_reference_source


def test_keyframe_database_adapter_reads_stale_scores_like_the_reference(world):
    TD.test_relocalization_reads_stale_scores_like_the_reference(world, 21, Reference("test_relocalization_reads_stale_scores_like_the_reference", {"seed": 21}))
