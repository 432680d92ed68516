"""CPU: the C++ adapters (reference class signatures) compile and link against libborb.so.  OpenCV C++ is
not installed here, so the compile check uses the oracle's cv shim purely as a header stand-in."""
import os
import subprocess
import textwrap

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

PROG = textwrap.dedent(r'''
    #include <opencv2/core/core.hpp>
    #include "borb_adapters.hpp"
    #include <cstdio>
    int main() {
        try {
            ORB_SLAM2::ORBextractor L(2000, 1.2f, 8, 20, 7), R(2000, 1.2f, 8, 20, 7);
            cv::Mat im(375, 1242, CV_8UC1), desc;
            std::vector<cv::KeyPoint> kps;
            L(im, cv::Mat(), kps, desc);
            std::vector<float> ur, dp;
            borb::ComputeStereoMatches(L, R, 386.1448f, 0.537f, (int)kps.size(), ur, dp);
            std::printf("levels %d\n", L.GetLevels());
        } catch (const std::exception& e) { std::printf("error: %s\n", e.what()); return 3; }
        return 0;
    }
''')


def test_adapters_compile_and_link(tmp_path):
    import __graft_entry__ as g
    so = os.path.join(ROOT, "orb_slam2_b200", "libborb.so")
    if not os.path.exists(so):
        g.build()
    src = tmp_path / "adapter_check.cpp"
    src.write_text(PROG)
    exe = tmp_path / "adapter_check"
    cmd = ["g++", "-std=c++17", "-I", os.path.join(ROOT, "include"), "-I", os.path.join(ROOT, "oracle", "cvshim"),
           str(src), "-o", str(exe), so, f"-Wl,-rpath,{os.path.dirname(so)}"]
    subprocess.check_call(cmd)
    r = subprocess.run([str(exe)], capture_output=True, text=True)
    # without a GPU the adapter must surface the library's error (no CPU fallback), with one it runs
    assert r.returncode in (0, 3), r
    if r.returncode == 3:
        assert "no CUDA device" in r.stdout or "no CPU path" in r.stdout or "CUDA" in r.stdout, r.stdout


def test_matcher_adapter_library_builds_and_exports_the_reference_entry_points():
    """integration/ORBmatcher_borb.cc (every ORBmatcher method through include/borb_matcher_adapters.hpp) compiles against the
    oracle's Frame / KeyFrame / MapPoint stand-ins and links libborb.so: oracle/libadaptmatch.so exports the same entry
    points as the verbatim libmatchref.so.  It is EXECUTED on the GPU by tests/test_gpu_adapters.py."""
    import ctypes
    from oracle import oracle_lib as O
    O.build()
    so = os.path.join(ROOT, "oracle", "libadaptmatch.so")
    lib = ctypes.CDLL(so)
    for name in ("matchref_search_by_projection", "matchref_search_by_projection_last", "matchref_search_by_projection_kf",
                 "matchref_search_by_projection_sim3", "matchref_search_by_bow_kf_f", "matchref_search_by_bow_kf_kf",
                 "matchref_search_for_triangulation", "matchref_search_for_initialization", "matchref_search_by_sim3", "matchref_fuse",
                 "matchref_descriptor_distance"):
        assert hasattr(lib, name), name
    # the adapter library depends on the product, not on the reference's matcher
    deps = subprocess.run(["ldd", so], capture_output=True, text=True).stdout
    assert "libborb.so" in deps


def test_keyframe_database_adapter_library_builds_and_fails_loudly_without_a_gpu():
    """integration/KeyFrameDatabase_borb.cc behind the reference's unchanged include/KeyFrameDatabase.h compiles against the
    dbowshim stand-ins and links libborb.so (oracle/libadaptdbow.so, same entry points as the verbatim libdbowref.so).
    Executed on the GPU by tests/test_gpu_adapters.py; here: the exports, the dependency, and — on a machine without a GPU —
    that a database call surfaces the library's error instead of falling back to anything."""
    import ctypes
    from oracle import oracle_lib as O
    O.build()
    so = os.path.join(ROOT, "oracle", "libadaptdbow.so")
    lib = ctypes.CDLL(so)
    for name in ("dbowref_voc_load_text", "dbowref_transform", "dbowref_score", "dbowref_detect_candidates", "dbowref_reloc_sequence"):
        assert hasattr(lib, name), name
    deps = subprocess.run(["ldd", so], capture_output=True, text=True).stdout
    assert "libborb.so" in deps
    syms = subprocess.run(["nm", "-DC", so], capture_output=True, text=True).stdout
    assert "borb_kfdb_query" in syms and "borb_kfdb_add" in syms            # undefined here, resolved by libborb.so


KFDB_MOCKS = {
    "ORBVocabulary.h": "#pragma once\nnamespace ORB_SLAM2 { struct ORBVocabulary { unsigned size() const { return 0; } }; }\n",
    "KeyFrameDatabase.h": r'''
#pragma once
#include <list>
#include <mutex>
#include <vector>
#include "ORBVocabulary.h"
namespace ORB_SLAM2 {
class KeyFrame; class Frame;
class KeyFrameDatabase {            // the interface of include/KeyFrameDatabase.h:41-75 (a declaration has to match)
public:
    KeyFrameDatabase(const ORBVocabulary& voc);
    void add(KeyFrame* pKF);
    void erase(KeyFrame* pKF);
    void clear();
    std::vector<KeyFrame*> DetectLoopCandidates(KeyFrame* pKF, float minScore);
    std::vector<KeyFrame*> DetectRelocalizationCandidates(Frame* F);
protected:
    const ORBVocabulary* mpVoc;
    std::vector<std::list<KeyFrame*> > mvInvertedFile;
    std::mutex mMutex;
};
}
''',
    "KeyFrame.h": r'''
#pragma once
#include <map>
#include <set>
#include <vector>
#include <opencv2/core/core.hpp>
namespace DBoW2 {
typedef std::map<unsigned, double> BowVector;
typedef std::map<unsigned, std::vector<unsigned> > FeatureVector;
}
namespace ORB_SLAM2 {
struct MapPoint { bool isBad() { return false; } };
class KeyFrame {                    // the members the adapters touch, with the reference's names
public:
    long unsigned int mnId = 0, mnLoopQuery = 0, mnRelocQuery = 0;
    int mnLoopWords = 0, mnRelocWords = 0;
    float mLoopScore = 0, mRelocScore = 0;
    DBoW2::BowVector mBowVec; DBoW2::FeatureVector mFeatVec;
    int N = 0;
    std::vector<cv::KeyPoint> mvKeysUn; cv::Mat mDescriptors; std::vector<float> mvuRight, mvScaleFactors, mvLevelSigma2;
    std::vector<MapPoint*> GetMapPointMatches() { return std::vector<MapPoint*>(N, nullptr); }
    std::set<KeyFrame*> GetConnectedKeyFrames() { return std::set<KeyFrame*>(); }
    std::vector<KeyFrame*> GetBestCovisibilityKeyFrames(const int&) { return std::vector<KeyFrame*>(); }
};
}
''',
    "Frame.h": "#pragma once\n#include \"KeyFrame.h\"\nnamespace ORB_SLAM2 { class Frame { public: long unsigned int mnId = 0; DBoW2::BowVector mBowVec; }; }\n",
}


def test_keyframe_database_drop_in_compiles_with_resident_features(tmp_path):
    """integration/KeyFrameDatabase_borb.cc in its default form (keyframe features uploaded for the resident SearchByBoW) against
    headers that carry the reference's member names: syntax and template instantiation only (the GPU run uses the scoring-only
    form because the verbatim build's KeyFrame stand-in has no features)."""
    for name, text in KFDB_MOCKS.items():
        (tmp_path / name).write_text(text)
    cmd = ["g++", "-std=c++14", "-fsyntax-only", "-DBORB_ADAPTER_NO_EXTRACTOR", "-I", str(tmp_path), "-I", os.path.join(ROOT, "oracle", "cvmini"),
           "-I", os.path.join(ROOT, "include"), os.path.join(ROOT, "integration", "KeyFrameDatabase_borb.cc")]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]


def test_multistream_host_example_builds_and_fails_loudly_without_a_gpu(tmp_path):
    """integration/example_multistream_host.cc — a C++ host written against the C ABI only (batched extraction, device-resident
    frames, one batched SearchByProjection for all streams, self-checking) — compiles and links; without a GPU it must stop at the
    first library call with the library's error (exit code 3), with one it runs its self-check (verified on the B200: every point
    of every stream matched to its own feature)."""
    so = os.path.join(ROOT, "orb_slam2_b200", "libborb.so")
    exe = tmp_path / "example_host"
    subprocess.check_call(["g++", "-std=c++14", "-I", os.path.join(ROOT, "include"), os.path.join(ROOT, "integration", "example_multistream_host.cc"),
                           so, f"-Wl,-rpath,{os.path.dirname(so)}", "-o", str(exe)])
    r = subprocess.run([str(exe), "2"], capture_output=True, text=True, timeout=300)
    assert r.returncode in (0, 3), r
    if r.returncode == 3:
        assert "no CUDA device" in r.stdout or "no CPU path" in r.stdout, r.stdout
    else:
        assert r.stdout.strip().endswith("ok")
