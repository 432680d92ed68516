"""CPU: pins the vocabulary / scoring / keyframe-database restatements — and the host bookkeeping the product does around the
GPU tree descent and the GPU database query — to the REFERENCE SOURCE: DBoW2 (TemplatedVocabulary.h, FORB.cpp, ScoringObject.cpp,
BowVector.cpp, FeatureVector.cpp) and src/KeyFrameDatabase.cc compiled verbatim (oracle/_ref/libdbowref.so, oracle/dbowref_wrap.cpp).
Where that build is absent, the results it gave are taken from tests/golden/reference.json (tests/reference_golden.py)."""
import numpy as np
import pytest

from tests import match_fixtures as mf
from tests.reference_golden import Reference, ref  # noqa: F401  (fixture)


def _live(world, fn):
    """fn on the reference-side library where it is built, else None (the stored results stand in)."""
    return fn if world["rv"] is not None else None


@pytest.fixture(scope="module")
def world(oracle, tmp_path_factory):
    pv = oracle.PortVocabulary.random(10, 3, 5)
    path = tmp_path_factory.mktemp("voc") / "voc.txt"
    pv.save_text(str(path))
    text = path.read_text()
    # The reference's loader loops `while(!f.eof()) getline(...)` (TemplatedVocabulary.h:1379-1420): a file that ends in a newline —
    # ORBvoc.txt does — makes it parse one more, empty, line into a bogus extra child of the root whose leaf flag, weight and
    # descriptor are whatever the previous iteration / the allocator left behind (undefined behaviour; see DESIGN.md §2).  The
    # pin below uses a file without the trailing newline, where the reference is well defined.
    path.write_text(text.rstrip("\n"))
    rv = oracle.RefVocabulary(path) if oracle.have_dbowref() else None   # the reference's own loadFromTextFile reads the file the port wrote
    with_nl = tmp_path_factory.mktemp("voc") / "voc_nl.txt"
    with_nl.write_text(text if text.endswith("\n") else text + "\n")
    return dict(O=oracle, pv=pv, rv=rv, v=mf.two_views(oracle, 7), with_nl=with_nl)


def test_reference_loader_trailing_newline_quirk(world, ref):
    """Documents the quirk: the same vocabulary with a trailing newline gains a node in the reference's loader."""
    assert ref.value(_live(world, lambda: world["rv"].words)) == 1000
    if world["rv"] is not None:
        rv2 = world["O"].RefVocabulary(world["with_nl"])
        assert rv2.words in (1000, 1001)        # 1001 when the stale leaf flag happens to be set


@pytest.mark.parametrize("levelsup", [1, 2, 3, 0])
def test_transform_equals_reference_dbow2(world, levelsup, ref):
    from orb_slam2_b200.matcher import bow_and_featvec
    O, pv, rv, v = world["O"], world["pv"], world["rv"], world["v"]
    assert rv is None or rv.words == 1000
    for d in (v["dl"], v["dr"][:137], v["dl"][:1]):
        bow_p, fv_p = bow_and_featvec(*pv.transform_raw(d, levelsup))
        words, values = np.fromiter(bow_p.keys(), np.uint32), np.fromiter(bow_p.values(), np.float64)   # bit-identical doubles
        ref.expect((words, values, fv_p.node_id, fv_p.start, fv_p.feat_idx),
                   _live(world, lambda: (lambda b, n, s, i: (np.fromiter(b.keys(), np.uint32), np.fromiter(b.values(), np.float64), n, s, i))(*rv.transform(d, levelsup))))
        assert abs(sum(bow_p.values()) - 1.0) < 1e-9


def test_l1_score_equals_reference_dbow2(world, ref):
    O, pv, rv, v = world["O"], world["pv"], world["rv"], world["v"]
    from orb_slam2_b200.matcher import bow_and_featvec
    rng = np.random.default_rng(3)
    bows = [bow_and_featvec(*pv.transform_raw(v["dl"][rng.choice(len(v["dl"]), 400, replace=False)], 2))[0] for _ in range(12)]
    bows.append({})
    ref.expect([O.port_bow_score(a, b)[0] for a in bows[:6] for b in bows],                     # identical doubles
               _live(world, lambda: [rv.score(a, b) for a in bows[:6] for b in bows]))


def test_keyframe_database_equals_reference_source(world, ref):
    """KeyFrameDatabase::add + DetectRelocalizationCandidates / DetectLoopCandidates of the reference source vs (i) the restatements
    with their own inverted file and (ii) the product's host logic fed with per-keyframe counts and scores."""
    from orb_slam2_b200 import matcher as M
    O, rv = world["O"], world["rv"]
    rng = np.random.default_rng(12)
    n_words, n_kf = 1000, 60
    assert rv is None or rv.words == n_words
    centers = [rng.choice(n_words, 90, replace=False) for _ in range(6)]

    def bow_near(c):
        keep = centers[c][rng.random(90) < 0.8]
        w = np.unique(np.concatenate([keep, rng.choice(n_words, 25, replace=False)]))
        val = rng.random(len(w)); val /= val.sum()
        return dict(zip(w.tolist(), val.tolist()))
    place = rng.integers(0, 6, n_kf)
    bows = [bow_near(int(p)) for p in place]
    neigh = np.full((n_kf, 10), -1, np.int32)
    for s in range(n_kf):
        same = [int(x) for x in np.nonzero(place == place[s])[0] if x != s]
        nb = [x for x in dict.fromkeys(same[:4] + rng.integers(0, n_kf, 3).tolist()) if x != s][:10]
        neigh[s, :len(nb)] = nb
    covis = lambda s: [int(x) for x in neigh[s] if x >= 0]
    seq = list(range(n_kf))
    total = 0
    for q in [bow_near(0), bow_near(3), bows[17], {5: 1.0}]:
        per = [O.port_bow_score(q, b) for b in bows]
        sc = np.array([np.float32(p[0]) for p in per], np.float32); cw = np.array([p[1] for p in per], np.int32); fw = np.array([p[2] for p in per], np.uint32)
        want = O.port_detect_reloc_candidates(bows, n_words, q, neigh).tolist()
        ref.expect(want, _live(world, lambda: rv.detect_candidates(False, bows, q, None, neigh)))
        assert M.relocalization_candidates(cw, sc, fw, seq, covis) == want
        for min_score, conn in [(0.0, []), (0.05, [3, 17, 20]), (0.3, list(range(0, n_kf, 2)))]:
            connected = np.zeros(n_kf, np.uint8); connected[conn] = 1
            want = O.port_detect_loop_candidates(bows, n_words, q, connected, neigh, min_score).tolist()
            ref.expect(want, _live(world, lambda: rv.detect_candidates(True, bows, q, connected, neigh, min_score)))
            assert M.loop_candidates(cw, sc, fw, seq, set(conn), covis, min_score) == want
            total += len(want)
    assert total > 10


@pytest.mark.parametrize("seed", [21, 22, 23, 24])
def test_relocalization_reads_stale_scores_like_the_reference(world, seed, ref):
    """KeyFrame::mRelocScore is assigned only to keyframes above minCommonWords (src/KeyFrameDatabase.cc:236-243) but read for every
    covisible neighbour that shares a word with the query (:262-275): on a long-running database a neighbour below the threshold
    contributes the score an EARLIER query left there.  The product keeps that field per slot (KeyFrameDatabase._reloc_score);
    a sequence of queries through the verbatim reference (one database, persistent KeyFrame objects) must give the same lists,
    and the sequence must differ somewhere from what a fresh database returns for the same query (otherwise the case is vacuous)."""
    from orb_slam2_b200 import matcher as M
    O, rv = world["O"], world["rv"]
    rng = np.random.default_rng(seed)
    n_words, n_kf = 1000, 80
    assert rv is None or rv.words == n_words
    centers = [rng.choice(n_words, 120, replace=False) for _ in range(5)]

    def bow_near(c, keep_p):
        keep = centers[c][rng.random(120) < keep_p]
        w = np.unique(np.concatenate([keep, rng.choice(n_words, 20, replace=False)]))
        val = rng.random(len(w)); val /= val.sum()
        return dict(zip(w.tolist(), val.tolist()))
    place = rng.integers(0, 5, n_kf)
    # keyframes share between 35 % and 95 % of their place's words: plenty of neighbours end up BELOW 0.8 x maxCommonWords
    bows = [bow_near(int(p), float(rng.uniform(0.35, 0.95))) for p in place]
    neigh = np.full((n_kf, 10), -1, np.int32)
    for s in range(n_kf):
        same = [int(x) for x in rng.permutation(np.nonzero(place == place[s])[0]) if x != s]
        nb = [x for x in dict.fromkeys(same[:8] + rng.integers(0, n_kf, 2).tolist()) if x != s][:10]
        neigh[s, :len(nb)] = nb
    covis = lambda s: [int(x) for x in neigh[s] if x >= 0]
    seq = list(range(n_kf))
    queries = [bow_near(int(c), float(kp)) for c, kp in zip(rng.integers(0, 5, 14), rng.uniform(0.5, 0.95, 14))]
    state = {}
    got_seq, differs_from_fresh = [], 0
    for q in queries:
        per = [O.port_bow_score(q, b) for b in bows]
        sc = np.array([np.float32(p[0]) for p in per], np.float32); cw = np.array([p[1] for p in per], np.int32); fw = np.array([p[2] for p in per], np.uint32)
        got_seq.append(M.relocalization_candidates(cw, sc, fw, seq, covis, state))
        differs_from_fresh += M.relocalization_candidates(cw, sc, fw, seq, covis) != got_seq[-1]
    ref.expect(got_seq, _live(world, lambda: rv.reloc_sequence(bows, queries, neigh)))
    assert sum(len(r) for r in got_seq) > 10
    if seed == 21:
        assert differs_from_fresh > 0, "no query of the sequence depended on a stale mRelocScore: strengthen the fixture"
