"""The oracle's restatement (oracle/*.cpp) held against THE REFERENCE ITSELF: oracle/_ref/libref.so is the reference's own
src/ORBextractor.cc, ORBmatcher.cc, LSDmatcher.cpp, ExtractLineSegment.cpp, Frame.cc, KeyFrame.cc, MapPoint.cc, MapLine.cpp and
Thirdparty/DBoW2, compiled unmodified by oracle/ref_build.sh.  What those calls returned is recorded in tests/golden/ref_parity.npz
(tests/ref_replay.py), so the comparisons run without the reference's sources.

Bit-exact everywhere (ints, bytes, indices, and the f32 keypoint fields)."""
import os
import numpy as np
import pytest

import ref_replay


@pytest.fixture(scope="module")
def ref_store():
    store = ref_replay.Store()
    yield store
    store.save()


@pytest.fixture
def ref(ref_store, request):
    return ref_store.reference(request.node.name)


_same = ref_replay.same


# ---------------------------------------------------------------------------------------------- ORB extractor
def test_orb_tables(oracle, ref):
    """ORBextractor constructor tables (ORBextractor.cc:410-470) — SURVEY.md §4 golden constants included."""
    for nf, sc, nl in [(1000, 1.2, 8), (2000, 1.2, 8), (4000, 1.2, 8), (500, 1.5, 4), (1500, 1.1, 12)]:
        t = ref.orb_tables(nf, sc, nl)
        o = oracle.OrbOracle(nf, sc, nl, 20, 7).tables()
        for key in ("scale", "invscale", "sigma2", "invsigma2", "nfeat", "umax"):
            assert np.array_equal(t[key], o[key]), (nf, sc, nl, key)
    assert list(ref.orb_tables(1000)["nfeat"]) == [217, 181, 151, 126, 105, 87, 73, 60]
    assert list(ref.orb_tables(4000)["nfeat"]) == [869, 724, 603, 503, 419, 349, 291, 242]
    assert list(ref.orb_tables(1000)["umax"]) == [15, 15, 15, 15, 14, 14, 14, 13, 13, 12, 11, 10, 9, 8, 6, 3]


def test_orb_icl_frame_known_answers(oracle, ref, icl_gray):
    """BASELINE.json config 1: the reference's ORBextractor on images/input.png — SURVEY.md §8(c) known answers reproduced by
    the reference code itself (bump allocator), and the oracle equal to it byte for byte."""
    import hashlib
    k, d, lc = ref.orb_extract(icl_gray, 1000)
    assert list(lc) == [218, 181, 151, 126, 105, 88, 73, 60] and len(k) == 1002
    ok, od = oracle.OrbOracle(1000, 1.2, 8, 20, 7).extract(icl_gray)
    assert _same(k, ok) and _same(d, od)
    # (the known answers, on the oracle's output: equal to the reference's above)
    assert hashlib.sha1(od.tobytes()).hexdigest() == "e8dce82582b67285476bbe582e3557644739a438"
    uva = np.stack([ok["x"], ok["y"], ok["angle"]], 1).astype(np.float32)
    assert hashlib.sha1(uva.tobytes()).hexdigest() == "1105debd69ac4a65f0375a9da3f130fe9fd64ca5"
    assert list(od[0]) == [176, 12, 22, 27, 144, 163, 2, 87, 84, 11, 99, 80, 66, 49, 32, 65, 81, 2, 2, 34, 49, 184, 81, 31, 36, 174, 48, 64, 72, 64, 224, 137]
    # the initialiser extractor (2 * nFeatures, Tracking.cc:120)
    k2, d2, _ = ref.orb_extract(icl_gray, 2000)
    ok2, od2 = oracle.OrbOracle(2000, 1.2, 8, 20, 7).extract(icl_gray)
    assert _same(k2, ok2) and _same(d2, od2)


@pytest.mark.parametrize("f", range(8))
def test_orb_synthetic_640(oracle, ref, synth, f):
    img = synth.frame(640, 480, f * 5)
    k, d, _ = ref.orb_extract(img, 1000)
    ok, od = oracle.OrbOracle(1000, 1.2, 8, 20, 7).extract(img)
    assert _same(k, ok) and _same(d, od) and len(k) > 900


def test_orb_1280_4000_and_other_parameters(oracle, ref, synth):
    img = synth.frame(1280, 960, 3)
    k, d, _ = ref.orb_extract(img, 4000)
    ok, od = oracle.OrbOracle(4000, 1.2, 8, 20, 7).extract(img)
    assert _same(k, ok) and _same(d, od) and len(k) > 3900
    small = synth.frame(640, 480, 2)[:241, :323]
    for nf, sc, nl, ini, mn in [(500, 1.5, 4, 30, 10), (300, 1.2, 8, 20, 7), (1500, 1.1, 6, 12, 5)]:
        k, d, _ = ref.orb_extract(small, nf, sc, nl, ini, mn)
        ok, od = oracle.OrbOracle(nf, sc, nl, ini, mn).extract(small)
        assert _same(k, ok) and _same(d, od), (nf, sc, nl)


def test_pyramid_levels(oracle, ref, icl_gray):
    """ComputePyramid (ORBextractor.cc:1107-1132): every level and its 19-px bordered view."""
    orc = oracle.OrbOracle(1000, 1.2, 8, 20, 7); orc.extract(icl_gray)
    for l in range(8):
        assert _same(ref.orb_pyramid_level(icl_gray, l, False), orc.level(l, False)), l
        assert _same(ref.orb_pyramid_level(icl_gray, l, True), orc.level(l, True)), l


def test_octree_tie_rule(oracle, ref):
    """DistributeOctTree (ORBextractor.cc:539-763) under the monotonic allocator == the oracle's (size, creation counter) key,
    on inputs full of equal-sized nodes (many equal responses, clustered points)."""
    rng = np.random.default_rng(7)
    for trial in range(60):
        n = int(rng.integers(1, 1500)); H = int(rng.integers(60, 480)); W = int(H * rng.uniform(0.6, 3.0))   # W < H/2 gives nIni = 0 and the reference indexes an empty vector (:548-569)
        if trial % 3 == 0:      # clusters => many nodes of equal size
            c = rng.integers(0, [W, H], (8, 2)); p = c[rng.integers(0, 8, n)] + rng.integers(-6, 7, (n, 2))
            xs = np.clip(p[:, 0], 0, W - 1); ys = np.clip(p[:, 1], 0, H - 1)
        else:
            xs = rng.integers(0, W, n); ys = rng.integers(0, H, n)
        resp = rng.integers(7, 12 if trial % 2 else 200, n)
        N = int(rng.integers(1, 400))
        got = ref.octree(xs, ys, resp, 0, W, 0, H, N)
        exp = oracle.octree(xs, ys, resp, 0, W, 0, H, N)
        assert _same(got, exp), trial


# ---------------------------------------------------------------------------------------------- point matchers
def _pair(oracle, synth, f0=0, nf=1000):
    orc = oracle.OrbOracle(nf, 1.2, 8, 20, 7)
    k1, d1 = orc.extract(synth.frame(640, 480, f0)); k2, d2 = orc.extract(synth.frame(640, 480, f0 + 1))
    return orc, k1, d1, k2, d2


def _fvs(oracle, synth, d1, d2, nwords):
    voc = synth.vocabulary(nwords)
    return oracle.feature_vector_csr(oracle.bow_assign(d1, voc)), oracle.feature_vector_csr(oracle.bow_assign(d2, voc))


def test_descriptor_distance(oracle, ref):
    rng = np.random.default_rng(5)
    for _ in range(200):
        a = rng.integers(0, 256, 32, dtype=np.uint8); b = rng.integers(0, 256, 32, dtype=np.uint8)
        e = oracle.descriptor_distance(a, b)
        assert ref.descriptor_distance(a, b) == e and ref.descriptor_distance(a, b, line=True) == e


@pytest.mark.parametrize("nwords,mask,ratio,ori,f0", [(100, False, 0.7, True, 0), (100, True, 0.7, True, 8), (10, True, 0.9, True, 16),
                                                       (100, True, 0.6, False, 1), (1000, True, 0.75, True, 2), (1, False, 0.7, True, 9)])
def test_search_by_bow(oracle, ref, synth, nwords, mask, ratio, ori, f0):
    """ORBmatcher::SearchByBoW(KeyFrame*, Frame&) :159-291 and (KeyFrame*, KeyFrame*) :525-658 — the parameter sets of the GPU tests."""
    _, k1, d1, k2, d2 = _pair(oracle, synth, f0)
    fv1, fv2 = _fvs(oracle, synth, d1, d2, nwords)
    rng = np.random.default_rng(99)
    valid1 = (rng.random(len(d1)) < 0.7).astype(np.uint8) if mask else np.ones(len(d1), np.uint8)
    n_o, m_o = oracle.search_by_bow(d1, d2, fv1, fv2, valid1, k1["angle"], k2["angle"], ratio, ori)
    # the reference skips BAD MapPoints exactly like missing ones (:197-200): make a third of the invalid ones bad instead of NULL
    state1 = valid1.copy(); inv = np.flatnonzero(valid1 == 0); state1[inv[::3]] = 2
    n_r, m_r = ref.search_by_bow(d1, k1, d2, k2, fv1, fv2, state1, ratio, ori)
    assert n_r == n_o and _same(m_r, m_o)
    valid2 = (rng.random(len(d2)) < 0.8).astype(np.uint8)
    n_o, m_o = oracle.search_by_bow_kf(d1, d2, fv1, fv2, valid1, valid2, k1["angle"], k2["angle"], ratio, ori)
    state2 = valid2.copy(); inv = np.flatnonzero(valid2 == 0); state2[inv[::2]] = 2
    n_r, m_r = ref.search_by_bow_kf(d1, k1, d2, k2, fv1, fv2, state1, state2, ratio, ori)
    assert n_r == n_o and _same(m_r, m_o)
    assert n_o > 10 or nwords == 1000


def test_search_by_bow_icl_shifted(oracle, ref, icl_gray, synth):
    """BASELINE.json config 3 on the ICL frame and its 2-px-shifted copy."""
    orc = oracle.OrbOracle(1000, 1.2, 8, 20, 7)
    k1, d1 = orc.extract(icl_gray); k2, d2 = orc.extract(np.roll(icl_gray, 2, axis=1))
    fv1, fv2 = _fvs(oracle, synth, d1, d2, 100)
    v = np.ones(len(d1), np.uint8)
    n_o, m_o = oracle.search_by_bow(d1, d2, fv1, fv2, v, k1["angle"], k2["angle"], 0.7, True)
    n_r, m_r = ref.search_by_bow(d1, k1, d2, k2, fv1, fv2, v, 0.7, True)
    assert n_r == n_o and _same(m_r, m_o) and n_o > 300


def _poses(rng, epi_inside):
    """Two camera poses (3x4 [R|t]) and F12 for K = CAM640; epi_inside puts the epipole of camera 1 inside image 2."""
    def rot(ax, a):
        c, s = np.cos(a), np.sin(a); R = np.eye(3); i, j = [(1, 2), (0, 2), (0, 1)][ax]
        R[i, i] = c; R[i, j] = -s; R[j, i] = s; R[j, j] = c; return R
    R1 = np.eye(3); t1 = np.zeros(3)
    R2 = rot(1, rng.uniform(-0.05, 0.05)) @ rot(0, rng.uniform(-0.03, 0.03))
    t2 = np.array([0.02, 0.01, -0.5]) if epi_inside else np.array([-0.4, 0.05, 0.02])
    K = np.array([[500, 0, 320], [0, 500, 240], [0, 0, 1.0]])
    R12 = R1 @ R2.T; t12 = -R1 @ R2.T @ t2 + t1
    tx = np.array([[0, -t12[2], t12[1]], [t12[2], 0, -t12[0]], [-t12[1], t12[0], 0]])
    F12 = np.linalg.inv(K).T @ tx @ R12 @ np.linalg.inv(K)
    T1 = np.hstack([R1, t1[:, None]]).astype(np.float32); T2 = np.hstack([R2, t2[:, None]]).astype(np.float32)
    return T1, T2, F12.astype(np.float32)


@pytest.mark.parametrize("nwords,ori,inside,f0", [(100, True, True, 0), (10, True, False, 8), (100, False, True, 3), (30, True, False, 17)])
def test_search_for_triangulation(oracle, ref, synth, nwords, ori, inside, f0):
    """ORBmatcher::SearchForTriangulation :660-826 + CheckDistEpipolarLine :140-157, epipole from the two KeyFrame poses."""
    orc, k1, d1, k2, d2 = _pair(oracle, synth, f0)
    fv1, fv2 = _fvs(oracle, synth, d1, d2, nwords)
    rng = np.random.default_rng(11 + f0)
    has1 = (rng.random(len(d1)) < 0.4).astype(np.uint8); has2 = (rng.random(len(d2)) < 0.4).astype(np.uint8)
    T1, T2, F12 = _poses(rng, inside)
    n_r, p_r, (ex, ey) = ref.search_for_triangulation(d1, k1, d2, k2, fv1, fv2, has1, has2, ref.CAM640, T1, T2, F12, ori)
    tb = orc.tables(); scale, sigma2 = tb["scale"], tb["sigma2"]
    n_o, p_o = oracle.search_for_triangulation(d1, d2, fv1, fv2, has1, has2, k1, k2, F12, ex, ey, scale, sigma2, ori)
    assert n_r == n_o and _same(p_r, p_o)
    assert (0 <= ex < 640 and 0 <= ey < 480) == inside


def test_features_in_area(oracle, ref, synth):
    """Frame::AssignFeaturesToGrid + GetFeaturesInArea (Frame.cc:133-148, :368-421)."""
    _, k1, d1, _, _ = _pair(oracle, synth, 4)
    rng = np.random.default_rng(3)
    camv = ref.CAM640
    for _ in range(60):
        x, y = rng.uniform(-20, 660), rng.uniform(-20, 500); r = rng.uniform(1, 120)
        lo, hi = (-1, -1) if rng.random() < 0.3 else (int(rng.integers(0, 5)), int(rng.integers(0, 8)))
        got = ref.features_in_area(k1, camv, x, y, r, lo, hi)
        exp = oracle.features_in_area(k1["x"], k1["y"], k1["octave"], (0, 640, 0, 480), x, y, r, lo, hi)
        assert _same(got, exp)


@pytest.mark.parametrize("seed,th,mono,ori,claimed", [(1, 15.0, True, True, 0.05), (2, 7.0, True, True, 0.0), (3, 30.0, True, False, 0.2),
                                                       (4, 15.0, False, True, 0.05), (5, 15.0, False, True, 0.0), (6, 100.0, True, True, 0.0)])
def test_search_by_projection_frame(oracle, ref, synth, seed, th, mono, ori, claimed):
    """ORBmatcher::SearchByProjection(Frame&, const Frame&, th, bMono) :1331-1473 (TrackWithMotionModel) — the scenarios of
    tests/test_projection_gpu.py, stereo ones included (forward / backward level windows, uRight test)."""
    from scenarios import projection_scenario
    last, cur, Tcw, Tlw, cam, bounds, sf = projection_scenario(oracle, synth, seed, n_claimed=claimed, stereo=not mono, f0=seed)
    n_o, a_o = oracle.search_by_projection_frame(last, cur, Tcw, Tlw, cam, bounds, sf, th, mono, ori)
    camv = ref.cam(cam[0], cam[1], cam[2], cam[3], *bounds)
    n_r, a_r = ref.search_by_projection_frame(last, cur, Tcw, Tlw, camv, 8, 1.2, th, mono, ori, mbf=cam[4])
    a_r = np.where(a_r == -2, -1, a_r)                           # -2 = the feature still holds the MapPoint it was 'claimed' with
    assert n_r == n_o and np.array_equal(a_r, a_o), (seed, n_r, n_o, int((a_r != a_o).sum()))
    assert n_o > 50 or th < 10
    if seed == 1:          # nothing valid / everything claimed / no observations (later points overwrite earlier ones, counted twice)
        for mod in ("novalid", "allclaimed", "noobs"):
            l2, c2 = dict(last), dict(cur)
            if mod == "novalid": l2["valid"] = np.zeros_like(last["valid"])
            if mod == "allclaimed": c2["claimed"] = np.ones(len(cur["x"]), np.uint8)
            if mod == "noobs": l2["obs"] = np.zeros_like(last["obs"]); l2["valid"] = np.ones_like(last["valid"])
            n_o, a_o = oracle.search_by_projection_frame(l2, c2, Tcw, Tlw, cam, bounds, sf, 20.0, True, True)
            n_r, a_r = ref.search_by_projection_frame(l2, c2, Tcw, Tlw, camv, 8, 1.2, 20.0, True, True, mbf=cam[4])
            assert n_r == n_o and np.array_equal(np.where(a_r == -2, -1, a_r), a_o), mod


@pytest.mark.parametrize("seed,th,ratio", [(1, 1.0, 0.8), (2, 3.0, 0.8), (3, 1.0, 0.6), (4, 5.0, 0.9)])
def test_search_by_projection_map_points(oracle, ref, synth, seed, th, ratio):
    """ORBmatcher::SearchByProjection(Frame&, const vector<MapPoint*>&, th) :45-129 — Tracking::SearchLocalPoints, every frame."""
    from scenarios import local_map_scenario
    mp, cur, bounds, sf = local_map_scenario(oracle, synth, seed, f0=seed)
    n_o, a_o = oracle.search_by_projection_mps(mp, cur, bounds, sf, ratio, th)
    n_r, a_r = ref.search_by_projection_mps(mp, cur, ref.cam(500, 500, 320, 240, *bounds), 8, 1.2, ratio, th)
    assert n_r == n_o and np.array_equal(np.where(a_r == -2, -1, a_r), a_o), (n_r, n_o, int((a_r != a_o).sum()))
    assert n_o > 300
    if seed == 1:
        for mod in ("none_in_view", "all_held", "no_obs"):
            m2, c2 = dict(mp), dict(cur)
            if mod == "none_in_view": m2["inview"] = np.zeros_like(mp["inview"])
            if mod == "all_held": c2["held"] = c2["claimed"] = np.ones(len(cur["x"]), np.uint8)
            if mod == "no_obs": m2["obs"] = np.zeros_like(mp["obs"])
            n_o, a_o = oracle.search_by_projection_mps(m2, c2, bounds, sf, ratio, th)
            n_r, a_r = ref.search_by_projection_mps(m2, c2, ref.cam(500, 500, 320, 240, *bounds), 8, 1.2, ratio, th)
            assert n_r == n_o and np.array_equal(np.where(a_r == -2, -1, a_r), a_o), mod


@pytest.mark.parametrize("f0,window,ratio,ori,nf", [(0, 100, 0.9, True, 2000), (8, 50, 0.9, True, 1000), (16, 100, 0.7, False, 2000), (3, 10, 0.9, True, 1000)])
def test_search_for_initialization(oracle, ref, synth, f0, window, ratio, ori, nf):
    """ORBmatcher::SearchForInitialization :408-523 (Tracking::MonocularInitialization, the 2 * nFeatures extractor)."""
    orc = oracle.OrbOracle(nf, 1.2, 8, 20, 7)
    k1, d1 = orc.extract(synth.frame(640, 480, f0)); k2, d2 = orc.extract(synth.frame(640, 480, f0 + 2))
    prev = np.stack([k1["x"], k1["y"]], 1)                                   # Tracking.cc:339-341: vbPrevMatched = keypoints of the first frame
    bounds = (0.0, 640.0, 0.0, 480.0)
    n_o, m_o, p_o = oracle.search_for_initialization(d1, k1, d2, k2, prev, bounds, ratio, ori, window)
    n_r, m_r, p_r = ref.search_for_initialization(d1, k1, d2, k2, prev, ref.cam(500, 500, 320, 240, *bounds), 8, 1.2, ratio, ori, window)
    assert n_r == n_o and _same(m_r, m_o) and _same(p_r, p_o)
    assert n_o > 50 or window < 20
    # second call, as Tracking does on the next frame with the updated vbPrevMatched
    n_o2, m_o2, _ = oracle.search_for_initialization(d1, k1, d2, k2, p_o, bounds, ratio, ori, window)
    n_r2, m_r2, _ = ref.search_for_initialization(d1, k1, d2, k2, p_r, ref.cam(500, 500, 320, 240, *bounds), 8, 1.2, ratio, ori, window)
    assert n_r2 == n_o2 and _same(m_r2, m_o2)


def test_descriptor_medoid(oracle, ref):
    """MapPoint::ComputeDistinctiveDescriptors (MapPoint.cc:247-312): least-median descriptor of each observation group."""
    rng = np.random.default_rng(8)
    sizes = [1, 2, 3, 4, 7, 20, 33]
    off = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int32)
    base = rng.integers(0, 256, (len(sizes), 32), dtype=np.uint8)
    desc = np.concatenate([np.repeat(base[g:g + 1], n, 0) for g, n in enumerate(sizes)])
    noise = (rng.random(desc.shape) < 0.15) * rng.integers(0, 256, desc.shape)
    desc = (desc ^ noise.astype(np.uint8)).astype(np.uint8)
    desc[off[5] + 3] = desc[off[5] + 9]                                   # duplicates inside a group: first minimum wins
    bi_o, _ = oracle.descriptor_medoid(desc, off)
    bi_r = ref.descriptor_medoid(desc, off)
    # the reference returns the descriptor, located here by content: equal rows are interchangeable
    for g in range(len(sizes)):
        assert np.array_equal(desc[off[g] + bi_r[g]], desc[off[g] + bi_o[g]]), g


# ---------------------------------------------------------------------------------------------- line matchers
@pytest.mark.parametrize("n1,n2,seed", [(40, 40, 0), (40, 37, 1), (500, 500, 2), (5, 2, 3), (64, 200, 4)])
def test_line_matchers(oracle, ref, n1, n2, seed):
    """LSDmatcher.cpp:143-183, 257-284, 286-327, 329-362, 382-415 and Frame::lineDescriptorMAD (Frame.cc:190-215)."""
    rng = np.random.default_rng(seed)
    d2 = rng.integers(0, 256, (n2, 32), dtype=np.uint8)
    d1 = d2[rng.integers(0, n2, n1)].copy()
    flip = rng.integers(0, 256, (n1, 32), dtype=np.uint8) & rng.integers(0, 256, (n1, 32), dtype=np.uint8) & rng.integers(0, 256, (n1, 32), dtype=np.uint8)
    d1 ^= flip; d1[::7] = rng.integers(0, 256, (len(d1[::7]), 32), dtype=np.uint8)
    h1 = (rng.random(n1) < 0.6).astype(np.uint8); h2 = (rng.random(n2) < 0.6).astype(np.uint8)
    knn = oracle.knn2(d1, d2)
    for mode in (0, 1, 2, 3):
        n_o, m_o = oracle.line_match(mode, d1, d2, h1, h2)
        n_r, m_r, mad = ref.line_match(mode, d1, d2, h1, h2)
        assert n_r == n_o and _same(m_r, m_o), mode
        assert mad == oracle.line_mad(knn)
    n_r, m_r, _ = ref.line_match(4, d1, d2, h1, h2)          # SearchByDescriptor(KF, F) has the body of SearchByProjection(KF, F)
    n_o, m_o = oracle.line_match(0, d1, d2, h1, h2)
    assert n_r == n_o and _same(m_r, m_o)


# ---------------------------------------------------------------------------------------------- DBoW2
def write_vocab_text(path, k, L, parent, desc, weight, is_leaf, scoring=0, weighting=0):
    """The text format TemplatedVocabulary::loadFromTextFile reads (:1338-1431): header 'k L scoring weighting', then one
    line per node (ids 1.. in file order): parent id, leaf flag, 32 descriptor bytes, weight.
    NO newline after the last line: the reference loops `while(!f.eof())` and turns a trailing empty line into a phantom extra
    child of the root whose leaf flag, descriptor and weight are indeterminate (failed extractions leave them untouched) — UB
    this build does not imitate; the package's loader skips blank lines."""
    lines = [f"{k} {L} {scoring} {weighting}"]
    for i in range(1, len(parent)):
        lines.append(f"{int(parent[i])} {int(is_leaf[i])} " + " ".join(str(int(v)) for v in desc[i]) + f" {float(weight[i])!r}")
    with open(path, "w") as f:
        f.write("\n".join(lines))


@pytest.mark.parametrize("k,L,stop,early", [(10, 3, 0.0, 0.0), (10, 3, 0.1, 0.2), (4, 5, 0.05, 0.3), (2, 1, 0.0, 0.0), (10, 2, 0.0, 0.0)])
def test_dbow2_transform(oracle, ref, pkg, synth, tmp_path, k, L, stop, early):
    """DBoW2's own loadFromTextFile + transform (TemplatedVocabulary.h:1127-1259, :1338-1431), as Frame::ComputeBoW calls it
    (levelsup = 4), against the oracle's restated descent and the package's host-side BowVector / FeatureVector assembly."""
    parent, nd, w, leaf = pkg.Vocabulary.random_arrays(k, L, seed=k * 100 + L, stop_fraction=stop, early_leaf_fraction=early)
    path = str(tmp_path / "voc.txt")
    write_vocab_text(path, k, L, parent, nd, w, leaf)
    voc = ref.Vocabulary(path)
    assert len(voc) == int(leaf.sum())
    _, _, d1, _, _ = _pair(oracle, synth, 2)
    feats = d1[:400].copy()
    m = min(20, len(nd) - 1)
    feats[:m] = nd[1:1 + m]                                          # exact hits on node descriptors
    nd2 = nd.copy()
    if len(nd) > 3:
        nd2[2] = nd2[1]                                              # identical siblings: ties -> first child (strict '<', :1241)
        write_vocab_text(path, k, L, parent, nd2, w, leaf); voc = ref.Vocabulary(path)
    V = pkg.Vocabulary.__new__(pkg.Vocabulary); V.scoring, V.weighting, V._h = 0, 0, None
    depth = np.zeros(len(parent), int)
    for i in range(1, len(parent)):
        depth[i] = depth[parent[i]] + 1
    leaves = np.flatnonzero(leaf)
    word_r, wt_r = voc.words(feats)
    for levelsup in (4, 1, 0, 10):
        node_r, ids_r, w_r = voc.transform(feats, levelsup)
        word_o, node_o, w_o = oracle.vocab_transform(L, parent, nd2, w, leaf, feats, levelsup)
        assert _same(word_r, word_o) and _same(wt_r, w_o)
        # stopped words are left out (:1162-1166).  A leaf that sits ABOVE level L - levelsup never assigns *nid (:1254): the
        # reference then files the feature under an indeterminate node (the caller's `NodeId nid` is uninitialised, :1150); the
        # oracle and the kernel file it under the root.  Real vocabularies (ORBvoc: k=10, L=6, levelsup=4) have no such leaves.
        defined = (depth[leaves[word_o]] >= L - levelsup) | (L - levelsup <= 0)
        exp = np.where(w_o > 0, node_o, -1)
        assert np.array_equal(node_r[defined], exp[defined]), levelsup
        assert np.all(node_o[~defined] == 0)
        node_o = np.where(defined, node_o, node_r)                # (compare the assemblies on the reference's filing)
        ids_p, vals_p = V.bow_vector(word_o, w_o)
        assert _same(ids_r, ids_p) and _same(w_r, vals_p)
        nodes_p, off_p, idx_p = pkg.Vocabulary.feature_vector(node_o, w_o)
        for j, nid in enumerate(nodes_p):
            assert np.array_equal(np.flatnonzero(node_r == nid), idx_p[off_p[j]:off_p[j + 1]])


# ---------------------------------------------------------------------------------------------- lines
def test_extract_line_segment(oracle, ref, icl_gray, synth):
    """LineSegment::ExtractLineSegment (ExtractLineSegment.cpp:18-69, lsdNFeatures = 40): the reference's own sort / cut /
    renumber / line-equation code over the oracle's LSD + KeyLine + LBD (those three are OpenCV's, not the reference's)."""
    for img in (icl_gray, synth.frame(640, 480, 0), synth.frame(640, 480, 13)):
        kl, ld, eq = ref.line_extract(img)
        okl, old, oeq = oracle.LineOracle(40).extract(img)
        assert len(kl) == len(okl) == 40
        # the reference's std::sort is unstable on exactly equal responses: compare as sets of rows when ties reach the cut
        if len(np.unique(okl["response"])) == len(okl):
            assert kl.tobytes() == okl.tobytes() and np.array_equal(ld, old) and np.array_equal(eq, oeq)
        else:
            key = lambda a: sorted(bytes(a[i].tobytes()[8:]) for i in range(len(a)))
            assert key(kl) == key(okl)


# ---------------------------------------------------------------------------------------------- Frame
def test_frame_constructor(oracle, ref, icl_gray):
    """Frame::Frame(imGray, ...) (Frame.cc:69-131): ExtractORB + ExtractLSD + UndistortKeyPoints + AssignFeaturesToGrid."""
    fr = ref.frame_from_image(icl_gray)
    ok, od = oracle.OrbOracle(1000, 1.2, 8, 20, 7).extract(icl_gray)
    assert _same(fr["keys"], ok) and _same(fr["keysUn"], ok) and _same(fr["desc"], od)
    okl, old, oeq = oracle.LineOracle(40).extract(icl_gray)
    assert _same(fr["keylines"], okl) and _same(fr["ldesc"], old) and _same(fr["lineeq"], oeq)
    assert list(fr["bounds"]) == [0, 640, 0, 480]
    # grid cell (c, r) holds the features whose rounded cell is (c, r), ascending
    rnd = lambda v: np.floor(v.astype(np.float32) + np.float32(0.5)).astype(int)      # C round() on non-negative floats (PosInGrid, Frame.cc:462-472)
    gx = rnd(ok["x"] * np.float32(64 / 640)); gy = rnd(ok["y"] * np.float32(48 / 480))
    for c, r in [(0, 0), (10, 7), (32, 24), (63, 47), (40, 13)]:
        cell = fr["grid_idx"][fr["grid_off"][c * 48 + r]:fr["grid_off"][c * 48 + r + 1]]
        assert np.array_equal(cell, np.flatnonzero((gx == c) & (gy == r)))


# ------------------------------------------------------------------------------------------------
# SURVEY.md 8(f) row 3: line projection matchers and Fuse
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("seed,th,mono,sign,ratio", [(1, 20.0, True, 0, 0.8), (2, 20.0, False, 1, 0.8), (3, 40.0, False, -1, 0.9), (4, 10.0, True, 0, 0.6)])
def test_line_search_by_projection_frame(oracle, ref, synth, seed, th, mono, sign, ratio):
    """LSDmatcher::SearchByProjection(Frame& Current, const Frame& Last, th, bMono) :22-141, forward / backward / mono level ranges."""
    from scenarios import line_scenario
    sc = line_scenario(oracle, synth, seed, f0=seed, stereo_sign=sign)
    last, cur = sc["last"], sc["cur"]
    q = oracle.line_project_frame(last["state"] == 1, last["Pw"], last["oct"], sc["Tcw"][:3], sc["Tlw"][:3], sc["cam5"], sc["bounds"], sc["sf"], th, mono)
    n_o, a_o = oracle.line_window_search(q, last["obs"], last["dml"], cur["ld"], cur["kl"], cur["oct"], cur["held"], ratio)
    cam = ref.cam(*sc["cam5"][:4], *sc["bounds"])
    n_r, a_r = ref.line_projection_frame(last, cur, sc["Tcw"], sc["Tlw"], cam, sc["cam5"][4], 8, 1.2, ratio, th, mono)
    assert n_r == n_o and np.array_equal(np.where(a_r == -2, -1, a_r), a_o), (n_r, n_o, int((a_r != a_o).sum()))
    assert n_o > 5 and q["active"].sum() > 100


@pytest.mark.parametrize("seed,th,ratio", [(1, 1.0, 0.8), (2, 3.0, 0.8), (3, 1.0, 0.6), (4, 0.5, 0.9)])
def test_line_search_by_projection_mls(oracle, ref, synth, seed, th, ratio):
    """LSDmatcher::SearchByProjection(Frame&, const vector<MapLine*>&, th) :185-255 — Tracking::SearchLocalLines (Tracking.cc:1783)."""
    from scenarios import local_lines_scenario
    ml, cur, sf = local_lines_scenario(oracle, synth, seed, f0=seed)
    q = oracle.line_project_mls(ml["inview"], ml["bad"], ml["level"], ml["viewcos"], sf, th); q["proj"] = ml["proj"]
    n_o, a_o = oracle.line_window_search(q, ml["obs"], ml["desc"], cur["ld"], cur["kl"], cur["oct"], cur["held"], ratio)
    n_r, a_r = ref.line_projection_mls(ml, cur, ref.cam(500, 500, 320, 240, 0, 640, 0, 480), 8, 1.2, ratio, th)
    assert n_r == n_o and np.array_equal(np.where(a_r == -2, -1, a_r), a_o), (n_r, n_o, int((a_r != a_o).sum()))
    assert n_o > 30
    if seed == 1:
        for mod in ("none_in_view", "all_held", "no_obs"):
            m2, c2 = dict(ml), dict(cur)
            if mod == "none_in_view": m2["inview"] = np.zeros_like(ml["inview"])
            if mod == "all_held": c2["held"] = np.ones(len(cur["oct"]), np.uint8)
            if mod == "no_obs": m2["obs"] = np.zeros_like(ml["obs"])
            q = oracle.line_project_mls(m2["inview"], m2["bad"], m2["level"], m2["viewcos"], sf, th); q["proj"] = m2["proj"]
            n_o, a_o = oracle.line_window_search(q, m2["obs"], m2["desc"], c2["ld"], c2["kl"], c2["oct"], c2["held"], ratio)
            n_r, a_r = ref.line_projection_mls(m2, c2, ref.cam(500, 500, 320, 240, 0, 640, 0, 480), 8, 1.2, ratio, th)
            assert n_r == n_o and np.array_equal(np.where(a_r == -2, -1, a_r), a_o), mod


def _fused(bi, bd, active):
    return np.where((np.asarray(active) != 0) & (bd <= 50) & (bi >= 0), bi, -1)


@pytest.mark.parametrize("seed,th,stereo", [(1, 3.0, False), (2, 3.0, True), (3, 5.0, False), (4, 1.5, True)])
def test_fuse_points(oracle, ref, synth, seed, th, stereo):
    """ORBmatcher::Fuse(KeyFrame*, const vector<MapPoint*>&, th) :828-973 (LocalMapping::SearchInNeighbors): projection gates, PredictScale,
    chi-square gates (mono / stereo), nearest descriptor; every fused MapPoint ends up at (or is replaced into) the feature the search chose."""
    from scenarios import fuse_points_scenario
    sc = fuse_points_scenario(oracle, synth, seed, f0=seed, stereo=stereo)
    mp, kf = sc["mp"], sc["kf"]
    cam = ref.cam(*sc["cam5"][:4], *sc["bounds"])
    n_r, f_r, acc = ref.fuse_points(mp, kf, sc["Tcw"], cam, sc["cam5"][4], 8, 1.2, th)
    q = oracle.fuse_project_points(mp["state"] != 1, mp["Xw"], mp["normal"], acc["min_inv"], acc["max_inv"], mp["max_raw"], sc["Tcw"][:3], acc["Ow"],
                                   sc["cam5"], sc["bounds"], 8, acc["log_scale"])
    bi, bd = oracle.fuse_points_search(q, mp["desc"], kf["desc"], kf["x"], kf["y"], kf["oct"], kf["uright"], sc["bounds"], sc["sf"], sc["inv_sigma2"], th)
    f_o = _fused(bi, bd, q["active"])
    assert np.array_equal(f_r, f_o), (int((f_r != f_o).sum()), np.nonzero(f_r != f_o)[0][:8])
    assert n_r == int((f_o >= 0).sum())
    assert n_r > 150 and q["active"].sum() < (mp["state"] == 1).sum()          # the gates dropped some


@pytest.mark.parametrize("seed,th", [(1, 3.0), (2, 5.0), (3, 10.0)])
def test_fuse_lines(oracle, ref, synth, seed, th):
    """LSDmatcher::Fuse(KeyFrame*, const vector<MapLine*>&, th) :417-548."""
    from scenarios import fuse_lines_scenario
    sc = fuse_lines_scenario(oracle, synth, seed, f0=seed)
    ml, kf = sc["ml"], sc["kf"]
    cam = ref.cam(*sc["cam5"][:4], *sc["bounds"])
    # MapLine::PredictScale is not clamped (MapLine.cpp:386-395): a level outside the pyramid makes the reference read mvScaleFactors out of
    # bounds, so the comparison keeps to lines whose level is inside (the oracle and the product drop the others)
    q0 = oracle.fuse_project_lines(ml["state"] != 1, ml["Pw"], ml["normal"], ml["min_raw"] * np.float32(0.8), ml["max_raw"] * np.float32(1.2), ml["max_raw"],
                                   sc["Tcw"][:3], np.zeros(3), sc["cam5"], sc["bounds"], 8, np.log(np.float32(1.2)))
    ml = dict(ml); ml["state"] = np.where((q0["level"] < 0) | (q0["level"] >= 8), 0, ml["state"]).astype(np.uint8)
    n_r, f_r, acc = ref.fuse_lines(ml, kf, sc["Tcw"], cam, 8, 1.2, th)
    q = oracle.fuse_project_lines(ml["state"] != 1, ml["Pw"], ml["normal"], acc["min_inv"], acc["max_inv"], ml["max_raw"], sc["Tcw"][:3], acc["Ow"],
                                  sc["cam5"], sc["bounds"], 8, acc["log_scale"])
    bi, bd = oracle.fuse_lines_search(q, ml["desc"], kf["ld"], kf["kl"], kf["oct"], sc["sf"], th)
    f_o = _fused(bi, bd, q["active"])
    assert np.array_equal(f_r, f_o), (int((f_r != f_o).sum()), np.nonzero(f_r != f_o)[0][:8])
    assert n_r == int((f_o >= 0).sum())
    assert n_r > 10
