"""GPU parity: CUDA line path (LSD + KeyLine packaging + LBD + line equations, through the C-ABI) vs the CPU oracle.
LSD endpoints within 1e-4 px (north_star tolerance; expected bit-equal) vs the oracle AND vs cv2's LSD; LBD bytes
bit-equal; angles within 1e-3 rad."""
import numpy as np
import cv2
import pytest

pytestmark = pytest.mark.gpu

BORDERLINE_OK = set()          # tags of inputs allowed one borderline LSD segment of difference (see _check_frame); empty: none is needed


def _check_frame(pkg, oracle, img, nfeat, tag, vs_cv2=True):
    ls = pkg.LineSegment(nfeat, max_width=img.shape[1], max_height=img.shape[0])
    kl, ld, eq = ls.ExtractLineSegment(img)
    raw = ls.raw_segments()
    lo = oracle.LineOracle(nfeat)
    okl, old, oeq = lo.extract(img)
    oraw = lo.raw_segments()
    if raw.shape != oraw.shape or np.max(np.abs(raw - oraw), initial=0) > 1e-4:
        # LSD decides whether the extreme pixels of a region are inside its rectangle from the LAST BIT of
        # cos/sin(theta) (they lie exactly on the end edges).  glibc mis-rounds ~0.14% of those; the device rounds
        # correctly (ddtrig.h).  Such a flip may add/remove ONE borderline segment (|log NFA| small).  It is tolerated only for
        # the inputs listed in BORDERLINE_OK (none of the committed test inputs needs it), and even then every KeyLine and LBD
        # descriptor of the segments both sides found is still compared.
        assert tag in BORDERLINE_OK, f"{tag}: LSD segments differ (GPU {len(raw)}, oracle {len(oraw)})"
        so = {tuple(np.round(r, 3)) for r in oraw}; sg = {tuple(np.round(r, 3)) for r in raw}
        assert len(so ^ sg) <= 1 and abs(len(raw) - len(oraw)) <= 1, f"{tag}: {len(so ^ sg)} segments differ (GPU {len(raw)}, oracle {len(oraw)})"
        res = cv2.createLineSegmentDetector(cv2.LSD_REFINE_ADV).detect(img)
        for seg in so - sg:
            j = [tuple(np.round(r, 3)) for r in oraw].index(seg)
            assert abs(float(res[3].ravel()[j])) < 3.0, f"{tag}: non-borderline segment missing (log NFA {res[3].ravel()[j]})"
        key = lambda k: (round(float(k["startPointX"]), 3), round(float(k["startPointY"]), 3), round(float(k["endPointX"]), 3), round(float(k["endPointY"]), 3))
        oidx = {key(k): i for i, k in enumerate(okl)}
        common = [(i, oidx[key(k)]) for i, k in enumerate(kl) if key(k) in oidx]
        assert len(common) >= min(len(kl), len(okl)) - 1
        for i, j in common:
            assert kl["numOfPixels"][i] == okl["numOfPixels"][j] and np.array_equal(ld[i], old[j]), f"{tag}: KeyLine / LBD of a common segment differs"
        return len(kl), len(raw)
    if vs_cv2:
        ref = cv2.createLineSegmentDetector(cv2.LSD_REFINE_ADV).detect(img)[0]
        ref = np.zeros((0, 4), np.float32) if ref is None else ref.reshape(-1, 4)
        assert ref.shape == raw.shape and np.max(np.abs(raw - ref), initial=0) <= 1e-4, f"{tag}: differs from cv2 LSD"
    assert len(kl) == len(okl), (tag, len(kl), len(okl))
    for fld in ("class_id", "octave", "numOfPixels"):
        assert np.array_equal(kl[fld], okl[fld]), (tag, fld)
    for fld in ("startPointX", "startPointY", "endPointX", "endPointY", "sPointInOctaveX", "sPointInOctaveY",
                "ePointInOctaveX", "ePointInOctaveY", "pt_x", "pt_y"):
        assert np.max(np.abs(kl[fld] - okl[fld]), initial=0) <= 1e-4, (tag, fld)
    assert np.max(np.abs(kl["angle"] - okl["angle"]), initial=0) <= 1e-3, tag
    assert np.allclose(kl["lineLength"], okl["lineLength"], rtol=1e-6) and np.allclose(kl["response"], okl["response"], rtol=1e-6)
    assert np.allclose(kl["size"], okl["size"], rtol=1e-5, atol=1e-3)
    assert np.allclose(eq, oeq, rtol=1e-9, atol=1e-9), tag
    nbad = int((ld != old).any(1).sum())
    assert nbad == 0, f"{tag}: {nbad} of {len(ld)} LBD descriptors differ"
    return len(kl), len(raw)


def test_icl_frame_lines(pkg, oracle, icl_gray):
    """BASELINE.json config 2: 640x480 ICL frame, LSD + LBD, lsdNFeatures = 40 (ExtractLineSegment.cpp:42)."""
    n, nraw = _check_frame(pkg, oracle, icl_gray, 40, "icl")
    assert n == 40 and nraw == 225


def test_icl_all_lines(pkg, oracle, icl_gray):
    n, _ = _check_frame(pkg, oracle, icl_gray, 1000, "icl-all")
    assert n == 225


@pytest.mark.parametrize("f", [0, 3, 8])
def test_synthetic_640_lines(pkg, oracle, synth, f):
    _check_frame(pkg, oracle, synth.frame(640, 480, f), 40, f"syn{f}")


def test_synthetic_1280_500_lines(pkg, oracle, synth):
    """BASELINE.json config 4: 1280x960, 500 lines."""
    n, nraw = _check_frame(pkg, oracle, synth.frame(1280, 960, 0), 500, "syn1280")
    assert n == 500 and nraw > 500


def test_line_edge_cases(pkg, oracle, synth):
    ls = pkg.LineSegment(40, max_width=640, max_height=480)
    kl, ld, eq = ls.ExtractLineSegment(np.full((240, 320), 90, np.uint8))          # flat image: no lines
    assert len(kl) == 0 and ld.shape == (0, 32)
    yy, xx = np.mgrid[0:120, 0:160]
    for im in [np.where(xx >= 80, 200, 50).astype(np.uint8), np.where(yy >= 60, 200, 50).astype(np.uint8),
               np.where((yy > 40) & (yy < 60) & (xx > 30) & (xx < 110), 200, 0).astype(np.uint8)]:
        _check_frame(pkg, oracle, np.ascontiguousarray(im), 40, "shape")
    _check_frame(pkg, oracle, synth.frame(320, 240, 1), 40, "syn320")


def test_line_odd_sizes(pkg, oracle, synth):
    """Widths that are not multiples of 4 (frame and 0.8x detection scale): the scalar store paths of the vectorised kernels."""
    for (w, h, seed) in [(333, 251, 2), (322, 243, 3)]:
        _check_frame(pkg, oracle, synth.frame(w, h, seed), 40, f"syn{w}x{h}")


def test_line_batch_equals_single(pkg, oracle, synth):
    frames = synth.batch(640, 480, 5)
    ls = pkg.LineSegment(40, max_width=640, max_height=480, max_batch=5)
    kl, ld, eq, n = ls.extract_batch(frames)
    for f in range(5):
        okl, old, oeq = oracle.LineOracle(40).extract(frames[f])
        assert n[f] == len(okl)
        assert np.array_equal(ld[f, :n[f]], old)
        assert np.max(np.abs(kl[f, :n[f]]["startPointX"] - okl["startPointX"]), initial=0) <= 1e-4


def test_max_walkers_knob_does_not_change_results(pkg, synth):
    """sslpl_line_set_max_walkers only bounds how many region-walker CTAs are resident (persistent grid pulling frames)."""
    frames = synth.batch(640, 480, 6)
    ls = pkg.LineSegment(40, max_width=640, max_height=480, max_batch=6)
    ref = ls.extract_batch(frames)
    for cap in (1, 4, 0):
        ls.set_max_walkers(cap)
        got = ls.extract_batch(frames)
        assert np.array_equal(got[3], ref[3]) and np.array_equal(got[1], ref[1]) and got[0].tobytes() == ref[0].tobytes(), cap


WALKERS = [("one warp, round-2a form", {"SSLPL_WALKER_WARPS": "-1"}),
           ("multi-warp round 2a, 16 warps", {"SSLPL_WALKER_WARPS": "16"}),
           ("multi-warp round 2a, 5 warps", {"SSLPL_WALKER_WARPS": "5"}),
           ("multi-warp round 2a, 2 warps", {"SSLPL_WALKER_WARPS": "2"}),
           ("multi-warp round 2a, 3 warps", {"SSLPL_WALKER_WARPS": "3"}),
           ("multi-warp round 2a, 4 warps", {"SSLPL_WALKER_WARPS": "4"}),
           ("multi-warp round 2a, 8 warps", {"SSLPL_WALKER_WARPS": "8"}),
           ("multi-warp round 2a, 12 warps", {"SSLPL_WALKER_WARPS": "12"}),
           ("automatic choice", {})]


@pytest.mark.parametrize("name,env", WALKERS, ids=[w[0] for w in WALKERS])
def test_every_region_walker_is_the_sequential_one(pkg, oracle, synth, icl_gray, monkeypatch, name, env):
    """The region stage exists in two forms (csrc/line.cu: one warp per frame, k_lsd_regions_solo, and the multi-warp speculative
    walker k_lsd_regions); the handle picks one by batch size.  Each of them, forced through SSLPL_WALKER_WARPS, which the handle
    reads when it is created, at several warp counts, and the automatic choice (16 warps for these single frames), has to reproduce
    the sequential detector: same raw segments, KeyLines and LBD bytes as the oracle, several runs each (the multi-warp form is
    timing dependent by construction)."""
    monkeypatch.delenv("SSLPL_WALKER_WARPS", raising=False)
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    reps = 1 if name.startswith("one warp") else 4
    for tag, img in (("icl", icl_gray), ("syn3", synth.frame(640, 480, 3)), ("syn8", synth.frame(640, 480, 8))):
        for _ in range(reps):
            _check_frame(pkg, oracle, img, 40, f"{name}/{tag}", vs_cv2=False)
    _check_frame(pkg, oracle, synth.frame(1280, 960, 0), 500, f"{name}/syn1280", vs_cv2=False)


def test_line_match_two_frames(pkg, oracle, synth):
    """config 3, line half: LSDmatcher::SearchByProjection(KF,F) (LSDmatcher.cpp:143) on LBD descriptors of two frames."""
    ls = pkg.LineSegment(40, max_width=640, max_height=480)
    _, l1, _ = ls.ExtractLineSegment(synth.frame(640, 480, 0))
    _, l2, _ = ls.ExtractLineSegment(synth.frame(640, 480, 1))
    has = np.ones(len(l1), np.uint8)
    n_g, t_g = pkg.LSDmatcher().SearchByProjection(l1, has, l2)
    n_o, t_o = oracle.line_match(0, l1, l2, has, None)
    assert n_g == n_o and np.array_equal(t_g, t_o)
    bf = cv2.BFMatcher(cv2.NORM_HAMMING, False).knnMatch(l1, l2, 2)
    knn = pkg.Matcher().knn2(l1, l2)
    assert [[m[0].trainIdx, int(m[0].distance), m[1].trainIdx, int(m[1].distance)] for m in bf] == knn.tolist()
