"""GPU parity: CUDA ORB path (through the C-ABI) vs the CPU oracle, stage by stage and end to end.
Bit-exact for integer work (pyramid, candidates, octree selection, descriptors); float outputs
(angle, scaled coordinates) are expected bit-equal too and are checked at 1e-4 px / 1e-3 rad."""
import os
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _compare_all(ext, orc, img, tag):
    kps, desc = ext(img)
    okps, odesc = orc.extract(img)
    L = ext.nlevels
    for l in range(L):
        assert ext.level_size(l) == orc.level_size(l), (tag, l)
        assert np.array_equal(ext.level(l), orc.level(l)), f"{tag}: pyramid level {l} differs"
    assert np.array_equal(ext.level(1, bordered=True), orc.level(1, bordered=True)), f"{tag}: bordered level"
    for l in range(L):
        gx, gy, gr = ext.candidates(l)
        ox, oy, orr = orc.candidates(l)
        assert len(gx) == len(ox), f"{tag}: level {l} candidate count {len(gx)} vs {len(ox)}"
        assert np.array_equal(gx, ox) and np.array_equal(gy, oy) and np.array_equal(gr, orr), f"{tag}: level {l} candidates"
    for l in range(L):
        gx, gy, gr = ext.level_keypoints(l)
        ox, oy, orr, _ = orc.level_keypoints(l)
        assert len(gx) == len(ox), f"{tag}: level {l} octree count {len(gx)} vs {len(ox)}"
        assert np.array_equal(gx, ox) and np.array_equal(gy, oy) and np.array_equal(gr, orr), f"{tag}: level {l} octree selection"
        if len(ox):
            assert np.array_equal(ext.blurred(l), orc.blurred(l)), f"{tag}: blurred level {l}"
    assert len(kps) == len(okps), (tag, len(kps), len(okps))
    for fld in ("octave", "class_id", "response", "size"):
        assert np.array_equal(kps[fld], okps[fld]), (tag, fld)
    assert np.max(np.abs(kps["x"] - okps["x"]), initial=0) <= 1e-4 and np.max(np.abs(kps["y"] - okps["y"]), initial=0) <= 1e-4
    dang = np.abs(kps["angle"] - okps["angle"]); dang = np.minimum(dang, 360 - dang)
    assert np.max(dang, initial=0) * np.pi / 180 <= 1e-3, (tag, float(np.max(dang)))
    assert np.array_equal(kps["angle"], okps["angle"]), f"{tag}: angles not bit-equal"
    assert np.array_equal(kps["x"], okps["x"]) and np.array_equal(kps["y"], okps["y"])
    assert np.array_equal(desc, odesc), f"{tag}: descriptors differ in {int((desc != odesc).any(1).sum())} rows"
    return len(kps)


def test_icl_frame_1000(pkg, oracle, icl_gray):
    """BASELINE.json config 1/2: 640x480 ICL-NUIM frame, nFeatures=1000, 8 levels."""
    ext = pkg.ORBextractor(1000, 1.2, 8, 20, 7, max_width=640, max_height=480)
    orc = oracle.OrbOracle(1000, 1.2, 8, 20, 7)
    n = _compare_all(ext, orc, icl_gray, "icl")
    assert n == 1002            # SURVEY.md 8(c) known answer
    t = ext._tables(); o = orc.tables()
    for k in t:
        assert np.array_equal(t[k], o[k]), k


def test_icl_frame_2000_initialiser(pkg, oracle, icl_gray):
    """The initialiser extractor uses 2*nFeatures (Tracking.cc:120)."""
    _compare_all(pkg.ORBextractor(2000, 1.2, 8, 20, 7, max_width=640, max_height=480), oracle.OrbOracle(2000, 1.2, 8, 20, 7), icl_gray, "icl2000")


@pytest.mark.parametrize("f", [0, 1, 5, 8])
def test_synthetic_640(pkg, oracle, synth, f):
    img = synth.frame(640, 480, f)
    _compare_all(pkg.ORBextractor(1000, 1.2, 8, 20, 7, max_width=640, max_height=480), oracle.OrbOracle(1000, 1.2, 8, 20, 7), img, f"syn{f}")


def test_synthetic_1280_4000(pkg, oracle, synth):
    """BASELINE.json config 4: 1280x960, nFeatures=4000."""
    img = synth.frame(1280, 960, 0)
    _compare_all(pkg.ORBextractor(4000, 1.2, 8, 20, 7, max_width=1280, max_height=960), oracle.OrbOracle(4000, 1.2, 8, 20, 7), img, "syn1280")


def test_edge_cases(pkg, oracle):
    rng = np.random.default_rng(7)
    ext = pkg.ORBextractor(500, 1.2, 8, 20, 7, max_width=800, max_height=600)
    orc = oracle.OrbOracle(500, 1.2, 8, 20, 7)
    # empty image: silent return (ORBextractor.cc:1046)
    k, d = ext(np.zeros((0, 0), np.uint8))
    assert len(k) == 0 and d.shape == (0, 32)
    # flat image: no corners anywhere
    k, d = ext(np.full((240, 320), 77, np.uint8))
    assert len(k) == 0
    # pure noise (many candidates per cell), odd sizes, non-contiguous pitch, different size on the same handle
    noise = rng.integers(0, 256, (333, 517), dtype=np.uint8)
    _compare_all(ext, orc, noise, "noise")
    big = rng.integers(0, 256, (480, 700), dtype=np.uint8)
    _compare_all(ext, orc, big[:, 30:670], "pitched-view")
    _compare_all(ext, orc, (rng.integers(0, 2, (200, 260)) * 255).astype(np.uint8), "binary")


def test_other_parameters(pkg, oracle, synth):
    img = synth.frame(640, 480, 3)
    _compare_all(pkg.ORBextractor(300, 1.5, 4, 30, 10, max_width=640, max_height=480), oracle.OrbOracle(300, 1.5, 4, 30, 10), img, "p300")
    _compare_all(pkg.ORBextractor(1500, 1.1, 12, 12, 5, max_width=640, max_height=480), oracle.OrbOracle(1500, 1.1, 12, 12, 5), img, "p1500")


def test_batch_equals_single(pkg, oracle, synth):
    """Batched frames (grid.z) must reproduce the per-frame results exactly, through HOST buffers."""
    frames = synth.batch(640, 480, 6)
    ext = pkg.ORBextractor(1000, 1.2, 8, 20, 7, max_width=640, max_height=480, max_batch=6)
    kps, desc, n = ext.extract_batch(frames)
    orc = oracle.OrbOracle(1000, 1.2, 8, 20, 7)
    for f in range(6):
        ok, od = orc.extract(frames[f])
        assert n[f] == len(ok)
        assert kps[f, :n[f]].tobytes() == ok.tobytes()
        assert np.array_equal(desc[f, :n[f]], od)


def test_non_tma_fallback_path(pkg, oracle, synth, icl_gray, monkeypatch):
    """The tile kernels stage their input with TMA (cp.async.bulk.tensor) by default; SSLPL_NO_TMA=1 and views that
    violate TMA's 16-byte rules use ordinary loads.  Both must give the oracle's result."""
    monkeypatch.setenv("SSLPL_NO_TMA", "1")
    ext = pkg.ORBextractor(1000, 1.2, 8, 20, 7, max_width=640, max_height=480)
    monkeypatch.delenv("SSLPL_NO_TMA")
    orc = oracle.OrbOracle(1000, 1.2, 8, 20, 7)
    _compare_all(ext, orc, icl_gray, "no-tma")
    _compare_all(ext, orc, synth.frame(640, 480, 2), "no-tma-syn")
    # a width that is not a multiple of 16 forces the fallback for level 0 on a TMA-enabled handle
    ext2 = pkg.ORBextractor(800, 1.2, 8, 20, 7, max_width=700, max_height=500)
    img = synth.frame(640, 480, 4)[:, :613]
    _compare_all(ext2, oracle.OrbOracle(800, 1.2, 8, 20, 7), np.ascontiguousarray(img), "w613")


def test_pyramid_odd_sizes(pkg, oracle, synth, icl_gray, monkeypatch):
    """The pyramid (k_resize, one launch per level) and the TMA-staged kernels that read it must give the oracle's planes and
    keypoints with and without TMA, also at sizes whose level widths are not multiples of the tiles."""
    orc = oracle.OrbOracle(1000, 1.2, 8, 20, 7)
    for env in ({}, {"SSLPL_NO_TMA": "1"}):
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        ext = pkg.ORBextractor(1000, 1.2, 8, 20, 7, max_width=700, max_height=500)
        for k in env:
            monkeypatch.delenv(k)
        _compare_all(ext, orc, icl_gray, f"pyr{env}")
        _compare_all(ext, orc, np.ascontiguousarray(synth.frame(640, 480, 5)[:437, :613]), f"pyr613{env}")
        _compare_all(ext, orc, np.ascontiguousarray(synth.frame(640, 480, 6)[:111, :171]), f"pyr171{env}")


def test_async_begin_and_device_paths(pkg, oracle, synth):
    """The asynchronous host-buffer form (pinned buffers, sslpl_orb_extract_batch_begin + sync) and the device-resident
    form must give the same keypoints/descriptors as the synchronous call."""
    frames = synth.batch(640, 480, 4)
    ext = pkg.ORBextractor(1000, 1.2, 8, 20, 7, max_width=640, max_height=480, max_batch=4)
    k0, d0, n0 = ext.extract_batch(frames)
    hp = pkg.host_alloc(frames.shape, np.uint8); hp[...] = frames
    out = (pkg.host_alloc((4, ext.cap), pkg.KEYPOINT_DTYPE), pkg.host_alloc((4, ext.cap, 32), np.uint8), pkg.host_alloc((4,), np.int32))
    ext.extract_batch_begin(hp, out)
    ext.sync()
    assert np.array_equal(out[2], n0)
    for f in range(4):
        assert out[0][f, :n0[f]].tobytes() == k0[f, :n0[f]].tobytes() and np.array_equal(out[1][f, :n0[f]], d0[f, :n0[f]])
    ls = pkg.LineSegment(40, max_width=640, max_height=480, max_batch=4)
    kl0, ld0, eq0, nl0 = ls.extract_batch(frames)
    lout = (pkg.host_alloc((4, 40), pkg.KEYLINE_DTYPE), pkg.host_alloc((4, 40, 32), np.uint8), pkg.host_alloc((4, 40, 3), np.float64), pkg.host_alloc((4,), np.int32))
    ls.extract_batch_begin(hp, lout)
    ls.sync()
    assert np.array_equal(lout[3], nl0)
    for f in range(4):
        assert np.array_equal(lout[1][f, :nl0[f]], ld0[f, :nl0[f]]) and lout[0][f, :nl0[f]].tobytes() == kl0[f, :nl0[f]].tobytes()
