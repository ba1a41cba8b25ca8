"""GPU: bench.py --dump-outputs writes what the last timed step computed.  The single1280 workload (17 frames a step, all of them
dumped), its last step's input frames rebuilt here: keypoints, descriptors and BoW matches against the oracle, lines against the
package's host API and their matches against the oracle's matcher on those lines."""
import json
import os
import subprocess
import sys
import numpy as np
import pytest

from conftest import ROOT

pytestmark = pytest.mark.gpu

NAMES = {"frames", "keypoint_counts", "keypoints", "descriptors", "point_matches", "point_match_counts", "line_counts", "keylines",
         "line_descriptors", "line_equations", "line_matches", "line_match_counts"}


def test_dump_outputs_hold_the_last_timed_step(pkg, oracle, synth, tmp_path):
    import bench
    steps, warmup = 2, 3
    out = tmp_path / "out"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "single1280", "--steps", str(steps), "--warmup", str(warmup),
                        "--no-cpu-baseline", "--dump-outputs", str(out)], capture_output=True, text=True, timeout=900,
                       env=dict(os.environ, SSLPL_BENCH_NO_TRACE="1"), cwd=ROOT)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    line = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    assert line["steps"] == steps and line["warmup"] == warmup
    d = {f[:-4]: np.load(out / f) for f in os.listdir(out)}
    assert set(d) == NAMES
    assert all(a.dtype in (np.float32, np.float64) for a in d.values()) and sum(a.nbytes for a in d.values()) <= 64e6

    cfg = bench.WORKLOADS["single1280"]
    W, H, NF, NL, B = cfg["width"], cfg["height"], cfg["nfeatures"], cfg["nlines"], cfg["frames_per_gpu"] + 1
    s = (warmup + steps - 1) % bench.n_input_sets(B, W, H)
    frames = bench.gen_frames(cfg, 0, s + 1, B)[s]
    assert np.array_equal(d["frames"], np.arange(1, B))
    n, nl = d["keypoint_counts"].astype(int), d["line_counts"].astype(int)
    assert len(d["keypoints"]) == len(d["descriptors"]) == n.sum() and len(d["keylines"]) == len(d["line_equations"]) == nl.sum()

    orc = oracle.OrbOracle(NF, 1.2, 8, 20, 7)
    voc = synth.vocabulary(bench.NWORDS)
    ls = pkg.LineSegment(NL, max_width=W, max_height=H, max_batch=B)
    kl_h, ld_h, eq_h, nl_h = ls.extract_batch(frames)
    ls.close()
    prev = orc.extract(frames[0])
    ko = lo = 0
    for i, f in enumerate(range(1, B)):
        k, desc = orc.extract(frames[f])
        assert n[i] == len(k)
        assert np.array_equal(d["keypoints"][ko:ko + n[i]], np.stack([k[c].astype(np.float32) for c in k.dtype.names], -1)), f
        assert np.array_equal(d["descriptors"][ko:ko + n[i]], desc), f
        (k1, d1), (k2, d2) = prev, (k, desc)
        fv1 = oracle.feature_vector_csr(oracle.bow_assign(d1, voc)); fv2 = oracle.feature_vector_csr(oracle.bow_assign(d2, voc))
        n_o, m_o = oracle.search_by_bow(d1, d2, fv1, fv2, np.ones(len(d1), np.uint8), k1["angle"], k2["angle"], bench.NNRATIO, True)
        assert d["point_match_counts"][i] == n_o and np.array_equal(d["point_matches"][i, :n[i]], m_o) and (d["point_matches"][i, n[i]:] == -1).all(), f

        assert nl[i] == nl_h[f]
        kl = kl_h[f, :nl[i]]
        assert np.array_equal(d["keylines"][lo:lo + nl[i]], np.stack([kl[c].astype(np.float32) for c in kl.dtype.names], -1)), f
        assert np.array_equal(d["line_descriptors"][lo:lo + nl[i]], ld_h[f, :nl[i]]) and np.array_equal(d["line_equations"][lo:lo + nl[i]], eq_h[f, :nl[i]]), f
        n_o, m_o = oracle.line_match(0, ld_h[f - 1, :nl_h[f - 1]], ld_h[f, :nl[i]], np.ones(nl_h[f - 1], np.uint8), None)
        assert d["line_match_counts"][i] == n_o and np.array_equal(d["line_matches"][i, :nl[i]], m_o), f
        prev = (k, desc); ko += n[i]; lo += nl[i]
