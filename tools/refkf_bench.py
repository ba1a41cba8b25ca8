"""Reference-keyframe matching on one GPU (sslpl_match_ref_kf_batch_device): prints one JSON line.

One step: ORB + LSD/LBD extraction of a 513-frame 640x480 batch on the device, K of its frames stored in a keyframe set (masks with
about 70 % of the features / lines set), then every frame matched against its reference keyframe = the latest keyframe before it
(Tracking::TrackReferenceKeyFrame's SearchByBoW + LSDmatcher::SearchByProjection).  For comparison, on the same frames: the
consecutive-pair batch calls (sslpl_match_bow_batch_device_vocab + sslpl_match_lines_batch_device) and the same matching as one
sslpl_search_by_bow + sslpl_line_match (mode 0) call per frame from host buffers, through the Python wrappers.
Times are CUDA events on the one stream all handles run on (host clock for the per-frame calls, which synchronise); median, min
and max over the timed runs after warm-up.  The 513 frames (157 MB) do not fit the 126 MB L2.

usage: python tools/refkf_bench.py [--runs 10] [--warmup 3] [--keyframes 8,32]"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tools"))

W, H, B, NF, NL, LEVELSUP = 640, 480, 513, 1000, 40, 1       # a k=10, L=3 tree at levelsup 1 = ORBvoc's node level at levelsup 4 (101 nodes)


def stats(xs):
    xs = sorted(xs)
    return {"median": round(float(np.median(xs)), 3), "min": round(xs[0], 3), "max": round(xs[-1], 3), "runs": len(xs)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--runs", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--keyframes", default="8,32")
    ap.add_argument("--single-runs", type=int, default=3)
    a = ap.parse_args()
    import torch
    import synth
    import __graft_entry__ as g
    if not torch.cuda.is_available():
        sys.exit("refkf_bench: no CUDA device")
    pkg = g.load_package()
    frames = synth.batch(W, H, B)
    dfr = torch.from_numpy(frames).cuda()
    ext = pkg.ORBextractor(NF, 1.2, 8, 20, 7, max_width=W, max_height=H, max_batch=B)
    ls = pkg.LineSegment(NL, max_width=W, max_height=H, max_batch=B)
    kk, d, n = ext.extract_batch(frames)                             # host copies for the per-frame calls
    _, ld, _, nl = ls.extract_batch(frames)
    voc = pkg.Vocabulary.random(10, 3, seed=1)
    nc = voc.level_nodes(LEVELSUP)
    st = torch.cuda.Stream()
    mt = pkg.Matcher(max_features=ext.cap, max_lines=NL, max_nodes=nc + 1, max_batch=B)
    for h in (ext, ls, mt):
        h.set_stream(st.cuda_stream)
    rng = np.random.default_rng(0)
    valid = [(rng.random(n[f]) < 0.7).astype(np.uint8) for f in range(B)]
    has_ml = [(rng.random(nl[f]) < 0.7).astype(np.uint8) for f in range(B)]
    i32 = dict(dtype=torch.int32, device="cuda")

    def extract():
        ext.extract_batch_device(dfr.data_ptr(), B, W, H, W, W * H)
        ls.extract_batch_device(dfr.data_ptr(), B, W, H, W, W * H)
        kps, desc, dn, cap = ext.device_results()
        _, ldesc, _, dnl, capl = ls.device_results()
        return kps, desc, dn, cap, ldesc, dnl, capl

    out = {"workload": f"{B} frames {W}x{H}, {NF} ORB features, {NL} lines, vocabulary level of {nc} nodes"}
    kps, desc, dn, cap, ldesc, dnl, capl = extract(); mt.sync()
    # consecutive pairs on the same frames
    pm, pn = torch.empty((B - 1, cap), **i32), torch.empty((B - 1,), **i32)
    plm, pln = torch.empty((B - 1, capl), **i32), torch.empty((B - 1,), **i32)
    with torch.cuda.stream(st):
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        ts = []
        for r in range(a.warmup + a.runs):
            ev[0].record(st)
            mt.match_bow_batch_device_vocab(desc, kps, dn, B, cap, voc, LEVELSUP, 0.9, True, pm.data_ptr(), pn.data_ptr())
            mt.match_lines_batch_device(ldesc, dnl, B, capl, plm.data_ptr(), pln.data_ptr())
            ev[1].record(st); ev[1].synchronize()
            if r >= a.warmup:
                ts.append(ev[0].elapsed_time(ev[1]))
    out["consecutive_pairs_ms"] = stats(ts)

    fvs = []
    for f in range(B):
        _, node, w = mt.bow_transform(voc, d[f, :n[f]], LEVELSUP)
        fvs.append(pkg.Vocabulary.feature_vector(node, w))
    out["per_k"] = {}
    for K in [int(x) for x in a.keyframes.split(",")]:
        kf_frames = [int(round(i * B / K)) for i in range(K)]
        ref = np.array([max([s for s, kf in enumerate(kf_frames) if kf < f], default=-1) for f in range(B)], np.int32)
        d_ref = torch.from_numpy(ref).cuda()
        kfs = pkg.KeyframeSet(K, cap, capl)
        m, nm = torch.empty((B, cap), **i32), torch.empty((B,), **i32)
        lm, nlm = torch.empty((B, capl), **i32), torch.empty((B,), **i32)
        step, match = [], []
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        for r in range(a.warmup + a.runs):
            ev[0].record(st)
            kps, desc, dn, cap, ldesc, dnl, capl = extract()
            for s, f in enumerate(kf_frames):
                kfs.store_device(mt, s, desc, kps, dn, cap, ldesc, dnl, capl, f, voc, LEVELSUP)
            for s, f in enumerate(kf_frames):
                kfs.set_masks(s, valid[f], has_ml[f])                 # host-synchronous: waits for the stores
            ev[1].record(st)
            mt.match_ref_kf_batch_device(kfs, d_ref.data_ptr(), B, desc, kps, dn, cap, ldesc, dnl, capl, voc, LEVELSUP, 0.9, True,
                                         m.data_ptr(), nm.data_ptr(), lm.data_ptr(), nlm.data_ptr())
            ev[2].record(st); ev[2].synchronize()
            if r >= a.warmup:
                step.append(ev[0].elapsed_time(ev[2])); match.append(ev[1].elapsed_time(ev[2]))
        got = (m.cpu().numpy(), nm.cpu().numpy(), lm.cpu().numpy(), nlm.cpu().numpy())
        # the same matching as one host-buffer call pair per frame
        om, lsd = pkg.ORBmatcher(0.9, True, mt), pkg.LSDmatcher(mt)
        single, agree = [], True
        for r in range(1 + a.single_runs):
            t0 = time.perf_counter()
            for f in range(B):
                s = ref[f]
                if s < 0:
                    continue
                kf = kf_frames[s]
                n_p, m_p = om.SearchByBoW(d[kf, :n[kf]], fvs[kf], valid[kf], kk[kf, :n[kf]]["angle"], d[f, :n[f]], fvs[f], kk[f, :n[f]]["angle"])
                n_l, m_l = (lsd.SearchByProjection(ld[kf, :nl[kf]], has_ml[kf], ld[f, :nl[f]]) if nl[f] >= 2 else (0, np.full(nl[f], -1, np.int32)))
                if r == 0:
                    agree &= bool(got[1][f] == n_p and np.array_equal(got[0][f, :n[f]], m_p) and got[3][f] == n_l and np.array_equal(got[2][f, :nl[f]], m_l))
            if r > 0:
                single.append((time.perf_counter() - t0) * 1e3)
        out["per_k"][str(K)] = {"step_ms": stats(step), "match_ms": stats(match), "per_frame_calls_ms": stats(single),
                                "equal_to_per_frame_calls": agree, "point_matches": int(got[1].sum()), "line_matches": int(got[3].sum())}
        kfs.close()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True).stdout
    out["gpu"] = smi.strip().splitlines()[0] if smi.strip() else torch.cuda.get_device_name()
    out["torch_device"] = torch.cuda.get_device_name()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
