#!/usr/bin/env python3
"""bench.py — features+matches/sec of the B200 point/line front-end (BASELINE.json metric).

A "step" is one pass of the hot path over one batch of synthetic frames on every GPU:
ORB extraction (+ line extraction when built) of the rank's frames, vocabulary-node assignment and
SearchByBoW matching of every consecutive frame pair, and one NCCL all-gather of the match tables (N>1).

  workload "batch640" (default; BASELINE.json config 5): 512 frames 640x480 per GPU (+1 halo frame so that the pair
            (last, first-of-next-rank) is local), nFeatures=1000, 8 levels, 40 lines; weak scaling over GPUs
  workload "single1280" (config 4): frames 1280x960, nFeatures=4000, 500 lines, 16 frames per GPU

`value`  : whole-job (features+matches)/s with the frames already resident in HBM (CUDA events, max over ranks)
`e2e`    : same metric through the host-buffer API: pinned-host frames H2D, results D2H, every step
`roofline`: dominant kernel's algorithmic bytes / CUDA-event duration vs MEASURED_PEAKS.json hbm_gbs
`cpu_baseline`: the same step on the host cores with the CPU oracle (port of the reference CPU path)
--impl reference : times the CPU oracle (the reference's OpenCV build is not compilable here, DESIGN.md) on
                   the same config/metric, all host threads.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

# The loops below keep ~30 CUDA streams busy (ten frame / line handles with two streams each, matchers, the gather's stream).  With the
# default of 8 hardware connections streams share queues and falsely serialise (measured: end-to-end step 28.3 ms at 8, 25.8-26.1 ms at 32).
# Must be set before the CUDA context exists.
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import numpy as np

METRIC = "features+matches/sec"
UNIT = "features+matches/s"

WORKLOADS = {
    # BASELINE.json config 5: a batch of 512 synthetic 640x480 frames (per GPU: the job is weak-scaled)
    "batch640": dict(width=640, height=480, nfeatures=1000, frames_per_gpu=512, nlines=40),
    # BASELINE.json config 4: 1280x960, nFeatures=4000, 500 lines
    "single1280": dict(width=1280, height=960, nfeatures=4000, frames_per_gpu=16, nlines=500),
}
NWORDS, NNRATIO = 100, 0.7


def host_cores():
    """Host threads this process can really use: the scheduler affinity mask capped by the cgroup CPU quota (os.cpu_count()
    reports the machine: the 1-GPU lease of round 1 showed 128 CPUs with a 16-CPU cpu.max quota)."""
    try:
        aff = len(os.sched_getaffinity(0))
    except AttributeError:
        aff = os.cpu_count() or 1
    quota = None
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    quota = float(txt[0]) / float(txt[1])
            else:
                q = float(txt[0])
                if q > 0:
                    quota = q / float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            break
        except Exception:
            continue
    eff = aff if quota is None else max(1, min(aff, int(quota + 0.5)))
    return eff, {"os_cpu_count": os.cpu_count(), "sched_affinity": aff, "cgroup_quota_cpus": quota}


def make_config(args, cfg, world, lines=True, ring=None, nsets=None, B=None):
    """The `config` object of the JSON line — the same keys and values in both arms (driver: same_config)."""
    W, H = cfg["width"], cfg["height"]
    total = cfg["frames_per_gpu"]
    per_gpu = total // world if args.scaling == "strong" else total
    c = {"workload": args.workload, "width": W, "height": H, "nfeatures": cfg["nfeatures"], "nlevels": 8,
         "frames_per_gpu": per_gpu, "halo_frames_per_gpu": 1, "pairs_per_gpu": per_gpu, "vocabulary_nodes": NWORDS,
         "lines": cfg["nlines"] if lines else 0, "scaling": args.scaling,
         "parallelism": f"frames sharded x{world}, one all_gather(point+line match tables) per step"}
    return c


def n_input_sets(B, W, H):
    """Distinct input batches the steps cycle through: more than 126 MB in all, so that inputs are never L2-resident."""
    return max(2, int(np.ceil(160e6 / (B * W * H))))


def gen_frames(cfg, rank, nsets, B=None):
    """nsets distinct input batches (so that the inputs cycle through more than the 126 MB L2)."""
    import synth
    B = B or cfg["frames_per_gpu"] + 1
    sets = []
    for s in range(nsets):
        start = (s * 977 + rank) * B * 3
        sets.append(synth.batch(cfg["width"], cfg["height"], B, start=start))
    return sets


# ------------------------------------------------------------------------------------------------
# CPU arm (oracle port of the reference CPU path), all host threads
# ------------------------------------------------------------------------------------------------
def cpu_step(O, cfg, frames, voc, nthreads, lines=True):
    """One step of the workload on the host: returns (features, matches, seconds)."""
    from concurrent.futures import ThreadPoolExecutor
    B = len(frames)
    tl = threading.local()

    def extract(i):
        if not hasattr(tl, "orb"):
            tl.orb = O.OrbOracle(cfg["nfeatures"], 1.2, 8, 20, 7)
            tl.line = O.LineOracle(cfg["nlines"])
        k, d = tl.orb.extract(frames[i])
        node = O.bow_assign(d, voc)
        kl, ld, _ = tl.line.extract(frames[i]) if lines else (np.zeros(0), np.zeros((0, 32), np.uint8), None)
        return k, d, O.feature_vector_csr(node), ld

    def match(i):
        (k1, d1, fv1, l1), (k2, d2, fv2, l2) = res[i], res[i + 1]
        n, _ = O.search_by_bow(d1, d2, fv1, fv2, np.ones(len(d1), np.uint8), k1["angle"], k2["angle"], NNRATIO, True)
        if lines and len(l1) >= 1 and len(l2) >= 2:
            n += O.line_match(0, l1, l2, np.ones(len(l1), np.uint8), None)[0]
        return n

    t0 = time.perf_counter()
    with ThreadPoolExecutor(nthreads) as ex:
        res = list(ex.map(extract, range(B)))
        nm = list(ex.map(match, range(B - 1)))
    dt = time.perf_counter() - t0
    feats = sum(len(r[0]) + len(r[3]) for r in res[:B - 1])
    return feats, sum(nm), dt


def _cv2_worker(job):
    """One host process: cv2's own (SIMD, single-threaded) ORB + LSD on a few frames and brute-force matching of consecutive pairs."""
    import cv2
    cv2.setNumThreads(1)
    frames, nfeat, nlines = job
    orb = cv2.ORB_create(nfeatures=nfeat, scaleFactor=1.2, nlevels=8, edgeThreshold=19, fastThreshold=20)
    lsd = cv2.createLineSegmentDetector(cv2.LSD_REFINE_ADV)
    bf = cv2.BFMatcher(cv2.NORM_HAMMING)
    feats, matches, prev = 0, 0, None
    for k, img in enumerate(frames):
        kps, desc = orb.detectAndCompute(img, None)
        seg = lsd.detect(img)[0]
        nl = 0 if seg is None else min(nlines, len(seg))
        if k + 1 < len(frames):
            feats += len(kps) + nl
        if prev is not None and desc is not None and prev is not None and len(prev) >= 2 and len(desc) >= 2:
            for m in bf.knnMatch(prev, desc, k=2):
                if len(m) == 2 and m[0].distance <= 50 and m[0].distance < 0.7 * m[1].distance:
                    matches += 1
        prev = desc
    return feats, matches


def cv2_baseline(cfg, frames, cores):
    """The second CPU line of SURVEY.md 8(d): what OpenCV's own SIMD code achieves on the same frames — cv2.ORB (not the
    reference's octree selection), cv2's LSD, brute-force 2-NN Hamming with the reference's thresholds; no LBD (opencv_contrib
    is not installed) and no line matching.  One fresh process per host core (no fork of a CUDA / OpenCV parent),
    cv2.setNumThreads(1) in each; throughput = all units / the slowest worker's compute time."""
    import tempfile
    n = len(frames)
    per = max(2, (n + cores - 1) // cores)
    spans = [(i, min(n, i + per + 1)) for i in range(0, n - 1, per)]
    with tempfile.TemporaryDirectory() as td:
        path = os.path.join(td, "frames.npy")
        np.save(path, np.ascontiguousarray(frames))
        procs = [subprocess.Popen([sys.executable, os.path.abspath(__file__), "--cv2-worker", path, str(a), str(b), str(cfg["nfeatures"]), str(cfg["nlines"])],
                                  stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True) for a, b in spans]
        outs = [p.communicate(timeout=600)[0] for p in procs]
    f = m = 0; tmax = 0.0
    for o in outs:
        ff, mm, tt = o.strip().split()[-3:]
        f += int(ff); m += int(mm); tmax = max(tmax, float(tt))
    return {"value": (f + m) / tmax, "unit": UNIT, "cores": len(spans), "kind": "cv2-composed",
            "sample": f"{n - 1} frames+pairs, cv2.ORB_create({cfg['nfeatures']}) + cv2 LSD (REFINE_ADV) + BFMatcher 2-NN, {len(spans)} processes x 1 thread",
            "note": "cv2.ORB's keypoint selection and cv2's brute-force matcher differ from the reference's octree / BoW-gated search; no LBD"}


def cv2_worker_main(argv):
    path, a, b, nfeat, nlines = argv[0], int(argv[1]), int(argv[2]), int(argv[3]), int(argv[4])
    frames = np.load(path)[a:b]
    _cv2_worker((frames[:2], nfeat, nlines))            # warm-up
    t0 = time.perf_counter()
    f, m = _cv2_worker((frames, nfeat, nlines))
    print(f, m, time.perf_counter() - t0)
    return 0


def run_reference(args, cfg):
    """--impl reference: the CPU implementation of the path on the box's host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    import __graft_entry__ as g
    O = g.load_oracle()
    import synth
    cores, core_info = host_cores()
    voc = synth.vocabulary(NWORDS)
    nsample = min(cfg["frames_per_gpu"] + 1, max(9, 4 * cores + 1))      # >= 4 frames per host thread: less tail imbalance
    frames = gen_frames(cfg, 0, 1)[0][:nsample]
    for _ in range(args.warmup):
        cpu_step(O, cfg, frames[:min(len(frames), cores + 1)], voc, cores)
    tot_units, tot_s = 0, 0.0
    for _ in range(args.steps):
        f, m, dt = cpu_step(O, cfg, frames, voc, cores)
        tot_units += f + m; tot_s += dt
    val = tot_units / tot_s
    sample = (f"{nsample - 1} frames+pairs of the {args.workload} workload per step, oracle C++ port (-O3), {cores} threads "
              f"(affinity {core_info['sched_affinity']}, cgroup quota {core_info['cgroup_quota_cpus']})")
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * tot_s / args.steps, "higher_is_better": True, "scaling": args.scaling,
            "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": make_config(args, cfg, args.gpus),
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample, "host": core_info},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))
    return 0


# ------------------------------------------------------------------------------------------------
DUMP_BYTES = 64 * 10**6


def last_step_outputs(pkg, dev_read, B, orb, match, nmatch, lines):
    """--dump-outputs: what a caller of the timed path receives for one step, as float32 (float64: line equations, counts, frame
    indices).  A fixed seeded sample of the step's frames f >= 1, as many as DUMP_BYTES holds at full capacity (so the sample depends on
    the arguments only); for each f its keypoints, descriptors and lines (rows of all sampled frames concatenated, with the counts) and
    the whole match-table rows of the pair (f - 1, f) (-1 = no match)."""
    kps, desc, n, cap = orb
    capl = lines[4] if lines else 0
    per_frame = cap * (7 + 32 + 1) * 4 + capl * ((17 + 32 + 1) * 4 + 3 * 8) + 6 * 8
    S = min(B - 1, DUMP_BYTES // per_frame)
    sel = np.sort(np.random.default_rng(0).choice(np.arange(1, B), S, replace=False))
    rows = lambda a, cnt: np.concatenate([a[i, :c] for i, c in enumerate(cnt)])
    fields = lambda a: np.stack([a[f].astype(np.float32) for f in a.dtype.names], -1)
    n = dev_read(n, np.int32, (B,))[sel]
    out = {"frames": sel.astype(np.float64), "keypoint_counts": n.astype(np.float64),
           "keypoints": fields(rows(dev_read(kps, pkg.KEYPOINT_DTYPE, (B, cap))[sel], n)),
           "descriptors": rows(dev_read(desc, np.uint8, (B, cap, 32))[sel], n).astype(np.float32),
           "point_matches": match.cpu().numpy()[sel - 1].astype(np.float32), "point_match_counts": nmatch.cpu().numpy()[sel - 1].astype(np.float64)}
    if lines:
        kl, ld, eq, nl, capl, lmatch, nlmatch = lines
        nl = dev_read(nl, np.int32, (B,))[sel]
        out.update(line_counts=nl.astype(np.float64),
                   keylines=fields(rows(dev_read(kl, pkg.KEYLINE_DTYPE, (B, capl))[sel], nl)),
                   line_descriptors=rows(dev_read(ld, np.uint8, (B, capl, 32))[sel], nl).astype(np.float32),
                   line_equations=rows(dev_read(eq, np.float64, (B, capl, 3))[sel], nl),
                   line_matches=lmatch.reshape(-1)[:(B - 1) * capl].view(B - 1, capl).cpu().numpy()[sel - 1].astype(np.float32),
                   line_match_counts=nlmatch.cpu().numpy()[sel - 1].astype(np.float64))
    return out


class ClockSampler:
    def __init__(self, device_index):
        self.idx = device_index; self.samples = []; self.proc = None

    def start(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(self.idx), "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            out = self.proc.communicate(timeout=5)[0]
        except Exception:
            out = ""
        sm, mx, reasons = [], [], set()
        for ln in out.strip().splitlines():
            p = [x.strip() for x in ln.split(",")]
            if len(p) < 6:
                continue
            try:
                sm.append(float(p[0])); mx.append(float(p[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons)}


def main():
    if len(sys.argv) > 1 and sys.argv[1] == "--cv2-worker":
        return cv2_worker_main(sys.argv[2:])
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="batch640", choices=list(WORKLOADS))
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: frames_per_gpu frames on every GPU; strong: BASELINE.json config 5 as written, the workload's frames in total, sharded")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-lines", action="store_true", help="ORB + point matching only")
    ap.add_argument("--line-ring", type=int, default=10, help="line / frame handles (streams + workspaces) kept in flight (measured: 10 gives the shortest step, device-resident and end to end; 6, 8, 12, 14 are 1-2 ms slower)")
    ap.add_argument("--walkers-per-sm", type=float, default=0.0, help="per line handle: resident LSD region walkers per SM (0 = one per frame)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed on rank 0 (a fixed sample of its frames, "
                    "at most 64 MB) to DIR/<name>.npy, to compare two builds output for output")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    cfg = WORKLOADS[args.workload]
    if args.impl == "reference":
        return run_reference(args, cfg)

    import torch
    import torch.distributed as dist
    import __graft_entry__ as g
    pkg = g.load_package()
    import synth

    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert world == args.gpus, f"WORLD_SIZE={world} but --gpus {args.gpus}"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        import datetime
        # the only collective is a ~2 MB all-gather per step: one channel with small CTAs is enough, and a small NCCL kernel
        # is dispatched promptly on SMs whose registers are mostly held by resident LSD region walkers
        os.environ.setdefault("NCCL_MAX_NCHANNELS", "1"); os.environ.setdefault("NCCL_NTHREADS", "64")
        dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(seconds=240))   # fail fast, never hang the box

    W, H, NF, Bf, NL = cfg["width"], cfg["height"], cfg["nfeatures"], cfg["frames_per_gpu"], cfg["nlines"]
    if args.scaling == "strong":
        assert Bf % world == 0, "strong scaling: the frames must divide over the GPUs"
        Bf //= world                                    # config 5: 512 frames in total, 512 / N (+ 1 halo frame) per GPU
    LINES = not args.no_lines
    B = Bf + 1                                          # + halo frame (first frame of the next rank's block)
    ext = pkg.ORBextractor(NF, 1.2, 8, 20, 7, max_width=W, max_height=H, max_batch=B, device=local)
    mt = pkg.Matcher(max_features=ext.cap, max_lines=NL, max_nodes=NWORDS, max_batch=B, device=local)
    # Lines: the LSD region walker is order-dependent inside a frame (one warp per frame, latency-bound), so a single
    # batch leaves most of the GPU idle.  A ring of R line handles (own stream + workspace each) keeps the walkers of R
    # consecutive steps in flight while the wide ORB kernels of later steps run — multi-stream pipelining, nothing is skipped:
    # every step's line results are finished (and gathered) before the timed region ends.
    R = max(1, args.line_ring) if LINES else 0
    lsr = [pkg.LineSegment(NL, max_width=W, max_height=H, max_batch=B, device=local) for _ in range(R)]
    lmr = [pkg.Matcher(max_features=64, max_lines=NL, max_nodes=2, max_batch=B, device=local) for _ in range(R)]
    if args.walkers_per_sm > 0:
        nsm = torch.cuda.get_device_properties(local).multi_processor_count
        for l in lsr:
            l.set_max_walkers(max(1, int(round(args.walkers_per_sm * nsm))))
    PRIO = -1 if os.environ.get('SSLPL_BENCH_PRIO', '1') == '1' else 0
    s_pts = torch.cuda.Stream(device=dev, priority=PRIO)   # points: ORB + BoW matching + NCCL + timing events; high priority so that
                                                          # its wide kernels are dispatched ahead of queued region-walker CTAs
    s_lin = [torch.cuda.Stream(device=dev) for _ in range(R)]
    torch.cuda.set_stream(s_pts)
    assert s_pts.cuda_stream != 0
    ext.set_stream(s_pts.cuda_stream); mt.set_stream(s_pts.cuda_stream)
    for r in range(R):
        lsr[r].set_stream(s_lin[r].cuda_stream); lmr[r].set_stream(s_lin[r].cuda_stream)
    cap = ext.cap
    voc = synth.vocabulary(NWORDS)
    d_voc = torch.from_numpy(voc).to(dev)
    nsets = n_input_sets(B, W, H)
    sets = gen_frames(cfg, rank, nsets, B)
    d_sets = [torch.from_numpy(s).to(dev) for s in sets]
    d_match = torch.empty((Bf, cap), dtype=torch.int32, device=dev)
    d_nmatch = torch.empty((Bf,), dtype=torch.int32, device=dev)
    d_lmatch = [torch.empty((Bf, NL), dtype=torch.int32, device=dev) for _ in range(R)]
    d_nlmatch = [torch.zeros((Bf,), dtype=torch.int32, device=dev) for _ in range(R)]
    d_gather = torch.empty((world * Bf, cap), dtype=torch.int32, device=dev) if world > 1 else None
    d_lgather = torch.empty((world * Bf, NL), dtype=torch.int32, device=dev) if world > 1 else None
    class _DevArr:                                      # a torch view of a device array owned by the library
        def __init__(self, ptr, n, typestr="<i4"):
            self.__cuda_array_interface__ = {"shape": (n,), "typestr": typestr, "data": (ptr, False), "version": 2}
    _views = {}
    def dev_i32(ptr, n):                                # (the result arrays exist after the handle's first call: looked up per step, cached)
        if (ptr, n) not in _views:
            _views[(ptr, n)] = torch.as_tensor(_DevArr(int(ptr), n), device=dev)
        return _views[(ptr, n)]
    def dev_read(ptr, dtype, shape):                    # host copy of a device array owned by the library
        nbytes = int(np.prod(shape)) * np.dtype(dtype).itemsize
        return torch.as_tensor(_DevArr(int(ptr), nbytes, "|u1"), device=dev).cpu().numpy().view(dtype).reshape(shape)
    u_pts = torch.zeros((), dtype=torch.int64, device=dev)     # features + matches of the timed loop, summed ON the device,
    u_lin = [torch.zeros((), dtype=torch.int64, device=dev) for _ in range(R)]   # inside the timed region (no separate counting pass)
    pending = [False] * R
    gather = [world > 1]                                # collectives on/off (off in the rank-0-only profiling pass)
    ev_free = [torch.cuda.Event() for _ in range(R)]    # slot r's tables have been consumed (gathered) on s_pts

    # One NCCL all-gather per step (north_star: "a single NCCL all-gather of match tables"): the point table of this step and
    # the line table of the ring slot that has just completed travel together in one [Bf, cap + NL] buffer (batch.PackedGather).
    from sslpl_b200 import batch as sbatch
    GBUF = int(os.environ.get("SSLPL_GATHER_BUFS", "4"))      # buffer sets of the packed all-gather: a rank may run 3 steps ahead of the slowest gather
    pgather = sbatch.PackedGather(Bf, cap, NL, world, dev, nbuf=GBUF) if world > 1 else None

    def finalize_slot(r, defer=False):
        """Join slot r's line results into the points stream; gather them across ranks (now, or with this step's point table)."""
        if not pending[r]:
            return
        s_pts.wait_stream(s_lin[r])
        if gather[0]:
            if defer:
                pgather.stage_lines(d_lmatch[r])
            else:
                dist.all_gather_into_tensor(d_lgather, d_lmatch[r])
        if world > 1:
            ev_free[r].record(s_pts)
        pending[r] = False

    def enqueue_lines_device(r, ptr):
        if world > 1:
            s_lin[r].wait_event(ev_free[r])
        lsr[r].extract_batch_device(ptr, B, W, H, W, W * H)
        _, ldesc, _, nl, capl = lsr[r].device_results()
        lmr[r].match_lines_batch_device(ldesc, nl, B, capl, d_lmatch[r].data_ptr(), d_nlmatch[r].data_ptr())
        with torch.cuda.stream(s_lin[r]):
            u_lin[r] += dev_i32(nl, B)[:Bf].sum() + d_nlmatch[r].sum()
        pending[r] = True

    def enqueue_points():
        kps, desc, n, c = ext.device_results()
        mt.match_bow_batch_device(desc, kps, n, B, c, d_voc.data_ptr(), NWORDS, NNRATIO, True, d_match.data_ptr(), d_nmatch.data_ptr())
        u_pts.add_(dev_i32(n, B)[:Bf].sum() + d_nmatch.sum())
        if gather[0]:
            pgather.gather(d_match)

    def step_device(i):
        fr = d_sets[i % nsets]
        if LINES:
            r = i % R
            finalize_slot(r, defer=True)
            enqueue_lines_device(r, fr.data_ptr())
        ext.extract_batch_device(fr.data_ptr(), B, W, H, W, W * H)
        enqueue_points()

    def drain():
        for r in range(R):
            finalize_slot(r)
        if gather[0]:
            pgather.wait()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def launches_now():
        return ext.launch_count + mt.launch_count + sum(l.launch_count for l in lsr) + sum(m.launch_count for m in lmr)

    # ---- every ring slot is used once before anything is timed (a handle's first call sizes its workspace, uploads tables and sets
    # kernel attributes: setup, not a step) ----
    for i in range(R if LINES else 0):
        step_device(i)
    drain()
    # ---- warm-up, then K timed steps, device-resident inputs ----
    for i in range(args.warmup):
        step_device(i)
    drain()
    ext.sync()
    for l in lsr:
        l.sync()
    u_pts.zero_()
    for u in u_lin:
        u.zero_()
    launches0 = launches_now()
    sampler = ClockSampler(local)
    barrier()
    if rank == 0:
        sampler.start()
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(args.steps):
        step_device(args.warmup + i)
    drain()
    e1.record()
    barrier()
    ms_total = e0.elapsed_time(e1)
    ext.sync()
    for l in lsr:
        l.sync()
    launches = launches_now() - launches0
    dumped = None                                       # read back now: the passes below reuse the handles' result buffers
    if args.dump_outputs and rank == 0:
        r = (args.warmup + args.steps - 1) % R if LINES else 0
        dumped = last_step_outputs(pkg, dev_read, B, ext.device_results(), d_match, d_nmatch,
                                   lsr[r].device_results() + (d_lmatch[r], d_nlmatch[r]) if LINES else None)
    clocks = sampler.stop() if rank == 0 else None
    units_timed = int(u_pts.item()) + sum(int(u.item()) for u in u_lin)      # counted inside the timed region, on the device

    # ---- N > 1: the gathered tables must be the single-GPU tables (every rank checks its rows and all ranks agree) ----
    gather_check = None
    if world > 1:
        torch.cuda.synchronize()
        pts_full, lin_full = pgather.fulls[pgather.last][:, :cap], pgather.fulls[pgather.last][:, cap:]
        mine_ok = bool(torch.equal(pts_full[rank * Bf:(rank + 1) * Bf], d_match))
        hsh = (pgather.fulls[pgather.last].to(torch.int64) * torch.arange(1, pgather.fulls[pgather.last].numel() + 1, device=dev).view_as(pgather.fulls[pgather.last])).sum()
        hmin = hsh.clone(); dist.all_reduce(hmin, op=dist.ReduceOp.MIN)
        hmax = hsh.clone(); dist.all_reduce(hmax, op=dist.ReduceOp.MAX)
        okt = torch.tensor([1 if (mine_ok and hmin.item() == hmax.item()) else 0], device=dev); dist.all_reduce(okt, op=dist.ReduceOp.MIN)
        gather_check = {"rows_of_this_rank_equal_local_table": mine_ok, "all_ranks_hold_the_same_tables": bool(hmin.item() == hmax.item()),
                        "ok_on_every_rank": bool(okt.item()), "checksum": int(hsh.item())}

    # ---- the same small job at every N (SURVEY.md 8(d) config 5: "gathered tables bit-equal to the 1-GPU run"): 64 frame pairs of the
    # synthetic sequence 0..64, split into world contiguous blocks (+ one halo frame each), extracted, matched, all-gathered; the
    # checksum of the gathered [64, cap + NL] table does not depend on N, so the lines printed at N = 1, 2, 4, 8 must agree on it.
    table_check = None
    if 64 % world == 0 and 64 // world + 1 <= B:            # (the handles are sized for the workload's batch: single1280 holds 17 frames)
        G = 64; per = G // world
        d_chk = torch.from_numpy(synth.batch(W, H, per + 1, start=rank * per)).to(dev)
        t_pts = torch.full((per, cap), -1, dtype=torch.int32, device=dev); t_np = torch.zeros((per,), dtype=torch.int32, device=dev)
        t_lin = torch.full((per, max(NL, 1)), -1, dtype=torch.int32, device=dev); t_nl = torch.zeros((per,), dtype=torch.int32, device=dev)
        ext.extract_batch_device(d_chk.data_ptr(), per + 1, W, H, W, W * H)
        kps_, desc_, n_, c_ = ext.device_results()
        mt.match_bow_batch_device(desc_, kps_, n_, per + 1, c_, d_voc.data_ptr(), NWORDS, NNRATIO, True, t_pts.data_ptr(), t_np.data_ptr())
        if LINES:
            s_lin[0].wait_stream(s_pts)
            lsr[0].extract_batch_device(d_chk.data_ptr(), per + 1, W, H, W, W * H)
            _, ld_, _, nl_, capl_ = lsr[0].device_results()
            lmr[0].match_lines_batch_device(ld_, nl_, per + 1, capl_, t_lin.data_ptr(), t_nl.data_ptr())
            s_pts.wait_stream(s_lin[0])
        packed = torch.cat([t_pts, t_lin[:, :NL]], 1).contiguous() if LINES else t_pts
        if world > 1:
            full = torch.empty((G, packed.shape[1]), dtype=torch.int32, device=dev)
            dist.all_gather_into_tensor(full, packed)
        else:
            full = packed
        wts = torch.arange(1, full.numel() + 1, device=dev, dtype=torch.int64).view_as(full)
        table_check = {"frames": "synthetic 0..64 (64 pairs), %d per GPU + 1 halo" % per, "rows": G, "cols": int(full.shape[1]),
                       "matches": int((full >= 0).sum().item()), "checksum": int(((full.to(torch.int64) + 2) * wts).sum().item())}
        ext.sync()
        for l in lsr[:1]:
            l.sync()

    units = units_timed
    t = torch.tensor([ms_total, float(units)], dtype=torch.float64, device=dev)
    if world > 1:
        tmax = t.clone(); dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        tsum = t.clone(); dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
        ms_total, units_all = float(tmax[0]), float(tsum[1])
    else:
        units_all = float(units)
    value = units_all / (ms_total * 1e-3)

    # ---- in-pipeline attribution (rank 0, outside the timed regions): CUPTI kernel intervals of a few steps of the SAME pipelined
    # device loop -> time per kernel per step and the union of GPU-busy time (the serial stage times of `roofline` cannot say
    # how much of a pipelined step is the region walker)
    in_pipeline = None
    if rank == 0 and not os.environ.get("SSLPL_BENCH_NO_TRACE"):
        try:
            from torch.profiler import profile, ProfilerActivity
            NT = 6
            gather_was = gather[0]; gather[0] = False       # rank 0 alone: no collectives in this pass
            torch.cuda.synchronize()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for i in range(NT):
                    step_device(args.warmup + i)
                drain(); torch.cuda.synchronize()
            gather[0] = gather_was
            evs = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
            iv = sorted((e.time_range.start, e.time_range.end, e.name) for e in evs)
            if iv:
                t0, t1 = iv[0][0], max(bb for _, bb, _ in iv)
                busy = 0.0; cur_a, cur_b = iv[0][0], iv[0][1]
                for a_, b_, _ in iv[1:]:
                    if a_ > cur_b:
                        busy += cur_b - cur_a; cur_a, cur_b = a_, b_
                    else:
                        cur_b = max(cur_b, b_)
                busy += cur_b - cur_a
                per = {}
                for a_, b_, n_ in iv:
                    k = n_.split("(")[0].split("::")[-1][:40]; per[k] = per.get(k, 0.0) + (b_ - a_)
                top = sorted(per.items(), key=lambda kv: -kv[1])[:12]
                in_pipeline = {"steps": NT, "wall_ms_per_step": (t1 - t0) / 1e3 / NT, "gpu_busy_union_ms_per_step": busy / 1e3 / NT,
                               "kernel_ms_per_step": {k: round(v / 1e3 / NT, 3) for k, v in top},
                               "how": "torch.profiler (CUPTI) over the pipelined device loop; kernels of different streams overlap, so the sums exceed the wall time"}
        except Exception as e:
            in_pipeline = {"unavailable": repr(e)[:200]}
    # ---- roofline of the dominant kernel (rank 0): CUDA events between the kernels of one handle ----
    roofline = None
    nkp_avg = float(dev_i32(ext.device_results()[2], B)[:Bf].float().mean().item())
    if rank == 0:
        gather[0] = False                               # this pass runs on rank 0 only: no collectives
        ext.set_profiling(True)
        if LINES:
            lsr[0].set_profiling(True)
        acc = {}
        nprof = 5
        for i in range(nprof):                          # serial: one handle at a time, so that the stage times are clean
            fr = d_sets[i % nsets]
            ext.extract_batch_device(fr.data_ptr(), B, W, H, W, W * H); ext.sync()
            st = dict(ext.stage_ms())
            if LINES:
                lsr[0].extract_batch_device(fr.data_ptr(), B, W, H, W, W * H); lsr[0].sync()
                st.update(lsr[0].stage_ms())
            for k, v in st.items():
                acc[k] = acc.get(k, 0.0) + v / nprof
        ext.set_profiling(False)
        if LINES:
            lsr[0].set_profiling(False)
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0)); which = "measured" if "hbm_gbs" in peaks else "fallback"
        P = sum(ext.level_size(l)[0] * ext.level_size(l)[1] for l in range(8))
        ncand = 0
        for l in range(8):
            ncand += len(ext.candidates(l, frame=0)[0])
        alg = {   # algorithmic bytes per frame, SURVEY.md 8(d) byte table
            "pyramid": 2 * P - W * H - ext.level_size(7)[0] * ext.level_size(7)[1],
            "fast": P + 5 * ncand,              # the FAST+NMS stage figure: read the pyramid once, write the candidates
            "blur": 2 * P,
            "orient_desc": (749 + 512 + 32 + 28 + 4) * nkp_avg,
            "octree": 8 * ncand,
            # line path, S = scaled pixels (0.64 W H): SURVEY.md 8(d)
            "lsd_prep": W * H + 2 * int(0.64 * W * H) + 2 * W * H,
            "lsd_ll_angle": int(0.64 * W * H) * (1 + 4 + 16 + 8 + 8),   # read u8, write angle, packed record, seed cos/sin, norm
            "lsd_seeds": int(0.64 * W * H) * (8 + 8) + 4 * int(0.3 * 0.64 * W * H),   # norm read twice, seed list written
            "lsd_regions": 17 * int(0.64 * W * H),          # SURVEY.md 8(d): angle + modgrad + used of the visited pixels, <= 17 S (latency-bound stage)
            "lsd_nfa": 4 * int(0.64 * W * H),
            "keylines_lbd": W * H + 8 * W * H + 63 * 4 * 60 * NL,
        }
        dom = max(acc, key=acc.get)
        achieved = alg.get(dom, 0) * B / (acc[dom] * 1e-3) / 1e9
        # dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed `ncu --set full` captures of the same
        # 513-frame batch (profiles/r01_ncu_k_lsd_regions_513_final.md, profiles/r01_ncu_orb_kernels_final.md); bytes
        ncu_traffic = {}
        try:                                            # written by tools/ncu_summary.py from the round's ncu capture of this workload
            tj = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
            ncu_traffic = tj.get(f"{args.workload}:{B}", {})
        except Exception:
            pass
        roofline = {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                    "traffic": ncu_traffic.get(dom), "traffic_unit": "bytes per launch (ncu dram read+write, profiles/ncu_traffic.json)", "peak_source": which, "stage_ms": acc,
                    "algorithmic_bytes_per_launch": alg.get(dom, 0) * B,
                    "note": ("lsd_regions is the order-dependent LSD region stage: latency / issue bound, reported against HBM "
                             "with SURVEY 8(d)'s 17 S bytes per frame" if dom == "lsd_regions" else ""),
                    "stage_gbs": {k: alg.get(k, 0) * B / (acc[k] * 1e-3) / 1e9 for k in acc}}

    # ---- e2e: pinned host frames -> ONE H2D per step -> kernels -> D2H of keypoints, descriptors, lines, counts, match tables ----
    # Through the frame-level entry point (sslpl_frame_extract_batch_begin: what Frame::Frame does with the two extractors): a ring of
    # FR frame handles, each with its ORB stream and its line stream fed by one upload, so that the upload of step i+1 overlaps the
    # kernels of step i and the region walkers of FR steps are in flight together.  Every step's results are read back into pinned
    # host memory and consumed (counted) on the host inside the timed region.
    nkp_avg_dev = float(dev_i32(ext.device_results()[2], B)[:Bf].float().mean().item())
    mt.close()
    for m_ in lmr:                # matchers first: they run on the extractors' streams
        m_.close()
    ext.close()
    for l in lsr:
        l.close()
    h_sets = []
    for s_ in sets:
        hp = pkg.host_alloc(s_.shape, np.uint8); hp[...] = s_; h_sets.append(hp)
    FR = max(2, R) if LINES else 2
    frs = [pkg.Frame(NF, 1.2, 8, 20, 7, NL, max_width=W, max_height=H, max_batch=B, device=local) for _ in range(FR)]
    mts = [pkg.Matcher(max_features=cap, max_lines=NL, max_nodes=NWORDS, max_batch=B, device=local) for _ in range(FR)]
    lms = [pkg.Matcher(max_features=64, max_lines=NL, max_nodes=2, max_batch=B, device=local) for _ in range(FR)]
    so = [torch.cuda.ExternalStream(frs[k].stream(0), device=dev) for k in range(FR)]      # the handles' own ORB / line streams
    sl = [torch.cuda.ExternalStream(frs[k].stream(1), device=dev) for k in range(FR)]
    for k in range(FR):
        mts[k].set_stream(frs[k].stream(0)); lms[k].set_stream(frs[k].stream(1))
    h_res = [dict(keys=pkg.host_alloc((B, cap), pkg.KEYPOINT_DTYPE), desc=pkg.host_alloc((B, cap, 32), np.uint8), n=pkg.host_alloc((B,), np.int32),
                  keylines=pkg.host_alloc((B, NL), pkg.KEYLINE_DTYPE), ldesc=pkg.host_alloc((B, NL, 32), np.uint8),
                  lineeq=pkg.host_alloc((B, NL, 3), np.float64), nl=pkg.host_alloc((B,), np.int32)) for _ in range(FR)]
    dm = [torch.empty((Bf, cap), dtype=torch.int32, device=dev) for _ in range(FR)]; dnm = [torch.empty((Bf,), dtype=torch.int32, device=dev) for _ in range(FR)]
    dl = [torch.empty((Bf, NL), dtype=torch.int32, device=dev) for _ in range(FR)]; dnl = [torch.zeros((Bf,), dtype=torch.int32, device=dev) for _ in range(FR)]
    h_match = [torch.empty((Bf, cap), dtype=torch.int32).pin_memory() for _ in range(FR)]
    h_nmatch = [torch.empty((Bf,), dtype=torch.int32).pin_memory() for _ in range(FR)]
    h_lmatch = [torch.empty((Bf, NL), dtype=torch.int32).pin_memory() for _ in range(FR)]
    h_nlmatch = [torch.zeros((Bf,), dtype=torch.int32).pin_memory() for _ in range(FR)]
    busy = [False] * FR
    pg_e = [sbatch.PackedGather(Bf, cap, NL, world, dev, nbuf=GBUF) for _ in range(FR)] if world > 1 else [None] * FR

    def e2e_finalize(k):
        """Host-side completion of ring slot k: both streams of the handle have finished, the results are in pinned host memory."""
        if not busy[k]:
            return 0
        frs[k].sync()                                                          # ORB + line streams, deferred device error checks
        busy[k] = False
        u = int(h_res[k]["n"][:Bf].sum()) + int(h_nmatch[k].sum())
        if LINES:
            u += int(h_res[k]["nl"][:Bf].sum()) + int(h_nlmatch[k].sum())
        if world > 1:                                                          # both tables of this step in ONE all-gather, on the gather's own stream
            with torch.cuda.stream(so[k]):
                pg_e[k].stage_lines(dl[k]); pg_e[k].gather(dm[k])
        return u

    def step_e2e(i):
        k = i % FR
        u = e2e_finalize(k)
        if world > 1:
            with torch.cuda.stream(so[k]):
                pg_e[k].wait()                                                 # the tables of this slot's previous step have been gathered
        frs[k].extract_batch_begin(h_sets[i % nsets], h_res[k])                # one H2D, ORB and LSD+LBD on two streams, D2H enqueued
        kps, desc, n, c = frs[k].orb.device_results()
        mts[k].match_bow_batch_device(desc, kps, n, B, c, d_voc.data_ptr(), NWORDS, NNRATIO, True, dm[k].data_ptr(), dnm[k].data_ptr())
        with torch.cuda.stream(so[k]):
            h_match[k].copy_(dm[k], non_blocking=True); h_nmatch[k].copy_(dnm[k], non_blocking=True)
        if LINES:
            _, ldesc, _, nl, capl = frs[k].line.device_results()
            lms[k].match_lines_batch_device(ldesc, nl, B, capl, dl[k].data_ptr(), dnl[k].data_ptr())
            with torch.cuda.stream(sl[k]):
                h_lmatch[k].copy_(dl[k], non_blocking=True); h_nlmatch[k].copy_(dnl[k], non_blocking=True)
        busy[k] = True
        return u

    def e2e_drain():
        u = sum(e2e_finalize(k) for k in range(FR))
        if world > 1:
            for pg in pg_e:
                pg.wait()
            torch.cuda.synchronize()
        return u

    # units of every distinct input set (untimed, host count): one synchronous pass per set; must equal the device-side count
    per_set = []
    for sidx in range(nsets):
        per_set.append(step_e2e(sidx) + e2e_drain())
    assert units_timed == sum(per_set[(args.warmup + i) % nsets] for i in range(args.steps)), "device count != host count of the same steps"

    for i in range(FR):                                  # every frame handle of the ring has been through one call before the timed region
        step_e2e(i)
    e2e_drain()
    for i in range(args.warmup):
        step_e2e(i)
    e2e_drain()
    barrier()
    e0.record()
    eu = 0
    for i in range(args.steps):
        eu += step_e2e(args.warmup + i)
    eu += e2e_drain()
    e1.record()
    barrier()
    e2e_ms = max(e0.elapsed_time(e1), 0.0)
    t = torch.tensor([e2e_ms, float(eu)], dtype=torch.float64, device=dev)
    if world > 1:
        tmax = t.clone(); dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        tsum = t.clone(); dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
        e2e_ms, eu_all = float(tmax[0]), float(tsum[1])
    else:
        eu_all = float(eu)
    h2d = B * W * H                                     # ONE upload per step (the frame-level entry point feeds both extractors)
    d2h = B * cap * (28 + 32) + B * 4 + Bf * cap * 4 + Bf * 4 + (B * NL * (68 + 32 + 24) + B * 4 + Bf * NL * 4 + Bf * 4 if LINES else 0)

    # ---- CPU baseline on the host cores (rank 0, N=1 only) ----
    cpu = None; cpu_cv2 = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        O = g.load_oracle()
        cores, core_info = host_cores()
        ns = min(B, max(9, 4 * cores + 1))              # >= 4 frames per host thread: less tail imbalance
        cpu_step(O, cfg, sets[0][:min(ns, cores + 1)], voc, cores, LINES)
        best = None
        for _ in range(2):
            f, m, dt = cpu_step(O, cfg, sets[0][:ns], voc, cores, LINES)
            v = (f + m) / dt
            best = v if best is None or v > best else best
        cpu = {"value": best, "unit": UNIT, "cores": cores, "kind": "port", "host": core_info,
               "sample": f"{ns - 1} frames+pairs of the {args.workload} workload, oracle C++ port, {cores} threads, best of 2"}
        try:
            cpu_cv2 = cv2_baseline(cfg, sets[0][:ns], cores)
        except Exception as e:                          # the second CPU line must never cost the bench line
            cpu_cv2 = {"unavailable": repr(e)[:200]}

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
                "dtype": "u8", "data": "synthetic",
                "config": make_config(args, cfg, world, LINES),
                "run": {"line_ring": R, "primed": "every ring handle called once before the warm-up steps", "cuda_device_max_connections": os.environ.get("CUDA_DEVICE_MAX_CONNECTIONS"), "e2e_frame_handles": FR, "l2": f"inputs cycle through {nsets} distinct batches ({nsets * B * W * H / 1e6:.0f} MB > 126 MB L2)",
                        "units_counted": "on the device inside the timed region"},
                "e2e": {"value": eu_all / (e2e_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                        "ms_per_step": e2e_ms / args.steps},
                "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu, "cpu_baseline_cv2": cpu_cv2,
                "gather_check": gather_check, "table_check": table_check, "in_pipeline": in_pipeline}
        if dumped:
            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, a in dumped.items():
                np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
        print(json.dumps(line)); sys.stdout.flush()
    # orderly teardown.  The pinned match tables were copied into on the frame handles' streams, and torch records an event on every such
    # stream when it frees a pinned block: they are freed while those streams exist.  The matchers run on the frame handles' streams, so
    # they are closed before the frames.
    torch.cuda.synchronize()
    del h_match, h_nmatch, h_lmatch, h_nlmatch
    torch.cuda.synchronize()
    for m_ in mts + lms:
        m_.close()
    for f_ in frs:
        f_.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    import faulthandler; faulthandler.enable()
    sys.exit(main())
