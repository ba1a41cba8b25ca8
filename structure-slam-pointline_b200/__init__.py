"""structure-slam-pointline_b200 — host-side Python mirror of the reference interface over libsslpl_b200.so.

The product is the C-ABI shared library (include/sslpl.h) built from csrc/*.cu for sm_100a; the C++
adapters with the reference's own class signatures live in host/.  This module is the thin ctypes layer
the tests and bench.py use; its classes carry the reference's names and argument meaning:

    ORBextractor(nfeatures, scaleFactor, nlevels, iniThFAST, minThFAST)   include/ORBextractor.h:45-111
        __call__(image) -> (keypoints, descriptors)                       src/ORBextractor.cc:1043
    LineSegment().ExtractLineSegment(img) -> (keylines, ldesc, keylineFunctions)   src/ExtractLineSegment.cpp:18
    ORBmatcher(nnratio, checkOri).SearchByBoW / SearchForTriangulation    src/ORBmatcher.cc:159,525,660
    LSDmatcher().SearchByProjection / SerachForInitialize / ...           src/LSDmatcher.cpp:143,257,286,329,382

There is no CPU fallback and nothing here imports oracle/: if the CUDA library is missing or no GPU is
present, construction raises.  (The package directory name contains '-', so import it through
`__graft_entry__.load_package()`, which registers it as module `sslpl_b200`.)
"""
import ctypes as C
import os
import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libsslpl_b200.so")

KEYPOINT_DTYPE = np.dtype([("x", "<f4"), ("y", "<f4"), ("size", "<f4"), ("angle", "<f4"), ("response", "<f4"),
                           ("octave", "<i4"), ("class_id", "<i4")])
KEYLINE_DTYPE = np.dtype([("angle", "<f4"), ("class_id", "<i4"), ("octave", "<i4"), ("pt_x", "<f4"), ("pt_y", "<f4"),
                          ("response", "<f4"), ("size", "<f4"),
                          ("startPointX", "<f4"), ("startPointY", "<f4"), ("endPointX", "<f4"), ("endPointY", "<f4"),
                          ("sPointInOctaveX", "<f4"), ("sPointInOctaveY", "<f4"),
                          ("ePointInOctaveX", "<f4"), ("ePointInOctaveY", "<f4"),
                          ("lineLength", "<f4"), ("numOfPixels", "<i4")])
assert KEYPOINT_DTYPE.itemsize == 28 and KEYLINE_DTYPE.itemsize == 68


class SslplError(RuntimeError):
    pass


class OrbParams(C.Structure):
    _fields_ = [("nfeatures", C.c_int), ("scaleFactor", C.c_float), ("nlevels", C.c_int), ("iniThFAST", C.c_int),
                ("minThFAST", C.c_int), ("max_width", C.c_int), ("max_height", C.c_int), ("max_batch", C.c_int),
                ("device", C.c_int)]


class MatcherParams(C.Structure):
    _fields_ = [("max_features", C.c_int), ("max_lines", C.c_int), ("max_nodes", C.c_int), ("max_batch", C.c_int),
                ("device", C.c_int)]


class LineParams(C.Structure):
    _fields_ = [("lsdNFeatures", C.c_int), ("max_width", C.c_int), ("max_height", C.c_int), ("max_batch", C.c_int),
                ("device", C.c_int)]


class FeatVec(C.Structure):
    _fields_ = [("nodes", C.c_void_p), ("off", C.c_void_p), ("idx", C.c_void_p), ("nn", C.c_int)]


_lib = None


def lib():
    """Load libsslpl_b200.so (fails loudly when it has not been built: run __graft_entry__.build())."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise SslplError(f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'`"
                             " (there is no CPU fallback)")
        L = C.CDLL(LIB_PATH)
        L.sslpl_last_error.restype = C.c_char_p
        L.sslpl_orb_stream.restype = C.c_void_p
        L.sslpl_orb_launch_count.restype = C.c_longlong
        for name in ("sslpl_matcher_stream", "sslpl_line_stream"):
            if hasattr(L, name):
                getattr(L, name).restype = C.c_void_p
        for name in ("sslpl_matcher_launch_count", "sslpl_line_launch_count"):
            if hasattr(L, name):
                getattr(L, name).restype = C.c_longlong
        _lib = L
    return _lib


def _check(rc):
    if rc != 0:
        raise SslplError(f"sslpl error {rc}: {lib().sslpl_last_error().decode(errors='replace')}")


def _p(a):
    if a is None:
        return None
    if isinstance(a, int):
        return C.c_void_p(a)
    return a.ctypes.data_as(C.c_void_p)


def device_count():
    return int(lib().sslpl_device_count())


def host_alloc(shape, dtype=np.uint8):
    """Pinned host ndarray (sslpl_host_alloc); keeps the allocation alive through .base."""
    dtype = np.dtype(dtype)
    nbytes = int(np.prod(shape)) * dtype.itemsize
    ptr = C.c_void_p()
    _check(lib().sslpl_host_alloc(C.byref(ptr), C.c_size_t(max(nbytes, 1))))
    buf = (C.c_uint8 * max(nbytes, 1)).from_address(ptr.value)
    arr = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)
    return arr


class ORBextractor:
    """Mirror of StructureSLAM::ORBextractor (include/ORBextractor.h:45-111)."""

    def __init__(self, nfeatures=1000, scaleFactor=1.2, nlevels=8, iniThFAST=20, minThFAST=7,
                 max_width=1280, max_height=960, max_batch=1, device=0):
        self.nfeatures, self.scaleFactor, self.nlevels = nfeatures, scaleFactor, nlevels
        p = OrbParams(nfeatures, scaleFactor, nlevels, iniThFAST, minThFAST, max_width, max_height, max_batch, device)
        self._h = C.c_void_p()
        _check(lib().sslpl_orb_create(C.byref(p), C.byref(self._h)))
        self.max_batch = max_batch
        self.cap = int(lib().sslpl_orb_max_keypoints(self._h))

    @classmethod
    def _borrow(cls, ptr, nfeatures, scaleFactor, nlevels, max_batch):
        """A view of an extractor owned by somebody else (Frame): same methods, never destroyed from here."""
        self = cls.__new__(cls)
        self.nfeatures, self.scaleFactor, self.nlevels, self.max_batch = nfeatures, scaleFactor, nlevels, max_batch
        self._h = C.c_void_p(ptr); self._borrowed = True
        self.cap = int(lib().sslpl_orb_max_keypoints(self._h))
        return self

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value and not getattr(self, "_borrowed", False):
            lib().sslpl_orb_destroy(self._h)
            self._h = C.c_void_p()

    __del__ = close

    # ORBextractor.h:60-77
    def GetLevels(self):
        return self.nlevels

    def GetScaleFactor(self):
        return self.scaleFactor

    def _tables(self):
        L = self.nlevels
        sc, isc, s2, is2 = (np.empty(L, np.float32) for _ in range(4))
        nf = np.empty(L, np.int32); um = np.empty(16, np.int32)
        _check(lib().sslpl_orb_tables(self._h, _p(sc), _p(isc), _p(s2), _p(is2), _p(nf), _p(um)))
        return dict(scale=sc, invscale=isc, sigma2=s2, invsigma2=is2, nfeat=nf, umax=um)

    def GetScaleFactors(self):
        return self._tables()["scale"]

    def GetInverseScaleFactors(self):
        return self._tables()["invscale"]

    def GetScaleSigmaSquares(self):
        return self._tables()["sigma2"]

    def GetInverseScaleSigmaSquares(self):
        return self._tables()["invsigma2"]

    def __call__(self, image, mask=None):
        """operator()(image, mask /*ignored*/, keypoints, descriptors) — ORBextractor.cc:1043."""
        if image is None or image.size == 0:
            return np.zeros(0, KEYPOINT_DTYPE), np.zeros((0, 32), np.uint8)      # silent return, ORBextractor.cc:1046
        assert image.dtype == np.uint8 and image.ndim == 2, "CV_8UC1 expected (ORBextractor.cc:1050)"
        if image.strides[1] != 1:
            image = np.ascontiguousarray(image)
        kps = np.zeros(self.cap, KEYPOINT_DTYPE); desc = np.zeros((self.cap, 32), np.uint8)
        n = C.c_int()
        _check(lib().sslpl_orb_extract(self._h, _p(image), image.shape[1], image.shape[0], image.strides[0],
                                       _p(kps), _p(desc), self.cap, C.byref(n)))
        return kps[:n.value].copy(), desc[:n.value].copy()

    def extract_batch(self, frames, out=None):
        """frames: (B,H,W) uint8 host array (pinned for full H2D speed). Returns (kps[B,cap], desc[B,cap,32], n[B])."""
        assert frames.dtype == np.uint8 and frames.ndim == 3 and frames.strides[2] == 1
        B, H, W = frames.shape
        if out is None:
            out = (np.zeros((B, self.cap), KEYPOINT_DTYPE), np.zeros((B, self.cap, 32), np.uint8), np.zeros(B, np.int32))
        kps, desc, n = out
        _check(lib().sslpl_orb_extract_batch(self._h, _p(frames), B, W, H, frames.strides[1], C.c_size_t(frames.strides[0]),
                                             _p(kps), _p(desc), self.cap, _p(n)))
        return kps, desc, n

    def extract_batch_begin(self, frames, out):
        """Asynchronous host-buffer form: returns immediately; `out` (pinned) is valid after sync()."""
        B, H, W = frames.shape
        kps, desc, n = out
        _check(lib().sslpl_orb_extract_batch_begin(self._h, _p(frames), B, W, H, frames.strides[1], C.c_size_t(frames.strides[0]),
                                                   _p(kps), _p(desc), self.cap, _p(n)))

    def extract_batch_device(self, d_ptr, nframes, width, height, pitch, frame_stride):
        """Frames already in HBM (raw device pointer, e.g. torch_tensor.data_ptr()); asynchronous."""
        _check(lib().sslpl_orb_extract_batch_device(self._h, C.c_void_p(d_ptr), nframes, width, height, pitch,
                                                    C.c_size_t(frame_stride)))

    def device_results(self):
        kps = C.c_void_p(); desc = C.c_void_p(); n = C.c_void_p(); cap = C.c_int()
        _check(lib().sslpl_orb_device_results(self._h, C.byref(kps), C.byref(desc), C.byref(n), C.byref(cap)))
        return kps.value, desc.value, n.value, cap.value

    def sync(self):
        _check(lib().sslpl_orb_sync(self._h))

    def set_stream(self, cuda_stream):
        _check(lib().sslpl_orb_set_stream(self._h, C.c_void_p(cuda_stream)))

    @property
    def stream(self):
        return lib().sslpl_orb_stream(self._h)

    @property
    def launch_count(self):
        return int(lib().sslpl_orb_launch_count(self._h))

    # ---- stage intermediates (parity tests) ----
    def level_size(self, l):
        w = C.c_int(); h = C.c_int()
        _check(lib().sslpl_orb_level_size(self._h, l, C.byref(w), C.byref(h)))
        return w.value, h.value

    def level(self, l, frame=0, bordered=False):
        """mvImagePyramid[l] (ORBextractor.h:79)."""
        w, h = self.level_size(l)
        b = 19 if bordered else 0
        out = np.empty((h + 2 * b, w + 2 * b), np.uint8)
        _check(lib().sslpl_orb_download_level(self._h, frame, l, int(bordered), _p(out), out.strides[0]))
        return out

    def blurred(self, l, frame=0):
        w, h = self.level_size(l)
        out = np.empty((h, w), np.uint8)
        _check(lib().sslpl_orb_download_blurred(self._h, frame, l, _p(out), out.strides[0]))
        return out

    def candidates(self, l, frame=0, cap=1 << 17):
        xs = np.empty(cap, np.int32); ys = np.empty(cap, np.int32); rs = np.empty(cap, np.int32); n = C.c_int()
        _check(lib().sslpl_orb_download_candidates(self._h, frame, l, _p(xs), _p(ys), _p(rs), cap, C.byref(n)))
        assert n.value <= cap
        return xs[:n.value].copy(), ys[:n.value].copy(), rs[:n.value].copy()

    def level_keypoints(self, l, frame=0, cap=1 << 15):
        xs = np.empty(cap, np.int32); ys = np.empty(cap, np.int32); rs = np.empty(cap, np.int32); n = C.c_int()
        _check(lib().sslpl_orb_download_level_keypoints(self._h, frame, l, _p(xs), _p(ys), _p(rs), cap, C.byref(n)))
        return xs[:n.value].copy(), ys[:n.value].copy(), rs[:n.value].copy()

    def set_profiling(self, on=True):
        _check(lib().sslpl_orb_set_profiling(self._h, int(on)))

    def stage_ms(self):
        ms = (C.c_float * 16)(); names = (C.c_char_p * 16)(); n = C.c_int()
        _check(lib().sslpl_orb_stage_ms(self._h, ms, 16, names, C.byref(n)))
        return {names[i].decode(): float(ms[i]) for i in range(n.value)}


# =====================================================================================================
# Matching
# =====================================================================================================
def _featvec(fv):
    """(nodes, off, idx) int32 arrays -> FeatVec struct (keeps references alive)."""
    nodes, off, idx = (np.ascontiguousarray(a, np.int32) for a in fv)
    s = FeatVec(_p(nodes) if len(nodes) else None, _p(off), _p(idx) if len(idx) else None, len(nodes))
    s._keep = (nodes, off, idx)
    return s


def feature_vector_csr(node):
    """DBoW2::FeatureVector (std::map<NodeId, vector<unsigned>>; FeatureVector.cpp:31-45) flattened to CSR."""
    node = np.asarray(node, np.int32)
    order = np.argsort(node, kind="stable").astype(np.int32)
    ids, counts = np.unique(node, return_counts=True)
    off = np.zeros(len(ids) + 1, np.int32)
    off[1:] = np.cumsum(counts)
    return ids.astype(np.int32), off, order


class Matcher:
    """Device context shared by ORBmatcher / LSDmatcher below (one stream + workspace; create one per thread)."""

    def __init__(self, max_features=4096, max_lines=512, max_nodes=1024, max_batch=1, device=0):
        p = MatcherParams(max_features, max_lines, max_nodes, max_batch, device)
        self._h = C.c_void_p()
        _check(lib().sslpl_matcher_create(C.byref(p), C.byref(self._h)))
        self.max_features, self.max_lines = max_features, max_lines

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            lib().sslpl_matcher_destroy(self._h)
            self._h = C.c_void_p()

    __del__ = close

    def sync(self):
        _check(lib().sslpl_matcher_sync(self._h))

    def set_stream(self, cuda_stream):
        _check(lib().sslpl_matcher_set_stream(self._h, C.c_void_p(cuda_stream)))

    @property
    def stream(self):
        return lib().sslpl_matcher_stream(self._h)

    @property
    def launch_count(self):
        return int(lib().sslpl_matcher_launch_count(self._h))

    def descriptor_distance(self, a, b):
        a = np.ascontiguousarray(a, np.uint8).reshape(-1, 32); b = np.ascontiguousarray(b, np.uint8).reshape(-1, 32)
        out = np.empty(len(a), np.int32)
        _check(lib().sslpl_descriptor_distance(self._h, _p(a), _p(b), len(a), _p(out)))
        return out

    def knn2(self, q, t):
        """cv::BFMatcher(NORM_HAMMING).knnMatch(q, t, k=2) -> int32 [nq,4] = idx0, d0, idx1, d1."""
        q = np.ascontiguousarray(q, np.uint8).reshape(-1, 32); t = np.ascontiguousarray(t, np.uint8).reshape(-1, 32)
        out = np.empty((len(q), 4), np.int32)
        _check(lib().sslpl_hamming_knn2(self._h, _p(q), len(q), _p(t), len(t), _p(out)))
        return out

    def bow_assign(self, desc, centroids):
        desc = np.ascontiguousarray(desc, np.uint8).reshape(-1, 32); centroids = np.ascontiguousarray(centroids, np.uint8).reshape(-1, 32)
        node = np.empty(len(desc), np.int32)
        _check(lib().sslpl_bow_assign(self._h, _p(desc), len(desc), _p(centroids), len(centroids), _p(node)))
        return node

    def match_bow_batch_device(self, d_desc, d_kps, d_n, nframes, cap, d_centroids, nc, nnratio, check_ori, d_match, d_nmatch):
        _check(lib().sslpl_match_bow_batch_device(self._h, C.c_void_p(d_desc), C.c_void_p(d_kps), C.c_void_p(d_n), nframes, cap,
                                                  C.c_void_p(d_centroids), nc, C.c_float(nnratio), int(check_ori),
                                                  C.c_void_p(d_match), C.c_void_p(d_nmatch)))

    def match_bow_batch_device_vocab(self, d_desc, d_kps, d_n, nframes, cap, vocab, levelsup, nnratio, check_ori, d_match, d_nmatch,
                                     d_word=0, d_node=0, d_weight=0):
        """Batched SearchByBoW with the DBoW2 tree transform (optional per-feature word / node / weight outputs in HBM)."""
        _check(lib().sslpl_match_bow_batch_device_vocab(self._h, C.c_void_p(d_desc), C.c_void_p(d_kps), C.c_void_p(d_n), nframes, cap,
                                                        vocab._h, int(levelsup), C.c_float(nnratio), int(check_ori),
                                                        C.c_void_p(d_match), C.c_void_p(d_nmatch),
                                                        C.c_void_p(d_word or None), C.c_void_p(d_node or None), C.c_void_p(d_weight or None)))

    def bow_transform(self, vocab, desc, levelsup=4):
        """TemplatedVocabulary::transform per feature (TemplatedVocabulary.h:1218-1259): (word, node, weight) arrays."""
        desc = np.ascontiguousarray(desc, np.uint8).reshape(-1, 32)
        n = len(desc)
        word = np.empty(max(n, 1), np.int32); node = np.empty(max(n, 1), np.int32); w = np.empty(max(n, 1), np.float64)
        _check(lib().sslpl_bow_transform(self._h, vocab._h, _p(desc), n, int(levelsup), _p(word), _p(node), _p(w)))
        return word[:n], node[:n], w[:n]

    def search_by_projection_mps(self, mp, cur, bounds, scale_factors, nnratio=0.8, th=1.0):
        """ORBmatcher::SearchByProjection(Frame&, const vector<MapPoint*>&, th) (ORBmatcher.cc:45-129).
        mp = dict(inview, bad, obs, projx, projy, level, viewcos, desc[, projxr]); cur = dict(desc, x, y, oct[, uright, held])."""
        f32 = lambda a: np.ascontiguousarray(a, np.float32); u8 = lambda a: np.ascontiguousarray(a, np.uint8)
        nmp = len(mp["inview"]); n2 = len(cur["x"])
        iv, bad, obs = u8(mp["inview"]), u8(mp["bad"]), u8(mp["obs"])
        px, py = f32(mp["projx"]), f32(mp["projy"]); pxr = f32(mp["projxr"]) if mp.get("projxr") is not None else None
        lv = np.ascontiguousarray(mp["level"], np.int32); vc = f32(mp["viewcos"]); dmp = u8(mp["desc"]).reshape(-1, 32)
        d2 = u8(cur["desc"]).reshape(-1, 32); x2, y2 = f32(cur["x"]), f32(cur["y"]); oc2 = np.ascontiguousarray(cur["oct"], np.int32)
        ur = f32(cur["uright"]) if cur.get("uright") is not None else None
        held = u8(cur["held"]) if cur.get("held") is not None else None
        sf = f32(scale_factors); out = np.full(max(n2, 1), -1, np.int32); nm = C.c_int()
        _check(lib().sslpl_search_by_projection_mps(self._h, nmp, _p(iv), _p(bad), _p(obs), _p(px), _p(py), _p(pxr) if pxr is not None else None,
                                                    _p(lv), _p(vc), _p(dmp), n2, _p(d2), _p(x2), _p(y2), _p(oc2), _p(ur) if ur is not None else None,
                                                    _p(held) if held is not None else None, _p(f32(bounds)), _p(sf), len(sf),
                                                    C.c_float(nnratio), C.c_float(th), _p(out), C.byref(nm)))
        return nm.value, out[:n2]

    def line_search_by_projection(self, q, obs, dml, ld2, kl2, oct2, held2=None, nnratio=0.8):
        """Search stage of LSDmatcher::SearchByProjection(Frame&, const Frame&, th, bMono) (LSDmatcher.cpp:98-137) and of
        LSDmatcher::SearchByProjection(Frame&, const vector<MapLine*>&, th) (:210-251).  q = dict(active, proj[n,4], radius, min_level,
        max_level) per MapLine (the projection stage's outputs), obs = Observations() > 0, dml their descriptors; ld2 / kl2[n,3] (pt.x,
        pt.y, angle) / oct2 / held2 the frame's lines -> (nmatches, assign2)."""
        f32 = lambda a: np.ascontiguousarray(a, np.float32); u8 = lambda a: np.ascontiguousarray(a, np.uint8); i32 = lambda a: np.ascontiguousarray(a, np.int32)
        nml = len(q["active"]); nl2 = len(oct2)
        out = np.full(max(nl2, 1), -1, np.int32); nm = C.c_int()
        _check(lib().sslpl_line_search_by_projection(self._h, nml, _p(u8(q["active"])), _p(u8(obs)), _p(f32(q["proj"])), _p(f32(q["radius"])),
                                                     _p(i32(q["min_level"])), _p(i32(q["max_level"])), _p(u8(dml)), nl2, _p(u8(ld2)), _p(f32(kl2)), _p(i32(oct2)),
                                                     _p(u8(held2)) if held2 is not None else None, C.c_float(nnratio), _p(out), C.byref(nm)))
        return nm.value, out[:nl2]

    def fuse_lines_search(self, q, dml, ld2, kl2, oct2, scale_factors, th=3.0):
        """Search stage of LSDmatcher::Fuse (LSDmatcher.cpp:495-523).  q = dict(active, proj[n,4], level) -> (best_idx, best_dist)."""
        f32 = lambda a: np.ascontiguousarray(a, np.float32); u8 = lambda a: np.ascontiguousarray(a, np.uint8); i32 = lambda a: np.ascontiguousarray(a, np.int32)
        n = len(q["active"]); sf = f32(scale_factors)
        bi = np.full(max(n, 1), -1, np.int32); bd = np.full(max(n, 1), 0x7fffffff, np.int32)
        _check(lib().sslpl_fuse_lines_search(self._h, n, _p(u8(q["active"])), _p(f32(q["proj"])), _p(i32(q["level"])), _p(u8(dml)), len(oct2), _p(u8(ld2)),
                                             _p(f32(kl2)), _p(i32(oct2)), _p(sf), len(sf), C.c_float(th), _p(bi), _p(bd)))
        return bi[:n], bd[:n]

    def fuse_points_search(self, q, dmp, d2, x2, y2, oct2, uright2, bounds, scale_factors, inv_level_sigma2, th=3.0):
        """Search stage of ORBmatcher::Fuse (ORBmatcher.cc:889-950).  q = dict(active, u, v, ur, level) -> (best_idx, best_dist)."""
        f32 = lambda a: np.ascontiguousarray(a, np.float32); u8 = lambda a: np.ascontiguousarray(a, np.uint8); i32 = lambda a: np.ascontiguousarray(a, np.int32)
        n = len(q["active"]); sf = f32(scale_factors)
        bi = np.full(max(n, 1), -1, np.int32); bd = np.full(max(n, 1), 256, np.int32)
        ur2 = f32(uright2) if uright2 is not None else None
        _check(lib().sslpl_fuse_points_search(self._h, n, _p(u8(q["active"])), _p(f32(q["u"])), _p(f32(q["v"])), _p(f32(q["ur"])), _p(i32(q["level"])), _p(u8(dmp)),
                                              len(x2), _p(u8(d2)), _p(f32(x2)), _p(f32(y2)), _p(i32(oct2)), _p(ur2) if ur2 is not None else None,
                                              _p(f32(bounds)), _p(sf), _p(f32(inv_level_sigma2)), len(sf), C.c_float(th), _p(bi), _p(bd)))
        return bi[:n], bd[:n]

    def search_for_initialization(self, d1, k1, d2, k2, prev, bounds, nnratio=0.9, check_ori=True, window=100):
        """ORBmatcher::SearchForInitialization (ORBmatcher.cc:408-523) -> (nmatches, matches12, prev_out)."""
        f32 = lambda a: np.ascontiguousarray(a, np.float32)
        d1 = np.ascontiguousarray(d1, np.uint8).reshape(-1, 32); d2 = np.ascontiguousarray(d2, np.uint8).reshape(-1, 32)
        prev = f32(prev).reshape(-1, 2).copy()
        m12 = np.full(max(len(k1), 1), -1, np.int32); nm = C.c_int()
        _check(lib().sslpl_search_for_initialization(self._h, len(k1), _p(d1), _p(np.ascontiguousarray(k1["octave"], np.int32)), _p(f32(k1["angle"])), _p(prev),
                                                     len(k2), _p(d2), _p(f32(k2["x"])), _p(f32(k2["y"])), _p(np.ascontiguousarray(k2["octave"], np.int32)),
                                                     _p(f32(k2["angle"])), _p(f32(bounds)), C.c_float(nnratio), int(check_ori), int(window), _p(m12), C.byref(nm)))
        return nm.value, m12[:len(k1)], prev

    def search_by_projection_frame(self, last, cur, Tcw, Tlw, cam, bounds, scale_factors, th, mono=True, check_ori=True, raw=False):
        """ORBmatcher::SearchByProjection(Frame &CurrentFrame, const Frame &LastFrame, th, bMono) (ORBmatcher.cc:1331-1473).
        last = dict(valid, obs, Xw[n,3], dmp[n,32], oct, angle); cur = dict(desc[n,32], x, y, oct, angle, uright|None, claimed|None);
        Tcw / Tlw 3x4 (or 4x4) row-major; cam = (fx, fy, cx, cy, mbf, mb); bounds = (minX, maxX, minY, maxY).
        Returns (nmatches, assign2) with assign2[j] = index of the last-frame MapPoint given to current feature j or -1."""
        f32 = lambda a: np.ascontiguousarray(a, np.float32)
        n1, n2 = len(last["valid"]), len(cur["x"])
        v1 = np.ascontiguousarray(last["valid"], np.uint8); o1 = np.ascontiguousarray(last["obs"], np.uint8)
        Xw = f32(last["Xw"]).reshape(-1, 3); dmp = np.ascontiguousarray(last["dmp"], np.uint8).reshape(-1, 32)
        oc1 = np.ascontiguousarray(last["oct"], np.int32); a1 = f32(last["angle"])
        d2 = np.ascontiguousarray(cur["desc"], np.uint8).reshape(-1, 32); x2 = f32(cur["x"]); y2 = f32(cur["y"])
        oc2 = np.ascontiguousarray(cur["oct"], np.int32); a2 = f32(cur["angle"])
        ur = f32(cur["uright"]) if cur.get("uright") is not None else None
        cl = np.ascontiguousarray(cur["claimed"], np.uint8) if cur.get("claimed") is not None else None
        Tc = f32(Tcw).reshape(-1)[:12].copy(); Tl = f32(Tlw).reshape(-1)[:12].copy() if Tlw is not None else None
        camv = f32(cam); bnd = f32(bounds); sf = f32(scale_factors)
        out = np.full(max(n2, 1), -1, np.int32); nm = C.c_int()
        _check(lib().sslpl_search_by_projection_frame(self._h, n1, _p(v1), _p(o1), _p(Xw), _p(dmp), _p(oc1), _p(a1),
                                                      n2, _p(d2), _p(x2), _p(y2), _p(oc2), _p(a2), _p(ur), _p(cl), _p(Tc), _p(Tl),
                                                      _p(camv), _p(bnd), _p(sf), len(sf), C.c_float(th), int(mono), int(check_ori),
                                                      _p(out), C.byref(nm)))
        # -2 = assigned, then removed by the rotation check (the reference writes NULL there, ORBmatcher.cc:1461); -1 = never assigned
        return nm.value, (out[:n2] if raw else np.where(out[:n2] == -2, -1, out[:n2]).astype(np.int32))

    def descriptor_medoid(self, desc, off):
        """ComputeDistinctiveDescriptors (MapPoint.cc:247-312 / MapLine.cpp:246-317) for CSR groups of descriptors."""
        desc = np.ascontiguousarray(desc, np.uint8).reshape(-1, 32); off = np.ascontiguousarray(off, np.int32)
        ng = len(off) - 1
        bi = np.empty(max(ng, 1), np.int32); bm = np.empty(max(ng, 1), np.int32)
        _check(lib().sslpl_descriptor_medoid_batch(self._h, _p(desc), _p(off), ng, _p(bi), _p(bm)))
        return bi[:ng], bm[:ng]

    def match_lines_batch_device(self, d_ldesc, d_nl, nframes, capl, d_lmatch, d_nlmatch):
        _check(lib().sslpl_match_lines_batch_device(self._h, C.c_void_p(d_ldesc), C.c_void_p(d_nl), nframes, capl,
                                                    C.c_void_p(d_lmatch), C.c_void_p(d_nlmatch)))

    def match_ref_kf_batch_device(self, kfset, d_ref, nframes, d_desc, d_kps, d_n, cap, d_ldesc, d_nl, capl, vocab, levelsup,
                                  nnratio, check_ori, d_match, d_nmatch, d_lmatch, d_nlmatch):
        """Tracking::TrackReferenceKeyFrame's two matchers for every frame f of a device batch against keyframe slot d_ref[f]
        (-1 = none): SearchByBoW -> d_match[f, j] / d_nmatch[f], LSDmatcher::SearchByProjection -> d_lmatch[f, t] / d_nlmatch[f]."""
        _check(lib().sslpl_match_ref_kf_batch_device(self._h, kfset._h, C.c_void_p(d_ref), nframes, C.c_void_p(d_desc), C.c_void_p(d_kps),
                                                     C.c_void_p(d_n), cap, C.c_void_p(d_ldesc), C.c_void_p(d_nl), capl, vocab._h, int(levelsup),
                                                     C.c_float(nnratio), int(check_ori), C.c_void_p(d_match), C.c_void_p(d_nmatch),
                                                     C.c_void_p(d_lmatch), C.c_void_p(d_nlmatch)))


class Vocabulary:
    """DBoW2 ORB vocabulary tree on the device (the reference's ORBVocabulary = TemplatedVocabulary<FORB::TDescriptor, FORB>,
    include/ORBVocabulary.h; used by Frame::ComputeBoW Frame.cc:474-481 with levelsup = 4).

    Vocabulary(k, L, parent, desc, weight, is_leaf)   from arrays (node 0 = root)
    Vocabulary.load_text(path)                          ORBvoc.txt (TemplatedVocabulary.h:1338-1420)
    Vocabulary.random(k, L, seed)                       synthetic tree for tests / benchmarks"""
    # scoring / weighting enums of DBoW2 (BowVector.h): the defaults of ORBvoc.txt are L1_NORM (0) and TF_IDF (0)
    TF_IDF, TF, IDF, BINARY = 0, 1, 2, 3

    def __init__(self, k, L, parent, desc, weight, is_leaf, device=0, scoring=0, weighting=0):
        self.parent = np.ascontiguousarray(parent, np.int32); self.desc = np.ascontiguousarray(desc, np.uint8).reshape(-1, 32)
        self.weight = np.ascontiguousarray(weight, np.float64); self.is_leaf = np.ascontiguousarray(is_leaf, np.uint8)
        self.k, self.L, self.scoring, self.weighting = int(k), int(L), int(scoring), int(weighting)
        self._h = C.c_void_p()
        _check(lib().sslpl_vocab_create(device, self.k, self.L, len(self.parent), _p(self.parent), _p(self.desc), _p(self.weight),
                                        _p(self.is_leaf), C.byref(self._h)))

    @classmethod
    def load_text(cls, path, device=0):
        self = cls.__new__(cls)
        self._h = C.c_void_p(); sc = C.c_int(); we = C.c_int()
        _check(lib().sslpl_vocab_load_text(device, str(path).encode(), C.byref(self._h), C.byref(sc), C.byref(we)))
        k = C.c_int(); L = C.c_int()
        _check(lib().sslpl_vocab_info(self._h, C.byref(k), C.byref(L), None, None))
        self.k, self.L, self.scoring, self.weighting = k.value, L.value, sc.value, we.value
        self.parent = self.desc = self.weight = self.is_leaf = None
        return self

    @staticmethod
    def random_arrays(k, L, seed=0, stop_fraction=0.0, early_leaf_fraction=0.0):
        """A random k-ary tree of depth L as arrays, in the node order loadFromTextFile produces for a file written level by
        level is NOT required: any order with parent[i] < i works.  Some leaves can be 'stopped' (weight 0) or sit above L."""
        rng = np.random.default_rng(seed)
        parent = [-1]; depth = [0]; frontier = [0]
        for d in range(1, L + 1):
            nxt = []
            for p in frontier:
                if d > 1 and rng.random() < early_leaf_fraction:
                    continue                                        # p stays a leaf above the last level
                for _ in range(k):
                    parent.append(p); depth.append(d); nxt.append(len(parent) - 1)
            frontier = nxt
        n = len(parent)
        parent = np.array(parent, np.int32)
        has_child = np.zeros(n, bool); has_child[parent[1:]] = True
        is_leaf = (~has_child).astype(np.uint8); is_leaf[0] = 0
        desc = rng.integers(0, 256, (n, 32), dtype=np.uint8)
        weight = np.where(is_leaf == 1, rng.random(n) * 5 + 0.1, 0.0)
        weight[(is_leaf == 1) & (rng.random(n) < stop_fraction)] = 0.0
        return parent, desc, weight.astype(np.float64), is_leaf

    @classmethod
    def random(cls, k=10, L=3, seed=0, device=0, **kw):
        parent, desc, weight, is_leaf = cls.random_arrays(k, L, seed, **kw)
        return cls(k, L, parent, desc, weight, is_leaf, device=device)

    def info(self):
        k = C.c_int(); L = C.c_int(); nn = C.c_int(); nw = C.c_int()
        _check(lib().sslpl_vocab_info(self._h, C.byref(k), C.byref(L), C.byref(nn), C.byref(nw)))
        return {"k": k.value, "L": L.value, "nodes": nn.value, "words": nw.value}

    def level_nodes(self, levelsup=4):
        c = C.c_int()
        _check(lib().sslpl_vocab_level_nodes(self._h, int(levelsup), C.byref(c)))
        return c.value

    def bow_vector(self, word, weight):
        """BowVector assembly of TemplatedVocabulary::transform (:1145-1195) from the per-feature arrays: a word -> value map
        (ascending word id), TF_IDF / TF: weights added in feature order then divided by the number of words unless the scoring
        normalises (L1 / L2 scoring types 0, 1 do); IDF / BINARY: first weight kept."""
        bv = {}
        for wid, w in zip(np.asarray(word).tolist(), np.asarray(weight).tolist()):
            if not w > 0:
                continue
            if self.weighting in (self.TF_IDF, self.TF):
                bv[wid] = bv.get(wid, 0.0) + w
            else:
                bv.setdefault(wid, w)
        must, l2 = self.scoring in (0, 1), self.scoring == 1      # L1_NORM, L2_NORM normalise (ScoringObject.cpp)
        keys = sorted(bv)
        if self.weighting in (self.TF_IDF, self.TF) and bv and not must:
            nd = float(len(bv))
            for kk in keys:
                bv[kk] /= nd
        if must and bv:
            norm = 0.0
            for kk in keys:
                norm += bv[kk] * bv[kk] if l2 else abs(bv[kk])
            if l2:
                norm = float(np.sqrt(norm))
            if norm > 0.0:
                for kk in keys:
                    bv[kk] /= norm
        return np.array(keys, np.int32), np.array([bv[kk] for kk in keys], np.float64)

    @staticmethod
    def feature_vector(node, weight):
        """FeatureVector (node id -> ascending feature indices) as CSR, without the stopped words (:1162-1166)."""
        node = np.asarray(node, np.int32); keep = np.nonzero(np.asarray(weight) > 0)[0].astype(np.int32)
        order = keep[np.argsort(node[keep], kind="stable")]
        ids, counts = np.unique(node[keep], return_counts=True)
        off = np.zeros(len(ids) + 1, np.int32); off[1:] = np.cumsum(counts)
        return ids.astype(np.int32), off, order.astype(np.int32)

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            lib().sslpl_vocab_destroy(self._h)
            self._h = C.c_void_p()

    __del__ = close


class KeyframeSet:
    """Reference keyframes kept in HBM for Matcher.match_ref_kf_batch_device (sslpl_kfset): max_keyframes slots of up to `cap`
    features and `capl` lines each, with their FeatureVectors and MapPoint / MapLine masks."""

    def __init__(self, max_keyframes, cap, capl, device=0):
        self._h = C.c_void_p()
        _check(lib().sslpl_kfset_create(device, max_keyframes, cap, capl, C.byref(self._h)))
        self.max_keyframes, self.cap, self.capl = max_keyframes, cap, capl

    def store_device(self, matcher, slot, d_desc, d_kps, d_n, cap, d_ldesc, d_nl, capl, frame, vocab, levelsup):
        """Copy frame `frame` of an extraction batch's device results into `slot` (asynchronous on the matcher's stream)."""
        _check(lib().sslpl_kfset_store_device(matcher._h, self._h, slot, C.c_void_p(d_desc), C.c_void_p(d_kps), C.c_void_p(d_n), cap,
                                              C.c_void_p(d_ldesc), C.c_void_p(d_nl), capl, frame, vocab._h, int(levelsup)))

    def store(self, matcher, slot, desc, angle, ldesc, vocab, levelsup):
        desc = np.ascontiguousarray(desc, np.uint8).reshape(-1, 32); angle = np.ascontiguousarray(angle, np.float32)
        ldesc = np.ascontiguousarray(ldesc, np.uint8).reshape(-1, 32)
        assert len(angle) == len(desc)
        _check(lib().sslpl_kfset_store(matcher._h, self._h, slot, _p(desc), _p(angle), len(desc), _p(ldesc), len(ldesc), vocab._h, int(levelsup)))

    def set_masks(self, slot, valid=None, has_ml=None):
        """valid[i] = feature i holds a non-bad MapPoint, has_ml[j] = line j holds a MapLine (None = all set)."""
        v = np.ascontiguousarray(valid, np.uint8) if valid is not None else None
        h = np.ascontiguousarray(has_ml, np.uint8) if has_ml is not None else None
        _check(lib().sslpl_kfset_set_masks(self._h, slot, _p(v), 0 if v is None else len(v), _p(h), 0 if h is None else len(h)))

    def clear(self, slot):
        _check(lib().sslpl_kfset_clear(self._h, slot))

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            lib().sslpl_kfset_destroy(self._h)
            self._h = C.c_void_p()

    __del__ = close


class ORBmatcher:
    """Mirror of StructureSLAM::ORBmatcher (include/ORBmatcher.h:36-101) on indices + masks instead of
    KeyFrame*/MapPoint* (the C++ adapter in host/ maps indices back to pointers)."""
    TH_HIGH, TH_LOW, HISTO_LENGTH = 100, 50, 30

    def __init__(self, nnratio=0.6, checkOri=True, ctx=None):
        self.mfNNratio, self.mbCheckOrientation = float(nnratio), bool(checkOri)
        self.ctx = ctx or Matcher()

    def DescriptorDistance(self, a, b):
        return int(self.ctx.descriptor_distance(a, b)[0])

    def SearchByBoW(self, d1, fv1, valid1, angle1, d2, fv2, angle2, valid2=None):
        """KeyFrame-vs-Frame (valid2 is None; ORBmatcher.cc:159) -> (nmatches, match2[n2] = KF index or -1);
        KeyFrame-vs-KeyFrame (valid2 given; ORBmatcher.cc:525) -> (nmatches, match12[n1] = KF2 index or -1)."""
        d1 = np.ascontiguousarray(d1, np.uint8).reshape(-1, 32); d2 = np.ascontiguousarray(d2, np.uint8).reshape(-1, 32)
        f1, f2 = _featvec(fv1), _featvec(fv2)
        valid1 = np.ascontiguousarray(valid1, np.uint8)
        angle1 = np.ascontiguousarray(angle1, np.float32); angle2 = np.ascontiguousarray(angle2, np.float32)
        nm = C.c_int()
        if valid2 is None:
            out = np.empty(len(d2), np.int32)
            _check(lib().sslpl_search_by_bow(self.ctx._h, _p(d1), len(d1), _p(d2), len(d2), C.byref(f1), C.byref(f2),
                                             _p(valid1), _p(angle1), _p(angle2), C.c_float(self.mfNNratio),
                                             int(self.mbCheckOrientation), _p(out), C.byref(nm)))
        else:
            valid2 = np.ascontiguousarray(valid2, np.uint8)
            out = np.empty(len(d1), np.int32)
            _check(lib().sslpl_search_by_bow_kf(self.ctx._h, _p(d1), len(d1), _p(d2), len(d2), C.byref(f1), C.byref(f2),
                                                _p(valid1), _p(valid2), _p(angle1), _p(angle2), C.c_float(self.mfNNratio),
                                                int(self.mbCheckOrientation), _p(out), C.byref(nm)))
        return nm.value, out

    def SearchForTriangulation(self, d1, fv1, has_mp1, kp1, d2, fv2, has_mp2, kp2, F12, ex, ey, scale, sigma2):
        """ORBmatcher.cc:660 (monocular) -> (nmatches, pairs[nmatches,2])."""
        d1 = np.ascontiguousarray(d1, np.uint8).reshape(-1, 32); d2 = np.ascontiguousarray(d2, np.uint8).reshape(-1, 32)
        f1, f2 = _featvec(fv1), _featvec(fv2)
        has_mp1 = np.ascontiguousarray(has_mp1, np.uint8); has_mp2 = np.ascontiguousarray(has_mp2, np.uint8)
        kp1 = np.ascontiguousarray(kp1, KEYPOINT_DTYPE); kp2 = np.ascontiguousarray(kp2, KEYPOINT_DTYPE)
        F12 = np.ascontiguousarray(F12, np.float32).reshape(9)
        scale = np.ascontiguousarray(scale, np.float32); sigma2 = np.ascontiguousarray(sigma2, np.float32)
        pairs = np.empty((max(len(d1), 1), 2), np.int32)
        nm = C.c_int()
        _check(lib().sslpl_search_for_triangulation(self.ctx._h, _p(d1), len(d1), _p(d2), len(d2), C.byref(f1), C.byref(f2),
                                                    _p(has_mp1), _p(has_mp2), _p(kp1), _p(kp2), _p(F12), C.c_float(ex), C.c_float(ey),
                                                    _p(scale), _p(sigma2), len(scale), int(self.mbCheckOrientation),
                                                    _p(pairs), C.byref(nm)))
        return nm.value, pairs[:nm.value].copy()


class LSDmatcher:
    """Mirror of the knnMatch-based entry points of StructureSLAM::LSDmatcher (include/LSDmatcher.h:36-64)."""

    def __init__(self, ctx=None):
        self.ctx = ctx or Matcher()

    def _run(self, mode, d1, d2, has_ml1, has_ml2):
        d1 = np.ascontiguousarray(d1, np.uint8).reshape(-1, 32); d2 = np.ascontiguousarray(d2, np.uint8).reshape(-1, 32)
        h1 = np.ascontiguousarray(has_ml1 if has_ml1 is not None else np.zeros(len(d1)), np.uint8)
        h2 = np.ascontiguousarray(has_ml2 if has_ml2 is not None else np.zeros(len(d2)), np.uint8)
        out = np.full(2 * max(len(d1), len(d2), 1), -1, np.int32)
        k = C.c_int(); nm = C.c_int(); mad = (C.c_double * 2)()
        _check(lib().sslpl_line_match(self.ctx._h, mode, _p(d1), len(d1), _p(d2), len(d2), _p(h1), _p(h2), _p(out),
                                      C.byref(k), C.byref(nm), mad))
        self.last_mad = (mad[0], mad[1])
        if mode == 0:
            return nm.value, out[:len(d2)].copy()
        if mode == 2:
            return nm.value, out[:len(d1)].copy()
        return nm.value, out[:2 * k.value].reshape(-1, 2).copy()

    def SearchByProjection(self, ldescKF, has_mapline_KF, ldescF):      # LSDmatcher.cpp:143 (KeyFrame*, Frame&)
        return self._run(0, ldescKF, ldescF, has_mapline_KF, None)

    SearchByDescriptor = SearchByProjection                             # LSDmatcher.cpp:286 (identical body)

    def SerachForInitialize(self, ldesc1, ldesc2):                      # LSDmatcher.cpp:257 (sic)
        return self._run(1, ldesc1, ldesc2, None, None)

    def SearchByDescriptorKF(self, ldesc1, ldesc2, has_mapline_KF2):    # LSDmatcher.cpp:329
        return self._run(2, ldesc1, ldesc2, None, has_mapline_KF2)

    def SearchForTriangulation(self, ldesc1, has_ml1, ldesc2, has_ml2):  # LSDmatcher.cpp:382
        return self._run(3, ldesc1, ldesc2, has_ml1, has_ml2)

    def DescriptorDistance(self, a, b):                                 # LSDmatcher.cpp:364
        return int(self.ctx.descriptor_distance(a, b)[0])


# =====================================================================================================
# Frame level
# =====================================================================================================
class FrameParams(C.Structure):
    _fields_ = [("orb", OrbParams), ("line", LineParams)]


class Frame:
    """What StructureSLAM::Frame::Frame(imGray, ...) does with the two extractors (src/Frame.cc:69-131): ONE upload of the frame,
    ORB and LSD+LBD on two streams, optional colour conversion in front (Tracking.cc:148-161) and keypoint undistortion behind
    (Frame.cc:483-513).  `extract(image)` -> dict(keys, keysUn, desc, keylines, ldesc, lineeq)."""

    def __init__(self, nfeatures=1000, scaleFactor=1.2, nlevels=8, iniThFAST=20, minThFAST=7, lsdNFeatures=40,
                 max_width=1280, max_height=960, max_batch=1, device=0):
        p = FrameParams(OrbParams(nfeatures, scaleFactor, nlevels, iniThFAST, minThFAST, max_width, max_height, max_batch, device),
                        LineParams(lsdNFeatures, max_width, max_height, max_batch, device))
        self._h = C.c_void_p()
        lib().sslpl_frame_create.argtypes = [C.c_void_p, C.c_void_p]
        _check(lib().sslpl_frame_create(C.byref(p), C.byref(self._h)))
        lib().sslpl_frame_orb.restype = C.c_void_p; lib().sslpl_frame_orb.argtypes = [C.c_void_p]
        lib().sslpl_frame_line.restype = C.c_void_p; lib().sslpl_frame_line.argtypes = [C.c_void_p]
        lib().sslpl_frame_stream.restype = C.c_void_p; lib().sslpl_frame_stream.argtypes = [C.c_void_p, C.c_int]
        self.orb = ORBextractor._borrow(lib().sslpl_frame_orb(self._h), nfeatures, scaleFactor, nlevels, max_batch)
        self.line = LineSegment._borrow(lib().sslpl_frame_line(self._h), lsdNFeatures, max_batch)
        self.cap = self.orb.cap
        self.lcap = lsdNFeatures
        self.max_batch = max_batch

    def stream(self, which):
        """CUDA stream handle of the ORB (0) or line (1) side."""
        return int(lib().sslpl_frame_stream(self._h, int(which)))

    def extract_batch_begin(self, frames, out):
        """Asynchronous: frames [B, H, W] uint8 in pinned memory (host_alloc); out = dict(keys, desc, n, keylines, ldesc, lineeq, nl) of
        pinned arrays with the handle's capacities.  Finish with sync()."""
        B, h, w = frames.shape[:3]
        cn = 1 if frames.ndim == 3 else frames.shape[3]
        assert out["keys"].shape[1] == self.cap and out["keylines"].shape[1] == self.lcap
        _check(lib().sslpl_frame_extract_batch_begin(self._h, _p(frames), B, w, h, frames.strides[1], C.c_size_t(frames.strides[0]), cn, 0,
                                                     _p(out["keys"]), None, _p(out["desc"]), self.cap, _p(out["n"]),
                                                     _p(out["keylines"]), _p(out["ldesc"]), _p(out["lineeq"]), self.lcap, _p(out["nl"])))

    def sync(self):
        _check(lib().sslpl_frame_sync(self._h))

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            lib().sslpl_frame_destroy.argtypes = [C.c_void_p]
            lib().sslpl_frame_destroy(self._h)
            self._h = C.c_void_p()

    __del__ = close

    def set_camera(self, fx, fy, cx, cy, dist=()):
        d = np.ascontiguousarray(dist, np.float32)
        _check(lib().sslpl_frame_set_camera(self._h, C.c_float(fx), C.c_float(fy), C.c_float(cx), C.c_float(cy), _p(d) if len(d) else None, len(d)))

    def image_bounds(self, cols, rows):
        b = np.zeros(4, np.float32)
        _check(lib().sslpl_frame_image_bounds(self._h, int(cols), int(rows), _p(b)))
        return b

    @property
    def launch_count(self):
        lib().sslpl_frame_launch_count.restype = C.c_longlong
        return int(lib().sslpl_frame_launch_count(self._h))

    def extract(self, image, rgb_order=False):
        """image: HxW (grey) or HxWx3 / HxWx4 uint8 (BGR[A] unless rgb_order)."""
        assert image.dtype == np.uint8 and image.ndim in (2, 3)
        image = np.ascontiguousarray(image)
        cn = 1 if image.ndim == 2 else image.shape[2]
        h, w = image.shape[:2]
        kps = np.zeros(self.cap, KEYPOINT_DTYPE); un = np.zeros(self.cap, KEYPOINT_DTYPE); desc = np.zeros((self.cap, 32), np.uint8)
        kl = np.zeros(self.lcap, KEYLINE_DTYPE); ld = np.zeros((self.lcap, 32), np.uint8); eq = np.zeros((self.lcap, 3), np.float64)
        n = C.c_int(); nl = C.c_int()
        _check(lib().sslpl_frame_extract(self._h, _p(image), w, h, image.strides[0], cn, int(rgb_order), _p(kps), _p(un), _p(desc), self.cap,
                                         C.byref(n), _p(kl), _p(ld), _p(eq), self.lcap, C.byref(nl)))
        n, nl = n.value, nl.value
        return dict(keys=kps[:n].copy(), keysUn=un[:n].copy(), desc=desc[:n].copy(), keylines=kl[:nl].copy(), ldesc=ld[:nl].copy(), lineeq=eq[:nl].copy())

    def extract_batch(self, frames, rgb_order=False):
        """frames: [B, H, W] or [B, H, W, C] uint8 -> dict of per-frame arrays (padded to the capacities) and counts."""
        frames = np.ascontiguousarray(frames)
        B, h, w = frames.shape[:3]
        cn = 1 if frames.ndim == 3 else frames.shape[3]
        kps = np.zeros((B, self.cap), KEYPOINT_DTYPE); un = np.zeros((B, self.cap), KEYPOINT_DTYPE); desc = np.zeros((B, self.cap, 32), np.uint8)
        kl = np.zeros((B, self.lcap), KEYLINE_DTYPE); ld = np.zeros((B, self.lcap, 32), np.uint8); eq = np.zeros((B, self.lcap, 3), np.float64)
        n = np.zeros(B, np.int32); nl = np.zeros(B, np.int32)
        _check(lib().sslpl_frame_extract_batch(self._h, _p(frames), B, w, h, frames.strides[1], C.c_size_t(frames.strides[0]), cn, int(rgb_order),
                                               _p(kps), _p(un), _p(desc), self.cap, _p(n), _p(kl), _p(ld), _p(eq), self.lcap, _p(nl)))
        return dict(keys=kps, keysUn=un, desc=desc, n=n, keylines=kl, ldesc=ld, lineeq=eq, nl=nl)


# =====================================================================================================
# Lines
# =====================================================================================================
class LineSegment:
    """Mirror of StructureSLAM::LineSegment (include/ExtractLineSegment.h:53-76).  lsdNFeatures is hard-coded to 40
    in the reference (ExtractLineSegment.cpp:42); it is a constructor parameter here (BASELINE.json config 4: 500)."""

    def __init__(self, lsdNFeatures=40, max_width=1280, max_height=960, max_batch=1, device=0):
        p = LineParams(lsdNFeatures, max_width, max_height, max_batch, device)
        self._h = C.c_void_p()
        _check(lib().sslpl_line_create(C.byref(p), C.byref(self._h)))
        self.cap = lsdNFeatures
        self.max_batch = max_batch

    @classmethod
    def _borrow(cls, ptr, lsdNFeatures, max_batch):
        self = cls.__new__(cls)
        self._h = C.c_void_p(ptr); self._borrowed = True; self.cap = lsdNFeatures; self.max_batch = max_batch
        return self

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value and not getattr(self, "_borrowed", False):
            lib().sslpl_line_destroy(self._h)
            self._h = C.c_void_p()

    __del__ = close

    def ExtractLineSegment(self, img, scale=1, numOctaves=1):
        """-> (keylines, ldesc, keylineFunctions): ExtractLineSegment.cpp:18-69 (scale / numOctaves as the reference
        passes them: int 1 and 1; other values are not supported)."""
        assert int(scale) == 1 and numOctaves == 1
        assert img.dtype == np.uint8 and img.ndim == 2
        if img.strides[1] != 1:
            img = np.ascontiguousarray(img)
        kl = np.zeros(self.cap, KEYLINE_DTYPE); ld = np.zeros((self.cap, 32), np.uint8); eq = np.zeros((self.cap, 3), np.float64)
        n = C.c_int()
        _check(lib().sslpl_line_extract(self._h, _p(img), img.shape[1], img.shape[0], img.strides[0], _p(kl), _p(ld), _p(eq),
                                        self.cap, C.byref(n)))
        return kl[:n.value].copy(), ld[:n.value].copy(), eq[:n.value].copy()

    def extract_batch(self, frames, out=None):
        assert frames.dtype == np.uint8 and frames.ndim == 3 and frames.strides[2] == 1
        B, H, W = frames.shape
        if out is None:
            out = (np.zeros((B, self.cap), KEYLINE_DTYPE), np.zeros((B, self.cap, 32), np.uint8),
                   np.zeros((B, self.cap, 3), np.float64), np.zeros(B, np.int32))
        kl, ld, eq, n = out
        _check(lib().sslpl_line_extract_batch(self._h, _p(frames), B, W, H, frames.strides[1], C.c_size_t(frames.strides[0]),
                                              _p(kl), _p(ld), _p(eq), self.cap, _p(n)))
        return kl, ld, eq, n

    def extract_batch_begin(self, frames, out):
        B, H, W = frames.shape
        kl, ld, eq, n = out
        _check(lib().sslpl_line_extract_batch_begin(self._h, _p(frames), B, W, H, frames.strides[1], C.c_size_t(frames.strides[0]),
                                                    _p(kl), _p(ld), _p(eq), self.cap, _p(n)))

    def extract_batch_device(self, d_ptr, nframes, width, height, pitch, frame_stride):
        _check(lib().sslpl_line_extract_batch_device(self._h, C.c_void_p(d_ptr), nframes, width, height, pitch, C.c_size_t(frame_stride)))

    def device_results(self):
        kl = C.c_void_p(); ld = C.c_void_p(); eq = C.c_void_p(); n = C.c_void_p(); cap = C.c_int()
        _check(lib().sslpl_line_device_results(self._h, C.byref(kl), C.byref(ld), C.byref(eq), C.byref(n), C.byref(cap)))
        return kl.value, ld.value, eq.value, n.value, cap.value

    def raw_segments(self, frame=0, cap=1 << 15):
        seg = np.empty((cap, 4), np.float32); n = C.c_int()
        _check(lib().sslpl_line_download_segments(self._h, frame, _p(seg), cap, C.byref(n)))
        return seg[:min(n.value, cap)].copy()

    def set_max_walkers(self, n):
        _check(lib().sslpl_line_set_max_walkers(self._h, int(n)))

    def set_profiling(self, on=True):
        _check(lib().sslpl_line_set_profiling(self._h, int(on)))

    def stage_ms(self):
        ms = (C.c_float * 16)(); names = (C.c_char_p * 16)(); n = C.c_int()
        _check(lib().sslpl_line_stage_ms(self._h, ms, 16, names, C.byref(n)))
        return {names[i].decode(): float(ms[i]) for i in range(n.value)}

    def walker_stats(self):
        out = (C.c_ulonglong * 16)()
        _check(lib().sslpl_line_walker_stats(self._h, out))
        names = ["turn_regions", "turn_cycles", "turn_pixels", "_", "seed_swallowed", "redo_abandoned", "redo_poisoned", "redo_invalid", "redo_presumed",
                 "committed_as_speculated", "speculated_pixels", "commit_lock_cycles", "claim_lock_cycles", "repeated_attempts", "frame_cycles", "claims"]
        return {k: int(out[i]) for i, k in enumerate(names)}

    def debug_trace(self, frame=0, cap=1 << 16):
        out = np.empty((cap, 10), np.float64); n = C.c_int()
        _check(lib().sslpl_line_debug_trace(self._h, frame, _p(out), cap, C.byref(n)))
        return out[:min(n.value, cap)].copy()

    def sync(self):
        _check(lib().sslpl_line_sync(self._h))

    def set_stream(self, cuda_stream):
        _check(lib().sslpl_line_set_stream(self._h, C.c_void_p(cuda_stream)))

    @property
    def launch_count(self):
        return int(lib().sslpl_line_launch_count(self._h))
