/*
 * include/sslpl.h — C ABI of the B200-native point/line front-end (libsslpl_b200.so).
 *
 * This is the drop-in boundary for the three data-parallel hot paths of
 * yanyan-li/Structure-SLAM-PointLine's Tracking::TrackWithPL():
 *   (1) ORBextractor::operator()            reference: include/ORBextractor.h:45-111, src/ORBextractor.cc:1043
 *   (2) LineSegment::ExtractLineSegment     reference: include/ExtractLineSegment.h:53-76, src/ExtractLineSegment.cpp:18
 *   (3) ORBmatcher / LSDmatcher Hamming     reference: include/ORBmatcher.h:36-101, include/LSDmatcher.h:36-64
 * and, widened after those met the parity + measurement bar (SURVEY.md 8(f) "next" rows 1-3): the DBoW2 vocabulary transform of
 * Frame::ComputeBoW, ORBmatcher::SearchByProjection(Frame&, const Frame&, ...) with the Frame feature grid, and the descriptor
 * medoid of MapPoint / MapLine ::ComputeDistinctiveDescriptors.
 * The reference has no FFI; its boundary is the C++ class surface.  The adapters in
 * structure-slam-pointline_b200/host/ re-expose those class signatures on top of this ABI
 * (see INTEGRATION.md).  Plain pointers and sizes only; no torch / OpenCV types.
 *
 * Conventions: every entry point returns 0 on success or a negative sslpl_status; nothing throws;
 * the callee never allocates caller-visible memory; `*_device` variants take device pointers and
 * enqueue on the handle's stream without synchronising (call sslpl_*_sync).  Handles are not
 * thread-safe individually, but any number of handles may be used concurrently from different
 * threads (the reference calls the matchers from Tracking and LocalMapping threads at once).
 * There is NO CPU fallback: without a CUDA device every create call fails with SSLPL_ERR_CUDA.
 */
#ifndef SSLPL_H
#define SSLPL_H
#include <stddef.h>
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define SSLPL_VERSION 1
#define SSLPL_MAX_LEVELS 16

typedef enum {
    SSLPL_OK = 0,
    SSLPL_ERR_ARG = -1,        /* bad argument (null pointer, size out of the handle's capacity, ...) */
    SSLPL_ERR_CUDA = -2,       /* CUDA runtime error; see sslpl_last_error() */
    SSLPL_ERR_CAPACITY = -3,   /* an internal or caller-provided buffer was too small (no partial result) */
    SSLPL_ERR_UNSUPPORTED = -4
} sslpl_status;

const char* sslpl_last_error(void);          /* thread-local message of the last failing call */
int  sslpl_version(void);
int  sslpl_device_count(void);               /* 0 when no CUDA device / driver */
int  sslpl_default_device(void);             /* CUDA ordinal the reference-side adapters use: $SSLPL_DEVICE, else 0 */

/* pinned host memory for frames / results (so H2D/D2H run at link speed) */
int  sslpl_host_alloc(void** p, size_t bytes);
int  sslpl_host_free(void* p);

/* ---- POD mirrors of the OpenCV types that cross the reference boundary (SURVEY.md 8(a) a15) ---- */
typedef struct { float x, y, size, angle, response; int32_t octave, class_id; } sslpl_keypoint;   /* cv::KeyPoint, 28 B */
typedef struct {                                                                                  /* cv::line_descriptor::KeyLine, 68 B */
    float angle; int32_t class_id; int32_t octave; float pt_x, pt_y; float response; float size;
    float startPointX, startPointY, endPointX, endPointY;
    float sPointInOctaveX, sPointInOctaveY, ePointInOctaveX, ePointInOctaveY;
    float lineLength; int32_t numOfPixels;
} sslpl_keyline;

/* =====================================================================================
 * (1) ORB extractor — replaces ORBextractor (src/ORBextractor.cc)
 * ===================================================================================== */
typedef struct {
    int   nfeatures;      /* ORBextractor.nFeatures   (Examples/ICL.yaml:41)  */
    float scaleFactor;    /* ORBextractor.scaleFactor (ICL.yaml:44)           */
    int   nlevels;        /* ORBextractor.nLevels     (ICL.yaml:47), <= SSLPL_MAX_LEVELS */
    int   iniThFAST;      /* ICL.yaml:53 */
    int   minThFAST;      /* ICL.yaml:54 */
    int   max_width, max_height;   /* largest frame this handle will see (device workspace is sized once) */
    int   max_batch;      /* frames per call for the batched entry points (>=1) */
    int   device;         /* CUDA device ordinal */
} sslpl_orb_params;

typedef struct sslpl_orb sslpl_orb;

int  sslpl_orb_create(const sslpl_orb_params* p, sslpl_orb** out);            /* ORBextractor::ORBextractor, ORBextractor.cc:410 */
void sslpl_orb_destroy(sslpl_orb* h);
/* GetScaleFactors / GetInverseScaleFactors / GetScaleSigmaSquares / GetInverseScaleSigmaSquares
   (ORBextractor.h:63-77) + mnFeaturesPerLevel + umax; each array has nlevels (umax: 16) entries; NULL = skip */
int  sslpl_orb_tables(const sslpl_orb* h, float* scale, float* invscale, float* sigma2, float* invsigma2,
                      int* nfeat_per_level, int* umax16);
/* the same tables without a device or a handle (host arithmetic only: the adapter's constructor runs before any frame is seen) */
int  sslpl_orb_tables_host(int nfeatures, float scaleFactor, int nlevels, float* scale, float* invscale, float* sigma2, float* invsigma2,
                           int* nfeat_per_level, int* umax16);
int  sslpl_orb_max_keypoints(const sslpl_orb* h);  /* capacity per frame: sum_l (mnFeaturesPerLevel[l] + 3) */

/* ORBextractor::operator() (ORBextractor.cc:1043) on one HOST frame (CV_8UC1, `pitch` bytes per row).
   kps[cap], desc[cap*32]; *n = number of keypoints (0 for an empty image, as the reference's silent return). */
int  sslpl_orb_extract(sslpl_orb* h, const uint8_t* img, int width, int height, int pitch,
                       sslpl_keypoint* kps, uint8_t* desc, int cap, int* n);
/* Batched frames, HOST buffers: frame f at imgs + f*frame_stride; outputs kps[f*cap + i], desc[(f*cap+i)*32], n[f]. */
int  sslpl_orb_extract_batch(sslpl_orb* h, const uint8_t* imgs, int nframes, int width, int height, int pitch,
                             size_t frame_stride, sslpl_keypoint* kps, uint8_t* desc, int cap, int* n);
/* Asynchronous form of the above: enqueues H2D + extraction + D2H on the handle's stream and returns; the host buffers
   (pinned, see sslpl_host_alloc) are valid after sslpl_orb_sync().  Needs cap >= sslpl_orb_max_keypoints(). */
int  sslpl_orb_extract_batch_begin(sslpl_orb* h, const uint8_t* imgs, int nframes, int width, int height, int pitch,
                                   size_t frame_stride, sslpl_keypoint* kps, uint8_t* desc, int cap, int* n);
/* Batched frames already resident in HBM; results stay in HBM (see sslpl_orb_device_results). Asynchronous. */
int  sslpl_orb_extract_batch_device(sslpl_orb* h, const uint8_t* d_imgs, int nframes, int width, int height, int pitch,
                                    size_t frame_stride);
/* Device result buffers of the last *_device call: d_kps[f*cap+i], d_desc[(f*cap+i)*32], d_n[f]. */
int  sslpl_orb_device_results(sslpl_orb* h, const sslpl_keypoint** d_kps, const uint8_t** d_desc, const int** d_n, int* cap);
int  sslpl_orb_sync(sslpl_orb* h);           /* wait for the handle's stream; reports deferred device-side errors */
void* sslpl_orb_stream(sslpl_orb* h);        /* cudaStream_t of the handle */
/* Run the handle on a caller-owned cudaStream_t (e.g. the framework's current stream) instead of its own. */
int  sslpl_orb_set_stream(sslpl_orb* h, void* cuda_stream);
/* mvImagePyramid[level] (ORBextractor.h:79) of frame f of the last call; bordered=1 adds the 19-px
   BORDER_REFLECT_101 frame of ComputePyramid (ORBextractor.cc:1107-1132). dst is a HOST buffer. */
int  sslpl_orb_level_size(const sslpl_orb* h, int level, int* w, int* hgt);
int  sslpl_orb_download_level(sslpl_orb* h, int frame, int level, int bordered, uint8_t* dst, int dpitch);
/* stage intermediates of the last call, for parity tests: FAST candidates (vToDistributeKeys order),
   per-level keypoints after DistributeOctTree, blurred level */
int  sslpl_orb_download_candidates(sslpl_orb* h, int frame, int level, int* xs, int* ys, int* resp, int cap, int* n);
int  sslpl_orb_download_level_keypoints(sslpl_orb* h, int frame, int level, int* xs, int* ys, int* resp, int cap, int* n);
int  sslpl_orb_download_blurred(sslpl_orb* h, int frame, int level, uint8_t* dst, int dpitch);
/* number of kernels this handle has launched since creation (bench.py's gpu_launches claim) */
long long sslpl_orb_launch_count(const sslpl_orb* h);
/* names + CUDA-event milliseconds of the kernels of the last profiled call (enable with sslpl_orb_set_profiling) */
int  sslpl_orb_set_profiling(sslpl_orb* h, int on);
int  sslpl_orb_stage_ms(sslpl_orb* h, float* ms, int cap, const char** names, int* nstages);

/* =====================================================================================
 * (3) Hamming matching — replaces ORBmatcher / LSDmatcher kernels of work
 * ===================================================================================== */
typedef struct sslpl_matcher sslpl_matcher;
typedef struct {
    int max_features;     /* largest N (points) per frame */
    int max_lines;        /* largest NL per frame */
    int max_nodes;        /* largest number of vocabulary nodes in a FeatureVector */
    int max_batch;        /* frame pairs per batched call */
    int device;
} sslpl_matcher_params;
int  sslpl_matcher_create(const sslpl_matcher_params* p, sslpl_matcher** out);
void sslpl_matcher_destroy(sslpl_matcher* m);
int  sslpl_matcher_sync(sslpl_matcher* m);
void* sslpl_matcher_stream(sslpl_matcher* m);
int  sslpl_matcher_set_stream(sslpl_matcher* m, void* cuda_stream);
long long sslpl_matcher_launch_count(const sslpl_matcher* m);

/* ORBmatcher::DescriptorDistance (ORBmatcher.cc:1650) for nq pairs a[i] vs b[i] (HOST buffers) */
int  sslpl_descriptor_distance(sslpl_matcher* m, const uint8_t* a, const uint8_t* b, int n, int32_t* dist);
/* cv::BFMatcher(NORM_HAMMING,false).knnMatch(q,t,.,2) as used by LSDmatcher.cpp:155,266,298,341,392:
   out[4*i+0..3] = trainIdx0, dist0, trainIdx1, dist1 (ties -> lower trainIdx; -1,-1 when nt < 2) */
int  sslpl_hamming_knn2(sslpl_matcher* m, const uint8_t* q, int nq, const uint8_t* t, int nt, int32_t* out);
/* Vocabulary-node assignment (synthetic one-level stand-in for DBoW2 transform, TemplatedVocabulary.h:1218-1259) */
int  sslpl_bow_assign(sslpl_matcher* m, const uint8_t* desc, int n, const uint8_t* centroids, int nc, int32_t* node);

/* DBoW2::FeatureVector flattened to CSR: nodes[nn] ascending, off[nn+1], idx[off[nn]] */
typedef struct { const int32_t* nodes; const int32_t* off; const int32_t* idx; int nn; } sslpl_featvec;

/* ORBmatcher::SearchByBoW(KeyFrame*,Frame&,vector<MapPoint*>&) (ORBmatcher.cc:159-291).
   valid1[i] != 0 <=> KF feature i has a non-bad MapPoint.  match2[j] = KF feature index matched to frame
   feature j, or -1 (the adapter maps indices back to MapPoint*).  *nmatches = return value of the reference. */
int  sslpl_search_by_bow(sslpl_matcher* m, const uint8_t* d1, int n1, const uint8_t* d2, int n2,
                         const sslpl_featvec* fv1, const sslpl_featvec* fv2,
                         const uint8_t* valid1, const float* angle1, const float* angle2,
                         float nnratio, int checkOrientation, int32_t* match2, int* nmatches);
/* ORBmatcher::SearchByBoW(KeyFrame*,KeyFrame*,vector<MapPoint*>&) (ORBmatcher.cc:525-658): match12[i] = KF2 index or -1 */
int  sslpl_search_by_bow_kf(sslpl_matcher* m, const uint8_t* d1, int n1, const uint8_t* d2, int n2,
                            const sslpl_featvec* fv1, const sslpl_featvec* fv2,
                            const uint8_t* valid1, const uint8_t* valid2, const float* angle1, const float* angle2,
                            float nnratio, int checkOrientation, int32_t* match12, int* nmatches);
/* ORBmatcher::SearchForTriangulation (ORBmatcher.cc:660-826), monocular (bOnlyStereo=false, mvuRight<0).
   kp1/kp2 = mvKeysUn; has_mp = "feature already has a MapPoint"; F12 row-major 3x3 f32; (ex,ey) epipole;
   scale = mvScaleFactors, sigma2 = mvLevelSigma2 of KF2.  pairs[2*k] = (idx1, idx2) sorted by idx1. */
int  sslpl_search_for_triangulation(sslpl_matcher* m, const uint8_t* d1, int n1, const uint8_t* d2, int n2,
                                    const sslpl_featvec* fv1, const sslpl_featvec* fv2,
                                    const uint8_t* has_mp1, const uint8_t* has_mp2,
                                    const sslpl_keypoint* kp1, const sslpl_keypoint* kp2,
                                    const float* F12, float ex, float ey, const float* scale, const float* sigma2, int nlevels,
                                    int checkOrientation, int32_t* pairs, int* nmatches);
/* LSDmatcher knnMatch-based entry points (LSDmatcher.cpp). mode 0: SearchByProjection(KF,F) :143 /
   SearchByDescriptor(KF,F) :286 -> out[tdx] = qdx table (n2 entries);  mode 1: SerachForInitialize :257 -> pairs;
   mode 2: SearchByDescriptor(KF,KF2) :329 -> out[qdx] = tdx table (n1 entries); mode 3: SearchForTriangulation :382 -> pairs.
   *nout = number of pairs written (modes 1,3); *nmatches = the reference's return value.
   Also returns Frame::lineDescriptorMAD (Frame.cc:190) in mad[0..1] when mad != NULL. */
int  sslpl_line_match(sslpl_matcher* m, int mode, const uint8_t* d1, int n1, const uint8_t* d2, int n2,
                      const uint8_t* has_ml1, const uint8_t* has_ml2, int32_t* out, int* nout, int* nmatches, double* mad);

/* Batched consecutive-frame matching, everything resident in HBM (config 5 of BASELINE.json):
   for pair p (frame p = "KeyFrame", frame p+1 = "Frame"): node assignment of both frames against the
   vocabulary, FeatureVector build, SearchByBoW (all KF features valid), rotation filter.
   d_desc/d_kps/d_n as produced by sslpl_orb_extract_batch_device (cap entries per frame, nframes frames);
   d_match[(p*cap)+j] = KF index or -1 for frame p+1's feature j; d_nmatch[p]. npairs = nframes-1. */
int  sslpl_match_bow_batch_device(sslpl_matcher* m, const uint8_t* d_desc, const sslpl_keypoint* d_kps, const int* d_n,
                                  int nframes, int cap, const uint8_t* d_centroids, int nc,
                                  float nnratio, int checkOrientation, int32_t* d_match, int32_t* d_nmatch);
/* ---- ORBmatcher::SearchByProjection(Frame &CurrentFrame, const Frame &LastFrame, th, bMono) (ORBmatcher.cc:1331-1473), the
   matcher of Tracking::TrackWithMotionModel (Tracking.cc:1227), with Frame::AssignFeaturesToGrid / GetFeaturesInArea
   (Frame.cc:133-148, 368-421) on the device.  SURVEY.md 8(f) row 2.  HOST buffers.
   Last frame (n1): valid1[i] = mvpMapPoints[i] && !mvbOutlier[i]; obs1[i] = that MapPoint's Observations() > 0; Xw[3i..] =
   GetWorldPos(); dmp[i][32] = GetDescriptor(); oct1 = mvKeys[i].octave; angle1 = mvKeysUn[i].angle.
   Current frame (n2): descriptors d2, mvKeysUn x2 / y2 / oct2 / angle2, mvuRight (NULL for monocular), claimed2[j] = the
   feature already holds a MapPoint with observations (NULL = none).  Tcw / Tlw: 3x4 row-major poses (Tlw only read when
   !bMono); cam = {fx, fy, cx, cy, mbf, mb}; bounds = {mnMinX, mnMaxX, mnMinY, mnMaxY}; scaleFactors[nlevels].
   Result: assign2[j] = index i of the last-frame MapPoint now held by current feature j; -1 = never assigned; -2 = assigned and
   then removed by the rotation check (the reference writes NULL there, ORBmatcher.cc:1461: the caller must too); *nmatches as
   returned by the reference.  The matcher handle needs max_nodes >= 3072 (grid cells) and at most 8192 features. */
int  sslpl_search_by_projection_frame(sslpl_matcher* m,
        int n1, const uint8_t* valid1, const uint8_t* obs1, const float* Xw, const uint8_t* dmp, const int32_t* oct1, const float* angle1,
        int n2, const uint8_t* d2, const float* x2, const float* y2, const int32_t* oct2, const float* angle2, const float* uright2,
        const uint8_t* claimed2, const float* Tcw, const float* Tlw, const float* cam, const float* bounds,
        const float* scaleFactors, int nlevels, float th, int bMono, int checkOrientation, int32_t* assign2, int* nmatches);

/* ---- ORBmatcher::SearchByProjection(Frame &F, const vector<MapPoint*> &vpMapPoints, th) (ORBmatcher.cc:45-129): the matcher of
   Tracking::SearchLocalPoints (Tracking.cc:1736), run on every frame.  Per MapPoint, in vector order, what Frame::isInFrustum left on
   it: inview = mbTrackInView, bad = isBad() (NULL = none), obs = Observations() > 0 (NULL = none), projx/projy = mTrackProjX/Y,
   projxr = mTrackProjXR (NULL for monocular), level = mnTrackScaleLevel, viewcos = mTrackViewCos, dmp = GetDescriptor().
   Frame (n2): descriptors, mvKeysUn x / y / octave, mvuRight (NULL), held2[j] = 0 nothing, 1 a MapPoint with observations (skipped),
   2 a MapPoint without (NULL = all 0).  assign2[j] = index of the MapPoint now written to F.mvpMapPoints[j] (-1: untouched). */
int  sslpl_search_by_projection_mps(sslpl_matcher* m,
        int nmp, const uint8_t* inview, const uint8_t* bad, const uint8_t* obs, const float* projx, const float* projy, const float* projxr,
        const int32_t* level, const float* viewcos, const uint8_t* dmp,
        int n2, const uint8_t* d2, const float* x2, const float* y2, const int32_t* oct2, const float* uright2, const uint8_t* held2,
        const float* bounds, const float* scaleFactors, int nlevels, float nnratio, float th, int32_t* assign2, int* nmatches);
/* ---- ORBmatcher::SearchForInitialization(F1, F2, vbPrevMatched, vnMatches12, windowSize) (ORBmatcher.cc:408-523,
   Tracking::MonocularInitialization Tracking.cc:366).  Keypoint fields are those of mvKeysUn; prev_xy[n1][2] = vbPrevMatched is
   updated like the reference does (:517-520); matches12[n1] = vnMatches12. */
int  sslpl_search_for_initialization(sslpl_matcher* m,
        int n1, const uint8_t* d1, const int32_t* oct1, const float* angle1, float* prev_xy,
        int n2, const uint8_t* d2, const float* x2, const float* y2, const int32_t* oct2, const float* angle2,
        const float* bounds, float nnratio, int checkOrientation, int windowSize, int32_t* matches12, int* nmatches);

/* ---- Line projection matchers and Fuse (SURVEY.md 8(f) row 3).  Each reference function is a projection stage (per map element:
   gates and projected quantities, arithmetic in the reference's own cv::Mat / Eigen types - it stays in the adapter, host/matcher_b200.cc,
   which calls the reference's own accessors, e.g. MapPoint::PredictScale) followed by a search stage (the Hamming scan over the frame's
   features), which is what these entry points run on the device.  HOST buffers; results identical to the reference's loops.

   sslpl_line_search_by_projection: search stage of LSDmatcher::SearchByProjection(Frame&, const Frame&, th, bMono) (LSDmatcher.cpp:98-137)
   and of LSDmatcher::SearchByProjection(Frame&, const vector<MapLine*>&, th) (:210-251).  Per MapLine, in the reference's visiting order:
   active (passed the gates), obs (Observations() > 0), proj[4] = projected end points x1 y1 x2 y2, radius, [minLevel, maxLevel] as handed to
   Frame::GetLinesInArea (Frame.cc:423-460), its descriptor.  Frame lines: descriptors, kl2[3] = pt.x pt.y angle of mvKeylinesUn, octaves,
   held2 (1 = holds a MapLine WITH observations: never a candidate).  assign2[j] = index of the MapLine written to mvpMapLines[j] (the last
   writer; -1 none), *nmatches = the function's return value. */
int  sslpl_line_search_by_projection(sslpl_matcher* m, int nml, const uint8_t* active, const uint8_t* obs, const float* proj, const float* radius,
        const int32_t* minLevel, const int32_t* maxLevel, const uint8_t* dml,
        int nl2, const uint8_t* ld2, const float* kl2, const int32_t* oct2, const uint8_t* held2,
        float nnratio, int32_t* assign2, int* nmatches);
/* Search stage of LSDmatcher::Fuse(KeyFrame*, const vector<MapLine*>&, th) (LSDmatcher.cpp:495-523): per MapLine the projected end points and
   the level MapLine::PredictScale returned; KeyFrame lines as above (oct2 = mvKeyLines[].octave).  best_idx[i] = nearest KeyFrame line of the
   window at level in [level-1, level] (first on ties; -1 none), best_dist[i] (INT_MAX when none); the caller fuses when best_dist <= 50.
   A level outside [0, nlevels) (PredictScale is not clamped, MapLine.cpp:386-395; the reference then reads mvScaleFactors out of bounds)
   drops the line. */
int  sslpl_fuse_lines_search(sslpl_matcher* m, int nml, const uint8_t* active, const float* proj, const int32_t* level, const uint8_t* dml,
        int nl2, const uint8_t* ld2, const float* kl2, const int32_t* oct2, const float* scaleFactors, int nlevels, float th,
        int32_t* best_idx, int32_t* best_dist);
/* Search stage of ORBmatcher::Fuse(KeyFrame*, const vector<MapPoint*>&, th) (ORBmatcher.cc:889-950): per MapPoint its projection (u, v, ur =
   u - bf / z; ur may be NULL when the KeyFrame has no stereo features) and predicted level; KeyFrame features: descriptors, mvKeysUn x / y /
   octave, mvuRight (NULL = monocular), image bounds, mvScaleFactors, mvInvLevelSigma2.  Window = KeyFrame::GetFeaturesInArea(u, v,
   th * scale[level]) (KeyFrame.cc:610-649), level gate, chi-square gate (5.99 mono / 7.8 stereo), nearest descriptor (first in the grid
   traversal order on ties).  best_idx[i] (-1 none), best_dist[i] (256 none); the caller fuses when best_dist <= 50. */
int  sslpl_fuse_points_search(sslpl_matcher* m, int nmp, const uint8_t* active, const float* u, const float* v, const float* ur,
        const int32_t* level, const uint8_t* dmp,
        int n2, const uint8_t* d2, const float* x2, const float* y2, const int32_t* oct2, const float* uright2,
        const float* bounds, const float* scaleFactors, const float* invLevelSigma2, int nlevels, float th,
        int32_t* best_idx, int32_t* best_dist);

/* MapPoint::ComputeDistinctiveDescriptors (MapPoint.cc:247-312) / MapLine::ComputeDistinctiveDescriptors (MapLine.cpp:246-317),
   batched (SURVEY.md 8(f) row 3): group g owns descriptors desc[off[g] .. off[g+1]) (HOST buffers, off[0] = 0);
   best_idx[g] = index inside the group of the descriptor with the least median Hamming distance to the others (median =
   sorted[int(0.5 (N - 1))], first minimum wins; -1 for an empty group), best_median[g] = that median. */
int  sslpl_descriptor_medoid_batch(sslpl_matcher* m, const uint8_t* desc, const int32_t* off, int ngroups,
                                   int32_t* best_idx, int32_t* best_median);

/* ---- DBoW2 vocabulary: Frame::ComputeBoW / KeyFrame::ComputeBoW (Frame.cc:474-481, KeyFrame.cc:71-80), i.e.
   TemplatedVocabulary<FORB>::transform(features, BowVector&, FeatureVector&, levelsup = 4)
   (Thirdparty/DBoW2/DBoW2/TemplatedVocabulary.h:1127-1259).  SURVEY.md 8(f) row 1. ---- */
typedef struct sslpl_vocab sslpl_vocab;
/* The tree as arrays (what loadFromTextFile :1338-1420 builds): node 0 = root, parent[i] < i (parent[0] ignored),
   desc[i][32], weight[i], is_leaf[i] (must agree with the structure).  Word ids number the leaves in node order. */
int  sslpl_vocab_create(int device, int k, int L, int nnodes, const int32_t* parent, const uint8_t* desc, const double* weight,
                        const uint8_t* is_leaf, sslpl_vocab** out);
/* ORBvoc.txt text format (System.cc:70 mpVocabulary->loadFromTextFile); scoring / weighting = the header's n1 / n2 */
int  sslpl_vocab_load_text(int device, const char* path, sslpl_vocab** out, int* scoring, int* weighting);
void sslpl_vocab_destroy(sslpl_vocab* v);
int  sslpl_vocab_info(const sslpl_vocab* v, int* k, int* L, int* nnodes, int* nwords);
/* number of distinct FeatureVector node values at level L - levelsup (+1 for node 0: root / leaves above that level) */
int  sslpl_vocab_level_nodes(const sslpl_vocab* v, int levelsup, int* count);
/* Per feature (HOST buffers): word id, NodeId at level L - levelsup, leaf weight.  weight <= 0 marks a stopped word, which
   the reference leaves out of both vectors (:1162-1166).  BowVector / FeatureVector assembly from these three arrays is a
   host-side map insertion (see the Python mirror's Vocabulary.bow_vector / feature_vector_csr). */
int  sslpl_bow_transform(sslpl_matcher* m, const sslpl_vocab* v, const uint8_t* desc, int n, int levelsup,
                         int32_t* word, int32_t* node, double* weight);
/* sslpl_match_bow_batch_device with the real tree instead of the one-level synthetic vocabulary.  Optional per-feature
   outputs d_word / d_node / d_weight ([nframes][cap], may be NULL) stay in HBM for the caller's BowVector build. */
int  sslpl_match_bow_batch_device_vocab(sslpl_matcher* m, const uint8_t* d_desc, const sslpl_keypoint* d_kps, const int* d_n,
                                        int nframes, int cap, const sslpl_vocab* v, int levelsup, float nnratio, int checkOrientation,
                                        int32_t* d_match, int32_t* d_nmatch, int32_t* d_word, int32_t* d_node, double* d_weight);
/* Batched line matching in HBM: knn2 + ratio rule of LSDmatcher::SearchByProjection(KF,F) (:143-183) with all
   KF lines valid: d_lmatch[p*capl + tdx] = qdx or -1; d_nlmatch[p]. */
int  sslpl_match_lines_batch_device(sslpl_matcher* m, const uint8_t* d_ldesc, const int* d_nl, int nframes, int capl,
                                    int32_t* d_lmatch, int32_t* d_nlmatch);

/* ---- Reference-keyframe matching of Tracking::TrackReferenceKeyFrame (Tracking.cc:1005-1034) against keyframes kept in HBM.
   A keyframe set has max_keyframes slots on one device; a slot holds up to `cap` ORB descriptors with their keypoint angles and
   MapPoint mask, their FeatureVector (built once, when the keyframe is stored), and up to `capl` LBD descriptors with their
   MapLine mask.  Slots start empty; an empty or cleared slot matches nothing. ---- */
typedef struct sslpl_kfset sslpl_kfset;
int  sslpl_kfset_create(int device, int max_keyframes, int cap, int capl, sslpl_kfset** out);
void sslpl_kfset_destroy(sslpl_kfset* k);
/* Copy frame `frame` of an extraction batch's device results (d_desc/d_kps/d_n with `cap` rows per frame, d_ldesc/d_nl with `capl`)
   into `slot` and build its FeatureVector with tree v at levelsup.  Masks are reset to all set.  Asynchronous on m's stream: the
   caller orders it after the extraction, and the extractor's results may be overwritten once it has run. */
int  sslpl_kfset_store_device(sslpl_matcher* m, sslpl_kfset* k, int slot,
                              const uint8_t* d_desc, const sslpl_keypoint* d_kps, const int* d_n, int cap,
                              const uint8_t* d_ldesc, const int* d_nl, int capl, int frame,
                              const sslpl_vocab* v, int levelsup);
/* The same from HOST buffers: n descriptors and keypoint angles, nl line descriptors.  Returns when the slot is written. */
int  sslpl_kfset_store(sslpl_matcher* m, sslpl_kfset* k, int slot, const uint8_t* desc, const float* angle, int n,
                       const uint8_t* ldesc, int nl, const sslpl_vocab* v, int levelsup);
/* valid[i] != 0 <=> feature i holds a non-bad MapPoint; has_ml[j] != 0 <=> line j holds a MapLine (HOST buffers; NULL = all set;
   entries past n / nl are set).  Returns when the masks are written, after the set's last store or match enqueued on a matcher's
   stream (sslpl_kfset_clear too). */
int  sslpl_kfset_set_masks(sslpl_kfset* k, int slot, const uint8_t* valid, int n, const uint8_t* has_ml, int nl);
int  sslpl_kfset_clear(sslpl_kfset* k, int slot);
/* For every frame f of a device extraction batch (layout as sslpl_match_bow_batch_device) with d_ref[f] = slot s (device int32
   array, never read by the host; -1, or any value outside the set, = no reference keyframe):
     ORBmatcher(nnratio, checkOrientation).SearchByBoW(KF s, frame f) (ORBmatcher.cc:159-291) with s's MapPoint mask:
       d_match[f*cap + j] = KF feature index or -1, d_nmatch[f] = the reference's return value;
     LSDmatcher::SearchByProjection(KF s, frame f) (LSDmatcher.cpp:143-183) with s's MapLine mask:
       d_lmatch[f*capl + t] = KF line index or -1 (the last writer in KF line order), d_nlmatch[f] = the reference's return value
       (0 when frame f has fewer than 2 lines, where the reference's knnMatch result is not usable).
   Frames without a reference keyframe get -1 rows and 0 counts.  Every stored slot must have been built with v and levelsup
   (SSLPL_ERR_ARG otherwise, nothing enqueued).  nframes <= max_batch + 1.  Asynchronous on m's stream. */
int  sslpl_match_ref_kf_batch_device(sslpl_matcher* m, const sslpl_kfset* k, const int32_t* d_ref, int nframes,
                                     const uint8_t* d_desc, const sslpl_keypoint* d_kps, const int* d_n, int cap,
                                     const uint8_t* d_ldesc, const int* d_nl, int capl,
                                     const sslpl_vocab* v, int levelsup, float nnratio, int checkOrientation,
                                     int32_t* d_match, int32_t* d_nmatch, int32_t* d_lmatch, int32_t* d_nlmatch);

/* =====================================================================================
 * (2) Line segments — replaces LineSegment::ExtractLineSegment (src/ExtractLineSegment.cpp:18-69)
 * ===================================================================================== */
typedef struct sslpl_line sslpl_line;
typedef struct {
    int lsdNFeatures;     /* hard-coded 40 in the reference (ExtractLineSegment.cpp:42) */
    int max_width, max_height, max_batch, device;
} sslpl_line_params;
int  sslpl_line_create(const sslpl_line_params* p, sslpl_line** out);
void sslpl_line_destroy(sslpl_line* h);
/* ExtractLineSegment(img, keylines, ldesc, keylineFunctions, scale=1, numOctaves=1): kl[cap], ldesc[cap*32], lineeq[cap*3] */
int  sslpl_line_extract(sslpl_line* h, const uint8_t* img, int width, int height, int pitch,
                        sslpl_keyline* kl, uint8_t* ldesc, double* lineeq, int cap, int* n);
int  sslpl_line_extract_batch(sslpl_line* h, const uint8_t* imgs, int nframes, int width, int height, int pitch,
                              size_t frame_stride, sslpl_keyline* kl, uint8_t* ldesc, double* lineeq, int cap, int* n);
/* asynchronous form (finish with sslpl_line_sync) */
int  sslpl_line_extract_batch_begin(sslpl_line* h, const uint8_t* imgs, int nframes, int width, int height, int pitch,
                                    size_t frame_stride, sslpl_keyline* kl, uint8_t* ldesc, double* lineeq, int cap, int* n);
int  sslpl_line_extract_batch_device(sslpl_line* h, const uint8_t* d_imgs, int nframes, int width, int height, int pitch,
                                     size_t frame_stride);
int  sslpl_line_device_results(sslpl_line* h, const sslpl_keyline** d_kl, const uint8_t** d_ldesc, const double** d_lineeq,
                               const int** d_n, int* cap);
int  sslpl_line_sync(sslpl_line* h);
void* sslpl_line_stream(sslpl_line* h);
int  sslpl_line_set_stream(sslpl_line* h, void* cuda_stream);
long long sslpl_line_launch_count(const sslpl_line* h);
/* Scheduling knob (no effect on results): the LSD region stage runs one multi-warp CTA per frame; bound how many of them one
   call keeps resident (0 = one per frame, the default).  Useful when several handles are in flight on one GPU next to wide
   kernels: resident walkers pin registers for milliseconds. */
int  sslpl_line_set_max_walkers(sslpl_line* h, int max_concurrent);
/* Statistics of the last region-walker launch, 16 values (see csrc/line.cu): regions grown by the turn holder / as speculated,
   redo causes, cycles under the commit and claim locks, cycles per frame.  Diagnostic only. */
int  sslpl_line_walker_stats(sslpl_line* h, unsigned long long* out16);
int  sslpl_line_set_profiling(sslpl_line* h, int on);
int  sslpl_line_stage_ms(sslpl_line* h, float* ms, int cap, const char** names, int* nstages);
/* raw LSD segments (before the top-N cut) of frame f of the last call: seg[4*i] = x1,y1,x2,y2 */
int  sslpl_line_download_segments(sslpl_line* h, int frame, float* seg4, int cap, int* n);
/* debug: with SSLPL_LINE_TRACE=1 in the environment at create time, one row of 10 doubles per LSD region that reached
   region2rect: seed pixel, size before/after refine, log_nfa, x1,y1,x2,y2,width,p (detection scale) */
int  sslpl_line_debug_trace(sslpl_line* h, int frame, double* out, int cap_rows, int* n);

/* =====================================================================================
 * (4) Frame level — what Frame::Frame(imGray, ...) does with the two extractors (src/Frame.cc:69-131), the colour conversion in
 *     front of it (Tracking::GrabImageMonocularWithPL, src/Tracking.cc:148-161) and Frame::UndistortKeyPoints /
 *     ComputeImageBounds behind it (src/Frame.cc:483-543).  ONE upload of the frame; ORB and LSD+LBD on two streams.
 * ===================================================================================== */
typedef struct sslpl_frame sslpl_frame;
typedef struct { sslpl_orb_params orb; sslpl_line_params line; } sslpl_frame_params;   /* device, max_batch and max size must agree */
int  sslpl_frame_create(const sslpl_frame_params* p, sslpl_frame** out);
void sslpl_frame_destroy(sslpl_frame* h);
sslpl_orb*  sslpl_frame_orb(sslpl_frame* h);     /* the extractors it owns (device results, tables, stage times) */
sslpl_line* sslpl_frame_line(sslpl_frame* h);
long long sslpl_frame_launch_count(const sslpl_frame* h);
/* Camera.fx/fy/cx/cy and k1 k2 p1 p2 [k3] (Tracking.cc:58-86); undistortion is skipped when k1 == 0 (Frame.cc:485) */
int  sslpl_frame_set_camera(sslpl_frame* h, float fx, float fy, float cx, float cy, const float* dist, int ndist);
int  sslpl_frame_image_bounds(sslpl_frame* h, int cols, int rows, float* bounds4 /* mnMinX mnMaxX mnMinY mnMaxY */);
/* channels 1 (grey), 3 or 4 (interleaved 8-bit; rgb_order 1 = RGB[A], 0 = BGR[A] as Camera.RGB says).  Any output pointer but the
   counts may be NULL.  kps / kps_un / desc hold `cap` entries per frame (>= sslpl_orb_max_keypoints), the line outputs `lcap`. */
int  sslpl_frame_extract(sslpl_frame* h, const uint8_t* img, int width, int height, int pitch, int channels, int rgb_order,
                         sslpl_keypoint* kps, sslpl_keypoint* kps_un, uint8_t* desc, int cap, int* nkp,
                         sslpl_keyline* kl, uint8_t* ldesc, double* lineeq, int lcap, int* nl);
int  sslpl_frame_extract_batch(sslpl_frame* h, const uint8_t* imgs, int nframes, int width, int height, int pitch, size_t frame_stride,
                               int channels, int rgb_order,
                               sslpl_keypoint* kps, sslpl_keypoint* kps_un, uint8_t* desc, int cap, int* nkp,
                               sslpl_keyline* kl, uint8_t* ldesc, double* lineeq, int lcap, int* nl);
/* asynchronous form: enqueue only (pinned host buffers), finish with sslpl_frame_sync */
int  sslpl_frame_extract_batch_begin(sslpl_frame* h, const uint8_t* imgs, int nframes, int width, int height, int pitch, size_t frame_stride,
                                     int channels, int rgb_order,
                                     sslpl_keypoint* kps, sslpl_keypoint* kps_un, uint8_t* desc, int cap, int* nkp,
                                     sslpl_keyline* kl, uint8_t* ldesc, double* lineeq, int lcap, int* nl);
int  sslpl_frame_sync(sslpl_frame* h);
void* sslpl_frame_stream(sslpl_frame* h, int which /* 0 = ORB stream, 1 = line stream */);
int  sslpl_frame_device_gray(sslpl_frame* h, const uint8_t** d_gray, int* pitch, size_t* frame_stride);

#ifdef __cplusplus
}
#endif
#endif /* SSLPL_H */
