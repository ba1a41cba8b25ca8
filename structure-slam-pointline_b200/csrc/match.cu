// match.cu — B200 (sm_100a) Hamming matchers: brute-force 2-NN (cv::BFMatcher knnMatch k=2), vocabulary-node
// assignment, SearchByBoW (KF-Frame and KF-KF), SearchForTriangulation, rotation-histogram filter, and the
// knn-based LSDmatcher entry points.  Replaces the distance work of src/ORBmatcher.cc and src/LSDmatcher.cpp.
//
// No tensor cores: 256-bit XOR + popcount per pair, reduced with warp shuffles.  Descriptors are read as
// 2 x uint4 per row.  The batched layout is "a set of frames": frame f owns desc[f*cap..], a CSR feature
// vector and optional masks; pair p matches frame p (KeyFrame role) against frame p+1 (Frame role), or, for reference-keyframe
// matching, frame f against the keyframe slot d_ref[f] of a keyframe set (sslpl_kfset).
#include "common.cuh"
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <vector>

namespace sslpl {

constexpr int TH_LOW = 50;          // ORBmatcher.cc:38
constexpr int MAX_DYN_SMEM = 200 * 1024;   // dynamic shared memory the two data-dependent kernels may ask for (sm_100: 227 KB per CTA, static included)
constexpr int HISTO_LENGTH = 30;    // ORBmatcher.cc:39

// A set of frames in HBM (strides in elements of the respective type)
struct FrameSet {
    const uint8_t* desc; long long desc_fs;                  // 32 B per row; frame stride in bytes
    const int* n; int n_const;                               // per-frame feature count (device array) or constant
    const int* nodes; const int* off; const int* idx; const int* nn; int nn_const;
    long long nodes_fs, off_fs, idx_fs;                      // CSR frame strides (ints)
    const uint8_t* flag; long long flag_fs;                  // valid / has-MapPoint mask (may be null)
    const float* angle; int angle_es; long long angle_fs;    // keypoint angle: element stride / frame stride in floats
    const float* x; const float* y; const int* oct;          // same strides as angle (fields of sslpl_keypoint)
};

__device__ __forceinline__ void load_desc(const uint8_t* p, uint4& a, uint4& b) {
    const uint4* q = reinterpret_cast<const uint4*>(p);
    a = __ldg(q); b = __ldg(q + 1);
}

// -------------------------------------------------------------------------------------------------
// knnMatch(k=2): one warp per query.  key = dist << 20 | trainIdx  => ascending distance, ties -> lower index
// -------------------------------------------------------------------------------------------------
__device__ __forceinline__ void top2_insert(unsigned& k0, unsigned& k1, unsigned k) {
    if (k < k0) { k1 = k0; k0 = k; } else if (k < k1) k1 = k;
}

// the two nearest of the nt train rows T to one query (a0, a1), computed by a whole warp; the result is in every lane
__device__ __forceinline__ int4 knn2_warp(uint4 a0, uint4 a1, const uint8_t* T, int nt, int lane) {
    unsigned k0 = 0xffffffffu, k1 = 0xffffffffu;
    for (int j = lane; j < nt; j += 32) {
        uint4 b0, b1;
        load_desc(T + (long long)j * 32, b0, b1);
        top2_insert(k0, k1, ((unsigned)popc256(a0, a1, b0, b1) << 20) | (unsigned)j);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const unsigned o0 = __shfl_xor_sync(0xffffffffu, k0, o), o1 = __shfl_xor_sync(0xffffffffu, k1, o);
        top2_insert(k0, k1, o0);
        top2_insert(k0, k1, o1);
    }
    int4 r;
    r.x = k0 == 0xffffffffu ? -1 : (int)(k0 & 0xfffff); r.y = k0 == 0xffffffffu ? -1 : (int)(k0 >> 20);
    r.z = k1 == 0xffffffffu ? -1 : (int)(k1 & 0xfffff); r.w = k1 == 0xffffffffu ? -1 : (int)(k1 >> 20);
    return r;
}

__global__ void __launch_bounds__(256) k_knn2(const uint8_t* q, long long q_fs, const int* nq_arr, int nq_const,
                                               const uint8_t* t, long long t_fs, const int* nt_arr, int nt_const,
                                               int32_t* out, long long out_fs, int qcap) {
    const int pair = blockIdx.y, lane = threadIdx.x & 31, qi = blockIdx.x * 8 + (threadIdx.x >> 5);
    const int nq = nq_arr ? min(nq_arr[pair], qcap) : nq_const, nt = nt_arr ? min(nt_arr[pair + 1], qcap) : nt_const;
    if (qi >= nq) return;
    uint4 a0, a1;
    load_desc(q + pair * q_fs + (long long)qi * 32, a0, a1);
    const int4 r = knn2_warp(a0, a1, t + pair * t_fs, nt, lane);
    if (lane == 0) reinterpret_cast<int4*>(out + pair * out_fs)[qi] = r;
}

// DescriptorDistance for n pairs (ORBmatcher.cc:1650): thread per pair
__global__ void k_pair_distance(const uint8_t* a, const uint8_t* b, int n, int32_t* dist) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint4 a0, a1, b0, b1;
    load_desc(a + (long long)i * 32, a0, a1); load_desc(b + (long long)i * 32, b0, b1);
    dist[i] = popc256(a0, a1, b0, b1);
}

// -------------------------------------------------------------------------------------------------
// Vocabulary node assignment: nearest centroid, strict '<' (first wins).  Thread per descriptor,
// centroids staged in shared memory.
// -------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) k_bow_assign(const uint8_t* desc, long long desc_fs, const int* n_arr, int n_const, int cap,
                                                     const uint8_t* centroids, int nc, int32_t* node, long long node_fs) {
    extern __shared__ uint4 s_cent[];
    const int f = blockIdx.y;
    for (int i = threadIdx.x; i < nc * 2; i += blockDim.x) s_cent[i] = __ldg(reinterpret_cast<const uint4*>(centroids) + i);
    __syncthreads();
    const int n = n_arr ? min(n_arr[f], cap) : n_const;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint4 a0, a1;
    load_desc(desc + f * desc_fs + (long long)i * 32, a0, a1);
    int best = 1 << 30, bi = 0;
    for (int c = 0; c < nc; c++) {
        const int d = popc256(a0, a1, s_cent[2 * c], s_cent[2 * c + 1]);
        if (d < best) { best = d; bi = c; }
    }
    node[f * node_fs + i] = bi;
}

// -------------------------------------------------------------------------------------------------
// DBoW2 TemplatedVocabulary<FORB>::transform (Thirdparty/DBoW2/DBoW2/TemplatedVocabulary.h:1218-1259): descend the
// k-ary tree by Hamming distance (strict '<': the first best child wins), one thread per descriptor.  The tree is
// stored as CSR children lists (ascending node id, as loadFromTextFile builds them) + 32-byte node descriptors; the
// upper levels stay resident in L1/L2 (ORBvoc: 1.1 M nodes x 32 B = 35 MB < 126 MB L2).
//   word  = word id of the leaf,  node = NodeId at level L - levelsup (0 if the leaf comes earlier),
//   rank  = dense index of `node` among the possible values (0 = root / early leaf, 1 + rank inside the level), or -1 for a
//           stopped word (weight <= 0), which the reference keeps out of the FeatureVector (:1162-1166).
// -------------------------------------------------------------------------------------------------
struct VocabView { const int* child_off; const int* child_ids; const uint8_t* desc; const double* weight; const int* word_id; const int* level_rank; };

__global__ void __launch_bounds__(128) k_vocab_transform(const uint8_t* desc, long long desc_fs, const int* n_arr, int n_const, int cap,
                                                          VocabView V, int nid_level, int32_t* word, int32_t* node, int32_t* rank,
                                                          double* weight, long long out_fs) {
    const int f = blockIdx.y;
    const int n = n_arr ? min(n_arr[f], cap) : n_const;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint4 a0, a1;
    load_desc(desc + f * desc_fs + (long long)i * 32, a0, a1);
    int cur = 0, nid = 0, level = 0;
    int cb = __ldg(V.child_off), ce = __ldg(V.child_off + 1);
    while (ce > cb) {
        ++level;
        int best = 1 << 30, bi = 0;
        for (int c = cb; c < ce; c++) {
            const int id = __ldg(V.child_ids + c);
            uint4 b0, b1;
            load_desc(V.desc + (long long)id * 32, b0, b1);
            const int d = popc256(a0, a1, b0, b1);
            if (d < best) { best = d; bi = id; }
        }
        cur = bi;
        if (level == nid_level) nid = cur;
        cb = __ldg(V.child_off + cur); ce = __ldg(V.child_off + cur + 1);
    }
    const double w = __ldg(V.weight + cur);
    const long long o = f * out_fs + i;
    if (word) word[o] = __ldg(V.word_id + cur);
    if (node) node[o] = nid;
    if (weight) weight[o] = w;
    if (rank) rank[o] = (w > 0) ? (nid == 0 ? 0 : 1 + __ldg(V.level_rank + nid)) : -1;
}

// FeatureVector build for a dense vocabulary (every node 0..nc-1 listed, possibly empty): CSR with
// ascending feature indices per node (FeatureVector.cpp:31-45).  One CTA per frame, thread per node.
__global__ void __launch_bounds__(128) k_build_csr(const int32_t* node, long long node_fs, const int* n_arr, int cap, int nc,
                                                    int* off, long long off_fs, int* idx, long long idx_fs) {
    __shared__ int s_warp[33];
    extern __shared__ int s_dyn[];        // nc + 1 counters, then the frame's node ids (cap ints)
    int* s_cnt = s_dyn; int* s_nd = s_dyn + nc + 1;
    const int f = blockIdx.x, tid = threadIdx.x;
    const int n = min(n_arr[f], cap);
    const int32_t* nd = node + f * node_fs;
    for (int c = tid; c <= nc; c += blockDim.x) s_cnt[c] = 0;
    __syncthreads();
    for (int i = tid; i < n; i += blockDim.x) { const int v = nd[i]; s_nd[i] = v; if (v >= 0) atomicAdd(&s_cnt[v], 1); }   // v < 0: stopped word, not in the FeatureVector
    __syncthreads();
    block_scan_array(s_cnt, nc + 1, s_warp);                  // exclusive offsets, s_cnt[nc] = n
    for (int c = tid; c <= nc; c += blockDim.x) off[f * off_fs + c] = s_cnt[c];
    __syncthreads();
    // stable fill: thread c walks the node ids in index order (broadcast reads from shared memory)
    for (int c = tid; c < nc; c += blockDim.x) {
        int o = s_cnt[c];
        const int e = s_cnt[c + 1];
        for (int i = 0; i < n && o < e; i++) if (s_nd[i] == c) idx[f * idx_fs + o++] = i;
    }
}

// -------------------------------------------------------------------------------------------------
// SearchByBoW — one warp per (pair, node of set 1).  Nodes are independent (a feature belongs to exactly
// one node), the greedy exclusion inside a node is sequential over the KF features in list order.
//   mode 0: KF vs Frame  (ORBmatcher.cc:159-291): out = match2[F idx] = KF idx, accept best <= TH_LOW
//   mode 1: KF vs KF     (ORBmatcher.cc:525-658): out = match12[idx1] = idx2, accept best <  TH_LOW, both need MapPoints
// rot[i] holds the rotation-histogram bin of the match written at out[i] (or 255).
// -------------------------------------------------------------------------------------------------
__device__ __forceinline__ int rot_bin(float a1, float a2) {                 // ORBmatcher.cc:241-246
    float rot = __fsub_rn(a1, a2);
    if (rot < 0.0f) rot = __fadd_rn(rot, 360.0f);
    int bin = (int)roundf(__fmul_rn(rot, 1.0f / HISTO_LENGTH));
    if (bin == HISTO_LENGTH) bin = 0;
    return bin;
}

__device__ __forceinline__ int find_node(const int* nodes, int nn, int id) {   // map::find on the ascending CSR node list
    int lo = 0, hi = nn;
    while (lo < hi) { int mid = (lo + hi) >> 1; if (nodes[mid] < id) lo = mid + 1; else hi = mid; }
    return (lo < nn && nodes[lo] == id) ? lo : -1;
}

// One node shared by both FeatureVectors: KF features idx1[b1..e1) against frame features idx2[b2..e2), in list order.
__device__ __forceinline__ void bow_match_node(int mode, float nnratio, int lane, int b1, int e1, int b2, int e2,
                                               const int* idx1, const int* idx2, const uint8_t* D1, const uint8_t* D2,
                                               const uint8_t* v1, const uint8_t* v2, const float* A1, int es1, const float* A2, int es2,
                                               int32_t* O, uint8_t* R, uint8_t* TK) {
    for (int i1 = b1; i1 < e1; i1++) {
        const int id1 = idx1[i1];
        if (v1 && !v1[id1]) continue;                                            // :196-200 / :563-567
        uint4 a0, a1;
        load_desc(D1 + (long long)id1 * 32, a0, a1);
        // per-lane best / second best over this lane's candidates, in list order: key = dist << 20 | position
        unsigned k0 = 0xffffffffu, k1 = 0xffffffffu;
        for (int i2 = b2 + lane; i2 < e2; i2 += 32) {
            const int id2 = idx2[i2];
            if (TK[id2]) continue;                                               // :212 / :579 (already matched)
            if (mode == 1 && v2 && !v2[id2]) continue;                           // :579-583
            uint4 c0, c1;
            load_desc(D2 + (long long)id2 * 32, c0, c1);
            top2_insert(k0, k1, ((unsigned)popc256(a0, a1, c0, c1) << 20) | (unsigned)(i2 - b2));
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const unsigned o0 = __shfl_xor_sync(0xffffffffu, k0, o), o1 = __shfl_xor_sync(0xffffffffu, k1, o);
            top2_insert(k0, k1, o0);
            top2_insert(k0, k1, o1);
        }
        // bestDist1 = smallest distance (first position wins), bestDist2 = second order statistic; both start at 256
        const int best1 = k0 == 0xffffffffu ? 256 : (int)(k0 >> 20);
        const int best2 = k1 == 0xffffffffu ? 256 : (int)(k1 >> 20);
        const bool th = mode == 0 ? best1 <= TH_LOW : best1 < TH_LOW;             // :231 / :601
        if (k0 != 0xffffffffu && th && (float)best1 < __fmul_rn(nnratio, (float)best2)) {      // :233
            const int id2 = idx2[b2 + (int)(k0 & 0xfffff)];
            if (lane == 0) {
                TK[id2] = 1;
                const int bin = rot_bin(A1[(long long)id1 * es1], A2[(long long)id2 * es2]);
                if (mode == 0) { O[id2] = id1; R[id2] = (uint8_t)bin; }
                else { O[id1] = id2; R[id1] = (uint8_t)bin; }
            }
        }
        __syncwarp();
    }
}

__global__ void __launch_bounds__(128) k_bow_match(FrameSet S, int mode, float nnratio, int cap,
                                                    int32_t* out, long long out_fs, uint8_t* rot, long long rot_fs,
                                                    uint8_t* taken, long long taken_fs) {
    const int pair = blockIdx.y, lane = threadIdx.x & 31, a = blockIdx.x * 4 + (threadIdx.x >> 5);
    const int f1 = pair, f2 = pair + 1;
    const int nn1 = S.nn ? S.nn[f1] : S.nn_const, nn2 = S.nn ? S.nn[f2] : S.nn_const;
    if (a >= nn1) return;
    const int* nodes1 = S.nodes + f1 * S.nodes_fs; const int* nodes2 = S.nodes + f2 * S.nodes_fs;
    const int b = find_node(nodes2, nn2, nodes1[a]);
    if (b < 0) return;
    const int* off1 = S.off + f1 * S.off_fs; const int* off2 = S.off + f2 * S.off_fs;
    const int* idx1 = S.idx + f1 * S.idx_fs; const int* idx2 = S.idx + f2 * S.idx_fs;
    const uint8_t* D1 = S.desc + f1 * S.desc_fs; const uint8_t* D2 = S.desc + f2 * S.desc_fs;
    const uint8_t* v1 = S.flag ? S.flag + f1 * S.flag_fs : nullptr;
    const uint8_t* v2 = S.flag ? S.flag + f2 * S.flag_fs : nullptr;
    const float* A1 = S.angle + f1 * S.angle_fs; const float* A2 = S.angle + f2 * S.angle_fs;
    int32_t* O = out + pair * out_fs; uint8_t* R = rot + pair * rot_fs; uint8_t* TK = taken + pair * taken_fs;
    bow_match_node(mode, nnratio, lane, off1[a], off1[a + 1], off2[b], off2[b + 1], idx1, idx2, D1, D2, v1, v2,
                   A1, S.angle_es, A2, S.angle_es, O, R, TK);
}

// -------------------------------------------------------------------------------------------------
// Keyframe set (sslpl_kfset): per slot s, `cap` ORB rows and `capl` LBD rows.  The FeatureVector is sparse: nn[s] non-empty
// nodes in ascending id, nodes[s*cap + a], off[s*(cap+1) + a], idx[s*cap + ..] (a node holds at least one feature, so
// nn <= cap).  An empty or cleared slot has nn = n = nl = 0 and matches nothing.
// -------------------------------------------------------------------------------------------------
struct KfView {
    uint8_t* desc; float* angle; uint8_t* valid;
    int* nodes; int* off; int* idx; int* nn;
    uint8_t* ldesc; uint8_t* has_ml; int* nl;
    int cap, capl, nslots;
};

__device__ __forceinline__ int kf_slot(const KfView& K, const int32_t* ref, int f) {
    const int s = ref[f];
    return (s >= 0 && s < K.nslots) ? s : -1;
}

// Keyframe side of a stored slot's FeatureVector: k_build_csr's dense offsets (nc + 1 entries) compacted to the non-empty
// nodes, and the slot's line count.  One CTA of 256 threads.
__global__ void __launch_bounds__(256) k_kf_compact(const int* dense_off, int nc, const int* nl_src, int capl_src,
                                                     int* nodes, int* off, int* nn, int* nl_out) {
    __shared__ int s_warp[33];
    int base = 0;
    for (int c0 = 0; c0 < nc; c0 += 256) {
        const int c = c0 + threadIdx.x;
        const int lo = c < nc ? dense_off[c] : 0;
        const int keep = c < nc && dense_off[c + 1] > lo;
        int total;
        const int o = base + block_exclusive_scan(keep, s_warp, &total);
        if (keep) { nodes[o] = c; off[o] = lo; }
        base += total;
    }
    if (threadIdx.x == 0) {
        off[base] = dense_off[nc];
        *nn = base;
        *nl_out = min(*nl_src, capl_src);
    }
}

// SearchByBoW(KF ref[f], frame f), mode 0 (ORBmatcher.cc:159-291): one warp per (frame, node of the keyframe).  The frame side
// is the batch's dense FeatureVector (S.nodes = 0..nc-1).
__global__ void __launch_bounds__(128) k_bow_match_ref(KfView K, const int32_t* ref, FrameSet S, float nnratio,
                                                        int32_t* out, long long out_fs, uint8_t* rot, long long rot_fs,
                                                        uint8_t* taken, long long taken_fs) {
    const int f = blockIdx.y, lane = threadIdx.x & 31, a = blockIdx.x * 4 + (threadIdx.x >> 5);
    const int s = kf_slot(K, ref, f);
    if (s < 0 || a >= K.nn[s]) return;
    const long long ks = (long long)s * K.cap;
    const int b = find_node(S.nodes, S.nn_const, K.nodes[ks + a]);
    if (b < 0) return;
    const int* off1 = K.off + (long long)s * (K.cap + 1); const int* off2 = S.off + f * S.off_fs;
    bow_match_node(0, nnratio, lane, off1[a], off1[a + 1], off2[b], off2[b + 1], K.idx + ks, S.idx + f * S.idx_fs,
                   K.desc + ks * 32, S.desc + f * S.desc_fs, K.valid + ks, nullptr, K.angle + ks, 1, S.angle + f * S.angle_fs, S.angle_es,
                   out + f * out_fs, rot + f * rot_fs, taken + f * taken_fs);
}

// knnMatch(KF ref[f] lines, frame f lines, k=2) for LSDmatcher::SearchByProjection(KF,F) (LSDmatcher.cpp:155): row q of frame f
// is the KF line q's two nearest frame lines, or -1s when the slot is empty, q is past its lines, or line q holds no MapLine
// (:169 rejects those rows whatever their distances), so k_line_ratio needs no mask.  Rows [0, qcap) are all written.
__global__ void __launch_bounds__(256) k_knn2_ref(KfView K, const int32_t* ref, const uint8_t* t, long long t_fs, const int* nt_arr, int ntcap,
                                                   int32_t* out, long long out_fs, int qcap) {
    const int f = blockIdx.y, lane = threadIdx.x & 31, qi = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (qi >= qcap) return;
    const int s = kf_slot(K, ref, f);
    const long long ks = (long long)max(s, 0) * K.capl;
    int4 r = make_int4(-1, -1, -1, -1);
    if (s >= 0 && qi < K.nl[s] && K.has_ml[ks + qi]) {
        uint4 a0, a1;
        load_desc(K.ldesc + (ks + qi) * 32, a0, a1);
        r = knn2_warp(a0, a1, t + f * t_fs, min(nt_arr[f], ntcap), lane);
    }
    if (lane == 0) reinterpret_cast<int4*>(out + f * out_fs)[qi] = r;
}

// SearchForTriangulation (ORBmatcher.cc:660-826, monocular): warp per node of set 1; no dependency between
// idx1's (vbMatched2 is never set), so the lanes only cooperate on the scan of the node's idx2 list.
struct TriArgs { float F[9]; float ex, ey; float scale[SSLPL_MAX_LEVELS]; float sigma2[SSLPL_MAX_LEVELS]; };

__global__ void __launch_bounds__(128) k_tri_match(FrameSet S, TriArgs T, int32_t* out, long long out_fs, uint8_t* rot, long long rot_fs) {
    const int pair = blockIdx.y, lane = threadIdx.x & 31, a = blockIdx.x * 4 + (threadIdx.x >> 5);
    const int f1 = pair, f2 = pair + 1;
    const int nn1 = S.nn ? S.nn[f1] : S.nn_const, nn2 = S.nn ? S.nn[f2] : S.nn_const;
    if (a >= nn1) return;
    const int* nodes1 = S.nodes + f1 * S.nodes_fs; const int* nodes2 = S.nodes + f2 * S.nodes_fs;
    const int b = find_node(nodes2, nn2, nodes1[a]);
    if (b < 0) return;
    const int* off1 = S.off + f1 * S.off_fs; const int* off2 = S.off + f2 * S.off_fs;
    const int* idx1 = S.idx + f1 * S.idx_fs; const int* idx2 = S.idx + f2 * S.idx_fs;
    const uint8_t* D1 = S.desc + f1 * S.desc_fs; const uint8_t* D2 = S.desc + f2 * S.desc_fs;
    const uint8_t* m1 = S.flag + f1 * S.flag_fs; const uint8_t* m2 = S.flag + f2 * S.flag_fs;
    const long long es = S.angle_es;
    const float* A1 = S.angle + f1 * S.angle_fs; const float* A2 = S.angle + f2 * S.angle_fs;
    const float* X1 = S.x + f1 * S.angle_fs; const float* Y1 = S.y + f1 * S.angle_fs;
    const float* X2 = S.x + f2 * S.angle_fs; const float* Y2 = S.y + f2 * S.angle_fs;
    const int* OC2 = S.oct + f2 * S.angle_fs;
    const int b1 = off1[a], e1 = off1[a + 1], b2 = off2[b], e2 = off2[b + 1];
    for (int i1 = b1; i1 < e1; i1++) {
        const int id1 = idx1[i1];
        if (m1[id1]) continue;                                                    // :702-706
        uint4 a0, a1;
        load_desc(D1 + (long long)id1 * 32, a0, a1);
        const float x1 = X1[id1 * es], y1 = Y1[id1 * es];
        // epipolar line l = x1' F12 (CheckDistEpipolarLine :143-145), f32 without contraction
        const float la = __fadd_rn(__fadd_rn(__fmul_rn(x1, T.F[0]), __fmul_rn(y1, T.F[3])), T.F[6]);
        const float lb = __fadd_rn(__fadd_rn(__fmul_rn(x1, T.F[1]), __fmul_rn(y1, T.F[4])), T.F[7]);
        const float lc = __fadd_rn(__fadd_rn(__fmul_rn(x1, T.F[2]), __fmul_rn(y1, T.F[5])), T.F[8]);
        const float den = __fadd_rn(__fmul_rn(la, la), __fmul_rn(lb, lb));
        unsigned best = 0xffffffffu;              // min over (dist << 20 | (0xfffff - position)): min distance, LAST wins (:741)
        for (int i2 = b2 + lane; i2 < e2; i2 += 32) {
            const int id2 = idx2[i2];
            if (m2[id2]) continue;                                                // :725-729
            uint4 c0, c1;
            load_desc(D2 + (long long)id2 * 32, c0, c1);
            const int dist = popc256(a0, a1, c0, c1);
            if (dist > TH_LOW) continue;
            const float x2 = X2[id2 * es], y2 = Y2[id2 * es];
            const int oc = OC2[id2 * es];
            const float dex = __fsub_rn(T.ex, x2), dey = __fsub_rn(T.ey, y2);
            if (__fadd_rn(__fmul_rn(dex, dex), __fmul_rn(dey, dey)) < __fmul_rn(100.f, T.scale[oc])) continue;    // :749-751
            const float num = __fadd_rn(__fadd_rn(__fmul_rn(la, x2), __fmul_rn(lb, y2)), lc);
            if (den == 0.f) continue;
            const float dsqr = __fdiv_rn(__fmul_rn(num, num), den);
            if (!((double)dsqr < 3.84 * (double)T.sigma2[oc])) continue;          // :156 (double compare)
            const unsigned key = ((unsigned)dist << 20) | (0xfffffu - (unsigned)(i2 - b2));
            best = min(best, key);
        }
        best = __reduce_min_sync(0xffffffffu, best);
        if (best != 0xffffffffu && lane == 0) {
            const int id2 = idx2[b2 + (int)(0xfffffu - (best & 0xfffffu))];
            out[pair * out_fs + id1] = id2;
            rot[pair * rot_fs + id1] = (uint8_t)rot_bin(A1[id1 * es], A2[id2 * es]);
        }
    }
}

// -------------------------------------------------------------------------------------------------
// SURVEY.md 8(f) row 2: Frame::AssignFeaturesToGrid (Frame.cc:133-148, PosInGrid :462-472) as a CSR over the 64 x 48 cells
// (cell id = ix * 48 + iy: the traversal order of GetFeaturesInArea, Frame.cc:368-421) and
// ORBmatcher::SearchByProjection(Frame &CurrentFrame, const Frame &LastFrame, th, bMono) (ORBmatcher.cc:1331-1473).
// The matcher is a greedy scan over the last frame's MapPoints in index order (a feature of the current frame that has
// received a MapPoint with observations is skipped by later points), so ONE WARP walks a frame pair sequentially; the lanes
// share the grid cells of each search window.  First-wins ties are kept by reducing (distance, traversal position) keys.
// -------------------------------------------------------------------------------------------------
constexpr int GRID_COLS = 64, GRID_ROWS = 48;        // Frame.h:45-46
constexpr int TH_HIGH = 100;                         // ORBmatcher.cc:37

struct ProjArgs {
    float T[12];                                     // Tcw, 3x4 row-major
    float fx, fy, cx, cy, mbf;
    float minX, maxX, minY, maxY, invW, invH;
    float th;
    int forward, backward, checkOri, use_right;
    float scale[32];                                 // mvScaleFactors
};

__global__ void __launch_bounds__(128) k_grid_cells(const float* x, const float* y, int n, float minX, float minY, float invW, float invH, int32_t* cell) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int px = (int)roundf(__fmul_rn(__fsub_rn(x[i], minX), invW)), py = (int)roundf(__fmul_rn(__fsub_rn(y[i], minY), invH));
    cell[i] = (px < 0 || px >= GRID_COLS || py < 0 || py >= GRID_ROWS) ? -1 : px * GRID_ROWS + py;
}

__global__ void __launch_bounds__(32) k_proj_match(const __grid_constant__ ProjArgs A, int n1, const uint8_t* flag1 /* bit0 valid, bit1 obs>0 */,
                                                    const float* Xw, const uint8_t* dmp, const int* oct1, const float* angle1,
                                                    int n2, const uint8_t* d2, const float* x2, const float* y2, const int* oct2, const float* angle2,
                                                    const float* uright2, uint8_t* claimed, const int* goff, const int* gidx,
                                                    int32_t* assign2, int32_t* sel, uint8_t* rbin, int32_t* nmatch) {
    __shared__ int s_hist[HISTO_LENGTH];
    __shared__ int s_keep[3];
    const int lane = threadIdx.x;
    for (int j = lane; j < n2; j += 32) assign2[j] = -1;
    if (lane < HISTO_LENGTH) s_hist[lane] = 0;
    __syncwarp();
    int nmatches = 0;
    for (int i = 0; i < n1; i++) {
        if (lane == 0) sel[i] = -1;
        const int fl = flag1[i];
        if (!(fl & 1)) continue;
        const float X0 = Xw[3 * i], X1 = Xw[3 * i + 1], X2 = Xw[3 * i + 2];
        // Rcw * x3Dw + tcw (ORBmatcher.cc:1364): cv::gemm runs a plain 3x3 * 3x1 (+ 3x1) CV_32F product in FLOAT, products summed
        // left to right, the addend last (probed on cv2 4.13, tools/probe_cv_gemm.py; the reference compiled over that model
        // agrees with the oracle in tests/test_ref_parity_cpu.py).  Explicit _rn intrinsics: no FMA contraction.
        const float xc = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(A.T[0], X0), __fmul_rn(A.T[1], X1)), __fmul_rn(A.T[2], X2)), A.T[3]);
        const float yc = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(A.T[4], X0), __fmul_rn(A.T[5], X1)), __fmul_rn(A.T[6], X2)), A.T[7]);
        const float zc = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(A.T[8], X0), __fmul_rn(A.T[9], X1)), __fmul_rn(A.T[10], X2)), A.T[11]);
        const float invzc = (float)(1.0 / (double)zc);
        if (invzc < 0) continue;
        const float u = __fadd_rn(__fmul_rn(__fmul_rn(A.fx, xc), invzc), A.cx), v = __fadd_rn(__fmul_rn(__fmul_rn(A.fy, yc), invzc), A.cy);
        if (u < A.minX || u > A.maxX || v < A.minY || v > A.maxY) continue;
        const int lo = oct1[i];
        const float r = __fmul_rn(A.th, A.scale[lo]);
        const int minLevel = A.forward ? lo : (A.backward ? 0 : lo - 1), maxLevel = A.forward ? -1 : (A.backward ? lo : lo + 1);
        // GetFeaturesInArea (Frame.cc:368-421)
        const int cx0 = max(0, (int)floorf(__fmul_rn(__fsub_rn(__fsub_rn(u, A.minX), r), A.invW)));
        if (cx0 >= GRID_COLS) continue;
        const int cx1 = min(GRID_COLS - 1, (int)ceilf(__fmul_rn(__fadd_rn(__fsub_rn(u, A.minX), r), A.invW)));
        if (cx1 < 0) continue;
        const int cy0 = max(0, (int)floorf(__fmul_rn(__fsub_rn(__fsub_rn(v, A.minY), r), A.invH)));
        if (cy0 >= GRID_ROWS) continue;
        const int cy1 = min(GRID_ROWS - 1, (int)ceilf(__fmul_rn(__fadd_rn(__fsub_rn(v, A.minY), r), A.invH)));
        if (cy1 < 0) continue;
        const bool checkLevels = (minLevel > 0) || (maxLevel >= 0);
        const int ny = cy1 - cy0 + 1, ncell = (cx1 - cx0 + 1) * ny;
        uint4 a0, a1;
        load_desc(dmp + (long long)i * 32, a0, a1);
        const float ur = __fsub_rn(u, __fmul_rn(A.mbf, invzc));
        unsigned long long best = ~0ull;                         // (dist << 40) | (cell rank << 20) | position in the cell
        for (int c = lane; c < ncell; c += 32) {
            const int ix = cx0 + c / ny, iy = cy0 + c % ny, cell = ix * GRID_ROWS + iy;
            const int b = goff[cell], e = goff[cell + 1];
            for (int q = b; q < e; q++) {
                const int j = gidx[q];
                if (checkLevels) {
                    const int o = oct2[j];
                    if (o < minLevel) continue;
                    if (maxLevel >= 0 && o > maxLevel) continue;
                }
                if (!(fabsf(__fsub_rn(x2[j], u)) < r && fabsf(__fsub_rn(y2[j], v)) < r)) continue;
                if (claimed[j]) continue;                        // :1400-1402
                if (A.use_right && uright2[j] > 0) { if (fabsf(__fsub_rn(ur, uright2[j])) > r) continue; }
                uint4 b0, b1;
                load_desc(d2 + (long long)j * 32, b0, b1);
                const unsigned long long key = ((unsigned long long)popc256(a0, a1, b0, b1) << 40) | ((unsigned long long)c << 20) | (unsigned)(q - b);
                if (key < best) best = key;
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) { const unsigned long long t = __shfl_xor_sync(0xffffffffu, best, o); best = t < best ? t : best; }
        const int bestDist = best == ~0ull ? 256 : (int)(best >> 40);
        if (bestDist <= TH_HIGH) {
            const int c = (int)((best >> 20) & 0xfffff), pos = (int)(best & 0xfffff);
            const int cell = (cx0 + c / ny) * GRID_ROWS + cy0 + c % ny;
            const int j = gidx[goff[cell] + pos];
            if (lane == 0) {
                assign2[j] = i; claimed[j] = (fl >> 1) & 1;
                sel[i] = j;
                const int bin = rot_bin(angle1[i], angle2[j]);
                rbin[i] = (uint8_t)bin;
                if (A.checkOri) s_hist[bin]++;
            }
            nmatches++;
        }
        __syncwarp();
    }
    __syncwarp();
    if (A.checkOri) {
        if (lane == 0) {                                         // ComputeThreeMaxima, ORBmatcher.cc:1604-1645
            int max1 = 0, max2 = 0, max3 = 0, ind1 = -1, ind2 = -1, ind3 = -1;
            for (int i = 0; i < HISTO_LENGTH; i++) {
                const int sv = s_hist[i];
                if (sv > max1) { max3 = max2; max2 = max1; max1 = sv; ind3 = ind2; ind2 = ind1; ind1 = i; }
                else if (sv > max2) { max3 = max2; max2 = sv; ind3 = ind2; ind2 = i; }
                else if (sv > max3) { max3 = sv; ind3 = i; }
            }
            if ((float)max2 < __fmul_rn(0.1f, (float)max1)) { ind2 = -1; ind3 = -1; }
            else if ((float)max3 < __fmul_rn(0.1f, (float)max1)) { ind3 = -1; }
            s_keep[0] = ind1; s_keep[1] = ind2; s_keep[2] = ind3;
        }
        __syncwarp();
        const int k0 = s_keep[0], k1 = s_keep[1], k2 = s_keep[2];
        for (int i0 = 0; i0 < n1; i0 += 32) {
            const int i = i0 + lane;
            bool drop = false;
            if (i < n1 && sel[i] >= 0) { const int b = rbin[i]; drop = (b != k0 && b != k1 && b != k2); }
            if (drop) assign2[sel[i]] = -2;                       // assigned, then removed by the rotation check: the reference NULLs it explicitly (:1461)
            nmatches -= __popc(__ballot_sync(0xffffffffu, drop));
        }
    }
    if (lane == 0) *nmatch = nmatches;
}

// -------------------------------------------------------------------------------------------------
// ORBmatcher::SearchByProjection(Frame &F, const vector<MapPoint*> &vpMapPoints, th) — ORBmatcher.cc:45-129 (Tracking::SearchLocalPoints,
// every frame) and ORBmatcher::SearchForInitialization — ORBmatcher.cc:408-523.  Both are greedy scans whose later iterations see
// what earlier ones wrote (a feature that received a MapPoint with observations is skipped; a feature matched at distance d only
// yields to a strictly smaller distance), so, like k_proj_match, ONE WARP walks the list in order and its lanes share the grid
// cells of each search window.  The reference's sequential best / second-best update keeps the two smallest candidates in
// (distance, traversal position) order: that is what the two-key reduction below computes.
// -------------------------------------------------------------------------------------------------
constexpr int TH_LOW_I = 50;                        // ORBmatcher.cc:38
struct WinArgs { float minX, minY, invW, invH, th, nnratio; int bFactor, use_right, checkOri, window; float scale[32]; };

__device__ __forceinline__ void top2_push(unsigned long long& a1, unsigned long long& a2, unsigned long long k) {
    if (k < a1) { a2 = a1; a1 = k; } else if (k < a2) a2 = k;
}
__device__ __forceinline__ void top2_warp(unsigned long long& a1, unsigned long long& a2) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const unsigned long long b1 = __shfl_xor_sync(0xffffffffu, a1, o), b2 = __shfl_xor_sync(0xffffffffu, a2, o);
        const unsigned long long lo = a1 < b1 ? a1 : b1, hi = a1 < b1 ? b1 : a1, m2 = a2 < b2 ? a2 : b2;
        a1 = lo; a2 = hi < m2 ? hi : m2;
    }
}
// the cell range of Frame::GetFeaturesInArea(x, y, r) (Frame.cc:375-393); false when the window misses the grid
__device__ __forceinline__ bool grid_window(const WinArgs& A, float x, float y, float r, int& cx0, int& cx1, int& cy0, int& cy1) {
    cx0 = max(0, (int)floorf(__fmul_rn(__fsub_rn(__fsub_rn(x, A.minX), r), A.invW)));
    if (cx0 >= GRID_COLS) return false;
    cx1 = min(GRID_COLS - 1, (int)ceilf(__fmul_rn(__fadd_rn(__fsub_rn(x, A.minX), r), A.invW)));
    if (cx1 < 0) return false;
    cy0 = max(0, (int)floorf(__fmul_rn(__fsub_rn(__fsub_rn(y, A.minY), r), A.invH)));
    if (cy0 >= GRID_ROWS) return false;
    cy1 = min(GRID_ROWS - 1, (int)ceilf(__fmul_rn(__fadd_rn(__fsub_rn(y, A.minY), r), A.invH)));
    return cy1 >= 0;
}

__global__ void __launch_bounds__(32) k_proj_match_mps(const __grid_constant__ WinArgs A, int nmp, const uint8_t* flag /* bit0 in view && !bad, bit1 obs>0 */,
                                                        const float* px, const float* py, const float* pxr, const int* level, const float* viewcos, const uint8_t* dmp,
                                                        int n2, const uint8_t* d2, const float* x2, const float* y2, const int* oct2, const float* uright2,
                                                        uint8_t* claimed, const int* goff, const int* gidx, int32_t* assign2, int32_t* nmatch) {
    const int lane = threadIdx.x;
    for (int j = lane; j < n2; j += 32) assign2[j] = -1;
    __syncwarp();
    int nmatches = 0;
    for (int i = 0; i < nmp; i++) {
        const int fl = flag[i];
        if (!(fl & 1)) continue;                                  // !mbTrackInView || isBad() (:54-58)
        const int lvl = level[i];
        float r = (double)viewcos[i] > 0.998 ? 2.5f : 4.0f;       // RadiusByViewingCos (:131-137)
        if (A.bFactor) r = __fmul_rn(r, A.th);
        const float rad = __fmul_rn(r, A.scale[lvl]);
        const float u = px[i], v = py[i];
        int cx0, cx1, cy0, cy1;
        if (!grid_window(A, u, v, rad, cx0, cx1, cy0, cy1)) continue;
        const int minLevel = lvl - 1, maxLevel = lvl;             // GetFeaturesInArea(..., nPredictedLevel-1, nPredictedLevel)
        const bool checkLevels = (minLevel > 0) || (maxLevel >= 0);
        const int ny = cy1 - cy0 + 1, ncell = (cx1 - cx0 + 1) * ny;
        uint4 a0, a1;
        load_desc(dmp + (long long)i * 32, a0, a1);
        unsigned long long b1 = ~0ull, b2 = ~0ull;                // (dist << 40) | (cell rank << 20) | position in the cell
        for (int c = lane; c < ncell; c += 32) {
            const int ix = cx0 + c / ny, iy = cy0 + c % ny, cell = ix * GRID_ROWS + iy;
            const int b = goff[cell], e = goff[cell + 1];
            for (int q = b; q < e; q++) {
                const int j = gidx[q];
                if (checkLevels) { const int o = oct2[j]; if (o < minLevel) continue; if (maxLevel >= 0 && o > maxLevel) continue; }
                if (!(fabsf(__fsub_rn(x2[j], u)) < rad && fabsf(__fsub_rn(y2[j], v)) < rad)) continue;
                if (claimed[j]) continue;                         // holds a MapPoint with observations (:86-88)
                if (A.use_right && uright2[j] > 0) { if (fabsf(__fsub_rn(pxr[i], uright2[j])) > rad) continue; }
                uint4 c0, c1;
                load_desc(d2 + (long long)j * 32, c0, c1);
                const int dist = popc256(a0, a1, c0, c1);
                if (dist >= 256) continue;                        // never below the initial bestDist = bestDist2 = 256
                top2_push(b1, b2, ((unsigned long long)dist << 40) | ((unsigned long long)c << 20) | (unsigned)(q - b));
            }
        }
        top2_warp(b1, b2);
        if (b1 == ~0ull) continue;
        const int bestDist = (int)(b1 >> 40);
        if (bestDist <= TH_HIGH) {
            const int c = (int)((b1 >> 20) & 0xfffff), pos = (int)(b1 & 0xfffff);
            const int j = gidx[goff[(cx0 + c / ny) * GRID_ROWS + cy0 + c % ny] + pos];
            int bestDist2 = 256, bestLevel2 = -1;
            if (b2 != ~0ull) {
                const int c2 = (int)((b2 >> 20) & 0xfffff), pos2 = (int)(b2 & 0xfffff);
                bestDist2 = (int)(b2 >> 40); bestLevel2 = oct2[gidx[goff[(cx0 + c2 / ny) * GRID_ROWS + cy0 + c2 % ny] + pos2]];
            }
            if (oct2[j] == bestLevel2 && (float)bestDist > __fmul_rn(A.nnratio, (float)bestDist2)) continue;   // :117
            if (lane == 0) { assign2[j] = i; claimed[j] = (fl >> 1) & 1; }
            nmatches++;
        }
        __syncwarp();
    }
    if (lane == 0) *nmatch = nmatches;
}

// ---------------- SURVEY.md 8(f) row 3: line projection search, Fuse search ----------------
// Frame::GetLinesInArea (Frame.cc:423-460) = KeyFrame::GetLinesInArea (KeyFrame.cc:651-684) for one frame line: the mid-point test is
// evaluated in double and narrowed (as the mixed float/double expression of the reference is), without FMA contraction.
struct LineWin { double mx, my; float r2, r, slope; double rs; int minLevel, maxLevel; bool checkLevels; };
__device__ __forceinline__ LineWin line_win(float x1, float y1, float x2, float y2, float r, int minLevel, int maxLevel) {
    LineWin w;
    w.mx = __dmul_rn(0.5, (double)__fadd_rn(x1, x2)); w.my = __dmul_rn(0.5, (double)__fadd_rn(y1, y2));
    w.r = r; w.r2 = __fmul_rn(r, r);
    w.slope = __fdiv_rn(__fsub_rn(y1, y2), __fsub_rn(x1, x2));
    w.rs = __dmul_rn((double)r, 0.01);
    w.minLevel = minLevel; w.maxLevel = maxLevel; w.checkLevels = (minLevel > 0) || (maxLevel > 0);
    return w;
}
__device__ __forceinline__ bool line_in_area(const LineWin& w, float ptx, float pty, float angle, int octave) {
    const double dx = __dsub_rn(w.mx, (double)ptx), dy = __dsub_rn(w.my, (double)pty);
    const float distance = __double2float_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)));
    if (distance > w.r2) return false;
    const float slope = __fsub_rn(w.slope, angle);
    if ((double)slope > w.rs) return false;
    if (w.checkLevels) {
        if (octave < w.minLevel) return false;
        if (w.maxLevel >= 0 && octave > w.maxLevel) return false;
    }
    return true;
}

// Search stage of both LSDmatcher::SearchByProjection overloads (LSDmatcher.cpp:98-137 = :210-251).  The MapLines are visited in
// vector order by ONE warp, because a frame line taken by a MapLine with observations is skipped by the later ones (:104-106);
// the lanes share the scan over the frame's lines.  keys: (distance << 32) | line index = the scan order of the reference.
__global__ void __launch_bounds__(32) k_line_window_search(int nml, const uint8_t* flag /* bit0 active, bit1 obs>0 */, const float4* proj, const float* radius,
                                                            const int* minLevel, const int* maxLevel, const uint8_t* dml,
                                                            int nl2, const uint8_t* ld2, const float* kl2, const int* oct2, uint8_t* claimed,
                                                            float nnratio, int32_t* assign2, int32_t* nmatch) {
    const int lane = threadIdx.x;
    for (int j = lane; j < nl2; j += 32) assign2[j] = -1;
    __syncwarp();
    int nmatches = 0;
    for (int i = 0; i < nml; i++) {
        const int fl = flag[i];
        if (!(fl & 1)) continue;
        const float4 p = proj[i];
        const LineWin w = line_win(p.x, p.y, p.z, p.w, radius[i], minLevel[i], maxLevel[i]);
        uint4 a0, a1;
        load_desc(dml + (long long)i * 32, a0, a1);
        unsigned long long b1 = ~0ull, b2 = ~0ull;
        for (int j = lane; j < nl2; j += 32) {
            if (!line_in_area(w, kl2[3 * j], kl2[3 * j + 1], kl2[3 * j + 2], oct2[j])) continue;
            if (claimed[j]) continue;
            uint4 c0, c1;
            load_desc(ld2 + (long long)j * 32, c0, c1);
            const int dist = popc256(a0, a1, c0, c1);
            if (dist >= 256) continue;                            // never below the initial bestDist = bestDist2 = 256
            top2_push(b1, b2, ((unsigned long long)dist << 32) | (unsigned)j);
        }
        top2_warp(b1, b2);
        if (b1 == ~0ull) continue;
        const int bestDist = (int)(b1 >> 32);
        if (bestDist <= TH_HIGH) {
            const int j = (int)(b1 & 0xffffffffu);
            int bestDist2 = 256, bestLevel2 = -1;
            if (b2 != ~0ull) { bestDist2 = (int)(b2 >> 32); bestLevel2 = oct2[(int)(b2 & 0xffffffffu)]; }
            if (oct2[j] == bestLevel2 && (float)bestDist > __fmul_rn(nnratio, (float)bestDist2)) continue;
            if (lane == 0) { assign2[j] = i; claimed[j] = (fl >> 1) & 1; }
            nmatches++;
        }
        __syncwarp();
    }
    if (lane == 0) *nmatch = nmatches;
}

// Search stage of LSDmatcher::Fuse (LSDmatcher.cpp:499-523): independent per MapLine, one warp each
__global__ void __launch_bounds__(128) k_line_fuse_search(int nml, const uint8_t* active, const float4* proj, const int* level, const uint8_t* dml,
                                                           int nl2, const uint8_t* ld2, const float* kl2, const int* oct2, const float* scale, float th,
                                                           int32_t* best_idx, int32_t* best_dist) {
    const int i = blockIdx.x * 4 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (i >= nml) return;
    unsigned long long b = ~0ull;
    if (active[i]) {
        const int lvl = level[i];
        const float4 p = proj[i];
        const LineWin w = line_win(p.x, p.y, p.z, p.w, __fmul_rn(th, scale[lvl]), -1, -1);
        uint4 a0, a1;
        load_desc(dml + (long long)i * 32, a0, a1);
        for (int j = lane; j < nl2; j += 32) {
            const int o = oct2[j];
            if (!line_in_area(w, kl2[3 * j], kl2[3 * j + 1], kl2[3 * j + 2], o)) continue;
            if (o < lvl - 1 || o > lvl) continue;
            uint4 c0, c1;
            load_desc(ld2 + (long long)j * 32, c0, c1);
            const unsigned long long k = ((unsigned long long)popc256(a0, a1, c0, c1) << 32) | (unsigned)j;
            b = k < b ? k : b;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) { const unsigned long long t = __shfl_xor_sync(0xffffffffu, b, o); b = t < b ? t : b; }
    }
    if (lane == 0) { best_idx[i] = b == ~0ull ? -1 : (int)(b & 0xffffffffu); best_dist[i] = b == ~0ull ? 0x7fffffff : (int)(b >> 32); }
}

// Search stage of ORBmatcher::Fuse (ORBmatcher.cc:896-950): independent per MapPoint, one warp each over the grid cells of the window
__global__ void __launch_bounds__(128) k_point_fuse_search(const __grid_constant__ WinArgs A, int nmp, const uint8_t* active, const float* pu, const float* pv, const float* pur,
                                                            const int* level, const uint8_t* dmp, const uint8_t* d2, const float* x2, const float* y2, const int* oct2,
                                                            const float* uright2, const float* invSigma2, const int* goff, const int* gidx,
                                                            int32_t* best_idx, int32_t* best_dist) {
    const int i = blockIdx.x * 4 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (i >= nmp) return;
    unsigned long long b = ~0ull;
    int cx0 = 0, cx1 = -1, cy0 = 0, cy1 = -1;
    if (active[i]) {
        const int lvl = level[i];
        const float u = pu[i], v = pv[i], ur = pur[i];
        const float rad = __fmul_rn(A.th, A.scale[lvl]);
        if (grid_window(A, u, v, rad, cx0, cx1, cy0, cy1)) {
            const int ny = cy1 - cy0 + 1, ncell = (cx1 - cx0 + 1) * ny;
            uint4 a0, a1;
            load_desc(dmp + (long long)i * 32, a0, a1);
            for (int c = lane; c < ncell; c += 32) {
                const int ix = cx0 + c / ny, iy = cy0 + c % ny, cell = ix * GRID_ROWS + iy;
                const int qb = goff[cell], qe = goff[cell + 1];
                for (int q = qb; q < qe; q++) {
                    const int j = gidx[q];
                    const float kx = x2[j], ky = y2[j];
                    if (!(fabsf(__fsub_rn(kx, u)) < rad && fabsf(__fsub_rn(ky, v)) < rad)) continue;     // KeyFrame::GetFeaturesInArea KeyFrame.cc:642
                    const int o = oct2[j];
                    if (o < lvl - 1 || o > lvl) continue;                                                 // :905
                    const float ex = __fsub_rn(u, kx), ey = __fsub_rn(v, ky);
                    float e2 = __fadd_rn(__fmul_rn(ex, ex), __fmul_rn(ey, ey));
                    const float kr = A.use_right ? uright2[j] : -1.f;
                    if (kr >= 0) {                                                                        // stereo chi-square, 3 dof (:908-921)
                        const float er = __fsub_rn(ur, kr);
                        e2 = __fadd_rn(e2, __fmul_rn(er, er));
                        if ((double)__fmul_rn(e2, invSigma2[o]) > 7.8) continue;
                    } else if ((double)__fmul_rn(e2, invSigma2[o]) > 5.99) continue;                      // :923-932
                    uint4 c0, c1;
                    load_desc(d2 + (long long)j * 32, c0, c1);
                    const int dist = popc256(a0, a1, c0, c1);
                    if (dist >= 256) continue;                                                            // bestDist starts at 256, strict <
                    const unsigned long long k = ((unsigned long long)dist << 40) | ((unsigned long long)c << 20) | (unsigned)(q - qb);
                    b = k < b ? k : b;
                }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) { const unsigned long long t = __shfl_xor_sync(0xffffffffu, b, o); b = t < b ? t : b; }
        }
    }
    if (lane == 0) {
        int bi = -1, bd = 256;
        if (b != ~0ull) {
            const int ny = cy1 - cy0 + 1, c = (int)((b >> 20) & 0xfffff), pos = (int)(b & 0xfffff);
            bi = gidx[goff[(cx0 + c / ny) * GRID_ROWS + cy0 + c % ny] + pos]; bd = (int)(b >> 40);
        }
        best_idx[i] = bi; best_dist[i] = bd;
    }
}

__global__ void __launch_bounds__(32) k_init_match(const __grid_constant__ WinArgs A, int n1, const uint8_t* d1, const int* oct1, const float* angle1,
                                                    float* prevx, float* prevy, int n2, const uint8_t* d2, const float* x2, const float* y2, const int* oct2,
                                                    const float* angle2, const int* goff, const int* gidx, int* matchedDist, int* matches21,
                                                    int32_t* matches12, uint8_t* rbin, int32_t* nmatch) {
    __shared__ int s_hist[HISTO_LENGTH];
    __shared__ int s_keep[3];
    const int lane = threadIdx.x;
    for (int j = lane; j < n2; j += 32) { matchedDist[j] = 0x7fffffff; matches21[j] = -1; }
    for (int i = lane; i < n1; i += 32) { matches12[i] = -1; rbin[i] = 255; }
    if (lane < HISTO_LENGTH) s_hist[lane] = 0;
    __syncwarp();
    int nmatches = 0;
    const float rad = (float)A.window;
    for (int i1 = 0; i1 < n1; i1++) {
        const int level1 = oct1[i1];
        if (level1 > 0) continue;                                 // :426
        const float u = prevx[i1], v = prevy[i1];
        int cx0, cx1, cy0, cy1;
        if (!grid_window(A, u, v, rad, cx0, cx1, cy0, cy1)) continue;
        const int ny = cy1 - cy0 + 1, ncell = (cx1 - cx0 + 1) * ny;
        uint4 a0, a1;
        load_desc(d1 + (long long)i1 * 32, a0, a1);
        unsigned long long b1 = ~0ull, b2 = ~0ull;
        for (int c = lane; c < ncell; c += 32) {
            const int ix = cx0 + c / ny, iy = cy0 + c % ny, cell = ix * GRID_ROWS + iy;
            const int b = goff[cell], e = goff[cell + 1];
            for (int q = b; q < e; q++) {
                const int j = gidx[q];
                { const int o = oct2[j]; if (o < level1 || o > level1) continue; }      // GetFeaturesInArea(..., level1, level1): levels are checked (maxLevel >= 0)
                if (!(fabsf(__fsub_rn(x2[j], u)) < rad && fabsf(__fsub_rn(y2[j], v)) < rad)) continue;
                uint4 c0, c1;
                load_desc(d2 + (long long)j * 32, c0, c1);
                const int dist = popc256(a0, a1, c0, c1);
                if (matchedDist[j] <= dist) continue;             // :448
                top2_push(b1, b2, ((unsigned long long)dist << 40) | ((unsigned long long)c << 20) | (unsigned)(q - b));
            }
        }
        top2_warp(b1, b2);
        if (b1 == ~0ull) continue;
        const int bestDist = (int)(b1 >> 40);
        const float bestDist2 = b2 == ~0ull ? (float)0x7fffffff : (float)(int)(b2 >> 40);
        if (bestDist <= TH_LOW_I && (float)bestDist < __fmul_rn(bestDist2, A.nnratio)) {       // :462-464
            const int c = (int)((b1 >> 20) & 0xfffff), pos = (int)(b1 & 0xfffff);
            const int j = gidx[goff[(cx0 + c / ny) * GRID_ROWS + cy0 + c % ny] + pos];
            const int old = matches21[j];
            if (old >= 0) nmatches--;
            if (lane == 0) {
                if (old >= 0) matches12[old] = -1;
                matches12[i1] = j; matches21[j] = i1; matchedDist[j] = bestDist;
                if (A.checkOri) { const int bin = rot_bin(angle1[i1], angle2[j]); rbin[i1] = (uint8_t)bin; s_hist[bin]++; }
            }
            nmatches++;
        }
        __syncwarp();
    }
    __syncwarp();
    if (A.checkOri) {
        if (lane == 0) {                                         // ComputeThreeMaxima, ORBmatcher.cc:1604-1645
            int max1 = 0, max2 = 0, max3 = 0, ind1 = -1, ind2 = -1, ind3 = -1;
            for (int i = 0; i < HISTO_LENGTH; i++) {
                const int sv = s_hist[i];
                if (sv > max1) { max3 = max2; max2 = max1; max1 = sv; ind3 = ind2; ind2 = ind1; ind1 = i; }
                else if (sv > max2) { max3 = max2; max2 = sv; ind3 = ind2; ind2 = i; }
                else if (sv > max3) { max3 = sv; ind3 = i; }
            }
            if ((float)max2 < __fmul_rn(0.1f, (float)max1)) { ind2 = -1; ind3 = -1; }
            else if ((float)max3 < __fmul_rn(0.1f, (float)max1)) { ind3 = -1; }
            s_keep[0] = ind1; s_keep[1] = ind2; s_keep[2] = ind3;
        }
        __syncwarp();
        const int k0 = s_keep[0], k1 = s_keep[1], k2 = s_keep[2];
        for (int i0 = 0; i0 < n1; i0 += 32) {
            const int i = i0 + lane;
            bool drop = false;
            if (i < n1 && rbin[i] != 255) { const int b = rbin[i]; drop = (b != k0 && b != k1 && b != k2) && matches12[i] >= 0; }
            if (drop) matches12[i] = -1;
            nmatches -= __popc(__ballot_sync(0xffffffffu, drop));
        }
    }
    __syncwarp();
    for (int i = lane; i < n1; i += 32) { const int j = matches12[i]; if (j >= 0) { prevx[i] = x2[j]; prevy[i] = y2[j]; } }   // :517-520
    if (lane == 0) *nmatch = nmatches;
}

// -------------------------------------------------------------------------------------------------
// MapPoint / MapLine ::ComputeDistinctiveDescriptors (MapPoint.cc:247-312, MapLine.cpp:246-317), batched over groups of
// observed descriptors (CSR): the descriptor with the least median Hamming distance to the others, first minimum wins.
// One CTA per group, one thread per row; the median of a row (rank r = int(0.5 (N-1)) of N distances in 0..256) is found by
// bisection on the value with count(d <= v) (8 passes over the row, descriptors stay in L1) — no sort, no per-thread arrays.
// -------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) k_medoid(const uint8_t* desc, const int32_t* off, int32_t* best_idx, int32_t* best_median) {
    __shared__ unsigned s_best;
    const int gI = blockIdx.x, b = off[gI], N = off[gI + 1] - b;
    if (threadIdx.x == 0) s_best = 0xffffffffu;
    __syncthreads();
    if (N > 0) {
        const int r = (int)(0.5 * (double)(N - 1));
        unsigned mine = 0xffffffffu;
        for (int i = threadIdx.x; i < N; i += blockDim.x) {
            uint4 a0, a1;
            load_desc(desc + (long long)(b + i) * 32, a0, a1);
            int lo = 0, hi = 256;                                        // smallest v with count(d <= v) >= r + 1
            while (lo < hi) {
                const int mid = (lo + hi) >> 1;
                int cnt = 0;
                for (int j = 0; j < N; j++) {
                    uint4 b0, b1;
                    load_desc(desc + (long long)(b + j) * 32, b0, b1);
                    cnt += (j == i ? 0 : popc256(a0, a1, b0, b1)) <= mid;
                }
                if (cnt >= r + 1) hi = mid; else lo = mid + 1;
            }
            const unsigned key = ((unsigned)lo << 20) | (unsigned)i;     // (median, row): the minimum is the first least median
            mine = min(mine, key);
        }
        atomicMin(&s_best, mine);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        best_idx[gI] = N > 0 ? (int)(s_best & 0xfffffu) : -1;
        best_median[gI] = N > 0 ? (int)(s_best >> 20) : -1;
    }
}

// Rotation-histogram filter (ComputeThreeMaxima, ORBmatcher.cc:1604-1645; application :270-288) and match
// count, one CTA per pair.  compact != 0 additionally writes the (i, out[i]) pairs in ascending i (:818-823).
__global__ void __launch_bounds__(256) k_rot_filter(int32_t* out, long long out_fs, const uint8_t* rot, long long rot_fs,
                                                     const int* n_arr, int n_frame_off, int n_const, int cap, int checkOri,
                                                     int32_t* nmatch, int32_t* pairs, long long pairs_fs) {
    __shared__ int s_hist[HISTO_LENGTH];
    __shared__ int s_keep[3];
    __shared__ int s_warp[33];
    const int pair = blockIdx.x, tid = threadIdx.x;
    const int n = n_arr ? min(n_arr[pair + n_frame_off], cap) : n_const;
    int32_t* O = out + pair * out_fs; const uint8_t* R = rot + pair * rot_fs;
    if (tid < HISTO_LENGTH) s_hist[tid] = 0;
    __syncthreads();
    if (checkOri) {
        for (int i = tid; i < n; i += 256) if (O[i] >= 0) atomicAdd(&s_hist[R[i]], 1);
        __syncthreads();
        if (tid == 0) {
            int max1 = 0, max2 = 0, max3 = 0, ind1 = -1, ind2 = -1, ind3 = -1;
            for (int i = 0; i < HISTO_LENGTH; i++) {
                const int s = s_hist[i];
                if (s > max1) { max3 = max2; max2 = max1; max1 = s; ind3 = ind2; ind2 = ind1; ind1 = i; }
                else if (s > max2) { max3 = max2; max2 = s; ind3 = ind2; ind2 = i; }
                else if (s > max3) { max3 = s; ind3 = i; }
            }
            if ((float)max2 < __fmul_rn(0.1f, (float)max1)) { ind2 = -1; ind3 = -1; }
            else if ((float)max3 < __fmul_rn(0.1f, (float)max1)) { ind3 = -1; }
            s_keep[0] = ind1; s_keep[1] = ind2; s_keep[2] = ind3;
        }
        __syncthreads();
        const int k0 = s_keep[0], k1 = s_keep[1], k2 = s_keep[2];
        for (int i = tid; i < n; i += 256)
            if (O[i] >= 0) { const int b = R[i]; if (b != k0 && b != k1 && b != k2) O[i] = -1; }
        __syncthreads();
    }
    // count (and optionally compact in ascending index order)
    const int chunk = (n + 255) / 256, pb = min(n, tid * chunk), pe = min(n, pb + chunk);
    int c = 0;
    for (int i = pb; i < pe; i++) c += O[i] >= 0;
    int total;
    int o = block_exclusive_scan(c, s_warp, &total);
    if (pairs) for (int i = pb; i < pe; i++) if (O[i] >= 0) { pairs[pair * pairs_fs + 2 * o] = i; pairs[pair * pairs_fs + 2 * o + 1] = O[i]; o++; }
    if (tid == 0) nmatch[pair] = total;
}

__global__ void k_fill_i32(int32_t* p, long long n, int v) {
    const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i < n) p[i] = v;
}

// LSDmatcher::SearchByProjection(KF,F) ratio rule on a knn2 table (LSDmatcher.cpp:161-180): out[tdx] = qdx, the
// LAST accepted query wins (atomicMax over ascending qdx), nmatch counts every acceptance like the reference.
__global__ void __launch_bounds__(128) k_line_ratio(const int32_t* knn, long long knn_fs, const int* n_arr, int n_const, int cap,
                                                     const uint8_t* has_ml1, long long ml_fs,
                                                     int32_t* out, long long out_fs, int32_t* nmatch) {
    const int pair = blockIdx.y, q = blockIdx.x * blockDim.x + threadIdx.x;
    const int nq = n_arr ? min(n_arr[pair], cap) : n_const;
    if (q >= nq) return;
    const int4 r = reinterpret_cast<const int4*>(knn + pair * knn_fs)[q];
    if (r.x < 0 || r.z < 0) return;
    const float ratio = __fdiv_rn((float)r.y, (float)r.w);                         // :167
    if ((double)ratio < (double)(1.0f / 1.5f)) {                                    // :169
        if (has_ml1 && !has_ml1[pair * ml_fs + q]) return;
        atomicMax(&out[pair * out_fs + r.x], q);
        atomicAdd(&nmatch[pair], 1);
    }
}

}  // namespace sslpl

// =================================================================================================
using namespace sslpl;

struct sslpl_vocab {
    int device = 0, k = 0, L = 0, nnodes = 0, nwords = 0;
    uint8_t* arena = nullptr;
    sslpl::VocabView view{};
    std::vector<int> depth;              // per node
    std::vector<int> level_count;        // nodes per depth
};

struct sslpl_matcher {
    sslpl_matcher_params p;
    cudaStream_t stream = nullptr, own_stream = nullptr;
    uint8_t* arena = nullptr; size_t arena_size = 0;
    int cap = 0;                     // rows per frame slot of the single-call staging (max(features, lines))
    // single-call staging: 2 frame slots
    uint8_t* desc; int* nodes; int* off; int* idx; uint8_t* flag; float* kpf; int* nn2; int* ncnt;
    int32_t* out; uint8_t* rot; uint8_t* taken; int32_t* pairs; int32_t* nmatch; int32_t* knn; uint8_t* cent; int32_t* node;
    int32_t* word; double* wgt;      // per-feature outputs of the vocabulary transform (single-call staging)
    uint8_t* scratch = nullptr; size_t scratch_size = 0;   // grow-only scratch of sslpl_descriptor_medoid_batch
    // batch workspace
    int32_t* b_node; int* b_off; int* b_idx; uint8_t* b_rot; uint8_t* b_taken; int32_t* b_knn; int* iota;
    int32_t* h_small = nullptr;      // pinned scratch
    long long launches = 0;
};

struct sslpl_kfset {
    int device = 0;
    sslpl::KfView view{};            // device arrays of every slot (layout above k_kf_compact)
    uint8_t* arena = nullptr;
    cudaStream_t stream = nullptr;   // host-buffer mask uploads and clears
    cudaEvent_t last_use = nullptr;  // recorded after every store / match enqueued on a matcher's stream
    struct Built { const sslpl_vocab* v; int levelsup; };
    std::vector<Built> built;        // tree and levelsup of each slot's FeatureVector; v == nullptr: empty slot
};

namespace {

int carve(sslpl_matcher* m, Arena& A) {
    const int cap = m->cap, NN = m->p.max_nodes + 1, B = m->p.max_batch + 1;
    m->desc = A.take<uint8_t>((size_t)2 * cap * 32);
    m->nodes = A.take<int>((size_t)2 * NN); m->off = A.take<int>((size_t)2 * (NN + 1)); m->idx = A.take<int>((size_t)2 * cap);
    m->flag = A.take<uint8_t>((size_t)2 * cap);
    m->kpf = A.take<float>((size_t)2 * cap * 7);
    m->nn2 = A.take<int>(2); m->ncnt = A.take<int>(2);
    m->out = A.take<int32_t>(cap); m->rot = A.take<uint8_t>(cap); m->taken = A.take<uint8_t>(cap);
    m->pairs = A.take<int32_t>((size_t)2 * cap); m->nmatch = A.take<int32_t>(B);
    m->knn = A.take<int32_t>((size_t)4 * cap);
    m->cent = A.take<uint8_t>((size_t)NN * 32); m->node = A.take<int32_t>(cap);
    m->word = A.take<int32_t>(cap); m->wgt = A.take<double>(cap);
    const int fc = m->p.max_features + 64, lc = m->p.max_lines + 64;
    m->b_node = A.take<int32_t>((size_t)B * fc); m->b_off = A.take<int>((size_t)B * (NN + 1)); m->b_idx = A.take<int>((size_t)B * fc);
    m->b_rot = A.take<uint8_t>((size_t)B * fc); m->b_taken = A.take<uint8_t>((size_t)B * fc);
    m->b_knn = A.take<int32_t>((size_t)B * lc * 4);
    m->iota = A.take<int>(NN);
    return 0;
}

// carve `count` elements out of a scratch arena and start their upload
template <class T> T* stage(Arena& A, const T* host, size_t count, cudaStream_t st, cudaError_t& err) {
    T* d = A.take<T>(count + 8);
    if (host && count && err == cudaSuccess) err = cudaMemcpyAsync(d, host, sizeof(T) * count, cudaMemcpyHostToDevice, st);
    return d;
}

int upload_featvec(sslpl_matcher* m, int slot, const sslpl_featvec* fv, int n) {
    const int NN = m->p.max_nodes + 1;
    SSLPL_REQUIRE(fv && fv->nn >= 0 && fv->nn <= m->p.max_nodes, SSLPL_ERR_ARG, "feature vector has more nodes than max_nodes");
    if (fv->nn == 0) return SSLPL_OK;
    SSLPL_REQUIRE(fv->nodes && fv->off && fv->idx, SSLPL_ERR_ARG, "null feature vector arrays");
    SSLPL_REQUIRE(fv->off[fv->nn] <= n, SSLPL_ERR_ARG, "feature vector indexes more features than given");
    SSLPL_CUDA(cudaMemcpyAsync(m->nodes + slot * NN, fv->nodes, sizeof(int) * fv->nn, cudaMemcpyHostToDevice, m->stream));
    SSLPL_CUDA(cudaMemcpyAsync(m->off + slot * (NN + 1), fv->off, sizeof(int) * (fv->nn + 1), cudaMemcpyHostToDevice, m->stream));
    SSLPL_CUDA(cudaMemcpyAsync(m->idx + slot * m->cap, fv->idx, sizeof(int) * fv->off[fv->nn], cudaMemcpyHostToDevice, m->stream));
    return SSLPL_OK;
}

FrameSet staging_set(sslpl_matcher* m, int nn1, int nn2, bool with_flags) {
    const int NN = m->p.max_nodes + 1;
    FrameSet S; memset(&S, 0, sizeof(S));
    S.desc = m->desc; S.desc_fs = (long long)m->cap * 32;
    S.nodes = m->nodes; S.off = m->off; S.idx = m->idx; S.nodes_fs = NN; S.off_fs = NN + 1; S.idx_fs = m->cap;
    S.nn = m->nn2; (void)nn1; (void)nn2;
    S.flag = with_flags ? m->flag : nullptr; S.flag_fs = m->cap;
    S.angle = m->kpf + 3; S.x = m->kpf; S.y = m->kpf + 1; S.oct = reinterpret_cast<const int*>(m->kpf + 5);
    S.angle_es = 7; S.angle_fs = (long long)m->cap * 7;
    return S;
}

int fill(sslpl_matcher* m, int32_t* p, long long n, int v) {
    if (n <= 0) return SSLPL_OK;
    k_fill_i32<<<(unsigned)((n + 255) / 256), 256, 0, m->stream>>>(p, n, v); m->launches++;
    return SSLPL_OK;
}

// upload angles (or full keypoints) into the 7-float-per-row staging of a slot
int upload_angles(sslpl_matcher* m, int slot, const float* angle, int n) {
    if (n == 0) return SSLPL_OK;
    SSLPL_CUDA(cudaMemcpy2DAsync(m->kpf + (size_t)slot * m->cap * 7 + 3, 7 * sizeof(float), angle, sizeof(float), sizeof(float), n,
                                 cudaMemcpyHostToDevice, m->stream));
    return SSLPL_OK;
}

int common_bow(sslpl_matcher* m, int mode, const uint8_t* d1, int n1, const uint8_t* d2, int n2,
               const sslpl_featvec* fv1, const sslpl_featvec* fv2, const uint8_t* valid1, const uint8_t* valid2,
               const float* angle1, const float* angle2, float nnratio, int checkOri, int32_t* match, int* nmatches) {
    SSLPL_REQUIRE(m && match && nmatches && fv1 && fv2, SSLPL_ERR_ARG, "null argument");
    SSLPL_REQUIRE(n1 >= 0 && n2 >= 0 && n1 <= m->p.max_features && n2 <= m->p.max_features, SSLPL_ERR_ARG, "feature count exceeds max_features");
    SSLPL_REQUIRE((n1 == 0 || (d1 && angle1 && valid1)) && (n2 == 0 || (d2 && angle2)), SSLPL_ERR_ARG, "null descriptor/angle/valid array");
    SSLPL_REQUIRE(mode == 0 || n2 == 0 || valid2, SSLPL_ERR_ARG, "valid2 required for the KF-KF variant");
    SSLPL_CUDA(cudaSetDevice(m->p.device));
    const int nout = mode == 0 ? n2 : n1;
    if (nout == 0) { *nmatches = 0; return SSLPL_OK; }
    cudaStream_t st = m->stream;
    const int cap = m->cap;
    if (n1) SSLPL_CUDA(cudaMemcpyAsync(m->desc, d1, (size_t)n1 * 32, cudaMemcpyHostToDevice, st));
    if (n2) SSLPL_CUDA(cudaMemcpyAsync(m->desc + (size_t)cap * 32, d2, (size_t)n2 * 32, cudaMemcpyHostToDevice, st));
    int rc;
    if ((rc = upload_featvec(m, 0, fv1, n1)) || (rc = upload_featvec(m, 1, fv2, n2))) return rc;
    if ((rc = upload_angles(m, 0, angle1, n1)) || (rc = upload_angles(m, 1, angle2, n2))) return rc;
    if (n1) SSLPL_CUDA(cudaMemcpyAsync(m->flag, valid1, n1, cudaMemcpyHostToDevice, st));
    if (n2 && valid2) SSLPL_CUDA(cudaMemcpyAsync(m->flag + cap, valid2, n2, cudaMemcpyHostToDevice, st));
    else if (n2) SSLPL_CUDA(cudaMemsetAsync(m->flag + cap, 1, n2, st));
    m->h_small[0] = fv1->nn; m->h_small[1] = fv2->nn;
    SSLPL_CUDA(cudaMemcpyAsync(m->nn2, m->h_small, 2 * sizeof(int), cudaMemcpyHostToDevice, st));
    fill(m, m->out, nout, -1);
    SSLPL_CUDA(cudaMemsetAsync(m->rot, 255, nout, st));
    SSLPL_CUDA(cudaMemsetAsync(m->taken, 0, std::max(n2, 1), st));
    FrameSet S = staging_set(m, fv1->nn, fv2->nn, true);
    if (fv1->nn > 0 && fv2->nn > 0) {
        k_bow_match<<<dim3((fv1->nn + 3) / 4, 1), 128, 0, st>>>(S, mode, nnratio, cap, m->out, 0, m->rot, 0, m->taken, 0);
        m->launches++;
    }
    k_rot_filter<<<1, 256, 0, st>>>(m->out, 0, m->rot, 0, nullptr, 0, nout, cap, checkOri, m->nmatch, nullptr, 0); m->launches++;
    SSLPL_CUDA(cudaGetLastError());
    SSLPL_CUDA(cudaMemcpyAsync(match, m->out, sizeof(int32_t) * nout, cudaMemcpyDeviceToHost, st));
    SSLPL_CUDA(cudaMemcpyAsync(m->h_small + 8, m->nmatch, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    SSLPL_CUDA(cudaStreamSynchronize(st));
    *nmatches = m->h_small[8];
    return SSLPL_OK;
}

int run_knn2(sslpl_matcher* m, const uint8_t* q, int nq, const uint8_t* t, int nt, int32_t* out_host) {
    SSLPL_REQUIRE(nq >= 0 && nt >= 0 && nq <= m->cap && nt <= m->cap, SSLPL_ERR_ARG, "row count exceeds the matcher capacity");
    SSLPL_REQUIRE(nt < (1 << 20), SSLPL_ERR_ARG, "too many train rows");
    if (nq == 0) return SSLPL_OK;
    cudaStream_t st = m->stream;
    SSLPL_CUDA(cudaMemcpyAsync(m->desc, q, (size_t)nq * 32, cudaMemcpyHostToDevice, st));
    if (nt) SSLPL_CUDA(cudaMemcpyAsync(m->desc + (size_t)m->cap * 32, t, (size_t)nt * 32, cudaMemcpyHostToDevice, st));
    k_knn2<<<dim3((nq + 7) / 8, 1), 256, 0, st>>>(m->desc, 0, nullptr, nq, m->desc + (size_t)m->cap * 32, 0, nullptr, nt, m->knn, 0, nq);
    m->launches++;
    SSLPL_CUDA(cudaGetLastError());
    if (out_host) {
        SSLPL_CUDA(cudaMemcpyAsync(out_host, m->knn, sizeof(int32_t) * 4 * nq, cudaMemcpyDeviceToHost, st));
        SSLPL_CUDA(cudaStreamSynchronize(st));
    }
    return SSLPL_OK;
}

// Frame::lineDescriptorMAD, Frame.cc:190-215 (host: two medians over <= NL values)
void line_mad(const int32_t* knn, int nq, double* nn_mad, double* nn12_mad) {
    if (nq <= 0) { *nn_mad = 0; *nn12_mad = 0; return; }
    std::vector<float> a(nq), g(nq);
    for (int i = 0; i < nq; i++) a[i] = (float)knn[4 * i + 1];
    std::sort(a.begin(), a.end());
    const double med = a[nq / 2];
    for (int i = 0; i < nq; i++) a[i] = fabsf((float)((float)knn[4 * i + 1] - med));
    std::sort(a.begin(), a.end());
    *nn_mad = 1.4826 * a[nq / 2];
    for (int i = 0; i < nq; i++) g[i] = (float)knn[4 * i + 3] - (float)knn[4 * i + 1];
    std::sort(g.begin(), g.end(), [](float x, float y) { return x > y; });
    const double med12 = g[nq / 2];
    for (int i = 0; i < nq; i++) a[i] = fabsf((float)((float)knn[4 * i + 3] - (float)knn[4 * i + 1] - med12));
    std::sort(a.begin(), a.end());
    *nn12_mad = 1.4826 * a[nq / 2];
}

}  // namespace

extern "C" {

void sslpl_matcher_destroy(sslpl_matcher* m);

int sslpl_matcher_create(const sslpl_matcher_params* p, sslpl_matcher** out) {
    SSLPL_REQUIRE(p && out, SSLPL_ERR_ARG, "null argument");
    SSLPL_REQUIRE(p->max_features >= 1 && p->max_lines >= 0 && p->max_nodes >= 1 && p->max_batch >= 1, SSLPL_ERR_ARG, "bad matcher capacity");
    SSLPL_REQUIRE(p->max_features < (1 << 20) && p->max_lines < (1 << 20), SSLPL_ERR_ARG, "capacity too large");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) { set_error("no CUDA device available: libsslpl_b200 has no CPU fallback"); return SSLPL_ERR_CUDA; }
    SSLPL_CUDA(cudaSetDevice(p->device));
    sslpl_matcher* m = new sslpl_matcher();
    m->p = *p;
    m->cap = std::max(p->max_features, p->max_lines) + 64;
    Arena A; carve(m, A);
    m->arena_size = A.used + (1 << 16);
    cudaError_t e = cudaMalloc(&m->arena, m->arena_size);
    if (e != cudaSuccess) { set_error("cudaMalloc(%zu) failed: %s", m->arena_size, cudaGetErrorString(e)); delete m; return SSLPL_ERR_CUDA; }
    cudaError_t e2 = cudaMemset(m->arena, 0, m->arena_size);
    Arena B; B.base = m->arena; B.size = m->arena_size; carve(m, B);
    if (e2 == cudaSuccess) e2 = cudaStreamCreateWithFlags(&m->own_stream, cudaStreamNonBlocking);
    m->stream = m->own_stream;
    if (e2 == cudaSuccess) e2 = cudaHostAlloc((void**)&m->h_small, 64 * sizeof(int32_t), cudaHostAllocDefault);
    if (e2 == cudaSuccess) {
        std::vector<int> iota(p->max_nodes + 1);
        for (int i = 0; i <= p->max_nodes; i++) iota[i] = i;
        e2 = cudaMemcpy(m->iota, iota.data(), sizeof(int) * iota.size(), cudaMemcpyHostToDevice);
    }
    // the two kernels with data-dependent dynamic shared memory may use the whole 227 KB of an sm_100 CTA
    if (e2 == cudaSuccess) e2 = cudaFuncSetAttribute(k_bow_assign, cudaFuncAttributeMaxDynamicSharedMemorySize, MAX_DYN_SMEM);
    if (e2 == cudaSuccess) e2 = cudaFuncSetAttribute(k_build_csr, cudaFuncAttributeMaxDynamicSharedMemorySize, MAX_DYN_SMEM);
    if (e2 != cudaSuccess) { set_error("sslpl_matcher_create: %s", cudaGetErrorString(e2)); sslpl_matcher_destroy(m); return SSLPL_ERR_CUDA; }
    *out = m;
    return SSLPL_OK;
}

void sslpl_matcher_destroy(sslpl_matcher* m) {
    if (!m) return;
    cudaSetDevice(m->p.device);
    // an external stream may already be gone (its owner was destroyed first): never touch it here
    if (m->stream && m->stream == m->own_stream) cudaStreamSynchronize(m->own_stream); else cudaDeviceSynchronize();
    if (m->own_stream) cudaStreamDestroy(m->own_stream);
    if (m->arena) cudaFree(m->arena);
    if (m->scratch) cudaFree(m->scratch);
    if (m->h_small) cudaFreeHost(m->h_small);
    delete m;
}

int sslpl_matcher_sync(sslpl_matcher* m) {
    SSLPL_REQUIRE(m, SSLPL_ERR_ARG, "null handle");
    SSLPL_CUDA(cudaSetDevice(m->p.device));
    SSLPL_CUDA(cudaStreamSynchronize(m->stream));
    return SSLPL_OK;
}
void* sslpl_matcher_stream(sslpl_matcher* m) { return m ? (void*)m->stream : nullptr; }
int sslpl_matcher_set_stream(sslpl_matcher* m, void* cuda_stream) {
    SSLPL_REQUIRE(m, SSLPL_ERR_ARG, "null handle");
    SSLPL_CUDA(cudaSetDevice(m->p.device));
    SSLPL_CUDA(cudaStreamSynchronize(m->stream));
    m->stream = cuda_stream ? (cudaStream_t)cuda_stream : m->own_stream;
    return SSLPL_OK;
}
long long sslpl_matcher_launch_count(const sslpl_matcher* m) { return m ? m->launches : 0; }

int sslpl_descriptor_distance(sslpl_matcher* m, const uint8_t* a, const uint8_t* b, int n, int32_t* dist) {
    SSLPL_REQUIRE(m && (n == 0 || (a && b && dist)), SSLPL_ERR_ARG, "null argument");
    SSLPL_REQUIRE(n >= 0 && n <= m->cap, SSLPL_ERR_ARG, "n exceeds the matcher capacity");
    if (n == 0) return SSLPL_OK;
    SSLPL_CUDA(cudaSetDevice(m->p.device));
    cudaStream_t st = m->stream;
    SSLPL_CUDA(cudaMemcpyAsync(m->desc, a, (size_t)n * 32, cudaMemcpyHostToDevice, st));
    SSLPL_CUDA(cudaMemcpyAsync(m->desc + (size_t)m->cap * 32, b, (size_t)n * 32, cudaMemcpyHostToDevice, st));
    k_pair_distance<<<(n + 127) / 128, 128, 0, st>>>(m->desc, m->desc + (size_t)m->cap * 32, n, m->out); m->launches++;
    SSLPL_CUDA(cudaGetLastError());
    SSLPL_CUDA(cudaMemcpyAsync(dist, m->out, sizeof(int32_t) * n, cudaMemcpyDeviceToHost, st));
    SSLPL_CUDA(cudaStreamSynchronize(st));
    return SSLPL_OK;
}

int sslpl_hamming_knn2(sslpl_matcher* m, const uint8_t* q, int nq, const uint8_t* t, int nt, int32_t* out) {
    SSLPL_REQUIRE(m && (nq == 0 || (q && out)) && (nt == 0 || t), SSLPL_ERR_ARG, "null argument");
    SSLPL_CUDA(cudaSetDevice(m->p.device));
    return run_knn2(m, q, nq, t, nt, out);
}

int sslpl_bow_assign(sslpl_matcher* m, const uint8_t* desc, int n, const uint8_t* centroids, int nc, int32_t* node) {
    SSLPL_REQUIRE(m && (n == 0 || (desc && node)) && centroids, SSLPL_ERR_ARG, "null argument");
    SSLPL_REQUIRE(n >= 0 && n <= m->cap && nc >= 1 && nc <= m->p.max_nodes, SSLPL_ERR_ARG, "n or nc exceeds the matcher capacity");
    if (n == 0) return SSLPL_OK;
    SSLPL_CUDA(cudaSetDevice(m->p.device));
    cudaStream_t st = m->stream;
    SSLPL_CUDA(cudaMemcpyAsync(m->desc, desc, (size_t)n * 32, cudaMemcpyHostToDevice, st));
    SSLPL_CUDA(cudaMemcpyAsync(m->cent, centroids, (size_t)nc * 32, cudaMemcpyHostToDevice, st));
    SSLPL_REQUIRE((size_t)(nc * 32) <= (size_t)MAX_DYN_SMEM, SSLPL_ERR_CAPACITY, "too many centroids for one shared-memory tile (nc <= 6400)");
    k_bow_assign<<<dim3((n + 127) / 128, 1), 128, nc * 32, st>>>(m->desc, 0, nullptr, n, n, m->cent, nc, m->node, 0); m->launches++;
    SSLPL_CUDA(cudaGetLastError());
    SSLPL_CUDA(cudaMemcpyAsync(node, m->node, sizeof(int32_t) * n, cudaMemcpyDeviceToHost, st));
    SSLPL_CUDA(cudaStreamSynchronize(st));
    return SSLPL_OK;
}

int sslpl_search_by_bow(sslpl_matcher* m, const uint8_t* d1, int n1, const uint8_t* d2, int n2,
                        const sslpl_featvec* fv1, const sslpl_featvec* fv2, const uint8_t* valid1, const float* angle1, const float* angle2,
                        float nnratio, int checkOri, int32_t* match2, int* nmatches) {
    return common_bow(m, 0, d1, n1, d2, n2, fv1, fv2, valid1, nullptr, angle1, angle2, nnratio, checkOri, match2, nmatches);
}

int sslpl_search_by_bow_kf(sslpl_matcher* m, const uint8_t* d1, int n1, const uint8_t* d2, int n2,
                           const sslpl_featvec* fv1, const sslpl_featvec* fv2, const uint8_t* valid1, const uint8_t* valid2,
                           const float* angle1, const float* angle2, float nnratio, int checkOri, int32_t* match12, int* nmatches) {
    return common_bow(m, 1, d1, n1, d2, n2, fv1, fv2, valid1, valid2, angle1, angle2, nnratio, checkOri, match12, nmatches);
}

int sslpl_search_for_triangulation(sslpl_matcher* m, const uint8_t* d1, int n1, const uint8_t* d2, int n2,
                                   const sslpl_featvec* fv1, const sslpl_featvec* fv2, const uint8_t* has_mp1, const uint8_t* has_mp2,
                                   const sslpl_keypoint* kp1, const sslpl_keypoint* kp2, const float* F12, float ex, float ey,
                                   const float* scale, const float* sigma2, int nlevels, int checkOri, int32_t* pairs, int* nmatches) {
    SSLPL_REQUIRE(m && pairs && nmatches && fv1 && fv2 && F12 && scale && sigma2, SSLPL_ERR_ARG, "null argument");
    SSLPL_REQUIRE(n1 >= 0 && n2 >= 0 && n1 <= m->p.max_features && n2 <= m->p.max_features, SSLPL_ERR_ARG, "feature count exceeds max_features");
    SSLPL_REQUIRE(nlevels >= 1 && nlevels <= SSLPL_MAX_LEVELS, SSLPL_ERR_ARG, "nlevels out of range");
    SSLPL_REQUIRE((n1 == 0 || (d1 && kp1 && has_mp1)) && (n2 == 0 || (d2 && kp2 && has_mp2)), SSLPL_ERR_ARG, "null array");
    *nmatches = 0;
    if (n1 == 0 || n2 == 0) return SSLPL_OK;
    for (int i = 0; i < n2; i++) SSLPL_REQUIRE(kp2[i].octave >= 0 && kp2[i].octave < nlevels, SSLPL_ERR_ARG, "keypoint octave out of range");
    SSLPL_CUDA(cudaSetDevice(m->p.device));
    cudaStream_t st = m->stream;
    const int cap = m->cap;
    SSLPL_CUDA(cudaMemcpyAsync(m->desc, d1, (size_t)n1 * 32, cudaMemcpyHostToDevice, st));
    SSLPL_CUDA(cudaMemcpyAsync(m->desc + (size_t)cap * 32, d2, (size_t)n2 * 32, cudaMemcpyHostToDevice, st));
    int rc;
    if ((rc = upload_featvec(m, 0, fv1, n1)) || (rc = upload_featvec(m, 1, fv2, n2))) return rc;
    SSLPL_CUDA(cudaMemcpyAsync(m->kpf, kp1, (size_t)n1 * 28, cudaMemcpyHostToDevice, st));
    SSLPL_CUDA(cudaMemcpyAsync(m->kpf + (size_t)cap * 7, kp2, (size_t)n2 * 28, cudaMemcpyHostToDevice, st));
    SSLPL_CUDA(cudaMemcpyAsync(m->flag, has_mp1, n1, cudaMemcpyHostToDevice, st));
    SSLPL_CUDA(cudaMemcpyAsync(m->flag + cap, has_mp2, n2, cudaMemcpyHostToDevice, st));
    m->h_small[0] = fv1->nn; m->h_small[1] = fv2->nn;
    SSLPL_CUDA(cudaMemcpyAsync(m->nn2, m->h_small, 2 * sizeof(int), cudaMemcpyHostToDevice, st));
    fill(m, m->out, n1, -1);
    SSLPL_CUDA(cudaMemsetAsync(m->rot, 255, n1, st));
    FrameSet S = staging_set(m, fv1->nn, fv2->nn, true);
    TriArgs T;
    for (int i = 0; i < 9; i++) T.F[i] = F12[i];
    T.ex = ex; T.ey = ey;
    for (int i = 0; i < SSLPL_MAX_LEVELS; i++) { T.scale[i] = i < nlevels ? scale[i] : 0.f; T.sigma2[i] = i < nlevels ? sigma2[i] : 0.f; }
    if (fv1->nn > 0 && fv2->nn > 0) { k_tri_match<<<dim3((fv1->nn + 3) / 4, 1), 128, 0, st>>>(S, T, m->out, 0, m->rot, 0); m->launches++; }
    k_rot_filter<<<1, 256, 0, st>>>(m->out, 0, m->rot, 0, nullptr, 0, n1, cap, checkOri, m->nmatch, m->pairs, 0); m->launches++;
    SSLPL_CUDA(cudaGetLastError());
    SSLPL_CUDA(cudaMemcpyAsync(m->h_small + 8, m->nmatch, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    SSLPL_CUDA(cudaStreamSynchronize(st));
    *nmatches = m->h_small[8];
    if (*nmatches > 0) {
        SSLPL_CUDA(cudaMemcpyAsync(pairs, m->pairs, sizeof(int32_t) * 2 * (*nmatches), cudaMemcpyDeviceToHost, st));
        SSLPL_CUDA(cudaStreamSynchronize(st));
    }
    return SSLPL_OK;
}

int sslpl_line_match(sslpl_matcher* m, int mode, const uint8_t* d1, int n1, const uint8_t* d2, int n2,
                     const uint8_t* has_ml1, const uint8_t* has_ml2, int32_t* out, int* nout, int* nmatches, double* mad) {
    SSLPL_REQUIRE(m && out && nmatches && mode >= 0 && mode <= 3, SSLPL_ERR_ARG, "bad argument");
    SSLPL_REQUIRE(n1 >= 0 && n2 >= 0 && n1 <= m->p.max_lines && n2 <= m->p.max_lines, SSLPL_ERR_ARG, "line count exceeds max_lines");
    // the reference indexes lmatches[i][1] unconditionally (LSDmatcher.cpp:167): it requires >= 2 train rows
    SSLPL_REQUIRE(n1 == 0 || n2 >= 2, SSLPL_ERR_ARG, "knnMatch(k=2) needs at least 2 train descriptors (reference reads out of bounds otherwise)");
    SSLPL_REQUIRE((mode != 0 && mode != 3) || n1 == 0 || has_ml1, SSLPL_ERR_ARG, "has_ml1 required");
    SSLPL_REQUIRE((mode != 2 && mode != 3) || n2 == 0 || has_ml2, SSLPL_ERR_ARG, "has_ml2 required");
    SSLPL_CUDA(cudaSetDevice(m->p.device));
    std::vector<int32_t> knn(4 * (size_t)std::max(n1, 1));
    int rc = run_knn2(m, d1, n1, d2, n2, knn.data());
    if (rc) return rc;
    double nn_mad = 0, nn12_mad = 0;
    line_mad(knn.data(), n1, &nn_mad, &nn12_mad);
    if (mad) { mad[0] = nn_mad; mad[1] = nn12_mad; }
    int nm = 0, k = 0;
    if (mode == 0) for (int j = 0; j < n2; j++) out[j] = -1;
    if (mode == 2) for (int i = 0; i < n1; i++) out[i] = -1;
    const float minRatio = 1.0f / 1.5f;
    for (int i = 0; i < n1; i++) {                      // knn rows are already in queryIdx order (:161)
        const int tdx = knn[4 * i];
        const float dist0 = (float)knn[4 * i + 1], dist1 = (float)knn[4 * i + 3];
        if (mode == 0) {
            const double dist_12 = dist0 / dist1;
            if (dist_12 < minRatio && has_ml1[i]) { out[tdx] = i; nm++; }
        } else if (mode == 1) {
            if ((double)(dist1 - dist0) > nn12_mad * 0.5) { out[2 * k] = i; out[2 * k + 1] = tdx; k++; nm++; }
        } else if (mode == 2) {
            if ((double)(dist1 - dist0) > nn12_mad * 0.5 && has_ml2[tdx]) { out[i] = tdx; nm++; }
        } else {
            if (has_ml1[i] || has_ml2[tdx]) continue;
            if ((double)(dist1 - dist0) > nn12_mad * 0.1) { out[2 * k] = i; out[2 * k + 1] = tdx; k++; nm++; }
        }
    }
    if (nout) *nout = k;
    *nmatches = nm;
    return SSLPL_OK;
}

// common tail of the batched consecutive-frame SearchByBoW: b_node holds the dense node index (or -1) of every feature
static int bow_batch_tail(sslpl_matcher* m, const uint8_t* d_desc, const sslpl_keypoint* d_kps, const int* d_n, int nframes, int cap, int nc,
                          float nnratio, int checkOri, int32_t* d_match, int32_t* d_nmatch) {
    cudaStream_t st = m->stream;
    const int npairs = nframes - 1, fc = m->p.max_features + 64, NN = m->p.max_nodes + 1;
    SSLPL_REQUIRE((size_t)((nc + 1 + cap) * sizeof(int)) <= (size_t)MAX_DYN_SMEM, SSLPL_ERR_CAPACITY, "nodes + features exceed the shared memory of one CTA ((nc + 1 + cap) * 4 <= 200 KB)");
    k_build_csr<<<nframes, 128, (nc + 1 + cap) * sizeof(int), st>>>(m->b_node, fc, d_n, cap, nc, m->b_off, NN + 1, m->b_idx, fc);
    m->launches += 1;
    fill(m, d_match, (long long)npairs * cap, -1);
    SSLPL_CUDA(cudaMemsetAsync(m->b_rot, 255, (size_t)npairs * fc, st));
    SSLPL_CUDA(cudaMemsetAsync(m->b_taken, 0, (size_t)npairs * fc, st));
    FrameSet S; memset(&S, 0, sizeof(S));
    S.desc = d_desc; S.desc_fs = (long long)cap * 32;
    S.n = d_n;
    S.nodes = nullptr; S.off = m->b_off; S.idx = m->b_idx; S.off_fs = NN + 1; S.idx_fs = fc;
    // dense vocabulary: node list is 0..nc-1 for every frame -> reuse one iota array
    S.nodes = m->iota; S.nodes_fs = 0; S.nn = nullptr; S.nn_const = nc;
    S.flag = nullptr;
    const float* kf = reinterpret_cast<const float*>(d_kps);
    S.angle = kf + 3; S.x = kf; S.y = kf + 1; S.oct = reinterpret_cast<const int*>(kf + 5); S.angle_es = 7; S.angle_fs = (long long)cap * 7;
    k_bow_match<<<dim3((nc + 3) / 4, npairs), 128, 0, st>>>(S, 0, nnratio, cap, d_match, cap, m->b_rot, fc, m->b_taken, fc);
    k_rot_filter<<<npairs, 256, 0, st>>>(d_match, cap, m->b_rot, fc, d_n, 1, 0, cap, checkOri, d_nmatch, nullptr, 0);
    m->launches += 2;
    SSLPL_CUDA(cudaGetLastError());
    return SSLPL_OK;
}

int sslpl_match_bow_batch_device(sslpl_matcher* m, const uint8_t* d_desc, const sslpl_keypoint* d_kps, const int* d_n,
                                 int nframes, int cap, const uint8_t* d_centroids, int nc, float nnratio, int checkOri,
                                 int32_t* d_match, int32_t* d_nmatch) {
    SSLPL_REQUIRE(m && d_desc && d_kps && d_n && d_centroids && d_match && d_nmatch, SSLPL_ERR_ARG, "null argument");
    SSLPL_REQUIRE(nframes >= 2 && nframes <= m->p.max_batch + 1, SSLPL_ERR_ARG, "nframes exceeds max_batch+1");
    SSLPL_REQUIRE(cap >= 1 && cap <= m->p.max_features + 64 && nc >= 1 && nc <= m->p.max_nodes, SSLPL_ERR_ARG, "cap or nc exceeds the matcher capacity");
    SSLPL_CUDA(cudaSetDevice(m->p.device));
    const int fc = m->p.max_features + 64;
    SSLPL_REQUIRE((size_t)(nc * 32) <= (size_t)MAX_DYN_SMEM, SSLPL_ERR_CAPACITY, "too many centroids for one shared-memory tile (nc <= 6400)");
    k_bow_assign<<<dim3((cap + 127) / 128, nframes), 128, nc * 32, m->stream>>>(d_desc, (long long)cap * 32, d_n, 0, cap, d_centroids, nc, m->b_node, fc);
    m->launches += 1;
    return bow_batch_tail(m, d_desc, d_kps, d_n, nframes, cap, nc, nnratio, checkOri, d_match, d_nmatch);
}

// ---------------- projection-gated matcher (SURVEY.md 8(f) row 2) ----------------
int sslpl_search_by_projection_frame(sslpl_matcher* m,
        int n1, const uint8_t* valid1, const uint8_t* obs1, const float* Xw, const uint8_t* dmp, const int32_t* oct1, const float* angle1,
        int n2, const uint8_t* d2, const float* x2, const float* y2, const int32_t* oct2, const float* angle2, const float* uright2,
        const uint8_t* claimed2, const float* Tcw, const float* Tlw, const float* cam, const float* bounds,
        const float* scaleFactors, int nlevels, float th, int bMono, int checkOri, int32_t* assign2, int* nmatches) {
    SSLPL_REQUIRE(m && assign2 && nmatches && Tcw && cam && bounds && scaleFactors, SSLPL_ERR_ARG, "null argument");
    SSLPL_REQUIRE(n1 >= 0 && n2 >= 0 && n1 <= m->cap && n2 <= m->cap && m->cap <= 8192 + 64, SSLPL_ERR_ARG, "n1 / n2 exceed the matcher capacity (<= 8192 features)");
    SSLPL_REQUIRE(m->p.max_nodes >= GRID_COLS * GRID_ROWS, SSLPL_ERR_ARG, "the matcher needs max_nodes >= 3072 (64 x 48 grid cells)");
    SSLPL_REQUIRE(nlevels >= 1 && nlevels <= 32, SSLPL_ERR_ARG, "nlevels out of range");
    SSLPL_REQUIRE(n1 == 0 || (valid1 && obs1 && Xw && dmp && oct1 && angle1), SSLPL_ERR_ARG, "null last-frame array");
    SSLPL_REQUIRE(n2 == 0 || (d2 && x2 && y2 && oct2 && angle2), SSLPL_ERR_ARG, "null current-frame array");
    SSLPL_REQUIRE(bMono || Tlw, SSLPL_ERR_ARG, "the stereo direction test needs the last frame's pose");
    for (int j = 0; j < n2; j++) assign2[j] = -1;
    *nmatches = 0;
    if (n1 == 0 || n2 == 0) return SSLPL_OK;
    for (int i = 0; i < n1; i++) SSLPL_REQUIRE(oct1[i] >= 0 && oct1[i] < nlevels, SSLPL_ERR_ARG, "last-frame octave outside the scale-factor table");
    SSLPL_CUDA(cudaSetDevice(m->p.device));
    cudaStream_t st = m->stream;
    const int cap = m->cap, NN = m->p.max_nodes + 1, nc = GRID_COLS * GRID_ROWS;
    ProjArgs A; memset(&A, 0, sizeof(A));
    for (int k = 0; k < 12; k++) A.T[k] = Tcw[k];
    A.fx = cam[0]; A.fy = cam[1]; A.cx = cam[2]; A.cy = cam[3]; A.mbf = cam[4];
    A.minX = bounds[0]; A.maxX = bounds[1]; A.minY = bounds[2]; A.maxY = bounds[3];
    A.invW = (float)GRID_COLS / (bounds[1] - bounds[0]); A.invH = (float)GRID_ROWS / (bounds[3] - bounds[2]);   // Frame.cc:115-116
    A.th = th; A.checkOri = checkOri ? 1 : 0; A.use_right = uright2 ? 1 : 0;
    for (int k = 0; k < nlevels; k++) A.scale[k] = scaleFactors[k];
    if (!bMono) {                                                        // tlc = Rlw * (-Rcw^T tcw) + tlw against the baseline (:1352-1353)
        float twc[3];
        for (int r = 0; r < 3; r++) twc[r] = (float)(-((double)Tcw[r] * Tcw[3] + (double)Tcw[4 + r] * Tcw[7] + (double)Tcw[8 + r] * Tcw[11]));
        // twc = -Rcw.t()*tcw carries a transpose flag => cv::gemm's general path (double accumulation, above); tlc = Rlw*twc+tlw
        // is a plain product => float path.  Host code: volatile keeps the compiler from contracting the float chain.
        volatile float s = Tlw[8] * twc[0]; s = s + Tlw[9] * twc[1]; s = s + Tlw[10] * twc[2];
        const float tlcz = s + Tlw[11];
        A.forward = tlcz > cam[5]; A.backward = -tlcz > cam[5];
    }
    // staging (pinned scratch would avoid the pageable copies; this entry point is per frame pair, not the batched path)
    std::vector<uint8_t> fl(n1);
    for (int i = 0; i < n1; i++) fl[i] = (uint8_t)((valid1[i] ? 1 : 0) | (obs1[i] ? 2 : 0));
    float* k0 = m->kpf; float* k1 = m->kpf + (size_t)cap * 7;
    SSLPL_CUDA(cudaMemcpyAsync(m->desc, dmp, (size_t)n1 * 32, cudaMemcpyHostToDevice, st));
    SSLPL_CUDA(cudaMemcpyAsync(m->desc + (size_t)cap * 32, d2, (size_t)n2 * 32, cudaMemcpyHostToDevice, st));
    SSLPL_CUDA(cudaMemcpyAsync(k0, Xw, sizeof(float) * 3 * n1, cudaMemcpyHostToDevice, st));
    SSLPL_CUDA(cudaMemcpyAsync(k0 + 3 * (size_t)cap, angle1, sizeof(float) * n1, cudaMemcpyHostToDevice, st));
    SSLPL_CUDA(cudaMemcpyAsync(k0 + 4 * (size_t)cap, oct1, sizeof(int) * n1, cudaMemcpyHostToDevice, st));
    SSLPL_CUDA(cudaMemcpyAsync(k1, x2, sizeof(float) * n2, cudaMemcpyHostToDevice, st));
    SSLPL_CUDA(cudaMemcpyAsync(k1 + (size_t)cap, y2, sizeof(float) * n2, cudaMemcpyHostToDevice, st));
    SSLPL_CUDA(cudaMemcpyAsync(k1 + 2 * (size_t)cap, angle2, sizeof(float) * n2, cudaMemcpyHostToDevice, st));
    if (uright2) SSLPL_CUDA(cudaMemcpyAsync(k1 + 3 * (size_t)cap, uright2, sizeof(float) * n2, cudaMemcpyHostToDevice, st));
    SSLPL_CUDA(cudaMemcpyAsync(k1 + 4 * (size_t)cap, oct2, sizeof(int) * n2, cudaMemcpyHostToDevice, st));
    SSLPL_CUDA(cudaMemcpyAsync(m->flag, fl.data(), n1, cudaMemcpyHostToDevice, st));
    if (claimed2) SSLPL_CUDA(cudaMemcpyAsync(m->flag + cap, claimed2, n2, cudaMemcpyHostToDevice, st));
    else SSLPL_CUDA(cudaMemsetAsync(m->flag + cap, 0, n2, st));
    m->h_small[0] = n2;
    SSLPL_CUDA(cudaMemcpyAsync(m->ncnt, m->h_small, sizeof(int), cudaMemcpyHostToDevice, st));
    SSLPL_CUDA(cudaStreamSynchronize(st));                               // fl (pageable) and h_small are reused by the caller / next call
    int* goff = m->off + (NN + 1); int* gidx = m->idx + cap;
    k_grid_cells<<<(n2 + 127) / 128, 128, 0, st>>>(k1, k1 + cap, n2, A.minX, A.minY, A.invW, A.invH, m->node);
    SSLPL_REQUIRE((size_t)((nc + 1 + cap) * sizeof(int)) <= (size_t)MAX_DYN_SMEM, SSLPL_ERR_CAPACITY, "nodes + features exceed the shared memory of one CTA ((nc + 1 + cap) * 4 <= 200 KB)");
    k_build_csr<<<1, 128, (nc + 1 + cap) * sizeof(int), st>>>(m->node, 0, m->ncnt, cap, nc, goff, 0, gidx, 0);
    k_proj_match<<<1, 32, 0, st>>>(A, n1, m->flag, k0, m->desc, reinterpret_cast<const int*>(k0 + 4 * (size_t)cap), k0 + 3 * (size_t)cap,
                                   n2, m->desc + (size_t)cap * 32, k1, k1 + cap, reinterpret_cast<const int*>(k1 + 4 * (size_t)cap), k1 + 2 * (size_t)cap,
                                   k1 + 3 * (size_t)cap, m->flag + cap, goff, gidx, m->out, m->pairs, m->rot, m->nmatch);
    m->launches += 3;
    SSLPL_CUDA(cudaGetLastError());
    SSLPL_CUDA(cudaMemcpyAsync(assign2, m->out, sizeof(int32_t) * n2, cudaMemcpyDeviceToHost, st));
    SSLPL_CUDA(cudaMemcpyAsync(m->h_small, m->nmatch, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    SSLPL_CUDA(cudaStreamSynchronize(st));
    *nmatches = m->h_small[0];
    return SSLPL_OK;
}

static void fill_win(WinArgs& A, const float* bounds, const float* scaleFactors, int nlevels) {
    memset(&A, 0, sizeof(A));
    A.minX = bounds[0]; A.minY = bounds[2];
    A.invW = (float)GRID_COLS / (bounds[1] - bounds[0]); A.invH = (float)GRID_ROWS / (bounds[3] - bounds[2]);   // Frame.cc:115-116
    for (int k = 0; k < nlevels && k < 32; k++) A.scale[k] = scaleFactors ? scaleFactors[k] : 1.f;
}

int sslpl_search_by_projection_mps(sslpl_matcher* m,
        int nmp, const uint8_t* inview, const uint8_t* bad, const uint8_t* obs, const float* projx, const float* projy, const float* projxr,
        const int32_t* level, const float* viewcos, const uint8_t* dmp,
        int n2, const uint8_t* d2, const float* x2, const float* y2, const int32_t* oct2, const float* uright2, const uint8_t* held2,
        const float* bounds, const float* scaleFactors, int nlevels, float nnratio, float th, int32_t* assign2, int* nmatches) {
    SSLPL_REQUIRE(m && assign2 && nmatches && bounds && scaleFactors, SSLPL_ERR_ARG, "null argument");
    SSLPL_REQUIRE(nmp >= 0 && n2 >= 0 && nmp <= m->cap && n2 <= m->cap && m->cap <= 8192 + 64, SSLPL_ERR_ARG, "nmp / n2 exceed the matcher capacity (<= 8192)");
    SSLPL_REQUIRE(m->p.max_nodes >= GRID_COLS * GRID_ROWS, SSLPL_ERR_ARG, "the matcher needs max_nodes >= 3072 (64 x 48 grid cells)");
    SSLPL_REQUIRE(nlevels >= 1 && nlevels <= 32, SSLPL_ERR_ARG, "nlevels out of range");
    SSLPL_REQUIRE(nmp == 0 || (inview && projx && projy && level && viewcos && dmp), SSLPL_ERR_ARG, "null MapPoint array");
    SSLPL_REQUIRE(n2 == 0 || (d2 && x2 && y2 && oct2), SSLPL_ERR_ARG, "null frame array");
    SSLPL_REQUIRE(!uright2 || projxr, SSLPL_ERR_ARG, "stereo frame features need mTrackProjXR");
    for (int j = 0; j < n2; j++) assign2[j] = -1;
    *nmatches = 0;
    if (nmp == 0 || n2 == 0) return SSLPL_OK;
    for (int i = 0; i < nmp; i++) SSLPL_REQUIRE(level[i] >= 0 && level[i] < nlevels, SSLPL_ERR_ARG, "predicted level outside the scale-factor table");
    SSLPL_CUDA(cudaSetDevice(m->p.device));
    cudaStream_t st = m->stream;
    const int cap = m->cap, NN = m->p.max_nodes + 1, nc = GRID_COLS * GRID_ROWS;
    WinArgs A; fill_win(A, bounds, scaleFactors, nlevels);
    A.th = th; A.nnratio = nnratio; A.bFactor = th != 1.0f; A.use_right = uright2 ? 1 : 0;
    std::vector<uint8_t> fl(nmp), cl(n2, 0);
    for (int i = 0; i < nmp; i++) fl[i] = (uint8_t)(((inview[i] && !(bad && bad[i])) ? 1 : 0) | ((obs && obs[i]) ? 2 : 0));
    if (held2) for (int j = 0; j < n2; j++) cl[j] = held2[j] == 1;
    float* k0 = m->kpf; float* k1 = m->kpf + (size_t)cap * 7;
    SSLPL_CUDA(cudaMemcpyAsync(m->desc, dmp, (size_t)nmp * 32, cudaMemcpyHostToDevice, st));
    SSLPL_CUDA(cudaMemcpyAsync(m->desc + (size_t)cap * 32, d2, (size_t)n2 * 32, cudaMemcpyHostToDevice, st));
    SSLPL_CUDA(cudaMemcpyAsync(k0, projx, sizeof(float) * nmp, cudaMemcpyHostToDevice, st));
    SSLPL_CUDA(cudaMemcpyAsync(k0 + (size_t)cap, projy, sizeof(float) * nmp, cudaMemcpyHostToDevice, st));
    if (projxr) SSLPL_CUDA(cudaMemcpyAsync(k0 + 2 * (size_t)cap, projxr, sizeof(float) * nmp, cudaMemcpyHostToDevice, st));
    SSLPL_CUDA(cudaMemcpyAsync(k0 + 3 * (size_t)cap, viewcos, sizeof(float) * nmp, cudaMemcpyHostToDevice, st));
    SSLPL_CUDA(cudaMemcpyAsync(k0 + 4 * (size_t)cap, level, sizeof(int) * nmp, cudaMemcpyHostToDevice, st));
    SSLPL_CUDA(cudaMemcpyAsync(k1, x2, sizeof(float) * n2, cudaMemcpyHostToDevice, st));
    SSLPL_CUDA(cudaMemcpyAsync(k1 + (size_t)cap, y2, sizeof(float) * n2, cudaMemcpyHostToDevice, st));
    if (uright2) SSLPL_CUDA(cudaMemcpyAsync(k1 + 3 * (size_t)cap, uright2, sizeof(float) * n2, cudaMemcpyHostToDevice, st));
    SSLPL_CUDA(cudaMemcpyAsync(k1 + 4 * (size_t)cap, oct2, sizeof(int) * n2, cudaMemcpyHostToDevice, st));
    SSLPL_CUDA(cudaMemcpyAsync(m->flag, fl.data(), nmp, cudaMemcpyHostToDevice, st));
    SSLPL_CUDA(cudaMemcpyAsync(m->flag + cap, cl.data(), n2, cudaMemcpyHostToDevice, st));
    m->h_small[0] = n2;
    SSLPL_CUDA(cudaMemcpyAsync(m->ncnt, m->h_small, sizeof(int), cudaMemcpyHostToDevice, st));
    SSLPL_CUDA(cudaStreamSynchronize(st));                               // pageable staging vectors go out of scope
    int* goff = m->off + (NN + 1); int* gidx = m->idx + cap;
    k_grid_cells<<<(n2 + 127) / 128, 128, 0, st>>>(k1, k1 + cap, n2, A.minX, A.minY, A.invW, A.invH, m->node);
    SSLPL_REQUIRE((size_t)((nc + 1 + cap) * sizeof(int)) <= (size_t)MAX_DYN_SMEM, SSLPL_ERR_CAPACITY, "nodes + features exceed the shared memory of one CTA ((nc + 1 + cap) * 4 <= 200 KB)");
    k_build_csr<<<1, 128, (nc + 1 + cap) * sizeof(int), st>>>(m->node, 0, m->ncnt, cap, nc, goff, 0, gidx, 0);
    k_proj_match_mps<<<1, 32, 0, st>>>(A, nmp, m->flag, k0, k0 + cap, k0 + 2 * (size_t)cap, reinterpret_cast<const int*>(k0 + 4 * (size_t)cap), k0 + 3 * (size_t)cap, m->desc,
                                       n2, m->desc + (size_t)cap * 32, k1, k1 + cap, reinterpret_cast<const int*>(k1 + 4 * (size_t)cap), k1 + 3 * (size_t)cap,
                                       m->flag + cap, goff, gidx, m->out, m->nmatch);
    m->launches += 3;
    SSLPL_CUDA(cudaGetLastError());
    SSLPL_CUDA(cudaMemcpyAsync(assign2, m->out, sizeof(int32_t) * n2, cudaMemcpyDeviceToHost, st));
    SSLPL_CUDA(cudaMemcpyAsync(m->h_small, m->nmatch, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    SSLPL_CUDA(cudaStreamSynchronize(st));
    *nmatches = m->h_small[0];
    return SSLPL_OK;
}

int sslpl_search_for_initialization(sslpl_matcher* m,
        int n1, const uint8_t* d1, const int32_t* oct1, const float* angle1, float* prev_xy /* [n1][2], in/out */,
        int n2, const uint8_t* d2, const float* x2, const float* y2, const int32_t* oct2, const float* angle2,
        const float* bounds, float nnratio, int checkOri, int windowSize, int32_t* matches12, int* nmatches) {
    SSLPL_REQUIRE(m && matches12 && nmatches && bounds, SSLPL_ERR_ARG, "null argument");
    SSLPL_REQUIRE(n1 >= 0 && n2 >= 0 && n1 <= m->cap && n2 <= m->cap && m->cap <= 8192 + 64, SSLPL_ERR_ARG, "n1 / n2 exceed the matcher capacity (<= 8192 features)");
    SSLPL_REQUIRE(m->p.max_nodes >= GRID_COLS * GRID_ROWS, SSLPL_ERR_ARG, "the matcher needs max_nodes >= 3072 (64 x 48 grid cells)");
    SSLPL_REQUIRE(n1 == 0 || (d1 && oct1 && angle1 && prev_xy), SSLPL_ERR_ARG, "null first-frame array");
    SSLPL_REQUIRE(n2 == 0 || (d2 && x2 && y2 && oct2 && angle2), SSLPL_ERR_ARG, "null second-frame array");
    for (int i = 0; i < n1; i++) matches12[i] = -1;
    *nmatches = 0;
    if (n1 == 0 || n2 == 0) return SSLPL_OK;
    SSLPL_CUDA(cudaSetDevice(m->p.device));
    cudaStream_t st = m->stream;
    const int cap = m->cap, NN = m->p.max_nodes + 1, nc = GRID_COLS * GRID_ROWS;
    WinArgs A; fill_win(A, bounds, nullptr, 0);
    A.nnratio = nnratio; A.checkOri = checkOri ? 1 : 0; A.window = windowSize;
    std::vector<float> px(n1), py(n1);
    for (int i = 0; i < n1; i++) { px[i] = prev_xy[2 * i]; py[i] = prev_xy[2 * i + 1]; }
    float* k0 = m->kpf; float* k1 = m->kpf + (size_t)cap * 7;
    SSLPL_CUDA(cudaMemcpyAsync(m->desc, d1, (size_t)n1 * 32, cudaMemcpyHostToDevice, st));
    SSLPL_CUDA(cudaMemcpyAsync(m->desc + (size_t)cap * 32, d2, (size_t)n2 * 32, cudaMemcpyHostToDevice, st));
    SSLPL_CUDA(cudaMemcpyAsync(k0, px.data(), sizeof(float) * n1, cudaMemcpyHostToDevice, st));
    SSLPL_CUDA(cudaMemcpyAsync(k0 + (size_t)cap, py.data(), sizeof(float) * n1, cudaMemcpyHostToDevice, st));
    SSLPL_CUDA(cudaMemcpyAsync(k0 + 3 * (size_t)cap, angle1, sizeof(float) * n1, cudaMemcpyHostToDevice, st));
    SSLPL_CUDA(cudaMemcpyAsync(k0 + 4 * (size_t)cap, oct1, sizeof(int) * n1, cudaMemcpyHostToDevice, st));
    SSLPL_CUDA(cudaMemcpyAsync(k1, x2, sizeof(float) * n2, cudaMemcpyHostToDevice, st));
    SSLPL_CUDA(cudaMemcpyAsync(k1 + (size_t)cap, y2, sizeof(float) * n2, cudaMemcpyHostToDevice, st));
    SSLPL_CUDA(cudaMemcpyAsync(k1 + 2 * (size_t)cap, angle2, sizeof(float) * n2, cudaMemcpyHostToDevice, st));
    SSLPL_CUDA(cudaMemcpyAsync(k1 + 4 * (size_t)cap, oct2, sizeof(int) * n2, cudaMemcpyHostToDevice, st));
    m->h_small[0] = n2;
    SSLPL_CUDA(cudaMemcpyAsync(m->ncnt, m->h_small, sizeof(int), cudaMemcpyHostToDevice, st));
    SSLPL_CUDA(cudaStreamSynchronize(st));
    int* goff = m->off + (NN + 1); int* gidx = m->idx + cap;
    k_grid_cells<<<(n2 + 127) / 128, 128, 0, st>>>(k1, k1 + cap, n2, A.minX, A.minY, A.invW, A.invH, m->node);
    SSLPL_REQUIRE((size_t)((nc + 1 + cap) * sizeof(int)) <= (size_t)MAX_DYN_SMEM, SSLPL_ERR_CAPACITY, "nodes + features exceed the shared memory of one CTA ((nc + 1 + cap) * 4 <= 200 KB)");
    k_build_csr<<<1, 128, (nc + 1 + cap) * sizeof(int), st>>>(m->node, 0, m->ncnt, cap, nc, goff, 0, gidx, 0);
    k_init_match<<<1, 32, 0, st>>>(A, n1, m->desc, reinterpret_cast<const int*>(k0 + 4 * (size_t)cap), k0 + 3 * (size_t)cap, k0, k0 + cap,
                                   n2, m->desc + (size_t)cap * 32, k1, k1 + cap, reinterpret_cast<const int*>(k1 + 4 * (size_t)cap), k1 + 2 * (size_t)cap,
                                   goff, gidx, m->knn, m->knn + cap, m->out, m->rot, m->nmatch);
    m->launches += 3;
    SSLPL_CUDA(cudaGetLastError());
    SSLPL_CUDA(cudaMemcpyAsync(matches12, m->out, sizeof(int32_t) * n1, cudaMemcpyDeviceToHost, st));
    SSLPL_CUDA(cudaMemcpyAsync(px.data(), k0, sizeof(float) * n1, cudaMemcpyDeviceToHost, st));
    SSLPL_CUDA(cudaMemcpyAsync(py.data(), k0 + cap, sizeof(float) * n1, cudaMemcpyDeviceToHost, st));
    SSLPL_CUDA(cudaMemcpyAsync(m->h_small, m->nmatch, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    SSLPL_CUDA(cudaStreamSynchronize(st));
    for (int i = 0; i < n1; i++) { prev_xy[2 * i] = px[i]; prev_xy[2 * i + 1] = py[i]; }
    *nmatches = m->h_small[0];
    return SSLPL_OK;
}

// Frame::GetFeaturesInArea on its own (Frame.cc:368-421) is host logic over the same CSR; the matcher above is its only
// device consumer.  (The per-frame grid build is k_grid_cells + k_build_csr.)

// ---------------- line projection search and Fuse search (SURVEY.md 8(f) row 3) ----------------
static int ensure_scratch(sslpl_matcher* m, size_t need) {           // grow-only scratch shared by the entry points below
    if (need <= m->scratch_size) return SSLPL_OK;
    SSLPL_CUDA(cudaStreamSynchronize(m->stream));
    if (m->scratch) cudaFree(m->scratch);
    m->scratch = nullptr; m->scratch_size = 0;
    cudaError_t e = cudaMalloc(&m->scratch, need);
    if (e != cudaSuccess) { set_error("cudaMalloc(%zu) failed: %s", need, cudaGetErrorString(e)); return SSLPL_ERR_CUDA; }
    m->scratch_size = need;
    return SSLPL_OK;
}

int sslpl_line_search_by_projection(sslpl_matcher* m, int nml, const uint8_t* active, const uint8_t* obs, const float* proj, const float* radius,
                                    const int32_t* minLevel, const int32_t* maxLevel, const uint8_t* dml,
                                    int nl2, const uint8_t* ld2, const float* kl2, const int32_t* oct2, const uint8_t* held2,
                                    float nnratio, int32_t* assign2, int* nmatches) {
    SSLPL_REQUIRE(m && nmatches && nml >= 0 && nl2 >= 0, SSLPL_ERR_ARG, "null argument");
    SSLPL_REQUIRE(nml == 0 || (active && proj && radius && minLevel && maxLevel && dml), SSLPL_ERR_ARG, "null MapLine array");
    SSLPL_REQUIRE(nl2 == 0 || (ld2 && kl2 && oct2 && assign2), SSLPL_ERR_ARG, "null frame-line array");
    for (int j = 0; j < nl2; j++) assign2[j] = -1;
    *nmatches = 0;
    if (nml == 0 || nl2 == 0) return SSLPL_OK;
    SSLPL_CUDA(cudaSetDevice(m->p.device));
    cudaStream_t st = m->stream;
    const size_t need = (size_t)nml * (1 + 16 + 4 + 4 + 4 + 32) + (size_t)nl2 * (32 + 12 + 4 + 1 + 4) + 16 * 256 + 4096;
    if (int rc = ensure_scratch(m, need)) return rc;
    std::vector<uint8_t> fl(nml), cl(nl2, 0);
    for (int i = 0; i < nml; i++) fl[i] = (uint8_t)((active[i] ? 1 : 0) | ((obs && obs[i]) ? 2 : 0));
    if (held2) for (int j = 0; j < nl2; j++) cl[j] = held2[j] == 1;
    Arena A; A.base = m->scratch; A.used = 0;
    cudaError_t e = cudaSuccess;
    uint8_t* d_fl = stage(A, fl.data(), nml, st, e); float* d_proj = stage(A, proj, (size_t)4 * nml, st, e); float* d_rad = stage(A, radius, nml, st, e);
    int32_t* d_min = stage(A, minLevel, nml, st, e); int32_t* d_max = stage(A, maxLevel, nml, st, e); uint8_t* d_dml = stage(A, dml, (size_t)32 * nml, st, e);
    uint8_t* d_ld2 = stage(A, ld2, (size_t)32 * nl2, st, e); float* d_kl2 = stage(A, kl2, (size_t)3 * nl2, st, e); int32_t* d_oct = stage(A, oct2, nl2, st, e);
    uint8_t* d_cl = stage(A, cl.data(), nl2, st, e); int32_t* d_out = A.take<int32_t>(nl2 + 8);
    SSLPL_CUDA(e);
    SSLPL_CUDA(cudaStreamSynchronize(st));                               // the pageable staging vectors go out of scope
    k_line_window_search<<<1, 32, 0, st>>>(nml, d_fl, reinterpret_cast<const float4*>(d_proj), d_rad, d_min, d_max, d_dml, nl2, d_ld2, d_kl2, d_oct, d_cl,
                                           nnratio, d_out, m->nmatch);
    m->launches++;
    SSLPL_CUDA(cudaGetLastError());
    SSLPL_CUDA(cudaMemcpyAsync(assign2, d_out, sizeof(int32_t) * nl2, cudaMemcpyDeviceToHost, st));
    SSLPL_CUDA(cudaMemcpyAsync(m->h_small, m->nmatch, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    SSLPL_CUDA(cudaStreamSynchronize(st));
    *nmatches = m->h_small[0];
    return SSLPL_OK;
}

int sslpl_fuse_lines_search(sslpl_matcher* m, int nml, const uint8_t* active, const float* proj, const int32_t* level, const uint8_t* dml,
                            int nl2, const uint8_t* ld2, const float* kl2, const int32_t* oct2, const float* scaleFactors, int nlevels, float th,
                            int32_t* best_idx, int32_t* best_dist) {
    SSLPL_REQUIRE(m && nml >= 0 && nl2 >= 0 && scaleFactors && nlevels >= 1 && nlevels <= 32, SSLPL_ERR_ARG, "bad argument");
    SSLPL_REQUIRE(nml == 0 || (active && proj && level && dml && best_idx && best_dist), SSLPL_ERR_ARG, "null MapLine array");
    SSLPL_REQUIRE(nl2 == 0 || (ld2 && kl2 && oct2), SSLPL_ERR_ARG, "null KeyFrame-line array");
    for (int i = 0; i < nml; i++) { best_idx[i] = -1; best_dist[i] = 0x7fffffff; }
    if (nml == 0 || nl2 == 0) return SSLPL_OK;
    std::vector<uint8_t> act(nml);
    for (int i = 0; i < nml; i++) act[i] = active[i] && level[i] >= 0 && level[i] < nlevels;      // MapLine::PredictScale is not clamped: out-of-pyramid levels are dropped
    SSLPL_CUDA(cudaSetDevice(m->p.device));
    cudaStream_t st = m->stream;
    const size_t need = (size_t)nml * (1 + 16 + 4 + 32 + 8) + (size_t)nl2 * (32 + 12 + 4) + 16 * 256 + 4096;
    if (int rc = ensure_scratch(m, need)) return rc;
    Arena A; A.base = m->scratch; A.used = 0;
    cudaError_t e = cudaSuccess;
    uint8_t* d_act = stage(A, act.data(), nml, st, e); float* d_proj = stage(A, proj, (size_t)4 * nml, st, e); int32_t* d_lvl = stage(A, level, nml, st, e);
    uint8_t* d_dml = stage(A, dml, (size_t)32 * nml, st, e); uint8_t* d_ld2 = stage(A, ld2, (size_t)32 * nl2, st, e);
    float* d_kl2 = stage(A, kl2, (size_t)3 * nl2, st, e); int32_t* d_oct = stage(A, oct2, nl2, st, e); float* d_sc = stage(A, scaleFactors, nlevels, st, e);
    int32_t* d_bi = A.take<int32_t>(nml + 8); int32_t* d_bd = A.take<int32_t>(nml + 8);
    SSLPL_CUDA(e);
    SSLPL_CUDA(cudaStreamSynchronize(st));
    k_line_fuse_search<<<(nml + 3) / 4, 128, 0, st>>>(nml, d_act, reinterpret_cast<const float4*>(d_proj), d_lvl, d_dml, nl2, d_ld2, d_kl2, d_oct, d_sc, th, d_bi, d_bd);
    m->launches++;
    SSLPL_CUDA(cudaGetLastError());
    SSLPL_CUDA(cudaMemcpyAsync(best_idx, d_bi, sizeof(int32_t) * nml, cudaMemcpyDeviceToHost, st));
    SSLPL_CUDA(cudaMemcpyAsync(best_dist, d_bd, sizeof(int32_t) * nml, cudaMemcpyDeviceToHost, st));
    SSLPL_CUDA(cudaStreamSynchronize(st));
    return SSLPL_OK;
}

int sslpl_fuse_points_search(sslpl_matcher* m, int nmp, const uint8_t* active, const float* u, const float* v, const float* ur, const int32_t* level, const uint8_t* dmp,
                             int n2, const uint8_t* d2, const float* x2, const float* y2, const int32_t* oct2, const float* uright2,
                             const float* bounds, const float* scaleFactors, const float* invLevelSigma2, int nlevels, float th,
                             int32_t* best_idx, int32_t* best_dist) {
    SSLPL_REQUIRE(m && nmp >= 0 && n2 >= 0 && bounds && scaleFactors && invLevelSigma2 && nlevels >= 1 && nlevels <= 32, SSLPL_ERR_ARG, "bad argument");
    SSLPL_REQUIRE(n2 <= m->cap && m->cap <= 8192 + 64, SSLPL_ERR_ARG, "n2 exceeds the matcher capacity (<= 8192 features)");
    SSLPL_REQUIRE(m->p.max_nodes >= GRID_COLS * GRID_ROWS, SSLPL_ERR_ARG, "the matcher needs max_nodes >= 3072 (64 x 48 grid cells)");
    SSLPL_REQUIRE(nmp == 0 || (active && u && v && level && dmp && best_idx && best_dist), SSLPL_ERR_ARG, "null MapPoint array");
    SSLPL_REQUIRE(n2 == 0 || (d2 && x2 && y2 && oct2), SSLPL_ERR_ARG, "null KeyFrame array");
    for (int i = 0; i < nmp; i++) { best_idx[i] = -1; best_dist[i] = 256; }
    if (nmp == 0 || n2 == 0) return SSLPL_OK;
    for (int i = 0; i < nmp; i++) SSLPL_REQUIRE(!active[i] || (level[i] >= 0 && level[i] < nlevels), SSLPL_ERR_ARG, "predicted level outside the pyramid");
    SSLPL_CUDA(cudaSetDevice(m->p.device));
    cudaStream_t st = m->stream;
    const int cap = m->cap, NN = m->p.max_nodes + 1, nc = GRID_COLS * GRID_ROWS;
    WinArgs A; fill_win(A, bounds, scaleFactors, nlevels);
    A.th = th; A.use_right = uright2 ? 1 : 0;
    const size_t need = (size_t)nmp * (1 + 12 + 4 + 32 + 8) + (size_t)n2 * (32 + 16) + 32 * 4 + 16 * 256 + 4096;
    if (int rc = ensure_scratch(m, need)) return rc;
    Arena S; S.base = m->scratch; S.used = 0;
    cudaError_t e = cudaSuccess;
    std::vector<float> urz;
    if (!ur) { urz.assign(nmp, 0.f); ur = urz.data(); }
    uint8_t* d_act = stage(S, active, nmp, st, e); float* d_u = stage(S, u, nmp, st, e); float* d_v = stage(S, v, nmp, st, e); float* d_ur = stage(S, ur, nmp, st, e);
    int32_t* d_lvl = stage(S, level, nmp, st, e); uint8_t* d_dmp = stage(S, dmp, (size_t)32 * nmp, st, e);
    uint8_t* d_d2 = stage(S, d2, (size_t)32 * n2, st, e); float* d_x2 = stage(S, x2, n2, st, e); float* d_y2 = stage(S, y2, n2, st, e);
    int32_t* d_oct = stage(S, oct2, n2, st, e); float* d_ur2 = stage(S, uright2, uright2 ? n2 : 0, st, e); float* d_is2 = stage(S, invLevelSigma2, nlevels, st, e);
    int32_t* d_bi = S.take<int32_t>(nmp + 8); int32_t* d_bd = S.take<int32_t>(nmp + 8);
    m->h_small[0] = n2;
    if (e == cudaSuccess) e = cudaMemcpyAsync(m->ncnt, m->h_small, sizeof(int), cudaMemcpyHostToDevice, st);
    SSLPL_CUDA(e);
    SSLPL_CUDA(cudaStreamSynchronize(st));
    int* goff = m->off + (NN + 1); int* gidx = m->idx + cap;
    k_grid_cells<<<(n2 + 127) / 128, 128, 0, st>>>(d_x2, d_y2, n2, A.minX, A.minY, A.invW, A.invH, m->node);
    SSLPL_REQUIRE((size_t)((nc + 1 + cap) * sizeof(int)) <= (size_t)MAX_DYN_SMEM, SSLPL_ERR_CAPACITY, "nodes + features exceed the shared memory of one CTA ((nc + 1 + cap) * 4 <= 200 KB)");
    k_build_csr<<<1, 128, (nc + 1 + cap) * sizeof(int), st>>>(m->node, 0, m->ncnt, cap, nc, goff, 0, gidx, 0);
    k_point_fuse_search<<<(nmp + 3) / 4, 128, 0, st>>>(A, nmp, d_act, d_u, d_v, d_ur, d_lvl, d_dmp, d_d2, d_x2, d_y2, d_oct, d_ur2, d_is2, goff, gidx, d_bi, d_bd);
    m->launches += 3;
    SSLPL_CUDA(cudaGetLastError());
    SSLPL_CUDA(cudaMemcpyAsync(best_idx, d_bi, sizeof(int32_t) * nmp, cudaMemcpyDeviceToHost, st));
    SSLPL_CUDA(cudaMemcpyAsync(best_dist, d_bd, sizeof(int32_t) * nmp, cudaMemcpyDeviceToHost, st));
    SSLPL_CUDA(cudaStreamSynchronize(st));
    return SSLPL_OK;
}

// ---------------- descriptor medoids (SURVEY.md 8(f) row 3) ----------------
int sslpl_descriptor_medoid_batch(sslpl_matcher* m, const uint8_t* desc, const int32_t* off, int ngroups, int32_t* best_idx, int32_t* best_median) {
    SSLPL_REQUIRE(m && off && ngroups >= 0 && (ngroups == 0 || (best_idx && best_median)), SSLPL_ERR_ARG, "null argument");
    if (ngroups == 0) return SSLPL_OK;
    const int total = off[ngroups];
    SSLPL_REQUIRE(off[0] == 0 && total >= 0 && (total == 0 || desc), SSLPL_ERR_ARG, "bad group offsets");
    for (int g = 0; g < ngroups; g++) SSLPL_REQUIRE(off[g + 1] >= off[g] && off[g + 1] - off[g] < (1 << 20), SSLPL_ERR_ARG, "group offsets must be non-decreasing (groups < 2^20 rows)");
    SSLPL_CUDA(cudaSetDevice(m->p.device));
    cudaStream_t st = m->stream;
    const size_t need = align_up((size_t)total * 32 + 256, 256) + align_up(sizeof(int32_t) * (size_t)(ngroups + 1), 256) + 2 * align_up(sizeof(int32_t) * (size_t)ngroups, 256);
    if (int rc = ensure_scratch(m, need)) return rc;
    Arena A; A.base = m->scratch; A.used = 0;
    uint8_t* d_desc = A.take<uint8_t>((size_t)total * 32 + 32); int32_t* d_off = A.take<int32_t>(ngroups + 1);
    int32_t* d_bi = A.take<int32_t>(ngroups); int32_t* d_bm = A.take<int32_t>(ngroups);
    if (total) SSLPL_CUDA(cudaMemcpyAsync(d_desc, desc, (size_t)total * 32, cudaMemcpyHostToDevice, st));
    SSLPL_CUDA(cudaMemcpyAsync(d_off, off, sizeof(int32_t) * (ngroups + 1), cudaMemcpyHostToDevice, st));
    k_medoid<<<ngroups, 128, 0, st>>>(d_desc, d_off, d_bi, d_bm);
    m->launches++;
    SSLPL_CUDA(cudaGetLastError());
    SSLPL_CUDA(cudaMemcpyAsync(best_idx, d_bi, sizeof(int32_t) * ngroups, cudaMemcpyDeviceToHost, st));
    SSLPL_CUDA(cudaMemcpyAsync(best_median, d_bm, sizeof(int32_t) * ngroups, cudaMemcpyDeviceToHost, st));
    SSLPL_CUDA(cudaStreamSynchronize(st));
    return SSLPL_OK;
}

// ---------------- DBoW2 vocabulary (SURVEY.md 8(f) row 1) ----------------
static int vocab_level_nodes(const sslpl_vocab* v, int levelsup) {
    const int lvl = v->L - levelsup;
    return 1 + ((lvl >= 1 && lvl < (int)v->level_count.size()) ? v->level_count[lvl] : 0);
}

int sslpl_vocab_create(int device, int k, int L, int nnodes, const int32_t* parent, const uint8_t* desc, const double* weight,
                       const uint8_t* is_leaf, sslpl_vocab** out) {
    SSLPL_REQUIRE(out && parent && desc && weight && is_leaf, SSLPL_ERR_ARG, "null argument");
    SSLPL_REQUIRE(k >= 1 && L >= 1 && nnodes >= 1, SSLPL_ERR_ARG, "bad vocabulary shape");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) { set_error("no CUDA device available: libsslpl_b200 has no CPU fallback"); return SSLPL_ERR_CUDA; }
    SSLPL_CUDA(cudaSetDevice(device));
    std::vector<int> cnt(nnodes + 1, 0), depth(nnodes, 0), word(nnodes, -1), rank(nnodes, 0);
    for (int i = 1; i < nnodes; i++) {
        SSLPL_REQUIRE(parent[i] >= 0 && parent[i] < i, SSLPL_ERR_ARG, "vocabulary: parent[i] must be an earlier node");
        cnt[parent[i] + 1]++; depth[i] = depth[parent[i]] + 1;
    }
    for (int i = 0; i < nnodes; i++) cnt[i + 1] += cnt[i];                    // CSR offsets
    std::vector<int> ids(std::max(nnodes - 1, 1)), fillp(cnt.begin(), cnt.end() - 1);
    for (int i = 1; i < nnodes; i++) ids[fillp[parent[i]]++] = i;             // ascending ids inside every list
    int nwords = 0, maxd = 0;
    for (int i = 1; i < nnodes; i++) {
        const bool leaf = cnt[i + 1] == cnt[i];
        SSLPL_REQUIRE(leaf == (is_leaf[i] != 0), SSLPL_ERR_ARG, "vocabulary: is_leaf disagrees with the tree structure");
        if (leaf) word[i] = nwords++;
        maxd = std::max(maxd, depth[i]);
    }
    sslpl_vocab* v = new sslpl_vocab();
    v->device = device; v->k = k; v->L = L; v->nnodes = nnodes; v->nwords = nwords; v->depth = depth;
    v->level_count.assign(maxd + 1, 0);
    for (int i = 0; i < nnodes; i++) rank[i] = v->level_count[depth[i]]++;    // rank among the nodes of the same depth, ascending id
    Arena A;
    A.base = nullptr; A.used = 0;
    auto carve_all = [&](Arena& a, sslpl::VocabView& w) {
        w.child_off = a.take<int>(nnodes + 1); w.child_ids = a.take<int>(ids.size()); w.desc = a.take<uint8_t>((size_t)nnodes * 32);
        w.weight = a.take<double>(nnodes); w.word_id = a.take<int>(nnodes); w.level_rank = a.take<int>(nnodes);
    };
    sslpl::VocabView dry{}; carve_all(A, dry);
    const size_t bytes = A.used + 256;
    cudaError_t e = cudaMalloc(&v->arena, bytes);
    if (e != cudaSuccess) { set_error("cudaMalloc(%zu) failed: %s", bytes, cudaGetErrorString(e)); delete v; return SSLPL_ERR_CUDA; }
    Arena B2; B2.base = v->arena; B2.used = 0;
    carve_all(B2, v->view);
    SSLPL_CUDA(cudaMemcpy(const_cast<int*>(v->view.child_off), cnt.data(), sizeof(int) * (nnodes + 1), cudaMemcpyHostToDevice));
    SSLPL_CUDA(cudaMemcpy(const_cast<int*>(v->view.child_ids), ids.data(), sizeof(int) * ids.size(), cudaMemcpyHostToDevice));
    SSLPL_CUDA(cudaMemcpy(const_cast<uint8_t*>(v->view.desc), desc, (size_t)nnodes * 32, cudaMemcpyHostToDevice));
    SSLPL_CUDA(cudaMemcpy(const_cast<double*>(v->view.weight), weight, sizeof(double) * nnodes, cudaMemcpyHostToDevice));
    SSLPL_CUDA(cudaMemcpy(const_cast<int*>(v->view.word_id), word.data(), sizeof(int) * nnodes, cudaMemcpyHostToDevice));
    SSLPL_CUDA(cudaMemcpy(const_cast<int*>(v->view.level_rank), rank.data(), sizeof(int) * nnodes, cudaMemcpyHostToDevice));
    *out = v;
    return SSLPL_OK;
}

// ORBvoc.txt text format of TemplatedVocabulary::loadFromTextFile (TemplatedVocabulary.h:1338-1420):
// "k L scoring weighting" then one line per node: "parent is_leaf b0 .. b31 weight".  Blank lines are skipped (the reference's
// `while(!f.eof())` loop turns the trailing newline into one bogus node with an uninitialised parent).
int sslpl_vocab_load_text(int device, const char* path, sslpl_vocab** out, int* scoring, int* weighting) {
    SSLPL_REQUIRE(path && out, SSLPL_ERR_ARG, "null argument");
    FILE* f = fopen(path, "r");
    if (!f) { set_error("cannot open vocabulary file %s", path); return SSLPL_ERR_ARG; }
    int k = 0, L = 0, n1 = 0, n2 = 0;
    if (fscanf(f, "%d %d %d %d", &k, &L, &n1, &n2) != 4 || k < 0 || k > 20 || L < 1 || L > 10 || n1 < 0 || n1 > 5 || n2 < 0 || n2 > 3) {
        fclose(f); set_error("%s is not a DBoW2 text vocabulary", path); return SSLPL_ERR_ARG;
    }
    std::vector<int32_t> parent(1, -1); std::vector<uint8_t> desc(32, 0), leaf(1, 0); std::vector<double> weight(1, 0.0);
    for (;;) {
        int pid, isleaf;
        if (fscanf(f, "%d %d", &pid, &isleaf) != 2) break;
        uint8_t d[32];
        bool ok = true;
        for (int i = 0; i < 32 && ok; i++) { int b; ok = fscanf(f, "%d", &b) == 1; d[i] = (uint8_t)b; }
        double w = 0;
        ok = ok && fscanf(f, "%lf", &w) == 1;
        if (!ok) { fclose(f); set_error("%s: truncated node line", path); return SSLPL_ERR_ARG; }
        parent.push_back(pid); leaf.push_back(isleaf > 0 ? 1 : 0); weight.push_back(w); desc.insert(desc.end(), d, d + 32);
    }
    fclose(f);
    if (scoring) *scoring = n1;
    if (weighting) *weighting = n2;
    return sslpl_vocab_create(device, k, L, (int)parent.size(), parent.data(), desc.data(), weight.data(), leaf.data(), out);
}

void sslpl_vocab_destroy(sslpl_vocab* v) {
    if (!v) return;
    cudaSetDevice(v->device);
    if (v->arena) cudaFree(v->arena);
    delete v;
}

int sslpl_vocab_info(const sslpl_vocab* v, int* k, int* L, int* nnodes, int* nwords) {
    SSLPL_REQUIRE(v, SSLPL_ERR_ARG, "null vocabulary");
    if (k) *k = v->k;
    if (L) *L = v->L;
    if (nnodes) *nnodes = v->nnodes;
    if (nwords) *nwords = v->nwords;
    return SSLPL_OK;
}

int sslpl_vocab_level_nodes(const sslpl_vocab* v, int levelsup, int* count) {
    SSLPL_REQUIRE(v && count, SSLPL_ERR_ARG, "null argument");
    *count = vocab_level_nodes(v, levelsup);
    return SSLPL_OK;
}

int sslpl_bow_transform(sslpl_matcher* m, const sslpl_vocab* v, const uint8_t* desc, int n, int levelsup,
                        int32_t* word, int32_t* node, double* weight) {
    SSLPL_REQUIRE(m && v && (n == 0 || (desc && word && node && weight)), SSLPL_ERR_ARG, "null argument");
    SSLPL_REQUIRE(n >= 0 && n <= m->cap, SSLPL_ERR_ARG, "n exceeds the matcher capacity");
    SSLPL_REQUIRE(v->device == m->p.device, SSLPL_ERR_ARG, "vocabulary and matcher live on different devices");
    if (n == 0) return SSLPL_OK;
    SSLPL_CUDA(cudaSetDevice(m->p.device));
    cudaStream_t st = m->stream;
    SSLPL_CUDA(cudaMemcpyAsync(m->desc, desc, (size_t)n * 32, cudaMemcpyHostToDevice, st));
    k_vocab_transform<<<dim3((n + 127) / 128, 1), 128, 0, st>>>(m->desc, 0, nullptr, n, n, v->view, v->L - levelsup, m->word, m->node, nullptr, m->wgt, 0);
    m->launches++;
    SSLPL_CUDA(cudaGetLastError());
    SSLPL_CUDA(cudaMemcpyAsync(word, m->word, sizeof(int32_t) * n, cudaMemcpyDeviceToHost, st));
    SSLPL_CUDA(cudaMemcpyAsync(node, m->node, sizeof(int32_t) * n, cudaMemcpyDeviceToHost, st));
    SSLPL_CUDA(cudaMemcpyAsync(weight, m->wgt, sizeof(double) * n, cudaMemcpyDeviceToHost, st));
    SSLPL_CUDA(cudaStreamSynchronize(st));
    return SSLPL_OK;
}

int sslpl_match_bow_batch_device_vocab(sslpl_matcher* m, const uint8_t* d_desc, const sslpl_keypoint* d_kps, const int* d_n,
                                       int nframes, int cap, const sslpl_vocab* v, int levelsup, float nnratio, int checkOri,
                                       int32_t* d_match, int32_t* d_nmatch, int32_t* d_word, int32_t* d_node, double* d_weight) {
    SSLPL_REQUIRE(m && v && d_desc && d_kps && d_n && d_match && d_nmatch, SSLPL_ERR_ARG, "null argument");
    SSLPL_REQUIRE(nframes >= 2 && nframes <= m->p.max_batch + 1, SSLPL_ERR_ARG, "nframes exceeds max_batch+1");
    const int nc = vocab_level_nodes(v, levelsup);
    SSLPL_REQUIRE(cap >= 1 && cap <= m->p.max_features + 64 && nc <= m->p.max_nodes, SSLPL_ERR_ARG, "cap or the vocabulary level exceeds the matcher capacity (max_nodes)");
    SSLPL_REQUIRE(v->device == m->p.device, SSLPL_ERR_ARG, "vocabulary and matcher live on different devices");
    SSLPL_CUDA(cudaSetDevice(m->p.device));
    const int fc = m->p.max_features + 64;
    // optional per-feature outputs use the caller's [nframes][cap] layout; the dense node index goes to the workspace ([..][fc])
    if (d_word || d_node || d_weight) {
        k_vocab_transform<<<dim3((cap + 127) / 128, nframes), 128, 0, m->stream>>>(d_desc, (long long)cap * 32, d_n, 0, cap, v->view, v->L - levelsup,
                                                                                      d_word, d_node, nullptr, d_weight, cap);
        m->launches += 1;
    }
    k_vocab_transform<<<dim3((cap + 127) / 128, nframes), 128, 0, m->stream>>>(d_desc, (long long)cap * 32, d_n, 0, cap, v->view, v->L - levelsup,
                                                                                  nullptr, nullptr, m->b_node, nullptr, fc);
    m->launches += 1;
    return bow_batch_tail(m, d_desc, d_kps, d_n, nframes, cap, nc, nnratio, checkOri, d_match, d_nmatch);
}

int sslpl_match_lines_batch_device(sslpl_matcher* m, const uint8_t* d_ldesc, const int* d_nl, int nframes, int capl,
                                   int32_t* d_lmatch, int32_t* d_nlmatch) {
    SSLPL_REQUIRE(m && d_ldesc && d_nl && d_lmatch && d_nlmatch, SSLPL_ERR_ARG, "null argument");
    SSLPL_REQUIRE(nframes >= 2 && nframes <= m->p.max_batch + 1 && capl >= 1 && capl <= m->p.max_lines + 64, SSLPL_ERR_ARG, "batch or capacity exceeds the matcher capacity");
    SSLPL_CUDA(cudaSetDevice(m->p.device));
    cudaStream_t st = m->stream;
    const int npairs = nframes - 1, lc = m->p.max_lines + 64;
    k_knn2<<<dim3((capl + 7) / 8, npairs), 256, 0, st>>>(d_ldesc, (long long)capl * 32, d_nl, 0, d_ldesc + (size_t)capl * 32, (long long)capl * 32,
                                                          d_nl, 0, m->b_knn, (long long)lc * 4, capl);
    m->launches++;
    fill(m, d_lmatch, (long long)npairs * capl, -1);
    SSLPL_CUDA(cudaMemsetAsync(d_nlmatch, 0, sizeof(int32_t) * npairs, st));
    k_line_ratio<<<dim3((capl + 127) / 128, npairs), 128, 0, st>>>(m->b_knn, (long long)lc * 4, d_nl, 0, capl, nullptr, 0, d_lmatch, capl, d_nlmatch);
    m->launches++;
    SSLPL_CUDA(cudaGetLastError());
    return SSLPL_OK;
}

// ---------------- keyframe set and reference-keyframe matching (Tracking::TrackReferenceKeyFrame, Tracking.cc:1005-1034) ----------------
void sslpl_kfset_destroy(sslpl_kfset* k);

int sslpl_kfset_create(int device, int max_keyframes, int cap, int capl, sslpl_kfset** out) {
    SSLPL_REQUIRE(out, SSLPL_ERR_ARG, "null argument");
    SSLPL_REQUIRE(max_keyframes >= 1 && cap >= 1 && capl >= 1 && cap < (1 << 20) && capl < (1 << 20), SSLPL_ERR_ARG, "bad keyframe set capacity");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) { set_error("no CUDA device available: libsslpl_b200 has no CPU fallback"); return SSLPL_ERR_CUDA; }
    SSLPL_CUDA(cudaSetDevice(device));
    const size_t K = max_keyframes;
    auto carve_all = [&](Arena& a, KfView& w) {
        w.desc = a.take<uint8_t>(K * cap * 32); w.angle = a.take<float>(K * cap); w.valid = a.take<uint8_t>(K * cap);
        w.nodes = a.take<int>(K * cap); w.off = a.take<int>(K * (cap + 1)); w.idx = a.take<int>(K * cap); w.nn = a.take<int>(K);
        w.ldesc = a.take<uint8_t>(K * capl * 32); w.has_ml = a.take<uint8_t>(K * capl); w.nl = a.take<int>(K);
    };
    Arena A; KfView dry{}; carve_all(A, dry);
    sslpl_kfset* k = new sslpl_kfset();
    k->device = device;
    k->built.assign(K, {nullptr, 0});
    cudaError_t e = cudaMalloc(&k->arena, A.used + 256);
    if (e != cudaSuccess) { set_error("cudaMalloc(%zu) failed: %s", A.used + 256, cudaGetErrorString(e)); delete k; return SSLPL_ERR_CUDA; }
    Arena B; B.base = k->arena; carve_all(B, k->view);
    k->view.cap = cap; k->view.capl = capl; k->view.nslots = max_keyframes;
    e = cudaMemset(k->arena, 0, A.used + 256);                      // every slot empty: nn = n = nl = 0
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&k->stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&k->last_use, cudaEventDisableTiming);
    if (e != cudaSuccess) { set_error("sslpl_kfset_create: %s", cudaGetErrorString(e)); sslpl_kfset_destroy(k); return SSLPL_ERR_CUDA; }
    *out = k;
    return SSLPL_OK;
}

void sslpl_kfset_destroy(sslpl_kfset* k) {
    if (!k) return;
    cudaSetDevice(k->device);
    if (k->last_use) { cudaEventSynchronize(k->last_use); cudaEventDestroy(k->last_use); }
    if (k->stream) { cudaStreamSynchronize(k->stream); cudaStreamDestroy(k->stream); }
    if (k->arena) cudaFree(k->arena);
    delete k;
}

// FeatureVector and counts of slot `slot`, whose descriptors are already (being) copied in, from n_src / nl_src (device)
static int kf_index(sslpl_matcher* m, sslpl_kfset* k, int slot, const int* n_src, int cap_src, const int* nl_src, int capl_src,
                    const sslpl_vocab* v, int levelsup) {
    cudaStream_t st = m->stream;
    const KfView& K = k->view;
    const long long ks = (long long)slot * K.cap;
    const int nc = vocab_level_nodes(v, levelsup);
    k_vocab_transform<<<dim3((cap_src + 127) / 128, 1), 128, 0, st>>>(K.desc + ks * 32, 0, n_src, 0, cap_src, v->view, v->L - levelsup,
                                                                       nullptr, nullptr, m->b_node, nullptr, 0);
    k_build_csr<<<1, 128, (nc + 1 + cap_src) * sizeof(int), st>>>(m->b_node, 0, n_src, cap_src, nc, m->b_off, 0, K.idx + ks, 0);
    k_kf_compact<<<1, 256, 0, st>>>(m->b_off, nc, nl_src, capl_src, K.nodes + ks, K.off + (long long)slot * (K.cap + 1), K.nn + slot, K.nl + slot);
    m->launches += 3;
    SSLPL_CUDA(cudaGetLastError());
    SSLPL_CUDA(cudaMemsetAsync(K.valid + ks, 1, K.cap, st));
    SSLPL_CUDA(cudaMemsetAsync(K.has_ml + (long long)slot * K.capl, 1, K.capl, st));
    SSLPL_CUDA(cudaEventRecord(k->last_use, st));
    k->built[slot] = {v, levelsup};
    return SSLPL_OK;
}

static int kf_store_checks(sslpl_matcher* m, sslpl_kfset* k, int slot, int cap, int capl, const sslpl_vocab* v, int levelsup) {
    SSLPL_REQUIRE(m && k && v, SSLPL_ERR_ARG, "null argument");
    SSLPL_REQUIRE(slot >= 0 && slot < k->view.nslots, SSLPL_ERR_ARG, "slot outside the keyframe set");
    SSLPL_REQUIRE(cap >= 0 && cap <= k->view.cap && cap <= m->p.max_features + 64, SSLPL_ERR_ARG, "cap exceeds the keyframe set or the matcher capacity");
    SSLPL_REQUIRE(capl >= 0 && capl <= k->view.capl, SSLPL_ERR_ARG, "capl exceeds the keyframe set capacity");
    SSLPL_REQUIRE(k->device == m->p.device && v->device == m->p.device, SSLPL_ERR_ARG, "keyframe set, vocabulary and matcher live on different devices");
    const int nc = vocab_level_nodes(v, levelsup);
    SSLPL_REQUIRE(nc <= m->p.max_nodes, SSLPL_ERR_ARG, "the vocabulary level exceeds the matcher capacity (max_nodes)");
    SSLPL_REQUIRE((size_t)((nc + 1 + cap) * sizeof(int)) <= (size_t)MAX_DYN_SMEM, SSLPL_ERR_CAPACITY, "nodes + features exceed the shared memory of one CTA ((nc + 1 + cap) * 4 <= 200 KB)");
    return SSLPL_OK;
}

int sslpl_kfset_store_device(sslpl_matcher* m, sslpl_kfset* k, int slot,
                             const uint8_t* d_desc, const sslpl_keypoint* d_kps, const int* d_n, int cap,
                             const uint8_t* d_ldesc, const int* d_nl, int capl, int frame,
                             const sslpl_vocab* v, int levelsup) {
    if (int rc = kf_store_checks(m, k, slot, cap, capl, v, levelsup)) return rc;
    SSLPL_REQUIRE(d_desc && d_kps && d_n && d_ldesc && d_nl && cap >= 1 && capl >= 1 && frame >= 0, SSLPL_ERR_ARG, "null argument or empty frame capacity");
    SSLPL_CUDA(cudaSetDevice(m->p.device));
    cudaStream_t st = m->stream;
    const KfView& K = k->view;
    const long long ks = (long long)slot * K.cap, f = frame;
    SSLPL_CUDA(cudaMemcpyAsync(K.desc + ks * 32, d_desc + f * cap * 32, (size_t)cap * 32, cudaMemcpyDeviceToDevice, st));
    SSLPL_CUDA(cudaMemcpy2DAsync(K.angle + ks, sizeof(float), reinterpret_cast<const float*>(d_kps + f * cap) + 3,
                                 sizeof(sslpl_keypoint), sizeof(float), cap, cudaMemcpyDeviceToDevice, st));
    SSLPL_CUDA(cudaMemcpyAsync(K.ldesc + (long long)slot * K.capl * 32, d_ldesc + f * capl * 32, (size_t)capl * 32,
                               cudaMemcpyDeviceToDevice, st));
    return kf_index(m, k, slot, d_n + frame, cap, d_nl + frame, capl, v, levelsup);
}

int sslpl_kfset_store(sslpl_matcher* m, sslpl_kfset* k, int slot, const uint8_t* desc, const float* angle, int n,
                      const uint8_t* ldesc, int nl, const sslpl_vocab* v, int levelsup) {
    if (int rc = kf_store_checks(m, k, slot, n, nl, v, levelsup)) return rc;
    SSLPL_REQUIRE((n == 0 || (desc && angle)) && (nl == 0 || ldesc), SSLPL_ERR_ARG, "null descriptor / angle array");
    SSLPL_CUDA(cudaSetDevice(m->p.device));
    cudaStream_t st = m->stream;
    const KfView& K = k->view;
    const long long ks = (long long)slot * K.cap;
    if (n) SSLPL_CUDA(cudaMemcpyAsync(K.desc + ks * 32, desc, (size_t)n * 32, cudaMemcpyHostToDevice, st));
    if (n) SSLPL_CUDA(cudaMemcpyAsync(K.angle + ks, angle, sizeof(float) * n, cudaMemcpyHostToDevice, st));
    if (nl) SSLPL_CUDA(cudaMemcpyAsync(K.ldesc + (long long)slot * K.capl * 32, ldesc, (size_t)nl * 32, cudaMemcpyHostToDevice, st));
    m->h_small[0] = n; m->h_small[1] = nl;
    SSLPL_CUDA(cudaMemcpyAsync(m->ncnt, m->h_small, 2 * sizeof(int), cudaMemcpyHostToDevice, st));
    if (int rc = kf_index(m, k, slot, m->ncnt, std::max(n, 1), m->ncnt + 1, std::max(nl, 1), v, levelsup)) return rc;
    SSLPL_CUDA(cudaStreamSynchronize(st));                                // the caller's host buffers and h_small are free again
    return SSLPL_OK;
}

int sslpl_kfset_set_masks(sslpl_kfset* k, int slot, const uint8_t* valid, int n, const uint8_t* has_ml, int nl) {
    SSLPL_REQUIRE(k, SSLPL_ERR_ARG, "null argument");
    SSLPL_REQUIRE(slot >= 0 && slot < k->view.nslots, SSLPL_ERR_ARG, "slot outside the keyframe set");
    SSLPL_REQUIRE(n >= 0 && n <= k->view.cap && nl >= 0 && nl <= k->view.capl, SSLPL_ERR_ARG, "mask longer than the keyframe set capacity");
    SSLPL_CUDA(cudaSetDevice(k->device));
    const KfView& K = k->view;
    uint8_t* mv = K.valid + (long long)slot * K.cap;
    uint8_t* ml = K.has_ml + (long long)slot * K.capl;
    SSLPL_CUDA(cudaStreamWaitEvent(k->stream, k->last_use, 0));          // after the store that reset them and the matches that read them
    SSLPL_CUDA(cudaMemsetAsync(mv, 1, K.cap, k->stream));
    if (valid && n) SSLPL_CUDA(cudaMemcpyAsync(mv, valid, n, cudaMemcpyHostToDevice, k->stream));
    SSLPL_CUDA(cudaMemsetAsync(ml, 1, K.capl, k->stream));
    if (has_ml && nl) SSLPL_CUDA(cudaMemcpyAsync(ml, has_ml, nl, cudaMemcpyHostToDevice, k->stream));
    SSLPL_CUDA(cudaStreamSynchronize(k->stream));
    return SSLPL_OK;
}

int sslpl_kfset_clear(sslpl_kfset* k, int slot) {
    SSLPL_REQUIRE(k, SSLPL_ERR_ARG, "null argument");
    SSLPL_REQUIRE(slot >= 0 && slot < k->view.nslots, SSLPL_ERR_ARG, "slot outside the keyframe set");
    SSLPL_CUDA(cudaSetDevice(k->device));
    SSLPL_CUDA(cudaStreamWaitEvent(k->stream, k->last_use, 0));
    SSLPL_CUDA(cudaMemsetAsync(k->view.nn + slot, 0, sizeof(int), k->stream));
    SSLPL_CUDA(cudaMemsetAsync(k->view.nl + slot, 0, sizeof(int), k->stream));
    SSLPL_CUDA(cudaStreamSynchronize(k->stream));
    k->built[slot] = {nullptr, 0};
    return SSLPL_OK;
}

int sslpl_match_ref_kf_batch_device(sslpl_matcher* m, const sslpl_kfset* k, const int32_t* d_ref, int nframes,
                                    const uint8_t* d_desc, const sslpl_keypoint* d_kps, const int* d_n, int cap,
                                    const uint8_t* d_ldesc, const int* d_nl, int capl,
                                    const sslpl_vocab* v, int levelsup, float nnratio, int checkOri,
                                    int32_t* d_match, int32_t* d_nmatch, int32_t* d_lmatch, int32_t* d_nlmatch) {
    SSLPL_REQUIRE(m && k && v && d_ref && d_desc && d_kps && d_n && d_ldesc && d_nl && d_match && d_nmatch && d_lmatch && d_nlmatch,
                  SSLPL_ERR_ARG, "null argument");
    SSLPL_REQUIRE(nframes >= 1 && nframes <= m->p.max_batch + 1, SSLPL_ERR_ARG, "nframes exceeds max_batch+1");
    const int fc = m->p.max_features + 64, lc = m->p.max_lines + 64, NN = m->p.max_nodes + 1;
    SSLPL_REQUIRE(cap >= 1 && cap <= fc && capl >= 1 && capl <= lc, SSLPL_ERR_ARG, "cap or capl exceeds the matcher capacity");
    SSLPL_REQUIRE(k->view.capl <= lc, SSLPL_ERR_ARG, "the keyframe set holds more lines per keyframe than the matcher's max_lines + 64");
    SSLPL_REQUIRE(k->device == m->p.device && v->device == m->p.device, SSLPL_ERR_ARG, "keyframe set, vocabulary and matcher live on different devices");
    const int nc = vocab_level_nodes(v, levelsup);
    SSLPL_REQUIRE(nc <= m->p.max_nodes, SSLPL_ERR_ARG, "the vocabulary level exceeds the matcher capacity (max_nodes)");
    for (const auto& b : k->built)
        SSLPL_REQUIRE(!b.v || (b.v == v && b.levelsup == levelsup), SSLPL_ERR_ARG, "a stored keyframe was built with another vocabulary tree or levelsup");
    SSLPL_REQUIRE((size_t)((nc + 1 + cap) * sizeof(int)) <= (size_t)MAX_DYN_SMEM, SSLPL_ERR_CAPACITY, "nodes + features exceed the shared memory of one CTA ((nc + 1 + cap) * 4 <= 200 KB)");
    SSLPL_CUDA(cudaSetDevice(m->p.device));
    cudaStream_t st = m->stream;
    // points: the batch's dense FeatureVectors (as sslpl_match_bow_batch_device_vocab), then SearchByBoW against the slots
    k_vocab_transform<<<dim3((cap + 127) / 128, nframes), 128, 0, st>>>(d_desc, (long long)cap * 32, d_n, 0, cap, v->view, v->L - levelsup,
                                                                         nullptr, nullptr, m->b_node, nullptr, fc);
    k_build_csr<<<nframes, 128, (nc + 1 + cap) * sizeof(int), st>>>(m->b_node, fc, d_n, cap, nc, m->b_off, NN + 1, m->b_idx, fc);
    m->launches += 2;
    fill(m, d_match, (long long)nframes * cap, -1);
    SSLPL_CUDA(cudaMemsetAsync(m->b_rot, 255, (size_t)nframes * fc, st));
    SSLPL_CUDA(cudaMemsetAsync(m->b_taken, 0, (size_t)nframes * fc, st));
    FrameSet S; memset(&S, 0, sizeof(S));
    S.desc = d_desc; S.desc_fs = (long long)cap * 32;
    S.nodes = m->iota; S.nn_const = nc; S.off = m->b_off; S.idx = m->b_idx; S.off_fs = NN + 1; S.idx_fs = fc;
    S.angle = reinterpret_cast<const float*>(d_kps) + 3; S.angle_es = 7; S.angle_fs = (long long)cap * 7;
    k_bow_match_ref<<<dim3((std::min(k->view.cap, nc) + 3) / 4, nframes), 128, 0, st>>>(k->view, d_ref, S, nnratio, d_match, cap, m->b_rot, fc,
                                                                                          m->b_taken, fc);
    k_rot_filter<<<nframes, 256, 0, st>>>(d_match, cap, m->b_rot, fc, d_n, 0, 0, cap, checkOri, d_nmatch, nullptr, 0);
    // lines: knn2 of the slot's MapLine-holding lines against frame f's, then the ratio rule
    const int qcap = k->view.capl;
    k_knn2_ref<<<dim3((qcap + 7) / 8, nframes), 256, 0, st>>>(k->view, d_ref, d_ldesc, (long long)capl * 32, d_nl, capl, m->b_knn, (long long)lc * 4, qcap);
    fill(m, d_lmatch, (long long)nframes * capl, -1);
    SSLPL_CUDA(cudaMemsetAsync(d_nlmatch, 0, sizeof(int32_t) * nframes, st));
    k_line_ratio<<<dim3((qcap + 127) / 128, nframes), 128, 0, st>>>(m->b_knn, (long long)lc * 4, nullptr, qcap, qcap, nullptr, 0, d_lmatch, capl, d_nlmatch);
    m->launches += 4;
    SSLPL_CUDA(cudaGetLastError());
    SSLPL_CUDA(cudaEventRecord(k->last_use, st));
    return SSLPL_OK;
}

}  // extern "C"
